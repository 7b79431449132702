"""The rank-route cases of tests/rank_cases.py on the float64 oracle: every case visits the rank bands and band changes it
claims, and no rank decision lies within 1e-3 of its threshold (|sigma_i mu - 1| >= 1e-3 for i = svp - 1, svp), so a correct
float32 solve cannot take a different rank.  This keeps device comparisons on these cases meaningful if the generator or the
oracle changes."""
import time

import pytest

import rank_cases as RC

MIN_MARGIN = 1e-3
MAX_SECONDS = 20.0              # ten times what a case takes (one to two seconds) on an idle 8-core host


@pytest.mark.parametrize("name", sorted(RC.CASES))
def test_case_visits_its_rank_bands(name):
    case = RC.CASES[name]
    D = RC.clip_of(case)
    log = []
    t0 = time.perf_counter()
    _L, _S, it, conv, _Y = RC.oracle_solve(case, D, log=log)
    seconds = time.perf_counter() - t0
    svp = [e["svp"] for e in log]
    bands = [RC.band(r) for r in svp]
    margins = RC.boundary_margin(log)
    worst = min(range(len(margins)), key=margins.__getitem__)
    print(f"[{name}] iters={it} converged={conv} {seconds:.1f}s svp={svp}")
    print(f"[{name}] smallest boundary margin {margins[worst]:.2e} at iteration {worst + 1}; "
          f"band changes at {RC.band_changes(svp)}")
    assert conv if "max_iter" not in case else it == case["max_iter"]
    assert set(bands) == case["bands"]
    assert {(a, b) for a, b in zip(bands, bands[1:]) if a != b} == case["transitions"]
    assert bands[-1] == case["final"]
    if case["mode"] == "flat":          # sv0 > 16: no implied first iterate, iteration 1 on the rank > 16 kernel
        assert case["sv0"] > 16 and bands[0] == ">16"
    assert margins[worst] >= MIN_MARGIN
    assert seconds <= MAX_SECONDS


def test_truncated_solve_is_a_prefix():
    """A solve stopped after k iterations is the first k iterations of the whole solve (what the hand-off tests rely on), and
    the multiplier it returns is Y_k = Y_{k-1} + mu_k (D - L_k - S_k)."""
    import numpy as np
    case = RC.CASES["flat_descent"]
    D = RC.clip_of(case)
    full, part = [], []
    RC.oracle_solve(case, D, log=full)
    L3, S3, it3, _c3, Y3 = RC.oracle_solve(case, D, max_iter=3, log=part)
    L2, S2, _it2, _c2, Y2 = RC.oracle_solve(case, D, max_iter=2)
    assert it3 == 3 and [e["svp"] for e in part] == [e["svp"] for e in full[:3]]
    assert np.allclose(Y3, Y2 + part[2]["mu"] * (D - L3 - S3), rtol=0, atol=1e-12)
