"""The rank-route cases of tests/rank_cases.py on the float64 oracle: every case visits the rank bands and band changes it
claims, and no rank decision lies within 1e-3 of its threshold (|sigma_i mu - 1| >= 1e-3 for i = svp - 1, svp), so a correct
float32 solve cannot take a different rank.  This keeps device comparisons on these cases meaningful if the generator or the
oracle changes."""
import time

import numpy as np
import pytest

import rank_cases as RC

MIN_MARGIN = 1e-3
# A converged case's stop decision (last err below tol, the one before above it) must lie this many times farther from tol than
# the float32 floor of err (how much err moves when the oracle's L and S are rounded to float32).  l1_climb at tol 1e-7 had 2.9
# and stopped one iteration late on every device path; flat_mid, the closest case that matched, has 4.9.
STOP_FLOOR_FACTOR = 4.0
MAX_SECONDS = 20.0              # ten times what a case takes (one to two seconds) on an idle 8-core host


@pytest.mark.parametrize("name", sorted(RC.CASES))
def test_case_visits_its_rank_bands(name):
    case = RC.CASES[name]
    D = RC.clip_of(case)
    log = []
    t0 = time.perf_counter()
    L, S, it, conv, _Y = RC.oracle_solve(case, D, log=log)
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
    if conv:
        tol = RC.TOL[case["mode"]]
        f32 = lambda a: a.astype(np.float32).astype(np.float64)          # noqa: E731
        floor = abs(np.linalg.norm(D - f32(L) - f32(S)) / np.linalg.norm(D) - log[-1]["err"]) / tol
        stop_margin = min(1 - log[-1]["err"] / tol, log[-2]["err"] / tol - 1)
        print(f"[{name}] stop decision: err/tol {log[-2]['err'] / tol:.3f} -> {log[-1]['err'] / tol:.3f}, "
              f"float32 floor {floor:.1e} of tol")
        assert stop_margin >= STOP_FLOOR_FACTOR * floor
    assert seconds <= MAX_SECONDS


@pytest.mark.parametrize("max_iter", [None, 3])
@pytest.mark.parametrize("name", sorted(RC.CASES))
def test_device_config_runs_the_oracle_loop(name, max_iter, monkeypatch):
    """The device solve of a case has the parameters of its oracle solve, so a wrong one shows up here and not as a rank
    mismatch on the GPU: the arguments oracle_solve hands to the oracle loop (defaults included) against RC.device_config."""
    import inspect
    from background_subtraction_b200 import _cabi as C
    from oracle import alm_oracle as O
    case = RC.CASES[name]
    rows, cols, n = case["shape"]
    seen, signature = {}, inspect.signature(O._alm)

    def spy(*args, **kw):
        bound = signature.bind(*args, **kw)
        bound.apply_defaults()
        seen.update(bound.arguments)
        return (None,) * 5
    monkeypatch.setattr(O, "_alm", spy)
    D = RC.clip_of(case)
    RC.oracle_solve(case, D, max_iter=max_iter)
    cfg, groups = RC.device_config(case, max_iter=max_iter)
    assert (cfg.m, cfg.n) == D.shape == (rows * cols, n)
    assert cfg.mu_scale == seen["mu_scale"] and cfg.delta == seen["delta"] and cfg.rho == seen["rho"]
    assert cfg.tol == seen["tol_out"] and cfg.max_iter == seen["max_iter"]
    assert bool(cfg.use_sv_prediction) == seen["use_sv_prediction"] and bool(cfg.break_on_rank0) == seen["break_on_rank0"]
    if seen["use_sv_prediction"]:
        assert cfg.sv0 == seen["sv0"]
    if case["mode"] == "l1":
        assert cfg.prox == C.PROX_L1 and groups is None
        G = np.random.default_rng(0).standard_normal((6, 5))
        assert np.array_equal(seen["prox_fn"](G, 0.3, 2.0), np.sign(G) * np.maximum(np.abs(G) - 0.15, 0))
    else:
        assert cfg.prox == C.PROX_FLAT_LINF and (cfg.rows, cfg.cols) == (rows, cols)
        assert (cfg.group_rows, cfg.group_cols) == (3, 3)
        assert np.array_equal(groups, O.flat_groups_nonoverlap((rows, cols), (3, 3)))
        G = np.asfortranarray(np.random.default_rng(0).standard_normal((rows * cols, 2)))
        assert np.array_equal(seen["prox_fn"](G, 0.3, 2.0), O.prox_flat(G, 0.15, groups))


def test_truncated_solve_is_a_prefix():
    """A solve stopped after k iterations is the first k iterations of the whole solve (what the hand-off tests rely on), and
    the multiplier it returns is Y_k = Y_{k-1} + mu_k (D - L_k - S_k)."""
    case = RC.CASES["flat_descent"]
    D = RC.clip_of(case)
    full, part = [], []
    RC.oracle_solve(case, D, log=full)
    L3, S3, it3, _c3, Y3 = RC.oracle_solve(case, D, max_iter=3, log=part)
    L2, S2, _it2, _c2, Y2 = RC.oracle_solve(case, D, max_iter=2)
    assert it3 == 3 and [e["svp"] for e in part] == [e["svp"] for e in full[:3]]
    assert np.allclose(Y3, Y2 + part[2]["mu"] * (D - L3 - S3), rtol=0, atol=1e-12)
