"""-m gpu: the ALM loop on the device above rank 8, held to the float64 oracle on the rank-route cases of tests/rank_cases.py.

The solver picks its shrink kernel on the device, once per iteration, from that iteration's rank svp (solver.cu step_shrink_impl):
  rank <= 8 from iteration 2 on, digit planes present   'flat'    shrink_flat_kernel; S stored only when the iteration may be the last
  rank 9..16, or <= 8 without planes                    'stream'  shrink_stream_kernel; T from project_planes_kernel when planes exist
  rank > 16                                             'tma'     shrink_tma_kernel; writes no planes, the next Gram is the fp64 one
  any rank when rows % 4 != 0                           'shrink'  shrink_kernel (shrink.cu) and the fp64 Gram throughout
No rank decision of these cases lies within 1e-3 of its threshold (tests/test_host_rank_routes.py), so a correct float32 solve
takes the oracle's rank in every iteration.  ALM corrects itself: a solve can still converge to the right L and S after one
slightly wrong iteration on a new kernel.  So besides whole solves, every case is stopped on both sides of each band change (and
after its first iteration) and compared there with the oracle stopped at the same iteration, to bounds set from measurement."""
import numpy as np
import pytest

import rank_cases as RC
from conftest import rel_fro

pytestmark = pytest.mark.gpu

NAMES = sorted(RC.CASES)
TOL_F = 1e-4            # whole solves: the north-star bound of test_gpu_parity.py
# Y = Y + mu Z adds float32 noise of Z times a mu that grows geometrically: rounding only the oracle's final L and S to float32
# moves Y of the converged flat cases by 4e-3 to 6e-3 relative.  Measured on a B200: 1.9e-3 (flat_high) at most.
TOL_Y = 5e-3
# err per iteration: rtol 1e-3 above a floor of 1e-8 (np.allclose's default atol, as in test_gpu_parity.py).  Near tol = 1e-7 the
# float32 floor of err is a few 1e-9 (rounding the oracle's final L and S to float32 moves it by 2e-9 to 3e-9), so no float32
# solve matches 1e-3 there; the flat cases measured 3e-3 to 1.6e-2 relative in their last iterations.
ERR_RTOL, ERR_ATOL = 1e-3, 1e-8
NNZ_ABS = 8             # |nnz(S) - oracle nnz| per iteration (measured on a B200: up to 5, l1_climb_odd_m): entries at the threshold

# Stopped solves: L and S by the kernel of the stopped (last) iteration, Y by mode.  Largest relF measured over all cases on one
# B200 (NVIDIA B200, 1000 W power limit):
#   stream  L 7.0e-7  S 1.06e-6      flat  L 3.4e-7  S 5.0e-7      tma  L 1.4e-7  S 3.2e-7      shrink  L 1.2e-7  S 2.7e-7
#   Y: l1 2.4e-7, flat 1.30e-5
# Bounds are at most 10x those and no looser than 1e-5, except flat-mode Y: there one float32 rounding of L and S alone moves Y
# by up to 2.0e-5 (flat_descent stopped at 6, mu = 3.2), so its bound sits at 2.3x the measured value.
STOPPED_BOUND = {
    "stream": {"L": 5e-6, "S": 1e-5},
    "flat": {"L": 3e-6, "S": 4e-6},
    "tma": {"L": 1e-6, "S": 3e-6},
    "shrink": {"L": 1e-6, "S": 2e-6},
}
STOPPED_BOUND_Y = {"l1": 2e-6, "flat": 3e-5}

# fast paths against fallbacks: environment (read when the handle is created) and config flags of the fallback solve, and the
# debug_info entries that must read 0 on even-m clips to show that the fallback was taken
FALLBACKS = {
    "no_flat": (dict(BSUB_NO_FLAT="1"), 0, ("flat_stages",)),
    "no_proj": (dict(BSUB_NO_PROJ="1"), 0, ("use_proj", "flat_stages")),
    "no_i8_no_stream": (dict(BSUB_NO_I8="1", BSUB_NO_STREAM="1"), 0, ("use_i8", "use_stream", "use_proj", "flat_stages")),
    "always_store_S": ({}, 1, ()),          # 1 = FLAG_ALWAYS_STORE_S: S stored every iteration instead of left stale
}


@pytest.fixture(autouse=True)
def _default_routes(monkeypatch):
    import os
    for k in [k for k in os.environ if k.startswith("BSUB_")]:
        monkeypatch.delenv(k)


@pytest.fixture(scope="module")
def clip():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = RC.clip_of(RC.CASES[name])
        return cache[name]
    return get


@pytest.fixture(scope="module")
def oracle(clip):
    """oracle(name, max_iter=None) -> dict(L, S, Y, it, conv, log), cached for the module."""
    cache = {}

    def get(name, max_iter=None):
        if (name, max_iter) not in cache:
            log = []
            L, S, it, conv, Y = RC.oracle_solve(RC.CASES[name], clip(name), max_iter=max_iter, log=log)
            cache[(name, max_iter)] = dict(L=L, S=S, Y=Y, it=it, conv=conv, log=log)
        return cache[(name, max_iter)]
    return get


@pytest.fixture(scope="module")
def device(clip):
    """device(name, max_iter=None, flags=0) -> dict(L, S, Y, it, conv, log, info) of the solve RC.device_config describes."""
    import background_subtraction_b200 as B

    def solve(name, max_iter=None, flags=0):
        cfg, groups = RC.device_config(RC.CASES[name], max_iter=max_iter, flags=flags)
        dec = B.Decomposition(cfg)
        try:
            if groups is not None:
                dec.set_flat_groups(groups)
            dec.load(clip(name))
            dec.run()
            st = dec.status()
            return dict(it=int(st.iter), conv=bool(st.converged), log=dec.log(), info=dec.debug_info(),
                        L=dec.download('L'), S=dec.download('S'), Y=dec.download('Y'))
        finally:
            dec.close()
    return solve


@pytest.fixture(scope="module")
def measured():
    """Largest relF of the stopped solves per (kernel, quantity), printed when the module ends."""
    worst = {}
    yield worst
    print("\n[rank routes] largest relF of the stopped solves, by kernel of the last iteration:")
    for kern in sorted(worst):
        print("  %-7s %s" % (kern, "  ".join("%s %.2e" % (q, v) for q, v in sorted(worst[kern].items()))))


def kernels(info, svp):
    """Shrink kernel of each iteration, as step_shrink_impl picks it from the rank sequence (a rank > 16 pass writes no planes)."""
    if not info["use_tma"]:
        return ["shrink"] * len(svp)
    out = []
    for i, r in enumerate(svp):
        planes = i > 0 and svp[i - 1] <= 16
        out.append("tma" if r > 16 else ("flat" if r <= 8 and planes and info["flat_stages"] > 0 else "stream"))
    return out


@pytest.mark.parametrize("name", NAMES)
def test_routes_are_what_the_case_claims(name, device):
    """The kernels each case is meant to exercise are the ones the handle selected: TMA, streamed, planes and single-pass kernels
    on the even-m clips (48 x 60 at 40 and 300 frames).  l1_climb_odd_m (m = 47 x 61, rows % 4 != 0) uses none of them: it tests
    shrink_kernel (shrink.cu) and the fp64 gram_dmma_kernel across all three rank bands."""
    info = device(name, max_iter=1)["info"]
    print(f"[{name}] debug_info {info}")
    if name == "l1_climb_odd_m":
        assert info["use_tma"] == info["use_stream"] == info["use_i8"] == 0
    else:
        assert info["use_tma"] == info["use_stream"] == info["use_i8"] == info["use_proj"] == 1
        assert info["stream_R"] == 48 and info["flat_stages"] > 0


@pytest.mark.parametrize("name", NAMES)
def test_whole_solve_matches_the_oracle(name, oracle, device):
    case = RC.CASES[name]
    ref, dev = oracle(name), device(name)
    dl, ol = dev["log"], ref["log"]
    svp, osvp = [e["svp"] for e in dl], [e["svp"] for e in ol]
    rel = {q: rel_fro(dev[q], ref[q]) for q in "LSY"}
    err_rel = max(abs(a["err"] - b["err"]) / b["err"] for a, b in zip(dl, ol)) if len(dl) == len(ol) else float("inf")
    err_ok = len(dl) == len(ol) and np.allclose([e["err"] for e in dl], [e["err"] for e in ol], rtol=ERR_RTOL, atol=ERR_ATOL)
    nnz_diff = max(abs(a["nnz"] - b["nnz"]) for a, b in zip(dl, ol)) if len(dl) == len(ol) else -1
    print(f"[{name}] debug_info {dev['info']}")
    print(f"[{name}] iters {dev['it']}/{ref['it']} converged {dev['conv']}/{ref['conv']} svp {svp}")
    print(f"[{name}] kernels {kernels(dev['info'], svp)}")
    print(f"[{name}] whole solve relF L {rel['L']:.2e} S {rel['S']:.2e} Y {rel['Y']:.2e}; max rel err diff {err_rel:.2e}; "
          f"max |nnz diff| {nnz_diff}")
    assert dev["it"] == ref["it"] and dev["conv"] == ref["conv"]
    if "max_iter" in case:
        assert dev["it"] == case["max_iter"] and not dev["conv"]
    assert svp == osvp
    assert [e["sv"] for e in dl] == [e["sv"] for e in ol]
    if case["mode"] == "l1":
        assert all(e["sv"] == case["shape"][2] for e in dl)
    cfg, _g = RC.device_config(case)
    assert dl[0]["mu"] == pytest.approx(ol[0]["mu"], rel=1e-6)
    assert all(b["mu"] == pytest.approx(a["mu"] * cfg.rho, rel=1e-12) for a, b in zip(dl, dl[1:]))
    assert err_ok
    assert rel["L"] <= TOL_F and rel["S"] <= TOL_F and rel["Y"] <= TOL_Y
    assert 0 <= nnz_diff <= NNZ_ABS


@pytest.mark.parametrize("name", NAMES)
def test_solves_stopped_at_band_changes(name, oracle, device, measured):
    """Stopped after the last iteration on the old kernel (k - 1) and after the first on the new one (k), for every band change
    k of the oracle run, and after iteration 1: L, S and Y against the oracle stopped at the same iteration.  The last iteration
    of a stopped solve stores S (shrink_flat_kernel: iter >= max_iter), and bsub_finalize rebuilds S when it is stale."""
    full = oracle(name)
    svp = [e["svp"] for e in full["log"]]
    stops = sorted({1} | {j for k in RC.band_changes(svp) for j in (k - 1, k)})
    results = []
    for k in stops:
        ref, dev = oracle(name, k), device(name, max_iter=k)
        kern = kernels(dev["info"], svp)[k - 1]
        rel = {q: rel_fro(dev[q], ref[q]) for q in "LSY"}
        mode = RC.CASES[name]["mode"]
        for key, q in ((kern, "L"), (kern, "S"), ("Y " + mode, "Y")):
            w = measured.setdefault(key, {})
            w[q] = max(w.get(q, 0.0), rel[q])
        print(f"[{name}] stopped at {k} (rank {svp[k - 1]}, {kern}): relF L {rel['L']:.2e} S {rel['S']:.2e} Y {rel['Y']:.2e}")
        results.append((k, kern, ref, dev, rel))
    for k, kern, ref, dev, rel in results:
        assert dev["it"] == ref["it"] == k and dev["conv"] == ref["conv"]
        assert [e["svp"] for e in dev["log"]] == svp[:k]
        for q in "LS":
            assert rel[q] <= STOPPED_BOUND[kern][q], f"stopped at {k} ({kern}): relF({q}) {rel[q]:.3e}"
        assert rel["Y"] <= STOPPED_BOUND_Y[mode], f"stopped at {k} ({kern}): relF(Y) {rel['Y']:.3e}"


@pytest.mark.parametrize("fallback", sorted(FALLBACKS))
@pytest.mark.parametrize("name", NAMES)
def test_fast_paths_match_fallbacks(name, fallback, device, monkeypatch):
    """The default kernels against the fallback the variable or flag selects, on the whole solve: single-pass kernel off, planes
    projection off, int8 Gram and streamed kernel off, and S stored in every iteration instead of rebuilt when stale."""
    env, flags, off = FALLBACKS[fallback]
    fast = device(name)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    slow = device(name, flags=flags)
    rl, rs = rel_fro(fast["L"], slow["L"]), rel_fro(fast["S"], slow["S"])
    print(f"[{name} vs {fallback}] iters {fast['it']}/{slow['it']} relF L {rl:.2e} S {rs:.2e} debug_info {slow['info']}")
    for key in off:
        assert slow["info"][key] == 0
    assert fast["it"] == slow["it"] and fast["conv"] == slow["conv"]
    assert [e["svp"] for e in fast["log"]] == [e["svp"] for e in slow["log"]]
    assert rl <= 2e-5 and rs <= 2e-4
