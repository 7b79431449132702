"""-m gpu: the generic graph prox (any non-nested SPAMS graph, one graph per frame) against the CPU oracle -- the operator on its own
and whole decompositions on WaterSurface crops -- plus the routing of the graphs that have dedicated kernels."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as ssp

from conftest import rel_fro

pytestmark = pytest.mark.gpu

TOL_F = 1e-4


@pytest.fixture(scope="module")
def B():
    import background_subtraction_b200 as B
    return B


def _dict(indptr, indices, eta, m):
    ng = len(indptr) - 1
    gv = ssp.csc_matrix((np.ones(len(indices), dtype=bool), np.asarray(indices, dtype=np.int32), np.asarray(indptr, dtype=np.int32)),
                        shape=(m, ng))
    return {'eta_g': np.asarray(eta, dtype=np.float64), 'groups': ssp.csc_matrix((ng, ng), dtype=bool), 'groups_var': gv}


def _random_graph(m, rng, sizes=(1, 9, 25, 33, 64, 230), count=6):
    """Irregular overlapping groups of the given sizes (pixels drawn from a local neighbourhood so that they overlap), an empty
    group, and weights that include 0 and 1.5."""
    groups = []
    for k in sizes:
        for _ in range(count):
            c = int(rng.integers(0, m))
            lo = max(0, min(c - 2 * k, m - 4 * k))
            groups.append(np.sort(rng.choice(np.arange(lo, min(m, lo + 4 * k)), size=k, replace=False)))
    groups.insert(3, np.zeros(0, dtype=np.int64))
    rng.shuffle(groups)
    indptr = np.concatenate([[0], np.cumsum([len(g) for g in groups])])
    eta = rng.choice([0.0, 0.5, 1.0, 1.5], size=len(groups))
    eta[:3] = [0.0, 1.5, 1.0]
    return _dict(indptr, np.concatenate(groups), eta, m)


def _signal(m, n, seed):
    rng = np.random.default_rng(seed)
    U = rng.standard_normal((m, n)) * 0.05
    U[rng.random((m, n)) < 0.02] += 0.4                      # a few strong pixels, like foreground
    return np.asfortranarray(U.astype(np.float32).astype(np.float64))


def _covered(graph, m):
    cov = np.zeros(m, dtype=bool)
    cov[graph['groups_var'].tocsc().indices] = True
    return cov


def _weighted(graph):
    """CSC triple of the groups with eta > 0.  A group of weight 0 adds nothing to the objective, so the prox is that of the graph
    without it; the oracle's l1-ball projection degenerates at radius 0 (theta stays 0 and it returns its input), so the
    reference solution is computed on this equivalent graph."""
    from oracle import alm_oracle as O
    ip, ix, eta = O.graph_from_spams_dict(graph)
    keep = eta > 0
    sizes = np.diff(ip)[keep]
    idx = np.concatenate([ix[ip[g]:ip[g + 1]] for g in np.nonzero(keep)[0]] or [np.zeros(0, dtype=np.int32)])
    return (np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32), idx.astype(np.int32), np.ascontiguousarray(eta[keep]))


def _check_prox(B, U, graphs, per_frame):
    from oracle import alm_oracle as O
    m, n = U.shape
    for lam in (0.003, 0.08):
        if per_frame:
            ref = O.prox_by_frame(U, lam, [_weighted(g) for g in graphs], tol=1e-12)
            out = B.prox_by_frame(U, lam, graphs)
        else:
            ref = O.prox_graph(U, lam, _weighted(graphs), tol=1e-12)
            out, sw = B.prox(U, lam, graphs, return_sweeps=True, tol=1e-6)
            assert 1 <= sw < 20000
        err = np.abs(out - ref).max()
        assert err <= 2e-5 * max(np.abs(U).max(), lam), (lam, err)
        for f in range(n):                                   # pixels in no group: the input, bit for bit in fp32
            cov = _covered(graphs[f] if per_frame else graphs, m)
            assert np.array_equal(out[~cov, f].astype(np.float32), U[~cov, f].astype(np.float32))


@pytest.mark.parametrize("win", [(5, 5), (2, 4), (1, 6)])
def test_prox_window_shapes(B, win):
    h, w, t = 37, 45, 3
    _check_prox(B, _signal(h * w, t, h * win[0] + win[1]), B.getGraphSPAMS_all_groups((h, w), win), False)


def test_prox_by_frame_radius2_centre_windows(B):
    h, w, t = 26, 31, 4
    rng = np.random.default_rng(4)
    weights = [np.where(rng.random((h, w)) < 0.3, rng.choice([1.0, 1.5], (h, w)), -1.0) for _ in range(t)]
    for wm in weights:
        wm[0, 0], wm[-1, -1], wm[1, w // 2] = 1.5, 1.0, 1.0               # windows clipped at corners and an edge
    graphs = [B.get_proximal_graph_group_centers((h, w), 2, wm) for wm in weights]
    _check_prox(B, _signal(h * w, t, 5), graphs, True)


def test_prox_irregular_groups_per_frame(B):
    """Random overlapping groups of sizes 1, 9, 25, 33, 64 and 230, an empty group, eta in {0, 0.5, 1, 1.5}, a different graph
    for every frame (and one repeated), all frames in one launch."""
    m, t = 1500, 4
    rng = np.random.default_rng(11)
    graphs = [_random_graph(m, rng) for _ in range(t - 1)]
    graphs.append(graphs[0])
    _check_prox(B, _signal(m, t, 12), graphs, True)


def test_prox_single_irregular_graph(B):
    m = 1200
    _check_prox(B, _signal(m, 3, 13), _random_graph(m, np.random.default_rng(14)), False)


def test_prox_workspace_cap_forces_small_batches(B, monkeypatch):
    """BSUB_GRAPH_XI_MB=1: the dual workspace holds one frame of (5,5) windows, so the frames run one cluster at a time."""
    monkeypatch.setenv("BSUB_GRAPH_XI_MB", "1")
    h, w, t = 90, 110, 5
    _check_prox(B, _signal(h * w, t, 15), B.getGraphSPAMS_all_groups((h, w), (5, 5)), False)


def test_prox_frame_larger_than_cluster_shared_memory(B):
    """A 520 x 540 frame: its dual sums do not fit the shared memory of an 8-CTA cluster and live in global memory."""
    from oracle import alm_oracle as O
    h, w = 520, 540
    m = h * w
    rng = np.random.default_rng(16)
    groups = [np.sort(rng.choice(np.arange(c, min(m, c + 60)), size=k, replace=False))
              for c, k in zip(rng.integers(0, m - 60, size=3000), rng.choice([4, 9, 25, 40], size=3000))]
    graph = _dict(np.concatenate([[0], np.cumsum([len(g) for g in groups])]), np.concatenate(groups), np.ones(len(groups)), m)
    U = _signal(m, 2, 17)
    for lam in (0.003, 0.08):
        ref = O.prox_graph(U, lam, O.graph_from_spams_dict(graph), tol=1e-12)
        out = B.prox(U, lam, graph, tol=1e-6)
        assert np.abs(out - ref).max() <= 2e-5 * max(np.abs(U).max(), lam)


# ------------------------------------------------------------------------------------------------------------- whole solves
def _centre_weights(h, w, t, seed):
    rng = np.random.default_rng(seed)
    return [np.where(rng.random((h, w)) < 0.15, rng.choice([1.0, 1.5], (h, w)), -1.0) for _ in range(t)]


def _graph_counters(dec):
    out = (ctypes.c_int64 * 4)()
    from background_subtraction_b200 import _cabi as C
    C.check(dec.lib.bsub_debug_graph(dec.h, out))
    return [int(v) for v in out]


def _compare_solve(B, D, dec, Lr, Sr, itr, convr, log):
    L, S, it, conv = B.api._finish(dec, D, False)
    rl, rs = rel_fro(L, Lr), rel_fro(S, Sr)
    ranks, ranks_ref = [l['svp'] for l in dec.log()], [l['svp'] for l in log]
    common = min(len(ranks), len(ranks_ref))
    from oracle import alm_oracle as O
    agree = float((dec.mask(2) == O.foreground_mask(D, Lr, Sr)).mean())
    cnt = _graph_counters(dec)
    print(f"iters {it}/{itr} conv {conv}/{convr} relF(L) {rl:.2e} relF(S) {rs:.2e} mask {agree:.5f} ranks {ranks} "
          f"graph counters {cnt}")
    assert abs(it - itr) <= 1 and conv == convr
    assert ranks[:common] == ranks_ref[:common]
    assert rl <= TOL_F and rs <= TOL_F and agree >= 0.999
    assert cnt[2] >= it and cnt[3] == 0                       # one prox call per iteration, none at the sweep cap


@pytest.mark.parametrize("case", ["win55", "win24", "centre_r2_per_frame"])
def test_lsd_generic_graph_vs_oracle(B, watersurface_u8, case):
    from oracle import alm_oracle as O
    from background_subtraction_b200 import _cabi as C
    h, w, t = 40, 50, 12
    D, _x, _mean = O.normalize_and_center(watersurface_u8[:h, :w, :t])
    if case == "win55":
        graphs = B.getGraphSPAMS_all_groups((h, w), (5, 5))
    elif case == "win24":
        graphs = B.getGraphSPAMS_all_groups((h, w), (2, 4))
    else:
        graphs = [B.get_proximal_graph_group_centers((h, w), 2, wm) for wm in _centre_weights(h, w, t, 21)]
    log = []
    Lr, Sr, itr, convr = O.inexact_alm_lsd(D, graphs=graphs, log=log, prox_tol=1e-12)
    dec = B.lsd_decomposition(D, graphs=graphs, graph_tol=1e-6, graph_max_sweeps=20000)
    assert dec.cfg.prox == C.PROX_GRAPH_GENERIC
    _compare_solve(B, D, dec, Lr, Sr, itr, convr, log)


def test_with_background_radius2_vs_oracle(B, watersurface_u8):
    from oracle import alm_oracle as O
    from background_subtraction_b200 import _cabi as C
    h, w, t = 40, 50, 12
    D, _x, _mean = O.normalize_and_center(watersurface_u8[:h, :w, :t])
    W = _centre_weights(h, w, t, 22)
    graphs = [B.get_proximal_graph_group_centers((h, w), 2, wm) for wm in W]
    bgm = [(wm < 0) & (np.random.default_rng(23 + f).random((h, w)) < 0.5) for f, wm in enumerate(W)]
    bgm = [b.flatten(order='F') for b in bgm]
    log = []
    Lr, Sr, itr, convr = O.inexact_alm_lsd_with_background(D, graphs, bgm, log=log, prox_tol=1e-12)
    dec = B.with_background_decomposition(D, graphs, bgm, graph_tol=1e-6, graph_max_sweeps=20000)
    assert dec.cfg.prox == C.PROX_GRAPH_GENERIC
    _compare_solve(B, D, dec, Lr, Sr, itr, convr, log)


# ------------------------------------------------------------------------------------------------------------- routing
def test_dedicated_graphs_keep_their_kernels(B, watersurface_u8):
    from oracle import alm_oracle as O
    from background_subtraction_b200 import _cabi as C
    h, w, t = 24, 30, 6
    D, _x, _mean = O.normalize_and_center(watersurface_u8[:h, :w, :t])
    g3 = B.getGraphSPAMS_all_groups((h, w), (3, 3))
    assert B.lsd_decomposition(D, graphs=g3, max_iter=1).cfg.prox == C.PROX_GRAPH_LINF
    assert B.lsd_decomposition(D, graphs=[g3] * t, max_iter=1).cfg.prox == C.PROX_GRAPH_LINF
    W = _centre_weights(h, w, t, 24)
    r1 = [B.get_proximal_graph_group_centers((h, w), 1, wm) for wm in W]
    bgm = [(wm < 0).flatten(order='F') for wm in W]
    assert B.with_background_decomposition(D, r1, bgm, max_iter=1).cfg.prox == C.PROX_GRAPH_CENTER_BG
    assert B.lsd_decomposition(D, graphs=B.getGraphSPAMS_all_groups((h, w), (5, 5)), max_iter=1).cfg.prox == C.PROX_GRAPH_GENERIC
    assert B.lsd_decomposition(D, graphs=r1, max_iter=1).cfg.prox == C.PROX_GRAPH_GENERIC


def test_batch_with_generic_graph_matches_one_at_a_time(B, watersurface_u8):
    from oracle import alm_oracle as O
    h, w, t = 40, 50, 12
    clips = [O.normalize_and_center(watersurface_u8[:h, 10 * i:10 * i + w, 5 * i:5 * i + t])[0] for i in range(2)]
    graph = B.getGraphSPAMS_all_groups((h, w), (2, 4))
    seq = [B.inexact_alm_lsd(D, graphs=graph) for D in clips]
    par = B.inexact_alm_lsd_batch(clips, graphs=graph, in_flight=2)
    for (L0, S0, it0, c0), (L1, S1, it1, c1) in zip(seq, par):
        assert it0 == it1 and c0 == c1 and c1
        assert rel_fro(L1, L0) <= 1e-6 and rel_fro(S1, S0) <= 1e-6
