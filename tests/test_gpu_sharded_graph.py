"""-m gpu: the graph modes that run their prox on whole frames (bsub_set_frame_* + bsub_step_prox_block) and the l1 mode, through
dist.ShardedLSD at world size 1 against bsub_run on the whole-clip handle; the prox of each iteration split into frame blocks with
explicit first frames (what the ranks of a multi-GPU run do, on one GPU); and the errors of the frame-range entry points."""
import ctypes

import numpy as np
import pytest

from conftest import rel_fro

pytestmark = pytest.mark.gpu

H, W, T = 48, 60, 12


@pytest.fixture(scope="module")
def B():
    import background_subtraction_b200 as B
    return B


class Solo:
    world, rank = 1, 0

    def all_reduce_sum(self, t_):
        pass

    def all_reduce_max(self, t_):
        pass


@pytest.fixture(scope="module")
def D(watersurface_u8):
    from oracle import alm_oracle as O
    D, _x, _mean = O.normalize_and_center(watersurface_u8[:H, :W, :T])
    return D


def _weight_mask(seed=2):
    """LSD_improved-style map [h, w, t]: positive = weight of the centre window, negative = background, 0 = neither; different in
    every frame (frame 4 has no window, frame 7 no background)."""
    rng = np.random.default_rng(seed)
    wm = np.zeros((H, W, T))
    for f in range(T):
        r = rng.random((H, W))
        if f != 4:
            wm[:, :, f] = np.where(r < 0.2, rng.uniform(0.5, 3.0, (H, W)), 0.0)
        if f != 7:
            wm[:, :, f] = np.where(r > 0.6, -1.0, wm[:, :, f])
    return wm


def _generic_graphs(B, seed=4):
    """Per-frame graphs the tile kernel does not take (radius-2 centre windows at random centres, 2 x 5 windows with random
    weights), different in every frame; frame 4 has no window.  Background masks: random, frame 7 empty."""
    rng = np.random.default_rng(seed)
    graphs, bg = [], []
    for f in range(T):
        if f == 4:
            graphs.append(B.get_proximal_graph_group_centers((H, W), 2, np.zeros((H, W))))
        elif f % 2:
            g = B.getGraphSPAMS_all_groups((H, W), (2, 5))
            g['eta_g'] = rng.uniform(0.5, 2.0, len(g['eta_g']))
            graphs.append(g)
        else:
            centres = np.where(rng.random((H, W)) < 0.15, rng.uniform(0.5, 2.0, (H, W)), -1.0)
            graphs.append(B.get_proximal_graph_group_centers((H, W), 2, centres))
        bg.append(np.zeros(H * W, dtype=bool) if f == 7 else rng.random(H * W) < 0.4)
    return graphs, bg


def _window_graph(B):
    g = B.getGraphSPAMS_all_groups((H, W), (3, 3))
    g['eta_g'] = np.random.default_rng(6).uniform(0.5, 2.0, len(g['eta_g']))
    return g


def _whole_clip(B, D, mode):
    """bsub_run on the handle the public solver builds, and the CudaStepSolver arguments of the same problem."""
    from background_subtraction_b200 import _cabi as C
    if mode == "generic":
        graphs, _ = _generic_graphs(B)
        return B.lsd_decomposition(D, graphs=graphs, img_shape=(H, W)), dict(graphs=graphs, graph_cols=W)
    if mode == "generic_bg":
        graphs, bg = _generic_graphs(B)
        return (B.with_background_decomposition(D, graphs, bg, img_shape=(H, W)),
                dict(graphs=graphs, background_masks=bg, graph_cols=W))
    if mode == "centre_bg":
        wm = _weight_mask()
        return B.center_window_decomposition(D, wm), dict(weight_mask=wm)
    if mode == "windows_eta":
        g = _window_graph(B)
        return B.lsd_decomposition(D, graphs=g), dict(graphs=g, graph_cols=W)
    if mode == "windows":                                        # the reference's default LSD(): unit weights, graph_cols alone
        return B.lsd_decomposition(D, graphs=B.getGraphSPAMS_all_groups((H, W), (3, 3))), dict(graph_cols=W)
    cfg = B.make_config(H * W, T, C.PROX_L1, 0, 0, delta=1.0, mu_scale=1.25, rho=1.2, use_sv_prediction=False)   # inexact_alm_rpca
    dec = B.Decomposition(cfg)
    dec.load(D)
    dec.run()
    return dec, dict(l1=True)


def _sharded(D, kw, cls=None):
    import torch
    from background_subtraction_b200 import dist as bdist
    s = (cls or bdist.CudaStepSolver)(H, W, T, H * W, **kw)
    s.load(np.ascontiguousarray(D.T, dtype=np.float32))
    drv = bdist.ShardedLSD(s, Solo())
    drv.solve()
    drv.finish(2.0, want_mask=False)
    torch.cuda.synchronize()
    return s


@pytest.mark.parametrize("mode,prox", [("generic", 5), ("generic_bg", 5), ("centre_bg", 4), ("windows_eta", 1), ("windows", 1),
                                       ("l1", 3)])
def test_mode_through_sharded_driver_matches_bsub_run(B, D, mode, prox):
    dec, kw = _whole_clip(B, D, mode)
    assert dec.cfg.prox == prox
    st0, log0, S0 = dec.status(), dec.log(), dec.download('S')
    s = _sharded(D, kw)
    assert s.dec.cfg.prox == prox
    st, log = s.status(), s.dec.log()
    assert st.iter == st0.iter and bool(st.converged) and bool(st0.converged)
    assert [l['svp'] for l in log] == [l['svp'] for l in log0]
    assert rel_fro(s.dec.download('S'), S0) <= 1e-6
    if mode != "l1":
        calls, capped = s.debug_graph()[2:]
        assert calls >= st.iter and capped == 0


@pytest.mark.parametrize("mode", ["generic_bg", "centre_bg", "windows_eta"])
def test_prox_in_frame_blocks_matches_one_block(B, D, mode):
    """The prox of every iteration as three frame blocks [0, 5), [5, 7), [7, 12) with their own first frame: with per-frame graphs,
    weights and backgrounds, a block that read another frame's description would change the result."""
    from background_subtraction_b200 import dist as bdist

    class Blocks(bdist.CudaStepSolver):
        def prox_frames(self, Uf, Vf, rows, cols, nf):
            assert nf == T and self.frame_range == (0, T)
            for a, b in ((0, 5), (5, 7), (7, 12)):
                self.prox_block(Uf[a:], Vf[a:], a, b - a)

    _dec, kw = _whole_clip(B, D, mode)
    one = _sharded(D, kw)
    three = _sharded(D, kw, Blocks)
    st1, st3 = one.status(), three.status()
    assert st3.iter == st1.iter and bool(st3.converged)
    assert [l['svp'] for l in three.dec.log()] == [l['svp'] for l in one.dec.log()]
    assert rel_fro(three.dec.download('S'), one.dec.download('S')) <= 1e-6
    assert three.debug_graph()[3] == 0 and three.debug_graph()[2] >= 3 * st3.iter


def test_frame_range_errors(B, D):
    import torch
    from background_subtraction_b200 import _cabi as C
    from background_subtraction_b200 import dist as bdist
    wm = _weight_mask()
    # a block outside the described range
    s = _sharded(D, dict(weight_mask=wm))
    U = torch.zeros((T, s.dec.m), dtype=torch.float32, device="cuda")
    with pytest.raises(Exception, match=r"frames \[10, 13\) are outside the described range \[0, 12\)"):
        s.prox_block(U, U, 10, 3)
    s.prox_block(U, U, 12, 0)                                    # an empty block at the end is a no-op
    # descriptions of the wrong size, refused before anything is uploaded
    dec = B.Decomposition(B.make_config(H * W, T, C.PROX_GRAPH_LINF, H, W))
    with pytest.raises(Exception, match="eta has 3 entries"):
        e = np.ones(3)
        C.check(dec.lib.bsub_set_frame_windows(dec.h, H, W, 0, T, e.ctypes.data_as(C.c_double_p), 3))
    with pytest.raises(Exception, match=r"frames \[6, 13\) are not a range of the 12 frames"):
        C.check(dec.lib.bsub_set_frame_windows(dec.h, H, W, 6, 7, None, 0))
    dec_g = B.Decomposition(B.make_config(H * W, T, C.PROX_GRAPH_GENERIC, H, W))
    route = B.api.route_graphs(B.getGraphSPAMS_all_groups((H + 1, W), (2, 2)), (H + 1) * W, T, (H + 1, W))
    route.rows = H                                               # graphs of a taller frame: pixel indices out of range
    with pytest.raises(Exception, match="not in \\[0, %d\\)" % (H * W)):
        dec_g.set_frame_route(route, 0, T)
    with pytest.raises(Exception, match="not created with BSUB_PROX_GRAPH_GENERIC"):
        dec.set_frame_route(route, 0, T)
    with pytest.raises(Exception, match="weight_mask must be"):
        bdist.CudaStepSolver(H, W, T, H * W, weight_mask=wm[:, :, :T - 1])
    # a handle with only a frame-range description has no graph of its own pixels
    dec_c = B.Decomposition(B.make_config(H * W, T, C.PROX_GRAPH_CENTER_BG, H, W))
    dec_c.set_frame_route(B.api.route_weight_mask(wm, H * W, T), 0, T)
    dec_c.load(D)
    with pytest.raises(Exception, match="only a frame-range description"):
        dec_c.run()
    # the frame range must be the rank's shard_frames
    s2 = bdist.CudaStepSolver(H, W, T, H * W, weight_mask=wm, frames=(0, 6))
    with pytest.raises(Exception, match=r"describes frames \[0, 6\), but rank 0 of 1 owns \[0, 12\)"):
        bdist.ShardedLSD(s2, Solo())
