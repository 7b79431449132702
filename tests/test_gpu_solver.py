"""-m gpu: end-to-end parity of the CUDA ALM solvers (through the Python mirror -> C ABI) against the CPU oracle
and the committed golden vectors.  Tolerances are the north-star ones: rel-Frobenius(L), (S) <= 1e-4 (fp32),
iteration count within +-1, masks identical on >= 99.9 % of the pixels."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, crop_D, rel_fro

pytestmark = pytest.mark.gpu

TOL_F = 1e-4


@pytest.fixture(scope="module")
def B():
    import background_subtraction_b200 as B
    return B


def _report(name, dec_or_log, it, conv, L, S, Lr, Sr):
    print(f"[{name}] iters={it} conv={conv} relF(L)={rel_fro(L, Lr):.3e} relF(S)={rel_fro(S, Sr):.3e}")


@pytest.mark.parametrize("case", ["flat_a", "flat_b"])
def test_flat_lsd_golden_small(B, golden_cases, watersurface_u8, case):
    D, shp = crop_D(watersurface_u8, golden_cases[case + "_crop"])
    groups = golden_cases[case + "_groups"]
    dec = B.lsd_decomposition(D, groups=groups)
    st = dec.status()
    L, S = dec.download('L'), dec.download('S')
    log = dec.log()
    _report(case, log, st.iter, st.converged, L, S, golden_cases[case + "_L"], golden_cases[case + "_S"])
    print("svp gpu", [l['svp'] for l in log], "ref", golden_cases[case + "_svp"].tolist())
    print("err gpu", ["%.2e" % l['err'] for l in log][-4:], "ref", golden_cases[case + "_err"][-4:])
    assert st.iter == int(golden_cases[case + "_iter"])
    assert bool(st.converged) == bool(golden_cases[case + "_conv"])
    assert [l['svp'] for l in log] == golden_cases[case + "_svp"].tolist()          # rank sequence of the reference run
    assert np.allclose([l['err'] for l in log], golden_cases[case + "_err"], rtol=2e-3)
    assert rel_fro(L, golden_cases[case + "_L"]) <= TOL_F
    assert rel_fro(S, golden_cases[case + "_S"]) <= TOL_F
    mask = dec.mask(2)
    ref = np.unpackbits(golden_cases[case + "_mask"])[:D.size].reshape(D.shape, order='F').astype(bool)
    assert (mask == ref).mean() >= 0.999


def test_flat_lsd_watersurface(B, watersurface_u8):
    from oracle import alm_oracle as O
    with open(os.path.join(GOLDEN, "golden_summary.json")) as f:
        gold = json.load(f)["watersurface_flat_delta10"]
    D, _x, _mean = O.normalize_and_center(watersurface_u8)
    groups = B.get_proximal_flat_groups_nonoverlap((128, 160), (3, 3))
    L, S, it, conv = B.inexact_alm_lsd(D, groups=groups)
    assert np.isfortran(L) and L.dtype == np.float64 and L.shape == D.shape
    olog = []
    Lr, Sr, itr, convr = O.inexact_alm_lsd(D, groups=groups, log=olog)
    _report("watersurface flat", None, it, conv, L, S, Lr, Sr)
    assert itr == gold["iters"] and [l["svp"] for l in olog] == gold["svp"]      # oracle == reference golden
    assert abs(it - gold["iters"]) <= 1 and conv == gold["converged"]
    assert rel_fro(L, Lr) <= TOL_F and rel_fro(S, Sr) <= TOL_F
    assert abs(np.linalg.norm(L) - gold["normL"]) <= 1e-4 * gold["normL"]
    mask = B.foreground_mask(D, L, S)
    mref = O.foreground_mask(D, Lr, Sr)
    assert (mask == mref).mean() >= 0.999
    gm = np.unpackbits(np.load(os.path.join(GOLDEN, "watersurface_flat_mask.npz"))["mask"])[:D.size]
    assert (mask.ravel(order='F') == gm.astype(bool)).mean() >= 0.999


def test_flat_lsd_delta1_and_tuning(B, watersurface_u8):
    from oracle import alm_oracle as O
    D, _x, _mean = O.normalize_and_center(watersurface_u8[:64, :96, :24])
    groups = B.get_proximal_flat_groups_nonoverlap((64, 96), (3, 3))
    Lr, Sr, itr, convr = O.inexact_alm_lsd(D, groups=groups, delta=1)
    for tune in (dict(), dict(tile_rows=12, cluster_frames=1), dict(tile_rows=24, cluster_frames=4), dict(tile_rows=60, cluster_frames=8)):
        L, S, it, conv = B.inexact_alm_lsd(D, groups=groups, delta=1, **tune)
        _report("delta1 %s" % tune, None, it, conv, L, S, Lr, Sr)
        assert abs(it - itr) <= 1 and conv == convr
        assert rel_fro(L, Lr) <= TOL_F and rel_fro(S, Sr) <= TOL_F


def test_flat_generic_groups(B, watersurface_u8):
    """An arbitrary partition (4x2 tiles) takes the generic two-phase path."""
    from oracle import alm_oracle as O
    D, _x, _mean = O.normalize_and_center(watersurface_u8[:40, :50, :12])
    groups = O.flat_groups_nonoverlap((40, 50), (4, 2))
    Lr, Sr, itr, convr = O.inexact_alm_lsd(D, groups=groups)
    L, S, it, conv = B.inexact_alm_lsd(D, groups=groups)
    _report("generic groups", None, it, conv, L, S, Lr, Sr)
    assert abs(it - itr) <= 1 and conv == convr
    assert rel_fro(L, Lr) <= TOL_F and rel_fro(S, Sr) <= TOL_F


def test_group_sparse_golden(B, golden_cases, watersurface_u8):
    D, shp = crop_D(watersurface_u8, golden_cases["gs_a_crop"])
    labels = golden_cases["gs_a_labels"]
    ptr, lam = golden_cases["gs_a_lam_ptr"], golden_cases["gs_a_lam"]
    n, m = labels.shape
    blocks = [[labels[f] == b + 1 for b in range(ptr[f + 1] - ptr[f])] for f in range(n)]
    lambdas = [[lam[ptr[f] + b] for b in range(ptr[f + 1] - ptr[f])] for f in range(n)]
    L, S, it, conv = B.inexact_alm_group_sparse_RPCA(D, blocks, lambdas, delta=10)
    _report("gs_a", None, it, conv, L, S, golden_cases["gs_a_L"], golden_cases["gs_a_S"])
    assert abs(it - int(golden_cases["gs_a_iter"])) <= 1
    assert conv == bool(golden_cases["gs_a_conv"])
    assert rel_fro(L, golden_cases["gs_a_L"]) <= TOL_F and rel_fro(S, golden_cases["gs_a_S"]) <= TOL_F


def test_graph_lsd_golden(B, golden_cases, watersurface_u8):
    D, shp = crop_D(watersurface_u8, golden_cases["graph_a_crop"])
    graph = B.getGraphSPAMS_all_groups(shp[:2], (3, 3))
    dec = B.lsd_decomposition(D, graphs=graph, graph_tol=1e-6, graph_max_sweeps=20000)
    L, S, it, conv = B.api._finish(dec, D, False)
    _report("graph_a", None, it, conv, L, S, golden_cases["graph_a_L"], golden_cases["graph_a_S"])
    assert it == int(golden_cases["graph_a_iter"]) and conv == bool(golden_cases["graph_a_conv"])
    assert [l['svp'] for l in dec.log()] == golden_cases["graph_a_svp"].tolist()
    mask = dec.mask(2)
    ref = np.unpackbits(golden_cases["graph_a_mask"])[:D.size].reshape(D.shape, order='F').astype(bool)
    assert (mask == ref).mean() >= 0.999
    assert rel_fro(L, golden_cases["graph_a_L"]) <= TOL_F and rel_fro(S, golden_cases["graph_a_S"]) <= TOL_F


def test_redescribed_graph_windows_replace_the_weights(B, watersurface_u8):
    """A whole-clip window handle given per-window weights and then re-described with unit weights (NULL) solves as a fresh
    unit-weight handle does: each description replaces the previous one."""
    from background_subtraction_b200 import _cabi as C
    from oracle import alm_oracle as O
    h, w, t = 48, 60, 12
    D, _x, _mean = O.normalize_and_center(watersurface_u8[:h, :w, :t])

    def solve(*etas):
        dec = B.Decomposition(B.make_config(h * w, t, C.PROX_GRAPH_LINF, h, w))
        for eta in etas:
            dec.set_graph_windows(eta)
        dec.load(D)
        dec.run()
        return dec.status(), [l['svp'] for l in dec.log()], dec.download('S')
    st0, svp0, S0 = solve(None)
    st1, svp1, S1 = solve(np.random.default_rng(7).uniform(0.2, 3.0, (h - 2) * (w - 2)), None)
    assert st1.iter == st0.iter and svp1 == svp0
    assert rel_fro(S1, S0) <= 1e-6


def test_with_background_golden(B, watersurface_u8):
    """inexact_alm_lsd_with_background (SURVEY 8f row 1) against what the reference's own loop produced: per-frame
    centre-window graphs (built here and handed over as SPAMS dicts) + background l2 shrink."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_bg.npz"))
    D, shp = crop_D(watersurface_u8, g["bg_a_crop"])
    W = g["bg_a_weights"].astype(np.float64)
    graphs = [B.get_proximal_graph_group_centers(shp[:2], 1, W[:, :, f]) for f in range(shp[2])]
    for gr in graphs[:3]:                          # exercise the detection from a bare SPAMS dict as the reference builds it
        gr.pop('_group_centers'); gr.pop('_group_radius')
    bgm = [(W[:, :, f] < 0).flatten(order='F') for f in range(shp[2])]
    L, S, it, conv = B.inexact_alm_lsd_with_background(D, graphs, bgm, graph_tol=1e-6, graph_max_sweeps=20000)
    _report("bg_a", None, it, conv, L, S, g["bg_a_L"], g["bg_a_S"])
    assert abs(it - int(g["bg_a_iter"])) <= 1 and conv == bool(g["bg_a_conv"])
    assert rel_fro(L, g["bg_a_L"]) <= TOL_F and rel_fro(S, g["bg_a_S"]) <= TOL_F
    with pytest.raises(Exception, match="graphs must be list/array"):
        B.inexact_alm_lsd_with_background(D, graphs[0], bgm)
    # stand-alone background operator (lsd_improvement.py:199-212)
    from oracle import alm_oracle as O
    rng = np.random.default_rng(3)
    G = np.asfortranarray(rng.standard_normal(D.shape) * 0.2)
    out = np.asfortranarray(rng.standard_normal(D.shape))
    ref = O.apply_background_shrinkage_operator(G, out.copy(order='F'), 0.7, bgm)
    got = B.apply_background_shrinkage_operator(G, out.copy(order='F'), 0.7, bgm)
    assert rel_fro(got, ref) <= 1e-6


def test_fmeasure_parity_synthetic(B):
    """north_star acceptance: the CUDA mask and the reference-algorithm mask score the same F-measure (compute_score.py
    metric, restated in oracle/score_oracle.py) against the known foreground of a synthetic clip; masks agree >= 99.9 %."""
    from background_subtraction_b200 import synth
    from oracle import alm_oracle as O
    from oracle import score_oracle as SC
    rows, cols, n = 48, 60, 24
    video, gt = synth.make_clip(rows, cols, n, seed=21, n_rect=2, return_gt=True)
    D = np.asfortranarray(synth.preprocess_u8(video).T.astype(np.float64))
    groups = B.get_proximal_flat_groups_nonoverlap((rows, cols), (3, 3))
    L, S, it, conv = B.inexact_alm_lsd(D, groups=groups)
    Lr, Sr, itr, convr = O.inexact_alm_lsd(D, groups=groups)
    assert abs(it - itr) <= 1 and conv == convr
    mask, mref = B.foreground_mask(D, L, S), O.foreground_mask(D, Lr, Sr)
    assert (mask == mref).mean() >= 0.999
    cube = lambda a: np.asarray(a).reshape((rows, cols, n), order='F')          # noqa: E731
    f_gpu, f_ref = SC.mean_fscore(cube(mask), cube(gt.T)), SC.mean_fscore(cube(mref), cube(gt.T))
    print("F-measure gpu %.4f  reference algorithm %.4f" % (f_gpu, f_ref))
    assert abs(f_gpu - f_ref) <= 1e-3


@pytest.mark.parametrize("rows,cols,n", [(48, 60, 600), (96, 63, 130)])
def test_fast_paths_match_fallback(B, rows, cols, n):
    """The tensor-core / streamed kernels (int8 Gram incl. the 5-block and 2-block layouts, rank cap 8 of long clips,
    implied first iterate) against the fp64-Gram + cluster-kernel fallback on the same clip."""
    from background_subtraction_b200 import synth
    video, _ = synth.make_clip(rows, cols, n, seed=33, n_rect=2)
    D = np.asfortranarray(synth.preprocess_u8(video).T.astype(np.float64))
    groups = B.get_proximal_flat_groups_nonoverlap((rows, cols), (3, 3))
    keys = ("BSUB_NO_I8", "BSUB_NO_STREAM")
    old = {k: os.environ.get(k) for k in keys}
    try:
        for k in keys:
            os.environ.pop(k, None)
        dec = B.lsd_decomposition(D, groups=groups, img_shape=(rows, cols))
        info = dec.debug_info()
        L1, S1, it1, c1 = B.api._finish(dec, D, False)
        for k in keys:
            os.environ[k] = "1"
        L0, S0, it0, c0 = B.inexact_alm_lsd(D, groups=groups, img_shape=(rows, cols))
    finally:
        for k in keys:
            if old[k] is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = old[k]
    assert info["use_stream"] == 1 and info["use_i8"] == 1
    assert it1 == it0 and c1 == c0
    assert rel_fro(L1, L0) <= 2e-5 and rel_fro(S1, S0) <= 2e-4


def test_batch_of_clips_in_flight(B):
    """BASELINE.json config 5 in miniature: independent clips decomposed with several solver handles in flight (threads +
    streams) give what one clip at a time gives."""
    from background_subtraction_b200 import synth
    rows, cols, n = 48, 63, 40
    clips = [np.asfortranarray(synth.preprocess_u8(synth.make_clip(rows, cols, n, seed=100 + i, n_rect=2)[0]).T.astype(np.float64))
             for i in range(6)]
    groups = B.get_proximal_flat_groups_nonoverlap((rows, cols), (3, 3))
    seq = [B.inexact_alm_lsd(D, groups=groups) for D in clips]
    par = B.inexact_alm_lsd_batch(clips, groups=groups, in_flight=3)
    for (L0, S0, it0, c0), (L1, S1, it1, c1) in zip(seq, par):
        assert it0 == it1 and c0 == c1 and c1
        assert rel_fro(L1, L0) <= 1e-6 and rel_fro(S1, S0) <= 1e-6      # (the kernels are deterministic: in practice identical)


def test_LSD_pipeline(B, watersurface_u8):
    """LSD() (inexact_alm_lsd.py:203-235, row a15): in-place normalisation, mean subtraction, solve, mask, reshapes."""
    from oracle import alm_oracle as O
    cube0 = np.asfortranarray(watersurface_u8[40:72, 60:100, 0:16].astype(np.float64))
    D, x_norm, mean = O.normalize_and_center(cube0)
    groups = O.flat_groups_nonoverlap((32, 40), (3, 3))
    Lr, Sr, itr, convr = O.inexact_alm_lsd(D, groups=groups)
    mref = O.foreground_mask(D, Lr, Sr)
    cube = cube0.copy(order='F')
    S, S_mask, L, ImData1, ImMean, shape, it, conv = B.LSD(cube, 0, 15, 1, use_flat=True)
    assert shape == (32, 40, 16) and S.shape == shape and S_mask.shape == shape and L.shape == shape
    assert ImData1 is cube and np.array_equal(cube, x_norm)            # normalised in place like the reference (SURVEY Q17)
    assert abs(ImMean - mean) <= 1e-15 and abs(it - itr) <= 1 and conv == convr
    assert rel_fro(L.reshape(D.shape, order='F'), Lr) <= TOL_F and rel_fro(S.reshape(D.shape, order='F'), Sr) <= TOL_F
    assert (S_mask.reshape(D.shape, order='F') == mref).mean() >= 0.999
    # default (overlapping graph) branch on a smaller crop
    cube2 = np.asfortranarray(watersurface_u8[50:74, 70:100, 0:10].astype(np.float64))
    D2, _x2, _m2 = O.normalize_and_center(cube2)
    Lg, Sg, itg, convg = O.inexact_alm_lsd(D2, graphs=O.graph_all_groups((24, 30), (3, 3)))
    out = B.LSD(cube2.copy(order='F'), 0, 9, 1)
    assert abs(out[6] - itg) <= 1 and out[7] == convg
    assert rel_fro(out[2].reshape(D2.shape, order='F'), Lg) <= TOL_F and rel_fro(out[0].reshape(D2.shape, order='F'), Sg) <= TOL_F


def test_device_side_u8_preprocessing(B):
    """bsub_load_u8_host: LSD()'s min-max normalisation and mean subtraction on the device (inexact_alm_lsd.py:211-225)."""
    from background_subtraction_b200 import synth
    from background_subtraction_b200 import _cabi as C
    rows, cols, n = 24, 30, 12
    video, _ = synth.make_clip(rows, cols, n, seed=3, n_rect=2)
    ref = synth.preprocess_u8(video)                                     # float32 [n][m], computed in fp64 on the host
    dec = B.Decomposition(B.make_config(rows * cols, n, C.PROX_FLAT_LINF, rows, cols))
    lo, hi, mean_raw = dec.load_u8(video)
    assert lo == float(video.min()) and hi == float(video.max())
    assert abs(mean_raw - float(video.mean(dtype=np.float64))) <= 1e-9 * max(1.0, abs(mean_raw))
    got = dec.device_tensor('D').cpu().numpy()
    assert np.abs(got - ref).max() <= 2e-7


def test_rpca_l1(B, watersurface_u8):
    from oracle import alm_oracle as O
    D, _x, _mean = O.normalize_and_center(watersurface_u8[:48, :60, :20])
    Lr, Sr, itr, convr = O.inexact_alm_rpca(D, delta=10)
    L, S, it, conv = B.inexact_alm_rpca(D, delta=10)
    _report("rpca", None, it, conv, L, S, Lr, Sr)
    assert abs(it - itr) <= 1 and conv == convr
    assert rel_fro(L, Lr) <= TOL_F and rel_fro(S, Sr) <= TOL_F


def test_errors(B):
    D = np.zeros((36, 4), order='F')
    with pytest.raises(Exception, match="one of graphs or groups must not be None"):
        B.inexact_alm_lsd(D)
    with pytest.raises(Exception, match="only one of graphs or groups"):
        B.inexact_alm_lsd(D, graphs=B.getGraphSPAMS_all_groups((6, 6), (3, 3)), groups=np.ones(36, dtype=np.int32))
    with pytest.raises(Exception):
        B.inexact_alm_lsd(D, groups=np.ones(35, dtype=np.int32))


def test_torch_cuda_input_returns_owning_tensors(B, watersurface_u8):
    """Drop-in call with a torch CUDA matrix: L and S come back as CUDA tensors that own their storage (they -- and views derived
    from them -- stay valid after the solver handle is gone, ADVICE r1) and equal the NumPy path."""
    import gc
    import torch
    from oracle import alm_oracle as O
    D, _x, _mean = O.normalize_and_center(watersurface_u8[:64, :60, :24])
    groups = B.get_proximal_flat_groups_nonoverlap((64, 60), (3, 3))
    Ln, Sn, itn, convn = B.inexact_alm_lsd(D, groups=groups)
    Dt = torch.from_numpy(np.ascontiguousarray(D.T, dtype=np.float32)).cuda().t()          # [m, n] view, F-order like the reference
    Lt, St, itt, convt = B.inexact_alm_lsd(Dt, groups=groups)
    assert Lt.is_cuda and St.is_cuda and tuple(Lt.shape) == D.shape and itt == itn and convt == convn
    view = Lt[:, :5]
    gc.collect()
    torch.cuda.synchronize()
    junk = [torch.full((1 << 22,), float("nan"), device="cuda") for _ in range(8)]          # recycle freed device memory, if any
    torch.cuda.synchronize()
    assert rel_fro(Lt.cpu().numpy().astype(np.float64), Ln) <= 1e-6 and rel_fro(St.cpu().numpy().astype(np.float64), Sn) <= 1e-6
    assert torch.isfinite(view).all()
    del junk
