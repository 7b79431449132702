"""-m gpu: the stage-2 saliency RPCA on slices the shared-memory kernel cannot hold (more than 640 frames, or too many rows for a
cluster of 8 CTAs), which run on the global-memory kernel of csrc/rpca_batch.cu, against the float64 oracle with an exact SVD
(oracle/flow_oracle.compute_RPCA) under the bars of test_gpu_flow.test_saliency_rpca_batch."""
import numpy as np
import pytest

from conftest import rel_fro

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    import background_subtraction_b200 as B
    return B


@pytest.fixture(scope="module")
def F():
    from oracle import flow_oracle as F
    return F


def _xt(seed, rows, cols, n):
    """n X-T slices of rows x cols (a rows-tall, n-wide synthetic clip of cols frames), float64 0..255, [n, rows, cols]."""
    from test_oracle_flow import saliency_slices
    return np.ascontiguousarray(saliency_slices(seed, rows, n, cols).transpose(2, 1, 0))


def _tol_l1(x):
    return x.shape[1] * x.shape[2] * 1e-4


def _check_against_oracle(F, x, L, S, info, sel, tol_l1, tag):
    Lr, Sr, its = F.compute_RPCA(x[sel], tol_l1)
    print("[%s] iters gpu" % tag, info["iters"][sel].tolist(), "oracle", its.tolist())
    assert np.all(np.abs(info["iters"][sel] - its) <= 1)
    for k, i in enumerate(sel):
        assert info["rank"][i] == 1
        assert rel_fro(L[i], Lr[k]) <= 1e-4
        if info["iters"][i] == its[k]:
            assert rel_fro(S[i], Sr[k]) <= 1e-4
        assert np.sum(np.abs(x[i] - L[i] - S[i])) <= 2 * tol_l1                # float32 L + S against the float64 input


@pytest.mark.parametrize("rows,cols,n,nsel", [(1080, 300, 4, 2), (2000, 96, 4, 2), (481, 301, 5, 3), (240, 862, 4, 2),
                                              (64, 1500, 6, 3), (3, 700, 6, 3)])
def test_large_slices_match_oracle(B, F, rows, cols, n, nsel):
    from background_subtraction_b200 import flow
    x = _xt(rows + cols, rows, cols, n)
    tol_l1 = _tol_l1(x)
    L, S, info = flow.inexact_alm_rpca_batch(x, delta=1.0, tol_l1=tol_l1, return_info=True)
    assert L.shape == x.shape and np.all(info["iters"] > 0)
    sel = np.linspace(0, n - 1, nsel).astype(int)
    _check_against_oracle(F, x, L, S, info, sel, tol_l1, "%dx%d" % (rows, cols))
    # determinism: the sampled slices again, reversed, as a smaller batch (fewer clusters, other positions)
    rev = sel[::-1].copy()
    L2, S2, info2 = flow.inexact_alm_rpca_batch(x[rev], delta=1.0, tol_l1=tol_l1, return_info=True)
    assert np.array_equal(L2, L[rev]) and np.array_equal(S2, S[rev])
    for key in ("iters", "err", "rank"):
        assert np.array_equal(info2[key], info[key][rev]), key


def test_degenerate_slices_in_a_large_batch(B, F):
    from background_subtraction_b200 import flow
    x = _xt(11, 64, 1500, 4)
    x[1] = 0.0
    x[2] = 37.0
    tol_l1 = _tol_l1(x)
    L, S, info = flow.inexact_alm_rpca_batch(x, delta=1.0, tol_l1=tol_l1, return_info=True)
    assert not L[1].any() and not S[1].any()
    assert (info["iters"][1], info["rank"][1], info["err"][1]) == (0, 0, 0.0)
    Lr, Sr, its = F.compute_RPCA(x[2:3], tol_l1)
    assert abs(info["iters"][2] - its[0]) <= 1 and info["rank"][2] == 1
    assert rel_fro(L[2], Lr[0]) <= 1e-4 and np.sum(np.abs(S[2])) <= tol_l1
    _check_against_oracle(F, x, L, S, info, np.array([0, 3]), tol_l1, "degenerate batch")


def test_iteration_cap(B, F):
    from background_subtraction_b200 import flow
    x = _xt(5, 481, 301, 3)
    tol_l1 = _tol_l1(x)
    L, S, info = flow.inexact_alm_rpca_batch(x, delta=1.0, tol_l1=tol_l1, max_iter=3, return_info=True)
    assert np.all(info["iters"] == -3)
    for i in range(x.shape[0]):
        Lr, Sr, it, conv = F.inexact_alm_rpca_capped(x[i], 1.0, 1, 1e-7, tol_l1, 3)
        assert (it, conv) == (3, False)
        assert rel_fro(L[i], Lr) <= 1e-4 and rel_fro(S[i], Sr) <= 1e-4


def test_saliency_chain_long_clip(B, F):
    """executeSaliencyRPCA -> computeSCube on a 700-frame clip (both stacks on the global-memory kernel) against the oracle chain."""
    from test_oracle_flow import saliency_slices
    video = saliency_slices(9, 24, 32, 700)                                 # [t, h, w]
    xl, xs, yl, ys = B.executeSaliencyRPCA(video, 1)
    rxl, rxs, ryl, rys = F.executeSaliencyRPCA(video, 1)
    assert xs.shape == (32, 24, 700) and ys.shape == (24, 32, 700)
    cube = B.computeSCube(xs, ys)
    ref = F.compute_scube_separable(rxs, rys)
    assert np.abs(cube - ref).max() <= 2e-3 * np.abs(ref).max()


def test_saliency_mixed_paths(B, F):
    """120 x 420 x 300: the X-T slices (120 x 300) fit the shared-memory kernel, the Y-T slices (420 x 300) do not."""
    from test_oracle_flow import saliency_slices
    video = saliency_slices(13, 120, 420, 300)
    xl, xs, yl, ys = B.executeSaliencyRPCA(video, 1)
    for lo, sp, stack, tag in ((xl, xs, video.transpose(2, 1, 0), "X-T"), (yl, ys, video.transpose(1, 2, 0), "Y-T")):
        x = np.ascontiguousarray(stack)
        tol_l1 = _tol_l1(x)
        Lc, Sc, info = B.compute_RPCA(x, True, tol_l1, return_info=True)
        assert np.array_equal(Lc, lo) and np.array_equal(Sc, sp)
        sel = np.linspace(0, x.shape[0] - 1, 2).astype(int)
        _check_against_oracle(F, x, Lc, Sc, info, sel, tol_l1, "120x420x300 " + tag)
    # compute_RPCA's info is inexact_alm_rpca_batch's, and the default return value is unchanged
    from background_subtraction_b200 import flow
    y = np.ascontiguousarray(video.transpose(1, 2, 0)[:6])
    tol_l1 = _tol_l1(y)
    L, S, info = flow.inexact_alm_rpca_batch(y, delta=1.0, tol_l1=tol_l1, return_info=True)
    Lc, Sc, infoc = B.compute_RPCA(y, True, tol_l1, return_info=True)
    assert np.array_equal(infoc["iters"], info["iters"]) and np.array_equal(Lc, L) and np.array_equal(Sc, S)
    plain = B.compute_RPCA(y, True, tol_l1)
    assert len(plain) == 2 and np.array_equal(plain[0], L)
