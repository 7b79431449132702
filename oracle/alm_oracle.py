"""oracle/alm_oracle.py -- TEST INFRASTRUCTURE ONLY (CPU oracle, NumPy float64).

CPU restatement of the reference's hot path (SURVEY.md section 8a), each
function citing the reference file:line it follows.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module; the product package never does.

Pinning (see tests/test_oracle.py and tests/golden/make_golden.py):
  * inexact_alm_group_sparse_RPCA, block_shrinkage_operator, foreground_mask,
    svd_k_largest and the two group builders are checked against the reference's
    own functions, imported in place from /root/reference by
    oracle/ref_harness.py (this container only), and against committed golden
    vectors generated the same way.
  * inexact_alm_lsd is checked against the reference's own loop executed
    unmodified around a `spams` stand-in (SPAMS is an un-vendored, unpinned
    third-party C++ dependency that is not installed: PARITY UNPINNED at the
    spams.proximalFlat / spams.proximalGraph boundary; the stand-in follows the
    published SPAMS definitions and is validated against an independent QP solve).
"""
import ctypes
import os

import numpy as np
from numpy import linalg as LA

from . import build_oracle

_lib = None


def _clib():
    global _lib
    if _lib is None:
        path = build_oracle.build()
        lib = ctypes.CDLL(path)
        dp = ctypes.POINTER(ctypes.c_double)
        ip = ctypes.POINTER(ctypes.c_int)
        lib.prox_flat_linf.argtypes = [dp, ctypes.c_long, ctypes.c_long, ip, ctypes.c_double, dp, ctypes.c_int]
        lib.prox_flat_linf.restype = ctypes.c_int
        lib.prox_graph_linf.argtypes = [dp, ctypes.c_long, ctypes.c_long, ip, ip, ctypes.c_long, dp,
                                        ctypes.c_double, ctypes.c_double, ctypes.c_int, dp, ip, ctypes.c_int]
        lib.prox_graph_linf.restype = ctypes.c_int
        lib.block_shrink_l2.argtypes = [dp, ctypes.c_long, ctypes.c_long, ip, ip, dp, ctypes.c_double,
                                        ctypes.c_double, dp]
        lib.block_shrink_l2.restype = ctypes.c_int
        lib.l1ball_project_export.argtypes = [dp, ctypes.c_int, ctypes.c_double, dp]
        lib.l1ball_project_export.restype = None
        _lib = lib
    return _lib


def _dptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def _iptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int))


def usable_cores():
    """numThreads the reference hands to SPAMS: cpu_count()-1 (/root/reference/utils.py:15-20)."""
    return max(1, (os.cpu_count() or 2) - 1)


# --------------------------------------------------------------------------
# group / graph builders (hot-path *types*)
# --------------------------------------------------------------------------
def flat_groups_nonoverlap(img_shape, batch_shape):
    """int32[m] 1-based tile ids in F-order; restates get_proximal_flat_groups_nonoverlap,
    /root/reference/lsd_improvement.py:14-34 (ragged right/bottom tiles are smaller)."""
    if len(img_shape) != 2 or len(batch_shape) != 2:
        raise Exception("Input lengths are incorrect")
    m, n = img_shape
    a, b = min(batch_shape[0], m), min(batch_shape[1], n)
    ti = np.arange(m) // a                       # tile row of each image row
    tj = np.arange(n) // b                       # tile col of each image col
    ntr = -(-m // a)
    ids = (tj[None, :] * ntr + ti[:, None] + 1).astype(np.int32)
    return np.asfortranarray(ids).flatten(order='F')


def window_pixels_top_left(i, j, group_shape, img_shape):
    """Pixel list of the window with top-left (i, j); restates get_vars_idx_top_left,
    /root/reference/utils.py:249-257 -- note min(shape, rows-1-i): the last image row
    and column are never covered and edge windows are truncated (SURVEY Q8)."""
    rows, cols = img_shape
    bottom = min(group_shape[0], rows - 1 - i)
    right = min(group_shape[1], cols - 1 - j)
    tl = j * rows + i
    return [tl + di + rows * dj for dj in range(right) for di in range(bottom)]


def graph_all_groups(img_shape, group_shape):
    """CSC (indptr, indices, eta) of the overlapping-window graph; restates
    getGraphSPAMS_all_groups, /root/reference/inexact_alm_lsd.py:13-46
    (groups enumerated j outer, i inner; eta_g = 1; no group nesting)."""
    if len(img_shape) != 2:
        raise Exception("Input lengths are incorrect")
    m, n = img_shape
    a, b = min(group_shape[0], m), min(group_shape[1], n)
    num_x, num_y = m - a + 1, n - b + 1
    indptr = [0]
    indices = []
    for j in range(num_y):
        for i in range(num_x):
            v = window_pixels_top_left(i, j, (a, b), img_shape)
            indices.extend(v)
            indptr.append(len(indices))
    return (np.asarray(indptr, dtype=np.int32), np.asarray(indices, dtype=np.int32),
            np.ones(num_x * num_y, dtype=np.float64))


def window_pixels_center(i, j, group_radius, img_shape):
    """Pixel list of the window centred on (i, j), clipped to the image; restates get_vars_idx_center,
    /root/reference/utils.py:234-246 (unlike the top-left variant the clipping here is exact)."""
    rows, cols = img_shape
    left, right = min(group_radius, j), min(group_radius, cols - 1 - j)
    top, bottom = min(group_radius, i), min(group_radius, rows - 1 - i)
    tl = (j - left) * rows + (i - top)
    return [tl + di + rows * dj for dj in range(left + right + 1) for di in range(top + bottom + 1)]


def graph_group_centers(img_shape, group_radius, group_centers):
    """CSC (indptr, indices, eta) of the per-frame graph of windows centred on the pixels with a positive weight;
    restates get_proximal_graph_group_centers, /root/reference/lsd_improvement.py:74-120 (centres enumerated
    column by column, eta_g = weight of the centre pixel, no nesting)."""
    rows, cols = img_shape
    gc = np.asarray(group_centers)
    cj, ci = np.where(gc.T > 0)
    indptr, indices, eta = [0], [], []
    for i, j in zip(ci, cj):
        indices.extend(window_pixels_center(int(i), int(j), group_radius, (rows, cols)))
        indptr.append(len(indices))
        eta.append(float(gc[i, j]))
    return (np.asarray(indptr, dtype=np.int32), np.asarray(indices, dtype=np.int32), np.asarray(eta, dtype=np.float64))


def graph_from_spams_dict(graph):
    """(indptr, indices, eta) from the SPAMS graph dict the reference passes around
    ({'eta_g','groups','groups_var'}, /root/reference/inexact_alm_lsd.py:45)."""
    gv = graph['groups_var'].tocsc()
    return (np.ascontiguousarray(gv.indptr, dtype=np.int32),
            np.ascontiguousarray(gv.indices, dtype=np.int32),
            np.ascontiguousarray(graph['eta_g'], dtype=np.float64))


# --------------------------------------------------------------------------
# proximal operators
# --------------------------------------------------------------------------
def l1ball_project(x, z):
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    _clib().l1ball_project_export(_dptr(x), x.size, float(z), _dptr(out))
    return out


def prox_flat(G_S, lambda1, groups, num_threads=None):
    """Stand-in for spams.proximalFlat(regul='group-lasso-linf'); call site
    /root/reference/inexact_alm_lsd.py:71-79."""
    U = np.asfortranarray(G_S, dtype=np.float64)
    m, n = U.shape
    g = np.ascontiguousarray(groups, dtype=np.int32).ravel()
    assert g.size == m
    V = np.empty_like(U, order='F')
    rc = _clib().prox_flat_linf(_dptr(U), m, n, _iptr(g), float(lambda1), _dptr(V),
                                int(num_threads or usable_cores()))
    if rc != 0:
        raise Exception("prox_flat: bad groups vector")
    return V


def prox_graph(G_S, lambda1, graph_csc, num_threads=None, tol=1e-13, max_sweeps=20000, return_sweeps=False):
    """Stand-in for spams.proximalGraph(regul='graph'); call site
    /root/reference/inexact_alm_lsd.py:49-57.  graph_csc = (indptr, indices, eta)."""
    U = np.asfortranarray(G_S, dtype=np.float64)
    if U.ndim == 1:
        U = U.reshape(-1, 1, order='F')
    m, n = U.shape
    indptr, indices, eta = graph_csc
    V = np.empty_like(U, order='F')
    sweeps = np.zeros(n, dtype=np.int32)
    _clib().prox_graph_linf(_dptr(U), m, n, _iptr(indptr), _iptr(indices), len(eta), _dptr(eta),
                            float(lambda1), float(tol), int(max_sweeps), _dptr(V), _iptr(sweeps),
                            int(num_threads or usable_cores()))
    return (V, sweeps) if return_sweeps else V


def prox_by_frame(G_S, lambda1, graphs_csc, **kw):
    """One graph per column; restates /root/reference/inexact_alm_lsd.py:60-68 (serial branch)."""
    out = np.zeros_like(G_S, order='F')
    for f in range(G_S.shape[1]):
        out[:, [f]] = prox_graph(G_S[:, [f]], lambda1, graphs_csc[f], **kw)
    return out


def blocks_to_labels(blocks_by_frame, m):
    """list[n] of lists of bool[m] masks -> (labels int32[n,m], lam_ptr); later blocks overwrite
    earlier ones exactly as the sequential assignment at /root/reference/group_sparse_RPCA.py:32-35 does."""
    n = len(blocks_by_frame)
    labels = np.zeros((n, m), dtype=np.int32)
    ptr = np.zeros(n + 1, dtype=np.int32)
    for f, blocks in enumerate(blocks_by_frame):
        for b, mask in enumerate(blocks):
            labels[f, np.asarray(mask, dtype=bool)] = b + 1
        ptr[f + 1] = ptr[f] + len(blocks)
    return labels, ptr


def block_shrinkage_operator(G, blocks_by_frame, lambdas_by_frame, mu, non_block_lambda):
    """Restates /root/reference/group_sparse_RPCA.py:13-42 (C loop over a label map)."""
    G = np.asfortranarray(G, dtype=np.float64)
    m, n = G.shape
    labels, ptr = blocks_to_labels(blocks_by_frame, m)
    lam = np.asarray([x for l in lambdas_by_frame for x in l] + [0.0], dtype=np.float64)
    R = np.empty_like(G, order='F')
    rc = _clib().block_shrink_l2(_dptr(G), m, n, _iptr(labels), _iptr(ptr), _dptr(lam), float(mu),
                                 float(non_block_lambda), _dptr(R))
    if rc != 0:
        raise Exception("block_shrinkage_operator: bad label map")
    return R


def block_shrinkage_operator_np(G, blocks_by_frame, lambdas_by_frame, mu, non_block_lambda):
    """Pure-NumPy line-by-line restatement of /root/reference/group_sparse_RPCA.py:13-42
    (small cases; cross-checks the C loop above)."""
    result = np.zeros_like(G)
    with np.errstate(divide='ignore', invalid='ignore'):
        for f in range(len(blocks_by_frame)):
            non_block = np.full(G.shape[0], True)
            for b, block in enumerate(blocks_by_frame[f]):
                eps = lambdas_by_frame[f][b] / mu
                non_block[block] = False
                g = G[block, f]
                result[block, f] = np.maximum(1 - eps / LA.norm(g, ord=2), 0) * g
            g = G[non_block, f]
            result[non_block, f] = np.maximum(1 - (non_block_lambda / mu) / LA.norm(g, ord=2), 0) * g
    return result


# --------------------------------------------------------------------------
# SVT helpers
# --------------------------------------------------------------------------
def svd_k_largest(G, k):
    """Top-k singular triplets, descending; /root/reference/utils.py:204-212.  The reference's
    ARPACK-vs-LAPACK switch (:189-201) is numerically irrelevant (SURVEY Q6): always full SVD."""
    u, s, vh = LA.svd(G, full_matrices=False)
    return u[:, :k], s[:k], vh[:k, :]


def rank_logic(s, sv, mu, d, use_sv_prediction=True):
    """svp and the next sv; /root/reference/inexact_alm_lsd.py:136-145 with
    get_last_nonzero_idx (/root/reference/utils.py:215-217).  round() is Python's (banker's)."""
    nz = np.nonzero(s - 1 / mu > 0)[0]
    svp = int(nz.max()) + 1 if nz.size else 0
    if use_sv_prediction:
        sv = svp + 1 if svp < sv else min(svp + round(0.05 * d), d)
    return svp, int(sv)


def foreground_mask(D, L, S, sigmas_from_mean=2):
    """Restates /root/reference/utils.py:139-149."""
    S_abs = np.abs(S)
    m = np.max(S_abs)
    S_back = S_abs < 0.5 * m
    S_diff = np.abs(D - L) * S_back
    pos = S_diff[S_diff > 0]
    th = np.mean(pos) + sigmas_from_mean * np.std(pos)
    return S_abs > th


# --------------------------------------------------------------------------
# the ALM loops
# --------------------------------------------------------------------------
def _alm(D0, prox_fn, mu_scale, delta, rho=1.6, tol_out=1e-7, max_iter=500, sv0=10,
         break_on_rank0=False, use_sv_prediction=True, L0=False, log=None, return_Y=False):
    """(L, S, iterations, converged), and the final multiplier Y after them when return_Y is set."""
    D = np.asfortranarray(D0, dtype=np.float64)
    m, n = D.shape
    d = min(m, n)
    lambda_param = (np.sqrt(max(m, n)) * delta) ** (-1)
    norm_two = LA.norm(D, ord=2)
    norm_inf = LA.norm(D, ord=np.inf) / lambda_param     # induced inf-norm = max ROW SUM (SURVEY Q1)
    dual_norm = max(norm_two, norm_inf)
    Y = D / dual_norm
    mu = mu_scale / norm_two
    norm_D = LA.norm(D, ord='fro')
    S = np.zeros(D.shape, order='F')
    L = np.zeros(D.shape, order='F') if L0 else None
    converged = False
    it = 0
    sv = sv0 if use_sv_prediction else d
    while not converged:
        it += 1
        G_L = D - S + Y / mu
        u, s, vh = svd_k_largest(G_L, sv)
        svp, sv_next = rank_logic(s, sv, mu, d, use_sv_prediction)
        if break_on_rank0 and svp == 0:
            if log is not None:
                log.append(dict(iter=it, svp=0, sv=sv, err=None, mu=mu, sigma=s.copy()))
            break
        sv_used = sv
        sv = sv_next
        L = np.asfortranarray((u[:, :svp] * (s[:svp] - 1 / mu)) @ vh[:svp, :])
        G_S = D - L + Y / mu
        S = prox_fn(G_S, lambda_param, mu)
        Z = D - L - S
        Y = Y + mu * Z
        mu_used = mu
        mu = min(mu * rho, mu * 1e7)
        err = LA.norm(Z, ord='fro') / norm_D
        if log is not None:
            log.append(dict(iter=it, svp=svp, sv=sv_used, err=float(err), mu=mu_used,
                            nnz=int(np.count_nonzero(S)), sigma=s.copy()))
        if err < tol_out:
            converged = True
        elif it >= max_iter:
            break
    return (L, S, it, converged, Y) if return_Y else (L, S, it, converged)


def inexact_alm_lsd(D0, graphs=None, groups=None, delta=10, log=None, prox_tol=1e-13, prox_max_sweeps=20000,
                    max_iter=500):
    """Restates /root/reference/inexact_alm_lsd.py:82-179.  graphs: (indptr, indices, eta) CSC triple or a
    SPAMS graph dict, or a list of those (one per frame); groups: int32[m]."""
    if graphs is None and groups is None:
        raise Exception("one of graphs or groups must not be None")
    if graphs is not None and groups is not None:
        raise Exception("only one of graphs or groups must not be None")

    def as_csc(g):
        return graph_from_spams_dict(g) if isinstance(g, dict) else g

    if groups is not None:
        def prox_fn(G_S, lam, mu):
            return prox_flat(G_S, lam / mu, groups)
    elif isinstance(graphs, list) or (isinstance(graphs, np.ndarray) and graphs.dtype == object):
        gl = [as_csc(g) for g in graphs]

        def prox_fn(G_S, lam, mu):
            return prox_by_frame(G_S, lam / mu, gl, tol=prox_tol, max_sweeps=prox_max_sweeps)
    else:
        gc = as_csc(graphs)

        def prox_fn(G_S, lam, mu):
            return prox_graph(G_S, lam / mu, gc, tol=prox_tol, max_sweeps=prox_max_sweeps)
    return _alm(D0, prox_fn, 12.5, delta, log=log, max_iter=max_iter)


def inexact_alm_group_sparse_RPCA(D0, blocks_by_frame, lambdas_by_frame, delta=10, use_sv_prediction=True,
                                  log=None, max_iter=500):
    """Restates /root/reference/group_sparse_RPCA.py:45-126 (mu0 = 1.25/||D||_2, L0 = S0 = 0, break on
    rank 0 BEFORE L/S are updated, non-block lambda = 100*lambda)."""
    m, n = np.shape(D0)
    lambda_param = (np.sqrt(max(m, n)) * delta) ** (-1)
    nbl = 1e2 * lambda_param

    def prox_fn(G_S, lam, mu):
        return block_shrinkage_operator(G_S, blocks_by_frame, lambdas_by_frame, mu, nbl)
    return _alm(D0, prox_fn, 1.25, delta, break_on_rank0=True, use_sv_prediction=use_sv_prediction, L0=True,
                log=log, max_iter=max_iter)


def inexact_alm_rpca(D0, delta=1.0, use_sv_prediction=False, log=None, max_iter=500):
    """Plain l1 RPCA sibling, /root/reference/lsd_improvement.py:123-196 (rho = 1.2, mu0 = 1.25/||D||_2,
    elementwise soft threshold) -- SURVEY 8f row 2; kept for the 'next' rows."""
    def prox_fn(G_S, lam, mu):
        return np.sign(G_S) * np.maximum(np.abs(G_S) - lam / mu, 0)
    return _alm(D0, prox_fn, 1.25, delta, rho=1.2, use_sv_prediction=use_sv_prediction,
                sv0=10, log=log, max_iter=max_iter)


def apply_background_shrinkage_operator(G, output, epsilon, background_masks):
    """One l2 group per frame over the frame's background pixels, written over `output`; restates
    /root/reference/lsd_improvement.py:199-212 (zero norm -> factor max(-inf, 0) = 0)."""
    for f in range(len(background_masks)):
        mask = np.asarray(background_masks[f], dtype=bool)
        g = G[mask, f]
        nrm = LA.norm(g, ord=2)
        fac = max(1 - epsilon / nrm, 0) if nrm > 0 else 0.0
        output[mask, f] = fac * g
    return output


def inexact_alm_lsd_with_background(D0, graphs, background_masks, delta=10, log=None, prox_tol=1e-13,
                                    prox_max_sweeps=20000, max_iter=500):
    """Restates /root/reference/lsd_improvement.py:215-304: the LSD loop with one graph per frame
    (prox_by_frame) followed by an l2 shrink of every frame's background pixels at 100 lambda / mu."""
    if not isinstance(graphs, list) and not isinstance(graphs, np.ndarray):
        raise Exception('graphs must be list/array')
    m, n = np.shape(D0)
    lambda_param = (np.sqrt(max(m, n)) * delta) ** (-1)
    background_lambda = 1e2 * lambda_param
    gl = [graph_from_spams_dict(g) if isinstance(g, dict) else g for g in graphs]

    def prox_fn(G_S, lam, mu):
        S = prox_by_frame(G_S, lam / mu, gl, tol=prox_tol, max_sweeps=prox_max_sweeps)
        return apply_background_shrinkage_operator(G_S, S, background_lambda / mu, background_masks)
    return _alm(D0, prox_fn, 12.5, delta, log=log, max_iter=max_iter)


def normalize_and_center(cube):
    """LSD() pre-processing, /root/reference/inexact_alm_lsd.py:211-225 with normalizeImage
    (/root/reference/utils.py:220-223): global min-max to [0,1], subtract global mean, F-reshape."""
    x = np.array(cube, dtype=np.float64, order='F')
    x -= np.min(x)
    x *= 1.0 / np.max(x)
    mean = np.mean(x)
    x2 = x - mean
    h, w, t = x2.shape
    return x2.reshape((h * w, t), order='F'), x, mean
