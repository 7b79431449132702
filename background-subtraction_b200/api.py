"""Host-side mirror of the reference's call surface for the hot path (SURVEY.md section 8b).

Same names, argument meaning, return tuples and error convention (`raise Exception(msg)`) as
  inexact_alm_lsd                    /root/reference/inexact_alm_lsd.py:82-179
  inexact_alm_group_sparse_RPCA      /root/reference/group_sparse_RPCA.py:45-126
  inexact_alm_rpca                   /root/reference/lsd_improvement.py:123-196
  foreground_mask                    /root/reference/utils.py:139-149
  LSD                                /root/reference/inexact_alm_lsd.py:203-235
  prox / prox_flat / prox_by_frame   /root/reference/inexact_alm_lsd.py:49-79
  block_shrinkage_operator           /root/reference/group_sparse_RPCA.py:13-42
  svd_k_largest                      /root/reference/utils.py:204-212
  getGraphSPAMS_all_groups           /root/reference/inexact_alm_lsd.py:13-46
  inexact_alm_lsd_with_background    /root/reference/lsd_improvement.py:215-304
  get_proximal_graph_group_centers   /root/reference/lsd_improvement.py:74-120
  apply_background_shrinkage_operator /root/reference/lsd_improvement.py:199-212
  get_proximal_flat_groups_nonoverlap /root/reference/lsd_improvement.py:14-34
Everything numerical happens in libbsub_b200.so (CUDA, sm_100a) behind the C ABI of include/bsub_b200.h;
this module only marshals arrays.  torch is used for device buffers and streams of the stand-alone operators.
"""
import ctypes

import numpy as np

from . import _cabi as C

BLOCK_SIZE = (3, 3)          # /root/reference/inexact_alm_lsd.py:11


# --------------------------------------------------------------------------------------------------------------
# group / graph builders (host, vectorised; same outputs as the reference builders)
# --------------------------------------------------------------------------------------------------------------
def get_proximal_flat_groups_nonoverlap(img_shape, batch_shape):
    if len(img_shape) != 2 or len(batch_shape) != 2:
        raise Exception("Input lengths are incorrect")
    m, n = int(img_shape[0]), int(img_shape[1])
    a, b = min(int(batch_shape[0]), m), min(int(batch_shape[1]), n)
    ntr = -(-m // a)
    ids = (np.arange(n)[None, :] // b) * ntr + (np.arange(m)[:, None] // a) + 1
    return np.asfortranarray(ids.astype(np.int32)).flatten(order='F')


def window_csc(img_shape, group_shape=BLOCK_SIZE):
    """(indptr, indices) of groups_var for all top-left windows, including the reference's edge quirk
    (utils.py:249-257: extent min(g, rows-1-i), so the last row/column is uncovered)."""
    rows, cols = int(img_shape[0]), int(img_shape[1])
    a, b = min(group_shape[0], rows), min(group_shape[1], cols)
    num_x, num_y = rows - a + 1, cols - b + 1
    ii, jj = np.meshgrid(np.arange(num_x), np.arange(num_y), indexing='ij')
    ii, jj = ii.ravel(order='F'), jj.ravel(order='F')          # j outer, i inner
    hh = np.minimum(a, rows - 1 - ii)
    ww = np.minimum(b, cols - 1 - jj)
    sizes = np.maximum(hh, 0) * np.maximum(ww, 0)
    indptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    idx = []
    for dj in range(b):
        for di in range(a):
            ok = (di < hh) & (dj < ww)
            idx.append((np.where(ok)[0], (jj[ok] + dj) * rows + ii[ok] + di, (dj * hh[ok] + di)))
    indices = np.empty(int(indptr[-1]), dtype=np.int32)
    for g, pix, slot in idx:
        indices[indptr[g] + slot] = pix
    return indptr, indices


def getGraphSPAMS_all_groups(img_shape, group_shape):
    if len(img_shape) != 2:
        raise Exception("Input lengths are incorrect")
    import scipy.sparse as ssp
    rows, cols = int(img_shape[0]), int(img_shape[1])
    indptr, indices = window_csc(img_shape, group_shape)
    ng = len(indptr) - 1
    groups_var = ssp.csc_matrix((np.full(len(indices), True), indices, indptr), shape=(rows * cols, ng), dtype=bool)
    return {'eta_g': np.ones(ng, dtype=np.float64), 'groups': ssp.csc_matrix((ng, ng), dtype=bool),
            'groups_var': groups_var}


def center_window_csc(img_shape, group_centers, group_radius=1):
    """(indptr, indices, eta) of the windows centred on the pixels with a positive weight, clipped to the image
    (get_vars_idx_center, utils.py:234-246), enumerated column by column like lsd_improvement.py:97-111."""
    rows, cols = int(img_shape[0]), int(img_shape[1])
    gc = np.asarray(group_centers)
    cj, ci = np.where(gc.T > 0)
    i0, i1 = np.maximum(ci - group_radius, 0), np.minimum(ci + group_radius, rows - 1)
    j0, j1 = np.maximum(cj - group_radius, 0), np.minimum(cj + group_radius, cols - 1)
    hh, ww = i1 - i0 + 1, j1 - j0 + 1
    indptr = np.concatenate([[0], np.cumsum(hh * ww)]).astype(np.int32)
    indices = np.empty(int(indptr[-1]), dtype=np.int32)
    w = 2 * group_radius + 1
    for dj in range(w):
        for di in range(w):
            ok = (di < hh) & (dj < ww)
            indices[indptr[:-1][ok] + dj * hh[ok] + di] = (j0[ok] + dj) * rows + i0[ok] + di
    return indptr, indices, np.ascontiguousarray(gc[ci, cj], dtype=np.float64)


def get_proximal_graph_group_centers(img_shape, group_size, group_centers):
    """Same SPAMS graph dict as /root/reference/lsd_improvement.py:74-120 (group_size is the window RADIUS there); the
    weight map is kept under a private key so that inexact_alm_lsd_with_background need not recover it."""
    import scipy.sparse as ssp
    rows, cols = int(img_shape[0]), int(img_shape[1])
    indptr, indices, eta = center_window_csc((rows, cols), group_centers, int(group_size))
    ng = len(eta)
    groups_var = ssp.csc_matrix((np.full(len(indices), True), indices, indptr), shape=(rows * cols, ng), dtype=bool)
    return {'eta_g': eta, 'groups': ssp.csc_matrix((ng, ng), dtype=bool), 'groups_var': groups_var,
            '_group_centers': np.array(group_centers, dtype=np.float64), '_group_radius': int(group_size)}


def detect_center_windows(graph, m, img_shape=None):
    """eta map float32[m] (F-order pixel index, 0 = no window) if the SPAMS graph dict is a radius-1 centre-window graph
    of get_proximal_graph_group_centers, else None.  The candidate map is verified by rebuilding the CSC arrays."""
    gc = graph.get('_group_centers', None) if isinstance(graph, dict) else None
    if gc is not None and graph.get('_group_radius', 1) == 1 and gc.size == m:
        return (int(gc.shape[0]), int(gc.shape[1])), np.where(gc > 0, gc, 0).astype(np.float32).flatten(order='F')
    gv = graph['groups_var'].tocsc()
    if gv.shape[0] != m:
        raise Exception("graph has %d variables, matrix has %d rows" % (gv.shape[0], m))
    nested = graph.get('groups', None)
    if nested is not None and getattr(nested, 'nnz', 0) != 0:
        return None
    ptr, idx = np.asarray(gv.indptr), np.asarray(gv.indices)
    eta = np.asarray(graph['eta_g'], dtype=np.float64)
    ng = len(ptr) - 1
    shapes = [tuple(int(v) for v in img_shape)] if img_shape is not None else []
    if not shapes:                                   # rows = jump between the first two columns of any multi-column window
        for g in range(min(ng, 64)):
            w = idx[ptr[g]:ptr[g + 1]]
            jump = np.nonzero(np.diff(w) != 1)[0]
            if jump.size:
                rows = int(w[jump[0] + 1] - w[0])
                if rows > 0 and m % rows == 0:
                    shapes.append((rows, m // rows))
                    break
    for rows, cols in shapes:
        if rows * cols != m:
            continue
        if ng == 0:
            return (rows, cols), np.zeros(m, dtype=np.float32)
        if np.any(np.diff(ptr) == 0):                  # a centre window is never empty (e.g. the 1 x k windows of the last row)
            return None
        first, size = idx[ptr[:-1]], np.diff(ptr)
        i0, j0 = first % rows, first // rows
        # height of the window = length of the first run of consecutive indices
        hh = np.array([(np.nonzero(np.diff(idx[ptr[g]:ptr[g + 1]]) != 1)[0][:1].tolist() or [size[g] - 1])[0] + 1
                       for g in range(ng)])
        hh = np.minimum(hh, rows)                     # a window as tall as the image runs on into its next column
        ww = size // np.maximum(hh, 1)
        ci = np.where(hh == 3, i0 + 1, np.where(i0 == 0, 0, rows - 1)) if rows > 2 else None
        cj = np.where(ww == 3, j0 + 1, np.where(j0 == 0, 0, cols - 1)) if cols > 2 else None
        if ci is None or cj is None or np.any(ci >= rows) or np.any(cj >= cols):   # the latter: not a centre-window graph
            continue
        emap = np.zeros((rows, cols), dtype=np.float64)
        emap[ci, cj] = eta
        p2, i2, e2 = center_window_csc((rows, cols), emap, 1)
        if np.array_equal(p2, ptr) and np.array_equal(i2, idx) and np.array_equal(e2, eta):
            return (rows, cols), emap.astype(np.float32).flatten(order='F')
    return None


def detect_flat_tiling(groups, img_shape=None):
    """Return (rows, cols) if `groups` is the 3x3 tiling produced by get_proximal_flat_groups_nonoverlap for some
    image shape, else None."""
    g = np.ascontiguousarray(groups, dtype=np.int32).ravel()
    m = g.size
    cands = []
    if img_shape is not None:
        cands.append((int(img_shape[0]), int(img_shape[1])))
    dec = np.nonzero(g[1:] < g[:-1])[0]
    if dec.size:
        cands.append((int(dec[0]) + 1, m // (int(dec[0]) + 1)))
    else:                                   # ids never decrease: at most 3 columns, or at most 3 rows
        for c in (1, 2, 3):
            if m % c == 0:
                cands.append((m // c, c))
                cands.append((c, m // c))
    for rows, cols in cands:
        if rows * cols == m and np.array_equal(get_proximal_flat_groups_nonoverlap((rows, cols), BLOCK_SIZE), g):
            return rows, cols
    return None


def detect_window_graph(graph, m, img_shape=None):
    """Return (rows, cols, eta) if the SPAMS graph dict is the all-windows 3x3 graph of getGraphSPAMS_all_groups."""
    gv = graph['groups_var'].tocsc()
    if gv.shape[0] != m:
        raise Exception("graph has %d variables, matrix has %d rows" % (gv.shape[0], m))
    cands = []
    if img_shape is not None:
        cands.append((int(img_shape[0]), int(img_shape[1])))
    ind = gv.indices[gv.indptr[0]:gv.indptr[1]] if gv.shape[1] else np.array([], dtype=np.int32)
    steps = np.nonzero(np.diff(ind) != 1)[0]
    if steps.size:
        hh = int(steps[0]) + 1
        rows = int(ind[hh] - ind[0])
        if rows > 0 and m % rows == 0:
            cands.append((rows, m // rows))
    for rows, cols in cands:
        if rows * cols != m:
            continue
        indptr, indices = window_csc((rows, cols), BLOCK_SIZE)
        if len(indptr) - 1 == gv.shape[1] and np.array_equal(indptr, gv.indptr) and np.array_equal(indices, gv.indices):
            nested = graph.get('groups', None)
            if nested is not None and getattr(nested, 'nnz', 0) != 0:
                return None
            return rows, cols, np.ascontiguousarray(graph['eta_g'], dtype=np.float64)
    return None


def _is_graph_list(graphs):
    return isinstance(graphs, (list, tuple)) or (isinstance(graphs, np.ndarray) and graphs.dtype == object)


def pack_graphs(graphs, m, n):
    """SPAMS graph dict, or a list of them with one per frame -> (csc, frame_graph): csc = list of distinct
    (indptr int32, indices int32, eta float64) triples, frame_graph int32[n] = which of them each frame uses.  A graph shared
    by several frames (the same object, or equal CSC arrays) is stored once.  Raises on nested groups (SPAMS DAG semantics
    are not restated), a variable count other than m, pixel indices out of range or twice in a group, and eta that is
    negative, non-finite or of the wrong length."""
    import hashlib
    glist = list(graphs) if _is_graph_list(graphs) else [graphs] * n
    if len(glist) != n:
        raise Exception("graphs must hold one graph per frame (%d graphs, %d frames)" % (len(glist), n))
    csc, frame_graph, by_id, by_hash = [], np.empty(n, dtype=np.int32), {}, {}
    for f, g in enumerate(glist):
        if id(g) in by_id:
            frame_graph[f] = by_id[id(g)]
            continue
        nested = g.get('groups', None)
        if nested is not None and getattr(nested, 'nnz', 0) != 0:
            raise Exception("frame %d: the graph has nested groups (graph['groups'] is not empty); only flat group "
                            "structures are implemented" % f)
        gv = g['groups_var'].tocsc()
        if gv.shape[0] != m:
            raise Exception("graph has %d variables, matrix has %d rows" % (gv.shape[0], m))
        ip = np.ascontiguousarray(gv.indptr, dtype=np.int32)
        ix = np.ascontiguousarray(gv.indices, dtype=np.int32)
        eta = np.ascontiguousarray(np.asarray(g['eta_g'], dtype=np.float64).ravel())
        ng = len(ip) - 1
        if eta.size != ng:
            raise Exception("frame %d: eta_g has %d entries, the graph has %d groups" % (f, eta.size, ng))
        if not np.all(np.isfinite(eta) & (eta >= 0)):
            raise Exception("frame %d: eta_g must be finite and >= 0" % f)
        if ix.size and (ix.min() < 0 or ix.max() >= m):
            raise Exception("frame %d: group pixel index out of range [0, %d)" % (f, m))
        owner = np.repeat(np.arange(ng, dtype=np.int64), np.diff(ip))
        if np.unique(owner * m + ix).size != ix.size:
            raise Exception("frame %d: a group holds the same pixel twice" % f)
        key = hashlib.sha1(ip.tobytes() + b'|' + ix.tobytes() + b'|' + eta.tobytes()).digest()
        k = by_hash.get(key)
        if k is None or not all(np.array_equal(a, b) for a, b in zip(csc[k], (ip, ix, eta))):
            k = len(csc)
            csc.append((ip, ix, eta))
            by_hash[key] = k
        by_id[id(g)] = k
        frame_graph[f] = k
    return csc, frame_graph


def _graph_pointers(csc):
    """ctypes arrays of bsub_set_graphs / bsub_prox_graph_dev for the triples of pack_graphs (which must stay alive)."""
    k = len(csc)
    ng = np.array([len(c[0]) - 1 for c in csc], dtype=np.int64)
    ip = (C.c_int32_p * k)(*[c[0].ctypes.data_as(C.c_int32_p) for c in csc])
    ix = (C.c_int32_p * k)(*[c[1].ctypes.data_as(C.c_int32_p) for c in csc])
    et = (C.c_double_p * k)(*[c[2].ctypes.data_as(C.c_double_p) for c in csc])
    return ng, ip, ix, et


class GraphRoute:
    """Which prox kernel runs a graph description -- the one decision shared by the solvers below and the sharded driver
    (dist.CudaStepSolver).  prox = C.PROX_GRAPH_LINF: the 3x3 all-window graph on the tile kernel, eta = float64 window weights
    or None (unit weights); C.PROX_GRAPH_CENTER_BG: radius-1 centre windows on the tile kernel, eta = float32 [n][m] map;
    C.PROX_GRAPH_GENERIC: any other graph on the generic kernel, csc / frame_graph as pack_graphs returns them.  background =
    uint8 [n][m] (non-zero: the frame's background pixels, l2-shrunk after the prox) or None; rows, cols = image geometry
    (0, 0 when the generic graphs came without one)."""

    def __init__(self, prox, rows, cols, eta=None, csc=None, frame_graph=None, background=None):
        self.prox, self.rows, self.cols = prox, int(rows), int(cols)
        self.eta, self.csc, self.frame_graph, self.background = eta, csc, frame_graph, background


def route_graphs(graphs, m, n, img_shape=None, background_masks=None):
    """GraphRoute of inexact_alm_lsd(graphs=...) (background_masks None: all-window graph or any other) or of
    inexact_alm_lsd_with_background (radius-1 centre windows or any other graphs, plus the background)."""
    if background_masks is None:
        if _is_graph_list(graphs):
            glist = list(graphs)
            if len(glist) != n:
                raise Exception("graphs must hold one graph per frame")
            first = detect_window_graph(glist[0], m, img_shape)
            same = first is not None and all(
                (g is glist[0]) or (detect_window_graph(g, m, img_shape) is not None and
                                    np.array_equal(g['eta_g'], glist[0]['eta_g'])) for g in glist[1:])
            geo = first if same else None
        else:
            geo = detect_window_graph(graphs, m, img_shape)
        if geo is None:                                  # any other graph, or per-frame graphs that differ
            csc, frame_graph = pack_graphs(graphs, m, n)
            return GraphRoute(C.PROX_GRAPH_GENERIC, *_geometry(img_shape, m), csc=csc, frame_graph=frame_graph)
        rows, cols, eta = geo
        return GraphRoute(C.PROX_GRAPH_LINF, rows, cols, eta=None if np.all(eta == 1.0) else eta)
    if not isinstance(graphs, list) and not isinstance(graphs, np.ndarray):
        raise Exception('graphs must be list/array')                       # lsd_improvement.py:223-224
    if len(graphs) != n or len(background_masks) != n:
        raise Exception("graphs and background_masks must have one entry per frame")
    eta = np.empty((n, m), dtype=np.float32)
    shape = tuple(img_shape) if img_shape is not None else None
    generic = False
    for f in range(n):
        det = detect_center_windows(graphs[f], m, shape)
        if det is None:                                  # not a radius-1 centre-window graph: the generic graph mode
            generic = True
            break
        if shape is None or graphs[f].get('_group_centers', None) is not None:
            shape = det[0] if shape is None else shape
        if det[0] != tuple(shape):
            raise Exception("frame %d: graph built for image shape %s, expected %s" % (f, det[0], tuple(shape)))
        eta[f] = det[1]
    bg = np.ascontiguousarray(np.stack([np.asarray(b, dtype=bool).ravel() for b in background_masks]).astype(np.uint8))
    if bg.shape != (n, m):
        raise Exception("background_masks must hold %d boolean masks of %d pixels" % (n, m))
    if generic:
        csc, frame_graph = pack_graphs(graphs, m, n)
        return GraphRoute(C.PROX_GRAPH_GENERIC, *_geometry(img_shape, m), csc=csc, frame_graph=frame_graph, background=bg)
    return GraphRoute(C.PROX_GRAPH_CENTER_BG, shape[0], shape[1], eta=eta, background=bg)


def route_weight_mask(weight_mask, m, n, img_shape=None):
    """GraphRoute of the [h, w, t] weight map of build_improved_LSD_graphs (center_window_decomposition): radius-1 centre windows
    weighted by the positive entries, background where an entry is negative."""
    wm = np.asarray(weight_mask)
    h, w = (int(v) for v in (img_shape if img_shape is not None else wm.shape[:2]))
    if wm.shape != (h, w, n) or h * w != m:
        raise Exception("weight_mask must be [h, w, t] with h*w = %d pixels and t = %d frames" % (m, n))
    flat = np.ascontiguousarray(wm.transpose(2, 1, 0)).reshape(n, m)          # [t][p], p = j*rows + i
    eta = np.where(flat > 0, flat, 0).astype(np.float32)
    bg = np.ascontiguousarray((flat < 0).astype(np.uint8))
    return GraphRoute(C.PROX_GRAPH_CENTER_BG, h, w, eta=eta, background=bg)


# --------------------------------------------------------------------------------------------------------------
# marshalling helpers
# --------------------------------------------------------------------------------------------------------------
def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise Exception("bsub_b200: no CUDA device -- the sm_100a path is the only implementation (no CPU fallback)")
    return torch


def _frames_major(D0):
    """Return a C-contiguous float64 [n][m] array sharing memory with the reference's Fortran-order m x n matrix."""
    D = np.asarray(D0)
    if D.ndim != 2:
        raise Exception("D must be a 2-D pixels x frames matrix")
    if D.dtype != np.float64:
        D = D.astype(np.float64)
    if not np.isfortran(D) and not (D.shape[0] == 1 or D.shape[1] == 1):
        D = np.asfortranarray(D)                       # the reference coerces too (inexact_alm_lsd.py:84-88)
    return np.ascontiguousarray(D.T)


def labels_from_blocks(blocks_by_frame, lambdas_by_frame, m):
    """blocks_by_frame (list[n] of lists of bool[m]) -> label map uint8[n][m] + CSR of lambdas; a later block of a
    frame overwrites an earlier one exactly like the sequential assignment of group_sparse_RPCA.py:32-35."""
    n = len(blocks_by_frame)
    if len(lambdas_by_frame) != n:
        raise Exception("blocks_by_frame and lambdas_by_frame must have one entry per frame")
    labels = np.zeros((n, m), dtype=np.uint8)
    ptr = np.zeros(n + 1, dtype=np.int32)
    lam = []
    for f in range(n):
        if len(blocks_by_frame[f]) != len(lambdas_by_frame[f]):
            raise Exception("frame %d: %d blocks but %d lambdas" % (f, len(blocks_by_frame[f]), len(lambdas_by_frame[f])))
        if len(blocks_by_frame[f]) > 254:
            raise Exception("more than 254 blocks in frame %d" % f)
        for b, mask in enumerate(blocks_by_frame[f]):
            labels[f, np.asarray(mask, dtype=bool)] = b + 1
            lam.append(float(lambdas_by_frame[f][b]))
        ptr[f + 1] = ptr[f] + len(blocks_by_frame[f])
    return labels, ptr, np.asarray(lam + [0.0], dtype=np.float64)


class Decomposition:
    """Device-resident result of one solve: owns the bsub_solver handle."""

    def __init__(self, cfg, stream=None):
        _require_cuda()
        self.lib = C.load()
        self.cfg = cfg
        h = ctypes.c_void_p()
        C.check(self.lib.bsub_create(ctypes.byref(cfg), ctypes.byref(h)))
        self.h = h
        self.m, self.n = int(cfg.m), int(cfg.n)
        self._stream = stream

    def stream(self):
        return self._stream if self._stream is not None else _stream_ptr()

    def close(self):
        if getattr(self, "h", None):
            self.lib.bsub_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- inputs
    def load(self, D):
        if _is_torch(D):
            import torch
            if not D.is_cuda:
                D = D.cuda()
            if D.dim() != 2:
                raise Exception("D must be 2-D")
            if tuple(D.shape) == (self.m, self.n):
                D = D.t()
            if tuple(D.shape) != (self.n, self.m):
                raise Exception("D has shape %s, expected (%d, %d)" % (tuple(D.shape), self.m, self.n))
            D = D.to(torch.float32).contiguous()
            self._keep = D
            C.check(self.lib.bsub_load_D_f32_dev(self.h, ctypes.c_void_p(D.data_ptr()), self.m, self.stream()))
        else:
            A = np.asarray(D)
            if A.dtype == np.float32 and A.shape == (self.n, self.m) and A.flags.c_contiguous:
                C.check(self.lib.bsub_load_D_f32_host(self.h, A.ctypes.data_as(ctypes.c_void_p), self.m, self.stream()))
            else:
                A = _frames_major(A)
                if A.shape != (self.n, self.m):
                    raise Exception("D has shape %s, expected (%d, %d)" % (A.shape[::-1], self.m, self.n))
                C.check(self.lib.bsub_load_D_f64_host(self.h, A.ctypes.data_as(ctypes.c_void_p), self.m, self.stream()))

    def load_u8(self, frames, force=None):
        """frames: uint8 [n][m] (frame-major).  Device-side LSD() pre-processing; returns (lo, hi, mean_raw)."""
        A = np.ascontiguousarray(frames, dtype=np.uint8)
        if A.shape != (self.n, self.m):
            raise Exception("frames has shape %s, expected (%d, %d)" % (A.shape, self.n, self.m))
        lo, hi, mean = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_double(0)
        if force is not None:
            lo.value, hi.value, mean.value = force
        C.check(self.lib.bsub_load_u8_host(self.h, A.ctypes.data_as(ctypes.c_void_p), ctypes.byref(lo), ctypes.byref(hi),
                                           ctypes.byref(mean), 1 if force is not None else 0, self.stream()))
        return lo.value, hi.value, mean.value

    def set_flat_groups(self, groups):
        g = np.ascontiguousarray(groups, dtype=np.int32).ravel()
        if g.size != self.m:
            raise Exception("groups has %d entries, matrix has %d rows" % (g.size, self.m))
        C.check(self.lib.bsub_set_flat_groups(self.h, g.ctypes.data_as(C.c_int32_p)))

    def set_graph_windows(self, eta=None):
        if eta is None:
            C.check(self.lib.bsub_set_graph_windows(self.h, None, 0))
        else:
            e = np.ascontiguousarray(eta, dtype=np.float64)
            C.check(self.lib.bsub_set_graph_windows(self.h, e.ctypes.data_as(C.c_double_p), e.size))

    def set_graphs(self, csc, frame_graph, background=None):
        """Any graphs (PROX_GRAPH_GENERIC): csc / frame_graph as returned by pack_graphs; background uint8[n][m] or None."""
        fg = np.ascontiguousarray(frame_graph, dtype=np.int32)
        ng, ip, ix, et = _graph_pointers(csc)
        bg = None if background is None else np.ascontiguousarray(background, dtype=np.uint8)
        C.check(self.lib.bsub_set_graphs(self.h, len(csc), fg.ctypes.data_as(C.c_int32_p), ng.ctypes.data_as(C.c_int64_p), ip, ix, et,
                                         None if bg is None else bg.ctypes.data_as(C.c_uint8_p)))

    def set_route(self, route):
        """The whole-clip description of a GraphRoute (this handle's pixels are whole frames)."""
        if route.prox == C.PROX_GRAPH_LINF:
            self.set_graph_windows(route.eta)
        elif route.prox == C.PROX_GRAPH_GENERIC:
            self.set_graphs(route.csc, route.frame_graph, route.background)
        else:
            C.check(self.lib.bsub_set_center_windows(self.h, route.eta.ctypes.data_as(C.c_float_p),
                                                     route.background.ctypes.data_as(C.c_uint8_p)))

    def set_frame_route(self, route, f0, f1):
        """Frame-range description of a GraphRoute: the prox of whole frames [f0, f1) (bsub_set_frame_*, run by
        bsub_step_prox_block).  Only those frames' graphs, weights and background are uploaded."""
        rows, cols, nf = route.rows, route.cols, f1 - f0
        bg = None if route.background is None else np.ascontiguousarray(route.background[f0:f1])
        bgp = None if bg is None else bg.ctypes.data_as(C.c_uint8_p)
        if route.prox == C.PROX_GRAPH_LINF:
            e = None if route.eta is None else np.ascontiguousarray(route.eta, dtype=np.float64)
            C.check(self.lib.bsub_set_frame_windows(self.h, rows, cols, f0, nf, None if e is None else e.ctypes.data_as(C.c_double_p),
                                                    0 if e is None else e.size))
        elif route.prox == C.PROX_GRAPH_CENTER_BG:
            eta = np.ascontiguousarray(route.eta[f0:f1], dtype=np.float32)
            C.check(self.lib.bsub_set_frame_center_windows(self.h, rows, cols, f0, nf, eta.ctypes.data_as(C.c_float_p), bgp))
        else:
            used, fg = np.unique(np.asarray(route.frame_graph[f0:f1]), return_inverse=True)
            csc = [route.csc[k] for k in used]
            fg = np.ascontiguousarray(fg, dtype=np.int32)
            ng, ip, ix, et = _graph_pointers(csc)
            C.check(self.lib.bsub_set_frame_graphs(self.h, rows, cols, f0, nf, len(csc), fg.ctypes.data_as(C.c_int32_p),
                                                   ng.ctypes.data_as(C.c_int64_p), ip, ix, et, bgp))

    def set_frame_weight_map(self, weight, rows, cols, f0):
        """Device variant of set_frame_route for LSD_improved's weight map: weight = CUDA tensor float32 [nf][rows * cols] (row pitch
        weight.stride(0)) of frames [f0, f0 + nf); > 0 centre-window weight, < 0 background (bsub_set_frame_weight_map_dev)."""
        import torch
        if not (_is_torch(weight) and weight.is_cuda and weight.dtype == torch.float32 and weight.dim() == 2 and
                weight.shape[1] == rows * cols and (weight.shape[0] == 0 or weight.stride(1) == 1)):
            raise Exception("weight map must be a CUDA float32 tensor [frames][%d] with unit pixel stride" % (rows * cols))
        nf = int(weight.shape[0])
        C.check(self.lib.bsub_set_frame_weight_map_dev(self.h, rows, cols, f0, nf, ctypes.c_void_p(weight.data_ptr()) if nf else None,
                                                       int(weight.stride(0)) if nf else rows * cols, self.stream()))

    def set_blocks(self, labels, lam_ptr, lam):
        labels = np.ascontiguousarray(labels, dtype=np.uint8)
        lam_ptr = np.ascontiguousarray(lam_ptr, dtype=np.int32)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        if labels.shape != (self.n, self.m):
            raise Exception("labels has shape %s, expected (%d, %d)" % (labels.shape, self.n, self.m))
        C.check(self.lib.bsub_set_blocks(self.h, labels.ctypes.data_as(C.c_uint8_p), lam_ptr.ctypes.data_as(C.c_int32_p),
                                         lam.ctypes.data_as(C.c_double_p)))

    # -- solve
    def run(self):
        C.check(self.lib.bsub_run(self.h, self.stream()))
        return self

    def status(self):
        st = C.Status()
        C.check(self.lib.bsub_sync_status(self.h, ctypes.byref(st), self.stream()))
        return st

    def poll(self):
        st = C.Status()
        C.check(self.lib.bsub_poll(self.h, ctypes.byref(st)))
        return st

    def debug_info(self):
        """Which kernel paths this solver uses (TMA / streamed shrink / int8 tcgen05 Gram) and their tile shapes."""
        out = (ctypes.c_int32 * 16)()
        C.check(self.lib.bsub_debug_info(self.h, out))
        keys = ["use_tma", "use_stream", "use_i8", "stream_R", "stream_FC", "stream_NS", "gram_types", "gram_kc", "eig_cluster",
                "tma_R", "tma_Cf", "ld", "use_proj", "proj_warps", "proj_depth", "flat_stages"]
        return dict(zip(keys, [int(v) for v in out]))

    def counters(self):
        out = (ctypes.c_int64 * 8)()
        C.check(self.lib.bsub_debug_counters(self.h, out))
        keys = ["eig_fast_iters", "eig_p", "eig_fast_steps", "eig_gb_ppm", "gram_mode", "wq_saturated", "force_dmma", "gram_err_ppm"]
        return dict(zip(keys, [int(v) for v in out]))

    def eig_fast_count(self):
        """Iterations of the last solve whose eigenpairs came from the warm-started subspace path."""
        return self.counters()["eig_fast_iters"]

    def log(self):
        buf = (C.IterLog * 512)()
        cnt = ctypes.c_int32(0)
        C.check(self.lib.bsub_get_log(self.h, buf, 512, ctypes.byref(cnt)))
        return [dict(iter=b.iter, svp=b.svp, sv=b.sv, err=b.err, mu=b.mu, nnz=int(b.nnz)) for b in buf[:cnt.value]]

    # -- outputs
    def finalize(self):
        C.check(self.lib.bsub_finalize(self.h, self.stream()))

    def download(self, which, dtype=np.float64):
        """which: 'L' | 'S' | 'D' | 'Y'.  Returns an m x n Fortran-order array (the reference's layout)."""
        sel = {'L': 0, 'S': 1, 'D': 2, 'Y': 3}[which]
        out = np.empty((self.n, self.m), dtype=dtype)
        fn = self.lib.bsub_download_f64 if dtype == np.float64 else self.lib.bsub_download_f32
        C.check(fn(self.h, sel, out.ctypes.data_as(ctypes.c_void_p), self.m, self.stream()))
        return out.T

    def device_tensor(self, which):
        """Zero-copy torch view [n][ld] of a device matrix (ld >= m, pad columns are zero)."""
        import torch
        fn = {'L': self.lib.bsub_get_L_f32_dev, 'S': self.lib.bsub_get_S_f32_dev, 'D': self.lib.bsub_get_D_f32_dev,
              'Y': self.lib.bsub_get_Y_f32_dev}[which]
        p, ld = ctypes.c_void_p(), ctypes.c_int64(0)
        if which in ('L', 'S'):
            self.finalize()
        C.check(fn(self.h, ctypes.byref(p), ctypes.byref(ld)))
        return _wrap_device(p.value, (self.n, ld.value), torch.float32)[:, :self.m]

    def mask(self, sigmas_from_mean=2):
        out = np.empty((self.n, self.m), dtype=np.uint8)
        C.check(self.lib.bsub_mask_host(self.h, float(sigmas_from_mean), out.ctypes.data_as(ctypes.c_void_p), self.stream()))
        return out.T.astype(bool)


class _CudaArray:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def _wrap_device(ptr, shape, dtype):
    import torch
    typestr = {torch.float32: "<f4", torch.float64: "<f8", torch.uint8: "|u1"}[dtype]
    return torch.as_tensor(_CudaArray(ptr, shape, typestr), device="cuda")


def make_config(m, n, prox, rows=0, cols=0, delta=10, mu_scale=12.5, rho=1.6, tol=1e-7, max_iter=500, sv0=10,
                use_sv_prediction=True, break_on_rank0=False, m_global=0, d_global=0, tile_rows=0, cluster_frames=0,
                graph_max_sweeps=0, graph_tol=0.0, flags=0):
    cfg = C.Config()
    C.load().bsub_default_config(ctypes.byref(cfg))
    cfg.m, cfg.n, cfg.prox, cfg.rows, cfg.cols = int(m), int(n), int(prox), int(rows), int(cols)
    cfg.delta, cfg.mu_scale, cfg.rho, cfg.tol = float(delta), float(mu_scale), float(rho), float(tol)
    cfg.max_iter, cfg.sv0 = int(max_iter), int(sv0)
    cfg.use_sv_prediction, cfg.break_on_rank0 = int(bool(use_sv_prediction)), int(bool(break_on_rank0))
    cfg.m_global, cfg.d_global = int(m_global), int(d_global)
    cfg.tile_rows, cfg.cluster_frames = int(tile_rows), int(cluster_frames)
    cfg.graph_max_sweeps, cfg.graph_tol = int(graph_max_sweeps), float(graph_tol)
    cfg.flags = int(flags)
    return cfg


def _shape_of(D0):
    if _is_torch(D0):
        return int(D0.shape[0]), int(D0.shape[1])
    return np.shape(D0)


def _geometry(img_shape, m):
    """(rows, cols) of img_shape when it describes the m pixels, else (0, 0) (the generic graph mode needs no geometry)."""
    if img_shape is not None and int(img_shape[0]) * int(img_shape[1]) == m:
        return int(img_shape[0]), int(img_shape[1])
    return 0, 0


def _finish(dec, D0, verbose):
    st = dec.status()
    if verbose:
        for l in dec.log():
            print(f"Iteration: {l['iter']:3d} rank(L): {l['svp']:2d} ||S||_0: {l['nnz']:.2E} err: {l['err']:.3E}")
        print('CONVERGED' if st.converged else ('L reached rank 0' if st.done == 3 else 'NOT CONVERGED'))
    if _is_torch(D0):
        # copies that own their storage: a view of solver memory would dangle as soon as a derived view (L[:, :k], .t(), ...)
        # outlives the handle (ADVICE r1).  Zero-copy access stays available through Decomposition.device_tensor().
        L = dec.device_tensor('L').clone().t()
        S = dec.device_tensor('S').clone().t()
    else:
        L = dec.download('L')
        S = dec.download('S')
    return L, S, int(st.iter), bool(st.converged)


# --------------------------------------------------------------------------------------------------------------
# the solvers
# --------------------------------------------------------------------------------------------------------------
def lsd_decomposition(D0, graphs=None, groups=None, delta=10, img_shape=None, max_iter=500, tile_rows=0, cluster_frames=0,
                      graph_max_sweeps=0, graph_tol=0.0):
    """Run inexact_alm_lsd on the GPU and keep everything resident; returns the Decomposition handle."""
    if graphs is None and groups is None:
        raise Exception("one of graphs or groups must not be None")
    if graphs is not None and groups is not None:
        raise Exception("only one of graphs or groups must not be None")
    m, n = _shape_of(D0)
    if groups is not None:
        geo = detect_flat_tiling(groups, img_shape)
        rows, cols = geo if geo is not None else (m, 1)
        cfg = make_config(m, n, C.PROX_FLAT_LINF, rows, cols, delta=delta, max_iter=max_iter, tile_rows=tile_rows,
                          cluster_frames=cluster_frames)
        dec = Decomposition(cfg)
        dec.set_flat_groups(groups)
    else:
        route = route_graphs(graphs, m, n, img_shape)
        cfg = make_config(m, n, route.prox, route.rows, route.cols, delta=delta, max_iter=max_iter, tile_rows=tile_rows,
                          cluster_frames=cluster_frames, graph_max_sweeps=graph_max_sweeps, graph_tol=graph_tol)
        dec = Decomposition(cfg)
        dec.set_route(route)
    dec.load(D0)
    dec.run()
    return dec


def inexact_alm_lsd(D0, graphs=None, groups=None, delta=10, img_shape=None, verbose=False, **tuning):
    """Drop-in for /root/reference/inexact_alm_lsd.py:82-179 -> (L, S, iter_out, converged)."""
    dec = lsd_decomposition(D0, graphs=graphs, groups=groups, delta=delta, img_shape=img_shape, **tuning)
    return _finish(dec, D0, verbose)


def inexact_alm_lsd_batch(clips, groups=None, graphs=None, delta=10, img_shape=None, in_flight=4, **tuning):
    """Independent decompositions of several clips (BASELINE.json config 5: "one decomposition per clip"), `in_flight` of
    them at a time on this GPU: one solver handle, host thread and CUDA stream per clip in flight, so the uploads and
    downloads of one clip and the 8-SM eigensolve of another overlap the streaming kernels of the rest.  Same arguments
    as inexact_alm_lsd for every clip; returns a list of (L, S, iter_out, converged) in input order."""
    import threading
    torch = _require_cuda()
    clips = list(clips)
    out = [None] * len(clips)
    errs = []
    nxt = [0]
    lock = threading.Lock()
    dev = torch.cuda.current_device()

    def worker():
        try:
            torch.cuda.set_device(dev)
            with torch.cuda.stream(torch.cuda.Stream()):
                while True:
                    with lock:
                        i = nxt[0]
                        nxt[0] += 1
                    if i >= len(clips) or errs:
                        return
                    out[i] = inexact_alm_lsd(clips[i], graphs=graphs, groups=groups, delta=delta, img_shape=img_shape, **tuning)
                    torch.cuda.current_stream().synchronize()
        except Exception as ex:                                  # re-raised in the caller
            errs.append(ex)

    th = [threading.Thread(target=worker) for _ in range(max(1, min(int(in_flight), len(clips))))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if errs:
        raise errs[0]
    return out


def with_background_decomposition(D0, graphs, background_masks, delta=10, img_shape=None, **tuning):
    m, n = _shape_of(D0)
    route = route_graphs(graphs, m, n, img_shape, background_masks=background_masks)
    dec = Decomposition(make_config(m, n, route.prox, route.rows, route.cols, delta=delta, **tuning))
    dec.set_route(route)
    dec.load(D0)
    dec.run()
    return dec


def center_window_decomposition(D0, weight_mask, delta=10, img_shape=None, **tuning):
    """inexact_alm_lsd_with_background straight from the [h, w, t] weight map of build_improved_LSD_graphs
    (/root/reference/lsd_improvement.py:406-436): a positive entry is the weight of the 3x3 window centred on that pixel of that
    frame, a negative one marks a background pixel -- the per-frame SPAMS graphs are never built."""
    m, n = _shape_of(D0)
    route = route_weight_mask(weight_mask, m, n, img_shape)
    dec = Decomposition(make_config(m, n, route.prox, route.rows, route.cols, delta=delta, **tuning))
    dec.set_route(route)
    dec.load(D0)
    dec.run()
    return dec


def inexact_alm_lsd_with_background(D0, graphs, background_masks, delta=10, img_shape=None, verbose=False, **tuning):
    """Drop-in for /root/reference/lsd_improvement.py:215-304 -> (L, S, iter_out, converged): one centre-window graph
    per frame (prox_by_frame) plus the l2 shrink of every frame's background pixels at 100 lambda / mu."""
    dec = with_background_decomposition(D0, graphs, background_masks, delta=delta, img_shape=img_shape, **tuning)
    return _finish(dec, D0, verbose)


def apply_background_shrinkage_operator(G, output, epsilon, background_masks):
    """Drop-in for /root/reference/lsd_improvement.py:199-212 (in place on `output`, which is also returned): every
    frame's background pixels become max(1 - epsilon/||G_bg||_2, 0) * G_bg.  Runs block_shrinkage_operator on the
    device with the background as the only (complement) group, mu = 1, non-block lambda = epsilon."""
    G = np.asarray(G)
    n = G.shape[1]
    fg_blocks = [[~np.asarray(background_masks[f], dtype=bool)] for f in range(n)]
    shrunk = block_shrinkage_operator(G, fg_blocks, [[0.0]] * n, 1.0, float(epsilon))
    for f in range(n):
        mk = np.asarray(background_masks[f], dtype=bool)
        output[mk, f] = shrunk[mk, f]
    return output


def group_sparse_decomposition(D0, blocks_by_frame, lambdas_by_frame, delta=10, use_sv_prediction=True, img_shape=None,
                               labels=None, max_iter=500):
    m, n = _shape_of(D0)
    if labels is None:
        labels, ptr, lam = labels_from_blocks(blocks_by_frame, lambdas_by_frame, m)
    else:
        labels, ptr, lam = labels
    rows, cols = img_shape if img_shape is not None else (0, 0)
    cfg = make_config(m, n, C.PROX_BLOCK_L2, rows, cols, delta=delta, mu_scale=1.25, break_on_rank0=True,
                      use_sv_prediction=use_sv_prediction, max_iter=max_iter)
    dec = Decomposition(cfg)
    dec.set_blocks(labels, ptr, lam)
    dec.load(D0)
    dec.run()
    return dec


def inexact_alm_group_sparse_RPCA(D0, blocks_by_frame, lambdas_by_frame, delta=10, use_sv_prediction=True, verbose=False,
                                  img_shape=None):
    """Drop-in for /root/reference/group_sparse_RPCA.py:45-126 -> (L, S, iter_out, converged)."""
    dec = group_sparse_decomposition(D0, blocks_by_frame, lambdas_by_frame, delta, use_sv_prediction, img_shape)
    return _finish(dec, D0, verbose)


def inexact_alm_rpca(D0, delta=1.0, use_sv_prediction=False, verbose=False):
    """Drop-in for /root/reference/lsd_improvement.py:123-196 (plain l1 RPCA; rho = 1.2, mu0 = 1.25/||D||_2)."""
    m, n = _shape_of(D0)
    cfg = make_config(m, n, C.PROX_L1, 0, 0, delta=delta, mu_scale=1.25, rho=1.2, use_sv_prediction=use_sv_prediction)
    dec = Decomposition(cfg)
    dec.load(D0)
    dec.run()
    return _finish(dec, D0, verbose)


# --------------------------------------------------------------------------------------------------------------
# mask and LSD()
# --------------------------------------------------------------------------------------------------------------
def _to_device_f32(A, m, n):
    """m x n (reference layout) host/torch matrix -> torch float32 [n][ld] with zero pad, ld % 32 == 0."""
    torch = _require_cuda()
    ld = (m + 31) // 32 * 32
    buf = torch.zeros((n, ld), dtype=torch.float32, device="cuda")
    if _is_torch(A):
        buf[:, :m] = A.t().to(torch.float32) if tuple(A.shape) == (m, n) else A.to(torch.float32)
    else:
        buf[:, :m] = torch.from_numpy(np.ascontiguousarray(np.asarray(A, dtype=np.float64).T)).to("cuda").to(torch.float32)
    return buf, ld


def foreground_mask(D, L, S, sigmas_from_mean=2):
    """Drop-in for /root/reference/utils.py:139-149: boolean m x n mask."""
    torch = _require_cuda()
    m, n = _shape_of(D)
    lib = C.load()
    d, ld = _to_device_f32(D, m, n)
    l, _ = _to_device_f32(L, m, n)
    s, _ = _to_device_f32(S, m, n)
    mask = torch.empty((n, m), dtype=torch.uint8, device="cuda")
    C.check(lib.bsub_foreground_mask_dev(ctypes.c_void_p(d.data_ptr()), ctypes.c_void_p(l.data_ptr()),
                                         ctypes.c_void_p(s.data_ptr()), ld, m, n, float(sigmas_from_mean),
                                         ctypes.c_void_p(mask.data_ptr()), _stream_ptr()))
    if _is_torch(D):
        return mask.t().bool()
    return mask.cpu().numpy().T.astype(bool)


def normalizeImage(image):
    """/root/reference/utils.py:220-223 (in place)."""
    image -= np.min(image)
    image *= 1.0 / np.max(image)


def resize_with_cv2(images, ratio):
    """/root/reference/utils.py:129-136 on the device (cv2.INTER_AREA / INTER_CUBIC restated in csrc/post.cu)."""
    from . import flow
    return flow.resize_with_cv2(images, ratio)


def LSD(ImData0, frame_start, frame_end, downsample_ratio, use_flat=False):
    """Drop-in for /root/reference/inexact_alm_lsd.py:203-235 -> (S, S_mask, L, ImData1, ImMean, shape, iterations,
    converged).  Like the reference it normalises ImData0 in place when downsample_ratio == 1 (SURVEY Q17).
    use_flat=True swaps the overlapping graph for the flat 3x3 tiling (the north-star fast path)."""
    if downsample_ratio == 1:
        ImData1 = ImData0
    else:
        ImData1 = resize_with_cv2(ImData0[:, :, frame_start:(frame_end + 1)], 1 / downsample_ratio)
    normalizeImage(ImData1)
    ImMean = np.mean(ImData1)
    ImData2 = ImData1 - ImMean
    shape = ImData2.shape
    h, w, frames = shape
    D = ImData2.reshape((h * w, frames), order='F')
    if use_flat:
        dec = lsd_decomposition(D, groups=get_proximal_flat_groups_nonoverlap((h, w), BLOCK_SIZE), img_shape=(h, w))
    else:
        dec = lsd_decomposition(D, graphs=getGraphSPAMS_all_groups((h, w), BLOCK_SIZE), img_shape=(h, w))
    L, S, iterations, converged = _finish(dec, D, False)
    S_mask = dec.mask(2)
    return (S.reshape(shape, order='F'), S_mask.reshape(shape, order='F'), L.reshape(shape, order='F'), ImData1, ImMean,
            shape, iterations, converged)


# --------------------------------------------------------------------------------------------------------------
# operator seams
# --------------------------------------------------------------------------------------------------------------
def _op_out(buf, m, like):
    if _is_torch(like):
        return buf[:, :m].t()
    return np.asfortranarray(buf[:, :m].t().double().cpu().numpy())


def prox_flat(G_S, lambda1, groups, num_threads=None, img_shape=None):
    """/root/reference/inexact_alm_lsd.py:71-79."""
    torch = _require_cuda()
    m, n = _shape_of(G_S)
    lib = C.load()
    u, ld = _to_device_f32(G_S, m, n)
    v = torch.zeros_like(u)
    geo = detect_flat_tiling(groups, img_shape)
    if geo is not None:
        C.check(lib.bsub_prox_flat3_dev(ctypes.c_void_p(u.data_ptr()), ctypes.c_void_p(v.data_ptr()), ld, geo[0], geo[1], n,
                                        float(lambda1), _stream_ptr()))
    else:
        g = np.ascontiguousarray(groups, dtype=np.int32).ravel()
        if g.size != m:
            raise Exception("groups has %d entries, matrix has %d rows" % (g.size, m))
        C.check(lib.bsub_prox_flat_groups_dev(ctypes.c_void_p(u.data_ptr()), ctypes.c_void_p(v.data_ptr()), ld, m, n,
                                              g.ctypes.data_as(C.c_int32_p), float(lambda1), _stream_ptr()))
    torch.cuda.current_stream().synchronize()
    return _op_out(v, m, G_S)


def prox(G_S, lambda1, graph, num_threads=None, img_shape=None, max_sweeps=20000, tol=1e-7, return_sweeps=False):
    """/root/reference/inexact_alm_lsd.py:49-57: the 3x3 all-windows graph and the radius-1 centre-window graphs on their
    dedicated kernels, any other graph on the generic one."""
    torch = _require_cuda()
    m, n = _shape_of(G_S)
    geo = detect_window_graph(graph, m, img_shape)
    if geo is None:
        ctr = detect_center_windows(graph, m, img_shape)           # a per-frame graph of get_proximal_graph_group_centers
        if ctr is None:
            return _prox_generic(G_S, lambda1, graph, max_sweeps, tol, return_sweeps)
        return _prox_center(G_S, lambda1, ctr[0], np.tile(ctr[1], (n, 1)), max_sweeps, tol, return_sweeps)
    rows, cols, eta = geo
    lib = C.load()
    u, ld = _to_device_f32(G_S, m, n)
    v = torch.zeros_like(u)
    sw = ctypes.c_int32(0)
    eta_p = None if np.all(eta == 1.0) else eta.ctypes.data_as(C.c_double_p)
    C.check(lib.bsub_prox_graph3_dev(ctypes.c_void_p(u.data_ptr()), ctypes.c_void_p(v.data_ptr()), ld, rows, cols, n,
                                     float(lambda1), eta_p, int(max_sweeps), float(tol) * float(lambda1), ctypes.byref(sw),
                                     _stream_ptr()))
    out = _op_out(v, m, G_S)
    return (out, sw.value) if return_sweeps else out


def _prox_center(G_S, lambda1, shape, eta_nm, max_sweeps=20000, tol=1e-7, return_sweeps=False):
    """Centre-window graphs, one weight map per frame (eta_nm float32 [n][m]); all frames in one launch."""
    torch = _require_cuda()
    m, n = _shape_of(G_S)
    lib = C.load()
    u, ld = _to_device_f32(G_S, m, n)
    v = torch.zeros_like(u)
    sw = ctypes.c_int32(0)
    eta_nm = np.ascontiguousarray(eta_nm, dtype=np.float32)
    C.check(lib.bsub_prox_center3_dev(ctypes.c_void_p(u.data_ptr()), ctypes.c_void_p(v.data_ptr()), ld, int(shape[0]), int(shape[1]), n,
                                      float(lambda1), eta_nm.ctypes.data_as(C.c_float_p), int(max_sweeps),
                                      float(tol) * float(lambda1), ctypes.byref(sw), _stream_ptr()))
    out = _op_out(v, m, G_S)
    return (out, sw.value) if return_sweeps else out


def _prox_generic(G_S, lambda1, graphs, max_sweeps=20000, tol=1e-7, return_sweeps=False):
    """Any graph, or one graph per frame (pack_graphs); all frames in one launch."""
    torch = _require_cuda()
    m, n = _shape_of(G_S)
    csc, frame_graph = pack_graphs(graphs, m, n)
    ng, ip, ix, et = _graph_pointers(csc)
    lib = C.load()
    u, ld = _to_device_f32(G_S, m, n)
    v = torch.zeros_like(u)
    sw = ctypes.c_int32(0)
    C.check(lib.bsub_prox_graph_dev(ctypes.c_void_p(u.data_ptr()), ctypes.c_void_p(v.data_ptr()), ld, m, n, float(lambda1), len(csc),
                                    frame_graph.ctypes.data_as(C.c_int32_p), ng.ctypes.data_as(C.c_int64_p), ip, ix, et,
                                    int(max_sweeps), float(tol) * float(lambda1), ctypes.byref(sw), _stream_ptr()))
    out = _op_out(v, m, G_S)
    return (out, sw.value) if return_sweeps else out


def prox_by_frame(G_S, lambda1, graphs, img_shape=None):
    """/root/reference/inexact_alm_lsd.py:60-68: one graph per column.  Centre-window graphs (the per-frame graphs the
    reference builds) go through one launch for all frames, as does any list with a graph the dedicated kernels do not take;
    lists of 3x3 all-window and radius-1 centre-window graphs go frame by frame through prox()."""
    m, n = _shape_of(G_S)
    win = [detect_window_graph(g, m, img_shape) is not None for g in graphs]
    dets = [detect_center_windows(g, m, img_shape) if not w else None for g, w in zip(graphs, win)]
    if len(dets) == n and all(d is not None for d in dets) and len({d[0] for d in dets}) == 1:
        return _prox_center(G_S, lambda1, dets[0][0], np.stack([d[1] for d in dets]))
    if len(dets) != n or not all(w or d is not None for w, d in zip(win, dets)):
        return _prox_generic(G_S, lambda1, list(graphs))
    cols = [prox(G_S[:, [f]], lambda1, graphs[f], img_shape=img_shape) for f in range(n)]
    return np.column_stack(cols)


def block_shrinkage_operator(G, blocks_by_frame, lambdas_by_frame, mu, non_block_lambda):
    """/root/reference/group_sparse_RPCA.py:13-42."""
    torch = _require_cuda()
    m, n = _shape_of(G)
    lib = C.load()
    labels, ptr, lam = labels_from_blocks(blocks_by_frame, lambdas_by_frame, m)
    u, ld = _to_device_f32(G, m, n)
    v = torch.zeros_like(u)
    C.check(lib.bsub_block_shrink_dev(ctypes.c_void_p(u.data_ptr()), ctypes.c_void_p(v.data_ptr()), ld, m, n,
                                      labels.ctypes.data_as(C.c_uint8_p), ptr.ctypes.data_as(C.c_int32_p),
                                      lam.ctypes.data_as(C.c_double_p), float(mu), float(non_block_lambda), _stream_ptr()))
    return _op_out(v, m, G)


def gram(D, S=None, Y=None, mu=1.0):
    """frames x frames Gram of W = D - S + Y/mu in fp64 (the n x n core that replaces the m x n SVD)."""
    _require_cuda()
    m, n = _shape_of(D)
    lib = C.load()
    d, ld = _to_device_f32(D, m, n)
    sp = yp = None
    if S is not None:
        s, _ = _to_device_f32(S, m, n)
        y, _ = _to_device_f32(Y, m, n)
        sp, yp = ctypes.c_void_p(s.data_ptr()), ctypes.c_void_p(y.data_ptr())
    G = np.empty((n, n), dtype=np.float64)
    C.check(lib.bsub_gram_dev(ctypes.c_void_p(d.data_ptr()), sp, yp, ld, m, n, float(mu), G.ctypes.data_as(C.c_double_p),
                              _stream_ptr()))
    return G


def eig_topk(G, k):
    """Top-k eigenpairs (descending) of a symmetric matrix with the device eigensolver."""
    _require_cuda()
    G = np.ascontiguousarray(G, dtype=np.float64)
    n = G.shape[0]
    lam = np.empty(k, dtype=np.float64)
    vec = np.empty((k, n), dtype=np.float64)
    C.check(C.load().bsub_eig_topk(G.ctypes.data_as(C.c_double_p), n, int(k), lam.ctypes.data_as(C.c_double_p),
                                   vec.ctypes.data_as(C.c_double_p)))
    return lam, vec


def svd_k_largest(G, k):
    """/root/reference/utils.py:204-212 through the Gram route: (u, s, vh) with s descending.  The left vectors are
    formed on the host (u = G v / s); the solver itself never needs them."""
    Gm = np.asarray(G, dtype=np.float64)
    gr = gram(Gm)
    lam, vec = eig_topk(gr, k)
    s = np.sqrt(np.maximum(lam, 0.0))
    with np.errstate(divide='ignore', invalid='ignore'):
        u = (Gm @ vec.T) / s
    return u, s, vec
