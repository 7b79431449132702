"""Host-side mirror of the reference's stages on either side of the decomposition, running on the device through the C ABI
(csrc/post.cu).  Same names, arguments and return values as the reference functions they replace:

    resize_with_cv2, resize_with_cv2_by_first_axis      /root/reference/utils.py:119-136
    filter_sparse_map                                   /root/reference/utils.py:404-420
    gkern, computeSCube                                 /root/reference/computeSCube.py:9-19, 82-92
    compute_groups_per_frame, filter_groups,
    run_motion_saliency_check                           /root/reference/motion_saliency_check.py:19-120
    get_footprint (disk), apply_morph_ops, merge_masks,
    calc_mask_percent, build_improved_LSD_graphs,
    LSD_improved                                        /root/reference/lsd_improvement.py:307-351, 369-487

There is no CPU fallback: every function raises without a CUDA device.  The pixel work (resampling, connected components and
their statistics, smoothing, morphology) runs in CUDA kernels; the host keeps only the per-component bookkeeping the reference
does on a handful of components per frame (bbox nesting, weight / size filter, lambda normalisation).
"""
import ctypes
import math

import numpy as np

from . import _cabi as C
from . import api as A


def _vp(t):
    return ctypes.c_void_p(t.data_ptr())


def _torch():
    return A._require_cuda()


# --------------------------------------------------------------------------------------------------------------
# resize
# --------------------------------------------------------------------------------------------------------------
def _resize(images, ratio, time_axis):
    """images: [h, w, T] (time_axis 2) or [T, h, w] (time_axis 0) host array or CUDA tensor."""
    torch = _torch()
    hw = [i for i in range(3) if i != time_axis]
    size = [int(np.ceil(images.shape[i] * ratio)) for i in hw]
    interp = 0 if ratio < 1 else 1                       # cv2.INTER_AREA if ratio < 1 else cv2.INTER_CUBIC
    on_dev = A._is_torch(images)
    src = images.to(torch.float32).contiguous() if on_dev else \
        torch.from_numpy(np.ascontiguousarray(images, dtype=np.float32)).to("cuda")
    T = src.shape[time_axis]
    out_shape = list(src.shape)
    out_shape[hw[0]], out_shape[hw[1]] = size
    dst = torch.empty(out_shape, dtype=torch.float32, device="cuda")
    ss, ds = src.stride(), dst.stride()
    C.check(C.load().bsub_resize_dev(_vp(src), ss[time_axis], ss[hw[0]], ss[hw[1]], src.shape[hw[0]], src.shape[hw[1]], T,
                                     _vp(dst), ds[time_axis], ds[hw[0]], ds[hw[1]], size[0], size[1], interp, A._stream_ptr()))
    return dst if on_dev else dst.double().cpu().numpy()


def resize_with_cv2(images, ratio):
    """/root/reference/utils.py:129-136: every [:, :, t] slice resized to ceil(shape * ratio)."""
    return _resize(images, ratio, 2)


def resize_with_cv2_by_first_axis(images, ratio):
    """/root/reference/utils.py:119-126: every [t, :, :] slice."""
    return _resize(images, ratio, 0)


# --------------------------------------------------------------------------------------------------------------
# connected components
# --------------------------------------------------------------------------------------------------------------
def _mask_to_device(cube_hwt):
    """[h, w, t] boolean cube -> uint8 [t][w*h] on the device (pixel p = j*rows + i, the solver's layout)."""
    torch = _torch()
    if A._is_torch(cube_hwt):
        h, w, t = cube_hwt.shape
        return (cube_hwt != 0).permute(2, 1, 0).contiguous().view(t, w * h).to(torch.uint8), (h, w, t)
    a = np.asarray(cube_hwt)
    h, w, t = a.shape
    host = np.ascontiguousarray((a != 0).transpose(2, 1, 0)).reshape(t, w * h).astype(np.uint8)
    return torch.from_numpy(host).to("cuda"), (h, w, t)


def _mask_from_device(dev, shape, like):
    h, w, t = shape
    out = dev.view(t, w, h).permute(2, 1, 0) != 0
    return out if A._is_torch(like) else np.ascontiguousarray(out.cpu().numpy())


class Components:
    """Per-frame 8-connected components of a binary video, resident on the device."""

    def __init__(self, mask_dev, shape, weight=None):
        torch = _torch()
        h, w, t = shape
        m = h * w
        lib = C.load()
        self.shape, self.m = shape, m
        self.labels = torch.empty((t, m), dtype=torch.int32, device="cuda")
        num = torch.empty(t, dtype=torch.int32, device="cuda")
        scratch = torch.empty((2, t, m), dtype=torch.int32, device="cuda")
        C.check(lib.bsub_cc_label_dev(_vp(mask_dev), m, h, w, t, _vp(self.labels), m, _vp(num), _vp(scratch), A._stream_ptr()))
        del scratch
        self.num = num.cpu().numpy().astype(np.int64)                       # components per frame (syncs)
        self.offsets = np.concatenate([[0], np.cumsum(self.num)]).astype(np.int64)
        total = int(self.offsets[-1])
        self.total = total
        self.offsets_dev = torch.from_numpy(self.offsets[:-1].astype(np.int32)).to("cuda")
        area = torch.zeros(max(total, 1), dtype=torch.int32, device="cuda")
        box = torch.zeros((max(total, 1), 5), dtype=torch.int32, device="cuda")
        wsum = torch.zeros(max(total, 1), dtype=torch.float64, device="cuda")
        if weight is not None:
            wt, (sf, sj, si) = weight
            C.check(lib.bsub_cc_stats_dev(_vp(self.labels), m, h, w, t, _vp(self.offsets_dev), total, _vp(wt), sf, sj, si, _vp(area),
                                          _vp(box), _vp(wsum), A._stream_ptr()))
        else:
            C.check(lib.bsub_cc_stats_dev(_vp(self.labels), m, h, w, t, _vp(self.offsets_dev), total, None, 0, 0, 0, _vp(area), _vp(box),
                                          None, A._stream_ptr()))
        self.area = area.cpu().numpy()[:total].astype(np.int64)
        self.box = box.cpu().numpy()[:total].astype(np.int64)              # min row, max row, min col, max col, first 2x2 block
        self.wsum = wsum.cpu().numpy()[:total]

    def frame_order(self, f):
        """Component slots of frame f in OpenCV's label order (labels 1..K of cv2.connectedComponentsWithStats)."""
        lo, hi = int(self.offsets[f]), int(self.offsets[f + 1])
        return lo + np.argsort(self.box[lo:hi, 4], kind="stable")

    def stats_cv2(self, f):
        """(left, top, width, height, area) rows for labels 1..K of frame f, in OpenCV's order."""
        idx = self.frame_order(f)
        b = self.box[idx]
        return np.stack([b[:, 2], b[:, 0], b[:, 3] - b[:, 2] + 1, b[:, 1] - b[:, 0] + 1, self.area[idx]], axis=1), idx

    def remap(self, table):
        """uint8 [t][m] device map: table[slot] for every pixel of component `slot`, 0 elsewhere."""
        torch = _torch()
        h, w, t = self.shape
        tb = torch.from_numpy(np.ascontiguousarray(table, dtype=np.uint8) if self.total else np.zeros(1, dtype=np.uint8)).to("cuda")
        out = torch.empty((t, self.m), dtype=torch.uint8, device="cuda")
        C.check(C.load().bsub_cc_remap_dev(_vp(self.labels), self.m, self.m, t, _vp(self.offsets_dev), _vp(tb), _vp(out), self.m,
                                           A._stream_ptr()))
        return out


def connected_components(cube_hwt):
    """Components of every [:, :, t] slice (8-connectivity): returns a Components object."""
    dev, shape = _mask_to_device(cube_hwt)
    return Components(dev, shape)


def filter_sparse_map(sparse_array, size_thresh=None):
    """/root/reference/utils.py:404-420: drop the 8-connected objects of every frame whose area is <= size_thresh."""
    torch = _torch()
    if size_thresh is None:
        size_thresh = (sparse_array.shape[0] * sparse_array.shape[1]) // 200
    dev, (h, w, t) = _mask_to_device(sparse_array)
    out = torch.empty_like(dev)
    scratch = torch.empty((3, t, h * w), dtype=torch.int32, device="cuda")
    # `area > size_thresh` on integers: a fractional threshold compares like its floor
    C.check(C.load().bsub_filter_sparse_map_dev(_vp(dev), h * w, h, w, t, int(math.floor(size_thresh)), _vp(out), h * w, _vp(scratch),
                                                A._stream_ptr()))
    res = _mask_from_device(out, (h, w, t), sparse_array)
    if not A._is_torch(sparse_array):
        res = res.astype(np.asarray(sparse_array).dtype)                   # np.zeros_like(sparse_array)
    return res


# --------------------------------------------------------------------------------------------------------------
# computeSCube
# --------------------------------------------------------------------------------------------------------------
def gkern(l=10, sig=1.):
    """/root/reference/computeSCube.py:9-19 (host; only used to describe the smoothing kernel)."""
    ax = np.linspace(-(l - 1) / 2., (l - 1) / 2., l)
    xx, yy, zz = np.meshgrid(ax, ax, ax)
    kernel = np.exp(-0.5 * (np.square(xx) + np.square(yy) + np.square(zz)) / np.square(sig))
    return kernel / np.sum(kernel)


def _gauss_taps(l, sig=1.):
    ax = np.linspace(-(l - 1) / 2., (l - 1) / 2., l)
    g = np.exp(-0.5 * np.square(ax) / np.square(sig))
    return g / g.sum()


def computeSCube(sparse_xt, sparse_yt, return_device=False):
    """/root/reference/computeSCube.py:82-92: |xt| * |yt| in video order [t, h, w], normalised to unit sum, smoothed with the
    int(min(h, w) / 10)^3-tap Gaussian of gkern (sigma 1) under scipy's 'reflect' boundary.  The Gaussian is separable, so the
    device runs three 1-D passes (the dense convolution the reference calls is O(l^3) per voxel)."""
    torch = _torch()
    lib = C.load()

    def dev32(a):
        return a.to(torch.float32).contiguous() if A._is_torch(a) else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to("cuda")
    xt, yt = dev32(sparse_xt), dev32(sparse_yt)
    W, H, T = xt.shape
    if tuple(yt.shape) != (H, W, T):
        raise Exception("computeSCube: sparse_xt must be [w, h, t] and sparse_yt [h, w, t]")
    cube = torch.empty((T, H, W), dtype=torch.float32, device="cuda")
    tmp = torch.empty_like(cube)
    total = torch.zeros(1, dtype=torch.float64, device="cuda")
    scratch = torch.empty(2048, dtype=torch.float64, device="cuda")
    st = A._stream_ptr()
    C.check(lib.bsub_scube_product_dev(_vp(xt), _vp(yt), _vp(cube), T, H, W, _vp(total), _vp(scratch), st))
    l = int(min(H, W) / 10)
    if l < 1:
        raise Exception("computeSCube: frames smaller than 10 pixels have an empty smoothing kernel")
    taps = torch.from_numpy(_gauss_taps(l)[::-1].astype(np.float32).copy()).to("cuda")      # convolution flips the kernel
    shift = l // 2 if l % 2 else l // 2 - 1                # scipy.ndimage.convolve moves the origin of an even kernel
    a, b = cube, tmp
    for axis, (outer, length, inner) in enumerate(((T * H, W, 1), (T, H, W), (1, T, H * W))):
        C.check(lib.bsub_conv1d_reflect_dev(_vp(a), _vp(b), outer, length, inner, _vp(taps), l, shift, _vp(total) if axis == 0 else None, st))
        a, b = b, a
    torch.cuda.current_stream().synchronize()
    if return_device or A._is_torch(sparse_xt):
        return a
    return a.double().cpu().numpy()


# --------------------------------------------------------------------------------------------------------------
# run_motion_saliency_check
# --------------------------------------------------------------------------------------------------------------
def _contained_in(cc1, cc2):
    x2, y2, w2, h2 = cc2
    x1, y1, w1, h1 = cc1
    return bool(x2 < x1 and y2 < y1 and x1 + w1 < x2 + w2 and y1 + h1 < y2 + h2)


def _nested_relabel(stats):
    """unite_nestedCCs (/root/reference/utils.py:351-401) as the label map it applies: labels are 1-based rows of `stats`
    (OpenCV order); the edges of the spanning forest of the bbox-nesting graph relabel the ORIGINAL label n2 as n1."""
    k = stats.shape[0]
    remap = list(range(k + 1))
    if k < 2:
        return remap
    cc = [None] + [tuple(int(v) for v in stats[i, :4]) for i in range(k)]
    nested = [(l1, l2) for l1 in range(1, k + 1) for l2 in range(1, k + 1) if l1 != l2 and _contained_in(cc[l1], cc[l2])]
    if not nested:
        return remap
    import networkx as nx                                   # the reference's own dependency for this step (utils.py:385-391)
    graph = nx.Graph()
    for l1, l2 in nested:
        graph.add_edge(l2, l1)
    for n1, n2 in nx.minimum_spanning_tree(graph).edges():
        remap[n2] = n1
    return remap


def _saliency_groups(cc):
    """(frame, weight, area, [component slots]) of every nest-merged component, frames ascending, OpenCV label order inside a
    frame (compute_groups_per_frame, /root/reference/motion_saliency_check.py:19-49)."""
    groups = []
    for f in range(cc.shape[2]):
        stats, idx = cc.stats_cv2(f)
        if len(idx) == 0:
            continue
        remap = _nested_relabel(stats)
        members = {}
        for l in range(1, len(idx) + 1):
            members.setdefault(remap[l], []).append(idx[l - 1])
        for l in sorted(members):                          # np.unique(new_labels): ascending label
            slots = members[l]
            area = int(cc.area[slots].sum())
            groups.append((f, float(cc.wsum[slots].sum() / area), area, slots))
    return groups


def _filter_groups(groups, size_thresh):
    """/root/reference/motion_saliency_check.py:52-63."""
    w = np.array([g[1] for g in groups])
    thr = np.mean(w) + np.std(w)
    kept = [g for g in groups if g[1] > thr and g[2] > size_thresh]
    return kept, min([g[1] for g in kept])


def motion_saliency_blocks(data_shape, sparse_binary_mat, sparse_cube, delta=10):
    """Device form of run_motion_saliency_check: returns (labels uint8 [n][m] CUDA tensor, lam_ptr int32[n+1], lam float64[k+1]) --
    the block map bsub_set_blocks takes (api.group_sparse_decomposition(..., labels=...)) -- without building host masks."""
    torch = _torch()
    h, w, n = data_shape
    dev, shape = _mask_to_device(sparse_binary_mat)
    if tuple(shape) != (h, w, n):
        raise Exception("sparse_binary_mat must have the shape of the data cube")
    cube = sparse_cube.to(torch.float32).contiguous() if A._is_torch(sparse_cube) else \
        torch.from_numpy(np.ascontiguousarray(sparse_cube, dtype=np.float32)).to("cuda")
    if tuple(cube.shape) != (h, w, n):
        raise Exception("sparse_cube must be [h, w, t] like the data cube")
    cs = cube.stride()
    cc = Components(dev, shape, weight=(cube, (cs[2], cs[1], cs[0])))
    groups = _saliency_groups(cc)
    kept, min_w = _filter_groups(groups, (h * w) / 1500)
    norm = 1.0 / (delta * np.sqrt(max(h * w, n))) * min_w
    table = np.zeros(max(cc.total, 1), dtype=np.uint8)
    ptr = np.zeros(n + 1, dtype=np.int32)
    lam = []
    per_frame = [0] * n
    for f, wgt, _area, slots in kept:                      # already sorted by frame (stable, like the reference's sort)
        per_frame[f] += 1
        if per_frame[f] > 254:
            raise Exception("more than 254 blocks in frame %d" % f)
        table[slots] = per_frame[f]
        lam.append(norm / wgt)
    ptr[1:] = np.cumsum(per_frame)
    return cc.remap(table), ptr, np.asarray(lam + [0.0], dtype=np.float64)


def run_motion_saliency_check(data, sparse_binary_mat, sparse_cube, delta=10):
    """Drop-in for /root/reference/motion_saliency_check.py:66-120 -> (groups_by_frame, weights_by_frame): lists over the frames
    of boolean F-order pixel masks and of the lambda_i of every kept group."""
    h, w, n = data.shape
    labels, ptr, lam = motion_saliency_blocks((h, w, n), sparse_binary_mat, sparse_cube, delta)
    host = labels.cpu().numpy()                             # [n][m], pixel index already F-order (p = j*rows + i)
    groups_by_frame, weights_by_frame = [], []
    for f in range(n):
        k = int(ptr[f + 1] - ptr[f])
        groups_by_frame.append([host[f] == (b + 1) for b in range(k)])
        weights_by_frame.append([float(v) for v in lam[ptr[f]:ptr[f + 1]]])
    return groups_by_frame, weights_by_frame


# --------------------------------------------------------------------------------------------------------------
# morphology and the two-pass LSD of lsd_improvement.py
# --------------------------------------------------------------------------------------------------------------
def disk_radius(footprint_name, size):
    """get_footprint (/root/reference/lsd_improvement.py:307-320): disk(ceil(size) // 2)."""
    if footprint_name != 'disk':
        raise Exception("only the 'disk' footprint (the reference's default and only use) is implemented in this build")
    return int(math.ceil(size)) // 2


def apply_morph_ops(input, footprint_name='disk', percetage=0.05):
    """/root/reference/lsd_improvement.py:323-335 on a [h, w, t] boolean cube: dilation, then closing (dilation + erosion), by
    disk(ceil(percetage * h) // 2), frame by frame (the footprint has extent 1 along time)."""
    r = disk_radius(footprint_name, percetage * input.shape[0])
    dev, (h, w, t) = _mask_to_device(input)
    return _mask_from_device(morph_frames_dev(dev, h, w, r), (h, w, t), input)


def morph_frames_dev(mask_dev, rows, cols, radius):
    """The morphology of apply_morph_ops on a uint8 [nf][rows * cols] CUDA tensor (pixel p = j*rows + i, non-zero = set, nf >= 1):
    dilation, then closing (dilation + erosion), by disk(radius), frame by frame.  Returns a new uint8 [nf][rows * cols] tensor."""
    torch = _torch()
    nf, m = int(mask_dev.shape[0]), rows * cols
    lib = C.load()
    st = A._stream_ptr()
    b1, b2 = (torch.empty((nf, m), dtype=torch.uint8, device="cuda") for _ in range(2))
    scratch = torch.empty(nf * m + 2 * radius + 1, dtype=torch.uint8, device="cuda")
    for src, dst, erode in ((mask_dev, b1, 0), (b1, b2, 0), (b2, b1, 1)):      # dilation; closing = dilation, erosion
        C.check(lib.bsub_morph_disk_dev(_vp(src), src.stride(0), _vp(dst), m, rows, cols, nf, radius, erode, _vp(scratch), st))
    return b1


def merge_masks(masks, weights, background_marker=-1):
    """/root/reference/lsd_improvement.py:338-351."""
    if len(masks) != len(weights):
        raise Exception('length of weights and masks must be equal')
    merged = np.ones(masks[0].shape) * background_marker
    for i in range(len(masks) - 1, -1, -1):
        merged[np.asarray(masks[i], dtype=bool)] = weights[i]
    return merged


def calc_mask_percent(mask):
    return np.sum(mask > 0) / mask.size


def improved_LSD_weight_mask(D, original_shape, weights, delta=1.0, proximal_object=None, mode=None):
    """First pass of build_improved_LSD_graphs (/root/reference/lsd_improvement.py:369-404): a plain decomposition, its
    foreground mask, the disk morphology with the mask-percentage back-off, merged into the weight map (-1 = background)."""
    if proximal_object is None:
        L, S, iter_count, convergence = A.inexact_alm_rpca(D, delta=10.0)
    elif mode == "NONOVERLAPPING_GRAPHS":
        L, S, iter_count, convergence = A.inexact_alm_lsd(D, graphs=proximal_object, delta=delta, img_shape=original_shape[:2])
    elif mode == "NONOVERLAPPING_GROUPS":
        L, S, iter_count, convergence = A.inexact_alm_lsd(D, groups=proximal_object, delta=delta, img_shape=original_shape[:2])
    else:
        raise Exception("Unknown improved LSD mode")
    S_mask = A.foreground_mask(D, L, S, sigmas_from_mean=2).reshape(original_shape, order='F')

    def weight_for(disk_ratio):
        weight_mask = merge_masks((S_mask, apply_morph_ops(S_mask, percetage=disk_ratio)), weights)
        return weight_mask, int(np.sum(weight_mask > 0))
    return mask_backoff(weight_for, original_shape[0], S_mask.size), iter_count, convergence


def mask_backoff(weight_for, rows, total):
    """The mask-percentage back-off of build_improved_LSD_graphs (/root/reference/lsd_improvement.py:385-404): weight_for(disk_ratio)
    -> (weight map, number of its positive entries), total = number of entries of the whole map (rows = image height).  Shrinks the
    disk ratio by 0.01 from 0.05 while more than 20 % of the map is positive; returns the last weight map.  The decision rests on the
    count alone, so a sharded caller whose callable returns the all-reduced count takes the same steps on every rank."""
    disk_ratio, step = 0.05, 0.01
    total_allowed_iterations, current_iteration, max_mask_percent = 5, 1, 20
    weight_mask, count = weight_for(disk_ratio)
    mask_percent = count / total * 100
    # the reference's loop raises its own iteration allowance every pass (lsd_improvement.py:396-398), so it only ends when the
    # mask shrinks below the cap; a disk of radius 0 cannot shrink further, which bounds it here
    while mask_percent > max_mask_percent and current_iteration < total_allowed_iterations:
        disk_ratio -= step
        total_allowed_iterations += 1
        if disk_ratio * rows <= 0:
            break
        weight_mask, count = weight_for(disk_ratio)
        mask_percent = count / total * 100
    return weight_mask


def build_improved_LSD_graphs(D, original_shape, weights, delta=1.0, proximal_object=None, mode=None):
    """Drop-in for /root/reference/lsd_improvement.py:369-438 -> (graphs, background_masks, iter_count, convergence)."""
    weight_mask, iter_count, convergence = improved_LSD_weight_mask(D, original_shape, weights, delta, proximal_object, mode)
    graphs = [A.get_proximal_graph_group_centers(weight_mask[:, :, i].shape, 1, group_centers=weight_mask[:, :, i])
              for i in range(weight_mask.shape[-1])]
    background_masks = [(weight_mask[:, :, i] < 0).flatten(order='F') for i in range(weight_mask.shape[-1])]
    return graphs, background_masks, iter_count, convergence


def LSD_improved(ImData0, frame_start=0, frame_end=47, downsample_ratio=1, delta=1, alg_ver=2):
    """Drop-in for /root/reference/lsd_improvement.py:441-487 -> (S, S_mask, L_recon, ImData1, ImMean, shape, iterations,
    converged, graph_iter, graph_converged).  The per-frame graphs are never materialised: the weight map of the first pass goes
    to the solver as the per-pixel window weights (bsub_set_center_windows)."""
    if downsample_ratio == 1:
        ImData1 = ImData0
    else:
        ImData1 = resize_with_cv2(ImData0[:, :, frame_start:(frame_end + 1)], 1 / downsample_ratio)
    A.normalizeImage(ImData1)
    ImMean = np.mean(ImData1)
    ImData2 = ImData1 - ImMean
    shape = ImData2.shape
    h, w, frames = shape
    D = ImData2.reshape((h * w, frames), order='F')
    weights = (1, 1.5)
    if alg_ver == 2:
        proximal_object, mode = A.get_proximal_flat_groups_nonoverlap((h, w), A.BLOCK_SIZE), "NONOVERLAPPING_GROUPS"
    elif alg_ver == 1:
        proximal_object, mode = None, None
    else:
        raise Exception("LSD_improved wrong alg ver")
    weight_mask, graph_iter, graph_converged = improved_LSD_weight_mask(D, shape, weights, delta=1.0, proximal_object=proximal_object,
                                                                        mode=mode)
    dec = A.center_window_decomposition(D, weight_mask, img_shape=(h, w))
    L, S, iterations, converged = A._finish(dec, D, False)
    S_mask = dec.mask(2).reshape(shape, order='F')
    return (S, S_mask, L.reshape(shape, order='F'), ImData1, ImMean, shape, iterations, converged, graph_iter, graph_converged)


# --------------------------------------------------------------------------------------------------------------
# stage 2: saliency RPCA over the X-T and Y-T slices (computeRPCADecomposition.py)
# --------------------------------------------------------------------------------------------------------------
def inexact_alm_rpca_batch(slices, delta=1.0, max_rank=1, tol=1e-7, tol_l1=0.0, max_iter=500, rho=1.2, return_info=False):
    """inexact_alm_rpca (/root/reference/lsd_improvement.py:123-196) on every slices[i, :, :] at once, the rank of L capped at
    max_rank = 1: one thread-block cluster per slice (csrc/rpca_batch.cu), its state resident in shared memory when the slice fits a
    cluster of 8 CTAs (at most 640 columns), otherwise iterated in global memory (any slice up to 4096 x 4096).  -> (L, S) like the
    input ([slices, rows, cols]); with return_info also the per-slice iteration counts (negative: not converged), errors, ranks."""
    if max_rank != 1:
        raise Exception("inexact_alm_rpca_batch: the batched kernel caps the rank at 1 (use inexact_alm_rpca for a free rank)")
    torch = _torch()
    on_dev = A._is_torch(slices)
    M = slices.to(torch.float32).contiguous() if on_dev else torch.from_numpy(np.ascontiguousarray(slices, dtype=np.float32)).to("cuda")
    if M.dim() != 3:
        raise Exception("inexact_alm_rpca_batch: slices must be [batch, rows, cols]")
    batch, rows, cols = (int(v) for v in M.shape)
    L, S = torch.empty_like(M), torch.empty_like(M)
    iters = torch.empty(batch, dtype=torch.int32, device="cuda")
    rank = torch.empty(batch, dtype=torch.int32, device="cuda")
    err = torch.empty(batch, dtype=torch.float32, device="cuda")
    C.check(C.load().bsub_rpca_rank1_batch_dev(_vp(M), batch, rows, cols, float(delta), float(rho), float(tol), float(tol_l1), int(max_iter),
                                               _vp(L), _vp(S), _vp(iters), _vp(err), _vp(rank), A._stream_ptr()))
    torch.cuda.current_stream().synchronize()
    if not on_dev:
        L, S = L.double().cpu().numpy(), S.double().cpu().numpy()
    if return_info:
        return L, S, {"iters": iters.cpu().numpy(), "err": err.cpu().numpy(), "rank": rank.cpu().numpy()}
    return L, S


def compute_RPCA(image_array, grayscale=True, max_error=None, max_iter=200000, return_info=False):
    """Drop-in for /root/reference/computeRPCADecomposition.py:12-48 (grayscale branch) -> (L_array, S_array): a max_rank = 1
    robust PCA of every image_array[i, :, :].  The reference hands each slice to RobustPCA(max_rank=1, tol=max_error) -- a package
    that is not vendored, pinned or installable (parity unpinned there); here every slice goes through the reference's own
    inexact_alm_rpca iteration with the rank capped at 1, stopped by the same residual test sum|M - L - S| <= max_error (or the
    iteration's own 1e-7 relative tolerance, whichever comes first; 500 iterations at most, like inexact_alm_rpca).
    return_info=True appends inexact_alm_rpca_batch's info dict (per-slice iters, negative where the cap was hit; err; rank)."""
    if not grayscale:
        raise Exception("compute_RPCA: only the grayscale work mode (the reference's default) is implemented in this build")
    if max_error is None:
        max_error = image_array.shape[1] * image_array.shape[2] * 0.0001
    return inexact_alm_rpca_batch(image_array, delta=1.0, tol_l1=float(max_error), max_iter=min(int(max_iter), 500),
                                  return_info=return_info)


def executeSaliencyRPCA(ImData, downsample_ratio, grayscale_workmode=True, grayscale_input=True):
    """Drop-in for /root/reference/computeRPCADecomposition.py:52-95 -> (xt_lowrank, xt_sparse, yt_lowrank, yt_sparse): the video
    [t, h, w] cut into X-T planes ([w, h, t]) and Y-T planes ([h, w, t]), each resized by 1/downsample_ratio over its first two
    axes (resize_with_cv2) and decomposed slice by slice.  Frames up to 4096 x 4096 pixels and clips up to 4096 frames; the X-T and
    Y-T stacks may take different kernels (inexact_alm_rpca_batch), with no effect on the result beyond float32 rounding."""
    if not (grayscale_workmode and grayscale_input):
        raise Exception("executeSaliencyRPCA: only the grayscale mode is implemented in this build")
    torch = _torch()
    v = ImData.to(torch.float32) if A._is_torch(ImData) else torch.from_numpy(np.ascontiguousarray(ImData, dtype=np.float32)).to("cuda")
    xt = v.permute(2, 1, 0).contiguous()
    yt = v.permute(1, 2, 0).contiguous()
    if downsample_ratio != 1:
        xt = resize_with_cv2(xt, 1 / downsample_ratio)
        yt = resize_with_cv2(yt, 1 / downsample_ratio)
    xt_l, xt_s = compute_RPCA(xt, True, xt.shape[1] * xt.shape[2] * 0.0001)
    yt_l, yt_s = compute_RPCA(yt, True, yt.shape[1] * yt.shape[2] * 0.0001)
    if A._is_torch(ImData):
        return xt_l, xt_s, yt_l, yt_s
    return tuple(x.double().cpu().numpy() for x in (xt_l, xt_s, yt_l, yt_s))
