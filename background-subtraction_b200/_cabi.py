"""ctypes binding of libbsub_b200.so (include/bsub_b200.h).  There is no CPU fallback: if the library is missing it
is built with nvcc (build.py); if that fails, or a compute call is made without a CUDA device, the call raises."""
import ctypes
import os

from . import build as _build

c_double_p = ctypes.POINTER(ctypes.c_double)
c_float_p = ctypes.POINTER(ctypes.c_float)
c_int32_p = ctypes.POINTER(ctypes.c_int32)
c_int64_p = ctypes.POINTER(ctypes.c_int64)
c_uint8_p = ctypes.POINTER(ctypes.c_uint8)
vp = ctypes.c_void_p


class Config(ctypes.Structure):
    _fields_ = [("m", ctypes.c_int64), ("m_global", ctypes.c_int64), ("n", ctypes.c_int32), ("rows", ctypes.c_int32),
                ("cols", ctypes.c_int32), ("prox", ctypes.c_int32), ("group_rows", ctypes.c_int32),
                ("group_cols", ctypes.c_int32), ("delta", ctypes.c_double), ("mu_scale", ctypes.c_double),
                ("rho", ctypes.c_double), ("tol", ctypes.c_double), ("max_iter", ctypes.c_int32), ("sv0", ctypes.c_int32),
                ("use_sv_prediction", ctypes.c_int32), ("break_on_rank0", ctypes.c_int32),
                ("non_block_lambda_scale", ctypes.c_double), ("d_global", ctypes.c_int32),
                ("graph_max_sweeps", ctypes.c_int32), ("graph_tol", ctypes.c_double), ("tile_rows", ctypes.c_int32),
                ("cluster_frames", ctypes.c_int32), ("flags", ctypes.c_int32), ("reserved", ctypes.c_int32 * 5)]


class Status(ctypes.Structure):
    _fields_ = [("iter", ctypes.c_int32), ("converged", ctypes.c_int32), ("done", ctypes.c_int32), ("svp", ctypes.c_int32),
                ("err", ctypes.c_double), ("mu", ctypes.c_double), ("norm_two", ctypes.c_double), ("norm_fro", ctypes.c_double),
                ("norm_rowsum", ctypes.c_double), ("lambda_", ctypes.c_double)]


class IterLog(ctypes.Structure):
    _fields_ = [("iter", ctypes.c_int32), ("svp", ctypes.c_int32), ("sv", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("err", ctypes.c_double), ("mu", ctypes.c_double), ("nnz", ctypes.c_uint64)]


PROX_FLAT_LINF, PROX_GRAPH_LINF, PROX_BLOCK_L2, PROX_L1, PROX_GRAPH_CENTER_BG, PROX_GRAPH_GENERIC = 0, 1, 2, 3, 4, 5
FLAG_ALWAYS_STORE_S = 1

# every symbol include/bsub_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "bsub_last_error": (ctypes.c_char_p, []),
    "bsub_version": (ctypes.c_int, []),
    "bsub_default_config": (None, [ctypes.POINTER(Config)]),
    "bsub_abi_sizes": (None, [c_int32_p]),
    "bsub_create": (ctypes.c_int, [ctypes.POINTER(Config), ctypes.POINTER(vp)]),
    "bsub_destroy": (ctypes.c_int, [vp]),
    "bsub_set_flat_groups": (ctypes.c_int, [vp, c_int32_p]),
    "bsub_set_graph_windows": (ctypes.c_int, [vp, c_double_p, ctypes.c_int64]),
    "bsub_set_blocks": (ctypes.c_int, [vp, c_uint8_p, c_int32_p, c_double_p]),
    "bsub_set_center_windows": (ctypes.c_int, [vp, c_float_p, c_uint8_p]),
    "bsub_set_graphs": (ctypes.c_int, [vp, ctypes.c_int32, c_int32_p, c_int64_p, ctypes.POINTER(c_int32_p), ctypes.POINTER(c_int32_p),
                                       ctypes.POINTER(c_double_p), c_uint8_p]),
    "bsub_load_D_f64_host": (ctypes.c_int, [vp, vp, ctypes.c_int64, vp]),
    "bsub_load_D_f32_host": (ctypes.c_int, [vp, vp, ctypes.c_int64, vp]),
    "bsub_load_D_f32_dev": (ctypes.c_int, [vp, vp, ctypes.c_int64, vp]),
    "bsub_load_u8_host": (ctypes.c_int, [vp, vp, c_double_p, c_double_p, c_double_p, ctypes.c_int, vp]),
    "bsub_run": (ctypes.c_int, [vp, vp]),
    "bsub_set_always_store_S": (ctypes.c_int, [vp, ctypes.c_int]),
    "bsub_comm_buffers": (ctypes.c_int, [vp, ctypes.POINTER(vp), c_int64_p, ctypes.POINTER(vp), c_int64_p]),
    "bsub_step_init_local": (ctypes.c_int, [vp, vp]),
    "bsub_step_init_finish": (ctypes.c_int, [vp, vp]),
    "bsub_step_gram": (ctypes.c_int, [vp, vp]),
    "bsub_step_solve": (ctypes.c_int, [vp, vp]),
    "bsub_step_project": (ctypes.c_int, [vp, vp]),
    "bsub_step_shrink": (ctypes.c_int, [vp, vp]),
    "bsub_step_finish_iter": (ctypes.c_int, [vp, vp]),
    "bsub_step_shrink_a": (ctypes.c_int, [vp, vp]),
    "bsub_step_shrink_b": (ctypes.c_int, [vp, vp]),
    "bsub_block_sums_buffer": (ctypes.c_int, [vp, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_int64)]),
    "bsub_step_prox_buffers": (ctypes.c_int, [vp, ctypes.POINTER(vp), ctypes.POINTER(vp), c_int64_p]),
    "bsub_set_frame_windows": (ctypes.c_int, [vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, c_double_p, ctypes.c_int64]),
    "bsub_set_frame_center_windows": (ctypes.c_int, [vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, c_float_p, c_uint8_p]),
    "bsub_set_frame_weight_map_dev": (ctypes.c_int, [vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, vp, ctypes.c_int64,
                                                     vp]),
    "bsub_set_frame_graphs": (ctypes.c_int, [vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, c_int32_p,
                                             c_int64_p, ctypes.POINTER(c_int32_p), ctypes.POINTER(c_int32_p), ctypes.POINTER(c_double_p),
                                             c_uint8_p]),
    "bsub_step_prox_block": (ctypes.c_int, [vp, vp, vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, vp]),
    "bsub_poll": (ctypes.c_int, [vp, ctypes.POINTER(Status)]),
    "bsub_sync_status": (ctypes.c_int, [vp, ctypes.POINTER(Status), vp]),
    "bsub_finalize": (ctypes.c_int, [vp, vp]),
    "bsub_get_L_f32_dev": (ctypes.c_int, [vp, ctypes.POINTER(vp), c_int64_p]),
    "bsub_get_S_f32_dev": (ctypes.c_int, [vp, ctypes.POINTER(vp), c_int64_p]),
    "bsub_get_D_f32_dev": (ctypes.c_int, [vp, ctypes.POINTER(vp), c_int64_p]),
    "bsub_get_Y_f32_dev": (ctypes.c_int, [vp, ctypes.POINTER(vp), c_int64_p]),
    "bsub_download_f64": (ctypes.c_int, [vp, ctypes.c_int, vp, ctypes.c_int64, vp]),
    "bsub_download_f32": (ctypes.c_int, [vp, ctypes.c_int, vp, ctypes.c_int64, vp]),
    "bsub_debug_eig_cycles": (ctypes.c_int, [vp, c_int64_p]),
    "bsub_debug_info": (ctypes.c_int, [vp, c_int32_p]),
    "bsub_debug_counters": (ctypes.c_int, [vp, c_int64_p]),
    "bsub_debug_graph": (ctypes.c_int, [vp, c_int64_p]),
    "bsub_get_log": (ctypes.c_int, [vp, ctypes.POINTER(IterLog), ctypes.c_int32, c_int32_p]),
    "bsub_mask_stats_local": (ctypes.c_int, [vp, ctypes.c_int, vp]),
    "bsub_mask_host": (ctypes.c_int, [vp, ctypes.c_double, vp, vp]),
    "bsub_mask_dev": (ctypes.c_int, [vp, ctypes.c_double, vp, vp]),
    "bsub_foreground_mask_dev": (ctypes.c_int, [vp, vp, vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_double, vp, vp]),
    "bsub_prox_flat3_dev": (ctypes.c_int, [vp, vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_double, vp]),
    "bsub_prox_flat_groups_dev": (ctypes.c_int, [vp, vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, c_int32_p, ctypes.c_double, vp]),
    "bsub_prox_graph3_dev": (ctypes.c_int, [vp, vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_double,
                                            c_double_p, ctypes.c_int32, ctypes.c_double, c_int32_p, vp]),
    "bsub_prox_center3_dev": (ctypes.c_int, [vp, vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_double,
                              c_float_p, ctypes.c_int32, ctypes.c_double, c_int32_p, vp]),
    "bsub_prox_graph_dev": (ctypes.c_int, [vp, vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_double, ctypes.c_int32, c_int32_p,
                                           c_int64_p, ctypes.POINTER(c_int32_p), ctypes.POINTER(c_int32_p), ctypes.POINTER(c_double_p),
                                           ctypes.c_int32, ctypes.c_double, c_int32_p, vp]),
    "bsub_block_shrink_dev": (ctypes.c_int, [vp, vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, c_uint8_p, c_int32_p, c_double_p,
                                             ctypes.c_double, ctypes.c_double, vp]),
    "bsub_gram_dev": (ctypes.c_int, [vp, vp, vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_double, c_double_p, vp]),
    "bsub_eig_topk": (ctypes.c_int, [c_double_p, ctypes.c_int32, ctypes.c_int32, c_double_p, c_double_p]),
    "bsub_gram_i8_test": (ctypes.c_int, [vp, ctypes.c_int32, ctypes.c_int64, vp]),
    "bsub_gram_i8_bench": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int64, ctypes.c_int32, vp]),
    "bsub_resize_dev": (ctypes.c_int, [vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                       vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, vp]),
    "bsub_cc_label_dev": (ctypes.c_int, [vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, vp, ctypes.c_int64, vp, vp, vp]),
    "bsub_cc_stats_dev": (ctypes.c_int, [vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, vp, ctypes.c_int32, vp,
                                         ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, vp, vp, vp, vp]),
    "bsub_cc_remap_dev": (ctypes.c_int, [vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, vp, vp, vp, ctypes.c_int64, vp]),
    "bsub_filter_sparse_map_dev": (ctypes.c_int, [vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, vp,
                                                  ctypes.c_int64, vp, vp]),
    "bsub_scube_product_dev": (ctypes.c_int, [vp, vp, vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, vp, vp, vp]),
    "bsub_conv1d_reflect_dev": (ctypes.c_int, [vp, vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int64, vp, ctypes.c_int32, ctypes.c_int32, vp, vp]),
    "bsub_rpca_rank1_batch_dev": (ctypes.c_int, [vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_double, ctypes.c_double,
                                                 ctypes.c_double, ctypes.c_double, ctypes.c_int32, vp, vp, vp, vp, vp, vp]),
    "bsub_morph_disk_dev": (ctypes.c_int, [vp, ctypes.c_int64, vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                           ctypes.c_int32, vp, vp]),
}

_lib = None


def lib_path():
    return _build.LIB


def load():
    """Load (building if necessary) the CUDA library.  Raises if it cannot be produced -- never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if not os.path.exists(path):
        path = _build.build()
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().bsub_last_error()
        raise Exception(msg.decode() if msg else "bsub_b200: error %d" % rc)
