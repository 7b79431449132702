"""background-subtraction_b200 -- B200-native (sm_100a) implementation of the inexact-ALM low-rank + structured-sparse
decomposition of yakovdan/Background-Subtraction (the LSD / group-sparse RPCA hot path), behind the reference's own
Python call surface.  All numerics run in libbsub_b200.so (hand-written CUDA) through the C ABI of
include/bsub_b200.h; there is no CPU fallback."""
from .api import (BLOCK_SIZE, Decomposition, center_window_decomposition, LSD, apply_background_shrinkage_operator, block_shrinkage_operator,
                  center_window_csc, detect_center_windows, detect_flat_tiling, detect_window_graph,
                  eig_topk, foreground_mask, getGraphSPAMS_all_groups, get_proximal_flat_groups_nonoverlap,
                  get_proximal_graph_group_centers, gram,
                  group_sparse_decomposition, inexact_alm_group_sparse_RPCA, inexact_alm_lsd,
                  inexact_alm_lsd_batch, inexact_alm_lsd_with_background, inexact_alm_rpca,
                  labels_from_blocks, lsd_decomposition, make_config, normalizeImage, pack_graphs, prox, prox_by_frame, prox_flat,
                  resize_with_cv2, svd_k_largest, window_csc, with_background_decomposition)
from .flow import (LSD_improved, apply_morph_ops, compute_RPCA, executeSaliencyRPCA, inexact_alm_rpca_batch, build_improved_LSD_graphs, calc_mask_percent, computeSCube, connected_components,
                   filter_sparse_map, gkern, improved_LSD_weight_mask, merge_masks, motion_saliency_blocks,
                   resize_with_cv2_by_first_axis, run_motion_saliency_check)
from . import _cabi, api, build, flow  # noqa: F401

__all__ = [n for n in dir() if not n.startswith("_")]
