/*
 * bsub_b200.h -- C ABI of libbsub_b200.so: the B200 (sm_100a) implementation of the reference's inexact-ALM
 * low-rank + structured-sparse decomposition (yakovdan/Background-Subtraction).
 *
 * The reference has no native plugin/FFI interface (it is pure Python, SURVEY.md section 2a); its boundary for
 * this path is the Python call surface.  Each entry point below names the reference interface it replaces
 * (file:line under /root/reference).  A binding only needs plain pointers and sizes (ctypes / cffi / cgo style);
 * no torch or CUDA types appear in the signatures -- streams are passed as void* (cudaStream_t, 0 = default).
 *
 * Matrix convention: the reference's pixels x frames matrix in Fortran order (inexact_alm_lsd.py:84-88,225) is
 * byte-for-byte a row-major [n_frames][m_pixels] array; every matrix pointer below uses that layout with a row
 * pitch `ld` (elements) >= m.  Pixel index p = j*rows + i for image row i, column j (utils.py:230-231).
 *
 * All functions return 0 on success and a non-zero status on failure; bsub_last_error() then returns a message
 * (the host-side mirror turns it into the reference's error convention, `raise Exception(msg)`).
 */
#ifndef BSUB_B200_H
#define BSUB_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bsub_solver bsub_solver;   /* opaque */

/* proximal operator of the S-step */
enum {
    BSUB_PROX_FLAT_LINF = 0,   /* spams.proximalFlat 'group-lasso-linf'      inexact_alm_lsd.py:71-79,153-155 */
    BSUB_PROX_GRAPH_LINF = 1,  /* spams.proximalGraph 'graph' (overlapping)   inexact_alm_lsd.py:49-57,159     */
    BSUB_PROX_BLOCK_L2 = 2,    /* block_shrinkage_operator                    group_sparse_RPCA.py:13-42       */
    BSUB_PROX_L1 = 3,          /* elementwise soft threshold                  lsd_improvement.py:176           */
    BSUB_PROX_GRAPH_CENTER_BG = 4, /* per-frame windows centred on weighted pixels (prox_by_frame, inexact_alm_lsd.py:60-68,
                                  graphs of lsd_improvement.py:74-120) + l2 shrink of each frame's background
                                  (lsd_improvement.py:199-212): inexact_alm_lsd_with_background, lsd_improvement.py:215-304 */
    BSUB_PROX_GRAPH_GENERIC = 5   /* spams.proximalGraph 'graph' for ANY non-nested graph, one graph per frame (bsub_set_graphs),
                                     optionally + the l2 shrink of each frame's background: every graph the reference accepts in
                                     inexact_alm_lsd / prox_by_frame / inexact_alm_lsd_with_background */
};

/* Replaces the hard-coded constants of inexact_alm_lsd.py:102-125 / group_sparse_RPCA.py:53-77. */
typedef struct {
    int64_t m;                 /* pixels held by THIS solver (a pixel-row shard in multi-GPU runs)            */
    int64_t m_global;          /* pixels of the whole matrix (lambda = 1/(sqrt(max(m_global,n))*delta)); 0 = m */
    int32_t n;                 /* frames                                                                       */
    int32_t rows, cols;        /* image geometry of this solver's pixels, rows*cols == m (0,0 if not an image) */
    int32_t prox;              /* BSUB_PROX_*                                                                  */
    int32_t group_rows, group_cols; /* tile / window shape; only 3x3 (the reference's BLOCK_SIZE) is fused      */
    double delta;              /* 10                                                                           */
    double mu_scale;           /* 12.5 (inexact_alm_lsd.py:114) or 1.25 (group_sparse_RPCA.py:67)              */
    double rho;                /* 1.6                                                                          */
    double tol;                /* 1e-7                                                                         */
    int32_t max_iter;          /* 500                                                                          */
    int32_t sv0;               /* 10                                                                           */
    int32_t use_sv_prediction; /* 1                                                                            */
    int32_t break_on_rank0;    /* 1 for group_sparse_RPCA.py:91-93                                             */
    double non_block_lambda_scale; /* 100 (group_sparse_RPCA.py:57)                                            */
    int32_t d_global;          /* min(m_global, n) used by the sv predictor; 0 = derive                        */
    int32_t graph_max_sweeps;  /* overlapping prox: BCD sweep cap per ALM iteration (0 = default 4000)         */
    double graph_tol;          /* overlapping prox: stop when the largest dual change of a sweep <= tol*lambda/mu (0 = 1e-6) */
    int32_t tile_rows;         /* tuning: rows per shrink tile (0 = default)                                   */
    int32_t cluster_frames;    /* tuning: CTAs per cluster splitting the frames (0 = default)                  */
    int32_t flags;             /* BSUB_FLAG_*                                                                  */
    int32_t reserved[5];
} bsub_config;

/* bsub_config.flags */
enum {
    BSUB_FLAG_ALWAYS_STORE_S = 1   /* store S in every iteration (default: only when the iteration may be the last; S is rebuilt
                                      from D, Y and the digit planes of W otherwise).  Set by drivers that use the step interface. */
};

typedef struct {
    int32_t iter;              /* reference iter_out                                                            */
    int32_t converged;         /* reference `converged`                                                         */
    int32_t done;              /* 0 running, 1 converged, 2 max_iter, 3 rank-0 break, 4 zero input              */
    int32_t svp;               /* rank of L                                                                     */
    double err;                /* ||Z||_F / ||D||_F of the last completed iteration                             */
    double mu;                 /* mu after the last update                                                      */
    double norm_two, norm_fro, norm_rowsum, lambda;
} bsub_status;

typedef struct {
    int32_t iter, svp, sv, reserved;
    double err, mu;
    uint64_t nnz;              /* ||S||_0 (the reference prints it every iteration, inexact_alm_lsd.py:170)      */
} bsub_iter_log;

const char* bsub_last_error(void);
int bsub_version(void);
void bsub_default_config(bsub_config* cfg);
/* sizeof(bsub_config), sizeof(bsub_status), sizeof(bsub_iter_log): lets a binding verify its struct layouts */
void bsub_abi_sizes(int32_t out3[3]);

/* ---- solver life cycle ------------------------------------------------------------------------------------
 * Threading / devices: a handle lives on the CUDA device that is current when bsub_create runs; call its entry points
 * from threads whose current device is that one (one process per GPU is the intended model: kernel attributes are set
 * once per process).  Different handles may be driven concurrently from different host threads on different streams
 * (error text is thread-local); one handle must not be used from two threads at once. */
int bsub_create(const bsub_config* cfg, bsub_solver** out);
int bsub_destroy(bsub_solver* s);

/* group / graph / block descriptions: the hot-path *types* of SURVEY.md 8a (a8-a11).
 * flat: int32[m] 1-based ids from get_proximal_flat_groups_nonoverlap (lsd_improvement.py:14-34); a regular 3x3
 *       tiling of the rows x cols image is recognised and fused, anything else takes the generic two-phase path. */
int bsub_set_flat_groups(bsub_solver* s, const int32_t* groups_host);
/* graph: overlapping windows of getGraphSPAMS_all_groups (inexact_alm_lsd.py:13-46); eta_host double[n_eta] one weight per window
 * (finite, >= 0), or NULL (all 1) */
int bsub_set_graph_windows(bsub_solver* s, const double* eta_host, int64_t n_eta);
/* blocks: blocks_by_frame / lambdas_by_frame of group_sparse_RPCA.py:45 as a label map uint8[n][m] (0 = complement,
 *       b = block b of that frame) plus the CSR (lam_ptr[n+1], lam) of the per-frame lambda lists. */
int bsub_set_blocks(bsub_solver* s, const uint8_t* labels_host, const int32_t* lam_ptr, const double* lam);
/* per-frame centre windows + background (BSUB_PROX_GRAPH_CENTER_BG): eta_host float32[n][m] = weight of the 3x3 window
 * centred on that pixel in that frame (finite; <= 0: no window; get_proximal_graph_group_centers, lsd_improvement.py:74-120),
 * background_host uint8[n][m] != 0 where the pixel belongs to the frame's background mask (lsd_improvement.py:434). */
int bsub_set_center_windows(bsub_solver* s, const float* eta_host, const uint8_t* background_host);
/* any graphs (BSUB_PROX_GRAPH_GENERIC): n_graphs SPAMS-style CSC groups_var matrices as the reference builds them -- graph k has
 * n_groups[k] groups, group g of it holds the pixels indices[k][indptr[k][g] .. indptr[k][g+1]) (0-based, < m, no pixel twice) and
 * weighs eta[k][g] (finite, >= 0); frame f uses graph frame_graph[f] (NULL: all frames use graph 0, n_graphs must be 1).
 * background_host uint8[n][m] (may be NULL): != 0 marks the frame's background pixels, which get the l2 shrink at
 * 100 lambda / mu after the prox (inexact_alm_lsd_with_background).  The library colours the graphs itself; the arrays are
 * copied, and every entry is validated before anything reaches the device. */
int bsub_set_graphs(bsub_solver* s, int32_t n_graphs, const int32_t* frame_graph, const int64_t* n_groups, const int32_t* const* indptr,
                    const int32_t* const* indices, const double* const* eta, const uint8_t* background_host);

/* ---- data in ---------------------------------------------------------------------------------------------- */
int bsub_load_D_f64_host(bsub_solver* s, const double* D, int64_t ld, void* stream);      /* host float64 (NumPy)   */
int bsub_load_D_f32_host(bsub_solver* s, const float* D, int64_t ld, void* stream);       /* host float32 (pinned)  */
int bsub_load_D_f32_dev(bsub_solver* s, const float* D, int64_t ld, void* stream);        /* device float32         */
/* LSD() pre-processing on the device (inexact_alm_lsd.py:211-225): uint8 cube [n][m] -> normalise to [0,1] over the
 * whole cube, subtract the global mean.  lo/hi/mean in raw units are returned (and may be forced by the caller for
 * sharded runs when force != 0). */
int bsub_load_u8_host(bsub_solver* s, const uint8_t* frames, double* lo, double* hi, double* mean_raw, int force, void* stream);

/* ---- whole solve on one GPU: inexact_alm_lsd.py:82-179 / group_sparse_RPCA.py:45-126 ------------------------ */
int bsub_run(bsub_solver* s, void* stream);

/* ---- step interface for pixel-sharded multi-GPU runs (the caller all-reduces between the steps) -------------- */
int bsub_comm_buffers(bsub_solver* s, double** sum_buf, int64_t* sum_count, double** max_buf, int64_t* max_count);
/* step drivers: a status with done == 5 means "a digit pass clipped while S was not being stored" -- switch this on and solve again
 * (bsub_run does that by itself) */
int bsub_set_always_store_S(bsub_solver* s, int on);
int bsub_step_init_local(bsub_solver* s, void* stream);    /* Gram(D) partial + row-sum max partial                */
int bsub_step_init_finish(bsub_solver* s, void* stream);   /* ||D||_2, mu0, Y0, S0                                  */
int bsub_step_gram(bsub_solver* s, void* stream);          /* partial Gram of W into sum_buf                        */
int bsub_step_solve(bsub_solver* s, void* stream);         /* eigensolve + rank logic                               */
int bsub_step_project(bsub_solver* s, void* stream);       /* optional: T = Vr^T W from the digit planes (else part of _shrink) */
int bsub_step_shrink(bsub_solver* s, void* stream);        /* fused pass B; leaves sum Z^2 etc. in the sum_buf tail  */
int bsub_step_finish_iter(bsub_solver* s, void* stream);   /* err, mu update, stop flags                            */
/* l2-block mode (group_sparse_RPCA.py:13-42) on pixel shards: a block -- and the frame-wide complement group, :37-40 -- spans the
 * shards, so its shrink factor needs the sum of squares over ALL of them.  _shrink_a leaves the local sums in the buffer
 * bsub_block_sums_buffer returns (double [n][labels], device memory), the driver all-reduces it (SUM), _shrink_b applies the
 * factors and finishes the pass.  For the other prox modes _shrink_a is the whole pass, _shrink_b does nothing and the buffer is NULL. */
int bsub_step_shrink_a(bsub_solver* s, void* stream);
int bsub_step_shrink_b(bsub_solver* s, void* stream);
int bsub_block_sums_buffer(bsub_solver* s, double** sums, int64_t* count);
/* Graph modes on pixel shards: the prox of a frame needs the whole image but no other frame, so between the two halves of the pass
 * the driver re-shards G_S by FRAMES (all-to-all), runs the prox of its frames and brings S back:
 *   _shrink_a (G_S of this pixel shard into the buffer _prox_buffers returns) -> exchange -> bsub_step_prox_block on whole frames
 *   (device pointers, lambda/mu and the stop flag from this handle's device state) -> exchange (result into the S pointer of
 *   _prox_buffers) -> _shrink_b.
 * The handle holds a frame-range description (bsub_set_frame_*, below).  _shrink_a then stops before the prox in every graph mode, as
 * it always does in BSUB_PROX_GRAPH_LINF, and _shrink_b finishes the pass.  The l1 mode (BSUB_PROX_L1) is elementwise and shards
 * with bsub_step_shrink alone. */
int bsub_step_prox_buffers(bsub_solver* s, float** G_S, float** S, int64_t* ld);
/* Frame-range descriptions: the prox of whole rows x cols frames [f0, f0 + nf) of the clip (the frames this rank owns after the
 * exchange; nf may be 0).  Only those frames' data is copied, and every entry is validated before anything reaches the device.  A
 * handle holds one graph description: each bsub_set_frame_* or whole-clip setter (bsub_set_graph_windows / _center_windows /
 * _graphs, which describe frames [0, n) of the handle's own pixels) replaces the previous one.  A handle whose description is a
 * frame range has no graph for its own pixels: bsub_run and bsub_step_shrink refuse it.
 *   _windows (BSUB_PROX_GRAPH_LINF): the 3x3 all-window graph, eta double[n_eta] one weight per window as bsub_set_graph_windows
 *     takes it (finite, >= 0), the same in every frame; NULL: unit weights.
 *   _center_windows (BSUB_PROX_GRAPH_CENTER_BG): eta float32[nf][rows*cols] and background uint8[nf][rows*cols] as
 *     bsub_set_center_windows takes them for frames f0 .. f0 + nf - 1.
 *   _graphs (BSUB_PROX_GRAPH_GENERIC): graphs as bsub_set_graphs takes them (indices < rows*cols), frame_graph[nf] for frames
 *     f0 .. f0 + nf - 1, background uint8[nf][rows*cols] or NULL. */
int bsub_set_frame_windows(bsub_solver* s, int32_t rows, int32_t cols, int32_t f0, int32_t nf, const double* eta_host, int64_t n_eta);
int bsub_set_frame_center_windows(bsub_solver* s, int32_t rows, int32_t cols, int32_t f0, int32_t nf, const float* eta_host,
                                  const uint8_t* background_host);
/* _center_windows from a weight map already on the device (BSUB_PROX_GRAPH_CENTER_BG): weight float32 [nf][ld] (device memory, row
 * pitch ld >= rows*cols), row f = frame f0 + f, pixel p = j*rows + i -- LSD_improved's merged map of those frames.  An entry > 0 is
 * the weight of the centre window at that pixel, < 0 marks a background pixel, 0 is neither: the same description
 * bsub_set_frame_center_windows builds from eta = max(weight, 0) and background = (weight < 0).  A kernel on `stream` writes it into
 * new device buffers; the call then waits for the stream and, if an entry is not finite, reports the first one (its row, pixel and
 * clip frame) and keeps the handle's previous description.  nf == 0 is accepted (weight may then be NULL). */
int bsub_set_frame_weight_map_dev(bsub_solver* s, int32_t rows, int32_t cols, int32_t f0, int32_t nf, const float* weight, int64_t ld,
                                  void* stream);
int bsub_set_frame_graphs(bsub_solver* s, int32_t rows, int32_t cols, int32_t f0, int32_t nf, int32_t n_graphs, const int32_t* frame_graph,
                          const int64_t* n_groups, const int32_t* const* indptr, const int32_t* const* indices, const double* const* eta,
                          const uint8_t* background_host);
/* prox of the whole frames [f0, f0 + nf) -- any sub-range of the described one, else an error; nf == 0 does nothing -- held in
 * U_frames / V_frames (row f - f0 = frame f, row pitch ld_frames >= rows*cols): the tile kernel (windows, centre windows) or the
 * generic kernel, then the l2 shrink of each frame's background when one was given.  Whole-frame workspaces are allocated once and
 * grow with the largest block (BSUB_GRAPH_XI_MB caps the duals); bsub_debug_graph counts the calls. */
int bsub_step_prox_block(bsub_solver* s, const float* U_frames, float* V_frames, int64_t ld_frames, int32_t f0, int32_t nf, void* stream);
int bsub_poll(bsub_solver* s, bsub_status* st);            /* non-blocking: host mirror written by the device       */
int bsub_sync_status(bsub_solver* s, bsub_status* st, void* stream);   /* blocking                                 */

/* ---- results ---------------------------------------------------------------------------------------------- */
int bsub_finalize(bsub_solver* s, void* stream);           /* materialise L = U (sigma - 1/mu) V^T                  */
int bsub_get_L_f32_dev(bsub_solver* s, float** L, int64_t* ld);
int bsub_get_S_f32_dev(bsub_solver* s, float** S, int64_t* ld);   /* after bsub_finalize (S may have to be rebuilt)          */
int bsub_get_D_f32_dev(bsub_solver* s, float** D, int64_t* ld);
int bsub_get_Y_f32_dev(bsub_solver* s, float** Y, int64_t* ld);
int bsub_download_f64(bsub_solver* s, int which /*0 L, 1 S, 2 D, 3 Y*/, double* dst_host, int64_t ld, void* stream);
int bsub_download_f32(bsub_solver* s, int which, float* dst_host, int64_t ld, void* stream);
int bsub_get_log(bsub_solver* s, bsub_iter_log* out, int32_t cap, int32_t* count);
/* diagnostics: SM clock at the phase boundaries of the last eigensolve (load, tridiag, eigenvalues, vectors, reorth, back-transform) */
int bsub_debug_eig_cycles(bsub_solver* s, int64_t* out16);
/* diagnostics: kernel paths chosen for this solver: use_tma, use_stream, use_i8, stream R/FC/NS, gram types/kc, eig cluster, tma R/Cf, ld */
int bsub_debug_info(bsub_solver* s, int32_t* out16);   /* ..., [12] plane projection on, [13] its warps, [14] its slot depth */
/* diagnostics: [0] iterations of the last solve whose eigenpairs came from the warm-started subspace path (eig.cu), [1] vectors
 * kept for the next warm start, [2] subspace steps of the last call, [3] 1e6 * last certificate ||G - X theta X^T||_F mu^2,
 * [4] Gram mode of the next iteration (0 fp64 DMMA, 1 int8 tcgen05), [5] last digit pass saturated, [6] the solve has switched
 * to the fp64 Gram for accuracy, [7] 1e6 * bound of the int8 Gram's truncation error relative to (1/mu)^2 */
int bsub_debug_counters(bsub_solver* s, int64_t* out8);
/* graph prox of this handle (SPILL pass or bsub_step_prox_block): out4 = {outer iterations of the last call, their total over all calls,
 * calls, calls that hit graph_max_sweeps} */
int bsub_debug_graph(bsub_solver* s, int64_t* out4);
/* foreground_mask(D, L, S, sigmas) of utils.py:139-149 on the solver's own D, L, S; mask uint8[n][m] on the host */
int bsub_mask_stats_local(bsub_solver* s, int phase /*0: max|S|, 1: count/sum/sumsq*/, void* stream);
int bsub_mask_host(bsub_solver* s, double sigmas, uint8_t* mask_host, void* stream);
int bsub_mask_dev(bsub_solver* s, double sigmas, uint8_t* mask_dev, void* stream);

/* ---- operator-level entry points (the reference's unit-test seams, SURVEY.md 8b); device pointers ------------ */
/* foreground_mask(D, L, S, sigmas_from_mean)   utils.py:139-149 */
int bsub_foreground_mask_dev(const float* D, const float* L, const float* S, int64_t ld, int64_t m, int32_t n, double sigmas,
                             uint8_t* mask, void* stream);
/* prox_flat(G_S, lambda1, groups) on the 3x3 tiling   inexact_alm_lsd.py:71-79 */
int bsub_prox_flat3_dev(const float* U, float* V, int64_t ld, int32_t rows, int32_t cols, int32_t n, double lambda1, void* stream);
/* prox_flat for an arbitrary groups vector (host int32[m]) */
int bsub_prox_flat_groups_dev(const float* U, float* V, int64_t ld, int64_t m, int32_t n, const int32_t* groups_host,
                              double lambda1, void* stream);
/* prox(G_S, lambda1, graph) on the overlapping 3x3 windows   inexact_alm_lsd.py:49-57; eta_host as for bsub_set_graph_windows.
 * The three graph operators validate their graphs and eta before anything else, as the setters do, and synchronise the stream. */
int bsub_prox_graph3_dev(const float* U, float* V, int64_t ld, int32_t rows, int32_t cols, int32_t n, double lambda1,
                         const double* eta_host, int32_t max_sweeps, double tol, int32_t* sweeps_used, void* stream);
/* prox_by_frame(G_S, lambda1, graphs) with the per-frame centre-window graphs of get_proximal_graph_group_centers
 * (inexact_alm_lsd.py:60-68, lsd_improvement.py:74-120): eta_host float32[n][rows*cols] = weight of the 3x3 window centred on
 * that pixel of that frame (finite; <= 0: no window) */
int bsub_prox_center3_dev(const float* U, float* V, int64_t ld, int32_t rows, int32_t cols, int32_t n, double lambda1,
                          const float* eta_host, int32_t max_sweeps, double tol, int32_t* sweeps_used, void* stream);
/* prox / prox_by_frame (inexact_alm_lsd.py:49-68) for any non-nested graphs, all frames in one launch: graphs and frame_graph as for
 * bsub_set_graphs; stop when the largest dual change of a sweep <= tol (absolute), at most max_sweeps (<= 0: 4000) per frame;
 * sweeps_used = the largest sweep count over the frames.  Synchronises the stream. */
int bsub_prox_graph_dev(const float* U, float* V, int64_t ld, int64_t m, int32_t n, double lambda1, int32_t n_graphs, const int32_t* frame_graph,
                        const int64_t* n_groups, const int32_t* const* indptr, const int32_t* const* indices, const double* const* eta,
                        int32_t max_sweeps, double tol, int32_t* sweeps_used, void* stream);
/* block_shrinkage_operator(G, blocks_by_frame, lambdas_by_frame, mu, non_block_lambda)   group_sparse_RPCA.py:13-42 */
int bsub_block_shrink_dev(const float* G, float* R, int64_t ld, int64_t m, int32_t n, const uint8_t* labels_host,
                          const int32_t* lam_ptr, const double* lam, double mu, double non_block_lambda, void* stream);
/* G = W W^T, W = D - S + Y/mu (S, Y may be NULL): fp64 frames x frames Gram, G_host double[n][n] */
int bsub_gram_dev(const float* D, const float* S, const float* Y, int64_t ld, int64_t m, int32_t n, double mu, double* G_host,
                  void* stream);
/* top-k eigenpairs of a symmetric double[n][n] host matrix: svd_k_largest's n x n core (utils.py:204-212).
 * lam_host double[k] descending, vec_host double[k][n] (row i = eigenvector i). */
int bsub_eig_topk(const double* G_host, int32_t n, int32_t k, double* lam_host, double* vec_host);
/* the tcgen05 int8 Gram on its own: slices int8[4][n][ldq] (host), G int64[n][n] = sum_p sum_{i+j>=3} 256^(i+j-3) d_i(f,p) d_j(g,p) */
int bsub_gram_i8_test(const int8_t* slices_host, int32_t n, int64_t ldq, int64_t* G_host);
/* profiling hook: mean milliseconds of `reps` launches of that Gram on device-resident planes [4][ldq/16][n][16] */
int bsub_gram_i8_bench(int32_t n, int64_t ldq, int32_t reps, float* ms_out);

/* ---- stages on either side of the decomposition (SURVEY.md 8f rows 1, 3, 4); device pointers, csrc/post.cu ---- */
/* resize_with_cv2 / resize_with_cv2_by_first_axis (utils.py:119-136): cv2.resize of n images, interp 0 = INTER_AREA (shrinking),
 * 1 = INTER_CUBIC.  Element (f, y, x) of src lives at f*src_stride_f + y*src_stride_y + x*src_stride_x (elements); same for dst.
 * Synchronises the stream before it returns. */
int bsub_resize_dev(const float* src, int64_t src_stride_f, int64_t src_stride_y, int64_t src_stride_x, int32_t src_h, int32_t src_w, int32_t n,
                    float* dst, int64_t dst_stride_f, int64_t dst_stride_y, int64_t dst_stride_x, int32_t dst_h, int32_t dst_w, int32_t interp,
                    void* stream);
/* cv2.connectedComponentsWithStats(frame, 8, CV_32S) for every frame (utils.py:411-416, motion_saliency_check.py:25-28):
 * mask uint8[n][ld_mask] (non-zero = foreground, pixel p = j*rows + i), labels int32[n][ld]: 0 = background, 1..num_labels[f]
 * numbered by the smallest pixel index of each component; num_labels int32[n] (device); scratch 2*n*ld int32. */
int bsub_cc_label_dev(const uint8_t* mask, int64_t ld_mask, int32_t rows, int32_t cols, int32_t n, int32_t* labels, int64_t ld, int32_t* num_labels,
                      int32_t* scratch, void* stream);
/* per-component area, box {min row, max row, min col, max col, key} and (optional) sum of weight[f, j, i] over the component
 * (compute_groups_per_frame, motion_saliency_check.py:44-47); key = index of the first 2x2 block (raster order) that meets the
 * component: sorting a frame's components by it reproduces OpenCV's label numbering.  offsets int32[n] = exclusive prefix sum of
 * num_labels (device), total = their sum; area int32[total], box int32[total][5], wsum double[total] (device). */
int bsub_cc_stats_dev(const int32_t* labels, int64_t ld, int32_t rows, int32_t cols, int32_t n, const int32_t* offsets, int32_t total,
                      const float* weight, int64_t w_stride_f, int64_t w_stride_j, int64_t w_stride_i, int32_t* area, int32_t* box, double* wsum,
                      void* stream);
/* label image -> uint8 map through a per-component table (uint8[total], device): out[f][p] = table[offsets[f] + label - 1], 0 stays 0.
 * Turns the components kept by run_motion_saliency_check (motion_saliency_check.py:66-120) into the block map of bsub_set_blocks. */
int bsub_cc_remap_dev(const int32_t* labels, int64_t ld, int64_t m, int32_t n, const int32_t* offsets, const uint8_t* table, uint8_t* out, int64_t ld_out,
                      void* stream);
/* filter_sparse_map(sparse_array, size_thresh) (utils.py:404-420): keep the pixels of 8-connected components with area > size_thresh.
 * mask, out uint8[n][ld]; scratch 3*n*rows*cols int32. */
int bsub_filter_sparse_map_dev(const uint8_t* mask, int64_t ld_mask, int32_t rows, int32_t cols, int32_t n, int32_t size_thresh, uint8_t* out,
                               int64_t ld_out, int32_t* scratch, void* stream);
/* computeSCube (computeSCube.py:22-50,82-92): cube[t][h][w] = |xt[w][h][t]| * |yt[h][w][t]| and its sum (double, device);
 * scratch >= 2048 doubles.  The normalisation by the sum is applied by the first smoothing pass (divide_by_dev). */
int bsub_scube_product_dev(const float* xt, const float* yt, float* cube, int32_t T, int32_t H, int32_t W, double* sum_out, double* scratch,
                           void* stream);
/* one axis of scipy.ndimage.convolve(..., mode='reflect') with a separable kernel (computeSCube.py:90):
 * dst[o, i, r] = (1/divide_by) * sum_k w[k] * src[o, reflect(i + k - shift), r], array viewed as [outer][len][inner]. */
int bsub_conv1d_reflect_dev(const float* src, float* dst, int64_t outer, int32_t len, int64_t inner, const float* weights_dev, int32_t taps,
                            int32_t shift, const double* divide_by_dev, void* stream);
/* binary dilation (erode = 0) / erosion (erode = 1) of every frame by skimage.morphology.disk(radius) (apply_morph_ops,
 * lsd_improvement.py:323-335); src, dst uint8[n][ld]; scratch n*rows*cols + 2*radius + 1 bytes. */
int bsub_morph_disk_dev(const uint8_t* src, int64_t ld_src, uint8_t* dst, int64_t ld_dst, int32_t rows, int32_t cols, int32_t n, int32_t radius,
                        int32_t erode, uint8_t* scratch, void* stream);
/* compute_RPCA (computeRPCADecomposition.py:12-48), grayscale branch: one rank-capped (max_rank = 1) robust PCA per slice D[b]
 * (float32 [batch][rows][cols], device), all slices in one launch.  Engine: the reference's own inexact_alm_rpca iteration
 * (lsd_improvement.py:123-196: lambda = 1/(sqrt(max(rows, cols)) delta), Y0 = D/max(||D||_2, ||D||_inf/lambda), mu0 = 1.25/||D||_2,
 * mu *= rho) with the rank of L capped at 1; stops when ||Z||_F/||D||_F < tol or (tol_l1 > 0) sum|Z| <= tol_l1 or after max_iter.
 * iters[b] > 0: iterations used; < 0: -max_iter, tolerance not met.  err[b] = last ||Z||_F/||D||_F, rank[b] in {0, 1}.
 * Two kernels, chosen by shape (csrc/rpca_batch.cu): a slice whose state fits the shared memory of a cluster of <= 8 CTAs (cols <= 640
 * and 4 * ceil(rows/C) * cols floats per CTA) is solved there; any other slice up to 4096 x 4096 iterates in global memory, S in S and
 * Y/mu in L (L holds the low-rank part on return).  A larger slice is an error before any launch. */
int bsub_rpca_rank1_batch_dev(const float* D, int32_t batch, int32_t rows, int32_t cols, double delta, double rho, double tol,
                              double tol_l1, int32_t max_iter, float* L, float* S, int32_t* iters, float* err, int32_t* rank, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BSUB_B200_H */
