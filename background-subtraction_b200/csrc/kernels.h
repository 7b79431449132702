// kernels.h -- host-side launch interfaces of the CUDA kernels (internal; the public boundary is
// include/bsub_b200.h).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <vector>
#include "common.cuh"

namespace bsub {

// ---------------------------------------------------------------- gram.cu
struct GramPlan {
    int n, npad, nb, ntasks, ntype, gridK, kc, nbox, boxrows;
    long long nchunks;
    size_t smem_bytes, partial_elems;
};
struct GramMaps { CUtensorMap D, S, Y; int narr; };     // TMA descriptors of the [n][ld] float32 matrices
GramPlan make_gram_plan(int n, long long ld, int num_sms);
void fill_gram_tasks(const GramPlan& p, int2* host_tasks);
int make_gram_maps(const GramPlan& p, const float* D, const float* S, const float* Y, long long ld, GramMaps* maps);
// combo: W = D - S + Y/mu (needs the S/Y maps); otherwise W = D
int launch_gram(const GramPlan& p, const GramMaps& maps, bool combo, const int2* dev_tasks, const DevState* st,
                float inv_mu_override, double* partial, double* G, cudaStream_t stream);

// ---------------------------------------------------------------- gram_i8.cu (tcgen05 int8 Gram from the W slices)
struct GramI8Plan { int n, nblk, nkb, grid; long long ldq; size_t smem_bytes;
                    long long m_real;       // pixels that hold real data (0: no correction of the dropped digit classes)
                    long long m_global; };  // pixels of the whole matrix (pixel-sharded runs), 0 = m_real
GramI8Plan make_gram_i8_plan(int n, long long ldq, int num_sms);
void fill_gram_i8_tables(const GramI8Plan& p, std::vector<int4>& cta_info, std::vector<int>& blk_n);
int make_gram_i8_map(const GramI8Plan& p, const signed char* Wq, CUtensorMap* map, int box_frames);
int gram_i8_last_block_n(const GramI8Plan& p);
int gram_i8_last_block_frames();
int launch_quantize_D(const float* D, long long ld, int n, long long ldq, signed char* Wq, const double* dmax, DevState* st,
                      cudaStream_t stream);
int launch_gram_i8(const GramI8Plan& p, const CUtensorMap& map, const CUtensorMap& map_last, const int4* cta_info_dev, int ncta, const int* blk_n_dev,
                   unsigned long long* Gint, double* G, int npad, const DevState* st, double scale_override, int require_mode,
                   cudaStream_t stream);

// ---------------------------------------------------------------- eig.cu
struct EigPlan {
    int n, npad, C, rows_per, in_smem, kcap;
    size_t smem_bytes;
    size_t work_doubles;       // total doubles of the device workspace
};
struct EigBuffers {
    double* work;              // workspace of EigPlan::work_doubles doubles
    double* lam;               // [n] eigenvalues, descending (top K valid)
    double* Z;                 // [n][n] eigenvectors, row k = vector k (top K valid)
    float* Vr;                 // [n][vstride] right singular vectors (fp32), columns 0..svp-1
    float* VC;                 // [n][vstride] Vr scaled by (1 - 1/(mu sigma_k))
    int vstride;
};
EigPlan make_eig_plan(int n, int npad);
// mode 0: init (K = 1; fills norm_two, normD2, dual_norm, mu, ...);  mode 1: ALM iteration control
// mode 2: stand-alone top-K (K = k_override), no state update except lam/Z
int launch_eig(const EigPlan& p, const double* G, const double* comm_max, EigBuffers b, DevState* st, int mode,
               int k_override, cudaStream_t stream);

// ---------------------------------------------------------------- shrink.cu
struct ShrinkPlan {
    int n, rows, cols, R, P, Cf, nf, threads, grid_clusters, kr;
    long long ld, m;
    int ntile_r, ntile_c;
    long long ntiles;
    size_t smem_bytes;
    size_t tpart_floats;       // cross-CTA T partial scratch
    int nparts;                // number of CTAs (length of the per-CTA partial arrays)
};
enum ShrinkMode { SHRINK_FLAT3 = 0, SHRINK_SPILL = 1, SHRINK_L1 = 2 };
ShrinkPlan make_shrink_plan(int n, int rows, int cols, long long ld, int num_sms, int R_hint, int Cf_hint);
struct ShrinkBuffers {
    const float* D; float* S; float* Y;
    float* T;                  // [tcap][ld] projected coefficients T = Vr^T W
    float* U;                  // SPILL mode: G_S = D - L + Y/mu  ([n][ld])
    float* tpart;              // scratch
    const float* Vr; const float* VC; int vstride;
    double* part_zz;           // [nparts]
    unsigned long long* part_nnz;
    float* part_max;
    float* part_wmax;          // [stream grid] max |W_next| written with the int8 slices (nullptr: slices off)
    int implied_first = 0;     // shrink_stream only: iteration 1 derives S0 = 0, Y0 = D / dual_norm from D (init_Y skipped)
    int have_flat = 0;         // shrink_stream only: shrink_flat.cu is launched too and takes the iterations it can (DevState decides)
    const float* Tt = nullptr; // shrink_stream only: T regrouped per tile by project.cu; when the planes of this W exist
                               // (DevState::gram_mode == 1) the kernel skips its own projection pass and streams every tile once
};
int launch_shrink(const ShrinkPlan& p, ShrinkBuffers b, const DevState* st, int mode, cudaStream_t stream);

// ---------------------------------------------------------------- shrink_tma.cu (fast path, rows % 4 == 0)
struct ShrinkTmaPlan {
    int n, rows, cols, R, P, Cf, nf, KR, grid_clusters, nparts, ntile_r, ntile_c, bufstride;
    long long ld, ntiles;
    size_t smem_bytes, tpart_floats;
};
struct ShrinkTmaMaps { CUtensorMap D, S, Y, U, Q, Vr, VC; bool has_U, has_Q; };
bool make_shrink_tma_plan(int n, int rows, int cols, long long ld, int num_sms, int R_hint, int Cf_hint, ShrinkTmaPlan* out);
int make_shrink_tma_maps(const ShrinkTmaPlan& p, const float* D, float* S, float* Y, float* U, ShrinkTmaMaps* m);
int launch_shrink_tma(const ShrinkTmaPlan& p, const ShrinkTmaMaps& maps, ShrinkBuffers b, const DevState* st, int mode,
                      int min_rank, cudaStream_t stream);

// ---------------------------------------------------------------- shrink_stream.cu (fastest path: rank <= 16, rows % 4 == 0)
struct ShrinkStreamPlan {
    int n, rows, cols, R, P, FC, NS, nchunkf, grid, nparts, ntile_r, ntile_c, bufstride;
    int kcap;                  // largest rank the streamed kernel takes (16)
    long long ld, ntiles;
    size_t smem_bytes;
};
constexpr int kStreamMaxRank = 16;
bool make_shrink_stream_plan(int n, int rows, int cols, long long ld, int num_sms, int R_hint, ShrinkStreamPlan* out);
int make_shrink_stream_maps(const ShrinkStreamPlan& p, const float* D, float* S, float* Y, float* U, ShrinkTmaMaps* m);
long long shrink_stream_ldq(const ShrinkStreamPlan& p);
int make_shrink_stream_vmaps(const ShrinkStreamPlan& p, const float* Vr, const float* VC, int vstride, ShrinkTmaMaps* m);
int make_shrink_stream_qmap(const ShrinkStreamPlan& p, signed char* Wq, ShrinkTmaMaps* m);
int launch_shrink_stream(const ShrinkStreamPlan& p, const ShrinkTmaMaps& maps, ShrinkBuffers b, const DevState* st, int mode,
                         cudaStream_t stream);

// ---------------------------------------------------------------- shrink_flat.cu (single-pass streamed shrink, rank <= 8, T from project.cu)
struct ShrinkFlatPlan { int n, rows, cols, FC, NS, nchunkf, ntile_r, grid; long long ld, ntiles; size_t smem_bytes; };
struct ShrinkFlatMaps { CUtensorMap D, S, Y, Q, VC; };
bool make_shrink_flat_plan(int n, int rows, int cols, long long ld, int num_sms, const ShrinkStreamPlan& sp, ShrinkFlatPlan* out);
int make_shrink_flat_maps(const ShrinkFlatPlan& p, const float* D, float* S, float* Y, signed char* Wq, long long ldq, const float* VC, int vstride,
                          ShrinkFlatMaps* m);
// part_*: [p.grid] partial results of this kernel (zeros when it leaves the iteration to a fallback kernel)
int launch_shrink_flat(const ShrinkFlatPlan& p, const ShrinkFlatMaps& maps, const float* Tt, DevState* st, int mode, int force_S, double* part_zz,
                       unsigned long long* part_nnz, float* part_max, float* part_wmax, cudaStream_t stream);
// S <- D + Y/mu - W_q from the digit planes when DevState::s_stale says the last passes skipped the store of S
int launch_rebuild_S(const ShrinkFlatPlan& p, const float* D, const float* Y, float* S, const signed char* Wq, long long ldq, DevState* st,
                     int min_rank, cudaStream_t stream);

// ---------------------------------------------------------------- project.cu (T = Vr^T W from the int8 digit planes)
struct ProjectPlan { int n, NW, DEPTH, slot_bytes, grid; long long ldq; size_t smem_bytes; };
bool make_project_plan(int n, int R, long long ldq, int num_sms, ProjectPlan* out);
// T: [kcap][ld] pixel order; Tt: [ntiles][16][4R] regrouped per tile / 3x3 group for shrink_stream's phase B
int launch_project(const ProjectPlan& p, const signed char* Wq, const float* Vr, int vstride, float* T, long long ld, float* Tt, int rows,
                   int cols, int R, int ntile_r, long long ntiles, int kcap, const DevState* st, cudaStream_t stream);

// ---------------------------------------------------------------- elementwise.cu
int launch_rowsum_max(const float* D, long long ld, long long m, int n, double* comm_max, cudaStream_t s);
int launch_init_Y(const float* D, float* Y, float* S, long long ld, int n, const DevState* st, cudaStream_t s);
int launch_control_post(DevState* st, const double* part_zz, const unsigned long long* part_nnz,
                        const float* part_max, int nparts, double* comm_sum_tail, IterLog* log, HostMirror* mirror,
                        int phase, const float* part_wmax, int nwmax, cudaStream_t s);
int launch_convert_f64(const double* src, long long src_ld, float* dst, long long ld, long long m, int n,
                       cudaStream_t s);
int launch_export_f64(const float* src, long long ld, double* dst, long long dst_ld, long long m, int n,
                      cudaStream_t s);
int launch_copy_f32(const float* src, long long src_ld, float* dst, long long ld, long long m, int n, cudaStream_t s);
int launch_u8_stats(const unsigned char* src, long long count, unsigned long long* sum_minmax, cudaStream_t s);
int launch_u8_to_D(const unsigned char* src, float* D, long long ld, long long m, int n, double lo, double scale,
                   double mean, cudaStream_t s);
// L = VC * T  (materialise the low-rank part), optionally masked statistics for foreground_mask
int launch_materialize_L(const float* T, const float* VC, int vstride, const DevState* st, float* L, long long ld,
                         long long m, int n, cudaStream_t s);
// second half of the two-phase shrink (SPILL mode): given S_new, recompute L from T and update Y
int launch_dual_update(const float* D, const float* Snew, float* S, float* Y, const float* T, const float* VC, int vstride,
                       const DevState* st, float* Lscratch, long long ld, int n, double* part_zz,
                       unsigned long long* part_nnz, float* part_max, int nparts, cudaStream_t s);

// ---------------------------------------------------------------- mask.cu
int launch_absmax(const float* S, long long ld, long long m, int n, double* out_max, cudaStream_t s);
int launch_maxS_from_state(const DevState* st, double* out_max, cudaStream_t s);
// scratch: mask_stats_scratch_doubles() doubles, zero before the first use (per-CTA partials + a ticket counter)
size_t mask_stats_scratch_doubles();
int launch_mask_stats(const float* D, const float* L, const float* S, long long ld, long long m, int n,
                      const double* absmax, double* stats /*[3]: count, sum, sumsq*/, double* scratch, cudaStream_t s);
int launch_mask_write(const float* S, long long ld, long long m, int n, const double* stats, double sigmas,
                      unsigned char* mask, long long mask_ld, cudaStream_t s);
// weight map float [nf][ld] -> eta [nf][m] (positive entries, else 0) and labels [nf][m] (0: negative entry, else 255); the flat
// index f * m + p of the first non-finite entry is atomicMin'ed into *first_bad (nf >= 1)
int launch_weight_map_describe(const float* w, long long ld, long long m, int nf, float* eta, unsigned char* labels,
                               unsigned long long* first_bad, cudaStream_t s);

// ---------------------------------------------------------------- prox.cu (operator-level + generic modes)
int launch_prox_flat3(const float* U, float* V, long long ld, int rows, int cols, int n, float lam, cudaStream_t s);
// st != nullptr: lambda1 = st->lambda / st->mu read on the device, and the kernel is skipped once st->done
int launch_prox_groups_csr(const float* U, float* V, long long ld, long long m, int n, const int* gptr,
                           const int* gidx, int ngroups, float lam, const DevState* st, cudaStream_t s);
int launch_block_l2_sums(const float* U, const unsigned char* labels, long long ld, long long m, int n, int nlab,
                         double* sums, const DevState* st, cudaStream_t s);
int launch_block_l2_apply(const float* U, float* V, const unsigned char* labels, long long ld, long long m, int n,
                          int nlab, const double* sums, const double* lam_table, const DevState* st,
                          double mu_override, double non_block_lambda, cudaStream_t s, int keep_other = 0);
int launch_prox_l1(const float* U, float* V, long long ld, long long m, int n, float lam, cudaStream_t s);
struct GraphProxPlan { int rows, cols, n; long long ld; size_t xi_floats; int max_sweeps; float tol; };
// workspace: xi = duals of whole frames (BSUB_GRAPH_XI_MB cap, default 8 GB: the kernel walks the frames in chunks that fit),
// tot = per-pixel dual sums of the frames held (ld floats each)
void prox_graph3_workspace(int rows, int cols, int n, long long ld, int center, long long* xi_floats, long long* tot_floats);
int launch_prox_graph3(const float* U, float* V, float* xi, long long xi_floats, float* tot, const float* eta, long long ld, int rows,
                       int cols, int n, float lam, int max_sweeps, float tol, int* sweeps_out, const DevState* st,
                       cudaStream_t s, int center = 0, long long eta_stride = 0);

// ---------------------------------------------------------------- prox_graph.cu (any non-nested graph, one graph per frame)
// Graphs coloured and stored colour-major by pack_generic_graphs: graph gr owns colours [gcol[gr], gcol[gr+1]); colour c owns
// groups [cbeg[c], cbeg[c+1]), of which [cbig[c], cbeg[c+1]) have more than 32 pixels; group g owns gidx[gptr[g] .. gptr[g+1])
// and its dual entries are the same positions minus gnz0[gr].
struct GenericGraphHost {
    std::vector<int> frame_graph, gcol, cbeg, cbig, gptr, gidx, gnz0;
    std::vector<float> eta;
    long long max_nnz = 0; int max_colours = 0;
};
struct GenericGraphDev {
    const int *frame_graph, *gcol, *cbeg, *cbig, *gptr, *gidx, *gnz0;
    const float* eta;
    long long max_nnz;
};
// where the per-pixel dual sums live (cs CTAs per cluster, 1 << shift pixels each, or global rows) and the workspace that takes
struct GenericGraphLayout { int cs, shift, slots; bool tot_global; long long xi_floats, tot_floats; size_t smem; };
// validates every input (bad input: error message, nothing launched), colours each graph and lays it out
int pack_generic_graphs(long long m, int n, int n_graphs, const int32_t* frame_graph, const int64_t* n_groups,
                        const int32_t* const* indptr, const int32_t* const* indices, const double* const* eta, GenericGraphHost* out,
                        const char* who);
// one device allocation for the index arrays (*ints) and one for eta; frees what the pointers held before
int upload_generic_graphs(const GenericGraphHost& H, int** ints, float** eta_dev, GenericGraphDev* dev);
// duals: BSUB_GRAPH_XI_MB cap (default 8 GB) on the clusters in flight
GenericGraphLayout prox_graph_generic_layout(long long m, long long ld, int n, long long max_nnz);
// status: the caller's zeroed int[8] ([0] sweeps of the last call, [4..6] running totals as for launch_prox_graph3)
int launch_prox_graph_generic(const float* U, float* V, long long ld, long long m, int n, const GenericGraphDev& g, const GenericGraphLayout& L,
                              float* xi, float* totg, float lam, int max_sweeps, float tol, int* status, const DevState* st, cudaStream_t s);

}  // namespace bsub
