// prox.cu -- stand-alone proximal operators (the reference's operator seams) and the prox stage of the two-phase
// shrink used by the modes that cannot be fused into shrink.cu:
//   prox_flat3        spams.proximalFlat 'group-lasso-linf' on the regular 3x3 tiling   (/root/reference/inexact_alm_lsd.py:71-79)
//   prox_groups_csr   the same regulariser for an ARBITRARY int32 groups vector (any partition of the pixels)
//   block_l2_*        block_shrinkage_operator                                           (/root/reference/group_sparse_RPCA.py:13-42)
//   prox_l1           elementwise soft threshold                                         (/root/reference/lsd_improvement.py:176)
//   prox_graph3       spams.proximalGraph 'graph' on the overlapping 3x3 windows         (/root/reference/inexact_alm_lsd.py:49-57)
#include <cooperative_groups.h>
#include <stdlib.h>
#include <algorithm>
#include "common.cuh"
#include "kernels.h"
#include "prox9.cuh"

namespace cg = cooperative_groups;

namespace bsub {

constexpr int PX_THREADS = 256;

__device__ __forceinline__ void px_cswap_desc(float& a, float& b) {
    float hi = fmaxf(a, b), lo = fminf(a, b);
    a = hi; b = lo;
}

// clip level theta of the l1-ball projection of k <= 9 non-negative values (sum a > z)
__device__ __forceinline__ float px_clip_level9(const float* a_in, float z) {
    float u[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) u[i] = a_in[i];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8 - i; ++j) px_cswap_desc(u[j], u[j + 1]);
    const float inv[9] = {1.f, 0.5f, 1.f / 3.f, 0.25f, 0.2f, 1.f / 6.f, 1.f / 7.f, 0.125f, 1.f / 9.f};
    float cs = 0.f, theta = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        cs += u[k];
        float t = (cs - z) * inv[k];
        if (u[k] > t) theta = t;
    }
    return theta;
}

// ---------------------------------------------------------------------------------------- flat 3x3 tiles
__global__ void prox_flat3_kernel(const float* __restrict__ U, float* __restrict__ V, long long ld, int rows, int cols, int n,
                                  float lam) {
    const int gr = (rows + 2) / 3, gc = (cols + 2) / 3;
    const long long ng = (long long)gr * gc;
    for (int f = blockIdx.y; f < n; f += gridDim.y) {
        const float* u = U + (size_t)f * ld;
        float* v = V + (size_t)f * ld;
        for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < ng; g += (long long)gridDim.x * blockDim.x) {
            const int tj = (int)(g / gr), ti = (int)(g - (long long)tj * gr);
            float x[9], ax[9];
            float sabs = 0.f;
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int dr = 0; dr < 3; ++dr) {
                    const int i = 3 * ti + dr, j = 3 * tj + c;
                    const bool ok = (i < rows) && (j < cols);
                    const float val = ok ? u[(long long)j * rows + i] : 0.f;
                    x[c * 3 + dr] = val; ax[c * 3 + dr] = fabsf(val); sabs += fabsf(val);
                }
            const bool nz = sabs > lam;
            const float theta = nz ? px_clip_level9(ax, lam) : 0.f;
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int dr = 0; dr < 3; ++dr) {
                    const int i = 3 * ti + dr, j = 3 * tj + c;
                    if (i < rows && j < cols) v[(long long)j * rows + i] = nz ? copysignf(fminf(ax[c * 3 + dr], theta), x[c * 3 + dr]) : 0.f;
                }
        }
    }
}

int launch_prox_flat3(const float* U, float* V, long long ld, int rows, int cols, int n, float lam, cudaStream_t s) {
    const long long ng = (long long)((rows + 2) / 3) * ((cols + 2) / 3);
    long long gx = (ng + PX_THREADS - 1) / PX_THREADS;
    if (gx > 2048) gx = 2048;
    if (gx < 1) gx = 1;
    dim3 g((unsigned)gx, n < 256 ? n : 256);
    prox_flat3_kernel<<<g, PX_THREADS, 0, s>>>(U, V, ld, rows, cols, n, lam);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------- arbitrary flat groups
// gptr/gidx: CSR of group -> pixel list for ids >= 1; pixels with id 0 are copied through by the caller
// (V is initialised with U).  One thread per (group, frame); Michelot's finite active-set iteration gives the
// exact clip level without sorting or local arrays.
__global__ void prox_groups_csr_kernel(const float* __restrict__ U, float* __restrict__ V, long long ld, int n,
                                       const int* __restrict__ gptr, const int* __restrict__ gidx, int ngroups, float lam,
                                       const DevState* st) {
    if (st != nullptr) { if (st->done) return; lam = (float)(st->lambda / st->mu); }
    for (int f = blockIdx.y; f < n; f += gridDim.y) {
        const float* u = U + (size_t)f * ld;
        float* v = V + (size_t)f * ld;
        for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += gridDim.x * blockDim.x) {
            const int b = gptr[g], e = gptr[g + 1];
            if (e <= b) continue;
            float sabs = 0.f;
            for (int q = b; q < e; ++q) sabs += fabsf(u[gidx[q]]);
            if (sabs <= lam) { for (int q = b; q < e; ++q) v[gidx[q]] = 0.f; continue; }
            float theta = (sabs - lam) / (float)(e - b);
            for (int it = 0; it < e - b; ++it) {
                float sum = 0.f; int cnt = 0;
                for (int q = b; q < e; ++q) { const float a = fabsf(u[gidx[q]]); if (a > theta) { sum += a; ++cnt; } }
                const float t2 = (sum - lam) / (float)cnt;
                if (!(t2 > theta)) break;
                theta = t2;
            }
            for (int q = b; q < e; ++q) { const float x = u[gidx[q]]; v[gidx[q]] = copysignf(fminf(fabsf(x), theta), x); }
        }
    }
}

// V <- U unless the solve has already stopped (the host enqueues a few iterations ahead of the device-side stop flag: an
// unconditional copy would overwrite the final S with the last G_S)
__global__ void prox_copy_through_kernel(const float* __restrict__ U, float* __restrict__ V, long long total4, const DevState* st) {
    if (st != nullptr && st->done) return;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total4; q += (long long)gridDim.x * blockDim.x)
        stg4(V + 4 * q, ldg4_stream(U + 4 * q));
}

int launch_prox_groups_csr(const float* U, float* V, long long ld, long long m, int n, const int* gptr, const int* gidx,
                           int ngroups, float lam, const DevState* st, cudaStream_t s) {
    (void)m;
    if (U != V) {
        if ((ld & 3) == 0 && ((reinterpret_cast<uintptr_t>(U) | reinterpret_cast<uintptr_t>(V)) & 15) == 0) {
            const long long total4 = ld * n / 4;
            long long gb = (total4 + PX_THREADS * 4 - 1) / (PX_THREADS * 4);
            if (gb > 148 * 8) gb = 148 * 8;
            if (gb < 1) gb = 1;
            prox_copy_through_kernel<<<(unsigned)gb, PX_THREADS, 0, s>>>(U, V, total4, st);
            BSUB_CUDA_CHECK(cudaGetLastError());
        } else {
            if (st != nullptr) { set_error("prox_groups_csr: unaligned matrices inside a solve"); return -1; }
            BSUB_CUDA_CHECK(cudaMemcpyAsync(V, U, sizeof(float) * (size_t)ld * n, cudaMemcpyDeviceToDevice, s));
        }
    }
    int gx = (ngroups + PX_THREADS - 1) / PX_THREADS;
    if (gx > 2048) gx = 2048;
    if (gx < 1) gx = 1;
    dim3 g((unsigned)gx, n < 256 ? n : 256);
    prox_groups_csr_kernel<<<g, PX_THREADS, 0, s>>>(U, V, ld, n, gptr, gidx, ngroups, lam, st);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------- per-frame l2 blocks
// labels[f][p] (uint8): 0 = complement group, b >= 1 = block b of that frame.  sums[f][nlab] = sum of squares.
__global__ void block_l2_sums_kernel(const float* __restrict__ U, const unsigned char* __restrict__ labels, long long ld,
                                     long long m, int nlab, double* __restrict__ sums, const DevState* st) {
    __shared__ double red[32];
    if (st != nullptr && st->done) return;
    const int f = blockIdx.y;
    const float* u = U + (size_t)f * ld;
    const unsigned char* lab = labels + (size_t)f * m;
    double s0 = 0.0;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (long long)gridDim.x * blockDim.x) {
        const float x = u[p];
        const int l = lab[p];
        if (l == 0) s0 += (double)x * (double)x;
        else if (l < nlab) atomicAdd(sums + (size_t)f * nlab + l, (double)x * (double)x);
    }
    s0 = block_sum(s0, red);
    if (threadIdx.x == 0) atomicAdd(sums + (size_t)f * nlab, s0);
}

int launch_block_l2_sums(const float* U, const unsigned char* labels, long long ld, long long m, int n, int nlab, double* sums,
                         const DevState* st, cudaStream_t s) {
    BSUB_CUDA_CHECK(cudaMemsetAsync(sums, 0, sizeof(double) * (size_t)n * nlab, s));
    long long gx = (m + PX_THREADS * 8 - 1) / (PX_THREADS * 8);
    if (gx < 1) gx = 1;
    if (gx > 256) gx = 256;
    dim3 g((unsigned)gx, n);
    block_l2_sums_kernel<<<g, PX_THREADS, 0, s>>>(U, labels, ld, m, nlab, sums, st);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// factor = max(1 - eps/||G_g||_2, 0), zero-norm group -> 0 (group_sparse_RPCA.py:35,40 with max(-inf, 0) = 0)
__global__ void block_l2_apply_kernel(const float* __restrict__ U, float* __restrict__ V, const unsigned char* __restrict__ labels,
                                      long long ld, long long m, int nlab, const double* __restrict__ sums,
                                      const double* __restrict__ lam_table, const DevState* st, double mu_override,
                                      double non_block_lambda, int keep_other) {
    extern __shared__ float fac_s[];
    if (st != nullptr && st->done) return;
    const int f = blockIdx.y;
    const double mu = (st != nullptr) ? st->mu : mu_override;
    if (st != nullptr) non_block_lambda = st->non_block_lambda;
    for (int l = threadIdx.x; l < nlab; l += blockDim.x) {
        const double eps = ((l == 0) ? non_block_lambda : lam_table[(size_t)f * nlab + l]) / mu;
        const double nrm = sqrt(sums[(size_t)f * nlab + l]);
        double t = (nrm > 0.0) ? 1.0 - eps / nrm : 0.0;
        fac_s[l] = (float)(t > 0.0 ? t : 0.0);
    }
    __syncthreads();
    const float* u = U + (size_t)f * ld;
    float* v = V + (size_t)f * ld;
    const unsigned char* lab = labels + (size_t)f * m;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (long long)gridDim.x * blockDim.x) {
        const int l = lab[p];
        if (l < nlab) v[p] = fac_s[l] * u[p];
        else if (!keep_other) v[p] = 0.f;               // keep_other: pixels outside every group keep what V already holds
    }
}

int launch_block_l2_apply(const float* U, float* V, const unsigned char* labels, long long ld, long long m, int n, int nlab,
                          const double* sums, const double* lam_table, const DevState* st, double mu_override,
                          double non_block_lambda, cudaStream_t s, int keep_other) {
    long long gx = (m + PX_THREADS * 8 - 1) / (PX_THREADS * 8);
    if (gx < 1) gx = 1;
    if (gx > 256) gx = 256;
    dim3 g((unsigned)gx, n);
    block_l2_apply_kernel<<<g, PX_THREADS, sizeof(float) * nlab, s>>>(U, V, labels, ld, m, nlab, sums, lam_table, st, mu_override,
                                                                     non_block_lambda, keep_other);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------- l1
__global__ void prox_l1_kernel(const float* __restrict__ U, float* __restrict__ V, long long total, float lam) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const float x = U[i];
        V[i] = copysignf(fmaxf(fabsf(x) - lam, 0.f), x);
    }
}
int launch_prox_l1(const float* U, float* V, long long ld, long long m, int n, float lam, cudaStream_t s) {
    (void)m;
    const long long total = ld * n;
    long long gx = (total + PX_THREADS * 8 - 1) / (PX_THREADS * 8);
    if (gx < 1) gx = 1;
    if (gx > 148 * 8) gx = 148 * 8;
    prox_l1_kernel<<<(unsigned)gx, PX_THREADS, 0, s>>>(U, V, total, lam);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------- overlapping 3x3 windows
// Dual block-coordinate descent with the 9-colouring (i mod 3, j mod 3) of the window top-lefts: windows of one
// colour are disjoint, so one colour step is one fully parallel pass.  Window geometry reproduces
// get_vars_idx_top_left (/root/reference/utils.py:249-257): top-lefts i in [0, rows-3], j in [0, cols-3],
// extent min(3, rows-1-i) x min(3, cols-1-j)  => last image row / column uncovered (SURVEY Q8).
// Per frame f: xi[f][w][9] dual variables, tot[f][p] = sum of duals on pixel p.
//
// The sweeps run in shared memory, not in HBM.  The early ALM iterations need thousands of sweeps (lambda/mu is large and the
// dual mass spreads like a diffusion: measured with the oracle, WaterSurface iteration 1 = 4292 sweeps, a 540 x 960 frame
// ~1900), and a grid-wide sweep over HBM moves ~180 B per matrix element and sweep and pays ten grid-wide barriers per sweep
// (one per colour, plus the stop test).  Here a CTA takes a GT_T x GT_T pixel tile of one frame, loads u, the per-pixel dual
// sums `tot` and the duals of the windows that lie ENTIRELY inside the tile (84 B per element), runs up to GT_INNER nine-colour sweeps on them in shared memory (block barriers only) and writes them back.  Windows that straddle
// a tile border stay frozen during that visit; the tiling is shifted diagonally by a third of a tile in each of three phases
// ((0,0), (11,11), (22,22)): a window straddles a row border in at most one phase and a column border in at most one phase,
// so it is interior -- and updated -- in at least one of the three.  Every update is still an exact block minimisation of
// the same dual objective and simultaneously updated windows never overlap, so the iteration converges to the same (unique)
// primal solution as the sequential sweep of the oracle; stop test: the largest dual change of a whole outer iteration
// (3 phases x inner sweeps) <= tol.  One grid-wide barrier per phase instead of per colour.
// The state is (xi, tot) with r = u - tot + xi and tot += xi' - xi: a window whose projection reproduces its dual bit for bit
// changes nothing, so the iteration reaches a true fixed point in fp32 (carrying x = u - tot instead re-rounds x at every
// visit: it never settles below ~1 ulp of u and drifts -- seen in round 2).
// Duals are not kept between calls (cold start, like the oracle), so frames are processed in chunks whose duals fit the
// caller's buffer (prox_graph3_workspace: capped, default 8 GB) -- 4K x 600 needs ~18 GB per 60-frame chunk instead of 179 GB.
constexpr int GT_T = 32, GT_PITCH = 33, GT_THREADS = 128, GT_INNER = 48, GT_SHIFT = 11;
constexpr int GT_TILE = GT_T * GT_PITCH;
constexpr size_t GT_SMEM = sizeof(float) * (size_t)GT_TILE * (3 + 9);
constexpr float GT_COUNT_FACTOR = 8.f;      // dead bands a dual change must exceed to count towards the stop test (see the kernel)

struct GraphTileArgs {
    const float* U; float* V; float* xi; float* tot; const float* eta;
    long long ld; int rows, cols, n; float lam; int max_outer; float tol;
    int* sweeps_out; unsigned int* change_bits;   // [3]: largest dual change of outer iteration k lives in slot k % 3
    unsigned int* item_ctr;                       // [3]: work counter of phase k lives in slot k % 3 (dynamic tile scheduling)
    float count_factor;                           // a change counts towards the stop test when it exceeds count_factor x the dead band
    int* stats;                                   // [3] running totals over the calls of a handle: outer iterations, calls, calls that hit the cap
    const DevState* st;
    // centre mode (get_proximal_graph_group_centers, /root/reference/lsd_improvement.py:74-120): one candidate window per
    // pixel, centred on it and clipped to the image (utils.py:234-246); eta[f][pixel] > 0 selects and weights it
    int center; long long eta_stride;
    int nwi, nwj, chunk;
};

// window (wi, wj) -> pixel rectangle [i0, i0 + hh) x [j0, j0 + ww)   (utils.py:249-257, or the clipped centre windows :234-246)
__device__ __forceinline__ void gt_geometry(bool ctr, int rows, int cols, int wi, int wj, int& i0, int& j0, int& hh, int& ww) {
    i0 = ctr ? max(wi - 1, 0) : wi; j0 = ctr ? max(wj - 1, 0) : wj;
    hh = ctr ? min(wi + 1, rows - 1) - i0 + 1 : min(3, rows - 1 - wi);
    ww = ctr ? min(wj + 1, cols - 1) - j0 + 1 : min(3, cols - 1 - wj);
}
// [lo, hi] lies inside one interval of the tiling whose borders sit at off + k GT_T
__device__ __forceinline__ bool gt_inside(int lo, int hi, int off) {
    return (lo - off + GT_T) / GT_T == (hi - off + GT_T) / GT_T;
}

__global__ void __launch_bounds__(GT_THREADS) prox_graph3_tile_kernel(GraphTileArgs a) {
    cg::grid_group grid = cg::this_grid();
    if (a.st != nullptr) {
        if (a.st->done) return;                                  // uniform over the grid
        a.lam = (float)(a.st->lambda / a.st->mu);
        a.tol = a.tol * a.lam;                                   // relative tolerance in solver mode
    }
    extern __shared__ __align__(16) float gt_smem[];
    float* us = gt_smem;                                         // u of the tile, column c at c * GT_PITCH
    float* ts = us + GT_TILE;                                    // tot (sum of the duals on each pixel)
    float* rads = ts + GT_TILE;                                  // lambda * eta of an owned window, < 0: not owned / no window
    float* xis = rads + GT_TILE;                                 // duals of candidate window (a, b) at (b * GT_PITCH + a) * 9
    const int rows = a.rows, cols = a.cols, nwi = a.nwi, nwj = a.nwj;
    const bool ctr = a.center != 0;
    const long long nw = (long long)nwi * nwj;
    const int tid = threadIdx.x;
    const long long gsz = (long long)gridDim.x * blockDim.x, gid = (long long)blockIdx.x * blockDim.x + tid;
    __shared__ long long item_s;
    if (blockIdx.x == 0 && tid < 3) { a.change_bits[tid] = 0u; a.item_ctr[tid] = 0u; }
    grid.sync();
    int oc = 0, most = 0, pc = 0;                                // outer iterations and phases done so far (slot rotation)
    for (int f0 = 0; f0 < a.n; f0 += a.chunk) {
        const int nf = min(a.chunk, a.n - f0);
        int outer = 0;
        while (outer < a.max_outer) {
            float mych = 0.f;
            for (int ph = 0; ph < 3; ++ph) {
                const int off = ph * GT_SHIFT;
                const int ntr = (max(rows - off, 0) + GT_T - 1) / GT_T + (off > 0 ? 1 : 0);
                const int ntc = (max(cols - off, 0) + GT_T - 1) / GT_T + (off > 0 ? 1 : 0);
                const long long per_frame = (long long)ntr * ntc, nitems = per_frame * nf;
                const bool first = (outer == 0 && ph == 0);      // nothing has been written yet: tot = 0, xi = 0
                // Tiles are handed out through a counter: a visit costs between 1 and GT_INNER sweeps, and with a fixed assignment
                // half of the warp time of a small clip was spent waiting at the grid barrier for the unluckiest CTA (ncu r2y).
                for (;;) {
                    if (tid == 0) item_s = (long long)atomicAdd(a.item_ctr + (pc % 3), 1u);
                    __syncthreads();
                    const long long item = item_s;
                    __syncthreads();
                    if (item >= nitems) break;
                    const int fl = (int)(item / per_frame);
                    const int tt = (int)(item - (long long)fl * per_frame);
                    const int tc = tt / ntr, tr = tt - tc * ntr;
                    const int rs = off - (off > 0 ? GT_T : 0) + tr * GT_T, cs = off - (off > 0 ? GT_T : 0) + tc * GT_T;
                    const int R0 = max(rs, 0), R1 = min(rs + GT_T, rows), C0 = max(cs, 0), C1 = min(cs + GT_T, cols);
                    if (R1 <= R0 || C1 <= C0) continue;           // uniform over the CTA
                    const int TR = R1 - R0, TC = C1 - C0;
                    const float* ug = a.U + (size_t)(f0 + fl) * a.ld;
                    float* tg = a.tot + (size_t)fl * a.ld;
                    float* xig = a.xi + (size_t)fl * nw * 9;
                    for (int idx = tid; idx < TR * TC; idx += GT_THREADS) {
                        const int c = idx / TR, r = idx - c * TR;
                        const size_t p = (size_t)(C0 + c) * rows + R0 + r;
                        us[c * GT_PITCH + r] = ug[p];
                        ts[c * GT_PITCH + r] = first ? 0.f : tg[p];
                    }
                    for (int idx = tid; idx < GT_T * GT_T; idx += GT_THREADS) {
                        const int b = idx / GT_T, aa = idx - b * GT_T;
                        const int wi = R0 + aa, wj = C0 + b;
                        float rad = -1.f;
                        if (aa < TR && b < TC && wi < nwi && wj < nwj) {
                            int i0, j0, hh, ww;
                            gt_geometry(ctr, rows, cols, wi, wj, i0, j0, hh, ww);
                            if (hh > 0 && ww > 0 && i0 >= R0 && i0 + hh <= R1 && j0 >= C0 && j0 + ww <= C1) {
                                const long long widx = (long long)wj * nwi + wi;
                                const float eta_w = ctr ? a.eta[(size_t)(f0 + fl) * a.eta_stride + widx] : (a.eta != nullptr ? a.eta[widx] : 1.f);
                                if (!ctr || eta_w > 0.f) rad = a.lam * eta_w;
                            }
                        }
                        rads[b * GT_PITCH + aa] = rad;
                    }
                    __syncthreads();
                    for (int idx = tid; idx < TC * TR * 9; idx += GT_THREADS) {
                        const int b = idx / (TR * 9), rem = idx - b * (TR * 9), aa = rem / 9, e = rem - aa * 9;
                        if (rads[b * GT_PITCH + aa] >= 0.f) {
                            float v = 0.f;
                            bool have = outer > 0;
                            if (!have && ph > 0) {                // first outer iteration: written only if an earlier phase owned it
                                int i0, j0, hh, ww;
                                gt_geometry(ctr, rows, cols, R0 + aa, C0 + b, i0, j0, hh, ww);
                                for (int q = 0; q < ph; ++q)
                                    have = have || (gt_inside(i0, i0 + hh - 1, q * GT_SHIFT) && gt_inside(j0, j0 + ww - 1, q * GT_SHIFT));
                            }
                            if (have) v = xig[((size_t)(C0 + b) * nwi + R0 + aa) * 9 + e];
                            xis[(b * GT_PITCH + aa) * 9 + e] = v;
                        }
                    }
                    __syncthreads();
                    float tile_ch = 0.f;
                    for (int sw = 0; sw < GT_INNER; ++sw) {
                        float ch = 0.f;
                        for (int col = 0; col < 9; ++col) {
                            const int ci = col % 3, cj = col / 3;
                            const int a0 = ((ci - R0) % 3 + 3) % 3, b0 = ((cj - C0) % 3 + 3) % 3;
                            const int na = (TR - a0 + 2) / 3, nb = (TC - b0 + 2) / 3;
                            for (int q = tid; q < na * nb; q += GT_THREADS) {
                                const int qb = q / na;
                                const int aa = a0 + 3 * (q - qb * na), b = b0 + 3 * qb;
                                const float radius = rads[b * GT_PITCH + aa];
                                if (radius < 0.f) continue;
                                int i0, j0, hh, ww;
                                gt_geometry(ctr, rows, cols, R0 + aa, C0 + b, i0, j0, hh, ww);
                                float* xw = xis + (b * GT_PITCH + aa) * 9;
                                const int po = (j0 - C0) * GT_PITCH + (i0 - R0);
                                float r[9], ar[9], xo[9];
                                float sabs = 0.f, wscale = 0.f;
#pragma unroll
                                for (int c = 0; c < 3; ++c)
#pragma unroll
                                    for (int dr = 0; dr < 3; ++dr) {
                                        const int e = c * 3 + dr;
                                        float val = 0.f, x0 = 0.f;
                                        if ((dr < hh) && (c < ww)) {
                                            const float uu = us[po + c * GT_PITCH + dr];
                                            const float tt0 = ts[po + c * GT_PITCH + dr];
                                            x0 = xw[e]; val = uu - tt0 + x0;
                                            wscale = fmaxf(wscale, fmaxf(fabsf(uu), fmaxf(fabsf(x0), fabsf(tt0))));
                                        }
                                        r[e] = val; ar[e] = fabsf(val); xo[e] = x0; sabs += fabsf(val);
                                    }
                                float theta = 0.f;
                                if (sabs > radius) theta = ss_clip_level9(ar, radius);        // depth-7 network: this loop is latency bound
                                float dmax = 0.f;
#pragma unroll
                                for (int e = 0; e < 9; ++e) {
                                    r[e] = copysignf(fmaxf(ar[e] - theta, 0.f), r[e]);                    // projection on the l1 ball
                                    dmax = fmaxf(dmax, fabsf(r[e] - xo[e]));
                                }
                                // Dead band of ~2 ulp of the operands: with three alternating tilings the fp32 iteration does not end in a
                                // bit-exact fixed point but in a limit cycle of 1-2 ulp changes, and each of them would add a rounding error
                                // to tot (a random walk: 7e-6 after 4000 outer iterations in the CPU emulation of this schedule).  A window
                                // whose projection moved by no more than that keeps its dual -- measured against the STORED dual, so slow
                                // systematic changes still accumulate and get applied.
                                if (dmax > 2.4e-7f * wscale) {
#pragma unroll
                                    for (int c = 0; c < 3; ++c)
#pragma unroll
                                        for (int dr = 0; dr < 3; ++dr) {
                                            const int e = c * 3 + dr;
                                            if ((dr < hh) && (c < ww)) {
                                                xw[e] = r[e];
                                                ts[po + c * GT_PITCH + dr] += r[e] - xo[e];
                                            }
                                        }
                                    // ... and it takes more than count_factor dead bands to keep the iteration going: among the 6e7 windows of
                                    // a 1080p clip a few keep trading 3-10 ulp with their neighbours for ever (theta sums nine values), which
                                    // held every call at the outer-iteration cap
                                    if (dmax > a.count_factor * 2.4e-7f * wscale) ch = fmaxf(ch, dmax);
                                }
                            }
                            __syncthreads();
                        }
                        tile_ch = fmaxf(tile_ch, ch);
                        if (!__syncthreads_or(ch > a.tol)) break;
                    }
                    mych = fmaxf(mych, tile_ch);
                    for (int idx = tid; idx < TC * TR * 9; idx += GT_THREADS) {
                        const int b = idx / (TR * 9), rem = idx - b * (TR * 9), aa = rem / 9, e = rem - aa * 9;
                        if (rads[b * GT_PITCH + aa] >= 0.f) xig[((size_t)(C0 + b) * nwi + R0 + aa) * 9 + e] = xis[(b * GT_PITCH + aa) * 9 + e];
                    }
                    for (int idx = tid; idx < TR * TC; idx += GT_THREADS) {
                        const int c = idx / TR, r = idx - c * TR;
                        tg[(size_t)(C0 + c) * rows + R0 + r] = ts[c * GT_PITCH + r];
                    }
                    __syncthreads();
                }
                if (ph == 2) {
                    mych = warp_max(mych);
                    if ((tid & 31) == 0 && mych > 0.f) atomicMax(a.change_bits + (oc % 3), __float_as_uint(mych));
                }
                grid.sync();
                if (blockIdx.x == 0 && tid == 0) a.item_ctr[(pc + 2) % 3] = 0u;      // next used two phases from now
                ++pc;
            }
            const float chg = __uint_as_float(*((volatile unsigned int*)(a.change_bits + (oc % 3))));
            if (blockIdx.x == 0 && tid == 0) a.change_bits[(oc + 2) % 3] = 0u;      // next written two outer iterations from now
            ++outer; ++oc;
            if (chg <= a.tol) break;
        }
        most = max(most, outer);
        // V = U - tot for the frames of this chunk (pixels no window covers have tot = 0: identity)
        const long long m = (long long)rows * cols;
        for (long long i = gid; i < (long long)nf * m; i += gsz) {
            const long long fl = i / m, p = i - fl * m;
            a.V[(size_t)(f0 + fl) * a.ld + p] = a.U[(size_t)(f0 + fl) * a.ld + p] - a.tot[(size_t)fl * a.ld + p];
        }
        grid.sync();                                             // tot and xi are reused by the next chunk
    }
    if (blockIdx.x == 0 && tid == 0 && a.sweeps_out != nullptr) {
        *a.sweeps_out = most;
        if (a.stats != nullptr) { a.stats[0] += most; a.stats[1] += 1; if (most >= a.max_outer) a.stats[2] += 1; }
    }
}

// workspace of launch_prox_graph3: duals xi (whole frames, capped) and per-pixel dual sums tot (one row of ld floats per frame held)
void prox_graph3_workspace(int rows, int cols, int n, long long ld, int center, long long* xi_floats, long long* tot_floats) {
    const long long nw = center ? (long long)rows * cols : (long long)(rows - std::min(3, rows) + 1) * (cols - std::min(3, cols) + 1);
    long long cap_mb = 8192;
    if (const char* e = getenv("BSUB_GRAPH_XI_MB")) cap_mb = std::max(1LL, atoll(e));
    const long long cap = cap_mb * (1LL << 20) / 4;
    const long long frames = std::max(1LL, std::min<long long>(n, cap / std::max(1LL, nw * 9)));
    *xi_floats = frames * nw * 9 + 16;            // + the three work counters of the tile kernel
    *tot_floats = frames * ld;
}

int launch_prox_graph3(const float* U, float* V, float* xi, long long xi_floats, float* tot, const float* eta, long long ld, int rows, int cols,
                       int n, float lam, int max_sweeps, float tol, int* sweeps_out, const DevState* st, cudaStream_t s, int center,
                       long long eta_stride) {
    if (xi == nullptr || tot == nullptr) { set_error("prox_graph3: missing workspace"); return -1; }
    if (sweeps_out == nullptr) { set_error("prox_graph3: the caller's int[8] status block is required"); return -1; }
    static int blocks_per_sm = 0, num_sms = 0;
    static unsigned long long attr_devs = 0;
    if (first_call_on_device(&attr_devs))
        BSUB_CUDA_CHECK(cudaFuncSetAttribute(prox_graph3_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GT_SMEM));
    if (blocks_per_sm == 0) {
        int dev = 0;
        BSUB_CUDA_CHECK(cudaGetDevice(&dev));
        BSUB_CUDA_CHECK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
        BSUB_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, prox_graph3_tile_kernel, GT_THREADS, GT_SMEM));
        if (blocks_per_sm < 1) { set_error("prox_graph3: kernel does not fit"); return -1; }
    }
    if (center && eta == nullptr) { set_error("prox_graph3: centre mode needs the per-frame eta map"); return -1; }
    GraphTileArgs a;
    a.U = U; a.V = V; a.xi = xi; a.tot = tot; a.eta = eta; a.ld = ld; a.rows = rows; a.cols = cols; a.n = n; a.lam = lam;
    a.max_outer = max_sweeps; a.tol = tol; a.sweeps_out = sweeps_out; a.st = st;
    // sweeps_out is an int[8] owned by the caller: [0] outer iterations used, [1..3] the rotating change flags (per
    // solver handle, so that handles running concurrently on different streams do not share them), [4..6] running totals
    a.change_bits = reinterpret_cast<unsigned int*>(sweeps_out + 1);
    a.stats = sweeps_out + 4;                                              // the caller's int[8]: [4..6] running totals
    a.count_factor = GT_COUNT_FACTOR;
    a.center = center; a.eta_stride = eta_stride;
    a.nwi = center ? rows : rows - std::min(3, rows) + 1;
    a.nwj = center ? cols : cols - std::min(3, cols) + 1;
    const long long per_frame = (long long)a.nwi * a.nwj * 9;
    if (xi_floats < per_frame + 16) { set_error("prox_graph3: dual buffer smaller than one frame"); return -1; }
    a.chunk = (int)std::max(1LL, std::min<long long>(n, (xi_floats - 16) / std::max(1LL, per_frame)));
    a.item_ctr = reinterpret_cast<unsigned int*>(xi + (xi_floats - 16));
    const long long tiles = (long long)((rows + GT_T - 1) / GT_T + 1) * ((cols + GT_T - 1) / GT_T + 1) * std::min(n, a.chunk);
    long long want = std::min<long long>(tiles, (long long)blocks_per_sm * num_sms);
    if (want < 1) want = 1;
    void* args[] = {&a};
    BSUB_CUDA_CHECK(cudaLaunchCooperativeKernel((void*)prox_graph3_tile_kernel, dim3((unsigned)want), dim3(GT_THREADS), args, GT_SMEM, s));
    return 0;
}

}  // namespace bsub
