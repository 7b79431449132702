// rpca_batch.cu -- the stage-2 saliency batch (SURVEY.md 8f row 2): hundreds of independent small rank-capped robust PCAs, one
// per X-T / Y-T slice of the video (/root/reference/computeRPCADecomposition.py:12-48: compute_RPCA fits a max_rank = 1 RPCA to
// every image_array[i, :, :]).
//
// The reference delegates those fits to the RobustPCA package, which is neither vendored nor pinned nor installable here (and its
// published fixed-penalty iteration does not reach the reference's tolerance under a hard rank cap -- DESIGN.md section 7), so the
// engine of the batch is the reference's OWN l1 RPCA, inexact_alm_rpca (/root/reference/lsd_improvement.py:123-196), with the
// rank of L capped at max_rank = 1 like RobustPCA(max_rank=1):
//     lambda = 1/(sqrt(max(m, n)) delta);  Y0 = D / max(||D||_2, ||D||_inf / lambda);  mu0 = 1.25/||D||_2;  rho = 1.2
//     repeat:  L = SVT_{1/mu}(D - S + Y/mu) cut to rank 1;  S = shrink(D - L + Y/mu, lambda/mu);  Z = D - L - S;  Y += mu Z;
//              mu *= rho;  stop when ||Z||_F / ||D||_F < tol (or sum |Z| <= tol_l1, the criterion compute_RPCA passes)
// With rank <= 1 the thresholding needs the leading singular triplet only: a warm-started power iteration (one or two steps per
// ALM iteration once it has locked on).
//
// One thread-block cluster per slice; every CTA keeps a band of rows of D, Q = Y/mu, S and X = D - S + Q in SHARED MEMORY for the
// whole solve, so the iteration never touches HBM (a 240 x 200 slice is 192 KB per array; the 560 slices of a 320 x 240 x 200 clip
// are a few waves of shared-memory sweeps).  Cross-CTA sums (X^T u, ||X v||^2, ||Z||^2, sum |Z|, ...) go through distributed shared
// memory: every CTA pushes its partials into a slot of every peer, one hardware cluster barrier, every CTA adds the slots in rank
// order -- all CTAs of a cluster take bit-identical decisions (deterministic, no atomics).
//
// Slices that do not fit that way (more than 640 columns, or too many rows for 8 CTAs of shared memory) take a second kernel with
// the same iteration whose state lives in GLOBAL memory (rpca_rank1_large_kernel below): S is iterated in the caller's S buffer,
// Q in the caller's L buffer (L is written from the rank-1 pair at the end), and X = D - S + Q is recomputed in every power sweep.
#include <cooperative_groups.h>
#include <math.h>
#include <algorithm>
#include "common.cuh"
#include "../../include/bsub_b200.h"

namespace cg = cooperative_groups;

namespace bsub {

constexpr int RB_THREADS = 256, RB_WARPS = 8, RB_KT = 20;          // columns <= 32 * RB_KT = 640 (one instantiation per 128 columns)
constexpr int RB_MAXC = 8, RB_NSCAL = 4;                           // scalars that travel with a push: [0] ||Xv||^2 [1] sum Z^2 [2] sum |Z| [3] spare
constexpr size_t RB_SMEM_CAP = 220 * 1024;

struct RpcaBatchArgs {
    const float* D; float* L; float* S;        // [batch][rows][cols]
    int batch, rows, cols, C, rl;              // rl = rows per CTA
    int tr;                                    // large kernel: rows per staged tile of a power sweep (a multiple of RB_WARPS)
    double delta, rho, tol, tol_l1;            // tol_l1 <= 0: unused
    int max_iter, max_power;
    int* iters; float* err; int* rank;
};

struct RbSmem {
    float *Ds, *Qs, *Ss, *Xs, *v, *vp, *u, *wpart, *part, *slots, *red;
    int t, rl, nr, C, my, width, buf;
};

__device__ __forceinline__ float rb_block_sum(float x, float* red8, int warp, int lane) {
    x = warp_sum(x);
    __syncthreads();
    if (lane == 0) red8[warp] = x;
    __syncthreads();
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < RB_WARPS; ++w) s += red8[w];
    return s;
}
__device__ __forceinline__ float rb_block_max(float x, float* red8, int warp, int lane) {
    x = warp_max(x);
    __syncthreads();
    if (lane == 0) red8[warp] = x;
    __syncthreads();
    float s = red8[0];
#pragma unroll
    for (int w = 1; w < RB_WARPS; ++w) s = fmaxf(s, red8[w]);
    return s;
}

// push part[0 .. count) into slot [buf][my] of every CTA of the cluster, barrier; afterwards slots[buf][c][.] hold everyone's values
__device__ __forceinline__ void rb_exchange(cg::cluster_group& cl, RbSmem& m, int first, int count) {
    for (int idx = threadIdx.x; idx < count * m.C; idx += blockDim.x) {
        const int peer = idx / count, j = first + idx - peer * count;
        float* dst = cl.map_shared_rank(m.slots, peer) + ((size_t)m.buf * m.C + m.my) * m.width + j;
        *dst = m.part[j];
    }
    cl.sync();
}
__device__ __forceinline__ float rb_slot_sum(const RbSmem& m, int j) {
    float s = 0.f;
    for (int c = 0; c < m.C; ++c) s += m.slots[((size_t)m.buf * m.C + c) * m.width + j];
    return s;
}
__device__ __forceinline__ float rb_slot_max(const RbSmem& m, int j) {
    float s = m.slots[((size_t)m.buf * m.C) * m.width + j];
    for (int c = 1; c < m.C; ++c) s = fmaxf(s, m.slots[((size_t)m.buf * m.C + c) * m.width + j]);
    return s;
}

// power iteration on X from the current v: returns ||X vp||^2 of the last sweep; (u, vp) is then an exact pair u = X vp
template <int KT>
__device__ float rb_power(cg::cluster_group& cl, RbSmem& m, int max_steps, float eps) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, t = m.t;
    float sigma2 = 0.f;
    for (int step = 0; step < max_steps; ++step) {
        float vreg[KT], wacc[KT];
#pragma unroll
        for (int k = 0; k < KT; ++k) { const int j = lane + 32 * k; vreg[k] = (j < t) ? m.v[j] : 0.f; wacc[k] = 0.f; }
        float uu = 0.f;
        for (int i = warp; i < m.nr; i += RB_WARPS) {
            const float* xr = m.Xs + (size_t)i * t;
            float x[KT], dot = 0.f;
#pragma unroll
            for (int k = 0; k < KT; ++k) { const int j = lane + 32 * k; x[k] = (j < t) ? xr[j] : 0.f; dot = fmaf(x[k], vreg[k], dot); }
            dot = warp_sum(dot);
            if (lane == 0) m.u[i] = dot;
            uu = fmaf(dot, dot, uu);
#pragma unroll
            for (int k = 0; k < KT; ++k) wacc[k] = fmaf(dot, x[k], wacc[k]);
        }
#pragma unroll
        for (int k = 0; k < KT; ++k) { const int j = lane + 32 * k; if (j < t) m.wpart[(size_t)warp * t + j] = wacc[k]; }
        if (lane == 0) m.red[warp] = uu;                        // all lanes of a warp hold the same uu
        __syncthreads();
        for (int j = threadIdx.x; j < t; j += blockDim.x) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < RB_WARPS; ++w) s += m.wpart[(size_t)w * t + j];
            m.part[j] = s;
            m.vp[j] = m.v[j];
        }
        if (threadIdx.x == 0) { float s = 0.f; for (int w = 0; w < RB_WARPS; ++w) s += m.red[w]; m.part[t] = s; }
        __syncthreads();
        rb_exchange(cl, m, 0, t + 1);
        // every CTA: w = sum of the slots in rank order, v <- w / ||w||, largest change of an entry
        float nrm2 = 0.f;
        for (int j = threadIdx.x; j < t; j += blockDim.x) {
            const float s = rb_slot_sum(m, j);
            m.part[j] = s;
            nrm2 = fmaf(s, s, nrm2);
        }
        sigma2 = rb_slot_sum(m, t);
        m.buf ^= 1;
        const float tot = rb_block_sum(nrm2, m.red, warp, lane);
        const float inv = (tot > 0.f) ? rsqrtf(tot) : 0.f;
        float delta = 0.f;
        for (int j = threadIdx.x; j < t; j += blockDim.x) {
            const float vn = m.part[j] * inv;
            delta = fmaxf(delta, fabsf(vn - m.v[j]));
            m.v[j] = vn;
        }
        const float dmax = rb_block_max(delta, m.red + 8, warp, lane);
        if (dmax <= eps || !(tot > 0.f)) break;                 // uniform over the cluster: identical inputs, identical order
    }
    return sigma2;
}

template <int KT>
__global__ void __launch_bounds__(RB_THREADS, 1) rpca_rank1_batch_kernel(RpcaBatchArgs a) {
    cg::cluster_group cl = cg::this_cluster();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    RbSmem m;
    m.C = a.C; m.my = (int)cl.block_rank(); m.t = a.cols; m.rl = a.rl; m.width = a.cols + RB_NSCAL; m.buf = 0;
    const int t = m.t, rl = m.rl;
    extern __shared__ __align__(16) float rb_smem[];
    m.Ds = rb_smem;                                            // [rl][t]
    m.Qs = m.Ds + (size_t)rl * t;
    m.Ss = m.Qs + (size_t)rl * t;
    m.Xs = m.Ss + (size_t)rl * t;
    m.v = m.Xs + (size_t)rl * t;                               // [t]   current right vector (unit)
    m.vp = m.v + t;                                            // [t]   the vector the last sweep used
    m.u = m.vp + t;                                            // [rl]  X vp of my rows
    m.wpart = m.u + rl;                                        // [RB_WARPS][t]
    m.part = m.wpart + (size_t)RB_WARPS * t;                   // [width] this CTA's partials
    m.slots = m.part + m.width;                                // [2][C][width]
    m.red = m.slots + (size_t)2 * m.C * m.width;               // [24] block reductions
    const int r0 = m.my * rl;
    m.nr = max(0, min(a.rows, r0 + rl) - r0);
    const int nr = m.nr;
    const int num_clusters = (int)(gridDim.x / m.C), cid = (int)(blockIdx.x / m.C);
    const double lambda = 1.0 / (sqrt((double)max(a.rows, a.cols)) * a.delta);

    for (int b = cid; b < a.batch; b += num_clusters) {
        const size_t goff = (size_t)b * a.rows * t + (size_t)r0 * t;
        // ---- load D; ||D||_F^2 and the largest row sum of |D| (NumPy's inf-norm, lsd_improvement.py:139)
        float fro = 0.f;
        for (int idx = threadIdx.x; idx < rl * t; idx += blockDim.x) {
            const float d = (idx < nr * t) ? a.D[goff + idx] : 0.f;
            m.Ds[idx] = d; m.Xs[idx] = d; m.Qs[idx] = 0.f; m.Ss[idx] = 0.f;
            fro = fmaf(d, d, fro);
        }
        const float v0 = rsqrtf((float)t);
        for (int j = threadIdx.x; j < t; j += blockDim.x) m.v[j] = v0;
        __syncthreads();
        float rmax = 0.f;
        for (int i = warp; i < nr; i += RB_WARPS) {
            float s = 0.f;
            for (int j = lane; j < t; j += 32) s += fabsf(m.Ds[(size_t)i * t + j]);
            rmax = fmaxf(rmax, warp_sum(s));
        }
        const float fro_b = rb_block_sum(fro, m.red, warp, lane);
        const float rmax_b = rb_block_max(rmax, m.red + 8, warp, lane);
        if (threadIdx.x == 0) { m.part[t + 1] = fro_b; m.part[t + 2] = rmax_b; }
        __syncthreads();
        rb_exchange(cl, m, t + 1, 2);
        const double normD2 = (double)rb_slot_sum(m, t + 1);
        const double norm_rowsum = (double)rb_slot_max(m, t + 2);
        m.buf ^= 1;
        // ---- ||D||_2 by power iteration on X = D
        const double norm_two = sqrt((double)rb_power<KT>(cl, m, 4 * a.max_power, 1e-7f));
        int it = 0, rank = 0, converged = 0;
        float err = 0.f;
        if (norm_two > 0.0) {
            const double dual_norm = fmax(norm_two, norm_rowsum / lambda);
            double mu = 1.25 / norm_two;
            // Y0 = D / dual_norm: Q = Y0 / mu0, X = D + Q
            const float q0 = (float)(1.0 / (dual_norm * mu));
            for (int idx = threadIdx.x; idx < nr * t; idx += blockDim.x) {
                const float d = m.Ds[idx];
                m.Qs[idx] = q0 * d;
                m.Xs[idx] = fmaf(q0, d, d);
            }
            __syncthreads();
            for (it = 1; it <= a.max_iter; ++it) {
                // ---- leading singular triplet of X (warm start), thresholded at 1/mu, rank cap 1
                const float sigma = sqrtf(rb_power<KT>(cl, m, a.max_power, 3e-7f));
                const float inv_mu = (float)(1.0 / mu), thr = (float)(lambda / mu);
                rank = (sigma > inv_mu) ? 1 : 0;
                const float cfac = rank ? (sigma - inv_mu) / sigma : 0.f;
                const float inv_rho = (float)(1.0 / a.rho);
                // ---- S = shrink(D - L + Q), Z = D - L - S, Y += mu Z, mu *= rho  =>  Q <- (Q + Z) / rho;  X = D - S + Q
                float zz = 0.f, za = 0.f;
                for (int idx = threadIdx.x; idx < nr * t; idx += blockDim.x) {
                    const int i = idx / t, j = idx - i * t;
                    const float l = cfac * m.u[i] * m.vp[j];
                    const float d = m.Ds[idx], q = m.Qs[idx];
                    const float g = d - l + q;
                    const float s = copysignf(fmaxf(fabsf(g) - thr, 0.f), g);
                    const float z = d - l - s;
                    zz = fmaf(z, z, zz);
                    za += fabsf(z);
                    m.Ss[idx] = s;
                    const float qn = (q + z) * inv_rho;
                    m.Qs[idx] = qn;
                    m.Xs[idx] = d - s + qn;
                }
                const float zz_b = rb_block_sum(zz, m.red, warp, lane);
                const float za_b = rb_block_sum(za, m.red + 8, warp, lane);
                if (threadIdx.x == 0) { m.part[t + 1] = zz_b; m.part[t + 2] = za_b; }
                __syncthreads();
                rb_exchange(cl, m, t + 1, 2);
                const float zz_t = rb_slot_sum(m, t + 1), za_t = rb_slot_sum(m, t + 2);
                m.buf ^= 1;
                mu = fmin(mu * a.rho, mu * 1e7);
                err = (float)(sqrt((double)zz_t) / sqrt(normD2));
                if ((double)err < a.tol || (a.tol_l1 > 0.0 && (double)za_t <= a.tol_l1)) { converged = 1; break; }
            }
            if (it > a.max_iter) it = a.max_iter;
        }
        // ---- outputs: the L and S of the last iteration.  L = cfac u vp^T with the pair of the last sweep; the threshold of that
        // iteration is recovered from mu (advanced once since)
        __syncthreads();
        if (norm_two > 0.0 && it > 0) {
            // recompute the factor of the last iteration: sigma = ||u|| (cluster sum of the squares of u)
            float uu = 0.f;
            for (int i = threadIdx.x; i < nr; i += blockDim.x) uu = fmaf(m.u[i], m.u[i], uu);
            const float uu_b = rb_block_sum(uu, m.red, warp, lane);
            if (threadIdx.x == 0) m.part[t + 1] = uu_b;
            __syncthreads();
            rb_exchange(cl, m, t + 1, 1);
            const float sigma = sqrtf(rb_slot_sum(m, t + 1));
            m.buf ^= 1;
            double mu_last = 1.25 / norm_two;
            for (int k = 1; k < it; ++k) mu_last = fmin(mu_last * a.rho, mu_last * 1e7);
            const float inv_mu = (float)(1.0 / mu_last);
            const float cfac = (sigma > inv_mu) ? (sigma - inv_mu) / sigma : 0.f;
            for (int idx = threadIdx.x; idx < nr * t; idx += blockDim.x) {
                const int i = idx / t, j = idx - i * t;
                a.L[goff + idx] = cfac * m.u[i] * m.vp[j];
                a.S[goff + idx] = m.Ss[idx];
            }
        } else {
            for (int idx = threadIdx.x; idx < nr * t; idx += blockDim.x) { a.L[goff + idx] = 0.f; a.S[goff + idx] = 0.f; }
        }
        if (m.my == 0 && threadIdx.x == 0) {
            a.iters[b] = converged ? it : -it;                  // negative: max_iter reached without meeting the tolerance
            a.err[b] = err;
            a.rank[b] = rank;
        }
        __syncthreads();
        cl.sync();                                              // nobody starts the next slice (and its pushes) before everyone is out
    }
}

// ---------------------------------------------------------------------------------------------------------------------------------
// Large slices: the same iteration with D, S and Q = Y/mu in global memory (S in the caller's S, Q in the caller's L).  One cluster per
// slice, a band of rows per CTA; only the vectors (v, vp, the band's u), a staged tile of X rows and the partials live in shared memory.
// A power sweep reads D, S, Q once (12 B per element) and rebuilds X = (D - S) + Q on the fly, rounded like the shared-memory kernel's
// stored X.  Every sum has a fixed order that depends on the slice shape only (u_i: lanes stride the columns then a warp tree; the
// band's X^T u: rows in ascending order per column; cluster sums: CTAs in rank order), so a slice's result does not depend on where in
// the batch it sits or on how many clusters run.
constexpr int RG_MAXDIM = 4096, RG_TILE = 32;

struct RgSmem {
    float *v, *vp, *u, *part, *tile, *red;
    int t, width, nr, C, tr, buf;
};

// Cluster sum (CTAs in rank order) / max of part[buf][j].  Every CTA READS its peers' partials over DSMEM after the cluster barrier
// that follows their writes, so a CTA needs 2 x (cols + RB_NSCAL) floats of exchange space whatever the cluster size.  A CTA writes
// buffer b again only after the next exchange's barrier, which no CTA reaches before it has finished reading buffer b.
__device__ __forceinline__ float rg_sum(cg::cluster_group& cl, const RgSmem& m, int j) {
    float* p = m.part + (size_t)m.buf * m.width + j;
    float s = 0.f;
    for (int c = 0; c < m.C; ++c) s += *cl.map_shared_rank(p, c);
    return s;
}
__device__ __forceinline__ float rg_max(cg::cluster_group& cl, const RgSmem& m, int j) {
    float* p = m.part + (size_t)m.buf * m.width + j;
    float s = *cl.map_shared_rank(p, 0);
    for (int c = 1; c < m.C; ++c) s = fmaxf(s, *cl.map_shared_rank(p, c));
    return s;
}
__device__ __forceinline__ double rg_block_sum(double x, double* red8, int warp, int lane) {
    x = warp_sum(x);
    __syncthreads();
    if (lane == 0) red8[warp] = x;
    __syncthreads();
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < RB_WARPS; ++w) s += red8[w];
    return s;
}

__device__ __forceinline__ float rg_x(const float* __restrict__ D, const float* S, const float* Q, size_t o, bool d_only) {
    return d_only ? D[o] : (D[o] - S[o]) + Q[o];
}

// rb_power on X = D - S + Q (or X = D) of the rows [goff, goff + nr * t): returns ||X vp||^2 of the last sweep, (u, vp) an exact pair
__device__ float rg_power(cg::cluster_group& cl, RgSmem& m, const float* __restrict__ D, const float* S, const float* Q, size_t goff,
                          bool d_only, int max_steps, float eps) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, t = m.t;
    float sigma2 = 0.f;
    for (int step = 0; step < max_steps; ++step) {
        float* part = m.part + (size_t)m.buf * m.width;
        for (int j = threadIdx.x; j < t; j += blockDim.x) { part[j] = 0.f; m.vp[j] = m.v[j]; }
        float uu = 0.f;
        for (int i0 = 0; i0 < m.nr; i0 += m.tr) {
            const int nt = min(m.tr, m.nr - i0);
            // u_i = X_i. v, warp per row; the row is staged for the X^T u pass
            for (int r = warp; r < nt; r += RB_WARPS) {
                const size_t o = goff + (size_t)(i0 + r) * t;
                float* xr = m.tile + (size_t)r * t;
                float dot = 0.f;
#pragma unroll 4
                for (int j = lane; j < t; j += 32) {
                    const float x = rg_x(D, S, Q, o + j, d_only);
                    xr[j] = x;
                    dot = fmaf(x, m.v[j], dot);
                }
                dot = warp_sum(dot);
                if (lane == 0) m.u[i0 + r] = dot;
                uu = fmaf(dot, dot, uu);
            }
            __syncthreads();
            // X^T u of the band, thread per column, rows in ascending order
            for (int j = threadIdx.x; j < t; j += blockDim.x) {
                float acc = part[j];
                for (int r = 0; r < nt; ++r) acc = fmaf(m.tile[(size_t)r * t + j], m.u[i0 + r], acc);
                part[j] = acc;
            }
            __syncthreads();
        }
        const float uu_b = rb_block_sum(lane == 0 ? uu : 0.f, m.red, warp, lane);   // all lanes of a warp hold the same uu
        if (threadIdx.x == 0) part[t] = uu_b;
        cl.sync();
        // every CTA: w = cluster sum, v <- w / ||w||, largest change of an entry
        float nrm2 = 0.f;
        for (int j = threadIdx.x; j < t; j += blockDim.x) {
            const float s = rg_sum(cl, m, j);
            m.v[j] = s;
            nrm2 = fmaf(s, s, nrm2);
        }
        sigma2 = rg_sum(cl, m, t);
        m.buf ^= 1;
        const float tot = rb_block_sum(nrm2, m.red, warp, lane);
        const float inv = (tot > 0.f) ? rsqrtf(tot) : 0.f;
        float delta = 0.f;
        for (int j = threadIdx.x; j < t; j += blockDim.x) {
            const float vn = m.v[j] * inv;
            delta = fmaxf(delta, fabsf(vn - m.vp[j]));
            m.v[j] = vn;
        }
        const float dmax = rb_block_max(delta, m.red + 8, warp, lane);
        if (dmax <= eps || !(tot > 0.f)) break;                 // uniform over the cluster: identical inputs, identical order
    }
    return sigma2;
}

__global__ void __launch_bounds__(RB_THREADS, 1) rpca_rank1_large_kernel(RpcaBatchArgs a) {
    cg::cluster_group cl = cg::this_cluster();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    RgSmem m;
    m.C = a.C; m.t = a.cols; m.width = a.cols + RB_NSCAL; m.tr = a.tr; m.buf = 0;
    const int my = (int)cl.block_rank(), t = m.t;
    extern __shared__ __align__(16) float rg_smem[];
    double* redd = reinterpret_cast<double*>(rg_smem);         // [8]   double block sums
    m.red = rg_smem + 16;                                      // [16]  float block sums / maxima
    m.v = m.red + 16;                                          // [t]
    m.vp = m.v + t;                                            // [t]
    m.part = m.vp + t;                                         // [2][width]
    m.u = m.part + (size_t)2 * m.width;                        // [rl]
    m.tile = m.u + a.rl;                                       // [tr][t]
    const int r0 = my * a.rl;
    m.nr = max(0, min(a.rows, r0 + a.rl) - r0);
    const int nr = m.nr;
    const int num_clusters = (int)(gridDim.x / m.C), cid = (int)(blockIdx.x / m.C);
    const double lambda = 1.0 / (sqrt((double)max(a.rows, a.cols)) * a.delta);
    const float* __restrict__ D = a.D;
    float* S = a.S;
    float* Q = a.L;

    for (int b = cid; b < a.batch; b += num_clusters) {
        const size_t goff = (size_t)b * a.rows * t + (size_t)r0 * t;
        // ---- ||D||_F^2 and the largest row sum of |D|
        double fro = 0.0;
        float rmax = 0.f;
        for (int i = warp; i < nr; i += RB_WARPS) {
            const size_t o = goff + (size_t)i * t;
            float s = 0.f;
            for (int j = lane; j < t; j += 32) {
                const float d = D[o + j];
                s += fabsf(d);
                fro = fma((double)d, (double)d, fro);
            }
            rmax = fmaxf(rmax, warp_sum(s));
        }
        const double fro_b = rg_block_sum(fro, redd, warp, lane);
        const float rmax_b = rb_block_max(rmax, m.red + 8, warp, lane);
        float* part = m.part + (size_t)m.buf * m.width;
        if (threadIdx.x == 0) { part[t + 1] = (float)fro_b; part[t + 2] = rmax_b; }
        const float v0 = rsqrtf((float)t);
        for (int j = threadIdx.x; j < t; j += blockDim.x) m.v[j] = v0;
        cl.sync();
        const double normD2 = (double)rg_sum(cl, m, t + 1);
        const double norm_rowsum = (double)rg_max(cl, m, t + 2);
        m.buf ^= 1;
        // ---- ||D||_2 by power iteration on X = D
        const double norm_two = sqrt((double)rg_power(cl, m, D, S, Q, goff, true, 4 * a.max_power, 1e-7f));
        int it = 0, rank = 0, converged = 0;
        float err = 0.f;
        if (norm_two > 0.0) {
            const double dual_norm = fmax(norm_two, norm_rowsum / lambda);
            double mu = 1.25 / norm_two;
            // Y0 = D / dual_norm: Q = Y0 / mu0, S = 0.  Row i, column j is read and written by warp i % RB_WARPS, lane j % 32 in every
            // pass of the solve, so the passes need no barrier between them for the global arrays.
            const float q0 = (float)(1.0 / (dual_norm * mu));
            for (int i = warp; i < nr; i += RB_WARPS) {
                const size_t o = goff + (size_t)i * t;
                for (int j = lane; j < t; j += 32) { S[o + j] = 0.f; Q[o + j] = q0 * D[o + j]; }
            }
            for (it = 1; it <= a.max_iter; ++it) {
                // ---- leading singular triplet of X (warm start), thresholded at 1/mu, rank cap 1
                const float sigma = sqrtf(rg_power(cl, m, D, S, Q, goff, false, a.max_power, 3e-7f));
                const float inv_mu = (float)(1.0 / mu), thr = (float)(lambda / mu);
                rank = (sigma > inv_mu) ? 1 : 0;
                const float cfac = rank ? (sigma - inv_mu) / sigma : 0.f;
                const float inv_rho = (float)(1.0 / a.rho);
                // ---- S = shrink(D - L + Q), Z = D - L - S, Q <- (Q + Z) / rho
                double zz = 0.0, za = 0.0;
                for (int i = warp; i < nr; i += RB_WARPS) {
                    const size_t o = goff + (size_t)i * t;
                    const float cu = cfac * m.u[i];
#pragma unroll 4
                    for (int j = lane; j < t; j += 32) {
                        const float l = cu * m.vp[j];
                        const float d = D[o + j], q = Q[o + j];
                        const float g = d - l + q;
                        const float s = copysignf(fmaxf(fabsf(g) - thr, 0.f), g);
                        const float z = d - l - s;
                        zz = fma((double)z, (double)z, zz);
                        za += (double)fabsf(z);
                        S[o + j] = s;
                        Q[o + j] = (q + z) * inv_rho;
                    }
                }
                const double zz_b = rg_block_sum(zz, redd, warp, lane);
                const double za_b = rg_block_sum(za, redd, warp, lane);
                part = m.part + (size_t)m.buf * m.width;
                if (threadIdx.x == 0) { part[t + 1] = (float)zz_b; part[t + 2] = (float)za_b; }
                cl.sync();
                const float zz_t = rg_sum(cl, m, t + 1), za_t = rg_sum(cl, m, t + 2);
                m.buf ^= 1;
                mu = fmin(mu * a.rho, mu * 1e7);
                err = (float)(sqrt((double)zz_t) / sqrt(normD2));
                if ((double)err < a.tol || (a.tol_l1 > 0.0 && (double)za_t <= a.tol_l1)) { converged = 1; break; }
            }
            if (it > a.max_iter) it = a.max_iter;
        }
        // ---- outputs: S is in place; L = cfac u vp^T of the last iteration overwrites Q
        __syncthreads();
        if (norm_two > 0.0 && it > 0) {
            float uu = 0.f;
            for (int i = threadIdx.x; i < nr; i += blockDim.x) uu = fmaf(m.u[i], m.u[i], uu);
            const float uu_b = rb_block_sum(uu, m.red, warp, lane);
            part = m.part + (size_t)m.buf * m.width;
            if (threadIdx.x == 0) part[t + 1] = uu_b;
            cl.sync();
            const float sigma = sqrtf(rg_sum(cl, m, t + 1));
            m.buf ^= 1;
            double mu_last = 1.25 / norm_two;
            for (int k = 1; k < it; ++k) mu_last = fmin(mu_last * a.rho, mu_last * 1e7);
            const float inv_mu = (float)(1.0 / mu_last);
            const float cfac = (sigma > inv_mu) ? (sigma - inv_mu) / sigma : 0.f;
            for (int i = warp; i < nr; i += RB_WARPS) {
                const size_t o = goff + (size_t)i * t;
                const float cu = cfac * m.u[i];
                for (int j = lane; j < t; j += 32) a.L[o + j] = cu * m.vp[j];
            }
        } else {
            for (int i = warp; i < nr; i += RB_WARPS) {
                const size_t o = goff + (size_t)i * t;
                for (int j = lane; j < t; j += 32) { a.L[o + j] = 0.f; a.S[o + j] = 0.f; }
            }
        }
        if (my == 0 && threadIdx.x == 0) {
            a.iters[b] = converged ? it : -it;                  // negative: max_iter reached without meeting the tolerance
            a.err[b] = err;
            a.rank[b] = rank;
        }
    }
    cl.sync();                                                  // no CTA leaves while a peer may still read its shared memory
}

}  // namespace bsub

using namespace bsub;

// Cluster size: the smallest power of two (at most RB_MAXC and the row count) for which one slice per C SMs keeps the in-flight working
// set (D, S and Q: 3 x rows x cols x 4 B per slice) within the L2; slices in flight: as many clusters as can be co-resident.  Capping
// the clusters further so that the in-flight slices fit the L2 measured slower (DESIGN.md section 4.7).  C and the tile follow from the
// shape and the device only, so no result depends on the batch.
static int rpca_large_launch(RpcaBatchArgs a, int dev, int sms, void* stream) {
    if (a.rows > RG_MAXDIM || a.cols > RG_MAXDIM) {
        set_error("bsub_rpca_rank1_batch_dev: a %d x %d slice is larger than %d x %d", a.rows, a.cols, RG_MAXDIM, RG_MAXDIM);
        return -1;
    }
    int l2 = 0;
    BSUB_CUDA_CHECK(cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev));
    const size_t slice = (size_t)3 * a.rows * a.cols * sizeof(float);
    int C = 1;
    while (C < RB_MAXC && 2 * C <= a.rows && (size_t)(sms / C) * slice > (size_t)l2) C *= 2;
    const int rl = (a.rows + C - 1) / C;
    const size_t fixed = 32 + 2 * (size_t)a.cols + 2 * ((size_t)a.cols + RB_NSCAL) + rl;          // floats before the tile
    const int tr = (int)std::min<size_t>(std::min<size_t>(RG_TILE, (rl + RB_WARPS - 1) / RB_WARPS * RB_WARPS),
                                         (RB_SMEM_CAP / sizeof(float) - fixed) / a.cols) / RB_WARPS * RB_WARPS;
    if (tr < RB_WARPS) { set_error("bsub_rpca_rank1_batch_dev: no tile of a %d x %d slice fits shared memory", a.rows, a.cols); return -1; }
    const size_t smem = (fixed + (size_t)tr * a.cols) * sizeof(float);
    a.C = C; a.rl = rl; a.tr = tr;
    // the attribute is a per-device upper bound shared by every host thread: always the cap, never one shape's size
    BSUB_CUDA_CHECK(cudaFuncSetAttribute(rpca_rank1_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RB_SMEM_CAP));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)C); cfg.blockDim = dim3(RB_THREADS);
    cfg.dynamicSmemBytes = smem; cfg.stream = reinterpret_cast<cudaStream_t>(stream);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int active = 0;
    BSUB_CUDA_CHECK(cudaOccupancyMaxActiveClusters(&active, rpca_rank1_large_kernel, &cfg));
    const int clusters = std::max(1, std::min(a.batch, active));
    cfg.gridDim = dim3((unsigned)(clusters * C));
    BSUB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, rpca_rank1_large_kernel, a));
    return 0;
}

extern "C" int bsub_rpca_rank1_batch_dev(const float* D, int32_t batch, int32_t rows, int32_t cols, double delta, double rho, double tol,
                                         double tol_l1, int32_t max_iter, float* L, float* S, int32_t* iters, float* err, int32_t* rank,
                                         void* stream) {
    if (!D || !L || !S || !iters || !err || !rank || batch < 1 || rows < 1 || cols < 1 || !(delta > 0) || !(rho > 1) || !(tol > 0) || max_iter < 1) {
        set_error("bsub_rpca_rank1_batch_dev: bad argument");
        return -1;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // smallest cluster whose CTAs hold their band of the four matrices in shared memory (scripts/bench_saliency_rpca.py copies this
    // rule to label its rows)
    int C = 0, rl = 0;
    size_t smem = 0;
    for (int c = 1; c <= RB_MAXC && cols <= 32 * RB_KT; c *= 2) {
        const int r = (rows + c - 1) / c;
        const size_t width = (size_t)cols + RB_NSCAL;
        const size_t fl = (size_t)4 * r * cols + 2 * (size_t)cols + r + (size_t)RB_WARPS * cols + width + (size_t)2 * c * width + 24;
        if (fl * sizeof(float) <= RB_SMEM_CAP) { C = c; rl = r; smem = fl * sizeof(float); break; }
    }
    RpcaBatchArgs a;
    a.D = D; a.L = L; a.S = S; a.batch = batch; a.rows = rows; a.cols = cols; a.C = C; a.rl = rl; a.tr = 0;
    a.delta = delta; a.rho = rho; a.tol = tol; a.tol_l1 = tol_l1; a.max_iter = max_iter; a.max_power = 40;
    a.iters = iters; a.err = err; a.rank = rank;
    if (C == 0) return rpca_large_launch(a, dev, sms, stream);
    void (*kern)(RpcaBatchArgs) = cols <= 128 ? rpca_rank1_batch_kernel<4> : cols <= 256 ? rpca_rank1_batch_kernel<8> :
                                  cols <= 384 ? rpca_rank1_batch_kernel<12> : cols <= 512 ? rpca_rank1_batch_kernel<16> : rpca_rank1_batch_kernel<RB_KT>;
    BSUB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RB_SMEM_CAP));
    const int clusters = std::max(1, std::min(batch, sms / C));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(clusters * C)); cfg.blockDim = dim3(RB_THREADS);
    cfg.dynamicSmemBytes = smem; cfg.stream = reinterpret_cast<cudaStream_t>(stream);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    BSUB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, a));
    return 0;
}
