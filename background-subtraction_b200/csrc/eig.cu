// eig.cu -- device-resident top-K symmetric eigensolver for the frames x frames Gram matrix and the
// data-dependent ALM control that follows it (no host round trip).
//
// Replaces the reference's svd_k_largest (/root/reference/utils.py:204-212: ARPACK svds or LAPACK gesdd on
// the m x n matrix) plus the rank logic of /root/reference/inexact_alm_lsd.py:136-145: the right singular
// vectors of W and sigma_i^2 are the eigenpairs of G = W^T W, so only the n x n problem is solved here.
//
// Algorithm (all fp64):
//   1. Householder tridiagonalisation of G by ONE thread-block cluster: rows are dealt cyclically to the C
//      CTAs of the cluster and kept in shared memory; per step the owner of row j builds the reflector, every
//      CTA does its slice of the symmetric matrix-vector product and of the rank-2 update; the two exchanges
//      per step go through L2 and are ordered by the hardware cluster barrier.
//   2. The K largest eigenvalues of the tridiagonal matrix by parallel multisection on Sturm counts
//      (every thread evaluates one shift per round; fixed number of rounds -> deterministic).
//   3. Eigenvectors by inverse iteration (one thread per vector, pivoted tridiagonal LU), CGS2
//      re-orthogonalisation, back-transformation through the stored reflectors (one warp per vector).
//   4. Control: sigma = sqrt(lambda); svp = #{sigma_i > 1/mu, i < sv}; next sv (reference predictor);
//      Vr and VC = Vr * diag(1 - 1/(mu sigma)) written in fp32 for the shrink pass.
#include <cooperative_groups.h>
#include <float.h>
#include <stdlib.h>
#include <algorithm>
#include "common.cuh"
#include "kernels.h"

namespace cg = cooperative_groups;

namespace bsub {

constexpr int EIG_THREADS = 512;
constexpr int EIG_WARPS = EIG_THREADS / 32;
constexpr int EIG_BT = 16;   // vectors back-transformed per batch (one warp each)

struct EigArgs {
    const double* G;           // [npad][npad]
    const double* comm_max;    // [0] = max row-sum of |D| (init mode)
    int n, npad, C, rows_per, in_smem, kcap, mode, k_override;
    int tail_off;              // doubles from the start of dynamic shared memory to the [3][n] exchange buffers
    double* Aglob;             // [C][rows_per][n]  (only when !in_smem)
    double* Vh;                // [n][n] reflectors
    double* tau;               // [n]
    double* dd;                // [n]
    double* ee;                // [n]
    double* pbuf;              // [2][n]
    double* dotbuf;            // [2][16]
    size_t iw_smem_doubles;    // shared-memory doubles available to the inverse-iteration workspace (aliases zs)
    double* lam;               // [n]
    double* Z;                 // [n][n]
    float* Vr; float* VC; int vstride;
    DevState* st;
    int fast_ok;               // warm-started subspace path allowed (mode 1; BSUB_NO_EIG_FAST unset)
    size_t smem_total;         // bytes of dynamic shared memory of this launch
};

__device__ __forceinline__ double ldcg_d(const double* p) { return __ldcg(p); }
__device__ __forceinline__ double warp_allsum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// number of eigenvalues of the tridiagonal (d, e2 = e^2) that are < x: sign changes of the Sturm sequence
//   p_0 = 1, p_1 = d_0 - x, p_i = (d_{i-1} - x) p_{i-1} - e2_{i-2} p_{i-2}
// evaluated in product form (one DFMA on the critical path per step instead of a division) with power-of-two
// rescaling; an exact zero is given the sign opposite to its predecessor (the pivmin rule of LAPACK dlaebz).
__device__ __forceinline__ int sturm_negcount(const double* d, const double* e2, int n, double x, double pivmin) {
    (void)pivmin;
    double pm = 1.0, p = d[0] - x;
    if (p == 0.0) p = -1e-300;
    int c = (p < 0.0);
    for (int i = 1; i < n; ++i) {
        const double t = e2[i - 1] * pm;
        double pn = fma(d[i] - x, p, -t);
        if (pn == 0.0) pn = -p * 0x1p-200;
        c += ((pn < 0.0) != (p < 0.0));
        pm = p; p = pn;
        const double ap = fabs(p);
        if (ap > 0x1p200) { p *= 0x1p-400; pm *= 0x1p-400; }
        else if (ap < 0x1p-200) { p *= 0x1p400; pm *= 0x1p400; }
    }
    return c;
}

__device__ __forceinline__ double hash_unit(unsigned a, unsigned b) {
    unsigned x = a * 0x9E3779B1u ^ (b + 0x7F4A7C15u) * 0x85EBCA77u;
    x ^= x >> 15; x *= 0x2C1B3C6Du; x ^= x >> 12; x *= 0x297A2D39u; x ^= x >> 15;
    return ((double)(x & 0xFFFFFFu) / (double)0x1000000u) * 2.0 - 1.0;
}

// ---- control that follows the eigensolve (runs in CTA 0).  lam_scale: the stored eigenvalues are those of G / lam_scale
//      (first iteration of the int8 path: G_1 = c^2 Gram(D), whose eigenpairs the initialisation already produced).
__device__ void eig_control(const EigArgs& a, DevState* st, int K, double mu, double lam_scale, double* red, double* bc) {
    const int n = a.n, tid = threadIdx.x;
    if (a.mode == 2) return;
    if (a.mode == 0) {
        double tr = 0.0;
        for (int i = tid; i < n; i += EIG_THREADS) tr += a.G[(size_t)i * a.npad + i];
        tr = block_sum(tr, red);
        if (tid == 0) {
            const double l0 = a.lam[0];
            const double norm_two = sqrt(fmax(l0, 0.0));
            st->norm_two = norm_two;
            st->normD2 = tr;
            st->norm_rowsum = a.comm_max[0];
            st->dual_norm = fmax(norm_two, a.comm_max[0] / st->lambda);
            st->mu = st->mu_scale / norm_two;
            st->thresh = 1.0 / st->mu;
            st->iter = 0; st->svp = 0; st->done = 0; st->converged = 0; st->zz = 0.0; st->err = 0.0;
            st->maxS = 0.f; st->nnzS = 0ull;
            // int8 Gram path: W_1 = c D, so iteration 1 reuses this eigen-decomposition (gram_mode 2);
            // |W_1| <= 1.08 max|D| (Y0/mu0 <= D/12.5)
            st->gram_mode = st->use_i8 ? 2 : 0; st->wq_saturated = 0; st->wmax = 1.08 * a.comm_max[2];
            st->force_dmma = 0; st->gram_err = 0.0;
            st->wq_scale = 0.0;
            st->wq_scale_next = (a.comm_max[2] > 0.0) ? exp2(ceil(log2(4.0 * 1.08 * a.comm_max[2]))) : 1.0;
            if (!(norm_two > 0.0)) { st->done = 4; }       // all-zero input
        }
        return;
    }
    // mode 1
    const double thresh = 1.0 / mu;
    if (tid == 0) {
        // truncation-error bound of the int8 Gram (gram_i8.cu; summed over the ranks by the all-reduce, 0 for the fp64 Gram):
        // beyond 0.3 (1/mu)^2 a singular value a little above the threshold could be lost, so the solve continues on gram.cu
        const double ge = a.G[(size_t)a.npad * a.npad + 8] / (thresh * thresh);
        st->gram_err = ge;
        if (ge > 0.3) st->force_dmma = 1;
        int svp = 0;
        for (int k = 0; k < K; ++k) {
            double sig = sqrt(fmax((a.lam[k] * lam_scale), 0.0));
            if (sig > thresh) svp = k + 1;               // last index with sigma > 1/mu (utils.py:215-217)
        }
        const int sv = K;
        st->iter += 1;
        st->sv_used = sv;                                // sv looked at this iteration
        st->svp = svp;
        st->thresh = thresh;
        int svn = sv;
        if (st->use_sv_prediction) svn = (svp < sv) ? svp + 1 : min(svp + st->round005d, st->d);
        st->sv = svn;                                    // inexact_alm_lsd.py:145
        if (st->break_on_rank0 && svp == 0) st->done = 3;  // group_sparse_RPCA.py:91-93
        bc[0] = (double)svp;
    }
    __syncthreads();
    const int svp = (int)bc[0];
    for (int idx = tid; idx < n * svp; idx += EIG_THREADS) {
        const int f = idx / svp, k = idx - f * svp;
        const double sig = sqrt(fmax((a.lam[k] * lam_scale), 0.0));
        const double z = a.Z[(size_t)k * n + f];
        a.Vr[(size_t)f * a.vstride + k] = (float)z;
        a.VC[(size_t)f * a.vstride + k] = (float)(z * (1.0 - thresh / sig));
    }
}

// =====================================================================================================================
// Warm-started fast path (mode 1).  The leading eigenpairs of G = W^T W change little between ALM iterations, and what
// lies below them is a tight cluster ~ (1/mu)^2 that only has to be PROVEN smaller than the threshold.
//   X <- eigenvectors of the previous iteration (p <= 16 columns).  Repeat: Y = G X (rows dealt to the CTAs of the
//   cluster, result pushed into every CTA through distributed shared memory); Rayleigh-Ritz on span(X) (H = X^T Y,
//   parallel Jacobi by one warp); residuals ||G x - theta x||; not converged -> X <- orth(Y) by a Cholesky QR of the
//   rotated (hence nearly orthogonal) Y.
// Certificate (Weyl): for any orthonormal X and theta >= 0, lambda_{p+1}(G) <= ||G - X diag(theta) X^T||_F =: gb.  With
// gb < (1/mu)^2 no eigenvalue outside the p Ritz values can exceed the threshold, so svp is decided by the Ritz values
// alone -- what the reference's rank logic (/root/reference/inexact_alm_lsd.py:133-145, utils.py:204-217) sees from a
// full SVD.  Anything ambiguous (not converged in 8 steps, gb too large, a Ritz value within its error bound of the
// threshold, Cholesky breakdown) returns 0 and the full tridiagonalisation runs instead.  Every CTA derives the same
// decisions from bit-identical data, so the cluster barriers stay uniform.
// =====================================================================================================================
constexpr int EIG_PMAX = 16;

struct EigFastLayout { int PM, RB, RG, NJ, JW, RBP, gsm; size_t doubles, scratch; };
__host__ __device__ inline EigFastLayout eig_fast_layout(int n, int C) {
    EigFastLayout L;
    L.PM = 16;
    L.RB = (n + C - 1) / C;
    L.RG = (L.RB + 31) / 32;
    L.RBP = L.RG * 32;
    L.NJ = EIG_WARPS / L.RG; if (L.NJ < 1) L.NJ = 1;
    {   // long clips: the partial-sum scratch [NJ][PM][RBP] must fit beside X and Y (fewer, longer column chunks)
        const size_t fixed0 = (size_t)2 * n * L.PM + (size_t)5 * L.PM * L.PM + (size_t)6 * L.PM + 16 + 8 + 64;
        while (L.NJ > 1 && (fixed0 + (size_t)L.NJ * L.PM * L.RBP) * sizeof(double) > (size_t)222 * 1024) --L.NJ;
    }
    L.JW = (n + L.NJ - 1) / L.NJ;
    // this CTA's rows of G in shared memory ([RB][n]) when they fit beside X and Y: the products then need no partial sums
    const size_t fixed = (size_t)2 * n * L.PM + (size_t)5 * L.PM * L.PM + (size_t)6 * L.PM + 16 + 8 + 64;
    const size_t with_g = fixed + (size_t)4 * EIG_THREADS + (size_t)L.RB * n;
    L.gsm = (with_g * sizeof(double) <= (size_t)220 * 1024) ? 1 : 0;
    size_t scratch = L.gsm ? (size_t)4 * EIG_THREADS : (size_t)L.NJ * L.PM * L.RBP;
    const size_t s2 = (size_t)4 * EIG_THREADS;             // small reductions: four doubles per thread
    if (scratch < s2) scratch = s2;
    L.scratch = scratch;
    L.doubles = fixed + scratch + (L.gsm ? (size_t)L.RB * n : 0);
    return L;
}

// Y rows of this CTA = G[rows, :] X, pushed into Ys of every CTA.  Thread = (row, column chunk): G is symmetric, so the
// lanes of a warp read G[j][i .. i+31] (coalesced) and X[j][0..p) is a shared-memory broadcast.
__device__ void eig_fast_matvec(const EigArgs& a, const EigFastLayout& L, int p, const double* Xs, double* Ys, double* Pp,
                                cg::cluster_group& cluster) {
    const int n = a.n, C = a.C, c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, PM = L.PM;
    const int row0 = c * L.RB, nrows = max(0, min(n, row0 + L.RB) - row0);
    const int rg = warp % L.RG, jc = warp / L.RG, rl = rg * 32 + lane, i = row0 + rl;
    if (jc < L.NJ) {
        double acc[EIG_PMAX];
#pragma unroll
        for (int k = 0; k < EIG_PMAX; ++k) acc[k] = 0.0;
        if (rl < nrows) {
            const int j1 = min(n, (jc + 1) * L.JW);
            for (int j = jc * L.JW; j < j1; ++j) {
                const double g = __ldg(a.G + (size_t)j * a.npad + i);
                const double* xr = Xs + (size_t)j * PM;
#pragma unroll
                for (int k = 0; k < EIG_PMAX; k += 2)
                    if (k < p) {
                        const double2 x2 = *reinterpret_cast<const double2*>(xr + k);
                        acc[k] = fma(g, x2.x, acc[k]); acc[k + 1] = fma(g, x2.y, acc[k + 1]);
                    }
            }
        }
#pragma unroll
        for (int k = 0; k < EIG_PMAX; ++k) if (k < p) Pp[((size_t)jc * PM + k) * L.RBP + rl] = acc[k];
    }
    __syncthreads();
    cluster.sync();                                   // every CTA has finished reading the previous Ys
    for (int item = tid; item < p * L.RBP; item += EIG_THREADS) {
        const int k = item / L.RBP, r2 = item - k * L.RBP;
        if (r2 < nrows) {
            double y = 0.0;
            for (int q = 0; q < L.NJ; ++q) y += Pp[((size_t)q * PM + k) * L.RBP + r2];
            for (int q = 0; q < C; ++q) cluster.map_shared_rank(Ys, q)[(size_t)(row0 + r2) * PM + k] = y;
        }
    }
    cluster.sync();                                   // Ys complete in every CTA
}

// The same product with this CTA's rows of G in shared memory (Gs[rl][j]): one thread per (row, vector) output, the row of G
// is a broadcast across the p threads of a row and X[j][0..p) is read conflict-free.
__device__ void eig_fast_matvec_smem(const EigArgs& a, const EigFastLayout& L, int p, const double* Gs, const double* Xs, double* Ys,
                                     cg::cluster_group& cluster) {
    const int n = a.n, C = a.C, c = blockIdx.x, tid = threadIdx.x, PM = L.PM;
    const int row0 = c * L.RB, nrows = max(0, min(n, row0 + L.RB) - row0);
    cluster.sync();                                   // every CTA has finished reading the previous Ys
    for (int item = tid; item < nrows * p; item += EIG_THREADS) {
        const int rl = item / p, k = item - rl * p;
        const double* gr = Gs + (size_t)rl * n;
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        int j = 0;
        for (; j + 3 < n; j += 4) {
            s0 = fma(gr[j], Xs[(size_t)j * PM + k], s0); s1 = fma(gr[j + 1], Xs[(size_t)(j + 1) * PM + k], s1);
            s2 = fma(gr[j + 2], Xs[(size_t)(j + 2) * PM + k], s2); s3 = fma(gr[j + 3], Xs[(size_t)(j + 3) * PM + k], s3);
        }
        for (; j < n; ++j) s0 = fma(gr[j], Xs[(size_t)j * PM + k], s0);
        const double y = (s0 + s1) + (s2 + s3);
        for (int q = 0; q < C; ++q) cluster.map_shared_rank(Ys, q)[(size_t)(row0 + rl) * PM + k] = y;
    }
    cluster.sync();                                   // Ys complete in every CTA
}

// out[a][b] = sum_i A[i][a] B[i][b]  (p x p, computed redundantly by every CTA); scratch: one double per thread
__device__ void eig_fast_gram(int n, int PM, int p, const double* A, const double* B, double* out, double* scratch, bool symmetrise) {
    const int tid = threadIdx.x, pairs = p * p, nparts = EIG_THREADS / pairs, part = tid / pairs, pr = tid - part * pairs;
    const int ia = pr / p, ib = pr - ia * p;
    if (part < nparts) {
        double acc = 0.0, acc2 = 0.0;
        int i = part;
        for (; i + nparts < n; i += 2 * nparts) {
            acc = fma(A[(size_t)i * PM + ia], B[(size_t)i * PM + ib], acc);
            acc2 = fma(A[(size_t)(i + nparts) * PM + ia], B[(size_t)(i + nparts) * PM + ib], acc2);
        }
        if (i < n) acc = fma(A[(size_t)i * PM + ia], B[(size_t)i * PM + ib], acc);
        scratch[tid] = acc + acc2;
    }
    __syncthreads();
    double t = 0.0;
    if (tid < pairs) for (int q = 0; q < nparts; ++q) t += scratch[(size_t)q * pairs + tid];
    __syncthreads();
    if (tid < pairs) out[ia * PM + ib] = t;
    __syncthreads();
    if (symmetrise) {
        double v = 0.0;
        if (tid < pairs) v = 0.5 * (out[ia * PM + ib] + out[ib * PM + ia]);
        __syncthreads();
        if (tid < pairs) out[ia * PM + ib] = v;
        __syncthreads();
    }
}

// Symmetric p x p eigenproblem by ONE warp: parallel (round-robin) Jacobi.  H is destroyed (its diagonal holds the
// eigenvalues), W = eigenvectors (columns); both then sorted in descending order through `tmp`.
__device__ void eig_fast_jacobi(int PM, int p, double* H, double* W, double* th, double* tmp, double* cs) {
    const int lane = threadIdx.x & 31;
    for (int idx = lane; idx < PM * PM; idx += 32) W[idx] = ((idx / PM) == (idx % PM)) ? 1.0 : 0.0;
    __syncwarp();
    const int pp = p + (p & 1), half = pp / 2;
    for (int sweep = 0; sweep < 12 && pp >= 2; ++sweep) {
        int rotated = 0;
        for (int round = 0; round < pp - 1; ++round) {
            if (lane < half) {
                const int ia = (lane == 0) ? pp - 1 : (round + lane) % (pp - 1);
                const int ib = (round + pp - 1 - lane) % (pp - 1);
                double cth = 1.0, sth = 0.0;
                if (ia < p && ib < p) {
                    const double apq = H[ia * PM + ib], app = H[ia * PM + ia], aqq = H[ib * PM + ib];
                    // rotate while the off-diagonal entry matters against the LARGER of the two diagonal entries (absolute accuracy
                    // eps * max is all the ALM needs: the threshold (1/mu)^2 is > 1e-12 of the leading value).  A test relative to
                    // sqrt(app aqq) never settles for a (leading, cluster) pair: the rounding of the leading entry alone leaves
                    // eps * app behind, far above eps * sqrt(app aqq).
                    const double amax = fmax(fabs(app), fabs(aqq));
                    if (fabs(apq) > DBL_EPSILON * amax && fabs(apq) > DBL_MIN) {
                        // rotation angle phi with tan(2 phi) = 2 apq / (aqq - app), |phi| <= pi/4:
                        //   cos(2 phi) = |d| / h, h = hypot(d, 2 apq);  c = sqrt((1 + cos 2phi) / 2);  s = sgn(d) apq / (h c)
                        // two reciprocal square roots instead of two square roots and three divisions
                        const double dd = aqq - app, bb = 2.0 * apq;
                        const double hinv = rsqrt(fma(dd, dd, bb * bb));
                        const double c2 = 0.5 * fma(fabs(dd), hinv, 1.0);          // cos^2 phi in [1/2, 1]
                        const double cinv = rsqrt(c2);
                        cth = c2 * cinv;
                        sth = copysign(apq * hinv * cinv, dd * apq);
                        if (dd == 0.0) sth = copysign(fabs(sth), apq);
                        rotated = 1;
                    }
                }
                cs[4 * lane] = cth; cs[4 * lane + 1] = sth; cs[4 * lane + 2] = (double)ia; cs[4 * lane + 3] = (double)ib;
            }
            __syncwarp();
            // columns a, b of H and of W:  (M[k][a], M[k][b]) <- (c M[k][a] - s M[k][b], s M[k][a] + c M[k][b])
            for (int item = lane; item < half * p; item += 32) {
                const int q = item / p, k = item - q * p;
                const double cth = cs[4 * q], sth = cs[4 * q + 1];
                const int ia = (int)cs[4 * q + 2], ib = (int)cs[4 * q + 3];
                if (sth != 0.0) {
                    const double ha = H[k * PM + ia], hb = H[k * PM + ib];
                    H[k * PM + ia] = cth * ha - sth * hb; H[k * PM + ib] = sth * ha + cth * hb;
                    const double wa = W[k * PM + ia], wb = W[k * PM + ib];
                    W[k * PM + ia] = cth * wa - sth * wb; W[k * PM + ib] = sth * wa + cth * wb;
                }
            }
            __syncwarp();
            // rows a, b of H
            for (int item = lane; item < half * p; item += 32) {
                const int q = item / p, k = item - q * p;
                const double cth = cs[4 * q], sth = cs[4 * q + 1];
                const int ia = (int)cs[4 * q + 2], ib = (int)cs[4 * q + 3];
                if (sth != 0.0) {
                    const double ha = H[ia * PM + k], hb = H[ib * PM + k];
                    H[ia * PM + k] = cth * ha - sth * hb; H[ib * PM + k] = sth * ha + cth * hb;
                }
            }
            __syncwarp();
        }
        if (!__any_sync(0xffffffffu, rotated)) break;
    }
    if (lane < p) {                                    // sort descending (rank by counting)
        const double v = H[lane * PM + lane];
        int rank = 0;
        for (int j = 0; j < p; ++j) { const double u = H[j * PM + j]; rank += (u > v) || (u == v && j < lane); }
        th[rank] = v;
        for (int k = 0; k < p; ++k) tmp[k * PM + rank] = W[k * PM + lane];
    }
    __syncwarp();
    for (int idx = lane; idx < PM * PM; idx += 32) { const int r = idx / PM, cc = idx - r * PM; if (r < p && cc < p) W[idx] = tmp[idx]; }
    __syncwarp();
}

// rows of M (n x p, row stride PM) <- row * W, in place: p lanes of one warp own a row (32 / p rows per warp pass), every lane
// reads the whole old row before the warp-level barrier and writes its element after it.
__device__ void eig_fast_rotate(int n, int PM, int p, double* M, const double* W) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int RP = 32 / p, rs = lane / p, k = lane - rs * p;
    for (int base = warp * RP; base < n; base += EIG_WARPS * RP) {
        const int i = base + rs;
        const bool act = rs < RP && i < n;
        double y0 = 0.0, y1 = 0.0;
        if (act) {
            const double* x = M + (size_t)i * PM;
            int aa = 0;
            for (; aa + 1 < p; aa += 2) { y0 = fma(x[aa], W[aa * PM + k], y0); y1 = fma(x[aa + 1], W[(aa + 1) * PM + k], y1); }
            if (aa < p) y0 = fma(x[aa], W[aa * PM + k], y0);
        }
        __syncwarp();
        if (act) M[(size_t)i * PM + k] = y0 + y1;
        __syncwarp();
    }
    __syncthreads();
}

// returns 1: CTA 0 has written lam[0..K) and Z[0..p), *p_out = p (all CTAs return 1); 0: nothing written -> full path
__device__ int eig_fast_path(const EigArgs& a, DevState* st, int K, double mu, double* esm, int* p_out, cg::cluster_group& cluster) {
    const int n = a.n, C = a.C, c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const EigFastLayout L = eig_fast_layout(n, C);
    const int PM = L.PM;
    const int p = st->eig_p;
    if (!a.fast_ok || p < 1 || n < 32 || 4 * p > n || p > PM || K < 1) return 0;
    if (L.doubles * sizeof(double) > a.smem_total) return 0;
    const double tau = 1.0 / (mu * mu);

    const size_t scratch_d = L.scratch;
    double* Xs = esm;                                   // [n][PM]
    double* Ys = Xs + (size_t)n * PM;                   // [n][PM]
    double* Pp = Ys + (size_t)n * PM;                   // [NJ][PM][RBP] partial products / scratch of the small reductions
    double* Hs = Pp + scratch_d;                        // [PM][PM]
    double* Bs = Hs + PM * PM;
    double* Ws = Bs + PM * PM;
    double* Ts = Ws + PM * PM;
    double* Rs = Ts + PM * PM;                          // Cholesky factor
    double* th = Rs + PM * PM;                          // [PM]
    double* res = th + PM;                              // [PM]
    double* cs = res + PM;                              // [4 * PM]
    double* gbp = cs + 4 * PM;                          // [16] per-CTA partials of gb^2
    double* flag = gbp + 16;                            // [8]
    double* red = flag + 8;                             // [64]
    double* Gs = red + 64;                              // [RB][n] this CTA's rows of G (only when L.gsm)
    if (L.gsm) {
        const int row0 = c * L.RB, nrows = max(0, min(n, row0 + L.RB) - row0);
        for (int idx = tid; idx < nrows * n; idx += EIG_THREADS) {
            const int rl = idx / n, j = idx - rl * n;
            Gs[idx] = __ldg(a.G + (size_t)(row0 + rl) * a.npad + j);
        }
    }

    for (int idx = tid; idx < n * PM; idx += EIG_THREADS) {
        const int i = idx / PM, k = idx - i * PM;
        Xs[idx] = (k < p) ? a.Z[(size_t)k * n + i] : 0.0;
    }
    __syncthreads();

    long long tph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tc = clock64();
#define EF_TICK(k) { __syncthreads(); const long long t_ = clock64(); tph[k] += t_ - tc; tc = t_; }
    EF_TICK(0)                                                  // load of X (and of the rows of G)
    const int max_steps = 8;
    int converged = 0, steps = 0;
    for (int step = 0; step < max_steps; ++step) {
        steps = step + 1;
        if (L.gsm) eig_fast_matvec_smem(a, L, p, Gs, Xs, Ys, cluster);
        else eig_fast_matvec(a, L, p, Xs, Ys, Pp, cluster);
        EF_TICK(1)
        eig_fast_gram(n, PM, p, Xs, Ys, Hs, Pp, true);          // H = X^T G X
        eig_fast_gram(n, PM, p, Ys, Ys, Bs, Pp, true);          // B = Y^T Y
        EF_TICK(2)
        if (warp == 0) eig_fast_jacobi(PM, p, Hs, Ws, th, Ts, cs);
        EF_TICK(3)
        eig_fast_rotate(n, PM, p, Xs, Ws);                      // Ritz vectors X W, and G (X W) = Y W
        eig_fast_rotate(n, PM, p, Ys, Ws);
        EF_TICK(4)
        // B' = W^T B W (Gram of the rotated Y):  Ts = B W, then Bs = W^T Ts
        if (tid < PM * PM) {
            const int r = tid / PM, cc = tid - r * PM;
            double t = 0.0;
            if (r < p && cc < p) for (int d = 0; d < p; ++d) t = fma(Bs[r * PM + d], Ws[d * PM + cc], t);
            Ts[tid] = t;
        }
        __syncthreads();
        if (tid < PM * PM) {
            const int r = tid / PM, cc = tid - r * PM;
            double t = 0.0;
            if (r < p && cc < p) for (int d = 0; d < p; ++d) t = fma(Ws[d * PM + r], Ts[d * PM + cc], t);
            Bs[tid] = t;
        }
        {   // residuals r_k = || Y_k - theta_k X_k ||
            const int k = tid % PM, part = tid / PM, nparts = EIG_THREADS / PM;
            double acc = 0.0;
            if (k < p) {
                const double t = th[k];
                for (int i = part; i < n; i += nparts) { const double d = fma(-t, Xs[(size_t)i * PM + k], Ys[(size_t)i * PM + k]); acc = fma(d, d, acc); }
            }
            Pp[tid] = acc;                                      // [part][PM]
        }
        __syncthreads();
        if (tid < PM) {
            double t = 0.0;
            const int nparts = EIG_THREADS / PM;
            for (int q = 0; q < nparts; ++q) t += Pp[(size_t)q * PM + tid];
            res[tid] = sqrt(t);
        }
        __syncthreads();
        if (tid == 0) {
            int ok = (th[0] > 0.0) ? 1 : 0;
            for (int k = 0; k < p; ++k) {
                if (!(th[k] == th[k])) ok = 0;                                      // NaN
                if (th[k] > 0.5 * tau && !(res[k] <= 1e-13 * th[0])) ok = 0;       // every pair that may be kept must have converged
            }
            flag[0] = (double)ok;
        }
        __syncthreads();
        EF_TICK(5)
        if (flag[0] != 0.0) { converged = 1; break; }
        if (step == max_steps - 1) break;
        // X <- orth(Y) by Cholesky QR: B' = R^T R, X = Y R^{-1}
        if (warp == 0) {
            int bad = 0;
            for (int idx = lane; idx < PM * PM; idx += 32) Rs[idx] = Bs[idx];
            __syncwarp();
            for (int j = 0; j < p; ++j) {
                const double d2 = Rs[j * PM + j];
                if (!(d2 > 0.0)) { bad = 1; break; }                                // uniform over the warp
                const double inv = rsqrt(d2);
                __syncwarp();
                if (lane > j && lane < p) Rs[j * PM + lane] *= inv;
                if (lane == j) Rs[j * PM + j] = inv;                                // the diagonal holds 1 / R_jj
                __syncwarp();
                const int m2 = p - 1 - j;                                           // trailing block, upper triangle incl. diagonal
                for (int item = lane; item < m2 * m2; item += 32) {
                    const int r = j + 1 + item / m2, cc = j + 1 + item % m2;
                    if (cc >= r) Rs[r * PM + cc] = fma(-Rs[j * PM + r], Rs[j * PM + cc], Rs[r * PM + cc]);
                }
                __syncwarp();
            }
            if (lane == 0) flag[1] = (double)bad;
        }
        __syncthreads();
        if (flag[1] != 0.0) return 0;
        for (int i = tid; i < n; i += EIG_THREADS) {
            double x[EIG_PMAX];
#pragma unroll
            for (int k = 0; k < EIG_PMAX; ++k) {
                x[k] = 0.0;
                if (k < p) {
                    double v = Ys[(size_t)i * PM + k];
#pragma unroll
                    for (int aa = 0; aa < EIG_PMAX; ++aa) if (aa < k) v = fma(-x[aa], Rs[aa * PM + k], v);
                    x[k] = v * Rs[k * PM + k];
                    Xs[(size_t)i * PM + k] = x[k];
                }
            }
        }
        EF_TICK(6)
    }
    if (!converged) return 0;

    // ---- certificate: gb = || G - X diag(theta) X^T + s (I - X X^T) ||_F (rows dealt as in the matvec) and the orthonormality
    // defect of X.  s >= 0 is the known downward bias of the int8 Gram on everything outside the leading pairs (half of the bound
    // in the error slot, see gram_i8.cu): the deflated matrix is re-centred before its norm is taken, and
    //     lambda_{p+1}(G) <= lambda_max(G - X theta X^T) <= gb - s.
    const double sshift = 0.5 * a.G[(size_t)a.npad * a.npad + 8];
    {
        const int row0 = c * L.RB, nrows = max(0, min(n, row0 + L.RB) - row0);
        const int rg = warp % L.RG, jc = warp / L.RG, rl = rg * 32 + lane, i = row0 + rl;
        double acc = 0.0;
        if (L.gsm) {
            // Y is no longer needed: keep X transposed there ([k][n]) so that threads with consecutive j read consecutive words
            double* Xt = Ys;
            for (int idx = tid; idx < n * p; idx += EIG_THREADS) { const int k = idx / n, j = idx - k * n; Xt[idx] = Xs[(size_t)j * PM + k]; }
            __syncthreads();
            for (int item = tid; item < nrows * n; item += EIG_THREADS) {
                const int r2 = item / n, j = item - r2 * n, i2 = row0 + r2;
                double g = Gs[item] + ((i2 == j) ? sshift : 0.0);
                for (int k = 0; k < p; ++k) if (th[k] > 0.0) g = fma(-(th[k] + sshift) * Xt[(size_t)k * n + i2], Xt[(size_t)k * n + j], g);
                acc = fma(g, g, acc);
            }
        } else if (jc < L.NJ && rl < nrows) {
            double xt[EIG_PMAX];
#pragma unroll
            for (int k = 0; k < EIG_PMAX; ++k) xt[k] = (k < p && th[k] > 0.0) ? (th[k] + sshift) * Xs[(size_t)i * PM + k] : 0.0;
            const int j1 = min(n, (jc + 1) * L.JW);
            for (int j = jc * L.JW; j < j1; ++j) {
                double g = (L.gsm ? Gs[(size_t)rl * n + j] : __ldg(a.G + (size_t)j * a.npad + i)) + ((i == j) ? sshift : 0.0);
                const double* xr = Xs + (size_t)j * PM;
#pragma unroll
                for (int k = 0; k < EIG_PMAX; ++k) if (k < p) g = fma(-xt[k], xr[k], g);
                acc = fma(g, g, acc);
            }
        }
        acc = block_sum(acc, red);                               // valid in thread 0
        if (tid == 0) for (int q = 0; q < C; ++q) cluster.map_shared_rank(gbp, q)[c] = acc;
        cluster.sync();
    }
    eig_fast_gram(n, PM, p, Xs, Xs, Ts, Pp, false);              // X^T X
    if (tid == 0) {
        double gb2 = 0.0;
        for (int q = 0; q < C; ++q) gb2 += gbp[q];
        const double gb = fmax(sqrt(gb2) - sshift, 0.0);
        double orth = 0.0;
        for (int r = 0; r < p; ++r)
            for (int cc = 0; cc < p; ++cc) orth = fmax(orth, fabs(Ts[r * PM + cc] - (r == cc ? 1.0 : 0.0)));
        const double slack = (8.0 * n * DBL_EPSILON + 2.0 * orth) * th[0];
        int ok = (gb * (1.0 + 1e-6) + slack < tau) && (gb2 == gb2);
        for (int k = 0; k < p; ++k) {
            if (th[k] > 0.5 * tau) { if (fabs(th[k] - tau) <= fmax(4.0 * res[k], 1e-13 * th[0])) ok = 0; }   // knife edge: let the full path decide
            else if (!(th[k] + gb + slack < tau)) ok = 0;                                                    // unconverged pair must be certainly below
        }
        flag[2] = (double)ok;
        if (c == 0) { st->eig_info = steps | (ok ? 0x100 : 0); st->eig_gb = gb / tau; }
    }
    EF_TICK(7)
    if (c == 0 && tid == 0) for (int k = 0; k < 8; ++k) st->eig_clk[8 + k] = tph[k];
#undef EF_TICK
    if (flag[2] == 0.0) return 0;
    if (c == 0) {
        for (int k = tid; k < K; k += EIG_THREADS) a.lam[k] = (k < p) ? th[k] : 0.0;     // everything else is certified below the threshold
        for (int idx = tid; idx < n * p; idx += EIG_THREADS) {
            const int k = idx / n, i = idx - k * n;
            a.Z[(size_t)k * n + i] = Xs[(size_t)i * PM + k];
        }
        __threadfence_block();
    }
    __syncthreads();
    *p_out = p;
    return 1;
}

// ---- back-transformation z <- H_0 H_1 ... H_{n-3} z of the tridiagonal eigenvectors, one warp per vector.  The vector
// lives in registers (lane owns entries lane + 32 t), the next reflector row is prefetched from L2 while the current one is
// applied: a step costs one register dot product, one warp all-reduce and one register update.
template <int NT>
__device__ void eig_backtransform(const EigArgs& a, int K, const double* tau_s, int warp, int lane) {
    const int n = a.n;
    auto load_row = [&](int j, auto& v) {          // reflector j: entries i > j (the rest of the row is not part of it)
        const double* vh = a.Vh + (size_t)(j < 0 ? 0 : j) * n;
#pragma unroll
        for (int t = 0; t < NT; ++t) { const int i = lane + 32 * t; v[t] = (j >= 0 && i > j && i < n) ? ldcg_d(vh + i) : 0.0; }
    };
    for (int k = warp; k < K; k += EIG_WARPS) {
        constexpr bool DEEP = (NT <= 10);                   // second prefetch level only while the registers last
        double z[NT], v0[NT], v1[NT], v2[DEEP ? NT : 1];    // current reflector and the next one or two (an L2 round trip is ~2 steps)
        double* zrow = a.Z + (size_t)k * n;
#pragma unroll
        for (int t = 0; t < NT; ++t) { const int i = lane + 32 * t; z[t] = (i < n) ? zrow[i] : 0.0; }
        load_row(n - 3, v0);
        load_row(n - 4, v1);
        for (int j = n - 3; j >= 0; --j) {
            if constexpr (DEEP) load_row(j - 2, v2);
            const double tau = tau_s[j];
            if (tau != 0.0) {
                double sa = 0.0, sb = 0.0;
#pragma unroll
                for (int t = 0; t < NT; ++t) { if (t & 1) sb = fma(v0[t], z[t], sb); else sa = fma(v0[t], z[t], sa); }
                const double s = warp_allsum(sa + sb) * tau;
#pragma unroll
                for (int t = 0; t < NT; ++t) z[t] = fma(-s, v0[t], z[t]);
            }
#pragma unroll
            for (int t = 0; t < NT; ++t) { v0[t] = v1[t]; if constexpr (DEEP) v1[t] = v2[t]; }
            if constexpr (!DEEP) load_row(j - 2, v1);
        }
#pragma unroll
        for (int t = 0; t < NT; ++t) { const int i = lane + 32 * t; if (i < n) zrow[i] = z[t]; }
    }
}

// ---- Householder tridiagonalisation with the matrix rows in shared memory, dealt cyclically over the cluster.
// Both exchanges of a step go through distributed shared memory: (1) after its rank-2 update every CTA pushes its
// entries of the next column into all CTAs, so every warp forms the reflector redundantly; (2) every CTA pushes its
// slice of p = tau A v into all CTAs.  Two hardware cluster barriers per step and nothing else: every warp keeps the
// reflector v and w = p + kc v in registers (lane owns columns lane + 32 t), so there is no block-level barrier or
// reduction, and a row is always touched by the same warp.
template <int NT>
__device__ void eig_tridiag_dsmem(const EigArgs& a, double* Asm, double* xb, double* pb, DevState* st) {
    cg::cluster_group cluster = cg::this_cluster();
    const int n = a.n, C = a.C, c = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cshift = 31 - __clz(C), cmask = C - 1;      // C is a power of two (make_eig_plan)
    double* xb_rem = (lane < C) ? cluster.map_shared_rank(xb, lane) : nullptr;
    double* pb_rem = (lane < C) ? cluster.map_shared_rank(pb, lane) : nullptr;
    for (int li = warp; li < a.rows_per; li += EIG_WARPS) {
        const int i = c + li * C;
        if (i >= 1 && i < n) { const double val = Asm[(size_t)li * n]; if (lane < C) xb_rem[i] = val; }
    }
    cluster.sync();
    long long tph[6] = {0, 0, 0, 0, 0, 0}, tc = clock64();
#define EIG_TICK(k) { const long long t_ = clock64(); tph[k] += t_ - tc; tc = t_; }
    for (int j = 0; j + 2 < n; ++j) {
        const int par = j & 1;
        const double* x = xb + par * n;
        const int t0 = (j + 1) >> 5;                        // first 32-column block holding a column > j
        // reflector from column j
        double v[NT], w[NT];
        double ssa = 0.0, ssb = 0.0;
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const int col = lane + 32 * t;
            v[t] = (t >= t0 && col > j && col < n) ? x[col] : 0.0;
        }
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const int col = lane + 32 * t;
            const double xv = (col >= j + 2) ? v[t] : 0.0;
            if (t & 1) ssb = fma(xv, xv, ssb); else ssa = fma(xv, xv, ssa);
        }
        const double ss = warp_allsum(ssa + ssb);
        const double alpha = x[j + 1];
        double beta, tau, scale;
        if (ss == 0.0) { tau = 0.0; beta = alpha; scale = 0.0; }
        else {
            // beta = -sgn(alpha) ||x||, tau = (beta - alpha) / beta = 1 + |alpha| / ||x||, scale = 1 / (alpha - beta):
            // one reciprocal square root and one independent reciprocal instead of sqrt + two divisions
            const double nrm2 = fma(alpha, alpha, ss), aa = fabs(alpha);
            const double rn = rsqrt(nrm2), nrm = nrm2 * rn;
            beta = -copysign(nrm, alpha);
            tau = fma(aa, rn, 1.0);
            scale = copysign(__drcp_rn(aa + nrm), alpha);
        }
#pragma unroll
        for (int t = 0; t < NT; ++t) v[t] = (lane + 32 * t == j + 1) ? 1.0 : v[t] * scale;
        if (c == (j & cmask) && warp == 0) {
            double* vh = a.Vh + (size_t)j * n;
#pragma unroll
            for (int t = 0; t < NT; ++t) { const int col = lane + 32 * t; if (t >= t0 && col > j && col < n) vh[col] = v[t]; }
            if (lane == 0) { a.tau[j] = tau; a.dd[j] = Asm[(size_t)(j >> cshift) * n + j]; a.ee[j] = beta; }
        }
        EIG_TICK(0)
        const int l0 = (j >= c) ? ((j - c) >> cshift) + 1 : 0;  // first local row with global index > j
        for (int lb = l0 + warp; lb < a.rows_per; lb += 3 * EIG_WARPS) {
            const int l1 = lb + EIG_WARPS, l2 = lb + 2 * EIG_WARPS;
            const int i0 = c + lb * C, i1 = c + l1 * C, i2 = c + l2 * C;
            const bool ok0 = i0 < n, ok1 = (l1 < a.rows_per) && i1 < n, ok2 = (l2 < a.rows_per) && i2 < n;
            const double* r0 = Asm + (size_t)lb * n;
            const double* r1 = ok1 ? Asm + (size_t)l1 * n : r0;
            const double* r2 = ok2 ? Asm + (size_t)l2 * n : r0;
            double s0 = 0.0, s1 = 0.0, s2 = 0.0;
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                const int col = lane + 32 * t;
                if (t >= t0 && col < n) { s0 = fma(r0[col], v[t], s0); s1 = fma(r1[col], v[t], s1); s2 = fma(r2[col], v[t], s2); }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                s2 += __shfl_xor_sync(0xffffffffu, s2, o);
            }
            if (lane < C) {
                if (ok0) pb_rem[i0] = tau * s0;
                if (ok1) pb_rem[i1] = tau * s1;
                if (ok2) pb_rem[i2] = tau * s2;
            }
        }
        EIG_TICK(1)
        cluster.sync();
        EIG_TICK(2)
        double dla = 0.0, dlb = 0.0;
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const int col = lane + 32 * t;
            w[t] = (t >= t0 && col > j && col < n) ? pb[col] : 0.0;
            if (t & 1) dlb = fma(w[t], v[t], dlb); else dla = fma(w[t], v[t], dla);
        }
        const double kc = -0.5 * tau * warp_allsum(dla + dlb);
#pragma unroll
        for (int t = 0; t < NT; ++t) w[t] = fma(kc, v[t], w[t]);
        EIG_TICK(3)
        double* xn = xb_rem + (par ^ 1) * n;
        const int fl = (j + 1) & 31;                        // lane / block (t0) that hold column j + 1
        if constexpr (NT <= 10) {
            // (a) the entries of the NEXT column first: they are all the other CTAs wait for.  A[i][j+1] -= v_i w_{j+1} + w_i v_{j+1}
            //     with v_{j+1} = 1.  Then arrive at the cluster barrier, (b) update the rest of my rows while the barrier
            //     completes, and only then wait.  Everything read from pb is taken before the arrive: a CTA that is through
            //     the barrier may already be writing the next p into it.
            double wsel = 0.0;
    #pragma unroll
            for (int t = 0; t < NT; ++t) if (t == t0) wsel = w[t];
            const double wnext = __shfl_sync(0xffffffffu, wsel, fl);
            double vi_[3], wi_[3];
            bool ok_[3];
    #pragma unroll
            for (int k = 0; k < 3; ++k) {
                const int li = l0 + warp + k * EIG_WARPS, i = c + li * C;
                ok_[k] = (li < a.rows_per) && (i < n);
                vi_[k] = 0.0; wi_[k] = 0.0;
                if (ok_[k]) {
                    double* r = Asm + (size_t)li * n;
                    vi_[k] = (i == j + 1) ? 1.0 : x[i] * scale;
                    wi_[k] = fma(kc, vi_[k], pb[i]);
                    const double nv = r[j + 1] - (vi_[k] * wnext + wi_[k]);
                    __syncwarp();
                    if (lane == 0) r[j + 1] = nv;
                    if (lane < C && i > j + 1) xn[i] = nv;     // this CTA's entry of the next column, into every CTA
                }
            }
            EIG_TICK(4)
            asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    #pragma unroll
            for (int k = 0; k < 3; ++k) {
                if (ok_[k]) {
                    double* r = Asm + (size_t)(l0 + warp + k * EIG_WARPS) * n;
                    const double vi = vi_[k], wi = wi_[k];
    #pragma unroll
                    for (int t = 0; t < NT; ++t) {
                        const int col = lane + 32 * t;
                        if (t >= t0 && col > j + 1 && col < n) r[col] -= vi * w[t] + wi * v[t];
                    }
                }
            }
            asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
        } else {
            // long rows: the split version costs registers that the NT > 10 instances do not have; one pass, full barrier
            for (int li = l0 + warp; li < a.rows_per; li += EIG_WARPS) {
                const int i = c + li * C;
                if (i < n) {
                    double* r = Asm + (size_t)li * n;
                    const double vi = (i == j + 1) ? 1.0 : x[i] * scale;
                    const double wi = fma(kc, vi, pb[i]);
                    double first = 0.0;
#pragma unroll
                    for (int t = 0; t < NT; ++t) {
                        const int col = lane + 32 * t;
                        if (t >= t0 && col > j && col < n) {
                            const double nv = r[col] - (vi * w[t] + wi * v[t]);
                            r[col] = nv;
                            if (t == t0) first = nv;
                        }
                    }
                    first = __shfl_sync(0xffffffffu, first, fl);
                    if (lane < C && i > j + 1) xn[i] = first;
                }
            }
            EIG_TICK(4)
            cluster.sync();
        }
        EIG_TICK(5)
    }
    if (c == 0 && tid == 0) for (int k = 0; k < 6; ++k) st->eig_clk[8 + k] = tph[k];
#undef EIG_TICK
}

__global__ void __launch_bounds__(EIG_THREADS, 1) eig_kernel(EigArgs a) {
    cg::cluster_group cluster = cg::this_cluster();
    DevState* st = a.st;
    if (a.mode == 1 && st->done) return;          // uniform over the cluster (see DESIGN.md 4.2)
    const int n = a.n, C = a.C, c = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // int8 path: the initialisation also produces the sv0 leading eigenpairs, which iteration 1 reuses (W_1 = c D)
    int K = (a.mode == 0) ? (st->use_i8 ? st->sv : 1) : ((a.mode == 1) ? st->sv : a.k_override);
    const bool reuse = (a.mode == 1) && (st->gram_mode == 2);
    if (K > n) K = n;
    if (K < 1) K = 1;
    const double mu = (a.mode == 1) ? st->mu : 0.0;

    extern __shared__ __align__(16) double esm[];
    double* v_s = esm;                 // [n]
    double* w_s = esm + n;             // [n]
    double* red = esm + 2 * n;         // [64]
    double* Asm = esm + 2 * n + 64;    // matrix rows / later phases
    __shared__ double bc[4];

    auto Arow = [&](int li) -> double* {
        return a.in_smem ? (Asm + (size_t)li * n) : (a.Aglob + ((size_t)c * a.rows_per + li) * n);
    };

    if (reuse) {
        if (c != 0) return;
        // W_1 = fma(Y0, 1/mu, D) with Y0 = D / dual_norm  ->  G_1 = c^2 Gram(D)
        const double cc = 1.0 + (1.0 / st->dual_norm) * (double)(float)(1.0 / mu);
        eig_control(a, st, K, mu, cc * cc, red, bc);
        if (tid == 0) st->eig_p = max(1, min(st->eig_p, st->svp + 2));
        return;
    }
    if (a.mode == 1) {
        int pf = 0;
        if (eig_fast_path(a, st, K, mu, esm, &pf, cluster)) {
            if (c != 0) return;
            eig_control(a, st, K, mu, 1.0, red, bc);
            if (tid == 0) { st->eig_p = max(1, min(pf, st->svp + 2)); st->eig_fast_iters += 1; }
            return;
        }
    }
    if (c == 0 && tid == 0) st->eig_clk[0] = clock64();
    // ---- load my rows -------------------------------------------------------------------------------------
    for (int li = warp; li < a.rows_per; li += EIG_WARPS) {
        int i = c + li * C;
        if (i < n) {
            double* r = Arow(li);
            const double* g = a.G + (size_t)i * a.npad;
            for (int col = lane; col < n; col += 32) r[col] = g[col];
        }
    }
    __syncthreads();

    // ---- 1. Householder tridiagonalisation ------------------------------------------------------------------
    if (a.in_smem) {
        double* xb = esm + a.tail_off;       // [2][n] column j of the current matrix, by parity of j
        double* pb = xb + 2 * n;             // [n]    p = tau * A v
        if (n <= 64) eig_tridiag_dsmem<2>(a, Asm, xb, pb, st);
        else if (n <= 128) eig_tridiag_dsmem<4>(a, Asm, xb, pb, st);
        else if (n <= 224) eig_tridiag_dsmem<7>(a, Asm, xb, pb, st);
        else if (n <= 320) eig_tridiag_dsmem<10>(a, Asm, xb, pb, st);
        else if (n <= 448) eig_tridiag_dsmem<14>(a, Asm, xb, pb, st);
        else eig_tridiag_dsmem<20>(a, Asm, xb, pb, st);
    } else {
        for (int j = 0; j + 2 < n; ++j) {
            const int par = j & 1;
            if (c == (j % C)) {
                const double* r = Arow(j / C);
                double ss = 0.0;
                for (int i = j + 2 + tid; i < n; i += EIG_THREADS) ss += r[i] * r[i];
                ss = block_sum(ss, red);
                if (tid == 0) {
                    double alpha = r[j + 1];
                    double beta, tau, scale;
                    if (ss == 0.0) { tau = 0.0; beta = alpha; scale = 0.0; }
                    else {
                        beta = -copysign(sqrt(alpha * alpha + ss), alpha);
                        tau = (beta - alpha) / beta;
                        scale = 1.0 / (alpha - beta);
                    }
                    bc[0] = scale;
                    a.tau[j] = tau; a.dd[j] = r[j]; a.ee[j] = beta;
                }
                __syncthreads();
                const double scale = bc[0];
                double* vh = a.Vh + (size_t)j * n;
                for (int i = j + 1 + tid; i < n; i += EIG_THREADS) vh[i] = (i == j + 1) ? 1.0 : r[i] * scale;
            }
            cluster.sync();
            const double tau = ldcg_d(a.tau + j);
            if (tau != 0.0) {
                const double* vh = a.Vh + (size_t)j * n;
                for (int i = tid; i < n; i += EIG_THREADS) v_s[i] = (i > j) ? ldcg_d(vh + i) : 0.0;
                __syncthreads();
                double pv = 0.0;
                for (int li = warp; li < a.rows_per; li += EIG_WARPS) {
                    int i = c + li * C;
                    if (i > j && i < n) {
                        const double* r = Arow(li);
                        double s = 0.0;
                        for (int col = j + 1 + lane; col < n; col += 32) s += r[col] * v_s[col];
                        s = warp_sum(s);
                        double p = tau * s;
                        if (lane == 0) { a.pbuf[par * n + i] = p; pv += p * v_s[i]; }
                    }
                }
                pv = block_sum(pv, red);
                if (tid == 0) a.dotbuf[par * 16 + c] = pv;
            }
            cluster.sync();
            if (tau != 0.0) {
                double dot = 0.0;
                for (int q = 0; q < C; ++q) dot += ldcg_d(a.dotbuf + par * 16 + q);
                const double kc = -0.5 * tau * dot;
                for (int i = tid; i < n; i += EIG_THREADS) w_s[i] = (i > j) ? (ldcg_d(a.pbuf + par * n + i) + kc * v_s[i]) : 0.0;
                __syncthreads();
                for (int li = warp; li < a.rows_per; li += EIG_WARPS) {
                    int i = c + li * C;
                    if (i > j && i < n) {
                        double* r = Arow(li);
                        const double vi = v_s[i], wi = w_s[i];
                        for (int col = j + 1 + lane; col < n; col += 32) r[col] -= vi * w_s[col] + wi * v_s[col];
                    }
                }
                __syncthreads();
            }
        }
    }
    // trailing 2x2 (or smaller)
    if (tid == 0) {
        if (n >= 2) {
            if (c == ((n - 2) % C)) { const double* r = Arow((n - 2) / C); a.dd[n - 2] = r[n - 2]; a.ee[n - 2] = r[n - 1]; a.tau[n - 2] = 0.0; }
            if (c == ((n - 1) % C)) { const double* r = Arow((n - 1) / C); a.dd[n - 1] = r[n - 1]; a.ee[n - 1] = 0.0; a.tau[n - 1] = 0.0; }
        } else if (c == 0) { const double* r = Arow(0); a.dd[0] = r[0]; a.ee[0] = 0.0; a.tau[0] = 0.0; }
    }
    cluster.sync();
    if (c == 0 && tid == 0) st->eig_clk[1] = clock64();

    // ---- 2. top-K eigenvalues of the tridiagonal matrix: multisection on Sturm counts, by the whole cluster -----
    // Every round cuts each bracket into C * S + 1 pieces: CTA c evaluates the shifts c*S .. c*S+S-1, tells every CTA how
    // many of its shifts lie at or below the eigenvalue (they form a prefix: the count is monotone in the shift), and all
    // CTAs update their identical copies of the brackets from the C counts.  One cluster barrier per round.
    // shared-memory carve-up for the remaining phases (the matrix rows are dead now)
    double* d_s = Asm;                 // [n]
    double* e2_s = Asm + n;            // [n]
    double* e_s = Asm + 2 * n;         // [n]
    double* lo_s = Asm + 3 * n;        // [EIG_THREADS]
    double* hi_s = lo_s + EIG_THREADS; // [EIG_THREADS]
    double* nlo_s = hi_s + EIG_THREADS;
    double* nhi_s = nlo_s + EIG_THREADS;
    int* flag_s = reinterpret_cast<int*>(nhi_s + EIG_THREADS);   // [EIG_THREADS]
    double* zs = nhi_s + EIG_THREADS + EIG_THREADS / 2;          // [EIG_BT][n]

    double gl = 1e300, gu = -1e300, emax = 0.0;
    for (int i = tid; i < n; i += EIG_THREADS) {
        double di = ldcg_d(a.dd + i);
        double ei = (i + 1 < n) ? ldcg_d(a.ee + i) : 0.0;
        double em = (i > 0) ? fabs(ldcg_d(a.ee + i - 1)) : 0.0;
        d_s[i] = di; e_s[i] = ei; e2_s[i] = ei * ei;
        gl = fmin(gl, di - fabs(ei) - em);
        gu = fmax(gu, di + fabs(ei) + em);
        emax = fmax(emax, ei * ei);
    }
    gu = block_max(gu, red);
    if (tid == 0) bc[0] = gu;
    gl = -block_max(-gl, red);
    if (tid == 0) bc[1] = gl;
    emax = block_max(emax, red);
    if (tid == 0) bc[2] = emax;
    __syncthreads();
    gu = bc[0]; gl = bc[1]; emax = bc[2];
    const double tnorm = fmax(fabs(gl), fabs(gu));
    const double pivmin = DBL_MIN * fmax(1.0, emax);
    {
        double widen = 2.1 * tnorm * DBL_EPSILON * n + 2.1 * pivmin;
        gl -= widen; gu += widen;
    }
    int* mycnt_s = reinterpret_cast<int*>(nlo_s);                 // [EIG_THREADS] my CTA's count per eigenvalue
    int* cnt_s = reinterpret_cast<int*>(zs);                      // [2][C][EIG_THREADS] counts of every CTA, by round parity
    int* cnt_rem = (lane < C) ? cluster.map_shared_rank(cnt_s, lane) : nullptr;
    int rr = 0;
    for (int kb = 0; kb < K; kb += EIG_THREADS) {
        const int Kb = min(K - kb, EIG_THREADS);
        const int S = max(1, EIG_THREADS / Kb), Stot = C * S;
        const int rounds = (int)ceil(62.0 / log2((double)Stot + 1.0)) + 1;
        const double inv_pieces = 1.0 / (double)(Stot + 1);
        for (int t = tid; t < Kb; t += EIG_THREADS) { lo_s[t] = gl; hi_s[t] = gu; }
        __syncthreads();
        const int kk = tid / S, s = tid - kk * S;
        const bool active = kk < Kb;
        for (int r = 0; r < rounds; ++r, ++rr) {
            const int par = rr & 1;
            int f = 0;
            if (active) {
                const double lo = lo_s[kk], hi = hi_s[kk];
                const double x = lo + (hi - lo) * ((double)(c * S + s + 1) * inv_pieces);
                const int cnt_ge = n - sturm_negcount(d_s, e2_s, n, x, pivmin);   // # eigenvalues >= x
                f = (cnt_ge >= kb + kk + 1);                                          // x <= lambda_k
            }
            flag_s[tid] = f;
            __syncthreads();
            if (active) {
                const int fn = (s + 1 < S) ? flag_s[tid + 1] : 0;
                if (f && !fn) mycnt_s[kk] = s + 1;
                if (s == 0 && !f) mycnt_s[kk] = 0;
            }
            __syncthreads();
            // one warp per eigenvalue group: lanes < C deliver this CTA's count to every CTA
            for (int k2 = warp; k2 < Kb; k2 += EIG_WARPS)
                if (lane < C) cnt_rem[(par * C + c) * EIG_THREADS + k2] = mycnt_s[k2];
            cluster.sync();
            if (tid < Kb) {
                int tot = 0;
                for (int q = 0; q < C; ++q) tot += cnt_s[(par * C + q) * EIG_THREADS + tid];
                const double lo = lo_s[tid], hi = hi_s[tid];
                if (tot > 0) lo_s[tid] = lo + (hi - lo) * ((double)tot * inv_pieces);
                if (tot < Stot) hi_s[tid] = lo + (hi - lo) * ((double)(tot + 1) * inv_pieces);
            }
            __syncthreads();
        }
        if (c == 0) for (int t = tid; t < Kb; t += EIG_THREADS) a.lam[kb + t] = 0.5 * (lo_s[t] + hi_s[t]);
        __syncthreads();
    }
    if (c != 0) return;                                           // the rest runs in CTA 0 (nobody writes into a CTA after its last barrier)
    __threadfence_block();
    __syncthreads();
    if (tid == 0) st->eig_clk[2] = clock64();

    // ---- 3. eigenvectors of the tridiagonal matrix: inverse iteration, one thread per vector ---------------------
    // The six work arrays of a vector live in shared memory ([array][i][slot], slot fastest -> conflict-free), so the
    // sequential recurrences run at shared-memory latency; vectors are processed in batches of `kbcap`.
    double* iw_s = zs;                                   // aliases the back-transformation scratch (later phase)
    const int kbcap = max(1, min(EIG_THREADS, (int)(a.iw_smem_doubles / ((size_t)6 * n))));
    for (int kb0 = 0; kb0 < K; kb0 += kbcap) {
        const int k = kb0 + tid;
        if (tid < kbcap && k < K) {
            const double lamk = a.lam[k];
            double* Up = iw_s + (size_t)0 * n * kbcap + tid;
            double* Uq = iw_s + (size_t)1 * n * kbcap + tid;
            double* Ur = iw_s + (size_t)2 * n * kbcap + tid;
            double* Mm = iw_s + (size_t)3 * n * kbcap + tid;
            double* Sw = iw_s + (size_t)4 * n * kbcap + tid;
            double* Bz = iw_s + (size_t)5 * n * kbcap + tid;
            const double ptol = fmax(DBL_EPSILON * tnorm, pivmin);
            // factor T - lam I = P L U  (partial pivoting; U has two super-diagonals)
            double p = d_s[0] - lamk, q = (n > 1) ? e_s[0] : 0.0, rr = 0.0;
            for (int i = 0; i + 1 < n; ++i) {
                const double sub = e_s[i];
                const double an = d_s[i + 1] - lamk;
                const double en = (i + 2 < n) ? e_s[i + 1] : 0.0;
                if (fabs(p) >= fabs(sub)) {
                    if (fabs(p) < ptol) p = copysign(ptol, p);
                    const double mlt = sub / p;
                    Up[(size_t)i * kbcap] = p; Uq[(size_t)i * kbcap] = q; Ur[(size_t)i * kbcap] = rr;
                    Mm[(size_t)i * kbcap] = mlt; Sw[(size_t)i * kbcap] = 0.0;
                    p = an - mlt * q; q = en - mlt * rr; rr = 0.0;
                } else {
                    const double mlt = p / sub;
                    Up[(size_t)i * kbcap] = sub; Uq[(size_t)i * kbcap] = an; Ur[(size_t)i * kbcap] = en;
                    Mm[(size_t)i * kbcap] = mlt; Sw[(size_t)i * kbcap] = 1.0;
                    p = q - mlt * an; q = rr - mlt * en; rr = 0.0;
                }
            }
            if (fabs(p) < ptol) p = copysign(ptol, p);
            Up[(size_t)(n - 1) * kbcap] = p; Uq[(size_t)(n - 1) * kbcap] = 0.0; Ur[(size_t)(n - 1) * kbcap] = 0.0;
            for (int i = 0; i < n; ++i) Bz[(size_t)i * kbcap] = hash_unit((unsigned)i, (unsigned)k);
            for (int itn = 0; itn < 3; ++itn) {
                // forward: apply P L^{-1}
                double bi = Bz[0];
                for (int i = 0; i + 1 < n; ++i) {
                    double bn = Bz[(size_t)(i + 1) * kbcap];
                    if (Sw[(size_t)i * kbcap] != 0.0) { double t = bi; bi = bn; bn = t; }
                    bn -= Mm[(size_t)i * kbcap] * bi;
                    Bz[(size_t)i * kbcap] = bi;
                    bi = bn;
                }
                Bz[(size_t)(n - 1) * kbcap] = bi;
                // backward: solve U z = b
                double z1 = 0.0, z2 = 0.0, zmax = 0.0;
                for (int i = n - 1; i >= 0; --i) {
                    double z = (Bz[(size_t)i * kbcap] - Uq[(size_t)i * kbcap] * z1 - Ur[(size_t)i * kbcap] * z2) / Up[(size_t)i * kbcap];
                    Bz[(size_t)i * kbcap] = z;
                    z2 = z1; z1 = z;
                    zmax = fmax(zmax, fabs(z));
                }
                const double sc = (zmax > 0.0) ? 1.0 / zmax : 1.0;
                for (int i = 0; i < n; ++i) Bz[(size_t)i * kbcap] *= sc;
            }
            double nn = 0.0;
            for (int i = 0; i < n; ++i) { double z = Bz[(size_t)i * kbcap]; nn += z * z; }
            const double sc = 1.0 / sqrt(nn);
            double* zrow = a.Z + (size_t)k * n;
            for (int i = 0; i < n; ++i) zrow[i] = Bz[(size_t)i * kbcap] * sc;
        }
        __syncthreads();
    }
    __threadfence_block();
    __syncthreads();
    if (tid == 0) st->eig_clk[3] = clock64();

    // ---- 3b. CGS2 re-orthogonalisation among close eigenvalues (descending order) -------------------------------
    {
        const double ortol = 1e-3 * tnorm;
        double* coef = lo_s;   // [<= EIG_THREADS] reuse
        for (int k = 1; k < K; ++k) {
            const double lamk = a.lam[k];
            int j0 = k;
            while (j0 > 0 && fabs(a.lam[j0 - 1] - lamk) <= ortol) --j0;
            if (j0 == k) continue;                       // uniform across the block
            double* zk = a.Z + (size_t)k * n;
            for (int pass = 0; pass < 2; ++pass) {
                for (int jb = j0; jb < k; jb += EIG_THREADS) {
                    const int je = min(k, jb + EIG_THREADS);
                    for (int j = jb + warp; j < je; j += EIG_WARPS) {
                        const double* zj = a.Z + (size_t)j * n;
                        double s = 0.0;
                        for (int i = lane; i < n; i += 32) s += zj[i] * zk[i];
                        s = warp_sum(s);
                        if (lane == 0) coef[j - jb] = s;
                    }
                    __syncthreads();
                    for (int i = tid; i < n; i += EIG_THREADS) {
                        double acc = zk[i];
                        for (int j = jb; j < je; ++j) acc -= coef[j - jb] * a.Z[(size_t)j * n + i];
                        zk[i] = acc;
                    }
                    __threadfence_block();
                    __syncthreads();
                }
            }
            double nn = 0.0;
            for (int i = tid; i < n; i += EIG_THREADS) nn += zk[i] * zk[i];
            nn = block_sum(nn, red);
            if (tid == 0) bc[0] = nn;
            __syncthreads();
            const double sc = 1.0 / sqrt(bc[0]);
            for (int i = tid; i < n; i += EIG_THREADS) zk[i] *= sc;
            __threadfence_block();
            __syncthreads();
        }
    }

    if (tid == 0) st->eig_clk[4] = clock64();
    // ---- 4. back-transformation z <- H_0 H_1 ... H_{n-3} z, one warp per vector ---------------------------------
    // tau is staged in shared memory and the next reflector row is prefetched into registers while the current one
    // is applied, so the chain of n dependent steps does not pay an L2 round trip per step.
    double* tau_s = d_s;                                  // d_s / e_s / e2_s are dead now
    for (int i = tid; i < n; i += EIG_THREADS) tau_s[i] = a.tau[i];
    __syncthreads();
    if (n <= 64) eig_backtransform<2>(a, K, tau_s, warp, lane);
    else if (n <= 128) eig_backtransform<4>(a, K, tau_s, warp, lane);
    else if (n <= 224) eig_backtransform<7>(a, K, tau_s, warp, lane);
    else if (n <= 320) eig_backtransform<10>(a, K, tau_s, warp, lane);
    else if (n <= 448) eig_backtransform<14>(a, K, tau_s, warp, lane);
    else eig_backtransform<20>(a, K, tau_s, warp, lane);
    __threadfence_block();
    __syncthreads();

    if (tid == 0) st->eig_clk[5] = clock64();
    eig_control(a, st, K, mu, 1.0, red, bc);
    // warm start of the next call: the kept vectors plus two guards (rows 0..eig_p-1 of Z)
    if (tid == 0 && a.mode != 2) {
        const int pcap = min(K, eig_fast_layout(n, C).PM);
        st->eig_p = (a.mode == 0) ? pcap : max(1, min(pcap, st->svp + 2));
        if (a.mode == 0) st->eig_fast_iters = 0;
    }
}

// -------------------------------------------------------------------------------------------------------------
static size_t eig_phase_doubles(int n) {
    return (size_t)3 * n + 4 * EIG_THREADS + EIG_THREADS / 2 + (size_t)EIG_BT * n + 16;
}

EigPlan make_eig_plan(int n, int npad) {
    EigPlan p;
    p.n = n; p.npad = npad;
    int C = 1;
    const int rows_target = 40;
    while (C < 16 && (n + C - 1) / C > rows_target) C *= 2;
    const size_t cap = 225 * 1024;
    auto bytes_for = [&](int Cc, bool in_smem) {
        size_t rows = (size_t)(n + Cc - 1) / Cc;
        size_t mat = in_smem ? rows * n + 3 * (size_t)n : 0;     // + exchange buffers of the tridiagonalisation
        size_t ph = eig_phase_doubles(n);
        return (2 * (size_t)n + 64 + (mat > ph ? mat : ph)) * sizeof(double);
    };
    p.in_smem = 1;
    while (bytes_for(C, true) > cap && C < 16) C *= 2;
    if (bytes_for(C, true) > cap) p.in_smem = 0;
    p.C = C;
    p.rows_per = (n + C - 1) / C;
    p.smem_bytes = std::max(bytes_for(C, p.in_smem != 0), cap);      // CTA 0 uses the slack for the inverse iteration
    p.kcap = n;
    // workspace: Aglob + Vh + tau + dd + ee + pbuf + dotbuf + iw
    p.work_doubles = (size_t)C * p.rows_per * n + (size_t)n * n + 3 * (size_t)n + 2 * (size_t)n + 32;
    return p;
}

int launch_eig(const EigPlan& p, const double* G, const double* comm_max, EigBuffers b, DevState* st, int mode,
               int k_override, cudaStream_t stream) {
    static unsigned long long attr_devs = 0;      // one bit per device: the attribute is per (function, device)
    if (first_call_on_device(&attr_devs)) {
        BSUB_CUDA_CHECK(cudaFuncSetAttribute(eig_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
        BSUB_CUDA_CHECK(cudaFuncSetAttribute(eig_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    }
    if (p.smem_bytes > 225 * 1024) { set_error("eig: n=%d needs %zu B of shared memory", p.n, p.smem_bytes); return -1; }
    EigArgs a;
    a.G = G; a.comm_max = comm_max; a.n = p.n; a.npad = p.npad; a.C = p.C; a.rows_per = p.rows_per;
    a.in_smem = p.in_smem; a.kcap = p.kcap; a.mode = mode; a.k_override = k_override;
    a.tail_off = 2 * p.n + 64 + p.rows_per * p.n;
    double* w = b.work;
    a.Aglob = w; w += (size_t)p.C * p.rows_per * p.n;
    a.Vh = w;    w += (size_t)p.n * p.n;
    a.tau = w;   w += p.n;
    a.dd = w;    w += p.n;
    a.ee = w;    w += p.n;
    a.pbuf = w;  w += 2 * (size_t)p.n;
    a.dotbuf = w; w += 32;
    a.iw_smem_doubles = (p.smem_bytes / sizeof(double)) - (2 * (size_t)p.n + 64) - (3 * (size_t)p.n + 4 * EIG_THREADS + EIG_THREADS / 2);
    a.lam = b.lam; a.Z = b.Z; a.Vr = b.Vr; a.VC = b.VC; a.vstride = b.vstride; a.st = st;
    a.fast_ok = (mode == 1 && getenv("BSUB_NO_EIG_FAST") == nullptr) ? 1 : 0;
    a.smem_total = p.smem_bytes;

    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(p.C); cfg.blockDim = dim3(EIG_THREADS); cfg.dynamicSmemBytes = p.smem_bytes; cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = p.C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    BSUB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, eig_kernel, a));
    return 0;
}

}  // namespace bsub
