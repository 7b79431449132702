// shrink_tma.cu -- pass B of the ALM iteration as a TMA + mbarrier pipelined kernel (the fast path; shrink.cu keeps
// the plain-load version for image heights that are not a multiple of 4, which TMA strides cannot express).
//
//   T = Vr^T W ; L = VC T ; G_S = D - L + Y/mu ; S = prox(G_S) ; Z = D - L - S ; Y += mu Z ; sum Z^2
//   (/root/reference/inexact_alm_lsd.py:131-167; prox_flat :71-79 as the closed-form l_inf tile prox)
//
// One persistent thread-block cluster of Cf CTAs walks tiles of 3 image columns x R rows x ALL frames; CTA `rank`
// owns frames [rank*nf, rank*nf + nf).  Per tile and CTA:
//   * one elected thread issues three 3-D TMA box loads {R rows, 3 cols, nf frames} of D, S, Y into a stage of
//     shared memory (out-of-image rows/cols/frames are zero-filled by the hardware, which is exactly the ragged
//     3x3 tile semantics); two stages, so the loads of tile i+2 and the stores of tile i overlap the math of i+1;
//   * sweep 1 accumulates the partial T over the CTA's frames from shared memory; partials of the Cf CTAs are
//     exchanged through L2 around ONE hardware cluster barrier;
//   * sweep 2 builds a = D - L in place, runs the prox + dual update per 3x3 group in shared memory, and the
//     results leave through two TMA box stores (S and Y; out-of-image elements are clipped by the hardware).
// Two CTAs share an SM (one when no tile fits half of shared memory) so that the barrier / exchange bubbles of one tile
// are filled by another CTA.
// HBM traffic is exactly read D,S,Y + write S,Y = 20 B per matrix element.
#include <cooperative_groups.h>
#include <algorithm>
#include "common.cuh"
#include "kernels.h"
#include "tma.cuh"

namespace cg = cooperative_groups;

namespace bsub {

constexpr int ST_KC = 8;          // singular vectors per register chunk
constexpr size_t ST_SMEM_CAP = 227 * 1024 - 256;
constexpr int ST_NT = 256;         // threads per CTA

struct ShrinkTmaArgs {
    float* T; float* tpart; const float* Vr; const float* VC; int vstride;
    long long ld;
    int n, rows, cols, R, P, NQ, NFL, Cf, nf, KR, BS;     // BS = floats per stage buffer (nf*P rounded up to 128 B)
    int ntile_r; long long ntiles; int nclusters;
    const DevState* st;
    double* part_zz; unsigned long long* part_nnz; float* part_max;
    int mode, min_rank;                                   // kernel is a no-op when svp < min_rank (the stream kernel did it)
};

#define ST_CE(i, j) { const float hi_ = fmaxf(u[i], u[j]), lo_ = fminf(u[i], u[j]); u[i] = hi_; u[j] = lo_; }
// Clip level of the l1-ball projection: theta >= 0 with sum_i max(a_i - theta, 0) = z, for a_i >= 0, sum a > z.
// Optimal 25-comparator sorting network for 9 inputs (descending), checked exhaustively by the 0-1 principle.
__device__ __forceinline__ float st_clip_level9(const float* a_in, float z) {
    float u[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) u[i] = a_in[i];
    ST_CE(0, 3) ST_CE(1, 7) ST_CE(2, 5) ST_CE(4, 8)
    ST_CE(0, 7) ST_CE(2, 4) ST_CE(3, 8) ST_CE(5, 6)
    ST_CE(0, 2) ST_CE(1, 3) ST_CE(4, 5) ST_CE(7, 8)
    ST_CE(1, 4) ST_CE(3, 6) ST_CE(5, 7)
    ST_CE(0, 1) ST_CE(2, 4) ST_CE(3, 5) ST_CE(6, 8)
    ST_CE(2, 3) ST_CE(4, 5) ST_CE(6, 7)
    ST_CE(1, 2) ST_CE(3, 4) ST_CE(5, 6)
    const float inv[9] = {1.f, 0.5f, 1.f / 3.f, 0.25f, 0.2f, 1.f / 6.f, 1.f / 7.f, 0.125f, 1.f / 9.f};
    float cs = 0.f, theta = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        cs += u[k];
        const float t = (cs - z) * inv[k];
        if (u[k] > t) theta = t;
    }
    return theta;
}

// partial T of this thread's pixel quad over its frames, KCNT live singular vectors of the chunk
template <int KCNT>
__device__ __forceinline__ void sweep1_acc(float (&acc)[ST_KC][4], const float* bD, const float* bS, const float* bY,
                                           const float* Vs, int P, int qd, int fl, int NFL, int nfr, float inv_mu) {
#pragma unroll 2
    for (int f = fl; f < nfr; f += NFL) {
        const float4 d4 = *reinterpret_cast<const float4*>(bD + (size_t)f * P + 4 * qd);
        const float4 s4 = *reinterpret_cast<const float4*>(bS + (size_t)f * P + 4 * qd);
        const float4 y4 = *reinterpret_cast<const float4*>(bY + (size_t)f * P + 4 * qd);
        float4 w;
        w.x = (d4.x - s4.x) + y4.x * inv_mu; w.y = (d4.y - s4.y) + y4.y * inv_mu;
        w.z = (d4.z - s4.z) + y4.z * inv_mu; w.w = (d4.w - s4.w) + y4.w * inv_mu;
        const float4 va = *reinterpret_cast<const float4*>(Vs + f * ST_KC);
        const float4 vb = *reinterpret_cast<const float4*>(Vs + f * ST_KC + 4);
        const float vv[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
#pragma unroll
        for (int k = 0; k < KCNT; ++k) {
            acc[k][0] = fmaf(vv[k], w.x, acc[k][0]); acc[k][1] = fmaf(vv[k], w.y, acc[k][1]);
            acc[k][2] = fmaf(vv[k], w.z, acc[k][2]); acc[k][3] = fmaf(vv[k], w.w, acc[k][3]);
        }
    }
}

// a = D - (VC chunk) * T chunk, in place in the D stage buffer
template <int KCNT>
__device__ __forceinline__ void sweep2a_sub(float* bD, const float* Tp, const float* Vs, int P, int qd, int fl, int NFL, int nfr) {
    float4 t4[KCNT];
#pragma unroll
    for (int k = 0; k < KCNT; ++k) t4[k] = *reinterpret_cast<const float4*>(Tp + (size_t)k * P + 4 * qd);
#pragma unroll 2
    for (int f = fl; f < nfr; f += NFL) {
        const float4 va = *reinterpret_cast<const float4*>(Vs + f * ST_KC);
        const float4 vb = *reinterpret_cast<const float4*>(Vs + f * ST_KC + 4);
        const float vv[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
        float4 l = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < KCNT; ++k) {
            l.x = fmaf(vv[k], t4[k].x, l.x); l.y = fmaf(vv[k], t4[k].y, l.y);
            l.z = fmaf(vv[k], t4[k].z, l.z); l.w = fmaf(vv[k], t4[k].w, l.w);
        }
        float4* dp = reinterpret_cast<float4*>(bD + (size_t)f * P + 4 * qd);
        float4 d4 = *dp;
        d4.x -= l.x; d4.y -= l.y; d4.z -= l.z; d4.w -= l.w;
        *dp = d4;
    }
}

#define ST_DISPATCH_K(kcnt, CALL)                 \
    switch (kcnt) {                               \
        case 1: { constexpr int K_ = 1; CALL; } break; \
        case 2: { constexpr int K_ = 2; CALL; } break; \
        case 3: { constexpr int K_ = 3; CALL; } break; \
        case 4: { constexpr int K_ = 4; CALL; } break; \
        case 5: { constexpr int K_ = 5; CALL; } break; \
        case 6: { constexpr int K_ = 6; CALL; } break; \
        case 7: { constexpr int K_ = 7; CALL; } break; \
        default: { constexpr int K_ = 8; CALL; } break; \
    }

__global__ void __launch_bounds__(ST_NT, 2)
shrink_tma_kernel(const __grid_constant__ CUtensorMap mapD, const __grid_constant__ CUtensorMap mapS,
                  const __grid_constant__ CUtensorMap mapY, const __grid_constant__ CUtensorMap mapOut, ShrinkTmaArgs a) {
    const DevState* st = a.st;
    if (st->done) return;
    if (st->svp < a.min_rank) {
        if (threadIdx.x == 0) { a.part_zz[blockIdx.x] = 0.0; a.part_nnz[blockIdx.x] = 0ull; a.part_max[blockIdx.x] = 0.f; }
        return;
    }
    cg::cluster_group cluster = cg::this_cluster();
    const int tid = threadIdx.x;
    const int rank = blockIdx.x % a.Cf, cl = blockIdx.x / a.Cf;
    const int f0 = rank * a.nf;
    const int nfr = max(0, min(a.nf, a.n - f0));
    const int P = a.P, NQ = a.NQ, NFL = a.NFL, R = a.R, KR = a.KR;
    const int r = st->svp;
    const double mu_d = st->mu;
    const float inv_mu = (float)(1.0 / mu_d), mu_f = (float)mu_d;
    const float lamq = (float)(st->lambda / mu_d);
    const int nchunk = (r + ST_KC - 1) / ST_KC;

    extern __shared__ __align__(128) unsigned char st_smem_raw[];
    const size_t stage_floats = (size_t)3 * a.BS;
    float* stage0 = reinterpret_cast<float*>(st_smem_raw);          // 2 stages x {D, S, Y} x [nf][P]
    float* scr = stage0 + 2 * stage_floats;                         // [NFL][KR][P]
    float* Tpart = scr + (size_t)NFL * KR * P;                      // [2][ST_KC][P]  this CTA's partial T (read by peers)
    float* Tp = Tpart + (size_t)2 * ST_KC * P;                      // [ST_KC][P]     summed T chunk
    float* Vr_s = Tp + (size_t)ST_KC * P;                           // [nf][ST_KC]
    float* VC_s = Vr_s + (size_t)a.nf * ST_KC;                      // [nf][ST_KC]
    uint64_t* full = reinterpret_cast<uint64_t*>(VC_s + (size_t)a.nf * ST_KC);   // [2]
    __shared__ double redd[32];

    const int qd = tid % NQ, fl = tid / NQ;
    const bool tact = fl < NFL;
    const int RQ = R / 4;

    if (tid == 0) {
        mbar_init(&full[0], 1); mbar_init(&full[1], 1);
        mbar_fence_init();
        tma_prefetch_desc(&mapD); tma_prefetch_desc(&mapS); tma_prefetch_desc(&mapY); tma_prefetch_desc(&mapOut);
    }
    auto load_V = [&](int kc) {                           // Vr / VC rows of my frames for singular vectors [8kc, 8kc+8)
        const int k0 = kc * ST_KC;
        for (int idx = tid; idx < nfr * ST_KC; idx += ST_NT) {
            const int f = idx / ST_KC, k = idx - f * ST_KC;
            const bool ok = (k0 + k) < r;
            Vr_s[idx] = ok ? a.Vr[(size_t)(f0 + f) * a.vstride + k0 + k] : 0.f;
            VC_s[idx] = ok ? a.VC[(size_t)(f0 + f) * a.vstride + k0 + k] : 0.f;
        }
    };
    if (nchunk == 1) load_V(0);                           // common case: once per kernel, not once per tile
    __syncthreads();

    const uint32_t tx_bytes = (uint32_t)((size_t)3 * a.nf * P * sizeof(float));
    auto tile_origin = [&](long long tl, int& j0, int& i0) {
        const int tcx = (int)(tl / a.ntile_r), trx = (int)(tl - (long long)tcx * a.ntile_r);
        j0 = 3 * tcx; i0 = trx * R;
    };
    auto issue_load = [&](long long tl, int s) {          // elected thread
        int j0, i0;
        tile_origin(tl, j0, i0);
        float* b = stage0 + (size_t)s * stage_floats;
        mbar_expect_tx(&full[s], tx_bytes);
        tma_load_3d(b, &mapD, &full[s], i0, j0, f0);
        tma_load_3d(b + (size_t)a.BS, &mapS, &full[s], i0, j0, f0);
        tma_load_3d(b + (size_t)2 * a.BS, &mapY, &full[s], i0, j0, f0);
    };

    double zz_acc = 0.0;
    unsigned int nnz_acc = 0u;
    float max_acc = 0.f;

    // prologue: two tiles in flight
    if (tid == 0) {
        if (cl < a.ntiles) issue_load(cl, 0);
        if (cl + a.nclusters < a.ntiles) issue_load(cl + a.nclusters, 1);
    }
    float* myscratch = a.tpart + (size_t)blockIdx.x * (size_t)a.n * P;    // only used when svp > 8

    int xslot = 0;                                        // parity of the DSMEM exchange step
    long long it = 0;
    for (long long tl = cl; tl < a.ntiles; tl += a.nclusters, ++it) {
        const int s = (int)(it & 1);
        const uint32_t par = (uint32_t)((it >> 1) & 1);
        int j0, i0;
        tile_origin(tl, j0, i0);
        float* bD = stage0 + (size_t)s * stage_floats;
        float* bS = bD + (size_t)a.BS;
        float* bY = bS + (size_t)a.BS;

        mbar_wait(&full[s], par);

        // ---------------- phase A: T chunk by chunk (sweep 1, CTA reduction, DSMEM exchange) ----------------
        for (int kc = 0; kc < nchunk; ++kc) {
            const int k0 = kc * ST_KC;
            const int kcnt = min(ST_KC, r - k0);
            if (nchunk > 1) { __syncthreads(); load_V(kc); __syncthreads(); }
            float acc[ST_KC][4];
#pragma unroll
            for (int k = 0; k < ST_KC; ++k) { acc[k][0] = acc[k][1] = acc[k][2] = acc[k][3] = 0.f; }
            if (tact) { ST_DISPATCH_K(kcnt, (sweep1_acc<K_>(acc, bD, bS, bY, Vr_s, P, qd, fl, NFL, nfr, inv_mu))); }
            float* tpart_mine = Tpart + (size_t)xslot * ST_KC * P;
            for (int kr0 = 0; kr0 < kcnt; kr0 += KR) {
                if (kr0 > 0) __syncthreads();                      // scr is reused by the next round
                if (tact) {
#pragma unroll
                    for (int k = 0; k < ST_KC; ++k)
                        if (k >= kr0 && k < kr0 + KR && k < kcnt)
                            *reinterpret_cast<float4*>(scr + ((size_t)(fl * KR + (k - kr0))) * P + 4 * qd) =
                                make_float4(acc[k][0], acc[k][1], acc[k][2], acc[k][3]);
                }
                __syncthreads();
                const int kend = min(KR, kcnt - kr0);
                for (int idx = tid; idx < kend * NQ; idx += ST_NT) {
                    const int k = idx / NQ, q = idx - k * NQ;
                    float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
                    for (int l = 0; l < NFL; ++l) {
                        const float4 v = *reinterpret_cast<const float4*>(scr + ((size_t)(l * KR + k)) * P + 4 * q);
                        sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
                    }
                    *reinterpret_cast<float4*>(tpart_mine + (size_t)(kr0 + k) * P + 4 * q) = sum;
                }
            }
            // all partials of the cluster are in place (this is also the CTA barrier after the reduction)
            cluster.sync();
            for (int idx = tid; idx < kcnt * NQ; idx += ST_NT) {
                const int k = idx / NQ, q = idx - k * NQ;
                float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int rk = 0; rk < a.Cf; ++rk) {                 // fixed order: every CTA gets bit-identical T
                    const float* rp = cluster.map_shared_rank(tpart_mine, rk);
                    const float4 v = *reinterpret_cast<const float4*>(rp + (size_t)k * P + 4 * q);
                    sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
                }
                if (rank == 0) {                  // keep T for the final materialisation of L (rows % 4 == 0 here)
                    const int c2 = q / RQ, i2 = (q - c2 * RQ) * 4;
                    const int j2 = j0 + c2, row2 = i0 + i2;
                    if (j2 < a.cols && row2 < a.rows) stg4(a.T + (size_t)(k0 + k) * a.ld + (long long)j2 * a.rows + row2, sum);
                }
                if (nchunk == 1) *reinterpret_cast<float4*>(Tp + (size_t)k * P + 4 * q) = sum;
                else *reinterpret_cast<float4*>(myscratch + (size_t)(k0 + k) * P + 4 * q) = sum;
            }
            xslot ^= 1;
        }

        // ---------------- phase B: a = D - L in place ----------------
        for (int kc = 0; kc < nchunk; ++kc) {
            const int k0 = kc * ST_KC;
            const int kcnt = min(ST_KC, r - k0);
            if (nchunk > 1) {
                __syncthreads();
                load_V(kc);
                for (int idx = tid; idx < kcnt * NQ; idx += ST_NT) {
                    const int k = idx / NQ, q = idx - k * NQ;
                    *reinterpret_cast<float4*>(Tp + (size_t)k * P + 4 * q) =
                        *reinterpret_cast<const float4*>(myscratch + (size_t)(k0 + k) * P + 4 * q);
                }
            }
            __syncthreads();
            if (tact) { ST_DISPATCH_K(kcnt, (sweep2a_sub<K_>(bD, Tp, VC_s, P, qd, fl, NFL, nfr))); }
        }
        __syncthreads();

        // ---------------- sweep 2b: prox + dual update in shared memory (S_new -> bS, Y_new -> bY) ----------------
        if (a.mode == SHRINK_FLAT3) {
            const int NG = R / 3;
            for (int itx = tid; itx < nfr * NG; itx += ST_NT) {
                const int f = itx / NG, g = itx - f * NG;
                const float* dsp = bD + (size_t)f * P + 3 * g;
                float* ssp = bS + (size_t)f * P + 3 * g;
                float* ysp = bY + (size_t)f * P + 3 * g;
                float av[9], yv[9], x[9], ax[9];
                float sabs = 0.f;
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int dr = 0; dr < 3; ++dr) {
                        const int e = c * 3 + dr;
                        av[e] = dsp[c * R + dr];
                        yv[e] = ysp[c * R + dr];
                        x[e] = fmaf(yv[e], inv_mu, av[e]);      // G_S
                        ax[e] = fabsf(x[e]);
                        sabs += ax[e];
                    }
                float zl = 0.f;
                if (!(sabs > lamq)) {
                    // whole tile inside the l1 ball: S = 0, Z = D - L
#pragma unroll
                    for (int c = 0; c < 3; ++c)
#pragma unroll
                        for (int dr = 0; dr < 3; ++dr) {
                            const int e = c * 3 + dr;
                            ssp[c * R + dr] = 0.f;
                            ysp[c * R + dr] = fmaf(mu_f, av[e], yv[e]);
                            zl = fmaf(av[e], av[e], zl);
                        }
                } else {
                    const float theta = st_clip_level9(ax, lamq);
#pragma unroll
                    for (int c = 0; c < 3; ++c)
#pragma unroll
                        for (int dr = 0; dr < 3; ++dr) {
                            const int e = c * 3 + dr;
                            const float sv = copysignf(fminf(ax[e], theta), x[e]);
                            const float z = av[e] - sv;                // Z = D - L - S
                            ssp[c * R + dr] = sv;
                            ysp[c * R + dr] = fmaf(mu_f, z, yv[e]);    // Y += mu Z
                            zl = fmaf(z, z, zl);
                            nnz_acc += (sv != 0.f);
                            max_acc = fmaxf(max_acc, fabsf(sv));
                        }
                }
                zz_acc += (double)zl;
            }
        } else if (a.mode == SHRINK_L1) {
            for (int itx = tid; itx < nfr * P; itx += ST_NT) {
                const float av = bD[itx], yv = bY[itx];
                const float x = av + yv * inv_mu;
                const float sv = copysignf(fmaxf(fabsf(x) - lamq, 0.f), x);
                const float z = av - sv;
                bS[itx] = sv; bY[itx] = fmaf(mu_f, z, yv);
                zz_acc += (double)(z * z);
                nnz_acc += (sv != 0.f);
                max_acc = fmaxf(max_acc, fabsf(sv));
            }
        } else {   // SHRINK_SPILL: G_S goes out through mapOut (= U); the dual update happens in lowrank_kernel<true>
            for (int itx = tid; itx < nfr * P; itx += ST_NT) bS[itx] = bD[itx] + bY[itx] * inv_mu;
        }
        fence_proxy_async_smem();          // my generic writes -> visible to the TMA store
        __syncthreads();

        // ---------------- stores + refill of this stage ----------------
        if (tid == 0) {
            tma_store_3d(&mapOut, bS, i0, j0, f0);
            if (a.mode != SHRINK_SPILL) tma_store_3d(&mapY, bY, i0, j0, f0);
            tma_store_commit();
            const long long nxt = tl + 2ll * a.nclusters;
            if (nxt < a.ntiles) {
                tma_store_wait_read<0>();  // the stores have read the stage; it may be overwritten
                issue_load(nxt, s);
            }
        }
    }
    if (tid == 0) tma_store_wait_all<0>();
    cluster.sync();                        // no CTA leaves while a peer may still read its partials through DSMEM

    double zt = block_sum(zz_acc, redd);
    if (tid == 0) a.part_zz[blockIdx.x] = zt;
    double nt = block_sum((double)nnz_acc, redd);
    if (tid == 0) a.part_nnz[blockIdx.x] = (unsigned long long)(nt + 0.5);
    double mt = block_max((double)max_acc, redd);
    if (tid == 0) a.part_max[blockIdx.x] = (float)mt;
}

// -------------------------------------------------------------------------------------------------------------
static size_t st_smem_bytes(int n, int R, int Cf, int KR) {
    const int P = 3 * R, NQ = P / 4, NFL = ST_NT / NQ;
    const int nf = (n + Cf - 1) / Cf;
    const size_t bs = ((size_t)nf * P + 31) / 32 * 32;
    size_t fl = (size_t)6 * bs + (size_t)NFL * KR * P + (size_t)3 * ST_KC * P + (size_t)2 * nf * ST_KC;
    return fl * sizeof(float) + 64;
}

bool make_shrink_tma_plan(int n, int rows, int cols, long long ld, int num_sms, int R_hint, int Cf_hint, ShrinkTmaPlan* out) {
    if (rows % 4 != 0 || rows < 12) return false;               // TMA global strides must be multiples of 16 B
    ShrinkTmaPlan p;
    p.n = n; p.rows = rows; p.cols = cols; p.ld = ld;
    int occ = 2;                                                // CTAs per SM the shared-memory budget is sized for
    const int rows12 = ((rows + 11) / 12) * 12;
    auto cap_for = [&](int o) { return (size_t)((228 * 1024) / o - 1024 - 512); };
    auto fits = [&](int Rr, int Cc, int Kr, int o) {
        return (n + Cc - 1) / Cc <= 256 && 3 * Rr / 4 <= ST_NT && st_smem_bytes(n, Rr, Cc, Kr) <= std::min(cap_for(o), ST_SMEM_CAP);
    };
    int R = 0, Cf = 0, KR = 0;
    for (; occ >= 1 && R == 0; --occ) {
        // largest tile (rows multiple of 12) first; clusters up to 8 CTAs split the frames
        const int r_hi = R_hint > 0 ? ((R_hint + 11) / 12) * 12 : 48;
        for (int krmin = 4; krmin >= 2 && R == 0; krmin -= 2)      // prefer few reduction rounds over tall tiles
            for (int Rr = std::min(std::min(r_hi, rows12), 252); Rr >= 24 && R == 0; Rr -= 12)
                for (int Cc = (Cf_hint > 0 ? Cf_hint : 1); Cc <= (Cf_hint > 0 ? Cf_hint : 8) && R == 0; Cc *= 2)
                    for (int Kr = 8; Kr >= krmin && R == 0; Kr >>= 1)
                        if (fits(Rr, Cc, Kr, occ)) { R = Rr; Cf = Cc; KR = Kr; }
        if (R == 0 && std::min(rows12, 252) < 24 && fits(12, Cf_hint > 0 ? Cf_hint : 8, 2, occ)) { R = 12; Cf = Cf_hint > 0 ? Cf_hint : 8; KR = 2; }
        if (R != 0) break;
    }
    if (R == 0) return false;
    p.R = R; p.P = 3 * R; p.Cf = Cf; p.nf = (n + Cf - 1) / Cf; p.KR = KR;
    p.bufstride = (int)(((size_t)p.nf * p.P + 31) / 32 * 32);
    p.smem_bytes = st_smem_bytes(n, R, Cf, KR);
    p.ntile_r = (rows + R - 1) / R;
    p.ntile_c = (cols + 2) / 3;
    p.ntiles = (long long)p.ntile_r * p.ntile_c;
    long long ncl = ((long long)num_sms * occ) / Cf;
    if (ncl < 1) ncl = 1;
    if (ncl > p.ntiles) ncl = p.ntiles;
    p.grid_clusters = (int)ncl;
    p.nparts = p.grid_clusters * Cf;
    p.tpart_floats = (size_t)p.grid_clusters * Cf * (size_t)n * p.P;      // per-CTA scratch, only touched when svp > 8
    *out = p;
    return true;
}

int make_shrink_tma_maps(const ShrinkTmaPlan& p, const float* D, float* S, float* Y, float* U, ShrinkTmaMaps* m) {
    const uint64_t dims[3] = {(uint64_t)p.rows, (uint64_t)p.cols, (uint64_t)p.n};
    const uint64_t strides[2] = {(uint64_t)p.rows * sizeof(float), (uint64_t)p.ld * sizeof(float)};
    const uint32_t box[3] = {(uint32_t)p.R, 3u, (uint32_t)p.nf};
    if (make_tensor_map_f32(&m->D, D, 3, dims, strides, box) != 0) return -1;
    if (make_tensor_map_f32(&m->S, S, 3, dims, strides, box) != 0) return -1;
    if (make_tensor_map_f32(&m->Y, Y, 3, dims, strides, box) != 0) return -1;
    m->has_U = false;
    if (U != nullptr) { if (make_tensor_map_f32(&m->U, U, 3, dims, strides, box) != 0) return -1; m->has_U = true; }
    else m->U = m->S;
    m->has_Q = false; m->Q = m->S;
    return 0;
}

int launch_shrink_tma(const ShrinkTmaPlan& p, const ShrinkTmaMaps& maps, ShrinkBuffers b, const DevState* st, int mode,
                      int min_rank, cudaStream_t stream) {
    if (mode == SHRINK_SPILL && !maps.has_U) { set_error("shrink_tma: spill buffer map missing"); return -1; }
    ShrinkTmaArgs a;
    a.T = b.T; a.tpart = b.tpart; a.Vr = b.Vr; a.VC = b.VC; a.vstride = b.vstride; a.ld = p.ld; a.n = p.n; a.rows = p.rows;
    a.cols = p.cols; a.R = p.R; a.P = p.P; a.NQ = p.P / 4; a.NFL = ST_NT / a.NQ; a.Cf = p.Cf; a.nf = p.nf; a.KR = p.KR;
    a.BS = p.bufstride;
    a.ntile_r = p.ntile_r; a.ntiles = p.ntiles; a.nclusters = p.grid_clusters; a.st = st; a.part_zz = b.part_zz;
    a.part_nnz = b.part_nnz; a.part_max = b.part_max; a.mode = mode; a.min_rank = min_rank;
    static unsigned long long attr_devs = 0;      // one bit per device: the attribute is per (function, device)
    if (first_call_on_device(&attr_devs)) {
        BSUB_CUDA_CHECK(cudaFuncSetAttribute(shrink_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ST_SMEM_CAP));
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(p.grid_clusters * p.Cf); cfg.blockDim = dim3(ST_NT);
    cfg.dynamicSmemBytes = p.smem_bytes; cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = p.Cf; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    const CUtensorMap& outmap = (mode == SHRINK_SPILL) ? maps.U : maps.S;
    BSUB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, shrink_tma_kernel, maps.D, maps.S, maps.Y, outmap, a));
    return 0;
}

}  // namespace bsub
