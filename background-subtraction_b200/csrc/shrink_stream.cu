// shrink_stream.cu -- pass B of the ALM iteration as a warp-specialised, TMA-ring streamed kernel (fast path for
// rank <= 16 and image heights that are a multiple of 4).
//
//   T = Vr^T W ; L = VC T ; G_S = D - L + Y/mu ; S = prox(G_S) ; Z = D - L - S ; Y += mu Z ; sum Z^2
//   (/root/reference/inexact_alm_lsd.py:131-167; prox_flat :71-79 as the closed-form l_inf tile prox)
//
// A persistent CTA (one per SM) owns tiles of 3 image columns x R rows x ALL n frames and streams each tile twice
// through a ring of shared-memory stages (FC frames per stage) filled by 3-D TMA box loads:
//   phase A  D,S,Y  -> W on the fly -> T accumulated in registers over all frames (one reduction per tile)
//   phase B  D,Y    -> per 3x3 group and frame: L from T, G_S, prox, dual update, results written in place and sent
//                      out with TMA box stores (S and Y).  The second read of D,Y partly hits L2 (a tile's D,Y are
//                      n*P*8 bytes; 148 tiles in flight ~ 51 MB of the 126 MB L2; measured hit rate ~60 %).
//                      With the int8 Gram on, W of the NEXT iteration is quantised here too and leaves as four digit
//                      planes (gram_i8.cu): the Gram pass then reads 4 B per element instead of D,S,Y.
// Every stage also carries the Vr (phase A) / VC (phase B) rows of its frames, so shared memory does not grow with n.
// Iteration 1 can run from D alone (S0 = 0, Y0 = D / dual_norm formed on the fly: `implied_first`).
// Roles: warp 0 lane 0 = loader (TMA loads), warp 1 lane 0 = storer (TMA stores, stage recycling), the remaining
// warps compute.  All hand-offs are mbarriers (full / done / free per stage); the only CTA-wide barriers are the two
// named barriers of the per-tile T reduction.  No thread-block clusters, no cross-CTA exchange.
// HBM traffic: read D,S,Y + write S,Y = 20 B per matrix element, + 4 B for the digit planes (+ the part of the 8 B
// phase-B re-read that misses L2).
#include <algorithm>
#include "common.cuh"
#include "kernels.h"
#include "tma.cuh"
#include "prox9.cuh"

namespace bsub {

constexpr int SS_KC = 16;                 // largest rank handled by this kernel (a plan may cap it at 8 to fit Vr, VC of long clips)
constexpr int SS_KRED = 8;                // singular vectors per round of the per-tile T reduction
constexpr size_t SS_SMEM_CAP = 227 * 1024 - 256;
constexpr int SS_NCW = 8;                 // consumer warps (block = 32 * (SS_NCW + 2))

struct ShrinkStreamArgs {
    float* T; const float* Vr; const float* VC; int vstride;
    long long ld;
    int n, rows, cols, R, P, NQ, NFL, FC, NS, BS, nchunkf;
    int ntile_r; long long ntiles;
    const DevState* st;
    double* part_zz; unsigned long long* part_nnz; float* part_max;
    float* part_wmax;                      // [grid] max |W_next| (negative: this kernel did not run -> no slices)
    int mode;
    int wq;                                // write the int8 slices of W_next (gram_i8.cu)
    int QS;                                // bytes per slice sub-buffer of a stage (FC*Pq rounded up to 128)
    int Pq;                                // = P (a multiple of 16 when the slices are on): bytes per frame of a tile
    int kcap;                              // ranks <= kcap (= SS_KC) are handled here; larger ones by the fallback kernel
    int implied_first;                     // iteration 1 takes S = 0, Y = D / dual_norm from D instead of reading them (no init pass)
    const float* Tt;                       // [ntiles][SS_KC][4R]: T of every tile from project.cu (nullptr: always project here)
    int have_flat;                         // shrink_flat.cu runs too: leave it the iterations it takes
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// phase A, one stage: T partial of this thread's pixel quad over its frames of the stage
template <int KCNT>
__device__ __forceinline__ void ss_accumulate(float (&acc)[SS_KC][4], const float* bD, const float* bS, const float* bY,
                                              const float* Vst, int P, int qd, int fl, int NFL, int FC, int fbase, int n,
                                              float inv_mu, bool first, double inv_dual) {
    for (int f = fl; f < FC; f += NFL) {
        const int fg = fbase + f;
        if (fg >= n) break;
        const float4 d4 = *reinterpret_cast<const float4*>(bD + (size_t)f * P + 4 * qd);
        float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f), y4;
        if (first) {                                      // S0 = 0, Y0 = D / dual_norm (inexact_alm_lsd.py:108-120), as init_Y_kernel forms it
            y4.x = (float)((double)d4.x * inv_dual); y4.y = (float)((double)d4.y * inv_dual);
            y4.z = (float)((double)d4.z * inv_dual); y4.w = (float)((double)d4.w * inv_dual);
        } else {
            s4 = *reinterpret_cast<const float4*>(bS + (size_t)f * P + 4 * qd);
            y4 = *reinterpret_cast<const float4*>(bY + (size_t)f * P + 4 * qd);
        }
        float4 w;
        w.x = (d4.x - s4.x) + y4.x * inv_mu; w.y = (d4.y - s4.y) + y4.y * inv_mu;
        w.z = (d4.z - s4.z) + y4.z * inv_mu; w.w = (d4.w - s4.w) + y4.w * inv_mu;
        const float* vrow = Vst + f * SS_KC;               // Vr rows of this stage's frames (TMA-loaded with the stage)
        float vv[SS_KC];
#pragma unroll
        for (int k4 = 0; k4 < (KCNT + 3) / 4; ++k4) {
            const float4 v = *reinterpret_cast<const float4*>(vrow + 4 * k4);
            vv[4 * k4] = v.x; vv[4 * k4 + 1] = v.y; vv[4 * k4 + 2] = v.z; vv[4 * k4 + 3] = v.w;
        }
#pragma unroll
        for (int k = 0; k < KCNT; ++k) {
            acc[k][0] = fmaf(vv[k], w.x, acc[k][0]); acc[k][1] = fmaf(vv[k], w.y, acc[k][1]);
            acc[k][2] = fmaf(vv[k], w.z, acc[k][2]); acc[k][3] = fmaf(vv[k], w.w, acc[k][3]);
        }
    }
}

// phase B, one 3x3 group of one frame: L from T, prox, dual update, in place in the stage
// W of the next iteration, exactly as the next pass will form it from the stored S and Y, as 32-bit fixed point
// q = rint(W * Q) split into four balanced base-256 digits (one byte plane each).  Stage layout per plane:
// [k16 block of the tile][frame][16 B]  (k-block-major, see gram_i8.cu).  Pixel order inside a tile (the Gram is a sum over
// pixels and does not care, project.cu and shrink_flat.cu use the same): position = e * NG + g for entry e = 3 c + dr of the
// 3x3 group g -- the 16 groups of a 48-row tile fill one k16 block per entry.
__device__ __forceinline__ void ss_emit_q(unsigned char* qb, int QS, int pix, int kstep, float d, float s_new, float y_new,
                                          float inv_mu_next, float Qf, float& wmax_acc) {
    const float wn = fmaf(y_new, inv_mu_next, d - s_new);
    wmax_acc = fmaxf(wmax_acc, fabsf(wn));
    // cvt saturates; a clipped value is detected afterwards through wmax (the slices are then discarded)
    const int q = __float2int_rn(wn * Qf);
    // balanced base-256 digits in one go: byte k of ((q + 0x808080) ^ 0x808080) is d_k as a signed byte
    const unsigned int u = ((unsigned int)q + 0x00808080u) ^ 0x00808080u;
    const int po = (pix >> 4) * kstep + (pix & 15);
    qb[po] = (unsigned char)u; qb[QS + po] = (unsigned char)(u >> 8); qb[2 * QS + po] = (unsigned char)(u >> 16);
    qb[3 * QS + po] = (unsigned char)(u >> 24);
}

// Tg: this group's T entries, regrouped as [k][group][12] (9 used) so that they come in as three 16-byte loads per k
template <int KCNT>
__device__ __forceinline__ void ss_group(float* dsp, float* ysp, const float* Tg, int tk_stride, const float* vc, int R, int P, float inv_mu,
                                         float mu_f, float lamq, int mode, double& zz_acc, unsigned int& nnz_acc, float& max_acc,
                                         unsigned char* qb, int QS, int o0, int qng, int kstep, float inv_mu_next, float Qf, float& wmax_acc,
                                         int& sat_acc, bool first, double inv_dual) {
    float vv[SS_KC];
#pragma unroll
    for (int k4 = 0; k4 < (KCNT + 3) / 4; ++k4) {
        const float4 v = *reinterpret_cast<const float4*>(vc + 4 * k4);
        vv[4 * k4] = v.x; vv[4 * k4 + 1] = v.y; vv[4 * k4 + 2] = v.z; vv[4 * k4 + 3] = v.w;
    }
    float av[9], yv[9], x[9], ax[9], dv[9];
    float lw[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) lw[e] = 0.f;
#pragma unroll
    for (int k = 0; k < KCNT; ++k) {
        const float4* tq = reinterpret_cast<const float4*>(Tg + (size_t)k * tk_stride);
        const float4 t0 = tq[0], t1 = tq[1], t2 = tq[2];
        lw[0] = fmaf(vv[k], t0.x, lw[0]); lw[1] = fmaf(vv[k], t0.y, lw[1]); lw[2] = fmaf(vv[k], t0.z, lw[2]);
        lw[3] = fmaf(vv[k], t0.w, lw[3]); lw[4] = fmaf(vv[k], t1.x, lw[4]); lw[5] = fmaf(vv[k], t1.y, lw[5]);
        lw[6] = fmaf(vv[k], t1.z, lw[6]); lw[7] = fmaf(vv[k], t1.w, lw[7]); lw[8] = fmaf(vv[k], t2.x, lw[8]);
    }
    float sabs = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int dr = 0; dr < 3; ++dr) {
            const int e = c * 3 + dr, o = c * R + dr;
            const float l = lw[e];
            dv[e] = dsp[o];
            av[e] = dv[e] - l;                            // a = D - L
            yv[e] = first ? (float)((double)dv[e] * inv_dual) : ysp[o];
            x[e] = fmaf(yv[e], inv_mu, av[e]);            // G_S
            ax[e] = fabsf(x[e]);
            sabs += ax[e];
        }
    float zl = 0.f;
    if (mode == SHRINK_FLAT3) {
        if (!(sabs > lamq)) {                             // whole tile inside the l1 ball: S = 0, Z = D - L
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int dr = 0; dr < 3; ++dr) {
                    const int e = c * 3 + dr, o = c * R + dr;
                    const float yn = fmaf(mu_f, av[e], yv[e]);
                    dsp[o] = 0.f;
                    ysp[o] = yn;
                    zl = fmaf(av[e], av[e], zl);
                    if (qb != nullptr) ss_emit_q(qb, QS, e * qng + o0, kstep, dv[e], 0.f, yn, inv_mu_next, Qf, wmax_acc);
                }
        } else {
            const float theta = ss_clip_level9(ax, lamq);
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int dr = 0; dr < 3; ++dr) {
                    const int e = c * 3 + dr, o = c * R + dr;
                    const float sv = copysignf(fminf(ax[e], theta), x[e]);
                    const float z = av[e] - sv;            // Z = D - L - S
                    const float yn = fmaf(mu_f, z, yv[e]);  // Y += mu Z
                    dsp[o] = sv;
                    ysp[o] = yn;
                    zl = fmaf(z, z, zl);
                    nnz_acc += (sv != 0.f);
                    max_acc = fmaxf(max_acc, fabsf(sv));
                    if (qb != nullptr) ss_emit_q(qb, QS, e * qng + o0, kstep, dv[e], sv, yn, inv_mu_next, Qf, wmax_acc);
                }
        }
        zz_acc += (double)zl;
    } else if (mode == SHRINK_L1) {
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int dr = 0; dr < 3; ++dr) {
                const int e = c * 3 + dr, o = c * R + dr;
                const float sv = copysignf(fmaxf(ax[e] - lamq, 0.f), x[e]);
                const float z = av[e] - sv;
                const float yn = fmaf(mu_f, z, yv[e]);
                dsp[o] = sv;
                ysp[o] = yn;
                zl = fmaf(z, z, zl);
                nnz_acc += (sv != 0.f);
                max_acc = fmaxf(max_acc, fabsf(sv));
                if (qb != nullptr) ss_emit_q(qb, QS, e * qng + o0, kstep, dv[e], sv, yn, inv_mu_next, Qf, wmax_acc);
            }
        zz_acc += (double)zl;
    } else {                                              // SHRINK_SPILL: hand G_S to a separate prox
#pragma unroll
        for (int e = 0; e < 9; ++e) dsp[(e / 3) * R + (e % 3)] = x[e];
    }
}

#define SS_DISPATCH_K(kcnt, CALL)                         \
    switch (kcnt) {                                       \
        case 0: { constexpr int K_ = 0; CALL; } break;    \
        case 1: { constexpr int K_ = 1; CALL; } break;    \
        case 2: { constexpr int K_ = 2; CALL; } break;    \
        case 3: { constexpr int K_ = 3; CALL; } break;    \
        case 4: { constexpr int K_ = 4; CALL; } break;    \
        case 5: { constexpr int K_ = 5; CALL; } break;    \
        case 6: { constexpr int K_ = 6; CALL; } break;    \
        case 7: { constexpr int K_ = 7; CALL; } break;    \
        case 8: { constexpr int K_ = 8; CALL; } break;    \
        case 9: case 10: { constexpr int K_ = 10; CALL; } break;  \
        case 11: case 12: { constexpr int K_ = 12; CALL; } break; \
        default: { constexpr int K_ = 16; CALL; } break;  \
    }

// phase B of one tile: every stage = FC frames; thread item = one 3x3 group of one frame
template <int KCNT, int NTC>
__device__ __forceinline__ void ss_phase_b(const ShrinkStreamArgs& a, float* ring, size_t stage_floats, const float* Tp, const float* Vst_all,
                                           uint64_t* full, uint64_t* done, long long& q, int ct, int lane, int NG, int R, int P, int FC,
                                           int BS, int QS, int VSS, int NS, int ncf, bool wq, float inv_mu, float mu_f, float lamq, float inv_mu_next, float Qf,
                                           double& zz_acc, unsigned int& nnz_acc, float& max_acc, float& wmax_acc, int& sat_acc, bool first,
                                           double inv_dual) {
    for (int c = 0; c < ncf; ++c, ++q) {
        const int s = (int)(q % NS);
        const long long u = q / NS;
        mbar_wait(&full[s], (uint32_t)(u & 1));
        float* b = ring + (size_t)s * stage_floats;
        const int fbase = c * FC;
        for (int itx = ct; itx < FC * NG; itx += NTC) {
            const int f = itx / NG, g = itx - f * NG;
            const int fg = fbase + f;
            if (fg >= a.n) continue;
            float* dsp = b + (size_t)f * P + 3 * g;
            float* ysp = b + (size_t)2 * BS + (size_t)f * P + 3 * g;
            unsigned char* qb = wq ? (reinterpret_cast<unsigned char*>(b + (size_t)BS) + (size_t)f * 16) : nullptr;
            ss_group<KCNT>(dsp, ysp, Tp + 12 * g, 12 * NG, Vst_all + (size_t)s * VSS + f * SS_KC, R, P, inv_mu, mu_f, lamq, a.mode, zz_acc, nnz_acc,
                           max_acc, qb, QS, g, NG, FC * 16, inv_mu_next, Qf, wmax_acc, sat_acc, first, inv_dual);
        }
        fence_proxy_async_smem();                   // my writes -> visible to the storer's TMA stores
        __syncwarp();
        if (lane == 0) mbar_arrive(&done[s]);
    }
}

// RT / FCT: tile rows and frames per stage as compile-time constants (0 = take them from the arguments): with the default
// plan (48 rows, 28 frames) every index computation of the inner loops folds into immediates and shifts.
template <int RT, int FCT>
__global__ void __launch_bounds__(32 * (SS_NCW + 2), 1)
shrink_stream_kernel(const __grid_constant__ CUtensorMap mapD, const __grid_constant__ CUtensorMap mapS,
                     const __grid_constant__ CUtensorMap mapY, const __grid_constant__ CUtensorMap mapOut,
                     const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapVr,
                     const __grid_constant__ CUtensorMap mapVC, ShrinkStreamArgs a) {
    constexpr int NTC = 32 * SS_NCW;
    const DevState* st = a.st;
    if (st->done) return;
    const int r = st->svp;
    if (a.have_flat && shrink_flat_takes(st)) {            // the single-pass kernel (shrink_flat.cu) does this iteration
        if (threadIdx.x == 0) { a.part_zz[blockIdx.x] = 0.0; a.part_nnz[blockIdx.x] = 0ull; a.part_max[blockIdx.x] = 0.f; if (a.part_wmax != nullptr) a.part_wmax[blockIdx.x] = 0.f; }
        return;
    }
    if (r > a.kcap) {                                      // large ranks take the fallback kernel launched next
        if (threadIdx.x == 0) { a.part_zz[blockIdx.x] = 0.0; a.part_nnz[blockIdx.x] = 0ull; a.part_max[blockIdx.x] = 0.f; if (a.part_wmax != nullptr) a.part_wmax[blockIdx.x] = -1.f; }
        return;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int R = RT ? RT : a.R, P = 3 * R, NQ = P / 4, NFL = (32 * SS_NCW) / NQ, FC = FCT ? FCT : a.FC, NS = a.NS;
    const int BS = (RT && FCT) ? ((FCT * 3 * RT + 127) / 128 * 128) : a.BS, QS = (RT && FCT) ? ((FCT * 3 * RT + 127) / 128 * 128) : a.QS;
    const double mu_d = st->mu;
    const float inv_mu = (float)(1.0 / mu_d), mu_f = (float)mu_d;
    const bool first = (a.implied_first != 0) && (st->iter == 1);
    const double inv_dual = 1.0 / st->dual_norm;
    const float lamq = (float)(st->lambda / mu_d);
    const bool wq = (a.wq != 0) && (a.mode != SHRINK_SPILL);
    // the next pass uses mu_next = min(mu rho, mu 1e7) (control_post_kernel): same double arithmetic here
    const float inv_mu_next = (float)(1.0 / fmin(mu_d * st->rho, mu_d * 1e7));
    const float Qf = wq ? (float)(2147483648.0 / st->wq_scale_next) : 0.f;
    float wmax_acc = 0.f;
    int sat_acc = 0;

    extern __shared__ __align__(128) unsigned char ss_smem_raw[];
    const size_t stage_floats = (size_t)3 * BS;
    float* ring = reinterpret_cast<float*>(ss_smem_raw);            // [NS][3][BS]
    float* scr = ring + (size_t)NS * stage_floats;                  // [NFL][SS_KRED][P]   (T reduction)
    float* Tp = scr + (size_t)NFL * SS_KRED * P;                    // [SS_KC][R/3 groups][12]: T of the tile, 9 entries per 3x3 group
    // Vr (phase A) / VC (phase B) rows of the frames of a stage, loaded by TMA together with the stage: the footprint does
    // not grow with the number of frames
    const int VSS = (FC * SS_KC + 31) / 32 * 32;                   // floats per stage slice (128-byte multiple: TMA destination)
    float* Vst = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(Tp + (size_t)SS_KC * (4 * R)) + 127) & ~(uintptr_t)127);   // [NS][VSS]
    uint64_t* full = reinterpret_cast<uint64_t*>(Vst + (size_t)NS * VSS);   // [NS]
    uint64_t* done = full + NS;                                     // [NS]
    uint64_t* freeb = done + NS;                                    // [NS]
    __shared__ double redd[32];

    if (threadIdx.x == 0) {
        for (int s = 0; s < NS; ++s) { mbar_init(&full[s], 1); mbar_init(&done[s], SS_NCW); mbar_init(&freeb[s], 1); }
        mbar_fence_init();
        tma_prefetch_desc(&mapD); tma_prefetch_desc(&mapS); tma_prefetch_desc(&mapY); tma_prefetch_desc(&mapOut);
        tma_prefetch_desc(&mapVr); tma_prefetch_desc(&mapVC);
    }
    for (int idx = threadIdx.x; idx < SS_KC * 4 * R; idx += blockDim.x) { Tp[idx] = 0.f; if (NFL * SS_KRED * P >= SS_KC * 4 * R) scr[idx] = 0.f; }   // rows >= svp stay zero (scr: second T buffer)
    __syncthreads();

    auto tile_origin = [&](long long tl, int& j0, int& i0) {
        const int tcx = (int)(tl / a.ntile_r), trx = (int)(tl - (long long)tcx * a.ntile_r);
        j0 = 3 * tcx; i0 = trx * R;
    };
    const int ncf = a.nchunkf;                              // frame chunks per tile
    // T already projected from the digit planes of this W (project.cu ran just before): one pass per tile
    const bool scr_ok = NFL * SS_KRED * P >= SS_KC * 4 * R;    // the reduction scratch doubles as the second T buffer
    const bool proj = (a.Tt != nullptr) && scr_ok && (st->gram_mode == 1) && !first && r > 0;
    const bool phaseA = r > 0 && !proj;                     // rank 0: L = 0, no T needed
    const int chunks_per_tile = (phaseA ? ncf : 0) + ncf;

    double zz_acc = 0.0;
    unsigned int nnz_acc = 0u;
    float max_acc = 0.f;

    if (warp == 0) {
        // ===================== loader =====================
        if (lane == 0) {
            // D and Y of a tile are read again in phase B: keep them in L2; everything else is streamed once
            const uint64_t pol_keep = l2_policy_evict_last(), pol_stream = l2_policy_evict_first();
            long long q = 0;
            for (long long tl = blockIdx.x; tl < a.ntiles; tl += gridDim.x) {
                int j0, i0;
                tile_origin(tl, j0, i0);
                for (int c = 0; c < chunks_per_tile; ++c, ++q) {
                    const int s = (int)(q % NS);
                    const long long u = q / NS;
                    if (u > 0) mbar_wait(&freeb[s], (uint32_t)((u - 1) & 1));
                    float* b = ring + (size_t)s * stage_floats;
                    const bool isA = phaseA && c < ncf;
                    const int fbase = (isA ? c : c - (phaseA ? ncf : 0)) * FC;
                    mbar_expect_tx(&full[s], (uint32_t)((first ? 1 : (isA ? 3 : 2)) * (size_t)FC * P * sizeof(float)) +
                                             (uint32_t)(FC * SS_KC * sizeof(float)));
                    tma_load_2d(Vst + (size_t)s * VSS, isA ? &mapVr : &mapVC, &full[s], 0, fbase);
                    const uint64_t pol = (isA && phaseA) ? pol_keep : pol_stream;
                    tma_load_3d_hint(b, &mapD, &full[s], i0, j0, fbase, pol);
                    if (!first) {
                        tma_load_3d_hint(b + (size_t)2 * a.BS, &mapY, &full[s], i0, j0, fbase, pol);
                        if (isA) tma_load_3d_hint(b + (size_t)a.BS, &mapS, &full[s], i0, j0, fbase, pol_stream);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== storer: TMA stores of finished phase-B stages, stage recycling =====================
        if (lane == 0) {
            const uint64_t pol_stream = l2_policy_evict_first();
            long long q = 0;
            for (long long tl = blockIdx.x; tl < a.ntiles; tl += gridDim.x) {
                int j0, i0;
                tile_origin(tl, j0, i0);
                for (int c = 0; c < chunks_per_tile; ++c, ++q) {
                    const int s = (int)(q % NS);
                    const long long u = q / NS;
                    mbar_wait(&done[s], (uint32_t)(u & 1));
                    const bool isA = phaseA && c < ncf;
                    if (!isA) {
                        float* b = ring + (size_t)s * stage_floats;
                        const int fbase = (c - (phaseA ? ncf : 0)) * FC;
                        tma_store_3d_hint(&mapOut, b, i0, j0, fbase, pol_stream);                  // S_new (or G_S)
                        if (a.mode != SHRINK_SPILL) tma_store_3d_hint(&mapY, b + (size_t)2 * a.BS, i0, j0, fbase, pol_stream);
                        if (wq) {                      // four byte planes of W_next, pixel order = tile-major (gram_i8.cu does not care)
                            const unsigned char* qbase = reinterpret_cast<const unsigned char*>(b + (size_t)a.BS);
                            for (int sl = 0; sl < 4; ++sl) tma_store_3d(&mapQ, qbase + (size_t)sl * a.QS, 2 * fbase, (int)(tl * (P / 16)), sl);
                        }
                        tma_store_commit();
                        tma_store_wait_read<0>();                                                  // stage may be overwritten
                    }
                    mbar_arrive(&freeb[s]);
                }
            }
            tma_store_wait_all<0>();
        }
        __syncwarp();
    } else {
        // ===================== consumers =====================
        const int ct = threadIdx.x - 64;                    // consumer thread id 0..NTC-1
        const int qd = ct % NQ, fl = ct / NQ;
        const bool tact = fl < NFL;
        const int NG = R / 3, RQ = R / 4;
        long long q = 0;
        // projected T of a tile: r rows of 4R floats, fetched with cp.async into one of two buffers (Tp, and the reduction
        // scratch, which is idle in this mode) one tile ahead
        const int tpieces = r * R;                          // 16-byte pieces (r rows x 4R floats)
        auto fetch_T = [&](long long tile, float* dst) {
            const float* src = a.Tt + (size_t)tile * SS_KC * (4 * R);
            for (int pc = ct; pc < tpieces; pc += NTC) cp_async16(dst + 4 * pc, src + 4 * pc);
        };
        int tpar = 0;
        if (proj && (long long)blockIdx.x < a.ntiles) { fetch_T(blockIdx.x, Tp); cp_async_wait_all(); named_bar_sync(1, NTC); }
        for (long long tl = blockIdx.x; tl < a.ntiles; tl += gridDim.x) {
            int j0, i0;
            tile_origin(tl, j0, i0);
            const float* Tcur = (proj && tpar) ? scr : Tp;
            if (proj && tl + gridDim.x < a.ntiles) fetch_T(tl + gridDim.x, tpar ? Tp : scr);
            if (phaseA) {
                float acc[SS_KC][4];
#pragma unroll
                for (int k = 0; k < SS_KC; ++k) { acc[k][0] = acc[k][1] = acc[k][2] = acc[k][3] = 0.f; }
                for (int c = 0; c < ncf; ++c, ++q) {
                    const int s = (int)(q % NS);
                    const long long u = q / NS;
                    mbar_wait(&full[s], (uint32_t)(u & 1));
                    const float* b = ring + (size_t)s * stage_floats;
                    if (tact) { SS_DISPATCH_K(r, (ss_accumulate<K_>(acc, b, b + BS, b + 2 * BS, Vst + (size_t)s * VSS, P, qd, fl, NFL, FC, c * FC, a.n, inv_mu, first, inv_dual))); }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&done[s]);
                }
                // one reduction per tile over the NFL frame lanes (SS_KRED vectors per round)
                for (int kr0 = 0; kr0 < r; kr0 += SS_KRED) {
                    if (tact) {
#pragma unroll
                        for (int k = 0; k < SS_KC; ++k)
                            if (k >= kr0 && k < kr0 + SS_KRED && k < r)
                                *reinterpret_cast<float4*>(scr + ((size_t)(fl * SS_KRED + (k - kr0))) * P + 4 * qd) =
                                    make_float4(acc[k][0], acc[k][1], acc[k][2], acc[k][3]);
                    }
                    named_bar_sync(1, NTC);
                    const int kend = min(SS_KRED, r - kr0);
                    for (int idx = ct; idx < kend * NQ; idx += NTC) {
                        const int k = idx / NQ, qq = idx - k * NQ;
                        float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
                        for (int l = 0; l < NFL; ++l) {
                            const float4 v = *reinterpret_cast<const float4*>(scr + ((size_t)(l * SS_KRED + k)) * P + 4 * qq);
                            sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
                        }
                        // keep T for the final materialisation of L (rows % 4 == 0 on this path)
                        const int c2 = qq / RQ, i2 = (qq - c2 * RQ) * 4;
                        {   // regrouped copy for phase B: entry e = 3 c + dr of group g = row / 3
                            float* tk = Tp + (size_t)(kr0 + k) * (4 * R);
                            const float sv4[4] = {sum.x, sum.y, sum.z, sum.w};
#pragma unroll
                            for (int t = 0; t < 4; ++t) { const int ir = i2 + t; tk[(ir / 3) * 12 + c2 * 3 + (ir % 3)] = sv4[t]; }
                        }
                        const int j2 = j0 + c2, row2 = i0 + i2;
                        if (j2 < a.cols && row2 < a.rows) stg4(a.T + (size_t)(kr0 + k) * a.ld + (long long)j2 * a.rows + row2, sum);
                    }
                    named_bar_sync(1, NTC);
                }
            }
            // phase B
            SS_DISPATCH_K(r, (ss_phase_b<K_, NTC>(a, ring, stage_floats, Tcur, Vst, full, done, q, ct, lane, NG, R, P, FC, BS, QS, VSS, NS, ncf, wq, inv_mu,
                                                  mu_f, lamq, inv_mu_next, Qf, zz_acc, nnz_acc, max_acc, wmax_acc, sat_acc, first, inv_dual)));
            if (proj) { cp_async_wait_all(); named_bar_sync(1, NTC); tpar ^= 1; }     // next tile's T has landed, this tile's buffer is free
        }
    }
    __syncthreads();
    double zt = block_sum(zz_acc, redd);
    if (threadIdx.x == 0) a.part_zz[blockIdx.x] = zt;
    double nt = block_sum((double)nnz_acc, redd);
    if (threadIdx.x == 0) a.part_nnz[blockIdx.x] = (unsigned long long)(nt + 0.5);
    double mt = block_max((double)max_acc, redd);
    if (threadIdx.x == 0) a.part_max[blockIdx.x] = (float)mt;
    // max |W_next| (+ a large sentinel if a slice was clipped) for the fixed-point scale of the following pass
    if (wq && !(wmax_acc * Qf < 2130706432.f)) sat_acc = 1;              // |q| must stay <= 2^31 - 2^24
    double wt = block_max((double)(sat_acc ? 3.0e38f : wmax_acc), redd);
    if (threadIdx.x == 0 && a.part_wmax != nullptr) a.part_wmax[blockIdx.x] = wq ? (float)wt : -1.f;
}

// -------------------------------------------------------------------------------------------------------------
static size_t ss_smem_bytes(int n, int R, int FC, int NS) {
    (void)n;
    const int P = 3 * R, NQ = P / 4, NFL = 32 * SS_NCW / NQ;
    const size_t bs = ((size_t)FC * P + 127) / 128 * 128;
    size_t fl = (size_t)NS * 3 * bs + (size_t)NFL * SS_KRED * P + (size_t)SS_KC * 4 * R + (size_t)NS * ((FC * SS_KC + 31) / 32 * 32) + 32;
    return fl * sizeof(float) + (size_t)3 * NS * sizeof(uint64_t) + 64;
}

bool make_shrink_stream_plan(int n, int rows, int cols, long long ld, int num_sms, int R_hint, ShrinkStreamPlan* out) {
    if (rows % 4 != 0 || rows < 12) return false;
    ShrinkStreamPlan p;
    p.n = n; p.rows = rows; p.cols = cols; p.ld = ld;
    const int NTC = 32 * SS_NCW;
    int R = R_hint > 0 ? ((R_hint + 11) / 12) * 12 : 48;
    const int rows12 = ((rows + 11) / 12) * 12;
    R = std::min(std::min(R, rows12), 252);
    for (; R >= 12; R -= 12) {
        const int NQ = 3 * R / 4;
        if (NQ > NTC) continue;
        const int NFL = NTC / NQ;
        const int FC = std::max(1, std::min(4 * NFL, std::min(n, 256)));
        int NS = 6;
        while (NS >= 3 && ss_smem_bytes(n, R, FC, NS) > SS_SMEM_CAP) --NS;
        if (NS < 3) continue;
        p.R = R; p.P = 3 * R; p.FC = FC; p.NS = NS; p.kcap = SS_KC;
        p.bufstride = (int)(((size_t)FC * p.P + 127) / 128 * 128);
        p.smem_bytes = ss_smem_bytes(n, R, FC, NS);
        p.nchunkf = (n + FC - 1) / FC;
        p.ntile_r = (rows + R - 1) / R;
        p.ntile_c = (cols + 2) / 3;
        p.ntiles = (long long)p.ntile_r * p.ntile_c;
        p.grid = (int)std::min<long long>(num_sms, p.ntiles);
        p.nparts = p.grid;
        *out = p;
        return true;
    }
    return false;
}

int make_shrink_stream_maps(const ShrinkStreamPlan& p, const float* D, float* S, float* Y, float* U, ShrinkTmaMaps* m) {
    const uint64_t dims[3] = {(uint64_t)p.rows, (uint64_t)p.cols, (uint64_t)p.n};
    const uint64_t strides[2] = {(uint64_t)p.rows * sizeof(float), (uint64_t)p.ld * sizeof(float)};
    const uint32_t box[3] = {(uint32_t)p.R, 3u, (uint32_t)p.FC};
    if (make_tensor_map_f32(&m->D, D, 3, dims, strides, box) != 0) return -1;
    if (make_tensor_map_f32(&m->S, S, 3, dims, strides, box) != 0) return -1;
    if (make_tensor_map_f32(&m->Y, Y, 3, dims, strides, box) != 0) return -1;
    m->has_U = false;
    if (U != nullptr) { if (make_tensor_map_f32(&m->U, U, 3, dims, strides, box) != 0) return -1; m->has_U = true; }
    else m->U = m->S;
    m->has_Q = false; m->Q = m->S;
    return 0;
}

int make_shrink_stream_vmaps(const ShrinkStreamPlan& p, const float* Vr, const float* VC, int vstride, ShrinkTmaMaps* m) {
    // Vr / VC: float32 [n frames][vstride]; a stage takes the first SS_KC columns of its FC frames (frames beyond n: zero)
    if (vstride < SS_KC) { set_error("shrink_stream: Vr row stride %d < %d", vstride, SS_KC); return -1; }
    const uint64_t dims[2] = {(uint64_t)vstride, (uint64_t)p.n};
    const uint64_t strides[1] = {(uint64_t)vstride * sizeof(float)};
    const uint32_t box[2] = {(uint32_t)SS_KC, (uint32_t)p.FC};
    if (make_tensor_map_f32(&m->Vr, Vr, 2, dims, strides, box) != 0) return -1;
    if (make_tensor_map_f32(&m->VC, VC, 2, dims, strides, box) != 0) return -1;
    return 0;
}

// slice matrix Wq: int8 [4][n][ldq], pixel order tile-major (tile tl of the shrink pass owns bytes [tl*P, tl*P + P) of every row)
// pixels per frame in the slice matrix (tile-major pixel order); 0 when the tile width does not split into 16-byte k-blocks
long long shrink_stream_ldq(const ShrinkStreamPlan& p) { return (p.P % 16 == 0) ? ((p.ntiles * (long long)p.P) + 63) / 64 * 64 : 0; }

int make_shrink_stream_qmap(const ShrinkStreamPlan& p, signed char* Wq, ShrinkTmaMaps* m) {
    const long long ldq = shrink_stream_ldq(p);
    // [slice][k16][frame][16 B]; the frames of a k16 block are contiguous, so the map views them as 2 n eight-byte elements:
    // a tile's chunk of FC frames is one box {2 FC, P/16, 1} per plane whose rows are 16 FC contiguous bytes
    const uint64_t dims[3] = {(uint64_t)2 * p.n, (uint64_t)(ldq / 16), 4};
    const uint64_t strides[2] = {(uint64_t)16 * p.n, (uint64_t)ldq * (uint64_t)p.n};
    const uint32_t box[3] = {(uint32_t)(2 * p.FC), (uint32_t)(p.P / 16), 1};
    if (make_tensor_map_u64(&m->Q, Wq, 3, dims, strides, box) != 0) return -1;
    m->has_Q = true;
    return 0;
}

template <int RT, int FCT>
static int launch_ss(const ShrinkStreamPlan& p, const ShrinkTmaMaps& maps, const ShrinkStreamArgs& a, int mode, cudaStream_t stream) {
    static unsigned long long attr_devs = 0;      // one bit per device: the attribute is per (function, device)
    if (first_call_on_device(&attr_devs)) {
        BSUB_CUDA_CHECK(cudaFuncSetAttribute(shrink_stream_kernel<RT, FCT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SS_SMEM_CAP));
    }
    const CUtensorMap& outmap = (mode == SHRINK_SPILL) ? maps.U : maps.S;
    shrink_stream_kernel<RT, FCT><<<p.grid, 32 * (SS_NCW + 2), p.smem_bytes, stream>>>(maps.D, maps.S, maps.Y, outmap, maps.Q, maps.Vr,
                                                                                      maps.VC, a);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_shrink_stream(const ShrinkStreamPlan& p, const ShrinkTmaMaps& maps, ShrinkBuffers b, const DevState* st, int mode,
                         cudaStream_t stream) {
    if (mode == SHRINK_SPILL && !maps.has_U) { set_error("shrink_stream: spill buffer map missing"); return -1; }
    ShrinkStreamArgs a;
    a.T = b.T; a.Vr = b.Vr; a.VC = b.VC; a.vstride = b.vstride; a.ld = p.ld; a.n = p.n; a.rows = p.rows; a.cols = p.cols;
    a.R = p.R; a.P = p.P; a.NQ = p.P / 4; a.NFL = (32 * SS_NCW) / a.NQ; a.FC = p.FC; a.NS = p.NS; a.BS = p.bufstride;
    a.nchunkf = p.nchunkf; a.ntile_r = p.ntile_r; a.ntiles = p.ntiles; a.st = st; a.part_zz = b.part_zz; a.part_nnz = b.part_nnz;
    a.part_max = b.part_max; a.part_wmax = b.part_wmax; a.mode = mode;
    a.wq = (maps.has_Q && b.part_wmax != nullptr) ? 1 : 0; a.Pq = p.P; a.implied_first = b.implied_first; a.kcap = p.kcap;
    a.Tt = (mode != SHRINK_SPILL) ? b.Tt : nullptr;
    a.have_flat = (mode != SHRINK_SPILL) ? b.have_flat : 0;
    a.QS = (int)(((size_t)p.FC * p.P + 127) / 128 * 128);
    if (p.R == 48 && p.FC == 28) return launch_ss<48, 28>(p, maps, a, mode, stream);
    return launch_ss<0, 0>(p, maps, a, mode, stream);
}

}  // namespace bsub
