// shrink_flat.cu -- the bandwidth pass of an ALM iteration as ONE streaming sweep (rank <= 8, 48-row tiles):
//
//   L = VC T ; G_S = D - L + Y/mu ; S = prox(G_S) ; Z = D - L - S ; Y += mu Z ; sum Z^2 ; W_next -> int8 digit planes
//   (/root/reference/inexact_alm_lsd.py:147-167; prox_flat :71-79 as the closed-form l_inf tile prox, or the l1
//   soft threshold of lsd_improvement.py:176)
//
// T = Vr^T W comes from project.cu (computed from the digit planes of W), so D and Y are read exactly once and S is not
// read at all: HBM traffic per matrix element = 8 B in (D, Y) + 12 B out (S, Y, 4 digit bytes).
//
// Persistent CTA per SM, warp-specialised like shrink_stream.cu (1 TMA loader warp, 1 TMA storer warp, 8 consumer warps,
// full / done / free mbarriers per stage), but organised around the instruction budget of the consumers:
//   * a consumer thread owns ONE 3x3 group of the tile and a frame lane (16 groups x 16 frame lanes = 256 threads); the
//     group's T (rank x 9) stays in registers for the whole tile, so L costs 9 r FMAs per frame and no shared-memory
//     traffic besides the 8 floats of VC;
//   * per frame and group: 18 scalar loads (conflict-free: 16 groups x 3 floats hit 16 distinct banks, the second frame
//     of the warp the other 16), the background test, and -- for the ~95 % of the groups inside the l1 ball -- a short
//     path without the sorting network;
//   * W_next leaves as one 32-bit word per pixel into a warp-private staging area; the warp (which holds two complete
//     frames of the tile) then transposes 4 pixels x 4 digits with byte permutes and writes 32-bit plane words, instead
//     of four one-byte stores per pixel.
// Loop order: a CTA owns a contiguous range of tiles and walks it in groups of 6 vertically adjacent tiles; inside a group the
// FRAME chunk is the outer loop and the tile the inner one, so the 192-byte runs that neighbouring tiles write into the same
// frame and image column reach L2 within a few microseconds of each other and leave for HBM as one long run.  Measured with
// scripts/micro/tma_pattern_bench.cu (same boxes, no compute): 4.27 -> 5.08 TB/s for 2 loads + 3 stores, 4.57 -> 5.19 TB/s
// for 2 + 2.  T of the whole group (6 x r x 768 B) sits in shared memory.
// Rank > 8, the first iteration (no planes of W yet), the spill modes and image heights that are not a multiple of 4
// stay on shrink_stream.cu / shrink_tma.cu / shrink.cu; the choice is made on the device from DevState.
#include <algorithm>
#include "common.cuh"
#include "kernels.h"
#include "tma.cuh"
#include "prox9.cuh"

namespace bsub {

constexpr int SF_R = 48, SF_P = 144, SF_NG = 16, SF_FL = 16, SF_NCW = 8, SF_NTC = 256, SF_KMAX = 8;
constexpr int SF_TFLOATS = SF_KMAX * 4 * SF_R;        // T of one tile: [8][16 groups][12]
constexpr int SF_TG = 6;                              // tiles per group (vertically adjacent): see the loop order below
constexpr size_t SF_SMEM_CAP = 227 * 1024 - 512;

struct ShrinkFlatArgs {
    const float* Tt;                       // [ntiles][16][4R] from project.cu
    int n, rows, cols, FC, NS, nchunkf, ntile_r; long long ntiles;
    const DevState* st;
    int* s_stale_next;                     // &DevState::s_stale_next (set when this launch leaves S in HBM untouched)
    int force_S;                           // always store S (pixel-sharded drivers, restart after a saturated digit pass)
    double* part_zz; unsigned long long* part_nnz; float* part_max; float* part_wmax;
    int mode;
};

__device__ __forceinline__ void sf_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void sf_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void sf_cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void sf_cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

static_assert(SF_KMAX == kFlatMaxRank, "rank cap of the single-pass kernel");

struct SfScal { float inv_mu, mu_f, lamq, c1, Qf; };

// one frame of one 3x3 group.  dsp / ysp: the group's first element in the D (-> S) and Y slots of the stage.
// uw: W_next of the 9 pixels as 32-bit fixed point with balanced base-256 digits (byte d = digit d); ws: S is stored
template <int KR, int MODE>
__device__ __forceinline__ void sf_item(float* dsp, float* ysp, const float (&T)[KR > 0 ? KR : 1][9], const float* vc, const SfScal& sc, const bool ws,
                                        unsigned int (&uw)[9], float& zl_acc, unsigned int& nnz_acc, float& max_acc, float& wmax_acc) {
    float l[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) l[e] = 0.f;
    if (KR > 0) {
        float vv[8];
        const float4 v0 = *reinterpret_cast<const float4*>(vc);
        vv[0] = v0.x; vv[1] = v0.y; vv[2] = v0.z; vv[3] = v0.w;
        if (KR > 4) { const float4 v1 = *reinterpret_cast<const float4*>(vc + 4); vv[4] = v1.x; vv[5] = v1.y; vv[6] = v1.z; vv[7] = v1.w; }
#pragma unroll
        for (int k = 0; k < KR; ++k)
#pragma unroll
            for (int e = 0; e < 9; ++e) l[e] = fmaf(vv[k], T[k][e], l[e]);
    }
    float d[9], y[9], a[9], x[9];
    float sabs = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int dr = 0; dr < 3; ++dr) {
            const int e = 3 * c + dr, o = c * SF_R + dr;
            d[e] = dsp[o]; y[e] = ysp[o];
            a[e] = d[e] - l[e];                               // D - L
            x[e] = fmaf(y[e], sc.inv_mu, a[e]);               // G_S
            sabs += fabsf(x[e]);
        }
    if (MODE == SHRINK_FLAT3 && !(sabs > sc.lamq)) {
        // the whole tile lies inside the l1 ball: S = 0, Z = D - L
        float zl = 0.f;
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int dr = 0; dr < 3; ++dr) {
                const int e = 3 * c + dr, o = c * SF_R + dr;
                const float yn = fmaf(sc.mu_f, a[e], y[e]);
                zl = fmaf(a[e], a[e], zl);
                if (ws) dsp[o] = 0.f;
                ysp[o] = yn;
                const float wq = fmaf(yn, sc.c1, d[e] * sc.Qf);          // W_next * Q, W_next = D - S + Y/mu_next
                wmax_acc = fmaxf(wmax_acc, fabsf(wq));
                uw[e] = ((unsigned int)__float2int_rn(wq) + 0x00808080u) ^ 0x00808080u;
            }
        zl_acc += zl;
        return;
    }
    float theta = 0.f;
    if (MODE == SHRINK_FLAT3) {
        float ax[9];
#pragma unroll
        for (int e = 0; e < 9; ++e) ax[e] = fabsf(x[e]);
        theta = ss_clip_level9(ax, sc.lamq);
    }
    float zl = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int dr = 0; dr < 3; ++dr) {
            const int e = 3 * c + dr, o = c * SF_R + dr;
            const float ax = fabsf(x[e]);
            const float sm = (MODE == SHRINK_FLAT3) ? fminf(ax, theta) : fmaxf(ax - sc.lamq, 0.f);
            const float sv = copysignf(sm, x[e]);
            const float z = a[e] - sv;                         // Z = D - L - S
            const float yn = fmaf(sc.mu_f, z, y[e]);           // Y += mu Z
            zl = fmaf(z, z, zl);
            nnz_acc += (sv != 0.f);
            max_acc = fmaxf(max_acc, sm);
            if (ws) dsp[o] = sv;
            ysp[o] = yn;
            const float wq = fmaf(yn, sc.c1, (d[e] - sv) * sc.Qf);
            wmax_acc = fmaxf(wmax_acc, fabsf(wq));
            uw[e] = ((unsigned int)__float2int_rn(wq) + 0x00808080u) ^ 0x00808080u;
        }
    zl_acc += zl;
}

// consumer side of one group of gt tiles: for every frame chunk, for every tile of the group: one stage of FC frames.
// The 9 words of a (group, frame) go to a warp-private staging area, and the warp transposes 4 pixels x 4 digits with byte
// permutes from there (dense plane boxes [4][9][FC][16 B] in the stage).  Kept over a transpose in registers across lanes
// (1080p x 300, ms per solve: 94.4 staged, 100.5 in registers with 128-byte-swizzled 8-frame boxes, 94.7 in registers with the
// dense boxes; profiles/r2r_shrink_variants.log): the bank conflicts of the staged stores do not bound the kernel.
template <int KR, int MODE>
__device__ __forceinline__ void sf_group(const ShrinkFlatArgs& a, const float* Tg, int gt, unsigned char* ring, size_t stage_bytes, const float* Vst_all,
                                         unsigned int* ustage, uint64_t* full, uint64_t* done, int& q, int lane, int cw, const SfScal& sc, const bool ws,
                                         float& zl_acc, unsigned int& nnz_acc, float& max_acc, float& wmax_acc) {
    const int g = lane & 15, flh = lane >> 4;
    const int FC = a.FC, NS = a.NS;
    unsigned int* ust = ustage + flh * SF_P + g;              // this thread's words of the warp's staging area: [frame half][entry][group]
    const size_t slot = (size_t)FC * SF_P * sizeof(float);
    for (int c = 0; c < a.nchunkf; ++c)
        for (int t = 0; t < gt; ++t, ++q) {
            float T[KR > 0 ? KR : 1][9];                      // the 3x3 group's T of this tile
            if (KR > 0) {
#pragma unroll
                for (int k = 0; k < KR; ++k) {
                    const float4* tq = reinterpret_cast<const float4*>(Tg + (size_t)t * SF_TFLOATS + (size_t)k * (4 * SF_R) + 12 * g);
                    const float4 t0 = tq[0], t1 = tq[1], t2 = tq[2];
                    T[k][0] = t0.x; T[k][1] = t0.y; T[k][2] = t0.z; T[k][3] = t0.w; T[k][4] = t1.x; T[k][5] = t1.y; T[k][6] = t1.z; T[k][7] = t1.w;
                    T[k][8] = t2.x;
                }
            }
            const int s = q % NS;
            mbar_wait(&full[s], (uint32_t)((q / NS) & 1));
            unsigned char* b = ring + (size_t)s * stage_bytes;
            float* bD = reinterpret_cast<float*>(b);
            float* bY = reinterpret_cast<float*>(b + slot);
            unsigned char* bP = b + 2 * slot;                     // [4 planes][9 k16 blocks][FC frames][16 B]
            const float* Vst = Vst_all + (size_t)s * FC * SF_KMAX;
            for (int f0 = 0; f0 < FC; f0 += SF_FL) {
                unsigned int uw[9];
                const int fw = f0 + 2 * cw, f = fw + flh;     // the warp's two frames of this round, and mine
                sf_item<KR, MODE>(bD + (size_t)f * SF_P + 3 * g, bY + (size_t)f * SF_P + 3 * g, T, Vst + f * SF_KMAX, sc, ws, uw, zl_acc, nnz_acc,
                                  max_acc, wmax_acc);
#pragma unroll
                for (int e = 0; e < 9; ++e) ust[e * SF_NG] = uw[e];
                __syncwarp();
                // 2 frames x 36 position quads: 4 pixels x 4 digits -> one 32-bit word per plane
#pragma unroll
                for (int tt = 0; tt < 3; ++tt) {
                    const int qi = lane + 32 * tt;
                    if (qi < 72) {
                        const int fh = qi / 36, pq = qi - 36 * fh;
                        const uint4 w = *reinterpret_cast<const uint4*>(ustage + fh * SF_P + 4 * pq);
                        const unsigned int t0 = __byte_perm(w.x, w.y, 0x5140), t1 = __byte_perm(w.z, w.w, 0x5140);
                        const unsigned int t2 = __byte_perm(w.x, w.y, 0x7362), t3 = __byte_perm(w.z, w.w, 0x7362);
                        unsigned char* dst = bP + ((size_t)(pq >> 2) * FC + (fw + fh)) * 16 + 4 * (pq & 3);
                        const size_t pstride = (size_t)9 * FC * 16;
                        *reinterpret_cast<unsigned int*>(dst) = __byte_perm(t0, t1, 0x5410);
                        *reinterpret_cast<unsigned int*>(dst + pstride) = __byte_perm(t0, t1, 0x7632);
                        *reinterpret_cast<unsigned int*>(dst + 2 * pstride) = __byte_perm(t2, t3, 0x5410);
                        *reinterpret_cast<unsigned int*>(dst + 3 * pstride) = __byte_perm(t2, t3, 0x7632);
                    }
                }
                __syncwarp();
            }
            fence_proxy_async_smem();                             // my writes -> visible to the storer's TMA stores
            __syncwarp();
            if (lane == 0) sf_mbar_arrive(&done[s]);
        }
}

template <int MODE>
__global__ void __launch_bounds__(32 * (SF_NCW + 2), 1)
shrink_flat_kernel(const __grid_constant__ CUtensorMap mapD, const __grid_constant__ CUtensorMap mapS, const __grid_constant__ CUtensorMap mapY,
                   const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapVC, ShrinkFlatArgs a) {
    const DevState* st = a.st;
    const bool run = !st->done && shrink_flat_takes(st);
    if (!run) {                                            // a fallback kernel does (or did) the work: contribute nothing
        if (threadIdx.x == 0) { a.part_zz[blockIdx.x] = 0.0; a.part_nnz[blockIdx.x] = 0ull; a.part_max[blockIdx.x] = 0.f; a.part_wmax[blockIdx.x] = 0.f; }
        return;
    }
    const int r = st->svp;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int FC = a.FC, NS = a.NS, ncf = a.nchunkf;
    // S is an output, not a state variable of this pass (G_S needs D, L and Y only), and it can be rebuilt from D, Y and the
    // digit planes of W_next = D - S + Y/mu_next (rebuild_S_kernel).  It is stored when this iteration may be the last one
    // (the residual of the previous iteration is within 4x of the tolerance, or max_iter is reached), when the next Gram
    // will read it (fp64 Gram), or when the caller insists; otherwise 4 of the 20 bytes per element stay on the chip.
    const bool write_S = a.force_S || st->force_dmma || !(st->err > 4.0 * st->tol) || st->iter >= st->max_iter;
    if (!write_S && blockIdx.x == 0 && threadIdx.x == 0) *a.s_stale_next = 1;
    const double mu_d = st->mu;
    SfScal sc;
    sc.inv_mu = (float)(1.0 / mu_d); sc.mu_f = (float)mu_d; sc.lamq = (float)(st->lambda / mu_d);
    // the next pass uses mu_next = min(mu rho, mu 1e7) (control_post_kernel): same double arithmetic here
    const float inv_mu_next = (float)(1.0 / fmin(mu_d * st->rho, mu_d * 1e7));
    sc.Qf = (float)(2147483648.0 / st->wq_scale_next);
    sc.c1 = inv_mu_next * sc.Qf;

    extern __shared__ __align__(128) unsigned char sf_smem[];
    const size_t slot = (size_t)FC * SF_P * sizeof(float), stage_bytes = 3 * slot;
    unsigned char* ring = sf_smem;                                                    // [NS][D | Y | planes]
    float* Vst = reinterpret_cast<float*>(ring + (size_t)NS * stage_bytes);           // [NS][FC][8]   VC rows of the stage's frames
    float* Tb = Vst + (size_t)NS * FC * SF_KMAX;                                      // [SF_TG][8][4R]  T of the tiles of the current group
    unsigned int* ustage_all = reinterpret_cast<unsigned int*>(Tb + SF_TG * SF_TFLOATS);  // [8 warps][2 frames][144]
    uint64_t* full = reinterpret_cast<uint64_t*>(ustage_all + SF_NCW * 2 * SF_P);
    uint64_t* done = full + NS;
    uint64_t* freeb = done + NS;
    __shared__ double redd[32];

    if (threadIdx.x == 0) {
        for (int s = 0; s < NS; ++s) { mbar_init(&full[s], 1); mbar_init(&done[s], SF_NCW); mbar_init(&freeb[s], 1); }
        mbar_fence_init();
        tma_prefetch_desc(&mapD); tma_prefetch_desc(&mapS); tma_prefetch_desc(&mapY); tma_prefetch_desc(&mapQ); tma_prefetch_desc(&mapVC);
    }
    for (int idx = threadIdx.x; idx < SF_TG * SF_TFLOATS; idx += blockDim.x) Tb[idx] = 0.f;
    __syncthreads();

    auto tile_origin = [&](long long tl, int& j0, int& i0) {
        const int tcx = (int)(tl / a.ntile_r), trx = (int)(tl - (long long)tcx * a.ntile_r);
        j0 = 3 * tcx; i0 = trx * SF_R;
    };
    float zl_acc = 0.f, max_acc = 0.f, wmax_acc = 0.f;
    unsigned int nnz_acc = 0u;
    double zz_acc = 0.0;
    // this CTA's tiles: a contiguous range, walked in groups of SF_TG
    const long long tile0 = (a.ntiles * blockIdx.x) / gridDim.x, tile1 = (a.ntiles * (blockIdx.x + 1)) / gridDim.x;

    if (warp == 0) {
        // ===================== loader =====================
        if (lane == 0) {
            int q = 0;
            for (long long g0 = tile0; g0 < tile1; g0 += SF_TG) {
                const int gt = (int)min((long long)SF_TG, tile1 - g0);
                for (int c = 0; c < ncf; ++c)
                    for (int t = 0; t < gt; ++t, ++q) {
                        int j0, i0;
                        tile_origin(g0 + t, j0, i0);
                        const int s = q % NS;
                        const int u = q / NS;
                        if (u > 0) mbar_wait(&freeb[s], (uint32_t)((u - 1) & 1));
                        unsigned char* b = ring + (size_t)s * stage_bytes;
                        mbar_expect_tx(&full[s], (uint32_t)(2 * slot) + (uint32_t)(FC * SF_KMAX * sizeof(float)));
                        tma_load_2d(Vst + (size_t)s * FC * SF_KMAX, &mapVC, &full[s], 0, c * FC);
                        // no L2 evict_first hint: on these loads it cost 2 % per solve, on the stores nothing (94.4 ms without,
                        // 96.4 on the loads, 94.4 on the stores; 1080p x 300, profiles/r2r_shrink_variants.log)
                        tma_load_3d(b, &mapD, &full[s], i0, j0, c * FC);
                        tma_load_3d(b + slot, &mapY, &full[s], i0, j0, c * FC);
                    }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== storer =====================
        if (lane == 0) {
            int q = 0;
            for (long long g0 = tile0; g0 < tile1; g0 += SF_TG) {
                const int gt = (int)min((long long)SF_TG, tile1 - g0);
                for (int c = 0; c < ncf; ++c)
                    for (int t = 0; t < gt; ++t, ++q) {
                        int j0, i0;
                        tile_origin(g0 + t, j0, i0);
                        const int s = q % NS;
                        mbar_wait(&done[s], (uint32_t)((q / NS) & 1));
                        unsigned char* b = ring + (size_t)s * stage_bytes;
                        if (write_S) tma_store_3d(&mapS, b, i0, j0, c * FC);
                        tma_store_3d(&mapY, b + slot, i0, j0, c * FC);
                        for (int sl = 0; sl < 4; ++sl)
                            tma_store_3d(&mapQ, b + 2 * slot + (size_t)sl * 9 * FC * 16, 2 * c * FC, (int)((g0 + t) * 9), sl);
                        tma_store_commit();
                        tma_store_wait_read<0>();
                        sf_mbar_arrive(&freeb[s]);
                    }
            }
            tma_store_wait_all<0>();
        }
        __syncwarp();
    } else {
        // ===================== consumers =====================
        const int ct = threadIdx.x - 64, cw = ct >> 5;
        unsigned int* ustage = ustage_all + (size_t)cw * 2 * SF_P;
        const int tpieces = r * SF_R;                              // 16-byte pieces of r rows x 4R floats (one tile)
        int q = 0;
        for (long long g0 = tile0; g0 < tile1; g0 += SF_TG) {
            const int gt = (int)min((long long)SF_TG, tile1 - g0);
            // T of the group's tiles -> shared memory (everyone is done with the previous group: barrier at the end of the loop body)
            for (int pc = ct; pc < gt * tpieces; pc += SF_NTC) {
                const int t = pc / tpieces, w = pc - t * tpieces;
                sf_cp_async16(Tb + (size_t)t * SF_TFLOATS + 4 * w, a.Tt + (size_t)(g0 + t) * 16 * (4 * SF_R) + 4 * w);
            }
            sf_cp_async_wait_all();
            sf_bar_sync(1, SF_NTC);
#define SF_CALL(KR_) sf_group<KR_, MODE>(a, Tb, gt, ring, stage_bytes, Vst, ustage, full, done, q, lane, cw, sc, write_S, zl_acc, nnz_acc, max_acc, wmax_acc)
            switch (r) {
                case 0: SF_CALL(0); break;
                case 1: SF_CALL(1); break;
                case 2: SF_CALL(2); break;
                case 3: SF_CALL(3); break;
                case 4: SF_CALL(4); break;
                case 5: SF_CALL(5); break;
                case 6: SF_CALL(6); break;
                case 7: SF_CALL(7); break;
                default: SF_CALL(8); break;
            }
#undef SF_CALL
            zz_acc += (double)zl_acc; zl_acc = 0.f;
            sf_bar_sync(1, SF_NTC);                               // the group's T buffer is free again
        }
    }
    __syncthreads();
    double zt = block_sum(zz_acc, redd);
    if (threadIdx.x == 0) a.part_zz[blockIdx.x] = zt;
    double nt = block_sum((double)nnz_acc, redd);
    if (threadIdx.x == 0) a.part_nnz[blockIdx.x] = (unsigned long long)(nt + 0.5);
    double mt = block_max((double)max_acc, redd);
    if (threadIdx.x == 0) a.part_max[blockIdx.x] = (float)mt;
    // max |W_next| (a large sentinel if a value left the 32-bit range: |q| must stay <= 2^31 - 2^24) for the next scale
    double wt = block_max((double)wmax_acc, redd);
    if (threadIdx.x == 0) a.part_wmax[blockIdx.x] = (wt < 2130706432.0) ? (float)(wt / (double)sc.Qf) : 3.0e38f;
}

// -------------------------------------------------------------------------------------------------------------
static size_t sf_smem_bytes(int FC, int NS) {
    const size_t slot = (size_t)FC * SF_P * sizeof(float);
    return (size_t)NS * 3 * slot + (size_t)NS * FC * SF_KMAX * sizeof(float) + (size_t)SF_TG * SF_TFLOATS * sizeof(float) +
           (size_t)SF_NCW * 2 * SF_P * sizeof(unsigned int) + (size_t)3 * NS * sizeof(uint64_t) + 128;
}

bool make_shrink_flat_plan(int n, int rows, int cols, long long ld, int num_sms, const ShrinkStreamPlan& sp, ShrinkFlatPlan* out) {
    // same tiles and the same digit-plane geometry as the streamed kernel (they alternate on the same buffers)
    if (sp.R != SF_R || rows % 4 != 0) return false;
    ShrinkFlatPlan p;
    p.n = n; p.rows = rows; p.cols = cols; p.ld = ld;
    p.FC = 16;
    p.NS = 8;
    while (p.NS >= 3 && sf_smem_bytes(p.FC, p.NS) > SF_SMEM_CAP) --p.NS;
    if (p.NS < 3) return false;
    p.nchunkf = (n + p.FC - 1) / p.FC;
    p.ntile_r = sp.ntile_r; p.ntiles = sp.ntiles;
    p.grid = (int)std::min<long long>(num_sms, (p.ntiles + SF_TG - 1) / SF_TG);     // every CTA at least one group
    p.smem_bytes = sf_smem_bytes(p.FC, p.NS);
    *out = p;
    return true;
}

int make_shrink_flat_maps(const ShrinkFlatPlan& p, const float* D, float* S, float* Y, signed char* Wq, long long ldq, const float* VC, int vstride,
                          ShrinkFlatMaps* m) {
    const uint64_t dims[3] = {(uint64_t)p.rows, (uint64_t)p.cols, (uint64_t)p.n};
    const uint64_t strides[2] = {(uint64_t)p.rows * sizeof(float), (uint64_t)p.ld * sizeof(float)};
    const uint32_t box[3] = {(uint32_t)SF_R, 3u, (uint32_t)p.FC};
    if (make_tensor_map_f32(&m->D, D, 3, dims, strides, box) != 0) return -1;
    if (make_tensor_map_f32(&m->S, S, 3, dims, strides, box) != 0) return -1;
    if (make_tensor_map_f32(&m->Y, Y, 3, dims, strides, box) != 0) return -1;
    // digit planes [slice][k16][frame][16 B] viewed as 8-byte elements (see make_shrink_stream_qmap)
    const uint64_t qdims[3] = {(uint64_t)2 * p.n, (uint64_t)(ldq / 16), 4};
    const uint64_t qstrides[2] = {(uint64_t)16 * p.n, (uint64_t)ldq * (uint64_t)p.n};
    const uint32_t qbox[3] = {(uint32_t)(2 * p.FC), 9u, 1u};
    if (make_tensor_map_u64(&m->Q, Wq, 3, qdims, qstrides, qbox) != 0) return -1;
    if (vstride < SF_KMAX) { set_error("shrink_flat: VC row stride %d < %d", vstride, SF_KMAX); return -1; }
    const uint64_t vdims[2] = {(uint64_t)vstride, (uint64_t)p.n};
    const uint64_t vstrides[1] = {(uint64_t)vstride * sizeof(float)};
    const uint32_t vbox[2] = {(uint32_t)SF_KMAX, (uint32_t)p.FC};
    if (make_tensor_map_f32(&m->VC, VC, 2, vdims, vstrides, vbox) != 0) return -1;
    return 0;
}

// S = D + Y/mu - W_q: undo W_next = D - S + Y/mu_next from the digit planes the last pass wrote (mu has been advanced since, so
// DevState::mu IS that mu_next, and wq_scale is the scale of the planes that exist).  Runs only when DevState::s_stale is set.
// Natural pixel order for D, Y, S (coalesced); the four digit bytes of a pixel are gathered from the tile-major planes.
__global__ void __launch_bounds__(256) rebuild_S_kernel(const float* __restrict__ D, const float* __restrict__ Y, float* __restrict__ S,
                                                        const signed char* __restrict__ Wq, long long ld, long long ldq, int n, int rows, int cols,
                                                        int ntile_r, DevState* st, int min_rank) {
    if (!st->s_stale || st->svp < min_rank) return;
    const float inv_mu = (float)(1.0 / st->mu);
    const float sc = (float)(st->wq_scale * (1.0 / 2147483648.0));
    const size_t plane = (size_t)ldq * n;
    const long long m = (long long)rows * cols;
    // a small persistent grid: this kernel is launched every iteration and nearly always returns at the first line
    for (long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x; w < m * n; w += (long long)gridDim.x * blockDim.x) {
        {
            const int f = (int)(w / m);
            const long long p = w - (long long)f * m;
            const int j = (int)(p / rows), i = (int)(p - (long long)j * rows);
            const int tcx = j / 3, c = j - 3 * tcx, trx = i / SF_R, il = i - trx * SF_R, g = il / 3, dr = il - 3 * g;
            const int pos = (3 * c + dr) * SF_NG + g;
            const long long unit = ((long long)tcx * ntile_r + trx) * 9 + (pos >> 4);
            const signed char* q0 = Wq + ((size_t)unit * n + f) * 16 + (pos & 15);
            const unsigned int u = (unsigned int)(unsigned char)q0[0] | ((unsigned int)(unsigned char)q0[plane] << 8) |
                                   ((unsigned int)(unsigned char)q0[2 * plane] << 16) | ((unsigned int)(unsigned char)q0[3 * plane] << 24);
            const float wq = (float)(int)((u ^ 0x00808080u) - 0x00808080u) * sc;
            const size_t off = (size_t)f * ld + p;
            S[off] = fmaf(Y[off], inv_mu, D[off]) - wq;
        }
    }
}
__global__ void rebuild_S_done_kernel(DevState* st, int min_rank) { if (threadIdx.x == 0 && blockIdx.x == 0 && st->s_stale && st->svp >= min_rank) st->s_stale = 0; }

// min_rank: rebuild only if the rank of the coming shrink pass is at least this (0 = unconditionally when stale)
int launch_rebuild_S(const ShrinkFlatPlan& p, const float* D, const float* Y, float* S, const signed char* Wq, long long ldq, DevState* st,
                     int min_rank, cudaStream_t stream) {
    const long long m = (long long)p.rows * p.cols;
    long long gx = (m * p.n + 255) / 256;
    if (gx > 148 * 8) gx = 148 * 8;
    dim3 g((unsigned)gx);
    rebuild_S_kernel<<<g, 256, 0, stream>>>(D, Y, S, Wq, p.ld, ldq, p.n, p.rows, p.cols, p.ntile_r, st, min_rank);
    BSUB_CUDA_CHECK(cudaGetLastError());
    rebuild_S_done_kernel<<<1, 32, 0, stream>>>(st, min_rank);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

template <int MODE>
static int launch_sf(const ShrinkFlatPlan& p, const ShrinkFlatMaps& maps, const ShrinkFlatArgs& a, cudaStream_t stream) {
    static unsigned long long attr_devs = 0;
    if (first_call_on_device(&attr_devs))
        BSUB_CUDA_CHECK(cudaFuncSetAttribute(shrink_flat_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SF_SMEM_CAP));
    shrink_flat_kernel<MODE><<<p.grid, 32 * (SF_NCW + 2), p.smem_bytes, stream>>>(maps.D, maps.S, maps.Y, maps.Q, maps.VC, a);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_shrink_flat(const ShrinkFlatPlan& p, const ShrinkFlatMaps& maps, const float* Tt, DevState* st, int mode, int force_S, double* part_zz,
                       unsigned long long* part_nnz, float* part_max, float* part_wmax, cudaStream_t stream) {
    ShrinkFlatArgs a;
    a.s_stale_next = &st->s_stale_next; a.force_S = force_S ? 1 : 0;
    a.Tt = Tt; a.n = p.n; a.rows = p.rows; a.cols = p.cols; a.FC = p.FC; a.NS = p.NS; a.nchunkf = p.nchunkf; a.ntile_r = p.ntile_r;
    a.ntiles = p.ntiles; a.st = st; a.part_zz = part_zz; a.part_nnz = part_nnz; a.part_max = part_max; a.part_wmax = part_wmax; a.mode = mode;
    if (mode == SHRINK_L1) return launch_sf<SHRINK_L1>(p, maps, a, stream);
    if (mode == SHRINK_FLAT3) return launch_sf<SHRINK_FLAT3>(p, maps, a, stream);
    set_error("shrink_flat: mode %d is not handled by this kernel", mode);
    return -1;
}

}  // namespace bsub
