// gram_i8.cu -- the frames x frames Gram on the 5th-generation tensor cores (tcgen05, sm_100a), exact in integers.
//
// W (fp32) is written by the shrink pass as 32-bit fixed point q = rint(W * 2^31 / S) split into four balanced base-256
// digits (int8 "slices" d0..d3, q = sum d_k 256^k).  Then
//     q_f . q_g = sum_{i,j} 256^{i+j} (d_i(f) . d_j(g))
// and every slice-pair product is an int8 GEMM with exact int32 accumulation (tcgen05.mma.kind::i8, accumulators in
// TMEM).  Pairs of equal weight i+j share one TMEM accumulator ("class"); classes 3..6 are kept (the dropped ones sit
// below 2^-32 of the top class), i.e. 10 MMAs per 32-pixel k-step.  Accumulators are flushed to a global int64 matrix
// with atomics before int32 could overflow -- integer adds commute, so the result is exact AND deterministic.
// This replaces the fp64 DMMA Gram (gram.cu, FP64-pipe bound at ~6.4 ms for 1080p x 300) wherever the slices exist.
//
// Kernel anatomy (one CTA = one 128 x N output tile of the upper block triangle x a range of pixels):
//   warp 0     TMA producer: one 8 KB box {16 B, 128 frames, 4 k-blocks} per slice and frame block -- the slice matrix is
//              stored k-block-major ([slice][k16][frame][16 B]) so every box is four contiguous 2 KB runs and lands in
//              shared memory directly in the canonical K-major no-swizzle UMMA layout (8x16 B core matrices)
//   warp 1     MMA issuer (one elected thread): tcgen05.mma, tcgen05.commit -> mbarriers
//   warp 2     TMEM allocator (512 columns = 4 classes x 128)
//   warps 4-7  epilogue: tcgen05.ld of the four class accumulators, recombination into int64, atomicAdd to global
#include <cooperative_groups.h>
#include <math.h>
#include <algorithm>
#include <vector>
#include "common.cuh"
#include "kernels.h"
#include "tma.cuh"

namespace cg = cooperative_groups;

namespace bsub {

constexpr int GI_THREADS = 256;
constexpr int GI_KB = 64;                 // pixels (bytes) per pipeline stage = 4 k16 blocks = 2 MMA k-steps
constexpr int GI_STAGES = 3;
constexpr int GI_FLUSH_KB = 448;          // K blocks between flushes: 4 pairs * 448*64 px * 2^14 < 2^31
constexpr int GI_TILE_BYTES = 128 * GI_KB;            // one slice of one 128-frame block
constexpr int GI_STAGE_BYTES = 8 * GI_TILE_BYTES;     // A (4 slices) + B (4 slices)

struct GramI8Args {
    int n, nblk;
    const int4* cta_info;                 // per CTA: (bi, bj, first stage index, stage stride); stages are 64-pixel blocks
    int nkb;                              // number of 64-pixel stages in the slice matrix
    const int* blk_n;                     // MMA N of each frame block (multiple of 16, <= 128)
    unsigned long long* Gint;             // [nblk*128][nblk*128] int64 accumulators (zeroed by the caller)
    const DevState* st;
    int require_mode;                     // kernel is a no-op unless st->gram_mode == require_mode (when st != nullptr)
};

__device__ __forceinline__ void gi_mbar_wait(uint64_t* bar, uint32_t parity) {
    unsigned long long spins = 0;
    while (!mbar_try_wait(bar, parity)) { if (++spins > (1ull << 31)) __trap(); }     // watchdog: never hang the GPU
}
__device__ __forceinline__ void gi_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ uint64_t gi_smem_desc(uint32_t saddr, uint32_t lbo_bytes) {
    // K-major, no swizzle ("interleave"): 8 x 16 B core matrices; the two core matrices of one K = 32 MMA are 2048 B
    // apart (LBO: next k16 block of the stage), consecutive 8-frame groups 128 B apart (SBO); descriptor version 1
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)(128 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
__device__ __forceinline__ uint32_t gi_instr_desc(int N) {
    // kind::i8: c_format S32 (2) at [4,6); a_format / b_format signed 8-bit (1) at [7,10) / [10,13); K-major A and B;
    // n_dim = N >> 3 at [17,23); m_dim = 128 >> 4 at [24,29)
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void gi_mma(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
        ::"r"(tmem_c), "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void gi_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// The MMA warp runs its loop with ALL 32 lanes on warp-uniform values and lets one elected lane issue (the `_w` forms below).
// With a single-thread `if (lane == 0)` region the compiler cannot prove the descriptors uniform and wraps every
// tcgen05.mma in ELECT + 4 R2UR.BROADCAST + a BRA.U.ANY waterfall: ~92 cycles of issue per MMA against 64 cycles of execution
// (measured with clock64 in round 2: the issuing thread, not the tensor pipe or the operand feed, set the 1.5 ms of this kernel).
__device__ __forceinline__ void gi_mma_w(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
        ::"r"(tmem_c), "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void gi_commit_w(uint64_t* bar) {
    asm volatile("{\n\t.reg .pred e;\n\telect.sync _|e, 0xffffffff;\n\t"
                 "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
// whole-warp wait: every lane polls (all see the phase flip), then the warp reconverges
__device__ __forceinline__ void gi_mbar_wait_w(uint64_t* bar, uint32_t parity) {
    gi_mbar_wait(bar, parity);
    __syncwarp();
}
__device__ __forceinline__ void gi_tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                   "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
}

__global__ void __launch_bounds__(GI_THREADS, 1)
gram_i8_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapQlast, GramI8Args a) {
    if (a.st != nullptr && (a.st->done || a.st->gram_mode != a.require_mode)) return;
    extern __shared__ __align__(1024) unsigned char gi_smem[];
    unsigned char* stages = gi_smem;                                             // [GI_STAGES][8][128][64]
    uint64_t* full = reinterpret_cast<uint64_t*>(gi_smem + (size_t)GI_STAGES * GI_STAGE_BYTES);   // [GI_STAGES]
    uint64_t* empty = full + GI_STAGES;                                          // [GI_STAGES]
    uint64_t* tmem_full = empty + GI_STAGES;                                     // accumulators ready for the epilogue
    uint64_t* tmem_empty = tmem_full + 1;                                        // accumulators drained
    uint32_t* tmem_base_s = reinterpret_cast<uint32_t*>(tmem_empty + 1);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;     // provably warp-uniform
    const int4 info = a.cta_info[blockIdx.x];
    const int bi = info.x, bj = info.y, kb0 = info.z, kstride = info.w;
    const bool diag = (bi == bj);
    const int Nj = a.blk_n[bj];
    // stages kb0, kb0 + kstride, ...: all CTAs sweep the pixels front to back together, so a frame block fetched for one
    // output tile is still in L2 when the other tiles need it
    const int nkb = (a.nkb > kb0) ? (a.nkb - kb0 + kstride - 1) / kstride : 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < GI_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, 128);
        mbar_fence_init();
        tma_prefetch_desc(&mapQ);
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_s)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_base_s, 0);

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            // the B block of the last frame block only needs its Nj (< 128) frames: narrower box, fewer bytes
            const bool narrowB = (!diag && Nj < 128);
            const uint32_t tx = (uint32_t)(4 * GI_TILE_BYTES + (diag ? 0 : 4 * Nj * GI_KB));
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % GI_STAGES;
                const int u = kb / GI_STAGES;
                if (u > 0) gi_mbar_wait(&empty[s], (uint32_t)((u - 1) & 1));
                unsigned char* base = stages + (size_t)s * GI_STAGE_BYTES;
                mbar_expect_tx(&full[s], tx);
                const int k16 = (kb0 + kb * kstride) * (GI_KB / 16);
                for (int sl = 0; sl < 4; ++sl) {
                    tma_load_3d(base + (size_t)sl * GI_TILE_BYTES, &mapQ, &full[s], bi * 256, k16, sl);
                    if (!diag) tma_load_3d(base + (size_t)(4 + sl) * GI_TILE_BYTES, narrowB ? &mapQlast : &mapQ, &full[s], bj * 256, k16, sl);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== MMA issuer (whole warp, one elected lane issues: see gi_mma_w) =====================
        {
            const uint32_t idesc = gi_instr_desc(Nj);
            const uint32_t lboB = (diag || Nj == 128) ? 2048u : (uint32_t)(Nj * 16);
            const uint64_t descA0 = gi_smem_desc(0u, 2048u), descB0 = gi_smem_desc(0u, lboB);
            int since_flush = 0, nflush = 0;
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % GI_STAGES;
                const int u = kb / GI_STAGES;
                if (since_flush == 0 && nflush > 0) {
                    gi_mbar_wait_w(tmem_empty, (uint32_t)((nflush - 1) & 1));        // epilogue has drained TMEM
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                gi_mbar_wait_w(&full[s], (uint32_t)(u & 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sbase = smem_u32(stages + (size_t)s * GI_STAGE_BYTES);
                // descriptors = per-kernel constant part + (address >> 4): one 64-bit add per operand
                const uint64_t sa = descA0 + (uint64_t)((sbase >> 4) & 0x3FFF);
                const uint64_t sb = descB0 + (uint64_t)(((sbase + (diag ? 0u : (uint32_t)(4 * GI_TILE_BYTES))) >> 4) & 0x3FFF);
#pragma unroll
                for (int ks = 0; ks < GI_KB / 32; ++ks) {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int cls = i + j - 3;
                            if (cls < 0) continue;
                            // diagonal tile: P_ji = P_ij^T, classes 0 and 2 keep the i < j half (7 of 10 products); the epilogue
                            // adds the transpose (as in gram_i8_c3_kernel)
                            if (diag && cls != 1 && i > j) continue;
                            const uint64_t da = sa + (uint64_t)((i * GI_TILE_BYTES + ks * 4096) >> 4);
                            const uint64_t db = sb + (uint64_t)((j * GI_TILE_BYTES) >> 4) + (uint64_t)ks * (uint64_t)((2 * lboB) >> 4);
                            // first pair of a class right after a flush overwrites the accumulator
                            const bool first = (since_flush == 0 && ks == 0 && j == 3);   // (i, 3) is the first pair of class i
                            gi_mma_w(tmem_base + (uint32_t)(cls * 128), da, db, idesc, first ? 0u : 1u);
                        }
                }
                gi_commit_w(&empty[s]);                                          // smem stage reusable when these MMAs finish
                ++since_flush;
                if (since_flush == GI_FLUSH_KB || kb == nkb - 1) {
                    gi_commit_w(tmem_full);                                      // accumulators complete -> epilogue
                    since_flush = 0; ++nflush;
                }
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ===================== epilogue =====================
        const int ew = warp - 4;                                                 // TMEM lanes 32*ew .. 32*ew+31
        const int nflush_total = (nkb + GI_FLUSH_KB - 1) / GI_FLUSH_KB;
        const int row = bi * 128 + ew * 32 + lane;
        const size_t ldg = (size_t)a.nblk * 128;
        for (int fl = 0; fl < nflush_total; ++fl) {
            gi_mbar_wait(tmem_full, (uint32_t)(fl & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int c0 = 0; c0 < Nj; c0 += 16) {
                uint32_t v3[16], v4[16], v5[16], v6[16];
                const uint32_t ta = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)c0;
                gi_tmem_ld16(ta + 0 * 128, v3);
                gi_tmem_ld16(ta + 1 * 128, v4);
                gi_tmem_ld16(ta + 2 * 128, v5);
                gi_tmem_ld16(ta + 3 * 128, v6);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (row < a.n) {
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        const int col = bj * 128 + c0 + e;
                        if (col < a.n) {
                            const long long half = (long long)(int)v3[e] + ((long long)(int)v5[e] << 16);
                            const long long val = half + ((long long)(int)v4[e] << 8) + ((long long)(int)v6[e] << 24);
                            if (val != 0) atomicAdd(a.Gint + (size_t)row * ldg + col, (unsigned long long)val);
                            if (diag && half != 0) atomicAdd(a.Gint + (size_t)col * ldg + row, (unsigned long long)half);
                        }
                    }
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            gi_mbar_arrive(tmem_empty);
        }
    }
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Three frame blocks (256 < n <= 384, the 300-frame clips): clusters of 3 CTAs share operand tiles through TMA multicast.
// gram_i8_kernel above is bound by L2 -> SM bytes: every 128-frame block is fetched by each of the block pairs that use it.
// Here the frames are cut into three blocks of nb = ceil(n / 3) frames (100 for n = 300: MMA N = 112 instead of 128; a box still
// carries 128 frames, the rows / columns beyond a block's own frames are never read by the epilogue) and the six tiles of the
// block triangle are dealt to two kinds of cluster:
//   type X (off-diagonal)  rank 0: (0,1)   rank 1: (0,2)   rank 2: (1,2)      10 digit pairs per k-step
//        block 0 -> slot A of ranks 0,1 (one multicast load by rank 0); block 2 -> slot B of ranks 1,2 (rank 1);
//        block 1 -> slot A of rank 2 (rank 2) and slot B of rank 0 (rank 0: a block can only be multicast to ONE slot offset)
//   type Y (diagonal)      rank r: (r,r), both operands from its own slot A     7 digit pairs per k-step
//        P_ji = P_ij^T on a diagonal tile, so classes 0 and 2 accumulate only H = sum_{i<j} P_ij and the epilogue adds H to
//        (r,c) AND (c,r); class 1 holds the symmetric pair P_22 and keeps all three of its products, class 3 is P_33 alone.
// X clusters cost 20 MMAs per 64-pixel stage, Y clusters 14: the pixel stages are split nX : nY ~ 20 : 14 between them.
// Stage hand-back: the MMA warp commits (tcgen05.commit ... multicast::cluster) to the `empty` barrier of every CTA that supplied
// one of its operands, and to its own `mine` barrier, which paces the re-arming of its `full` barrier.
struct GramI8C3Args {
    int n, nkb;                           // frames; 64-pixel stages in the slice matrix
    int nX, nY;                           // clusters of each type (cluster id < nX: type X)
    int nb, N;                            // frames per block, MMA N (nb rounded up to 16)
    unsigned long long* Gint;
    const DevState* st;
    int require_mode;
};

__device__ __forceinline__ void gi_tma_load_3d_mc(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                                  uint16_t cta_mask) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, %5}], [%2], %6;"
                 ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void gi_commit_mc_w(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("{\n\t.reg .pred e;\n\telect.sync _|e, 0xffffffff;\n\t"
                 "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}"
                 ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}

__global__ void __launch_bounds__(GI_THREADS, 1)
gram_i8_c3_kernel(const __grid_constant__ CUtensorMap mapQ, GramI8C3Args a) {
    if (a.st != nullptr && (a.st->done || a.st->gram_mode != a.require_mode)) return;      // uniform over the grid
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(1024) unsigned char gi_smem[];
    unsigned char* stages = gi_smem;                                             // [GI_STAGES][A: 4 planes | B: 4 planes][128][64]
    uint64_t* full = reinterpret_cast<uint64_t*>(gi_smem + (size_t)GI_STAGES * GI_STAGE_BYTES);   // [GI_STAGES]
    uint64_t* empty = full + GI_STAGES;                                          // [GI_STAGES] consumers of the slots I load are done
    uint64_t* mine = empty + GI_STAGES;                                          // [GI_STAGES] my own MMAs on the stage are done
    uint64_t* tmem_full = mine + GI_STAGES;
    uint64_t* tmem_empty = tmem_full + 1;
    uint32_t* tmem_base_s = reinterpret_cast<uint32_t*>(tmem_empty + 1);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;     // provably warp-uniform
    const int rank = (int)cluster.block_rank();
    const int cid = blockIdx.x / 3;
    const bool tX = cid < a.nX;
    const int kb0 = tX ? cid : cid - a.nX, kstride = tX ? a.nX : a.nY;
    const int nkb = (a.nkb > kb0) ? (a.nkb - kb0 + kstride - 1) / kstride : 0;
    // role table (see the header comment)
    const int bi = tX ? (rank == 2 ? 1 : 0) : rank;
    const int bj = tX ? (rank == 0 ? 1 : 2) : rank;
    const bool diag = !tX;
    // what I load: up to two (slot, frame block, destination CTAs)
    int ld0_slot, ld0_blk, ld1_slot = -1, ld1_blk = 0; uint16_t ld0_mask, ld1_mask = 0;
    uint16_t sup_mask; int n_consumers;
    if (tX) {
        if (rank == 0)      { ld0_slot = 0; ld0_blk = 0; ld0_mask = 0x3; ld1_slot = 1; ld1_blk = 1; ld1_mask = 0x1; sup_mask = 0x1; n_consumers = 2; }
        else if (rank == 1) { ld0_slot = 1; ld0_blk = 2; ld0_mask = 0x6; sup_mask = 0x3; n_consumers = 2; }
        else                { ld0_slot = 0; ld0_blk = 1; ld0_mask = 0x4; sup_mask = 0x6; n_consumers = 1; }
    } else { ld0_slot = 0; ld0_blk = rank; ld0_mask = (uint16_t)(1u << rank); sup_mask = ld0_mask; n_consumers = 1; }

    if (threadIdx.x == 0) {
        for (int s = 0; s < GI_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], n_consumers); mbar_init(&mine[s], 1); }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, 128);
        mbar_fence_init();
        tma_prefetch_desc(&mapQ);
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_s)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster.sync();                                        // barriers of all three CTAs exist before anything is signalled
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_base_s, 0);

    if (warp == 0) {
        // ===================== TMA producer: arms my full barrier, loads the slots I own =====================
        if (lane == 0) {
            const uint32_t tx = (uint32_t)(tX ? 8 : 4) * GI_TILE_BYTES;
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % GI_STAGES;
                const int u = kb / GI_STAGES;
                if (u > 0) gi_mbar_wait(&mine[s], (uint32_t)((u - 1) & 1));           // my MMAs of the previous round are done
                mbar_expect_tx(&full[s], tx);
                if (u > 0) gi_mbar_wait(&empty[s], (uint32_t)((u - 1) & 1));          // and so are those of everyone I feed
                unsigned char* base = stages + (size_t)s * GI_STAGE_BYTES;
                const int k16 = (kb0 + kb * kstride) * (GI_KB / 16);
                for (int sl = 0; sl < 4; ++sl)
                    gi_tma_load_3d_mc(base + (size_t)(ld0_slot * 4 + sl) * GI_TILE_BYTES, &mapQ, &full[s], ld0_blk * 2 * a.nb, k16, sl, ld0_mask);
                if (ld1_slot >= 0)
                    for (int sl = 0; sl < 4; ++sl)
                        gi_tma_load_3d_mc(base + (size_t)(ld1_slot * 4 + sl) * GI_TILE_BYTES, &mapQ, &full[s], ld1_blk * 2 * a.nb, k16, sl, ld1_mask);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== MMA issuer (whole warp, one elected lane issues: see gi_mma_w) =====================
        {
            const uint32_t idesc = gi_instr_desc(a.N);
            const uint32_t offB = diag ? 0u : (uint32_t)(4 * GI_TILE_BYTES);
            const uint64_t desc0 = gi_smem_desc(0u, 2048u);      // constant part of the operand descriptors (see gram_i8_kernel)
            int since_flush = 0, nflush = 0;
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % GI_STAGES;
                const int u = kb / GI_STAGES;
                if (since_flush == 0 && nflush > 0) {
                    gi_mbar_wait_w(tmem_empty, (uint32_t)((nflush - 1) & 1));
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                gi_mbar_wait_w(&full[s], (uint32_t)(u & 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sbase = smem_u32(stages + (size_t)s * GI_STAGE_BYTES);
                // (in a cluster launch the shared-window address carries CTA-rank bits above the 14-bit descriptor field: mask)
                const uint64_t sa = desc0 + (uint64_t)((sbase >> 4) & 0x3FFF), sb = desc0 + (uint64_t)(((sbase + offB) >> 4) & 0x3FFF);
                if (!diag) {
#pragma unroll
                    for (int ks = 0; ks < GI_KB / 32; ++ks) {
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const int cls = i + j - 3;
                                if (cls < 0) continue;
                                const uint64_t da = sa + (uint64_t)((i * GI_TILE_BYTES + ks * 4096) >> 4);
                                const uint64_t db = sb + (uint64_t)((j * GI_TILE_BYTES + ks * 4096) >> 4);
                                const bool first = (since_flush == 0 && ks == 0 && j == 3);
                                gi_mma_w(tmem_base + (uint32_t)(cls * 128), da, db, idesc, first ? 0u : 1u);
                            }
                    }
                } else {
#pragma unroll
                    for (int ks = 0; ks < GI_KB / 32; ++ks) {
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const int cls = i + j - 3;
                                if (cls < 0) continue;
                                if (cls != 1 && i > j) continue;       // classes 0 and 2: the i < j half; the epilogue adds the transpose
                                const uint64_t da = sa + (uint64_t)((i * GI_TILE_BYTES + ks * 4096) >> 4);
                                const uint64_t db = sb + (uint64_t)((j * GI_TILE_BYTES + ks * 4096) >> 4);
                                const bool first = (since_flush == 0 && ks == 0 && j == 3);
                                gi_mma_w(tmem_base + (uint32_t)(cls * 128), da, db, idesc, first ? 0u : 1u);
                            }
                    }
                }
                gi_commit_mc_w(&empty[s], sup_mask);                               // hand the operand slots back to their loaders
                gi_commit_w(&mine[s]);
                ++since_flush;
                if (since_flush == GI_FLUSH_KB || kb == nkb - 1) {
                    gi_commit_w(tmem_full);
                    since_flush = 0; ++nflush;
                }
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ===================== epilogue =====================
        const int ew = warp - 4;
        const int nflush_total = (nkb + GI_FLUSH_KB - 1) / GI_FLUSH_KB;
        const int lrow = ew * 32 + lane;
        const int row = bi * a.nb + lrow;
        const bool row_ok = lrow < a.nb && row < a.n;
        const size_t ldg = (size_t)3 * 128;
        for (int fl = 0; fl < nflush_total; ++fl) {
            gi_mbar_wait(tmem_full, (uint32_t)(fl & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int c0 = 0; c0 < a.N; c0 += 16) {
                uint32_t v3[16], v4[16], v5[16], v6[16];
                const uint32_t ta = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)c0;
                gi_tmem_ld16(ta + 0 * 128, v3);
                gi_tmem_ld16(ta + 1 * 128, v4);
                gi_tmem_ld16(ta + 2 * 128, v5);
                gi_tmem_ld16(ta + 3 * 128, v6);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (row_ok) {
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        const int lcol = c0 + e, col = bj * a.nb + lcol;
                        if (lcol < a.nb && col < a.n) {
                            const long long half = (long long)(int)v3[e] + ((long long)(int)v5[e] << 16);
                            const long long whole = ((long long)(int)v4[e] << 8) + ((long long)(int)v6[e] << 24);
                            const long long val = half + whole;
                            if (val != 0) atomicAdd(a.Gint + (size_t)row * ldg + col, (unsigned long long)val);
                            if (diag && half != 0) atomicAdd(a.Gint + (size_t)col * ldg + row, (unsigned long long)half);
                        }
                    }
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            gi_mbar_arrive(tmem_empty);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster.sync();                                        // nobody leaves while a neighbour may still write or signal here
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ---- D -> the four int8 digit planes (initialisation: Gram(D) runs on the tensor cores too).  The planes use the natural
// pixel order here; the Gram is a sum over pixels and does not care as long as all frames agree.
// scale S = 2^ceil(log2(2 max|D|)) is left in st->wq_scale for gram_i8_finish_kernel.
__global__ void __launch_bounds__(256) quantize_D_kernel(const float* __restrict__ D, long long ld, int n, long long ldq,
                                                         signed char* __restrict__ Wq, const double* __restrict__ dmax, DevState* st) {
    // tile = QD_F frames x QD_KB k-blocks (16 pixels each): coalesced 1 KB row reads, digits staged in shared memory,
    // then every plane is written as runs of QD_F * 16 contiguous bytes ([k16][frame][16 B] layout)
    constexpr int QD_F = 32, QD_KB = 16;
    __shared__ uint4 stage[4][QD_KB][QD_F + 1];
    const double mx = *dmax;
    const double S = (mx > 0.0) ? exp2(ceil(log2(2.0 * mx))) : 1.0;
    if (blockIdx.x == 0 && threadIdx.x == 0) st->wq_scale = S;
    const float Qf = (float)(2147483648.0 / S);
    const long long nkb = ldq / 16, plane = ldq * (long long)n;
    const long long ntk = (nkb + QD_KB - 1) / QD_KB;
    const int ntf = (n + QD_F - 1) / QD_F;
    const long long ntiles = ntk * ntf;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long kb0 = (tile / ntf) * QD_KB;
        const int f0 = (int)(tile % ntf) * QD_F;
        // read: a frame's share of the tile is 16 k-blocks x 16 floats = 64 float4 (1 KB contiguous)
#pragma unroll
        for (int pass = 0; pass < 8; ++pass) {
            const int idx = pass * 256 + threadIdx.x;        // 0 .. 2047 = 32 frames x 64 float4
            const int fl = idx >> 6, q4 = idx & 63;          // frame in tile, float4 index within the 256-pixel run
            const int f = f0 + fl;
            const long long p = kb0 * 16 + 4 * q4;
            float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
            if (f < n && p < ld) d = ldg4_stream(D + (size_t)f * ld + p);
            // balanced base-256 digits: byte k of ((q + 0x808080) ^ 0x808080) is digit k as a signed byte (shrink_stream.cu)
            const unsigned int u0 = ((unsigned int)__float2int_rn(d.x * Qf) + 0x00808080u) ^ 0x00808080u;
            const unsigned int u1 = ((unsigned int)__float2int_rn(d.y * Qf) + 0x00808080u) ^ 0x00808080u;
            const unsigned int u2 = ((unsigned int)__float2int_rn(d.z * Qf) + 0x00808080u) ^ 0x00808080u;
            const unsigned int u3 = ((unsigned int)__float2int_rn(d.w * Qf) + 0x00808080u) ^ 0x00808080u;
            const int kbl = q4 >> 2, wq = q4 & 3;             // k-block within tile, 32-bit word within its 16 bytes
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const unsigned int sel = (unsigned int)k | ((unsigned int)(4 + k) << 4);
                reinterpret_cast<unsigned int*>(&stage[k][kbl][fl])[wq] =
                    __byte_perm(__byte_perm(u0, u1, sel), __byte_perm(u2, u3, sel), 0x5410);
            }
        }
        __syncthreads();
        // write: per plane and k-block a run of QD_F x 16 B
#pragma unroll
        for (int pass = 0; pass < 8; ++pass) {
            const int idx = pass * 256 + threadIdx.x;        // 0 .. 2047 = 4 planes x 16 k-blocks x 32 frames
            const int fl = idx & 31, kbl = (idx >> 5) & 15, k = idx >> 9;
            const int f = f0 + fl;
            const long long kb = kb0 + kbl;
            if (f < n && kb < nkb) *reinterpret_cast<uint4*>(Wq + (size_t)k * plane + ((size_t)kb * n + f) * 16) = stage[k][kbl][fl];
        }
        __syncthreads();
    }
}

int launch_quantize_D(const float* D, long long ld, int n, long long ldq, signed char* Wq, const double* dmax, DevState* st,
                      cudaStream_t stream) {
    const long long ntiles = ((ldq / 16 + 15) / 16) * ((n + 31) / 32);
    const int grid = (int)std::min<long long>(ntiles, 148LL * 8);
    quantize_D_kernel<<<grid, 256, 0, stream>>>(D, ld, n, ldq, Wq, dmax, st);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// G[i][j] (double, [npad][npad], symmetric) = Gint * scale   with  scale = S^2 * 2^-38
__global__ void gram_i8_finish_kernel(const unsigned long long* __restrict__ Gint, int nblk, int blk, int n, int npad, double* __restrict__ G,
                                      const DevState* st, double scale_override, int require_mode, double diag_bias, double err_units,
                                      double* err_slot) {
    const bool runs = !(st != nullptr && (st->done || st->gram_mode != require_mode));
    const double scale = (st != nullptr) ? st->wq_scale * st->wq_scale * 0x1p-38 : scale_override;
    // bound of what the dropped digit classes may have taken from an eigenvalue of this rank's partial Gram (0 when the fp64
    // Gram did the work); it travels with the Gram through the all-reduce, so every rank sees the same total (eig.cu)
    if (err_slot != nullptr && blockIdx.x == 0 && threadIdx.x == 0 && !(st != nullptr && st->done)) *err_slot = runs ? 2.0 * err_units * scale : 0.0;
    if (!runs) return;
    const size_t ldg = (size_t)nblk * 128;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < npad * npad; idx += gridDim.x * blockDim.x) {
        const int i = idx / npad, j = idx - i * npad;
        double v = 0.0;
        if (i < n && j < n) {
            const int r = (i / blk <= j / blk) ? i : j, c = (i / blk <= j / blk) ? j : i;     // upper block triangle holds the data (blk frames per block)
            // diag_bias: expected value of the digit products the kernel drops (classes i + j <= 2), see launch_gram_i8
            v = ((double)(long long)Gint[(size_t)r * ldg + c] + ((i == j) ? diag_bias : 0.0)) * scale;
        }
        G[idx] = v;
    }
}

// -------------------------------------------------------------------------------------------------------------
GramI8Plan make_gram_i8_plan(int n, long long ldq, int num_sms) {
    GramI8Plan p;
    p.n = n; p.ldq = ldq; p.m_real = 0; p.m_global = 0;
    p.nblk = (n + 127) / 128;
    p.nkb = (int)(ldq / GI_KB);          // ldq = pixels per frame in the slice matrix, a multiple of 64
    p.smem_bytes = (size_t)GI_STAGES * GI_STAGE_BYTES + 256 + 1024;
    p.grid = num_sms;
    return p;
}

void fill_gram_i8_tables(const GramI8Plan& p, std::vector<int4>& cta_info, std::vector<int>& blk_n) {
    blk_n.assign(p.nblk, 128);
    const int last = p.n - (p.nblk - 1) * 128;
    blk_n[p.nblk - 1] = std::min(128, ((last + 15) / 16) * 16);
    // CTAs per output tile proportional to its MMA cost (N of the column block); every tile gets at least one
    std::vector<std::pair<int, int>> tiles;
    std::vector<double> w;
    double wsum = 0.0;
    for (int bi = 0; bi < p.nblk; ++bi)
        for (int bj = bi; bj < p.nblk; ++bj) {
            // half operand bytes per 64-pixel stage (one block on the diagonal, two off it), half MMAs (14 vs 20 per stage, x N / 128)
            const double cost = 0.5 * (128.0 + (bi == bj ? 0.0 : (double)blk_n[bj])) / 256.0 +
                                0.5 * (bi == bj ? 0.7 : 1.0) * (double)blk_n[bj] / 128.0;
            tiles.push_back({bi, bj}); w.push_back(cost); wsum += cost;
        }
    std::vector<int> cnt(tiles.size(), 1);
    int left = p.grid - (int)tiles.size();
    if (left < 0) left = 0;
    // largest-remainder apportionment
    std::vector<double> want(tiles.size());
    int given = 0;
    for (size_t t = 0; t < tiles.size(); ++t) { want[t] = w[t] / wsum * left; cnt[t] += (int)want[t]; given += (int)want[t]; }
    while (given < left) {
        size_t best = 0; double br = -1.0;
        for (size_t t = 0; t < tiles.size(); ++t) { double r = want[t] - (int)want[t]; if (r > br) { br = r; best = t; } }
        cnt[best]++; want[best] = (int)want[best]; ++given;
    }
    cta_info.clear();
    for (size_t t = 0; t < tiles.size(); ++t) {
        const int c = std::min(cnt[t], std::max(1, p.nkb));
        for (int k = 0; k < c; ++k) cta_info.push_back(make_int4(tiles[t].first, tiles[t].second, k, c));
    }
}

int gram_i8_last_block_n(const GramI8Plan& p) {
    const int last = p.n - (p.nblk - 1) * 128;
    return std::min(128, ((last + 15) / 16) * 16);
}

int make_gram_i8_map(const GramI8Plan& p, const signed char* Wq, CUtensorMap* map, int box_frames) {
    // k-block-major slice matrix [slice][k16][frame][16 B]: the frames of one k16 block are contiguous (16 n bytes), so the
    // map views them as 2 n eight-byte elements and a box row carries 16 * box_frames contiguous bytes (a 16-byte inner
    // dimension would make the TMA unit issue one request per frame and cap the feed rate); boxes {2 box_frames, 4, 1};
    // frames beyond n read as zero
    const uint64_t dims[3] = {(uint64_t)2 * p.n, (uint64_t)(p.ldq / 16), 4};
    const uint64_t strides[2] = {(uint64_t)16 * p.n, (uint64_t)p.ldq * (uint64_t)p.n};
    const uint32_t box[3] = {(uint32_t)(2 * box_frames), 4, 1};
    return make_tensor_map_u64(map, Wq, 3, dims, strides, box);
}

static int g_last_block_frames = 128;
// frames per block of the upper block triangle the most recent launch left in Gint (test hook: bsub_gram_i8_test reads Gint itself)
int gram_i8_last_block_frames() { return g_last_block_frames; }

int launch_gram_i8(const GramI8Plan& p, const CUtensorMap& map, const CUtensorMap& map_last, const int4* cta_info_dev, int ncta, const int* blk_n_dev,
                   unsigned long long* Gint, double* G, int npad, const DevState* st, double scale_override, int require_mode,
                   cudaStream_t stream) {
    static unsigned long long attr_devs = 0;      // one bit per device: the attribute is per (function, device)
    if (first_call_on_device(&attr_devs)) {
        BSUB_CUDA_CHECK(cudaFuncSetAttribute(gram_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_bytes));
    }
    // The kernel keeps the digit-pair classes i + j >= 3 of q_f q_g = sum 256^(i+j) d_i(f) d_j(g).  With q = A 2^16 + B
    // (B = d0 + 256 d1, the low 16 bits as a balanced number) the dropped part is B_f B_g + 2^16 (d0_f d2_g + d2_f d0_g):
    //   * on the diagonal its mean is E_d = E[d0^2] + 512 E[d0] E[d1] + 65536 E[d1^2] + 2^17 E[d0] E[d2] per pixel for uniformly
    //     distributed low digits (d uniform on -128..127: E[d] = -1/2, E[d^2] = 5461.5), i.e. the raw sums are too SMALL by
    //     m E_d: every eigenvalue sits ~1e-10 lambda_1 too low -- the size of (1/mu)^2 after ~20 ALM iterations;
    //   * off the diagonal it is a zero-mean sum over the pixels: a random symmetric matrix with entry deviation
    //     sqrt(m) E_o (E_o^2 = E[B^2]^2 + 2 (65536 sd(d0) sd(d2))^2) and spectral norm ~ 2 sqrt(n m) E_o.
    //   * worse, the d0 x d2 part is COHERENT: the third digit of a pixel is nearly the same in every frame (static background),
    //     so sum_p d0_f d2_g ~ r_f for all g: a rank-2 perturbation r 1^T + 1 r^T of norm <= n sqrt(m) 65536 sd(d0) max|d2|.
    // Adding back m E_d alone would centre this noise on zero and let it push cluster eigenvalues ABOVE the threshold in late
    // iterations (seen: rank inflation at iteration 21+ of WaterSurface delta = 1, iteration 20 of a 48x60x600 clip).  So the
    // diagonal gets m E_d - err with err = sqrt(m) (n + 3 sqrt(n)) E_o, a bound of the noise norm: the Gram then errs LOW by
    // at most 2 err -- it can never invent rank.  2 err (in the units of G) is handed to the eigensolver, which switches the
    // solve to the fp64 Gram (gram.cu) once that bound stops being small against the threshold (1/mu)^2 (eig.cu, force_dmma).
    // m_real = 0 (operator test) keeps the raw integer sums.  (The int64 accumulators hold the kept classes / 256^3: 2^-24.)
    const double E_d = 5461.5 + 128.0 + 65536.0 * 5461.5 + 131072.0 * 0.25, E_o = 6.2e8;
    // Pixel-sharded runs: the noise is a sum over ALL pixels of zero-mean terms, so its norm grows like sqrt(m_global); every rank
    // takes its share m / m_global of that global bound, and the all-reduce of the slot adds the shares up again.
    const double mg = (double)std::max(p.m_global, p.m_real);
    const double err_units = (p.m_real > 0) ? ((double)p.m_real / sqrt(mg)) * ((double)p.n + 3.0 * sqrt((double)p.n)) * E_o * 0x1p-24 : 0.0;
    const double diag_bias = (p.m_real > 0) ? (double)p.m_real * E_d * 0x1p-24 - err_units : 0.0;
    const size_t gbytes = sizeof(unsigned long long) * (size_t)p.nblk * 128 * p.nblk * 128;
    BSUB_CUDA_CHECK(cudaMemsetAsync(Gint, 0, gbytes, stream));
    // three frame blocks: the 3-CTA multicast clusters (gram_i8_c3_kernel); anything else: independent CTAs
    static int c3_clusters = -1;                           // -1: not probed yet, 0: unavailable
    if (p.nblk == 3 && c3_clusters != 0) {
        cudaLaunchConfig_t cfg = {};
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 3; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.blockDim = dim3(GI_THREADS); cfg.dynamicSmemBytes = p.smem_bytes; cfg.stream = stream; cfg.attrs = at; cfg.numAttrs = 1;
        if (c3_clusters < 0) {
            c3_clusters = 0;
            if (getenv("BSUB_NO_GRAM_CLUSTER") == nullptr &&
                cudaFuncSetAttribute(gram_i8_c3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_bytes) == cudaSuccess) {
                cfg.gridDim = dim3(3 * (p.grid / 3));
                int ncl = 0;
                if (cudaOccupancyMaxActiveClusters(&ncl, gram_i8_c3_kernel, &cfg) == cudaSuccess && ncl >= 2) c3_clusters = std::min(ncl, p.grid / 3);
            }
            (void)cudaGetLastError();
        }
        if (c3_clusters >= 2) {
            GramI8C3Args c;
            c.n = p.n; c.nkb = p.nkb;
            c.nb = (p.n + 2) / 3; c.N = ((c.nb + 15) / 16) * 16;
            // pixel stages in proportion to the MMAs per stage: 20 on the off-diagonal clusters, 14 on the diagonal ones
            c.nX = std::min(c3_clusters - 1, std::max(1, (int)lround(c3_clusters * 20.0 / 34.0))); c.nY = c3_clusters - c.nX;
            c.Gint = Gint; c.st = st; c.require_mode = require_mode;
            g_last_block_frames = c.nb;
            cfg.gridDim = dim3(3 * c3_clusters);
            BSUB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, gram_i8_c3_kernel, map, c));
            gram_i8_finish_kernel<<<64, 256, 0, stream>>>(Gint, p.nblk, c.nb, p.n, npad, G, st, scale_override, require_mode, diag_bias, err_units,
                                                          (st != nullptr) ? G + (size_t)npad * npad + 8 : nullptr);
            BSUB_CUDA_CHECK(cudaGetLastError());
            return 0;
        }
    }
    GramI8Args a;
    a.n = p.n; a.nblk = p.nblk; a.nkb = p.nkb; a.cta_info = cta_info_dev; a.blk_n = blk_n_dev; a.Gint = Gint; a.st = st; a.require_mode = require_mode;
    gram_i8_kernel<<<ncta, GI_THREADS, p.smem_bytes, stream>>>(map, map_last, a);
    BSUB_CUDA_CHECK(cudaGetLastError());
    g_last_block_frames = 128;
    gram_i8_finish_kernel<<<64, 256, 0, stream>>>(Gint, p.nblk, 128, p.n, npad, G, st, scale_override, require_mode, diag_bias, err_units,
                                                          (st != nullptr) ? G + (size_t)npad * npad + 8 : nullptr);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

}  // namespace bsub
