// project.cu -- T = Vr^T W straight from the int8 digit planes of W (first half of the SVT reconstruction,
// /root/reference/utils.py:185-186 with L = (W Vr) diag(1 - 1/(mu sigma)) Vr^T).
//
// The shrink pass of the previous iteration left W of THIS iteration in HBM as four int8 digit planes (32-bit fixed
// point, 4 B per element, layout [plane][k16 block][frame][16 B], pixels in the tile-major order of shrink_stream.cu);
// the tensor-core Gram has just read them.  Projecting onto the svp <= 16 right singular vectors from the same planes
// costs 4 B per element instead of re-reading D, S and Y (12 B) inside the shrink kernel, and lets that kernel stream
// every tile once instead of twice.
//
// One warp owns a k16 block (16 pixels x all frames = 64 n contiguous bytes per plane) at a time: lane 0 fetches the four
// plane runs with 1-D bulk copies (cp.async.bulk, mbarrier complete_tx) into the warp's own double-buffered slot, the
// lanes split the block as (frame mod 8) x (4-pixel word), rebuild the 32-bit integers with byte permutes, accumulate
// r x 4 partial sums in registers and reduce over the 8 frame lanes with shuffles.  Output: T in pixel order ([k][ld], for
// the final materialisation of L) and regrouped per tile and 3x3 group ([tile][k][group][12]) for the shrink kernel.
// HBM traffic: 4 B per matrix element read (+ r/n of that written).
#include <algorithm>
#include "common.cuh"
#include "kernels.h"
#include "tma.cuh"

namespace bsub {

constexpr int PJ_MAXW = 12;

struct ProjectArgs {
    const signed char* Wq; long long ldq; int n;
    const float* Vr; int vstride;
    float* T; long long ld;
    float* Tt;
    int rows, cols, R, ntile_r; long long ntiles;
    const DevState* st;
    int kcap, NW, DEPTH, slot_bytes;
};

__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

template <int KC>
__device__ __forceinline__ void pj_unit(const ProjectArgs& a, const unsigned char* slot, const float* Vs, long long unit, int r, float sc, int lane) {
    const int n = a.n, f8 = lane >> 2, quad = lane & 3;
    float acc[KC][4];
#pragma unroll
    for (int k = 0; k < KC; ++k) { acc[k][0] = acc[k][1] = acc[k][2] = acc[k][3] = 0.f; }
    const size_t pstride = (size_t)n * 16;
    auto one_frame = [&](int f, unsigned int a0, unsigned int a1, unsigned int a2, unsigned int a3) {
        // 4 x 4 byte transpose: word i of the result holds the four digits of pixel i (digit k = byte k)
        const unsigned int t0 = __byte_perm(a0, a1, 0x5140), t1 = __byte_perm(a2, a3, 0x5140);
        const unsigned int t2 = __byte_perm(a0, a1, 0x7362), t3 = __byte_perm(a2, a3, 0x7362);
        const unsigned int u0 = __byte_perm(t0, t1, 0x5410), u1 = __byte_perm(t0, t1, 0x7632);
        const unsigned int u2 = __byte_perm(t2, t3, 0x5410), u3 = __byte_perm(t2, t3, 0x7632);
        // inverse of the balanced-digit encoding u = (q + 0x808080) ^ 0x808080 of shrink_stream.cu
        float q[4];
        q[0] = (float)(int)((u0 ^ 0x00808080u) - 0x00808080u);
        q[1] = (float)(int)((u1 ^ 0x00808080u) - 0x00808080u);
        q[2] = (float)(int)((u2 ^ 0x00808080u) - 0x00808080u);
        q[3] = (float)(int)((u3 ^ 0x00808080u) - 0x00808080u);
        const float4* vrow = reinterpret_cast<const float4*>(Vs + (size_t)f * 16);
#pragma unroll
        for (int k4 = 0; k4 < (KC + 3) / 4; ++k4) {
            const float4 v = vrow[k4];
            const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const int k = 4 * k4 + kk;
                if (k < KC) {
                    acc[k][0] = fmaf(vv[kk], q[0], acc[k][0]); acc[k][1] = fmaf(vv[kk], q[1], acc[k][1]);
                    acc[k][2] = fmaf(vv[kk], q[2], acc[k][2]); acc[k][3] = fmaf(vv[kk], q[3], acc[k][3]);
                }
            }
        }
    };
    int f = f8;
    for (; f + 8 < n; f += 16) {                       // two frames per trip: eight independent loads in flight
        const unsigned char* p = slot + (size_t)f * 16 + quad * 4;
        const unsigned int a0 = *reinterpret_cast<const unsigned int*>(p), b0 = *reinterpret_cast<const unsigned int*>(p + 128);
        const unsigned int a1 = *reinterpret_cast<const unsigned int*>(p + pstride), b1 = *reinterpret_cast<const unsigned int*>(p + pstride + 128);
        const unsigned int a2 = *reinterpret_cast<const unsigned int*>(p + 2 * pstride), b2 = *reinterpret_cast<const unsigned int*>(p + 2 * pstride + 128);
        const unsigned int a3 = *reinterpret_cast<const unsigned int*>(p + 3 * pstride), b3 = *reinterpret_cast<const unsigned int*>(p + 3 * pstride + 128);
        one_frame(f, a0, a1, a2, a3);
        one_frame(f + 8, b0, b1, b2, b3);
    }
    if (f < n) {
        const unsigned char* p = slot + (size_t)f * 16 + quad * 4;
        one_frame(f, *reinterpret_cast<const unsigned int*>(p), *reinterpret_cast<const unsigned int*>(p + pstride),
                  *reinterpret_cast<const unsigned int*>(p + 2 * pstride), *reinterpret_cast<const unsigned int*>(p + 3 * pstride));
    }
#pragma unroll
    for (int k = 0; k < KC; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float v = acc[k][i];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            acc[k][i] = v * sc;
        }
    // every lane holds the totals of its 4 pixels (xor butterfly); the ranks are spread over the 8 frame lanes for the stores.
    // Pixel order inside a tile (shrink_stream.cu / shrink_flat.cu): position = e * NG + g for entry e = 3 c + dr of the 3x3
    // group g, so a k16 block holds 16 consecutive groups of one entry.
    const int NG = a.R / 3, bpt = (3 * a.R) / 16;               // groups per tile, k16 blocks per tile
    const long long tl = unit / bpt;
    const int kb = (int)(unit - tl * bpt);
    if (tl >= a.ntiles) return;
    const int pos0 = 16 * kb + 4 * quad;                        // 4 consecutive positions: same entry (NG % 4 == 0), groups g0 .. g0+3
    const int e = pos0 / NG, g0 = pos0 - e * NG, c = e / 3, dr = e - 3 * c;
    const int tcx = (int)(tl / a.ntile_r), trx = (int)(tl - (long long)tcx * a.ntile_r);
    const int j = 3 * tcx + c, row0 = trx * a.R + 3 * g0 + dr;
    float* tt = a.Tt + (size_t)tl * 16 * (4 * a.R);
#pragma unroll
    for (int k = 0; k < KC; ++k) {
        if ((k & 7) == f8 && k < r) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                tt[(size_t)k * (4 * a.R) + (g0 + i) * 12 + e] = acc[k][i];
                const int row = row0 + 3 * i;
                if (j < a.cols && row < a.rows) a.T[(size_t)k * a.ld + (long long)j * a.rows + row] = acc[k][i];
            }
        }
    }
}

__global__ void __launch_bounds__(32 * PJ_MAXW, 1) project_planes_kernel(ProjectArgs a) {
    const DevState* st = a.st;
    if (st->done || st->gram_mode != 1) return;            // no valid planes of this iteration's W: the shrink kernel projects itself
    const int r = st->svp;
    if (r <= 0 || r > a.kcap) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n = a.n;
    extern __shared__ __align__(128) unsigned char pj_smem[];
    float* Vs = reinterpret_cast<float*>(pj_smem);                                   // [n][16]
    unsigned char* slots = pj_smem + (((size_t)n * 16 * sizeof(float) + 127) & ~(size_t)127);
    __shared__ uint64_t full[PJ_MAXW * 2];
    if (threadIdx.x == 0) {
        for (int i = 0; i < a.NW * a.DEPTH; ++i) mbar_init(&full[i], 1);
        mbar_fence_init();
    }
    for (int idx = threadIdx.x; idx < n * 16; idx += blockDim.x) {
        const int f = idx >> 4, k = idx & 15;
        Vs[idx] = (k < r) ? a.Vr[(size_t)f * a.vstride + k] : 0.f;
    }
    __syncthreads();
    if (warp >= a.NW) return;
    const float sc = (float)(st->wq_scale * (1.0 / 2147483648.0));
    const long long nunits = a.ldq / 16;
    const long long stride = (long long)gridDim.x * a.NW;
    const long long u0 = (long long)blockIdx.x * a.NW + warp;
    const size_t plane = (size_t)a.ldq * n;
    const uint32_t run = (uint32_t)n * 16;
    unsigned char* myslots = slots + (size_t)warp * a.DEPTH * a.slot_bytes;
    uint64_t* mybar = &full[warp * a.DEPTH];
    auto issue = [&](long long u, int d) {
        if (lane == 0) {
            mbar_expect_tx(&mybar[d], 4 * run);
            unsigned char* dst = myslots + (size_t)d * a.slot_bytes;
#pragma unroll
            for (int pl = 0; pl < 4; ++pl)
                bulk_load_1d(dst + (size_t)pl * run, a.Wq + (size_t)pl * plane + (size_t)u * run, run, &mybar[d]);
        }
    };
    for (int d = 0; d < a.DEPTH; ++d) if (u0 + d * stride < nunits) issue(u0 + d * stride, d);
    long long it = 0;
    for (long long u = u0; u < nunits; u += stride, ++it) {
        const int d = (int)(it % a.DEPTH);
        mbar_wait(&mybar[d], (uint32_t)((it / a.DEPTH) & 1));
        const unsigned char* slot = myslots + (size_t)d * a.slot_bytes;
        if (r <= 2) pj_unit<2>(a, slot, Vs, u, r, sc, lane);
        else if (r <= 4) pj_unit<4>(a, slot, Vs, u, r, sc, lane);
        else if (r == 5) pj_unit<5>(a, slot, Vs, u, r, sc, lane);
        else if (r == 6) pj_unit<6>(a, slot, Vs, u, r, sc, lane);
        else if (r <= 8) pj_unit<8>(a, slot, Vs, u, r, sc, lane);
        else if (r <= 12) pj_unit<12>(a, slot, Vs, u, r, sc, lane);
        else pj_unit<16>(a, slot, Vs, u, r, sc, lane);
        __syncwarp();                                      // every lane is done with the slot before it is refilled
        const long long un = u + (long long)a.DEPTH * stride;
        if (un < nunits) issue(un, d);
    }
}

bool make_project_plan(int n, int R, long long ldq, int num_sms, ProjectPlan* out) {
    if (R % 48 != 0 || ldq <= 0) return false;          // whole k16 blocks per entry: (R / 3) % 16 == 0
    ProjectPlan p;
    p.n = n; p.ldq = ldq;
    p.slot_bytes = 64 * n;
    const size_t vs = (((size_t)n * 16 * sizeof(float)) + 127) & ~(size_t)127;
    const size_t cap = 225 * 1024;
    if (vs + (size_t)p.slot_bytes > cap) return false;
    const int nslots = (int)((cap - vs) / p.slot_bytes);
    // the per-block arithmetic (~2400 warp instructions for n = 300) outweighs the load: many warps with one slot each beat few
    // warps with a prefetch slot; two slots per warp only when shared memory holds them for a full set of warps
    if (nslots >= 2 * PJ_MAXW) { p.DEPTH = 2; p.NW = PJ_MAXW; }
    else { p.DEPTH = 1; p.NW = std::min(PJ_MAXW, nslots); }
    p.smem_bytes = vs + (size_t)p.NW * p.DEPTH * p.slot_bytes;
    const long long nunits = ldq / 16;
    p.grid = (int)std::max<long long>(1, std::min<long long>(num_sms, (nunits + p.NW - 1) / p.NW));
    *out = p;
    return true;
}

int launch_project(const ProjectPlan& p, const signed char* Wq, const float* Vr, int vstride, float* T, long long ld, float* Tt, int rows,
                   int cols, int R, int ntile_r, long long ntiles, int kcap, const DevState* st, cudaStream_t stream) {
    static unsigned long long attr_devs = 0;
    if (first_call_on_device(&attr_devs))
        BSUB_CUDA_CHECK(cudaFuncSetAttribute(project_planes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
    ProjectArgs a;
    a.Wq = Wq; a.ldq = p.ldq; a.n = p.n; a.Vr = Vr; a.vstride = vstride; a.T = T; a.ld = ld; a.Tt = Tt; a.rows = rows; a.cols = cols;
    a.R = R; a.ntile_r = ntile_r; a.ntiles = ntiles; a.st = st; a.kcap = kcap; a.NW = p.NW; a.DEPTH = p.DEPTH; a.slot_bytes = p.slot_bytes;
    project_planes_kernel<<<p.grid, 32 * PJ_MAXW, p.smem_bytes, stream>>>(a);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

}  // namespace bsub
