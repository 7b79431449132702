// gram.cu -- pass A of the ALM iteration: G = W W^T (frames x frames) with
//   W = D - S + Y/mu   formed on the fly in fp32   (/root/reference/inexact_alm_lsd.py:131)
// accumulated in fp64 on the FP64 tensor pipe (DMMA m8n8k4), which is what the Gram-route
// singular-value thresholding needs (SURVEY H1: the small eigenvalues near (1/mu)^2 sit ~1e-10
// below sigma_1^2, so products and sums must be fp64-grade).
//
// Work decomposition (DESIGN.md section 4.1):
//   * the symmetric output is cut into 32x32 "macro tiles" (bi <= bj); one warp owns one macro tile
//     = 4x4 DMMA blocks = 32 fp64 accumulators per thread;
//   * a CTA has 14 MMA warps (14 macro tiles); ceil(ntasks/14) CTA "types" cover the whole upper triangle,
//     CTAs of different type that share a k-slot walk the same pixel chunks at the same time so the
//     re-reads hit L2;
//   * the raw D, S, Y chunks ([frames][kc pixels]) are brought in by TMA (cp.async.bulk.tensor.2d, frames
//     beyond n zero-filled by the hardware) one whole chunk ahead of the math: ncu r1a showed that two
//     producer warps with plain loads could not keep the DMMA pipe fed (35 % active);
//   * all 16 warps combine raw -> W (fp32, padded rows) between two chunks; fragments are widened to fp64 at
//     load time;
//   * K (= pixels) is split across k-slots; every CTA writes its partial tile to a scratch buffer and a
//     second kernel sums the k-slots in a fixed order (deterministic, no atomics).
#include "common.cuh"
#include "kernels.h"
#include "tma.cuh"

namespace bsub {

constexpr int GR_MMA_WARPS = 14;
constexpr int GR_THREADS = 512;
constexpr size_t GR_SMEM_CAP = 227 * 1024 - 256;

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

struct GramArgs {
    int n, npad, ntasks, ntype, gridK, narr, kc, nbox, boxrows;
    long long nchunks;                                  // ld / kc
    const int2* tasks;                                  // (bi, bj), bi <= bj
    const DevState* st;                                 // may be nullptr (stand-alone use)
    float inv_mu_override;                              // used when st == nullptr
    double* partial;                                    // [gridK][ntasks][32*32]
};

__global__ void __launch_bounds__(GR_THREADS, 1)
gram_dmma_kernel(const __grid_constant__ CUtensorMap mapD, const __grid_constant__ CUtensorMap mapS,
                 const __grid_constant__ CUtensorMap mapY, GramArgs a) {
    if (a.st != nullptr && (a.st->done || a.st->gram_mode != 0)) return;      // gram_mode 1: gram_i8.cu does this iteration
    extern __shared__ __align__(128) unsigned char gram_smem_raw[];
    const int kc = a.kc, lds = kc + 4;
    const int rawrows = a.nbox * a.boxrows;
    float* raw = reinterpret_cast<float*>(gram_smem_raw);                       // [3][rawrows][kc]
    float* wt = raw + (size_t)3 * rawrows * kc;                                 // [2][npad][lds]
    uint64_t* bar = reinterpret_cast<uint64_t*>(wt + (size_t)2 * a.npad * lds); // full barrier

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int type = blockIdx.x % a.ntype;
    const int kslot = blockIdx.x / a.ntype;
    const int task = type * GR_MMA_WARPS + warp;
    const bool has_task = warp < GR_MMA_WARPS && task < a.ntasks;
    int bi = 0, bj = 0;
    if (has_task) { int2 t = a.tasks[task]; bi = t.x; bj = t.y; }
    const bool diag = (bi == bj);
    float inv_mu = 0.f;
    if (a.narr == 3) inv_mu = (a.st != nullptr) ? (float)(1.0 / a.st->mu) : a.inv_mu_override;

    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

    long long niter = 0;
    if (kslot < a.nchunks) niter = (a.nchunks - kslot + a.gridK - 1) / a.gridK;

    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
        tma_prefetch_desc(&mapD);
        if (a.narr == 3) { tma_prefetch_desc(&mapS); tma_prefetch_desc(&mapY); }
    }
    __syncthreads();

    const uint32_t tx_bytes = (uint32_t)(a.narr * rawrows * kc * sizeof(float));
    auto issue = [&](long long chunk) {        // one elected thread
        mbar_expect_tx(bar, tx_bytes);
        const int x = (int)(chunk * kc);
        for (int b = 0; b < a.nbox; ++b) {
            tma_load_2d(raw + (size_t)(0 * rawrows + b * a.boxrows) * kc, &mapD, bar, x, b * a.boxrows);
            if (a.narr == 3) {
                tma_load_2d(raw + (size_t)(1 * rawrows + b * a.boxrows) * kc, &mapS, bar, x, b * a.boxrows);
                tma_load_2d(raw + (size_t)(2 * rawrows + b * a.boxrows) * kc, &mapY, bar, x, b * a.boxrows);
            }
        }
    };
    const int qpr = kc >> 2;
    auto combine = [&](float* dst) {           // all threads: W = (D - S) + Y/mu, rows >= n are zero (TMA OOB fill)
        const float* rd = raw;
        const float* rs = raw + (size_t)rawrows * kc;
        const float* ry = raw + (size_t)2 * rawrows * kc;
        for (int idx = threadIdx.x; idx < a.npad * qpr; idx += GR_THREADS) {
            const int row = idx / qpr, q = idx - row * qpr;
            const float4 d = *reinterpret_cast<const float4*>(rd + (size_t)row * kc + 4 * q);
            float4 w = d;
            if (a.narr == 3) {
                const float4 s = *reinterpret_cast<const float4*>(rs + (size_t)row * kc + 4 * q);
                const float4 y = *reinterpret_cast<const float4*>(ry + (size_t)row * kc + 4 * q);
                // same fp32 expression as the shrink pass so that both passes see the same W
                w.x = (d.x - s.x) + y.x * inv_mu; w.y = (d.y - s.y) + y.y * inv_mu;
                w.z = (d.z - s.z) + y.z * inv_mu; w.w = (d.w - s.w) + y.w * inv_mu;
            }
            *reinterpret_cast<float4*>(dst + (size_t)row * lds + 4 * q) = w;
        }
    };

    if (niter > 0) {
        if (threadIdx.x == 0) issue(kslot);
        mbar_wait(bar, 0);
        combine(wt);
        __syncthreads();
        if (niter > 1 && threadIdx.x == 0) issue(kslot + a.gridK);
    }
    const int fr = lane >> 2, fc = lane & 3;
    const int nks = kc >> 2, rs8 = 8 * lds;
    for (long long it = 0; it < niter; ++it) {
        const int cur = (int)(it & 1);
        if (has_task) {
            const float* wb = wt + (size_t)cur * a.npad * lds;
            const float* rowA = wb + (size_t)(bi * 32 + fr) * lds + fc;
            const float* rowB = wb + (size_t)(bj * 32 + fr) * lds + fc;
#pragma unroll 2
            for (int ks = 0; ks < nks; ++ks) {
                double af[4], bf[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    af[i] = (double)rowA[i * rs8 + ks * 4];
                    bf[i] = (double)rowB[i * rs8 + ks * 4];
                }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (!diag || i <= j) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
            }
        }
        if (it + 1 < niter) {
            mbar_wait(bar, (uint32_t)((it + 1) & 1));              // chunk it+1 has landed in raw
            combine(wt + (size_t)(cur ^ 1) * a.npad * lds);        // wt[cur^1] was last read in iteration it-1
            __syncthreads();                                       // raw is free, wt[cur^1] is complete
            if (it + 2 < niter && threadIdx.x == 0) issue(kslot + (it + 2) * a.gridK);
        }
    }
    if (has_task) {
        double* out = a.partial + ((size_t)kslot * a.ntasks + task) * 1024;
        const int row = lane >> 2, col = 2 * (lane & 3);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                double2 v = make_double2(acc[i][j][0], acc[i][j][1]);
                *reinterpret_cast<double2*>(out + (i * 8 + row) * 32 + j * 8 + col) = v;
            }
    }
}

// Sum the k-slot partials in a fixed order and scatter the symmetric result into G[npad][npad].
__global__ void gram_reduce_kernel(const double* __restrict__ partial, const int2* __restrict__ tasks, int ntasks,
                                   int gridK, int npad, double* __restrict__ G, const DevState* st) {
    if (st != nullptr && (st->done || st->gram_mode != 0)) return;
    const int task = blockIdx.x;
    const int2 t = tasks[task];
    for (int e = threadIdx.x; e < 1024; e += blockDim.x) {
        const int r = e >> 5, c = e & 31;
        if (t.x == t.y && r > c) continue;
        double s = 0.0;
        for (int k = 0; k < gridK; ++k) s += partial[((size_t)k * ntasks + task) * 1024 + e];
        const int i = t.x * 32 + r, j = t.y * 32 + c;
        G[(size_t)i * npad + j] = s;
        G[(size_t)j * npad + i] = s;
    }
}

// ---------------------------------------------------------------------------------------------------------
static size_t gram_smem_bytes(int npad, int kc, int nbox, int boxrows) {
    return (size_t)3 * nbox * boxrows * kc * sizeof(float) + (size_t)2 * npad * (kc + 4) * sizeof(float) + 16;
}

GramPlan make_gram_plan(int n, long long ld, int num_sms) {
    GramPlan p;
    p.n = n;
    p.npad = ((n + 31) / 32) * 32;
    p.nb = p.npad / 32;
    p.ntasks = p.nb * (p.nb + 1) / 2;
    p.ntype = (p.ntasks + GR_MMA_WARPS - 1) / GR_MMA_WARPS;
    p.nbox = (p.npad + 255) / 256;
    p.boxrows = (((p.npad + p.nbox - 1) / p.nbox) + 7) / 8 * 8;
    p.kc = 32;
    while (p.kc > 8 && gram_smem_bytes(p.npad, p.kc, p.nbox, p.boxrows) > GR_SMEM_CAP) p.kc >>= 1;
    p.nchunks = ld / p.kc;
    long long gk = num_sms / p.ntype;
    if (gk < 1) gk = 1;
    if (gk > p.nchunks) gk = p.nchunks;
    if (gk < 1) gk = 1;
    p.gridK = (int)gk;
    p.smem_bytes = gram_smem_bytes(p.npad, p.kc, p.nbox, p.boxrows);
    p.partial_elems = (size_t)p.gridK * p.ntasks * 1024;
    return p;
}

void fill_gram_tasks(const GramPlan& p, int2* host_tasks) {
    int t = 0;
    for (int bi = 0; bi < p.nb; ++bi)
        for (int bj = bi; bj < p.nb; ++bj) host_tasks[t++] = make_int2(bi, bj);
}

int make_gram_maps(const GramPlan& p, const float* D, const float* S, const float* Y, long long ld, GramMaps* maps) {
    const uint64_t dims[2] = {(uint64_t)ld, (uint64_t)p.n};
    const uint64_t strides[1] = {(uint64_t)ld * sizeof(float)};
    const uint32_t box[2] = {(uint32_t)p.kc, (uint32_t)p.boxrows};
    if (make_tensor_map_f32(&maps->D, D, 2, dims, strides, box) != 0) return -1;
    maps->narr = 1;
    if (S != nullptr && Y != nullptr) {
        if (make_tensor_map_f32(&maps->S, S, 2, dims, strides, box) != 0) return -1;
        if (make_tensor_map_f32(&maps->Y, Y, 2, dims, strides, box) != 0) return -1;
        maps->narr = 3;
    } else {
        maps->S = maps->D; maps->Y = maps->D;
    }
    return 0;
}

int launch_gram(const GramPlan& p, const GramMaps& maps, bool combo, const int2* dev_tasks, const DevState* st,
                float inv_mu_override, double* partial, double* G, cudaStream_t stream) {
    static unsigned long long attr_devs = 0;      // one bit per device: the attribute is per (function, device)
    if (first_call_on_device(&attr_devs)) {
        BSUB_CUDA_CHECK(cudaFuncSetAttribute(gram_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GR_SMEM_CAP));
    }
    if (p.smem_bytes > GR_SMEM_CAP) { set_error("gram: n=%d too large for the shared-memory tiles", p.n); return -1; }
    if (combo && maps.narr != 3) { set_error("gram: S/Y tensor maps missing"); return -1; }
    GramArgs a;
    a.n = p.n; a.npad = p.npad; a.ntasks = p.ntasks; a.ntype = p.ntype; a.gridK = p.gridK; a.narr = combo ? 3 : 1;
    a.kc = p.kc; a.nbox = p.nbox; a.boxrows = p.boxrows; a.nchunks = p.nchunks; a.tasks = dev_tasks; a.st = st;
    a.inv_mu_override = inv_mu_override; a.partial = partial;
    gram_dmma_kernel<<<p.gridK * p.ntype, GR_THREADS, p.smem_bytes, stream>>>(maps.D, maps.S, maps.Y, a);
    BSUB_CUDA_CHECK(cudaGetLastError());
    gram_reduce_kernel<<<p.ntasks, 256, 0, stream>>>(partial, dev_tasks, p.ntasks, p.gridK, p.npad, G, st);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------
// tensor-map creation through the driver entry point
typedef CUresult (*PFN_tmap_encode)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_tensor_map_any(CUtensorMap* map, const void* base, CUtensorMapDataType dtype, int rank, const uint64_t* dims,
                               const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swz);

int make_tensor_map_f32(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                        const uint32_t* box) {
    return make_tensor_map_any(map, base, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, rank, dims, strides_bytes, box, CU_TENSOR_MAP_SWIZZLE_NONE);
}

int make_tensor_map_u64(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                        const uint32_t* box) {
    return make_tensor_map_any(map, base, CU_TENSOR_MAP_DATA_TYPE_UINT64, rank, dims, strides_bytes, box, CU_TENSOR_MAP_SWIZZLE_NONE);
}

int make_tensor_map_u8(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                       const uint32_t* box, int swizzle_bytes) {
    const CUtensorMapSwizzle swz = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B :
                                   swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
    return make_tensor_map_any(map, base, CU_TENSOR_MAP_DATA_TYPE_UINT8, rank, dims, strides_bytes, box, swz);
}

static int make_tensor_map_any(CUtensorMap* map, const void* base, CUtensorMapDataType dtype, int rank, const uint64_t* dims,
                               const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swz) {
    static PFN_tmap_encode fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
        if (e != cudaSuccess || p == nullptr || qres != cudaDriverEntryPointSuccess) {
            set_error("cuTensorMapEncodeTiled is not available from this driver (%s)", cudaGetErrorString(e));
            return -1;
        }
        fn = reinterpret_cast<PFN_tmap_encode>(p);
    }
    cuuint64_t gdim[5]; cuuint64_t gstr[4]; cuuint32_t bx[5]; cuuint32_t es[5];
    for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
    CUresult r = fn(map, dtype, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d): rank %d dims %llu,%llu,%llu box %u,%u,%u", (int)r, rank,
                  (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0), (unsigned long long)(rank > 2 ? dims[2] : 0),
                  box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0);
        return -1;
    }
    return 0;
}

}  // namespace bsub
