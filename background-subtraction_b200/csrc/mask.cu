// mask.cu -- foreground_mask (/root/reference/utils.py:139-149):
//   A = |S| ; M = max A ; B = A < 0.5 M ; Delta = |D - L| * B ; over Delta > 0: mean and POPULATION std ;
//   th = mean + k std ; mask = A > th          (strict comparisons, global statistics -- SURVEY Q15)
// Three streaming passes (max; count/sum/sum^2 in fp64; threshold + write).  The statistics buffers are plain
// device memory so that a pixel-sharded run can all-reduce them between the passes.
#include "common.cuh"
#include "kernels.h"

namespace bsub {

constexpr int MK_THREADS = 256;

static inline int mk_grid(long long work4) {
    long long g = (work4 + MK_THREADS * 4 - 1) / (MK_THREADS * 4);
    if (g < 1) g = 1;
    if (g > 148 * 8) g = 148 * 8;
    return (int)g;
}

__global__ void absmax_kernel(const float* __restrict__ S, long long total4, double* out_max) {
    __shared__ double red[32];
    float mx = 0.f;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total4; q += (long long)gridDim.x * blockDim.x) {
        const float4 s = ldg4_stream(S + 4 * q);
        mx = fmaxf(mx, fmaxf(fmaxf(fabsf(s.x), fabsf(s.y)), fmaxf(fabsf(s.z), fabsf(s.w))));
    }
    double m = block_max((double)mx, red);
    if (threadIdx.x == 0) atomicMax(reinterpret_cast<unsigned long long*>(out_max), (unsigned long long)__double_as_longlong(m));
}

// out_max (double, non-negative, ordered like its bit pattern) must be zero on entry
int launch_absmax(const float* S, long long ld, long long m, int n, double* out_max, cudaStream_t s) {
    (void)m;
    const long long total4 = ld * n / 4;   // pad columns are zero
    absmax_kernel<<<mk_grid(total4), MK_THREADS, 0, s>>>(S, total4, out_max);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// Statistics in a fixed order (bit-reproducible threshold): every CTA writes its three fp64 partials, the last CTA to
// finish (ticket counter) adds them up in CTA order and stores stats[0..2].  scratch: [3 * grid] doubles + one counter.
__global__ void mask_stats_kernel(const float* __restrict__ D, const float* __restrict__ L, const float* __restrict__ S,
                                  long long total4, const double* absmax, double* stats, double* scratch) {
    __shared__ double red[32];
    __shared__ int is_last;
    const float half_m = 0.5f * (float)absmax[0];
    double cnt = 0.0, sum = 0.0, sq = 0.0;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total4; q += (long long)gridDim.x * blockDim.x) {
        const float4 d = ldg4_stream(D + 4 * q), l = ldg4_stream(L + 4 * q), s = ldg4_stream(S + 4 * q);
        const float dv[4] = {d.x, d.y, d.z, d.w}, lv[4] = {l.x, l.y, l.z, l.w}, sv[4] = {s.x, s.y, s.z, s.w};
        float c4 = 0.f; double s4 = 0.0, q4 = 0.0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float dl = fabsf(dv[e] - lv[e]);
            if (fabsf(sv[e]) < half_m && dl > 0.f) { c4 += 1.f; s4 += (double)dl; q4 += (double)dl * (double)dl; }
        }
        cnt += (double)c4; sum += s4; sq += q4;
    }
    unsigned int* ticket = reinterpret_cast<unsigned int*>(scratch + 3 * (size_t)gridDim.x);
    double a = block_sum(cnt, red);
    if (threadIdx.x == 0) scratch[3 * (size_t)blockIdx.x + 0] = a;
    double b = block_sum(sum, red);
    if (threadIdx.x == 0) scratch[3 * (size_t)blockIdx.x + 1] = b;
    double c = block_sum(sq, red);
    if (threadIdx.x == 0) {
        scratch[3 * (size_t)blockIdx.x + 2] = c;
        __threadfence();
        is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1 : 0;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    double t0 = 0.0, t1 = 0.0, t2 = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
        t0 += __ldcg(scratch + 3 * (size_t)i); t1 += __ldcg(scratch + 3 * (size_t)i + 1); t2 += __ldcg(scratch + 3 * (size_t)i + 2);
    }
    t0 = block_sum(t0, red);
    if (threadIdx.x == 0) stats[0] = t0;
    t1 = block_sum(t1, red);
    if (threadIdx.x == 0) stats[1] = t1;
    t2 = block_sum(t2, red);
    if (threadIdx.x == 0) { stats[2] = t2; *ticket = 0u; }
}

size_t mask_stats_scratch_doubles() { return (size_t)3 * 148 * 8 + 2; }

int launch_mask_stats(const float* D, const float* L, const float* S, long long ld, long long m, int n, const double* absmax,
                      double* stats, double* scratch, cudaStream_t s) {
    (void)m;
    const long long total4 = ld * n / 4;   // pad columns: D = L = 0 -> Delta = 0 -> excluded
    mask_stats_kernel<<<mk_grid(total4), MK_THREADS, 0, s>>>(D, L, S, total4, absmax, stats, scratch);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

__global__ void mask_write_kernel(const float* __restrict__ S, long long ld, long long m, int n, const double* stats,
                                  double sigmas, unsigned char* __restrict__ mask, long long mask_ld) {
    const double cnt = stats[0];
    double th;
    if (cnt > 0.0) {
        const double mean = stats[1] / cnt;
        double var = stats[2] / cnt - mean * mean;
        if (var < 0.0) var = 0.0;
        th = mean + sigmas * sqrt(var);
    } else {
        th = nan("");                       // np.mean of an empty selection is nan -> mask all False
    }
    if (((m | mask_ld) & 3) == 0 && (reinterpret_cast<uintptr_t>(mask) & 3) == 0) {
        // four pixels per thread: 16-byte loads, 4-byte stores (same comparison in double as the scalar path)
        const long long m4 = m / 4;
        for (int f = blockIdx.y; f < n; f += gridDim.y)
            for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < m4; q += (long long)gridDim.x * blockDim.x) {
                const float4 v = ldg4_stream(S + (size_t)f * ld + 4 * q);
                uchar4 o;
                o.x = ((double)fabsf(v.x) > th) ? 1 : 0; o.y = ((double)fabsf(v.y) > th) ? 1 : 0;
                o.z = ((double)fabsf(v.z) > th) ? 1 : 0; o.w = ((double)fabsf(v.w) > th) ? 1 : 0;
                *reinterpret_cast<uchar4*>(mask + (size_t)f * mask_ld + 4 * q) = o;
            }
        return;
    }
    for (int f = blockIdx.y; f < n; f += gridDim.y)
        for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (long long)gridDim.x * blockDim.x)
            mask[(size_t)f * mask_ld + p] = ((double)fabsf(S[(size_t)f * ld + p]) > th) ? 1 : 0;
}

// max |S| of a finished solve is already known on the device (control_post keeps the last iteration's value)
__global__ void maxS_from_state_kernel(const DevState* st, double* out_max) {
    if (threadIdx.x == 0 && blockIdx.x == 0) *out_max = (double)st->maxS;
}
int launch_maxS_from_state(const DevState* st, double* out_max, cudaStream_t s) {
    maxS_from_state_kernel<<<1, 32, 0, s>>>(st, out_max);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_mask_write(const float* S, long long ld, long long m, int n, const double* stats, double sigmas, unsigned char* mask,
                      long long mask_ld, cudaStream_t s) {
    long long gx = (m + MK_THREADS * 4 - 1) / (MK_THREADS * 4);
    if (gx < 1) gx = 1;
    if (gx > 1024) gx = 1024;
    dim3 g((unsigned)gx, n < 512 ? n : 512);
    mask_write_kernel<<<g, MK_THREADS, 0, s>>>(S, ld, m, n, stats, sigmas, mask, mask_ld);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// LSD_improved's weight map -> centre-window description: eta = the positive entries (0 elsewhere), label 0 where the entry is
// negative (background) and 255 elsewhere; the flat index f * m + p of the first non-finite entry goes to *first_bad (atomicMin)
__global__ void weight_map_describe_kernel(const float* __restrict__ w, long long ld, long long m, int nf, float* __restrict__ eta,
                                           unsigned char* __restrict__ labels, unsigned long long* first_bad) {
    for (int f = blockIdx.y; f < nf; f += gridDim.y)
        for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (long long)gridDim.x * blockDim.x) {
            const float v = w[(size_t)f * ld + p];
            const size_t i = (size_t)f * m + p;
            if (!isfinite(v)) atomicMin(first_bad, (unsigned long long)i);
            eta[i] = v > 0.f ? v : 0.f;
            labels[i] = v < 0.f ? 0 : 255;
        }
}

int launch_weight_map_describe(const float* w, long long ld, long long m, int nf, float* eta, unsigned char* labels,
                               unsigned long long* first_bad, cudaStream_t s) {
    long long gx = (m + MK_THREADS - 1) / MK_THREADS;
    if (gx < 1) gx = 1;
    if (gx > 1024) gx = 1024;
    dim3 g((unsigned)gx, nf < 512 ? nf : 512);
    weight_map_describe_kernel<<<g, MK_THREADS, 0, s>>>(w, ld, m, nf, eta, labels, first_bad);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

}  // namespace bsub
