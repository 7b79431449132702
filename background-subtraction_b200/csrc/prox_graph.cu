// prox_graph.cu -- spams.proximalGraph 'graph' for an ARBITRARY non-nested group structure (/root/reference/inexact_alm_lsd.py:49-68):
// per frame f,  argmin_v 1/2 ||u - v||^2 + lam sum_g eta_g ||v_g||_inf  with the groups g given as a SPAMS-style CSC
// (indptr, indices, eta) -- any window shape, the centre windows of any radius, irregular groups of any size and overlap, and a
// different graph for every frame.
//
// Same dual block-coordinate descent as the oracle (oracle/prox_oracle.c:prox_graph_linf) and the 3x3 tile kernel (prox.cu):
// xi_g <- Proj_{l1-ball(lam eta_g)}(u - tot + xi_g), tot = sum of the duals on each pixel, v = u - tot.  The sweep order is free
// (every order converges to the same unique primal solution), so the host colours each graph greedily (two groups conflict when
// they share a pixel) and stores its groups colour-major: one colour is a set of disjoint groups that update in parallel without
// atomics.
//
// Frames are independent: a thread-block cluster takes one frame at a time from a work counter, sweeps it to its own stop test
// and takes the next one -- there is no grid-wide barrier (DESIGN.md 4.6 on why a barrier per colour is unusable).  The per-pixel
// dual sums `tot` of the frame live in the distributed shared memory of the cluster (pixel p in CTA p >> shift, slot p & mask);
// the cluster is the smallest power of two <= 8 whose shared memory holds the frame, enlarged while the frames alone would not
// fill the GPU.  Larger frames keep `tot` in global memory (one row per cluster).  u is read through the read-only path, the
// duals live in global memory in the graph's nnz order (one slot of max_nnz floats per cluster in flight: the workspace cap
// bounds the number of clusters, not the frame count).
//
// Projection: Michelot's finite active-set iteration (the active set shrinks monotonically and the clip level is the closed form
// (sum_active - z) / |active| of the final set, exact to fp32 rounding for every group size).  Groups of <= PG_SMALL pixels take
// one thread each (no local arrays: the operands are re-read from shared memory on each pass), larger ones one warp.
// fp32 hazards handled as in the tile kernel: the state is (xi, tot), not x = u - tot; a projection that moved by <= ~2 ulp of its
// operands keeps its dual, and a change counts towards the stop test only above PG_COUNT_FACTOR of those dead bands.
#include <cooperative_groups.h>
#include <math.h>
#include <stdlib.h>
#include <algorithm>
#include <vector>
#include "common.cuh"
#include "kernels.h"

namespace cg = cooperative_groups;

namespace bsub {

constexpr int PG_THREADS = 256;
constexpr int PG_SMALL = 32;                       // groups up to this size: one thread; larger: one warp
constexpr int PG_MAX_SHIFT = 15;                   // <= 32768 pixels (128 KB of tot) per CTA
constexpr float PG_BAND = 2.4e-7f;                 // ~2 ulp
constexpr float PG_COUNT_FACTOR = 8.f;             // dead bands a dual change must exceed to count towards the stop test

struct PgArgs {
    const float* U; float* V; long long ld; int m, n;
    float lam, tol; int max_sweeps; float count_factor;
    GenericGraphDev g;
    float* xi;                 // [clusters][max_nnz]
    float* totg;               // [clusters][ld] when tot does not fit the cluster's shared memory, else nullptr
    int shift;                 // pixels per CTA = 1 << shift (distributed mode)
    int* status;               // int[8]: [1] work counter, [3] largest sweep count of this call
    const DevState* st;
};

struct PgTot {
    float* s; float* g; int shift, cs;
    __device__ __forceinline__ float* at(const cg::cluster_group& cl, int p) const {
        if (g != nullptr) return g + p;
        if (cs == 1) return s + p;
        return cl.map_shared_rank(s + (p & ((1 << shift) - 1)), (unsigned)(p >> shift));
    }
};

// a / b for a count b >= 1: hardware reciprocal + one Newton step on the quotient (within an ulp of the rounded quotient; the
// IEEE division calls a slow-path subroutine that makes the kernel spill)
__device__ __forceinline__ float pg_div(float a, float b) {
    const float r = __fdividef(1.f, b), q = a * r;
    return fmaf(fmaf(-b, q, a), r, q);
}

__device__ __forceinline__ double pg_ddiv(double a, double b) {   // the same for lambda / mu (b > 0, normal)
    double r = (double)__fdividef(1.f, (float)b);
    r = fma(r, fma(-b, r, 1.0), r);
    r = fma(r, fma(-b, r, 1.0), r);
    const double q = a * r;
    return fma(fma(-b, q, a), r, q);
}

// one group, one thread.  Returns the dual change that counts towards the stop test.
__device__ __forceinline__ float pg_update_small(const cg::cluster_group& cl, const PgTot T, const float* __restrict__ u,
                                                 const int* __restrict__ idx, float* xi, int k, float z, float cf) {
    float sabs = 0.f, wscale = 0.f;
    for (int q = 0; q < k; ++q) {
        const int p = __ldg(idx + q);
        const float uu = __ldg(u + p), tt = *T.at(cl, p), x0 = xi[q];
        const float r = uu - tt + x0;
        sabs += fabsf(r);
        wscale = fmaxf(wscale, fmaxf(fabsf(uu), fmaxf(fabsf(x0), fabsf(tt))));
    }
    float theta = 0.f;
    if (!(z > 0.f)) theta = INFINITY;                              // radius 0: the dual is 0
    else if (sabs > z) {
        theta = pg_div(sabs - z, (float)k);
        for (int it = 0; it < k; ++it) {
            float sum = 0.f; int cnt = 0;
            for (int q = 0; q < k; ++q) {
                const int p = __ldg(idx + q);
                const float a = fabsf(__ldg(u + p) - *T.at(cl, p) + xi[q]);
                if (a > theta) { sum += a; ++cnt; }
            }
            const float t2 = pg_div(sum - z, (float)cnt);
            if (!(t2 > theta)) break;
            theta = t2;
        }
    }
    float dmax = 0.f;
    for (int q = 0; q < k; ++q) {
        const int p = __ldg(idx + q);
        const float x0 = xi[q], r = __ldg(u + p) - *T.at(cl, p) + x0;
        dmax = fmaxf(dmax, fabsf(copysignf(fmaxf(fabsf(r) - theta, 0.f), r) - x0));
    }
    if (!(dmax > PG_BAND * wscale)) return 0.f;                   // dead band: keep the dual
    for (int q = 0; q < k; ++q) {
        const int p = __ldg(idx + q);
        float* tp = T.at(cl, p);
        const float x0 = xi[q], r = __ldg(u + p) - *tp + x0;
        const float xn = copysignf(fmaxf(fabsf(r) - theta, 0.f), r);
        xi[q] = xn;
        *tp += xn - x0;
    }
    return dmax > cf * PG_BAND * wscale ? dmax : 0.f;
}

// one group, one warp (all lanes get the same result)
__device__ __forceinline__ float pg_update_warp(const cg::cluster_group& cl, const PgTot T, const float* __restrict__ u,
                                                const int* __restrict__ idx, float* xi, int k, float z, float cf, int lane) {
    float sabs = 0.f, wscale = 0.f;
    for (int q = lane; q < k; q += 32) {
        const int p = __ldg(idx + q);
        const float uu = __ldg(u + p), tt = *T.at(cl, p), x0 = xi[q];
        sabs += fabsf(uu - tt + x0);
        wscale = fmaxf(wscale, fmaxf(fabsf(uu), fmaxf(fabsf(x0), fabsf(tt))));
    }
    sabs = warp_sum(sabs);
    wscale = warp_max(wscale);
    float theta = 0.f;
    if (!(z > 0.f)) theta = INFINITY;
    else if (sabs > z) {
        theta = pg_div(sabs - z, (float)k);
        for (int it = 0; it < k; ++it) {
            float sum = 0.f, cnt = 0.f;
            for (int q = lane; q < k; q += 32) {
                const int p = __ldg(idx + q);
                const float a = fabsf(__ldg(u + p) - *T.at(cl, p) + xi[q]);
                if (a > theta) { sum += a; cnt += 1.f; }
            }
            sum = warp_sum(sum);
            cnt = warp_sum(cnt);                                   // exact: counts < 2^24
            const float t2 = pg_div(sum - z, cnt);
            if (!(t2 > theta)) break;
            theta = t2;
        }
    }
    float dmax = 0.f;
    for (int q = lane; q < k; q += 32) {
        const int p = __ldg(idx + q);
        const float x0 = xi[q], r = __ldg(u + p) - *T.at(cl, p) + x0;
        dmax = fmaxf(dmax, fabsf(copysignf(fmaxf(fabsf(r) - theta, 0.f), r) - x0));
    }
    dmax = warp_max(dmax);
    if (!(dmax > PG_BAND * wscale)) return 0.f;
    for (int q = lane; q < k; q += 32) {
        const int p = __ldg(idx + q);
        float* tp = T.at(cl, p);
        const float x0 = xi[q], r = __ldg(u + p) - *tp + x0;
        const float xn = copysignf(fmaxf(fabsf(r) - theta, 0.f), r);
        xi[q] = xn;
        *tp += xn - x0;
    }
    return dmax > cf * PG_BAND * wscale ? dmax : 0.f;
}

__global__ void __launch_bounds__(PG_THREADS, 4) prox_graph_generic_kernel(PgArgs a) {
    float lam = a.lam, tol = a.tol;
    if (a.st != nullptr) {
        if (a.st->done) return;                                    // uniform over the grid
        lam = (float)pg_ddiv(a.st->lambda, a.st->mu);
        tol = tol * lam;                                           // relative tolerance in solver mode
    }
    cg::cluster_group cl = cg::this_cluster();
    const int cs = (int)cl.num_blocks(), rank = (int)cl.block_rank();
    const int cid = (int)(blockIdx.x >> __ffs(cs) - 1);             // cs is a power of two
    const int tid = threadIdx.x, lane = tid & 31;
    const int ctid = rank * PG_THREADS + tid, cthreads = cs * PG_THREADS;
    extern __shared__ __align__(16) float pg_smem[];
    __shared__ int item_s;
    __shared__ float red_s[PG_THREADS / 32];
    __shared__ float chg_s[2];
    PgTot T;
    T.s = pg_smem; T.g = a.totg ? a.totg + (size_t)cid * a.ld : nullptr; T.shift = a.shift; T.cs = cs;
    float* xi = a.xi + (size_t)cid * a.g.max_nnz;
    const GenericGraphDev G = a.g;
    const int p_lo = T.g ? 0 : min(rank << a.shift, a.m), p_hi = T.g ? a.m : min((rank + 1) << a.shift, a.m);
    const int p_step = T.g ? cthreads : PG_THREADS, p_off = T.g ? ctid : tid;
    for (;;) {
        if (rank == 0 && tid == 0) item_s = atomicAdd(a.status + 1, 1);
        cl.sync();
        const int f = *cl.map_shared_rank(&item_s, 0);
        cl.sync();                                                 // read before rank 0 takes the next frame
        if (f >= a.n) break;
        const int gr = G.frame_graph[f];
        const int c0 = G.gcol[gr], c1 = G.gcol[gr + 1];
        const int nz0 = G.gnz0[gr], nnz = G.gptr[G.cbeg[c1]] - nz0;
        const float* u = a.U + (size_t)f * a.ld;
        for (int p = p_lo + p_off; p < p_hi; p += p_step) {
            if (T.g) T.g[p] = 0.f; else pg_smem[p - p_lo] = 0.f;
        }
        for (int q = ctid; q < nnz; q += cthreads) xi[q] = 0.f;
        cl.sync();
        int sw = 0;
        for (; sw < a.max_sweeps; ++sw) {
            float ch = 0.f;
            for (int c = c0; c < c1; ++c) {
                const int gb = G.cbeg[c], gbig = G.cbig[c], ge = G.cbeg[c + 1];
                for (int g = gb + ctid; g < gbig; g += cthreads) {
                    const int b = G.gptr[g];
                    ch = fmaxf(ch, pg_update_small(cl, T, u, G.gidx + b, xi + (b - nz0), G.gptr[g + 1] - b, lam * G.eta[g],
                                                   a.count_factor));
                }
                for (int g = gbig + (ctid >> 5); g < ge; g += cthreads >> 5) {
                    const int b = G.gptr[g];
                    ch = fmaxf(ch, pg_update_warp(cl, T, u, G.gidx + b, xi + (b - nz0), G.gptr[g + 1] - b, lam * G.eta[g],
                                                  a.count_factor, lane));
                }
                cl.sync();
            }
            // largest counted change of this sweep over the cluster (slot sw & 1 is next written two sweeps later, after a
            // cluster barrier that every reader of this one has passed)
            ch = warp_max(ch);
            if (lane == 0) red_s[tid >> 5] = ch;
            __syncthreads();
            if (tid == 0) {
                float mx = 0.f;
                for (int w = 0; w < PG_THREADS / 32; ++w) mx = fmaxf(mx, red_s[w]);
                chg_s[sw & 1] = mx;
            }
            cl.sync();
            float all = 0.f;
            for (int r = 0; r < cs; ++r) all = fmaxf(all, *cl.map_shared_rank(&chg_s[sw & 1], (unsigned)r));
            if (all <= tol) { ++sw; break; }
        }
        // v = u - tot (pixels in no group have tot = 0: bit-exact identity)
        float* v = a.V + (size_t)f * a.ld;
        for (int p = p_lo + p_off; p < p_hi; p += p_step) v[p] = u[p] - (T.g ? T.g[p] : pg_smem[p - p_lo]);
        if (rank == 0 && tid == 0) atomicMax(a.status + 3, sw);
    }
}

// [0] = sweeps of this call, running totals [4] sweeps, [5] calls, [6] calls at the cap; resets the per-call slots
__global__ void prox_graph_generic_stats_kernel(int* status, int max_sweeps, const DevState* st) {
    if (st != nullptr && st->done) return;
    const int sw = status[3];
    status[0] = sw;
    status[4] += sw; status[5] += 1; if (sw >= max_sweeps) status[6] += 1;
    status[1] = 0; status[3] = 0;
}

// ------------------------------------------------------------------------------------------------------------- host side
static int pg_ceil_log2(long long v) { int s = 0; while ((1LL << s) < v) ++s; return s; }

GenericGraphLayout prox_graph_generic_layout(long long m, long long ld, int n, long long max_nnz) {
    GenericGraphLayout L;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    L.cs = 1;
    while (L.cs < 8 && pg_ceil_log2((m + L.cs - 1) / L.cs) > PG_MAX_SHIFT) L.cs *= 2;
    L.shift = pg_ceil_log2(std::max(1LL, (m + L.cs - 1) / L.cs));
    L.tot_global = L.shift > PG_MAX_SHIFT;
    if (L.tot_global) { L.cs = 1; L.shift = 0; }
    else
        while (L.cs < 8 && (long long)n * L.cs < sms) {             // few frames: spread each over more SMs
            L.cs *= 2;
            L.shift = pg_ceil_log2(std::max(1LL, (m + L.cs - 1) / L.cs));
        }
    long long cap_mb = 8192;
    if (const char* e = getenv("BSUB_GRAPH_XI_MB")) cap_mb = std::max(1LL, atoll(e));
    const long long per = std::max(1LL, max_nnz) + (L.tot_global ? ld : 0);
    long long slots = std::min<long long>(n, std::max(1LL, cap_mb * (1LL << 20) / 4 / per));
    slots = std::min<long long>(slots, (long long)sms * 8);
    L.slots = (int)std::max(1LL, slots);
    L.xi_floats = (long long)L.slots * std::max(1LL, max_nnz);
    L.tot_floats = L.tot_global ? (long long)L.slots * ld : 0;
    L.smem = L.tot_global ? 0 : sizeof(float) * ((size_t)1 << L.shift);
    return L;
}

int pack_generic_graphs(long long m, int n, int n_graphs, const int32_t* frame_graph, const int64_t* n_groups,
                        const int32_t* const* indptr, const int32_t* const* indices, const double* const* eta, GenericGraphHost* out,
                        const char* who) {
    if (m <= 0 || m > (1LL << 30) || n <= 0) { set_error("%s: bad matrix size (m=%lld, n=%d)", who, m, n); return -1; }
    if (n_graphs < 1 || !n_groups || !indptr || !indices || !eta) { set_error("%s: need at least one graph (n_graphs=%d)", who, n_graphs); return -1; }
    if (!frame_graph && n_graphs != 1) { set_error("%s: frame_graph is required with %d graphs", who, n_graphs); return -1; }
    GenericGraphHost& H = *out;
    H.frame_graph.assign(n, 0);
    for (int f = 0; f < n && frame_graph; ++f) {
        if (frame_graph[f] < 0 || frame_graph[f] >= n_graphs) {
            set_error("%s: frame_graph[%d] = %d is not a graph index in [0, %d)", who, f, frame_graph[f], n_graphs); return -1;
        }
        H.frame_graph[f] = frame_graph[f];
    }
    H.gcol.assign(1, 0); H.cbeg.clear(); H.cbig.clear(); H.gptr.assign(1, 0); H.gidx.clear(); H.eta.clear(); H.gnz0.clear();
    H.max_nnz = 0; H.max_colours = 0;
    std::vector<int> stamp((size_t)m, -1);
    for (int gi = 0; gi < n_graphs; ++gi) {
        const long long ng = n_groups[gi];
        const int32_t* ip = indptr[gi]; const int32_t* ix = indices[gi]; const double* et = eta[gi];
        if (ng < 0 || ng >= (1LL << 30)) { set_error("%s: graph %d: bad group count %lld", who, gi, ng); return -1; }
        if (ng > 0 && (!ip || !et)) { set_error("%s: graph %d: null indptr or eta", who, gi); return -1; }
        if (ng > 0 && ip[0] != 0) { set_error("%s: graph %d: indptr[0] = %d, expected 0", who, gi, ip[0]); return -1; }
        for (long long g = 0; g < ng; ++g) {
            if (ip[g + 1] < ip[g]) { set_error("%s: graph %d: indptr decreases at group %lld", who, gi, g); return -1; }
            if (!(std::isfinite(et[g]) && et[g] >= 0.0)) { set_error("%s: graph %d: eta[%lld] = %g is not finite and >= 0", who, gi, g, et[g]); return -1; }
        }
        const long long nnz = ng > 0 ? ip[ng] : 0;
        if (nnz > 0 && !ix) { set_error("%s: graph %d: null indices", who, gi); return -1; }
        if ((long long)H.gidx.size() + nnz >= (1LL << 31) - 1) { set_error("%s: more than 2^31 graph entries", who); return -1; }
        // validate and build the pixel -> groups transpose
        std::vector<int> pcnt((size_t)m + 1, 0);
        for (long long g = 0; g < ng; ++g)
            for (long long q = ip[g]; q < ip[g + 1]; ++q) {
                const int p = ix[q];
                if (p < 0 || p >= m) { set_error("%s: graph %d: group %lld holds pixel %d, not in [0, %lld)", who, gi, g, p, m); return -1; }
                if (stamp[p] == (int)g) {
                    set_error("%s: graph %d: group %lld holds pixel %d twice", who, gi, g, p); return -1;
                }
                stamp[p] = (int)g;
                pcnt[p + 1]++;
            }
        std::fill(stamp.begin(), stamp.end(), -1);
        for (long long p = 0; p < m; ++p) pcnt[p + 1] += pcnt[p];
        std::vector<int> pg((size_t)std::max(1LL, nnz)), fill(pcnt.begin(), pcnt.end() - 1);
        for (long long g = 0; g < ng; ++g)
            for (long long q = ip[g]; q < ip[g + 1]; ++q) pg[fill[ix[q]]++] = (int)g;
        // greedy colouring in input order
        std::vector<int> colour((size_t)ng, -1), mark;
        int ncol = 0;
        for (long long g = 0; g < ng; ++g) {
            if (ip[g + 1] == ip[g]) continue;                       // empty group: no effect on the solution
            for (long long q = ip[g]; q < ip[g + 1]; ++q) {
                const int p = ix[q];
                for (int t = pcnt[p]; t < pcnt[p + 1]; ++t) {
                    const int c = colour[pg[t]];
                    if (c >= 0) mark[c] = (int)g;
                }
            }
            int c = 0;
            while (c < ncol && mark[c] == (int)g) ++c;
            if (c == ncol) { ++ncol; mark.push_back(-1); }
            colour[g] = c;
        }
        // colour-major layout, small groups before large ones within a colour
        std::vector<int> cnt_small(ncol, 0), cnt_all(ncol, 0);
        for (long long g = 0; g < ng; ++g)
            if (colour[g] >= 0) { cnt_all[colour[g]]++; if (ip[g + 1] - ip[g] <= PG_SMALL) cnt_small[colour[g]]++; }
        std::vector<int> pos_small(ncol), pos_big(ncol);
        int base = (int)H.gptr.size() - 1;
        for (int c = 0; c < ncol; ++c) {
            H.cbeg.push_back(base); H.cbig.push_back(base + cnt_small[c]);
            pos_small[c] = base; pos_big[c] = base + cnt_small[c];
            base += cnt_all[c];
        }
        const int g0 = (int)H.gptr.size() - 1, nzbase = (int)H.gidx.size();
        std::vector<int> order((size_t)(base - g0));
        for (long long g = 0; g < ng; ++g)
            if (colour[g] >= 0) order[(ip[g + 1] - ip[g] <= PG_SMALL ? pos_small[colour[g]]++ : pos_big[colour[g]]++) - g0] = (int)g;
        H.gnz0.push_back(nzbase);
        for (int g : order) {
            for (long long q = ip[g]; q < ip[g + 1]; ++q) H.gidx.push_back(ix[q]);
            H.gptr.push_back((int)H.gidx.size());
            H.eta.push_back((float)et[g]);
        }
        H.gcol.push_back((int)H.cbeg.size());
        H.max_nnz = std::max<long long>(H.max_nnz, (long long)H.gidx.size() - nzbase);
        H.max_colours = std::max(H.max_colours, ncol);
    }
    H.cbeg.push_back((int)H.gptr.size() - 1);                       // end of the last colour
    return 0;
}

int upload_generic_graphs(const GenericGraphHost& H, int** ints, float** eta_dev, GenericGraphDev* dev) {
    const size_t nint = H.frame_graph.size() + H.gcol.size() + H.cbeg.size() + H.cbig.size() + H.gptr.size() + H.gidx.size() + H.gnz0.size();
    std::vector<int> all;
    all.reserve(nint);
    size_t off[7], k = 0;
    for (const std::vector<int>* v : {&H.frame_graph, &H.gcol, &H.cbeg, &H.cbig, &H.gptr, &H.gidx, &H.gnz0}) {
        off[k++] = all.size();
        all.insert(all.end(), v->begin(), v->end());
    }
    if (*ints) { cudaFree(*ints); *ints = nullptr; }
    if (*eta_dev) { cudaFree(*eta_dev); *eta_dev = nullptr; }
    BSUB_CUDA_CHECK(cudaMalloc((void**)ints, sizeof(int) * std::max<size_t>(1, all.size())));
    BSUB_CUDA_CHECK(cudaMalloc((void**)eta_dev, sizeof(float) * std::max<size_t>(1, H.eta.size())));
    BSUB_CUDA_CHECK(cudaMemcpy(*ints, all.data(), sizeof(int) * all.size(), cudaMemcpyHostToDevice));
    if (!H.eta.empty()) BSUB_CUDA_CHECK(cudaMemcpy(*eta_dev, H.eta.data(), sizeof(float) * H.eta.size(), cudaMemcpyHostToDevice));
    dev->frame_graph = *ints + off[0]; dev->gcol = *ints + off[1]; dev->cbeg = *ints + off[2]; dev->cbig = *ints + off[3];
    dev->gptr = *ints + off[4]; dev->gidx = *ints + off[5]; dev->gnz0 = *ints + off[6]; dev->eta = *eta_dev;
    dev->max_nnz = H.max_nnz;
    return 0;
}

int launch_prox_graph_generic(const float* U, float* V, long long ld, long long m, int n, const GenericGraphDev& g, const GenericGraphLayout& L,
                              float* xi, float* totg, float lam, int max_sweeps, float tol, int* status, const DevState* st, cudaStream_t s) {
    if (!xi || !status || (L.tot_global && !totg)) { set_error("prox_graph_generic: missing workspace"); return -1; }
    static unsigned long long attr_devs = 0;
    if (first_call_on_device(&attr_devs))
        BSUB_CUDA_CHECK(cudaFuncSetAttribute(prox_graph_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)(sizeof(float) << PG_MAX_SHIFT)));
    PgArgs a;
    a.U = U; a.V = V; a.ld = ld; a.m = (int)m; a.n = n; a.lam = lam; a.tol = tol; a.max_sweeps = max_sweeps;
    a.count_factor = PG_COUNT_FACTOR;
    a.g = g; a.xi = xi; a.totg = L.tot_global ? totg : nullptr; a.shift = L.shift; a.status = status; a.st = st;
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = L.cs; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.blockDim = dim3(PG_THREADS); cfg.dynamicSmemBytes = L.smem; cfg.stream = s; cfg.attrs = attr; cfg.numAttrs = 1;
    int clusters = L.slots;
    {
        cfg.gridDim = dim3((unsigned)(L.cs * clusters));
        int active = 0;
        BSUB_CUDA_CHECK(cudaOccupancyMaxActiveClusters(&active, (void*)prox_graph_generic_kernel, &cfg));
        if (active < 1) { set_error("prox_graph_generic: a cluster of %d CTAs with %zu B of shared memory does not fit", L.cs, L.smem); return -1; }
        clusters = std::min(clusters, active);
    }
    cfg.gridDim = dim3((unsigned)(L.cs * clusters));
    BSUB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, prox_graph_generic_kernel, a));
    prox_graph_generic_stats_kernel<<<1, 1, 0, s>>>(status, max_sweeps, st);
    BSUB_CUDA_CHECK(cudaGetLastError());
    return 0;
}

}  // namespace bsub
