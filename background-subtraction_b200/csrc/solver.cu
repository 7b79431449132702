// solver.cu -- host orchestration and the extern "C" boundary (include/bsub_b200.h).
//
// One bsub_solver owns the device-resident state of one decomposition (D, S, Y, T, eigen workspace, control
// state) on one GPU and one stream.  bsub_run() is the whole single-GPU solve; the bsub_step_* functions expose
// the same sequence in pieces so that a pixel-sharded multi-GPU driver can all-reduce the frames x frames Gram
// and a few scalars between them (DESIGN.md section 6).  The ALM loop never waits on the host: every kernel
// reads its scalars (mu, rank, stop flag) from DevState and returns immediately once the stop flag is set; the
// host only limits how far ahead it enqueues by watching a mapped status word.
#include <math.h>
#include <stdarg.h>
#include <cmath>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include <algorithm>
#include "../../include/bsub_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace bsub {
static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
}  // namespace bsub

using namespace bsub;

#define CK(expr) BSUB_CUDA_CHECK(expr)
#define RET_IF(expr) do { int _rc = (expr); if (_rc != 0) return _rc; } while (0)

static const int kCommTail = 16;     // doubles after the Gram in the sum buffer
static const int kRunAhead = 3;      // iterations the host may enqueue ahead of the device

// The prox of whole rows x cols frames [f0, f0 + nf) of a clip (m pixels each; the generic kernel needs m alone), as one setter or
// one stand-alone operator describes it.  Built by describe_windows / _centre / _graphs, run by graph_prox.
struct GraphDesc {
    int kind = 0;                                       // BSUB_PROX_GRAPH_LINF (windows), _CENTER_BG (centre map), _GENERIC; 0: none
    int rows = 0, cols = 0, f0 = 0, nf = 0;
    long long m = 0;
    float* eta = nullptr; long long eta_stride = 0;     // tile kernel: window weights (stride 0; NULL: unit) or centre map [nf][m]
    int* ints = nullptr; GenericGraphDev graphs = {};   // generic kernel: packed graphs, their eta in graphs.eta, frame_graph[nf]
    unsigned char* labels = nullptr; double* bsums = nullptr;   // background (label 0) [nf][m] and its per-frame sums, or none
    void release() {
        for (void* p : {(void*)eta, (void*)ints, (void*)graphs.eta, (void*)labels, (void*)bsums}) if (p) cudaFree(p);
        *this = GraphDesc();
    }
};

// duals of the graph prox: allocated once, grown when a call needs more
struct ProxWork {
    float *xi = nullptr, *tot = nullptr;
    long long xi_floats = 0, tot_floats = 0;
    void release() {
        for (float* p : {xi, tot}) if (p) cudaFree(p);
        *this = ProxWork();
    }
};

struct bsub_solver {
    bsub_config cfg;
    int device = 0, num_sms = 148;
    long long m = 0, ld = 0;
    int n = 0, npad = 0;
    float *D = nullptr, *S = nullptr, *Y = nullptr, *T = nullptr, *L = nullptr, *U = nullptr;
    DevState* st = nullptr;
    IterLog* log = nullptr;
    HostMirror* mirror = nullptr;       // mapped pinned host memory
    HostMirror* mirror_dev = nullptr;
    double* comm_sum = nullptr;         // [npad*npad + kCommTail]
    double* comm_max = nullptr;         // [8]
    GramPlan gp; GramMaps gmaps; int2* tasks_dev = nullptr; double* gram_partial = nullptr;
    EigPlan ep; EigBuffers eb;
    ShrinkPlan sp; ShrinkTmaPlan stp; ShrinkTmaMaps stmaps; bool use_tma = false, stmaps_ready = false;
    ShrinkStreamPlan ssp; ShrinkTmaMaps ssmaps; bool use_stream = false;
    // int8 tcgen05 Gram from the W slices written by the streamed shrink pass
    bool use_i8 = false; signed char* Wq = nullptr; unsigned long long* Gint = nullptr; GramI8Plan gip; CUtensorMap gimap, gimap_last;
    int4* gi_info = nullptr; int* gi_blkn = nullptr; int gi_ncta = 0; float* part_wmax = nullptr;
    // T = Vr^T W from the digit planes (project.cu): lets the streamed shrink kernel read every tile once
    bool use_proj = false; ProjectPlan pjp; float* Tt = nullptr;
    bool use_flat = false, sfmaps_ready = false; ShrinkFlatPlan sfp; ShrinkFlatMaps sfmaps;     // single-pass shrink (shrink_flat.cu)
    bool force_S = false;                     // store S in every iteration (BSUB_FLAG_ALWAYS_STORE_S, or after a restart)
    int proj_iter = -1;                       // iteration (iters_enqueued) whose projection has already been launched (bsub_step_project)
    float* tpart = nullptr; double* part_zz = nullptr; unsigned long long* part_nnz = nullptr;
    float* part_max = nullptr;
    int shrink_mode = SHRINK_FLAT3;
    // generic flat groups
    int* gptr = nullptr; int* gidx = nullptr; int ngroups = 0; bool groups_set = false;
    // graph modes: the one description (whole-clip: bsub_set_graph_windows / _center_windows / _graphs, run by the SPILL pass; else
    // a frame range: bsub_set_frame_*, run by bsub_step_prox_block on the frames a pixel-sharded driver has gathered), the duals of
    // its prox and the counters bsub_debug_graph reads
    GraphDesc graph; bool graph_whole = false; ProxWork work; int* sweeps_dev = nullptr;
    // l2 blocks
    unsigned char* labels_dev = nullptr; double* lam_table = nullptr; double* bsums = nullptr; int nlab = 0; bool blocks_set = false;
    unsigned char* mask_stage = nullptr;      // bsub_mask_host staging
    double* mask_scratch = nullptr;           // per-CTA partials of the mask statistics (fixed-order reduction)
    double* stage64 = nullptr; size_t stage64_doubles = 0;   // fp64 staging of bsub_load_D_f64_host / bsub_download_f64 (allocated once)
    cudaStream_t last_stream = nullptr; bool stream_seen = false;
    bool implied_first = false;               // see bsub_step_init_finish
    bool loaded = false, finalized = false, initialised = false;
    cudaEvent_t ev[kRunAhead + 1];
    int iters_enqueued = 0;
};

static cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static cudaStream_t use_stream(bsub_solver* s, void* stream) {
    s->last_stream = as_stream(stream); s->stream_seen = true;
    return s->last_stream;
}
static int ensure_stage64(bsub_solver* s, size_t doubles) {
    if (s->stage64_doubles >= doubles) return 0;
    if (s->stage64) { cudaFree(s->stage64); s->stage64 = nullptr; s->stage64_doubles = 0; }
    BSUB_CUDA_CHECK(cudaMalloc((void**)&s->stage64, sizeof(double) * doubles));
    s->stage64_doubles = doubles;
    return 0;
}
// whole-frame prox workspaces: allocated once, grown when a call needs more
static int grow_floats(float** p, long long* have, long long want) {
    if (want <= *have) return 0;
    if (*p) cudaFree(*p);
    *p = nullptr; *have = 0;
    CK(cudaMalloc((void**)p, sizeof(float) * (size_t)want));
    *have = want;
    return 0;
}

// frees whatever a stand-alone operator allocated, on every return path
struct DevScope {
    std::vector<void*> ptrs;
    ~DevScope() { for (void* p : ptrs) if (p) cudaFree(p); }
    template <typename T> int alloc(T** out, size_t bytes) {
        void* p = nullptr;
        if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(cudaGetLastError())); return -1; }
        ptrs.push_back(p);
        *out = reinterpret_cast<T*>(p);
        return 0;
    }
};

// ----------------------------------------------------------------------------------------------------- graph prox descriptions
// Each builder validates every entry, then uploads *d; on failure *d holds nothing.  args_ok = false: the caller's own arguments are
// bad, reported after the description's errors and before any device call.
static long long window_count(int rows, int cols) { return (long long)(rows - std::min(3, rows) + 1) * (cols - std::min(3, cols) + 1); }

// eta float[n_eta] (n_eta may be 0) and background uint8[nf][m] (may be NULL) -> label 0 (the complement group of the l2 kernels) /
// 255 (keeps the graph prox result)
static int describe_upload(GraphDesc* d, const float* eta, size_t n_eta, const uint8_t* background) {
    const int rc = [&]() -> int {
        if (n_eta > 0) {
            CK(cudaMalloc((void**)&d->eta, sizeof(float) * n_eta));
            CK(cudaMemcpy(d->eta, eta, sizeof(float) * n_eta, cudaMemcpyHostToDevice));
        }
        if (background == nullptr || d->nf == 0) return 0;
        const size_t nm = (size_t)d->nf * d->m;
        std::vector<unsigned char> lab(nm);
        for (size_t i = 0; i < nm; ++i) lab[i] = background[i] ? 0 : 255;
        CK(cudaMalloc((void**)&d->labels, nm));
        CK(cudaMalloc((void**)&d->bsums, sizeof(double) * d->nf));
        CK(cudaMemcpy(d->labels, lab.data(), nm, cudaMemcpyHostToDevice));
        return 0;
    }();
    if (rc != 0) d->release();
    return rc;
}

// the 3x3 all-window graph, eta double[n_eta] one weight per window (finite, >= 0) the same in every frame; NULL: unit weights
static int describe_windows(GraphDesc* d, int rows, int cols, int f0, int nf, const double* eta, long long n_eta, const char* who,
                            bool args_ok = true) {
    const long long nw = window_count(rows, cols);
    std::vector<float> ef;
    if (eta != nullptr) {
        if (n_eta != nw) { set_error("%s: eta has %lld entries, the %dx%d image has %lld windows", who, n_eta, rows, cols, nw); return -1; }
        ef.resize((size_t)nw);
        for (long long i = 0; i < nw; ++i) {
            if (!(std::isfinite(eta[i]) && eta[i] >= 0.0)) { set_error("%s: eta[%lld] = %g is not finite and >= 0", who, i, eta[i]); return -1; }
            ef[i] = (float)eta[i];
        }
    }
    if (!args_ok) { set_error("%s: bad argument", who); return -1; }
    *d = GraphDesc{BSUB_PROX_GRAPH_LINF, rows, cols, f0, nf, (long long)rows * cols};
    return describe_upload(d, ef.data(), ef.size(), nullptr);
}

// radius-1 centre windows, eta float32[nf][rows*cols] (finite) = weight of the window centred on that pixel in that frame
static int describe_centre(GraphDesc* d, int rows, int cols, int f0, int nf, const float* eta, const uint8_t* background, const char* who,
                           bool args_ok = true) {
    const size_t nm = (rows > 0 && cols > 0 && nf > 0) ? (size_t)nf * rows * cols : 0;
    for (size_t i = 0; i < nm; ++i)
        if (!std::isfinite(eta[i])) { set_error("%s: eta[%zu] = %g is not finite", who, i, (double)eta[i]); return -1; }
    if (!args_ok) { set_error("%s: bad argument", who); return -1; }
    *d = GraphDesc{BSUB_PROX_GRAPH_CENTER_BG, rows, cols, f0, nf, (long long)rows * cols};
    d->eta_stride = d->m;
    return describe_upload(d, eta, nm, background);
}

// any non-nested graphs (the generic kernel), frame_graph[nf] for the frames of the range
static int describe_graphs(GraphDesc* d, int rows, int cols, long long m, int f0, int nf, int n_graphs, const int32_t* frame_graph,
                           const int64_t* n_groups, const int32_t* const* indptr, const int32_t* const* indices, const double* const* eta,
                           const uint8_t* background, const char* who, bool args_ok = true) {
    GenericGraphHost H;
    if (nf > 0) RET_IF(pack_generic_graphs(m, nf, n_graphs, frame_graph, n_groups, indptr, indices, eta, &H, who));
    if (!args_ok) { set_error("%s: bad argument", who); return -1; }
    *d = GraphDesc{BSUB_PROX_GRAPH_GENERIC, rows, cols, f0, nf, m};
    if (nf > 0) {
        float* geta = nullptr;
        const int rc = upload_generic_graphs(H, &d->ints, &geta, &d->graphs);
        d->graphs.eta = geta;                           // d owns it whether or not the upload finished
        if (rc != 0) { d->release(); return rc; }
    }
    return describe_upload(d, nullptr, 0, background);
}

// the duals of nf frames of d at row pitch ld, grown in *w; *L: the generic kernel's layout
static int size_work(const GraphDesc& d, long long ld, int nf, ProxWork* w, long long* xi_floats, GenericGraphLayout* L) {
    long long tot_floats = 0;
    if (d.kind == BSUB_PROX_GRAPH_GENERIC) {
        *L = prox_graph_generic_layout(d.m, ld, nf, d.graphs.max_nnz);
        *xi_floats = L->xi_floats; tot_floats = L->tot_floats;
    } else {
        prox_graph3_workspace(d.rows, d.cols, nf, ld, d.kind == BSUB_PROX_GRAPH_CENTER_BG ? 1 : 0, xi_floats, &tot_floats);
    }
    RET_IF(grow_floats(&w->xi, &w->xi_floats, *xi_floats));
    return grow_floats(&w->tot, &w->tot_floats, tot_floats);
}

// prox of the whole frames [f0, f0 + nf) -- within d's range -- held in U / V (row f - f0 = frame f, row pitch ld): the tile or the
// generic kernel, then the l2 shrink of each frame's background.  st != nullptr: lambda / mu and the stop flag come from the device
// state, else lam is lambda1.  sweeps: the int[8] status block of the prox kernels.
static int graph_prox(const GraphDesc& d, const float* U, float* V, long long ld, int f0, int nf, const DevState* st, float lam,
                      int max_sweeps, float tol, int* sweeps, ProxWork* w, cudaStream_t stream) {
    if (nf == 0) return 0;
    const int lf = f0 - d.f0;
    long long xi_floats = 0;
    GenericGraphLayout L;
    RET_IF(size_work(d, ld, nf, w, &xi_floats, &L));
    if (d.kind == BSUB_PROX_GRAPH_GENERIC) {
        GenericGraphDev g = d.graphs;
        g.frame_graph += lf;
        RET_IF(launch_prox_graph_generic(U, V, ld, d.m, nf, g, L, w->xi, w->tot, lam, max_sweeps, tol, sweeps, st, stream));
    } else {
        const float* eta = d.eta ? d.eta + (size_t)lf * d.eta_stride : nullptr;
        RET_IF(launch_prox_graph3(U, V, w->xi, xi_floats, w->tot, eta, ld, d.rows, d.cols, nf, lam, max_sweeps, tol, sweeps, st, stream,
                                  d.kind == BSUB_PROX_GRAPH_CENTER_BG ? 1 : 0, d.eta_stride));
    }
    if (d.labels) {       // background pixels: their frame's l2 shrink of G_S at non_block_lambda / mu, over the graph prox result
        const unsigned char* lab = d.labels + (size_t)lf * d.m;
        RET_IF(launch_block_l2_sums(U, lab, ld, d.m, nf, 1, d.bsums, st, stream));
        RET_IF(launch_block_l2_apply(U, V, lab, ld, d.m, nf, 1, d.bsums, nullptr, st, 0.0, 0.0, stream, 1));
    }
    return 0;
}

static int round_half_even_005(int d) {
    // Python round(0.05 * d) -- banker's rounding on the double product (SURVEY Q5)
    return (int)nearbyint(0.05 * (double)d);
}

extern "C" {

const char* bsub_last_error(void) { return g_err; }
int bsub_version(void) { return 100; }

void bsub_abi_sizes(int32_t out3[3]) {
    out3[0] = (int32_t)sizeof(bsub_config); out3[1] = (int32_t)sizeof(bsub_status); out3[2] = (int32_t)sizeof(bsub_iter_log);
}

void bsub_default_config(bsub_config* c) {
    memset(c, 0, sizeof(*c));
    c->prox = BSUB_PROX_FLAT_LINF; c->group_rows = 3; c->group_cols = 3; c->delta = 10.0; c->mu_scale = 12.5; c->rho = 1.6;
    c->tol = 1e-7; c->max_iter = 500; c->sv0 = 10; c->use_sv_prediction = 1; c->break_on_rank0 = 0;
    c->non_block_lambda_scale = 100.0; c->graph_max_sweeps = 4000; c->graph_tol = 1e-6;
}

int bsub_destroy(bsub_solver* s) {
    if (!s) return 0;
    int cur = 0;
    cudaGetDevice(&cur);
    if (cur != s->device) cudaSetDevice(s->device);
    // only this solver's work has to drain: a device-wide synchronise would stall the other clips in flight
    if (s->stream_seen) cudaStreamSynchronize(s->last_stream); else cudaDeviceSynchronize();
    void* ptrs[] = {s->D, s->S, s->Y, s->T, s->L, s->U, s->st, s->log, s->comm_sum, s->comm_max, s->tasks_dev, s->gram_partial,
                    s->eb.work, s->eb.lam, s->eb.Z, s->eb.Vr, s->eb.VC, s->tpart, s->part_zz, s->part_nnz, s->part_max, s->gptr,
                    s->gidx, s->sweeps_dev, s->labels_dev, s->lam_table, s->bsums, s->Wq, s->Gint, s->gi_info, s->gi_blkn, s->part_wmax,
                    s->mask_stage, s->mask_scratch, s->stage64, s->Tt};
    for (void* p : ptrs) if (p) cudaFree(p);
    s->graph.release();
    s->work.release();
    if (s->mirror) cudaFreeHost((void*)s->mirror);
    for (int i = 0; i <= kRunAhead; ++i) if (s->ev[i]) cudaEventDestroy(s->ev[i]);
    const int own = s->device;
    delete s;
    if (cur != own) cudaSetDevice(cur);
    return 0;
}

int bsub_create(const bsub_config* cfg, bsub_solver** out) {
    if (!cfg || !out) { set_error("bsub_create: null argument"); return -1; }
    if (cfg->m <= 0 || cfg->n <= 0) { set_error("bsub_create: empty matrix (m=%lld, n=%d)", (long long)cfg->m, cfg->n); return -1; }
    if (cfg->prox < 0 || cfg->prox > 5) { set_error("bsub_create: unknown prox %d", cfg->prox); return -1; }
    if ((cfg->prox == BSUB_PROX_FLAT_LINF || cfg->prox == BSUB_PROX_GRAPH_LINF || cfg->prox == BSUB_PROX_GRAPH_CENTER_BG) &&
        ((long long)cfg->rows * cfg->cols != cfg->m)) {
        set_error("bsub_create: rows*cols (%d*%d) != m (%lld)", cfg->rows, cfg->cols, (long long)cfg->m); return -1;
    }
    if ((cfg->prox == BSUB_PROX_GRAPH_LINF || cfg->prox == BSUB_PROX_GRAPH_CENTER_BG) && (cfg->group_rows != 3 || cfg->group_cols != 3)) {
        set_error("bsub_create: overlapping windows are implemented for the reference's 3x3 BLOCK_SIZE only"); return -1;
    }
    bsub_solver* s = new bsub_solver();
    for (int i = 0; i <= kRunAhead; ++i) s->ev[i] = nullptr;
    memset(&s->eb, 0, sizeof(s->eb));
    s->cfg = *cfg;
    if (s->cfg.m_global <= 0) s->cfg.m_global = cfg->m;
    if (s->cfg.max_iter <= 0) s->cfg.max_iter = 500;
    if (s->cfg.max_iter > kMaxIterLog) s->cfg.max_iter = kMaxIterLog;
    if (s->cfg.graph_max_sweeps <= 0) s->cfg.graph_max_sweeps = 4000;
    if (s->cfg.graph_tol <= 0) s->cfg.graph_tol = 1e-6;
    if (s->cfg.non_block_lambda_scale <= 0) s->cfg.non_block_lambda_scale = 100.0;
    s->m = cfg->m; s->n = cfg->n;
    s->force_S = (cfg->flags & BSUB_FLAG_ALWAYS_STORE_S) != 0;
    s->ld = ((cfg->m + 31) / 32) * 32;
    s->npad = ((cfg->n + 31) / 32) * 32;
    int rc = 0;
    do {
        if (cudaGetDevice(&s->device) != cudaSuccess) { set_error("bsub_create: no CUDA device (the CUDA path is mandatory; there is no CPU fallback)"); rc = -1; break; }
        cudaDeviceGetAttribute(&s->num_sms, cudaDevAttrMultiProcessorCount, s->device);
        const size_t mat = sizeof(float) * (size_t)s->ld * s->n;
#define ALLOC(ptr, bytes) if (cudaMalloc((void**)&(ptr), (bytes)) != cudaSuccess) { set_error("bsub_create: cudaMalloc(%zu) failed: %s", (size_t)(bytes), cudaGetErrorString(cudaGetLastError())); rc = -1; break; }
        ALLOC(s->D, mat); ALLOC(s->S, mat); ALLOC(s->Y, mat);
        cudaMemset(s->S, 0, mat); cudaMemset(s->Y, 0, mat);     // pad columns stay zero even when init_Y is skipped
        ALLOC(s->T, mat);                                    // T has up to n rows (rank <= n)
        cudaMemset(s->T, 0, mat);                            // pad columns must read as zero
        ALLOC(s->st, sizeof(DevState)); ALLOC(s->log, sizeof(IterLog) * kMaxIterLog);
        ALLOC(s->comm_sum, sizeof(double) * ((size_t)s->npad * s->npad + kCommTail));
        ALLOC(s->comm_max, sizeof(double) * 8);
        ALLOC(s->sweeps_dev, sizeof(int) * 8);
        cudaMemset(s->sweeps_dev, 0, sizeof(int) * 8);
        ALLOC(s->mask_scratch, sizeof(double) * mask_stats_scratch_doubles());
        cudaMemset(s->mask_scratch, 0, sizeof(double) * mask_stats_scratch_doubles());
        cudaMemset(s->comm_sum, 0, sizeof(double) * ((size_t)s->npad * s->npad + kCommTail));
        cudaMemset(s->comm_max, 0, sizeof(double) * 8);
        cudaMemset(s->log, 0, sizeof(IterLog) * kMaxIterLog);
        if (cudaHostAlloc((void**)&s->mirror, sizeof(HostMirror), cudaHostAllocMapped) != cudaSuccess) { set_error("bsub_create: cudaHostAlloc failed"); rc = -1; break; }
        memset((void*)s->mirror, 0, sizeof(HostMirror));
        if (cudaHostGetDevicePointer((void**)&s->mirror_dev, (void*)s->mirror, 0) != cudaSuccess) { set_error("bsub_create: cudaHostGetDevicePointer failed"); rc = -1; break; }
        // Gram
        s->gp = make_gram_plan(s->n, s->ld, s->num_sms);
        if (make_gram_maps(s->gp, s->D, s->S, s->Y, s->ld, &s->gmaps) != 0) { rc = -1; break; }
        std::vector<int2> tasks(s->gp.ntasks);
        fill_gram_tasks(s->gp, tasks.data());
        ALLOC(s->tasks_dev, sizeof(int2) * s->gp.ntasks);
        cudaMemcpy(s->tasks_dev, tasks.data(), sizeof(int2) * s->gp.ntasks, cudaMemcpyHostToDevice);
        ALLOC(s->gram_partial, sizeof(double) * s->gp.partial_elems);
        // eigen solver
        s->ep = make_eig_plan(s->n, s->npad);
        ALLOC(s->eb.work, sizeof(double) * s->ep.work_doubles);
        ALLOC(s->eb.lam, sizeof(double) * s->n);
        ALLOC(s->eb.Z, sizeof(double) * (size_t)s->n * s->n);
        s->eb.vstride = std::max(16, ((s->n + 3) / 4) * 4);        // >= 16: the streamed shrink loads 16-column boxes
        ALLOC(s->eb.Vr, sizeof(float) * (size_t)s->n * s->eb.vstride);
        ALLOC(s->eb.VC, sizeof(float) * (size_t)s->n * s->eb.vstride);
        cudaMemset(s->eb.Vr, 0, sizeof(float) * (size_t)s->n * s->eb.vstride);
        cudaMemset(s->eb.VC, 0, sizeof(float) * (size_t)s->n * s->eb.vstride);
        // shrink
        int rows = cfg->rows, cols = cfg->cols;
        if ((long long)rows * cols != s->m) {
            // no image geometry (block-l2 / l1 modes do not depend on it): pick any factorisation m = rows*cols that
            // tiles well (rows a multiple of 4, as large as fits a few tiles), else one long column.
            rows = (int)s->m; cols = 1;
            for (int r = 4096; r >= 48; r -= 4)
                if (s->m % r == 0) { rows = r; cols = (int)(s->m / r); break; }
        }
        s->sp = make_shrink_plan(s->n, rows, cols, s->ld, s->num_sms, cfg->tile_rows, cfg->cluster_frames);
        s->use_tma = make_shrink_tma_plan(s->n, rows, cols, s->ld, s->num_sms, cfg->tile_rows, cfg->cluster_frames, &s->stp);
        s->use_stream = s->use_tma && (getenv("BSUB_NO_STREAM") == nullptr) &&
                        make_shrink_stream_plan(s->n, rows, cols, s->ld, s->num_sms, cfg->tile_rows, &s->ssp);
        ALLOC(s->tpart, sizeof(float) * std::max(s->sp.tpart_floats, s->use_tma ? s->stp.tpart_floats : (size_t)0));
        int nparts = std::max(std::max(s->sp.nparts, (s->use_tma ? s->stp.nparts : 0) + (s->use_stream ? s->ssp.nparts : 0) + s->num_sms), s->num_sms * 8);
        ALLOC(s->part_zz, sizeof(double) * nparts); ALLOC(s->part_nnz, sizeof(unsigned long long) * nparts);
        ALLOC(s->part_max, sizeof(float) * nparts);
        cudaMemset(s->part_zz, 0, sizeof(double) * nparts); cudaMemset(s->part_nnz, 0, sizeof(unsigned long long) * nparts);
        cudaMemset(s->part_max, 0, sizeof(float) * nparts);
        s->use_i8 = s->use_stream && (shrink_stream_ldq(s->ssp) > 0) && (getenv("BSUB_NO_I8") == nullptr) &&
                    (cfg->prox == BSUB_PROX_FLAT_LINF || cfg->prox == BSUB_PROX_L1);
        if (s->use_i8) {
            const long long ldq = shrink_stream_ldq(s->ssp);
            s->gip = make_gram_i8_plan(s->n, ldq, s->num_sms);
            s->gip.m_real = s->m;
            s->gip.m_global = s->cfg.m_global;
            std::vector<int4> info; std::vector<int> blkn;
            fill_gram_i8_tables(s->gip, info, blkn);
            s->gi_ncta = (int)info.size();
            ALLOC(s->Wq, (size_t)4 * s->n * ldq);
            cudaMemset(s->Wq, 0, (size_t)4 * s->n * ldq);                     // the row tails (ldq padding) stay zero
            ALLOC(s->Gint, sizeof(unsigned long long) * (size_t)s->gip.nblk * 128 * s->gip.nblk * 128);
            ALLOC(s->gi_info, sizeof(int4) * info.size());
            ALLOC(s->gi_blkn, sizeof(int) * blkn.size());
            ALLOC(s->part_wmax, sizeof(float) * (s->ssp.grid + s->num_sms));
            cudaMemcpy(s->gi_info, info.data(), sizeof(int4) * info.size(), cudaMemcpyHostToDevice);
            cudaMemcpy(s->gi_blkn, blkn.data(), sizeof(int) * blkn.size(), cudaMemcpyHostToDevice);
            cudaMemset(s->part_wmax, 0, sizeof(float) * (s->ssp.grid + s->num_sms));
            if (make_gram_i8_map(s->gip, s->Wq, &s->gimap, 128) != 0) { rc = -1; break; }
            if (make_gram_i8_map(s->gip, s->Wq, &s->gimap_last, gram_i8_last_block_n(s->gip)) != 0) { rc = -1; break; }
            s->use_proj = (getenv("BSUB_NO_PROJ") == nullptr) && make_project_plan(s->n, s->ssp.R, ldq, s->num_sms, &s->pjp);
            if (s->use_proj) {
                const size_t tt = sizeof(float) * (size_t)s->ssp.ntiles * 16 * 4 * s->ssp.R;
                ALLOC(s->Tt, tt);
                cudaMemset(s->Tt, 0, tt);
                s->use_flat = (getenv("BSUB_NO_FLAT") == nullptr) && make_shrink_flat_plan(s->n, s->ssp.rows, s->ssp.cols, s->ld, s->num_sms, s->ssp, &s->sfp);
            }
        }
        for (int i = 0; i <= kRunAhead; ++i)
            if (cudaEventCreateWithFlags(&s->ev[i], cudaEventDisableTiming) != cudaSuccess) { set_error("bsub_create: event"); rc = -1; break; }
        if (rc) break;
        switch (cfg->prox) {
            case BSUB_PROX_FLAT_LINF: s->shrink_mode = (cfg->group_rows == 3 && cfg->group_cols == 3) ? SHRINK_FLAT3 : SHRINK_SPILL; break;
            case BSUB_PROX_L1: s->shrink_mode = SHRINK_L1; break;
            default: s->shrink_mode = SHRINK_SPILL; break;
        }
        s->implied_first = s->use_i8 && s->use_stream && s->shrink_mode != SHRINK_SPILL && s->cfg.use_sv_prediction &&
                           s->cfg.sv0 >= 1 && s->cfg.sv0 <= s->ssp.kcap;
        if (s->shrink_mode == SHRINK_SPILL) { ALLOC(s->U, mat); ALLOC(s->L, mat); cudaMemset(s->U, 0, mat); cudaMemset(s->L, 0, mat); }
#undef ALLOC
        if (cudaGetLastError() != cudaSuccess) { /* clear sticky-less errors from memset probing */ }
    } while (0);
    if (rc != 0) { bsub_destroy(s); return rc; }
    *out = s;
    return 0;
}

// --------------------------------------------------------------------------------------------------- groups
int bsub_set_flat_groups(bsub_solver* s, const int32_t* g) {
    if (!s || !g) { set_error("bsub_set_flat_groups: null argument"); return -1; }
    if (s->cfg.prox != BSUB_PROX_FLAT_LINF) { set_error("bsub_set_flat_groups: solver was not created with BSUB_PROX_FLAT_LINF"); return -1; }
    const long long m = s->m;
    const int rows = s->cfg.rows, cols = s->cfg.cols;
    // is it the regular 3x3 tiling of get_proximal_flat_groups_nonoverlap (lsd_improvement.py:24-34)?
    bool regular = ((long long)rows * cols == m);
    if (regular) {
        const int ntr = (rows + 2) / 3;
        for (int j = 0; j < cols && regular; ++j)
            for (int i = 0; i < rows; ++i)
                if (g[(long long)j * rows + i] != (j / 3) * ntr + (i / 3) + 1) { regular = false; break; }
    }
    s->groups_set = true;
    if (regular) { s->shrink_mode = SHRINK_FLAT3; return 0; }
    // generic partition: CSR of the ids >= 1
    int gmax = 0;
    for (long long p = 0; p < m; ++p) { if (g[p] < 0) { set_error("bsub_set_flat_groups: negative group id"); return -1; } gmax = std::max(gmax, (int)g[p]); }
    std::vector<int> ptr((size_t)gmax + 1, 0), idx;
    for (long long p = 0; p < m; ++p) if (g[p] > 0) ptr[g[p]]++;       // ptr[k] = size of group k (k >= 1)
    std::vector<int> start((size_t)gmax + 1, 0);
    int acc = 0;
    for (int k = 1; k <= gmax; ++k) { start[k - 1] = acc; acc += ptr[k]; }
    start[gmax] = acc;
    idx.resize((size_t)std::max(acc, 1));
    std::vector<int> fill(start.begin(), start.end());
    for (long long p = 0; p < m; ++p) if (g[p] > 0) idx[fill[g[p] - 1]++] = (int)p;
    if (s->gptr) cudaFree(s->gptr);
    if (s->gidx) cudaFree(s->gidx);
    CK(cudaMalloc((void**)&s->gptr, sizeof(int) * ((size_t)gmax + 1)));
    CK(cudaMalloc((void**)&s->gidx, sizeof(int) * idx.size()));
    CK(cudaMemcpy(s->gptr, start.data(), sizeof(int) * ((size_t)gmax + 1), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(s->gidx, idx.data(), sizeof(int) * idx.size(), cudaMemcpyHostToDevice));
    s->ngroups = gmax;
    s->shrink_mode = SHRINK_SPILL;
    s->implied_first = false;      // the two-phase path reads Y from HBM: init_Y must store Y0 = D / dual_norm
    s->stmaps_ready = false;
    const size_t mat = sizeof(float) * (size_t)s->ld * s->n;
    if (!s->U) { CK(cudaMalloc((void**)&s->U, mat)); CK(cudaMemset(s->U, 0, mat)); }
    if (!s->L) { CK(cudaMalloc((void**)&s->L, mat)); CK(cudaMemset(s->L, 0, mat)); }
    return 0;
}

static int check_prox(bsub_solver* s, int prox, const char* prox_name, const char* who) {
    if (!s) { set_error("%s: null solver", who); return -1; }
    if (s->cfg.prox != prox) { set_error("%s: solver was not created with %s", who, prox_name); return -1; }
    return 0;
}

// d becomes the handle's description and the previous one is released.  A whole-clip one gets the duals of all n frames at the
// handle's ld here, so that bsub_run allocates nothing inside its loop.
static int set_graph(bsub_solver* s, const GraphDesc& d, bool whole) {
    s->graph.release();
    s->graph = d;
    s->graph_whole = whole;
    if (!whole) return 0;
    long long xi_floats = 0;
    GenericGraphLayout L;
    return size_work(s->graph, s->ld, s->n, &s->work, &xi_floats, &L);
}

// a frame-range description only: the handle has no graph of its own pixels
static bool frame_range_only(const bsub_solver* s) { return s->graph.kind != 0 && !s->graph_whole; }

int bsub_set_graph_windows(bsub_solver* s, const double* eta, int64_t n_eta) {
    RET_IF(check_prox(s, BSUB_PROX_GRAPH_LINF, "BSUB_PROX_GRAPH_LINF", "bsub_set_graph_windows"));
    GraphDesc d;
    RET_IF(describe_windows(&d, s->cfg.rows, s->cfg.cols, 0, s->n, eta, n_eta, "bsub_set_graph_windows"));
    return set_graph(s, d, true);
}

int bsub_set_center_windows(bsub_solver* s, const float* eta, const uint8_t* background) {
    if (!s || !eta || !background) { set_error("bsub_set_center_windows: null argument"); return -1; }
    RET_IF(check_prox(s, BSUB_PROX_GRAPH_CENTER_BG, "BSUB_PROX_GRAPH_CENTER_BG", "bsub_set_center_windows"));
    GraphDesc d;
    RET_IF(describe_centre(&d, s->cfg.rows, s->cfg.cols, 0, s->n, eta, background, "bsub_set_center_windows"));
    return set_graph(s, d, true);
}

int bsub_set_graphs(bsub_solver* s, int32_t n_graphs, const int32_t* frame_graph, const int64_t* n_groups, const int32_t* const* indptr,
                    const int32_t* const* indices, const double* const* eta, const uint8_t* background) {
    RET_IF(check_prox(s, BSUB_PROX_GRAPH_GENERIC, "BSUB_PROX_GRAPH_GENERIC", "bsub_set_graphs"));
    GraphDesc d;                  // the handle's m: the generic kernel needs no image geometry
    RET_IF(describe_graphs(&d, s->cfg.rows, s->cfg.cols, s->m, 0, s->n, n_graphs, frame_graph, n_groups, indptr, indices, eta, background,
                           "bsub_set_graphs"));
    return set_graph(s, d, true);
}

// ---------------------------------------------------------------------------- frame-range descriptions (bsub_step_prox_block)
static int frame_range_check(bsub_solver* s, int prox, const char* prox_name, int32_t rows, int32_t cols, int32_t f0, int32_t nf,
                             const char* who) {
    RET_IF(check_prox(s, prox, prox_name, who));
    if (rows <= 0 || cols <= 0 || (long long)rows * cols > (1LL << 30)) { set_error("%s: bad frame geometry %d x %d", who, rows, cols); return -1; }
    if (f0 < 0 || nf < 0 || (long long)f0 + nf > s->n) {
        set_error("%s: frames [%d, %lld) are not a range of the %d frames of the clip", who, f0, (long long)f0 + nf, s->n); return -1;
    }
    return 0;
}

int bsub_set_frame_windows(bsub_solver* s, int32_t rows, int32_t cols, int32_t f0, int32_t nf, const double* eta, int64_t n_eta) {
    RET_IF(frame_range_check(s, BSUB_PROX_GRAPH_LINF, "BSUB_PROX_GRAPH_LINF", rows, cols, f0, nf, "bsub_set_frame_windows"));
    GraphDesc d;
    RET_IF(describe_windows(&d, rows, cols, f0, nf, eta, n_eta, "bsub_set_frame_windows"));
    return set_graph(s, d, false);
}

int bsub_set_frame_center_windows(bsub_solver* s, int32_t rows, int32_t cols, int32_t f0, int32_t nf, const float* eta, const uint8_t* background) {
    RET_IF(frame_range_check(s, BSUB_PROX_GRAPH_CENTER_BG, "BSUB_PROX_GRAPH_CENTER_BG", rows, cols, f0, nf, "bsub_set_frame_center_windows"));
    if (nf > 0 && (!eta || !background)) { set_error("bsub_set_frame_center_windows: null argument"); return -1; }
    GraphDesc d;
    RET_IF(describe_centre(&d, rows, cols, f0, nf, eta, background, "bsub_set_frame_center_windows"));
    return set_graph(s, d, false);
}

int bsub_set_frame_weight_map_dev(bsub_solver* s, int32_t rows, int32_t cols, int32_t f0, int32_t nf, const float* weight, int64_t ld,
                                  void* stream) {
    const char* who = "bsub_set_frame_weight_map_dev";
    RET_IF(frame_range_check(s, BSUB_PROX_GRAPH_CENTER_BG, "BSUB_PROX_GRAPH_CENTER_BG", rows, cols, f0, nf, who));
    const long long m = (long long)rows * cols;
    if (nf > 0 && !weight) { set_error("%s: null argument", who); return -1; }
    if (nf > 0 && ld < m) { set_error("%s: ld = %lld is less than rows*cols = %lld", who, (long long)ld, m); return -1; }
    GraphDesc d{BSUB_PROX_GRAPH_CENTER_BG, rows, cols, f0, nf, m};
    d.eta_stride = m;
    if (nf > 0) {
        cudaStream_t st = use_stream(s, stream);
        DevScope scope;
        unsigned long long* bad_dev = nullptr;
        unsigned long long bad = 0;
        const size_t nm = (size_t)nf * m;
        // the same buffers describe_upload makes from a host map with a background array: eta, labels and their per-frame sums
        const int rc = [&]() -> int {
            RET_IF(scope.alloc(&bad_dev, sizeof(unsigned long long)));
            CK(cudaMalloc((void**)&d.eta, sizeof(float) * nm));
            CK(cudaMalloc((void**)&d.labels, nm));
            CK(cudaMalloc((void**)&d.bsums, sizeof(double) * nf));
            CK(cudaMemsetAsync(bad_dev, 0xff, sizeof(unsigned long long), st));
            RET_IF(launch_weight_map_describe(weight, ld, m, nf, d.eta, d.labels, bad_dev, st));
            CK(cudaMemcpyAsync(&bad, bad_dev, sizeof(bad), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (bad == ~0ULL) return 0;
            const long long f = (long long)(bad / (unsigned long long)m), p = (long long)(bad % (unsigned long long)m);
            float v = 0.f;
            CK(cudaMemcpyAsync(&v, weight + (size_t)f * ld + p, sizeof(float), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            set_error("%s: weight[%lld][%lld] (frame %lld, pixel %lld) = %g is not finite", who, f, p, f0 + f, p, (double)v);
            return -1;
        }();
        if (rc != 0) { d.release(); return rc; }       // the handle keeps its previous description
    }
    return set_graph(s, d, false);
}

int bsub_set_frame_graphs(bsub_solver* s, int32_t rows, int32_t cols, int32_t f0, int32_t nf, int32_t n_graphs, const int32_t* frame_graph,
                          const int64_t* n_groups, const int32_t* const* indptr, const int32_t* const* indices, const double* const* eta,
                          const uint8_t* background) {
    RET_IF(frame_range_check(s, BSUB_PROX_GRAPH_GENERIC, "BSUB_PROX_GRAPH_GENERIC", rows, cols, f0, nf, "bsub_set_frame_graphs"));
    GraphDesc d;
    RET_IF(describe_graphs(&d, rows, cols, (long long)rows * cols, f0, nf, n_graphs, frame_graph, n_groups, indptr, indices, eta, background,
                           "bsub_set_frame_graphs"));
    return set_graph(s, d, false);
}

int bsub_set_blocks(bsub_solver* s, const uint8_t* labels, const int32_t* lam_ptr, const double* lam) {
    if (!s || !labels || !lam_ptr) { set_error("bsub_set_blocks: null argument"); return -1; }
    if (s->cfg.prox != BSUB_PROX_BLOCK_L2) { set_error("bsub_set_blocks: solver was not created with BSUB_PROX_BLOCK_L2"); return -1; }
    int maxb = 0;
    for (int f = 0; f < s->n; ++f) maxb = std::max(maxb, lam_ptr[f + 1] - lam_ptr[f]);
    if (maxb > 254) { set_error("bsub_set_blocks: more than 254 blocks in one frame"); return -1; }
    s->nlab = maxb + 1;
    std::vector<double> table((size_t)s->n * s->nlab, 0.0);
    for (int f = 0; f < s->n; ++f)
        for (int b = 0; b < lam_ptr[f + 1] - lam_ptr[f]; ++b) table[(size_t)f * s->nlab + b + 1] = lam[lam_ptr[f] + b];
    if (s->labels_dev) cudaFree(s->labels_dev);
    if (s->lam_table) cudaFree(s->lam_table);
    if (s->bsums) cudaFree(s->bsums);
    CK(cudaMalloc((void**)&s->labels_dev, (size_t)s->n * s->m));
    CK(cudaMalloc((void**)&s->lam_table, sizeof(double) * table.size()));
    CK(cudaMalloc((void**)&s->bsums, sizeof(double) * table.size()));
    CK(cudaMemcpy(s->labels_dev, labels, (size_t)s->n * s->m, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(s->lam_table, table.data(), sizeof(double) * table.size(), cudaMemcpyHostToDevice));
    s->blocks_set = true;
    return 0;
}

// --------------------------------------------------------------------------------------------------- data in
static int after_load(bsub_solver* s) { s->loaded = true; s->finalized = false; s->initialised = false; return 0; }

int bsub_load_D_f32_dev(bsub_solver* s, const float* D, int64_t ld, void* stream) {
    if (!s || !D || ld < s->m) { set_error("bsub_load_D_f32_dev: bad argument"); return -1; }
    RET_IF(launch_copy_f32(D, ld, s->D, s->ld, s->m, s->n, as_stream(stream)));
    return after_load(s);
}

int bsub_load_D_f32_host(bsub_solver* s, const float* D, int64_t ld, void* stream) {
    if (!s || !D || ld < s->m) { set_error("bsub_load_D_f32_host: bad argument"); return -1; }
    cudaStream_t st = use_stream(s, stream);
    if (s->ld != s->m) CK(cudaMemsetAsync(s->D, 0, sizeof(float) * (size_t)s->ld * s->n, st));
    if (ld == s->m && s->ld == s->m) CK(cudaMemcpyAsync(s->D, D, sizeof(float) * (size_t)s->m * s->n, cudaMemcpyHostToDevice, st));
    else CK(cudaMemcpy2DAsync(s->D, sizeof(float) * s->ld, D, sizeof(float) * ld, sizeof(float) * s->m, s->n, cudaMemcpyHostToDevice, st));
    return after_load(s);
}

int bsub_load_D_f64_host(bsub_solver* s, const double* D, int64_t ld, void* stream) {
    if (!s || !D || ld < s->m) { set_error("bsub_load_D_f64_host: bad argument"); return -1; }
    cudaStream_t st = use_stream(s, stream);
    // narrow on the device through a staging buffer that is allocated once: two halves alternate so that the conversion
    // of one batch overlaps the copy of the next; a batch is a whole number of frames, or a piece of one long frame
    const size_t half = (size_t)4 << 20;                       // doubles per half (32 MB)
    RET_IF(ensure_stage64(s, 2 * half));
    if (s->ld != s->m) CK(cudaMemsetAsync(s->D, 0, sizeof(float) * (size_t)s->ld * s->n, st));
    int flip = 0;
    if ((size_t)s->m <= half) {
        const long long cap_frames = (long long)(half / (size_t)s->m);
        for (long long f0 = 0; f0 < s->n; f0 += cap_frames, flip ^= 1) {
            const int nf = (int)std::min<long long>(cap_frames, s->n - f0);
            double* stage = s->stage64 + (size_t)flip * half;
            CK(cudaMemcpy2DAsync(stage, sizeof(double) * s->m, D + (size_t)f0 * ld, sizeof(double) * ld, sizeof(double) * s->m, nf,
                                 cudaMemcpyHostToDevice, st));
            RET_IF(launch_convert_f64(stage, s->m, s->D + (size_t)f0 * s->ld, s->ld, s->m, nf, st));
        }
    } else {
        for (long long f = 0; f < s->n; ++f)
            for (long long p0 = 0; p0 < s->m; p0 += (long long)half, flip ^= 1) {
                const long long np = std::min<long long>((long long)half, s->m - p0);
                double* stage = s->stage64 + (size_t)flip * half;
                CK(cudaMemcpyAsync(stage, D + (size_t)f * ld + p0, sizeof(double) * np, cudaMemcpyHostToDevice, st));
                RET_IF(launch_convert_f64(stage, np, s->D + (size_t)f * s->ld + p0, s->ld, np, 1, st));
            }
    }
    return after_load(s);
}

int bsub_load_u8_host(bsub_solver* s, const uint8_t* frames, double* lo, double* hi, double* mean_raw, int force, void* stream) {
    if (!s || !frames) { set_error("bsub_load_u8_host: bad argument"); return -1; }
    cudaStream_t st = use_stream(s, stream);
    unsigned char* stage = reinterpret_cast<unsigned char*>(s->T);
    const long long count = (long long)s->m * s->n;
    CK(cudaMemcpyAsync(stage, frames, (size_t)count, cudaMemcpyHostToDevice, st));
    double vlo, vhi, vmean;
    if (force && lo && hi && mean_raw) { vlo = *lo; vhi = *hi; vmean = *mean_raw; }
    else {
        unsigned long long* acc = reinterpret_cast<unsigned long long*>(s->comm_max);   // scratch: 3 x u64
        unsigned long long init[3] = {0ull, 255ull, 0ull}, res[3];
        CK(cudaMemcpyAsync(acc, init, sizeof(init), cudaMemcpyHostToDevice, st));
        RET_IF(launch_u8_stats(stage, count, acc, st));
        CK(cudaMemcpyAsync(res, acc, sizeof(res), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        CK(cudaMemsetAsync(s->comm_max, 0, sizeof(double) * 8, st));
        vlo = (double)res[1]; vhi = (double)res[2]; vmean = (double)res[0] / (double)count;
        if (lo) *lo = vlo; if (hi) *hi = vhi; if (mean_raw) *mean_raw = vmean;
    }
    // normalizeImage: x -= min; x *= 1/max(x)  (utils.py:220-223); then subtract the mean of the normalised cube
    const double scale = (vhi > vlo) ? 1.0 / (vhi - vlo) : 0.0;
    const double mean_n = (vmean - vlo) * scale;
    RET_IF(launch_u8_to_D(stage, s->D, s->ld, s->m, s->n, vlo, scale, mean_n, st));
    CK(cudaMemsetAsync(s->T, 0, sizeof(float) * (size_t)s->ld * s->n, st));     // T was the staging buffer
    return after_load(s);
}

// --------------------------------------------------------------------------------------------------- steps
static int upload_state(bsub_solver* s, cudaStream_t st) {
    DevState h;
    memset(&h, 0, sizeof(h));
    const bsub_config& c = s->cfg;
    const double mx = (double)std::max<long long>(c.m_global, c.n);
    h.lambda = 1.0 / (sqrt(mx) * c.delta);
    h.non_block_lambda = c.non_block_lambda_scale * h.lambda;
    h.rho = c.rho; h.tol = c.tol; h.mu_scale = c.mu_scale;
    h.max_iter = c.max_iter;
    h.d = c.d_global > 0 ? c.d_global : (int)std::min<long long>(c.m_global, c.n);
    h.round005d = round_half_even_005(h.d);
    h.use_sv_prediction = c.use_sv_prediction;
    h.break_on_rank0 = c.break_on_rank0;
    h.sv = c.use_sv_prediction ? c.sv0 : h.d;
    h.use_i8 = s->use_i8 ? 1 : 0;
    CK(cudaMemcpyAsync(s->st, &h, sizeof(h), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));     // h is a stack object
    memset((void*)s->mirror, 0, sizeof(HostMirror));
    return 0;
}

int bsub_set_always_store_S(bsub_solver* s, int on) {
    if (!s) { set_error("bsub_set_always_store_S: null solver"); return -1; }
    s->force_S = on != 0;
    return 0;
}

int bsub_comm_buffers(bsub_solver* s, double** sum_buf, int64_t* sum_count, double** max_buf, int64_t* max_count) {
    if (!s) { set_error("bsub_comm_buffers: null solver"); return -1; }
    if (sum_buf) *sum_buf = s->comm_sum;
    if (sum_count) *sum_count = (int64_t)s->npad * s->npad + kCommTail;
    if (max_buf) *max_buf = s->comm_max;
    if (max_count) *max_count = 8;
    return 0;
}

static int check_ready(bsub_solver* s) {
    if (!s) { set_error("null solver"); return -1; }
    if (!s->loaded) { set_error("no data loaded (call bsub_load_* first)"); return -1; }
    if (s->cfg.prox == BSUB_PROX_FLAT_LINF && !s->groups_set) { set_error("one of graphs or groups must not be None"); return -1; }
    if ((s->cfg.prox == BSUB_PROX_GRAPH_LINF || s->cfg.prox == BSUB_PROX_GRAPH_CENTER_BG || s->cfg.prox == BSUB_PROX_GRAPH_GENERIC) &&
        s->graph.kind == 0) { set_error("one of graphs or groups must not be None"); return -1; }
    if (s->cfg.prox == BSUB_PROX_BLOCK_L2 && !s->blocks_set) { set_error("blocks_by_frame / lambdas_by_frame not set"); return -1; }
    return 0;
}

int bsub_step_init_local(bsub_solver* s, void* stream) {
    RET_IF(check_ready(s));
    cudaStream_t st = use_stream(s, stream);
    RET_IF(upload_state(s, st));
    CK(cudaMemsetAsync(s->comm_max, 0, sizeof(double) * 8, st));
    CK(cudaMemsetAsync(s->comm_sum + (size_t)s->npad * s->npad, 0, sizeof(double) * kCommTail, st));
    RET_IF(launch_rowsum_max(s->D, s->ld, s->m, s->n, s->comm_max, st));
    if (s->use_i8) {
        // Gram(D) on the int8 tensor-core path: quantise D into the slice planes (scale from max|D|), then the exact Gram
        RET_IF(launch_quantize_D(s->D, s->ld, s->n, s->gip.ldq, s->Wq, s->comm_max + 2, s->st, st));
        RET_IF(launch_gram_i8(s->gip, s->gimap, s->gimap_last, s->gi_info, s->gi_ncta, s->gi_blkn, s->Gint, s->comm_sum, s->npad, s->st, 0.0, 0,
                              st));
    } else {
        RET_IF(launch_gram(s->gp, s->gmaps, false, s->tasks_dev, nullptr, 0.f, s->gram_partial, s->comm_sum, st));
    }
    s->iters_enqueued = 0;
    s->proj_iter = -1;
    s->finalized = false;
    return 0;
}

int bsub_step_init_finish(bsub_solver* s, void* stream) {
    RET_IF(check_ready(s));
    cudaStream_t st = use_stream(s, stream);
    RET_IF(launch_eig(s->ep, s->comm_sum, s->comm_max, s->eb, s->st, 0, 1, st));
    // S0 = 0 and Y0 = D / dual_norm are only materialised when some kernel of iteration 1 reads them: with the int8 path
    // iteration 1 has no Gram pass and the streamed shrink kernel forms both from D on the fly
    if (!s->implied_first) RET_IF(launch_init_Y(s->D, s->Y, s->S, s->ld, s->n, s->st, st));
    s->initialised = true;
    return 0;
}

int bsub_step_gram(bsub_solver* s, void* stream) {
    if (!s || !s->initialised) { set_error("bsub_step_gram: solver not initialised"); return -1; }
    use_stream(s, stream);
    // both Gram kernels are enqueued; DevState.gram_mode (set on the device) decides which one does the work
    RET_IF(launch_gram(s->gp, s->gmaps, true, s->tasks_dev, s->st, 0.f, s->gram_partial, s->comm_sum, as_stream(stream)));
    if (s->use_i8)
        RET_IF(launch_gram_i8(s->gip, s->gimap, s->gimap_last, s->gi_info, s->gi_ncta, s->gi_blkn, s->Gint, s->comm_sum, s->npad, s->st, 0.0, 1,
                              as_stream(stream)));
    return 0;
}

int bsub_step_solve(bsub_solver* s, void* stream) {
    if (!s || !s->initialised) { set_error("bsub_step_solve: solver not initialised"); return -1; }
    return launch_eig(s->ep, s->comm_sum, s->comm_max, s->eb, s->st, 1, 0, as_stream(stream));
}

// T = Vr^T W from the digit planes (project.cu) as a step of its own, so that a driver can time it; bsub_step_shrink launches it
// itself when the driver did not.
int bsub_step_project(bsub_solver* s, void* stream) {
    if (!s || !s->initialised) { set_error("bsub_step_project: solver not initialised"); return -1; }
    cudaStream_t st = use_stream(s, stream);
    const bool proj = s->use_proj && s->use_stream && s->use_i8 && s->shrink_mode != SHRINK_SPILL;
    if (!proj || s->proj_iter == s->iters_enqueued) return 0;
    RET_IF(launch_project(s->pjp, s->Wq, s->eb.Vr, s->eb.vstride, s->T, s->ld, s->Tt, s->ssp.rows, s->ssp.cols, s->ssp.R, s->ssp.ntile_r,
                          s->ssp.ntiles, s->ssp.kcap, s->st, st));
    s->proj_iter = s->iters_enqueued;
    return 0;
}

// part: 0 = the whole pass; 1 / 2 = the two halves of the l2-block mode around the all-reduce of the per-(frame, group) sums of
// squares (pixel-sharded drivers: a block -- and the frame-wide complement group -- spans the shards).  For every other mode part 1
// is the whole pass and part 2 does nothing.
static int step_shrink_impl(bsub_solver* s, void* stream, int part) {
    if (!s || !s->initialised) { set_error("bsub_step_shrink: solver not initialised"); return -1; }
    cudaStream_t st = use_stream(s, stream);
    // the overlapping-window mode splits too: between the halves the driver re-shards G_S by FRAMES (the prox of a frame needs the
    // whole image), runs bsub_step_prox_block and brings S back; so does every graph mode with a frame-range description
    const bool split = s->shrink_mode == SHRINK_SPILL &&
                       (s->cfg.prox == BSUB_PROX_BLOCK_L2 || s->cfg.prox == BSUB_PROX_GRAPH_LINF || frame_range_only(s));
    if (part == 2 && !split) return 0;
    if (part == 0 && frame_range_only(s)) {
        set_error("bsub_step_shrink: the handle holds only a frame-range description; use _shrink_a, bsub_step_prox_block, _shrink_b");
        return -1;
    }
    if (part == 2) {
        if (s->cfg.prox == BSUB_PROX_BLOCK_L2)
            RET_IF(launch_block_l2_apply(s->U, s->S, s->labels_dev, s->ld, s->m, s->n, s->nlab, s->bsums, s->lam_table, s->st, 0.0, 0.0, st));
        const int np2 = s->num_sms * 8;
        RET_IF(launch_dual_update(s->D, s->S, s->S, s->Y, s->T, s->eb.VC, s->eb.vstride, s->st, s->L, s->ld, s->n, s->part_zz,
                                  s->part_nnz, s->part_max, np2, st));
        RET_IF(launch_control_post(s->st, s->part_zz, s->part_nnz, s->part_max, np2, s->comm_sum + (size_t)s->npad * s->npad, s->log,
                                   s->mirror_dev, 1 | 4, nullptr, 0, st));
        return 0;
    }
    ShrinkBuffers b;
    b.D = s->D; b.S = s->S; b.Y = s->Y; b.T = s->T; b.U = s->U; b.tpart = s->tpart; b.Vr = s->eb.Vr; b.VC = s->eb.VC;
    b.vstride = s->eb.vstride; b.part_zz = s->part_zz; b.part_nnz = s->part_nnz; b.part_max = s->part_max;
    b.part_wmax = s->use_i8 ? s->part_wmax : nullptr;
    b.implied_first = s->implied_first ? 1 : 0;
    const bool proj = s->use_proj && s->use_stream && s->use_i8 && s->shrink_mode != SHRINK_SPILL;
    const bool flat = proj && s->use_flat;
    b.Tt = proj ? s->Tt : nullptr;
    b.have_flat = flat ? 1 : 0;
    int nparts = s->sp.nparts;
    if (s->use_tma) {
        if (!s->stmaps_ready) {
            RET_IF(make_shrink_tma_maps(s->stp, s->D, s->S, s->Y, s->U, &s->stmaps));
            if (s->use_stream) RET_IF(make_shrink_stream_maps(s->ssp, s->D, s->S, s->Y, s->U, &s->ssmaps));
            if (s->use_stream) RET_IF(make_shrink_stream_vmaps(s->ssp, s->eb.Vr, s->eb.VC, s->eb.vstride, &s->ssmaps));
            if (s->use_stream && s->use_i8) RET_IF(make_shrink_stream_qmap(s->ssp, s->Wq, &s->ssmaps));
            s->stmaps_ready = true;
        }
        int off = 0, min_rank = 0;
        if (s->use_stream) {          // rank <= 16: streamed kernel; larger ranks fall through to the cluster kernel
            if (proj)                 // T = Vr^T W from the planes the Gram just read (skips itself when they do not exist)
                RET_IF(bsub_step_project(s, stream));
            RET_IF(launch_shrink_stream(s->ssp, s->ssmaps, b, s->st, s->shrink_mode, st));
            off = s->ssp.nparts; min_rank = s->ssp.kcap + 1;
            if (flat) {               // rank <= 8 from the second iteration on: the single-pass kernel (the one above then exits at once)
                if (!s->sfmaps_ready) {
                    RET_IF(make_shrink_flat_maps(s->sfp, s->D, s->S, s->Y, s->Wq, s->gip.ldq, s->eb.VC, s->eb.vstride, &s->sfmaps));
                    s->sfmaps_ready = true;
                }
                RET_IF(launch_shrink_flat(s->sfp, s->sfmaps, s->Tt, s->st, s->shrink_mode, s->force_S ? 1 : 0, s->part_zz + off, s->part_nnz + off,
                                          s->part_max + off, s->part_wmax + s->ssp.grid, st));
                off += s->sfp.grid;
                // the rank > 16 fallback below reads S from HBM: bring it up to date if the single-pass kernel has been skipping its store
                if (!s->force_S) RET_IF(launch_rebuild_S(s->sfp, s->D, s->Y, s->S, s->Wq, s->gip.ldq, s->st, s->ssp.kcap + 1, st));
            }
        }
        ShrinkBuffers b2 = b;
        b2.part_zz += off; b2.part_nnz += off; b2.part_max += off;
        RET_IF(launch_shrink_tma(s->stp, s->stmaps, b2, s->st, s->shrink_mode, min_rank, st));
        nparts = off + s->stp.nparts;
    } else {
        RET_IF(launch_shrink(s->sp, b, s->st, s->shrink_mode, st));
    }
    if (s->shrink_mode == SHRINK_SPILL) {
        // two-phase: U = G_S -> prox -> S_new (written over S) -> dual update
        if (s->cfg.prox == BSUB_PROX_FLAT_LINF) {
            RET_IF(launch_prox_groups_csr(s->U, s->S, s->ld, s->m, s->n, s->gptr, s->gidx, s->ngroups, 0.f, s->st, st));
        } else if (s->cfg.prox == BSUB_PROX_BLOCK_L2) {
            RET_IF(launch_block_l2_sums(s->U, s->labels_dev, s->ld, s->m, s->n, s->nlab, s->bsums, s->st, st));
            if (part == 1) return 0;                       // the driver all-reduces bsums, then calls part 2
            RET_IF(launch_block_l2_apply(s->U, s->S, s->labels_dev, s->ld, s->m, s->n, s->nlab, s->bsums, s->lam_table, s->st, 0.0,
                                         0.0, st));
        } else {   // graph modes
            if (part == 1 && split) return 0;              // the driver runs the prox on frame shards, then calls part 2
            RET_IF(graph_prox(s->graph, s->U, s->S, s->ld, 0, s->n, s->st, 0.f, s->cfg.graph_max_sweeps, (float)s->cfg.graph_tol,
                              s->sweeps_dev, &s->work, st));
        }
        nparts = s->num_sms * 8;
        RET_IF(launch_dual_update(s->D, s->S, s->S, s->Y, s->T, s->eb.VC, s->eb.vstride, s->st, s->L, s->ld, s->n, s->part_zz,
                                  s->part_nnz, s->part_max, nparts, st));
    }
    RET_IF(launch_control_post(s->st, s->part_zz, s->part_nnz, s->part_max, nparts, s->comm_sum + (size_t)s->npad * s->npad, s->log,
                               s->mirror_dev, 1 | 4, (s->use_i8 && s->use_stream) ? s->part_wmax : nullptr,
                               s->use_i8 ? s->ssp.grid + (flat ? s->sfp.grid : 0) : 0, st));
    return 0;
}

int bsub_step_shrink(bsub_solver* s, void* stream) { return step_shrink_impl(s, stream, 0); }
int bsub_step_shrink_a(bsub_solver* s, void* stream) { return step_shrink_impl(s, stream, 1); }
int bsub_step_shrink_b(bsub_solver* s, void* stream) { return step_shrink_impl(s, stream, 2); }

int bsub_step_prox_buffers(bsub_solver* s, float** G_S, float** S, int64_t* ld) {
    if (!s || !s->initialised) { set_error("bsub_step_prox_buffers: solver not initialised"); return -1; }
    if (G_S) *G_S = s->U;
    if (S) *S = s->S;
    if (ld) *ld = s->ld;
    return 0;
}

int bsub_step_prox_block(bsub_solver* s, const float* Uf, float* Vf, int64_t ldf, int32_t f0, int32_t nf, void* stream) {
    if (!s || !s->initialised) { set_error("bsub_step_prox_block: solver not initialised"); return -1; }
    if (!frame_range_only(s)) { set_error("bsub_step_prox_block: the handle has no frame-range description (bsub_set_frame_*)"); return -1; }
    const GraphDesc& d = s->graph;
    if (nf < 0 || f0 < d.f0 || (long long)f0 + nf > (long long)d.f0 + d.nf) {
        set_error("bsub_step_prox_block: frames [%d, %lld) are outside the described range [%d, %d)", f0, (long long)f0 + nf, d.f0, d.f0 + d.nf);
        return -1;
    }
    if (nf == 0) return 0;
    if (!Uf || !Vf || ldf < d.m) { set_error("bsub_step_prox_block: bad argument"); return -1; }
    // lambda / mu and the stop flag come from the device state, exactly as in the unsharded pass
    return graph_prox(d, Uf, Vf, ldf, f0, nf, s->st, 0.f, s->cfg.graph_max_sweeps, (float)s->cfg.graph_tol, s->sweeps_dev, &s->work,
                      use_stream(s, stream));
}

int bsub_block_sums_buffer(bsub_solver* s, double** sums, int64_t* count) {
    if (!s) { set_error("bsub_block_sums_buffer: null solver"); return -1; }
    const bool have = s->cfg.prox == BSUB_PROX_BLOCK_L2 && s->bsums != nullptr;
    if (sums) *sums = have ? s->bsums : nullptr;
    if (count) *count = have ? (int64_t)s->n * s->nlab : 0;
    return 0;
}

int bsub_step_finish_iter(bsub_solver* s, void* stream) {
    if (!s || !s->initialised) { set_error("bsub_step_finish_iter: solver not initialised"); return -1; }
    cudaStream_t st = use_stream(s, stream);
    RET_IF(launch_control_post(s->st, s->part_zz, s->part_nnz, s->part_max, 0, s->comm_sum + (size_t)s->npad * s->npad, s->log,
                               s->mirror_dev, 2, nullptr, 0, st));
    CK(cudaEventRecord(s->ev[s->iters_enqueued % (kRunAhead + 1)], st));
    s->iters_enqueued++;
    return 0;
}

static void fill_status(bsub_solver* s, bsub_status* out, const DevState* h) {
    memset(out, 0, sizeof(*out));
    if (h) {
        out->iter = h->iter; out->converged = h->converged; out->done = h->done; out->svp = h->svp_L; out->err = h->err; out->mu = h->mu;
        out->norm_two = h->norm_two; out->norm_fro = sqrt(h->normD2); out->norm_rowsum = h->norm_rowsum; out->lambda = h->lambda;
    } else {
        out->iter = s->mirror->iter; out->converged = s->mirror->converged; out->done = s->mirror->done; out->svp = s->mirror->svp;
        out->err = s->mirror->err;
    }
}

int bsub_poll(bsub_solver* s, bsub_status* out) {
    if (!s || !out) { set_error("bsub_poll: null argument"); return -1; }
    fill_status(s, out, nullptr);
    return 0;
}

int bsub_sync_status(bsub_solver* s, bsub_status* out, void* stream) {
    if (!s || !out) { set_error("bsub_sync_status: null argument"); return -1; }
    DevState h;
    CK(cudaMemcpyAsync(&h, s->st, sizeof(h), cudaMemcpyDeviceToHost, as_stream(stream)));
    CK(cudaStreamSynchronize(as_stream(stream)));
    fill_status(s, out, &h);
    return 0;
}

int bsub_run(bsub_solver* s, void* stream) {
    if (s && frame_range_only(s)) {
        set_error("bsub_run: the handle holds only a frame-range description (bsub_set_frame_*), not the graphs of its own pixels");
        return -1;
    }
    for (int attempt = 0; attempt < 2; ++attempt) {
        RET_IF(bsub_step_init_local(s, stream));
        RET_IF(bsub_step_init_finish(s, stream));
        const int max_iter = s->cfg.max_iter;
        for (int it = 0; it < max_iter + 1; ++it) {
            // bounded run-ahead: wait for iteration it - kRunAhead, then look at the mapped stop flag (no device sync)
            if (it >= kRunAhead) {
                CK(cudaEventSynchronize(s->ev[(it - kRunAhead) % (kRunAhead + 1)]));
                if (s->mirror->done) break;
            }
            RET_IF(bsub_step_gram(s, stream));
            RET_IF(bsub_step_solve(s, stream));
            RET_IF(bsub_step_shrink(s, stream));
            RET_IF(bsub_step_finish_iter(s, stream));
        }
        if (!s->use_flat || s->force_S) return 0;
        // the single-pass shrink skips the store of S in iterations that cannot be the last; a clipped digit pass in such an
        // iteration (never seen: the fixed-point scale has 4x head-room) leaves the state unrecoverable -> the device stops with
        // done == 5 and the solve is repeated with S stored every time.  This needs the final flag: drain the last iterations.
        CK(cudaEventSynchronize(s->ev[(s->iters_enqueued + kRunAhead) % (kRunAhead + 1)]));
        if (s->mirror->done != 5) return 0;
        s->force_S = true;
    }
    return 0;
}

// --------------------------------------------------------------------------------------------------- results
int bsub_finalize(bsub_solver* s, void* stream) {
    if (!s || !s->initialised) { set_error("bsub_finalize: nothing has been solved"); return -1; }
    if (s->finalized) return 0;
    if (!s->L) { CK(cudaMalloc((void**)&s->L, sizeof(float) * (size_t)s->ld * s->n)); }
    // S is an output: if the last shrink passes skipped its store (shrink_flat.cu), rebuild it from D, Y and the digit planes
    if (s->use_flat && s->iters_enqueued > 0 && !s->force_S)
        RET_IF(launch_rebuild_S(s->sfp, s->D, s->Y, s->S, s->Wq, s->gip.ldq, s->st, 0, as_stream(stream)));
    RET_IF(launch_materialize_L(s->T, s->eb.VC, s->eb.vstride, s->st, s->L, s->ld, s->m, s->n, as_stream(stream)));
    s->finalized = true;
    return 0;
}

static float* pick(bsub_solver* s, int which) {
    switch (which) { case 0: return s->L; case 1: return s->S; case 2: return s->D; case 3: return s->Y; default: return nullptr; }
}
int bsub_get_L_f32_dev(bsub_solver* s, float** L, int64_t* ld) {
    if (!s || !s->finalized) { set_error("bsub_get_L_f32_dev: call bsub_finalize first"); return -1; }
    *L = s->L; if (ld) *ld = s->ld; return 0;
}
int bsub_get_S_f32_dev(bsub_solver* s, float** S, int64_t* ld) {
    if (!s || (s->iters_enqueued > 0 && !s->finalized)) { set_error("bsub_get_S_f32_dev: call bsub_finalize first"); return -1; }
    *S = s->S; if (ld) *ld = s->ld; return 0;
}
int bsub_get_D_f32_dev(bsub_solver* s, float** D, int64_t* ld) { if (!s) return -1; *D = s->D; if (ld) *ld = s->ld; return 0; }
int bsub_get_Y_f32_dev(bsub_solver* s, float** Y, int64_t* ld) { if (!s) return -1; *Y = s->Y; if (ld) *ld = s->ld; return 0; }

int bsub_download_f32(bsub_solver* s, int which, float* dst, int64_t ld, void* stream) {
    if (!s || !dst || ld < s->m) { set_error("bsub_download_f32: bad argument"); return -1; }
    if (which <= 1 && !s->finalized && s->initialised) RET_IF(bsub_finalize(s, stream));
    float* src = pick(s, which);
    if (!src) { set_error("bsub_download_f32: bad selector %d", which); return -1; }
    if (ld == s->m && s->ld == s->m) CK(cudaMemcpyAsync(dst, src, sizeof(float) * (size_t)s->m * s->n, cudaMemcpyDeviceToHost, as_stream(stream)));
    else CK(cudaMemcpy2DAsync(dst, sizeof(float) * ld, src, sizeof(float) * s->ld, sizeof(float) * s->m, s->n, cudaMemcpyDeviceToHost,
                              as_stream(stream)));
    CK(cudaStreamSynchronize(as_stream(stream)));
    return 0;
}

int bsub_download_f64(bsub_solver* s, int which, double* dst, int64_t ld, void* stream) {
    if (!s || !dst || ld < s->m) { set_error("bsub_download_f64: bad argument"); return -1; }
    cudaStream_t st = use_stream(s, stream);
    if (which <= 1 && !s->finalized && s->initialised) RET_IF(bsub_finalize(s, stream));
    float* src = pick(s, which);
    if (!src) { set_error("bsub_download_f64: bad selector %d", which); return -1; }
    // widen on the device in batches through the staging buffer (allocated once, no per-call cudaMalloc and a single
    // synchronise at the end); stream order keeps a half from being overwritten before its copy has left
    const size_t half = (size_t)4 << 20;
    RET_IF(ensure_stage64(s, 2 * half));
    int rc = 0, flip = 0;
    auto piece = [&](const float* from, long long from_ld, double* to, long long to_ld, long long np, int nf) {
        double* stage = s->stage64 + (size_t)flip * half;
        if (rc == 0) rc = launch_export_f64(from, from_ld, stage, np, np, nf, st);
        if (rc == 0 && cudaMemcpy2DAsync(to, sizeof(double) * to_ld, stage, sizeof(double) * np, sizeof(double) * np, nf, cudaMemcpyDeviceToHost, st) != cudaSuccess) { set_error("bsub_download_f64: copy failed"); rc = -1; }
        flip ^= 1;
    };
    if ((size_t)s->m <= half) {
        const long long batch = (long long)(half / (size_t)s->m);
        for (long long f0 = 0; f0 < s->n && rc == 0; f0 += batch)
            piece(src + (size_t)f0 * s->ld, s->ld, dst + (size_t)f0 * ld, ld, s->m, (int)std::min<long long>(batch, s->n - f0));
    } else {
        for (long long f = 0; f < s->n && rc == 0; ++f)
            for (long long p0 = 0; p0 < s->m && rc == 0; p0 += (long long)half)
                piece(src + (size_t)f * s->ld + p0, s->ld, dst + (size_t)f * ld + p0, ld, std::min<long long>((long long)half, s->m - p0), 1);
    }
    if (cudaStreamSynchronize(st) != cudaSuccess && rc == 0) { set_error("bsub_download_f64: sync failed: %s", cudaGetErrorString(cudaGetLastError())); rc = -1; }
    return rc;
}

int bsub_debug_info(bsub_solver* s, int32_t* o) {
    if (!s || !o) { set_error("bsub_debug_info: null argument"); return -1; }
    o[0] = s->use_tma; o[1] = s->use_stream; o[2] = s->use_i8; o[3] = s->use_stream ? s->ssp.R : 0; o[4] = s->use_stream ? s->ssp.FC : 0;
    o[5] = s->use_stream ? s->ssp.NS : 0; o[6] = s->gp.ntype; o[7] = s->gp.kc; o[8] = s->ep.C; o[9] = s->use_tma ? s->stp.R : s->sp.R;
    o[10] = s->use_tma ? s->stp.Cf : s->sp.Cf; o[11] = (int32_t)s->ld; o[12] = s->use_proj ? 1 : 0; o[13] = s->use_proj ? s->pjp.NW : 0;
    o[14] = s->use_proj ? s->pjp.DEPTH : 0; o[15] = s->use_flat ? s->sfp.NS : 0;
    return 0;
}

int bsub_debug_eig_cycles(bsub_solver* s, int64_t* out16) {
    if (!s || !out16) { set_error("bsub_debug_eig_cycles: null argument"); return -1; }
    DevState h;
    CK(cudaMemcpy(&h, s->st, sizeof(h), cudaMemcpyDeviceToHost));
    for (int i = 0; i < 16; ++i) out16[i] = (int64_t)h.eig_clk[i];
    return 0;
}

int bsub_debug_counters(bsub_solver* s, int64_t* out8) {
    if (!s || !out8) { set_error("bsub_debug_counters: null argument"); return -1; }
    DevState h;
    CK(cudaMemcpy(&h, s->st, sizeof(h), cudaMemcpyDeviceToHost));
    memset(out8, 0, sizeof(int64_t) * 8);
    out8[0] = h.eig_fast_iters; out8[1] = h.eig_p; out8[2] = h.eig_info & 0xff; out8[3] = (int64_t)(h.eig_gb * 1e6);
    out8[4] = h.gram_mode; out8[5] = h.wq_saturated; out8[6] = h.force_dmma; out8[7] = (int64_t)(h.gram_err * 1e6);
    return 0;
}

int bsub_debug_graph(bsub_solver* s, int64_t* out4) {
    if (!s || !out4) { set_error("bsub_debug_graph: null argument"); return -1; }
    int h[8];
    CK(cudaMemcpy(h, s->sweeps_dev, sizeof(h), cudaMemcpyDeviceToHost));
    out4[0] = h[0]; out4[1] = h[4]; out4[2] = h[5]; out4[3] = h[6];
    return 0;
}

int bsub_get_log(bsub_solver* s, bsub_iter_log* out, int32_t cap, int32_t* count) {
    if (!s || !out || !count) { set_error("bsub_get_log: null argument"); return -1; }
    DevState h;
    CK(cudaMemcpy(&h, s->st, sizeof(h), cudaMemcpyDeviceToHost));
    std::vector<IterLog> tmp(kMaxIterLog);
    CK(cudaMemcpy(tmp.data(), s->log, sizeof(IterLog) * kMaxIterLog, cudaMemcpyDeviceToHost));
    int n = 0;
    for (int i = 0; i < kMaxIterLog && i < h.iter && n < cap; ++i) {
        if (tmp[i].iter != i + 1) break;         // an aborted (rank-0) iteration has no log line, like the reference
        out[n].iter = tmp[i].iter; out[n].svp = tmp[i].svp; out[n].sv = tmp[i].sv; out[n].reserved = 0; out[n].err = tmp[i].err;
        out[n].mu = tmp[i].mu; out[n].nnz = tmp[i].nnz; ++n;
    }
    *count = n;
    return 0;
}

// foreground mask on the solver's own buffers -------------------------------------------------------------------
int bsub_mask_stats_local(bsub_solver* s, int phase, void* stream) {
    if (!s || !s->initialised) { set_error("bsub_mask_stats_local: nothing has been solved"); return -1; }
    cudaStream_t st = use_stream(s, stream);
    if (!s->finalized) RET_IF(bsub_finalize(s, stream));
    double* tail = s->comm_sum + (size_t)s->npad * s->npad;
    if (phase == 0) {
        CK(cudaMemsetAsync(s->comm_max, 0, sizeof(double) * 8, st));
        // one shard holding the whole matrix: max |S| is what the last shrink pass reported; shards need the pass (the
        // per-iteration maximum is not all-reduced)
        if (s->cfg.m_global == s->m && s->iters_enqueued > 0)
            return launch_maxS_from_state(s->st, s->comm_max + 1, st);
        return launch_absmax(s->S, s->ld, s->m, s->n, s->comm_max + 1, st);
    }
    CK(cudaMemsetAsync(tail + 4, 0, sizeof(double) * 3, st));
    return launch_mask_stats(s->D, s->L, s->S, s->ld, s->m, s->n, s->comm_max + 1, tail + 4, s->mask_scratch, st);
}

int bsub_mask_dev(bsub_solver* s, double sigmas, uint8_t* mask_dev, void* stream) {
    if (!s || !mask_dev) { set_error("bsub_mask_dev: null argument"); return -1; }
    double* tail = s->comm_sum + (size_t)s->npad * s->npad;
    return launch_mask_write(s->S, s->ld, s->m, s->n, tail + 4, sigmas, mask_dev, s->m, as_stream(stream));
}

int bsub_mask_host(bsub_solver* s, double sigmas, uint8_t* mask_host, void* stream) {
    if (!s || !mask_host) { set_error("bsub_mask_host: null argument"); return -1; }
    cudaStream_t st = use_stream(s, stream);
    RET_IF(bsub_mask_stats_local(s, 0, stream));
    RET_IF(bsub_mask_stats_local(s, 1, stream));
    // device staging buffer, allocated once (a cudaMalloc/cudaFree per call would synchronise the whole device)
    if (!s->mask_stage) CK(cudaMalloc((void**)&s->mask_stage, (size_t)s->n * s->m));
    unsigned char* dev = s->mask_stage;
    int rc = bsub_mask_dev(s, sigmas, dev, stream);
    if (rc == 0 && cudaMemcpyAsync(mask_host, dev, (size_t)s->n * s->m, cudaMemcpyDeviceToHost, st) != cudaSuccess) { set_error("bsub_mask_host: copy failed"); rc = -1; }
    if (rc == 0 && cudaStreamSynchronize(st) != cudaSuccess) { set_error("bsub_mask_host: %s", cudaGetErrorString(cudaGetLastError())); rc = -1; }
    return rc;
}

// --------------------------------------------------------------------------------------------------- operators
int bsub_foreground_mask_dev(const float* D, const float* L, const float* S, int64_t ld, int64_t m, int32_t n, double sigmas,
                             uint8_t* mask, void* stream) {
    if (!D || !L || !S || !mask || ld < m || (ld % 4) != 0) { set_error("bsub_foreground_mask_dev: bad argument (ld must be a multiple of 4, pad columns zero)"); return -1; }
    cudaStream_t st = as_stream(stream);
    DevScope mem;
    double* buf = nullptr;
    const size_t nd = 4 + mask_stats_scratch_doubles();
    RET_IF(mem.alloc(&buf, sizeof(double) * nd));
    CK(cudaMemsetAsync(buf, 0, sizeof(double) * nd, st));
    RET_IF(launch_absmax(S, ld, m, n, buf, st));
    RET_IF(launch_mask_stats(D, L, S, ld, m, n, buf, buf + 1, buf + 4, st));
    RET_IF(launch_mask_write(S, ld, m, n, buf + 1, sigmas, mask, m, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

int bsub_prox_flat3_dev(const float* U, float* V, int64_t ld, int32_t rows, int32_t cols, int32_t n, double lambda1, void* stream) {
    if (!U || !V || (long long)rows * cols > ld) { set_error("bsub_prox_flat3_dev: bad argument"); return -1; }
    return launch_prox_flat3(U, V, ld, rows, cols, n, (float)lambda1, as_stream(stream));
}

// CSR of the group ids >= 1 (ptr[k] .. ptr[k+1]: pixels of group k+1); returns the largest id
static int groups_to_csr(const int32_t* g, long long m, std::vector<int>& start, std::vector<int>& idx) {
    int gmax = 0;
    for (long long p = 0; p < m; ++p) { if (g[p] < 0) return -1; gmax = std::max(gmax, (int)g[p]); }
    std::vector<int> cnt((size_t)gmax + 1, 0);
    start.assign((size_t)gmax + 1, 0);
    for (long long p = 0; p < m; ++p) if (g[p] > 0) cnt[g[p]]++;
    int acc = 0;
    for (int k = 1; k <= gmax; ++k) { start[k - 1] = acc; acc += cnt[k]; }
    start[gmax] = acc;
    idx.assign((size_t)std::max(acc, 1), 0);
    std::vector<int> fill(start.begin(), start.end());
    for (long long p = 0; p < m; ++p) if (g[p] > 0) idx[fill[g[p] - 1]++] = (int)p;
    return gmax;
}

int bsub_prox_flat_groups_dev(const float* U, float* V, int64_t ld, int64_t m, int32_t n, const int32_t* g, double lambda1, void* stream) {
    if (!U || !V || !g || ld < m) { set_error("bsub_prox_flat_groups_dev: bad argument"); return -1; }
    std::vector<int> start, idx;
    const int gmax = groups_to_csr(g, m, start, idx);
    if (gmax < 0) { set_error("bsub_prox_flat_groups_dev: negative group id"); return -1; }
    DevScope mem;
    int *gptr = nullptr, *gidx = nullptr;
    RET_IF(mem.alloc(&gptr, sizeof(int) * ((size_t)gmax + 1)));
    RET_IF(mem.alloc(&gidx, sizeof(int) * idx.size()));
    CK(cudaMemcpy(gptr, start.data(), sizeof(int) * ((size_t)gmax + 1), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(gidx, idx.data(), sizeof(int) * idx.size(), cudaMemcpyHostToDevice));
    RET_IF(launch_prox_groups_csr(U, V, ld, m, n, gptr, gidx, gmax, (float)lambda1, nullptr, as_stream(stream)));
    CK(cudaStreamSynchronize(as_stream(stream)));
    return 0;
}

// the prox of the operators: all n frames of d at lambda1, the sweep count of the call; synchronises the stream and releases d
static int prox_once(GraphDesc* d, const float* U, float* V, long long ld, int n, double lambda1, int max_sweeps, double tol,
                     int32_t* sweeps_used, void* stream) {
    cudaStream_t st = as_stream(stream);
    ProxWork w;
    DevScope mem;
    int* sw = nullptr;
    int sw_h = 0;
    const int rc = [&]() -> int {
        RET_IF(mem.alloc(&sw, sizeof(int) * 8));
        CK(cudaMemsetAsync(sw, 0, sizeof(int) * 8, st));
        RET_IF(graph_prox(*d, U, V, ld, 0, n, nullptr, (float)lambda1, max_sweeps > 0 ? max_sweeps : 4000, (float)tol, sw, &w, st));
        CK(cudaMemcpyAsync(&sw_h, sw, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return 0;
    }();
    w.release();
    d->release();
    if (rc == 0 && sweeps_used) *sweeps_used = sw_h;
    return rc;
}

int bsub_prox_graph3_dev(const float* U, float* V, int64_t ld, int32_t rows, int32_t cols, int32_t n, double lambda1,
                         const double* eta_host, int32_t max_sweeps, double tol, int32_t* sweeps_used, void* stream) {
    GraphDesc d;
    RET_IF(describe_windows(&d, rows, cols, 0, n, eta_host, window_count(rows, cols), "bsub_prox_graph3_dev",
                            U && V && (long long)rows * cols <= ld));
    return prox_once(&d, U, V, ld, n, lambda1, max_sweeps, tol, sweeps_used, stream);
}

int bsub_prox_center3_dev(const float* U, float* V, int64_t ld, int32_t rows, int32_t cols, int32_t n, double lambda1,
                          const float* eta_host, int32_t max_sweeps, double tol, int32_t* sweeps_used, void* stream) {
    if (!eta_host) { set_error("bsub_prox_center3_dev: bad argument"); return -1; }
    GraphDesc d;
    RET_IF(describe_centre(&d, rows, cols, 0, n, eta_host, nullptr, "bsub_prox_center3_dev", U && V && (long long)rows * cols <= ld));
    return prox_once(&d, U, V, ld, n, lambda1, max_sweeps, tol, sweeps_used, stream);
}

int bsub_prox_graph_dev(const float* U, float* V, int64_t ld, int64_t m, int32_t n, double lambda1, int32_t n_graphs, const int32_t* frame_graph,
                        const int64_t* n_groups, const int32_t* const* indptr, const int32_t* const* indices, const double* const* eta,
                        int32_t max_sweeps, double tol, int32_t* sweeps_used, void* stream) {
    GraphDesc d;
    RET_IF(describe_graphs(&d, 0, 0, m, 0, n, n_graphs, frame_graph, n_groups, indptr, indices, eta, nullptr, "bsub_prox_graph_dev",
                           U && V && ld >= m));
    return prox_once(&d, U, V, ld, n, lambda1, max_sweeps, tol, sweeps_used, stream);
}

int bsub_block_shrink_dev(const float* G, float* R, int64_t ld, int64_t m, int32_t n, const uint8_t* labels, const int32_t* lam_ptr,
                          const double* lam, double mu, double non_block_lambda, void* stream) {
    if (!G || !R || !labels || !lam_ptr || ld < m) { set_error("bsub_block_shrink_dev: bad argument"); return -1; }
    cudaStream_t st = as_stream(stream);
    int maxb = 0;
    for (int f = 0; f < n; ++f) maxb = std::max(maxb, lam_ptr[f + 1] - lam_ptr[f]);
    const int nlab = maxb + 1;
    std::vector<double> table((size_t)n * nlab, 0.0);
    for (int f = 0; f < n; ++f)
        for (int b = 0; b < lam_ptr[f + 1] - lam_ptr[f]; ++b) table[(size_t)f * nlab + b + 1] = lam[lam_ptr[f] + b];
    DevScope mem;
    unsigned char* lab_d = nullptr; double *tab_d = nullptr, *sums = nullptr;
    RET_IF(mem.alloc(&lab_d, (size_t)n * m));
    RET_IF(mem.alloc(&tab_d, sizeof(double) * table.size()));
    RET_IF(mem.alloc(&sums, sizeof(double) * table.size()));
    CK(cudaMemcpy(lab_d, labels, (size_t)n * m, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(tab_d, table.data(), sizeof(double) * table.size(), cudaMemcpyHostToDevice));
    RET_IF(launch_block_l2_sums(G, lab_d, ld, m, n, nlab, sums, nullptr, st));
    RET_IF(launch_block_l2_apply(G, R, lab_d, ld, m, n, nlab, sums, tab_d, nullptr, mu, non_block_lambda, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

int bsub_gram_dev(const float* D, const float* S, const float* Y, int64_t ld, int64_t m, int32_t n, double mu, double* G_host,
                  void* stream) {
    if (!D || !G_host || ld < m || (ld % 32) != 0) { set_error("bsub_gram_dev: bad argument (ld must be a multiple of 32, pad columns zero)"); return -1; }
    if ((S == nullptr) != (Y == nullptr)) { set_error("bsub_gram_dev: S and Y must both be given or both be NULL"); return -1; }
    cudaStream_t st = as_stream(stream);
    int dev = 0, sms = 148;
    CK(cudaGetDevice(&dev));
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    GramPlan gp = make_gram_plan(n, ld, sms);
    std::vector<int2> tasks(gp.ntasks);
    fill_gram_tasks(gp, tasks.data());
    DevScope mem;
    int2* tasks_d = nullptr; double *partial = nullptr, *G = nullptr;
    RET_IF(mem.alloc(&tasks_d, sizeof(int2) * gp.ntasks));
    RET_IF(mem.alloc(&partial, sizeof(double) * gp.partial_elems));
    RET_IF(mem.alloc(&G, sizeof(double) * (size_t)gp.npad * gp.npad));
    CK(cudaMemcpy(tasks_d, tasks.data(), sizeof(int2) * gp.ntasks, cudaMemcpyHostToDevice));
    GramMaps gm;
    RET_IF(make_gram_maps(gp, D, S, Y, ld, &gm));
    RET_IF(launch_gram(gp, gm, S != nullptr, tasks_d, nullptr, (float)(S ? 1.0 / mu : 0.0), partial, G, st));
    CK(cudaMemcpy2DAsync(G_host, sizeof(double) * n, G, sizeof(double) * gp.npad, sizeof(double) * n, n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

int bsub_gram_i8_test(const int8_t* slices_host, int32_t n, int64_t ldq, int64_t* G_host) {
    // slices_host: int8 [4][n][ldq] (ldq a multiple of 64); G_host: int64 [n][n] = sum over pixels and slice pairs (i + j >= 3)
    // of 256^(i+j-3) d_i(f) d_j(g)  -- exact integers; exercises the tcgen05 kernel on its own
    if (!slices_host || !G_host || n <= 0 || ldq <= 0 || (ldq % 64) != 0) { set_error("bsub_gram_i8_test: bad argument"); return -1; }
    int dev = 0, sms = 148;
    CK(cudaGetDevice(&dev));
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    GramI8Plan gp = make_gram_i8_plan(n, ldq, sms);
    std::vector<int4> info; std::vector<int> blkn;
    fill_gram_i8_tables(gp, info, blkn);
    DevScope mem;
    signed char* q = nullptr; int4* info_d = nullptr; int* blkn_d = nullptr; unsigned long long* Gint = nullptr; double* G = nullptr;
    const size_t qbytes = (size_t)4 * n * ldq, gn = (size_t)gp.nblk * 128;
    const int npad = ((n + 31) / 32) * 32;
    RET_IF(mem.alloc(&q, qbytes));
    RET_IF(mem.alloc(&info_d, sizeof(int4) * info.size()));
    RET_IF(mem.alloc(&blkn_d, sizeof(int) * blkn.size()));
    RET_IF(mem.alloc(&Gint, sizeof(unsigned long long) * gn * gn));
    RET_IF(mem.alloc(&G, sizeof(double) * (size_t)npad * npad));
    {   // repack [4][n][ldq] (row-major, as the caller gives it) into the k-block-major layout [4][ldq/16][n][16]
        std::vector<signed char> packed(qbytes);
        for (int sl = 0; sl < 4; ++sl)
            for (int f = 0; f < n; ++f)
                for (long long k = 0; k < ldq / 16; ++k)
                    memcpy(&packed[(((size_t)sl * (ldq / 16) + k) * n + f) * 16], &slices_host[((size_t)sl * n + f) * ldq + k * 16], 16);
        CK(cudaMemcpy(q, packed.data(), qbytes, cudaMemcpyHostToDevice));
    }
    CK(cudaMemcpy(info_d, info.data(), sizeof(int4) * info.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(blkn_d, blkn.data(), sizeof(int) * blkn.size(), cudaMemcpyHostToDevice));
    CUtensorMap map, map_last;
    RET_IF(make_gram_i8_map(gp, q, &map, 128));
    RET_IF(make_gram_i8_map(gp, q, &map_last, gram_i8_last_block_n(gp)));
    RET_IF(launch_gram_i8(gp, map, map_last, info_d, (int)info.size(), blkn_d, Gint, G, npad, nullptr, 1.0, 1, 0));
    CK(cudaDeviceSynchronize());
    std::vector<long long> tmp(gn * gn);
    CK(cudaMemcpy(tmp.data(), Gint, sizeof(long long) * gn * gn, cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            const int blk = gram_i8_last_block_frames();
            const int r = (i / blk <= j / blk) ? i : j, c = (i / blk <= j / blk) ? j : i;
            G_host[(size_t)i * n + j] = tmp[(size_t)r * gn + c];
        }
    return 0;
}

int bsub_gram_i8_bench(int32_t n, int64_t ldq, int32_t reps, float* ms_out) {
    // profiling hook: average time of `reps` launches of the int8 Gram on device-resident digit planes of arbitrary content
    if (!ms_out || n <= 0 || ldq <= 0 || (ldq % 64) != 0 || reps <= 0) { set_error("bsub_gram_i8_bench: bad argument"); return -1; }
    int dev = 0, sms = 148;
    CK(cudaGetDevice(&dev));
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    GramI8Plan gp = make_gram_i8_plan(n, ldq, sms);
    std::vector<int4> info; std::vector<int> blkn;
    fill_gram_i8_tables(gp, info, blkn);
    DevScope mem;
    signed char* q = nullptr; int4* info_d = nullptr; int* blkn_d = nullptr; unsigned long long* Gint = nullptr; double* G = nullptr;
    const size_t qbytes = (size_t)4 * n * ldq, gn = (size_t)gp.nblk * 128;
    const int npad = ((n + 31) / 32) * 32;
    RET_IF(mem.alloc(&q, qbytes));
    RET_IF(mem.alloc(&info_d, sizeof(int4) * info.size()));
    RET_IF(mem.alloc(&blkn_d, sizeof(int) * blkn.size()));
    RET_IF(mem.alloc(&Gint, sizeof(unsigned long long) * gn * gn));
    RET_IF(mem.alloc(&G, sizeof(double) * ((size_t)npad * npad + 16)));
    CK(cudaMemset(q, 0x35, qbytes));
    CK(cudaMemcpy(info_d, info.data(), sizeof(int4) * info.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(blkn_d, blkn.data(), sizeof(int) * blkn.size(), cudaMemcpyHostToDevice));
    CUtensorMap map, map_last;
    RET_IF(make_gram_i8_map(gp, q, &map, 128));
    RET_IF(make_gram_i8_map(gp, q, &map_last, gram_i8_last_block_n(gp)));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    for (int r = 0; r < 2; ++r) RET_IF(launch_gram_i8(gp, map, map_last, info_d, (int)info.size(), blkn_d, Gint, G, npad, nullptr, 1.0, 1, 0));
    CK(cudaEventRecord(e0, 0));
    for (int r = 0; r < reps; ++r) RET_IF(launch_gram_i8(gp, map, map_last, info_d, (int)info.size(), blkn_d, Gint, G, npad, nullptr, 1.0, 1, 0));
    CK(cudaEventRecord(e1, 0));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *ms_out = ms / (float)reps;
    return 0;
}

int bsub_eig_topk(const double* G_host, int32_t n, int32_t k, double* lam_host, double* vec_host) {
    if (!G_host || n <= 0 || k <= 0 || k > n || !lam_host) { set_error("bsub_eig_topk: bad argument"); return -1; }
    const int npad = ((n + 31) / 32) * 32;
    EigPlan ep = make_eig_plan(n, npad);
    EigBuffers eb;
    memset(&eb, 0, sizeof(eb));
    DevScope mem;
    double* G = nullptr; DevState* st = nullptr;
    RET_IF(mem.alloc(&G, sizeof(double) * (size_t)npad * npad));
    CK(cudaMemset(G, 0, sizeof(double) * (size_t)npad * npad));
    CK(cudaMemcpy2D(G, sizeof(double) * npad, G_host, sizeof(double) * n, sizeof(double) * n, n, cudaMemcpyHostToDevice));
    RET_IF(mem.alloc(&eb.work, sizeof(double) * ep.work_doubles));
    RET_IF(mem.alloc(&eb.lam, sizeof(double) * n));
    RET_IF(mem.alloc(&eb.Z, sizeof(double) * (size_t)n * n));
    RET_IF(mem.alloc(&st, sizeof(DevState)));
    CK(cudaMemset(st, 0, sizeof(DevState)));
    eb.vstride = n;
    RET_IF(launch_eig(ep, G, nullptr, eb, st, 2, k, 0));
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(lam_host, eb.lam, sizeof(double) * k, cudaMemcpyDeviceToHost));
    if (vec_host) CK(cudaMemcpy(vec_host, eb.Z, sizeof(double) * (size_t)k * n, cudaMemcpyDeviceToHost));
    return 0;
}

}  // extern "C"
