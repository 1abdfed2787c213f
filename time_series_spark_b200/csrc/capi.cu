// C ABI of libprophet_b200.so (see include/prophet_b200.h).  Host-side orchestration only:
// length classes, work queues, launches, staging copies.  All arithmetic is in the kernels.
#define PB200_WITH_PREP 1
#include "fit_kernel.cuh"
#include "launch.h"
#include "predict_kernel.cuh"
#include "mc_kernel.cuh"
#include "newton_kernel.cuh"
#include "csv_kernel.cuh"
#include "csv_reader.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

namespace {

thread_local std::string g_err;

int fail(int code, const char* what, cudaError_t e = cudaSuccess) {
    char buf[512];
    if (e != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
    else snprintf(buf, sizeof buf, "%s", what);
    g_err = buf;
    return code;
}

#define CK(call)                                                      \
    do {                                                              \
        cudaError_t e_ = (call);                                      \
        if (e_ != cudaSuccess) return fail(PB200_E_CUDA, #call, e_);  \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = n + n / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

struct HostBuf {   // pinned
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        size_t want = n + n / 8 + 256;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

constexpr int NLC = 3;
const int LC_NT[NLC] = {32, 64, 128};

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

}  // namespace

// Everything one in-flight fit call needs besides its inputs and outputs.  NWS of them: the *_host entry point cuts
// a big batch into series chunks, one (stream, workspace) pair each, so that the H2D copy of chunk i + 1 overlaps the
// fit of chunk i and the later chunks' kernels fill the SMs an earlier chunk's stragglers leave idle.  (With two
// pairs chunk i + 2 had to wait for chunk i's LAST series before it could start: r2i, e2e / value 0.86.)
struct FitWs {
    cudaStream_t stream = nullptr;
    cudaEvent_t ctl_ev = nullptr;   // recorded after the H2D copies out of h_ctl
    bool ctl_pending = false;
    DevBuf d_offsets, d_order, d_lenclass, d_qitems, d_qctl;   // control workspace (device)
    DevBuf d_qkey, d_qhist;         // counting sort of the work queues by expected cost (prep_kernel, queue_*_kernel)
    DevBuf d_nq;                    // [0] count, [1] head, [2..] series whose L-BFGS failed its line search (Newton retry queue)
    DevBuf d_planes;                // fit kernels' per-series workspace (one slice per resident CTA / series slot)
    HostBuf h_ctl;                  // pinned staging for offsets / order / lenclass
};

constexpr int NWS = 4;

struct pb200_ctx {
    int device = 0;
    int sms = 0;
    FitWs ws[NWS];
    cudaStream_t stream = nullptr;  // = ws[0].stream: the stream of every single-workspace call
    cudaEvent_t fork_ev = nullptr;
    int64_t launches = 0;
    DevBuf d_vcount;                // series of the last fit call per kernel variant x seasonality class
    // data staging for the *_host entry points
    DevBuf d_ds, d_y, d_cap, d_params, d_tchange, d_mi32, d_mi64, d_mf64;
    DevBuf d_fut, d_floor, d_yhat, d_lo, d_hi, d_yint;
    DevBuf d_mc;     // MC workspace
    int lc_max[NLC];
    bool lc_auto = true;   // false when PB200_LC*_MAX pins the CTA width
    bool tab_on = true;    // PB200_NO_TAB=1 disables the seasonal-table variants (A/B runs)
    int grp_g = -1;        // lanes per series of the grouped day-table kernel (fit_group.cuh); PB200_GROUP=0|8|16|32 pins it
                           // (0 = point_pass_tab), unset = by batch size: 8 from grp_min series on, 16 below
    DevBuf d_trace;        // trajectory rows of pb200_fit_trace_host
    DevBuf d_nq_all, d_offsets_full;   // pb200_fit_host: per-chunk Newton retry queues, the call's offsets on the device
    int plain_grp = 0;     // PB200_PLAIN_GROUP=1: the class WITHOUT seasonality (regular grid; reference config #4) on the grouped kernel
                           // too.  Off: measured 6 % faster than one warp per series at 500k short series, 3 % slower at 100k and
                           // 35 % slower at 30k (r2s) -- its rounds are longer, and small batches are latency bound
    int grp_min = 16384;   // PB200_GROUP_MIN: smallest batch that gets 8 lanes per series; smaller ones get 16 (a warp with 4
                           // series drains longer once the queue is empty).  r2o, ms per step at 6 250 / 12 500 / 50 000 series:
                           // G = 8: 78 / 113 / 333, G = 16: 73 / 110 / 352, one warp per series (round-1 kernel): 76 / 125 / 455
    int host_chunks = 1;   // PB200_HOST_CHUNKS: series chunks of pb200_fit_host.  Default 1 (one pass): measured on 50k x 1440
                           // (r2j / r2k) 1 / 2 / 4 / 8 chunks = 397 / 407 / 440 / 500 ms -- the 865 MB copy is only ~25 ms at
                           // PCIe 5 speed, and every chunk pays its own straggler drain, which costs more than it hides
};

namespace {

using pb200::FitArgs;
using pb200::FitOptsDev;
using pb200::NQ;

typedef cudaError_t (*launch_fn)(int, int, int, const FitArgs&, int, size_t, cudaStream_t, int*);
const launch_fn LAUNCH[8] = {pb200::launch_fit_mask0, pb200::launch_fit_mask1, pb200::launch_fit_mask2,
                             pb200::launch_fit_mask3, pb200::launch_fit_mask4, pb200::launch_fit_mask5,
                             pb200::launch_fit_mask6, pb200::launch_fit_mask7};

int check_opts(const pb200_options* o) {
    if (!o) return fail(PB200_E_ARG, "options is null");
    if (o->abi_version != PB200_ABI_VERSION) return fail(PB200_E_ARG, "options.abi_version mismatch");
    if (o->growth != PB200_GROWTH_LINEAR && o->growth != PB200_GROWTH_LOGISTIC) return fail(PB200_E_ARG, "growth");
    if (o->n_changepoints < 0 || o->n_changepoints > 30) return fail(PB200_E_UNSUPPORTED, "n_changepoints must be in [0, 30]");
    if (o->history_size < 1 || o->history_size > pb200::HMAX) return fail(PB200_E_UNSUPPORTED, "history_size must be in [1, 5]");
    if (!(o->changepoint_range > 0.0 && o->changepoint_range <= 1.0)) return fail(PB200_E_ARG, "changepoint_range");
    if (!(o->changepoint_prior_scale > 0.0) || !(o->seasonality_prior_scale > 0.0)) return fail(PB200_E_ARG, "prior scales");
    for (int v : {o->yearly, o->weekly, o->daily})
        if (v != PB200_SEAS_AUTO && v != 0 && v != 1) return fail(PB200_E_UNSUPPORTED, "seasonality switch must be AUTO, 0 or 1");
    if (o->max_iter < 1) return fail(PB200_E_ARG, "max_iter");
    if (o->algorithm < PB200_ALG_LBFGS_NEWTON || o->algorithm > PB200_ALG_NEWTON) return fail(PB200_E_ARG, "algorithm");
    return PB200_OK;
}

FitOptsDev to_dev(const pb200_options* o) {
    FitOptsDev d;
    const double eps = 2.220446049250313e-16;
    d.growth = o->growth;
    d.mult = o->multiplicative ? 1 : 0;
    d.n_changepoints = o->n_changepoints;
    d.max_iter = o->max_iter;
    d.history = o->history_size;
    d.yearly = o->yearly;
    d.weekly = o->weekly;
    d.daily = o->daily;
    d.changepoint_range = o->changepoint_range;
    d.tau = o->changepoint_prior_scale;
    d.seas_prior = o->seasonality_prior_scale;
    d.rtau = 1.0 / o->changepoint_prior_scale;
    d.inv_seas2 = 1.0 / (o->seasonality_prior_scale * o->seasonality_prior_scale);
    d.init_alpha = o->init_alpha;
    d.tol_obj = o->tol_obj;
    d.tol_rel_obj_eps = o->tol_rel_obj * eps;
    d.tol_grad = o->tol_grad;
    d.tol_rel_grad_eps = o->tol_rel_grad * eps;
    d.tol_param = o->tol_param;
    return d;
}

int mask_nseas(int m) { return pb200::stored_planes((m & 1) ? 10 : 0, (m & 2) ? 3 : 0, (m & 4) ? 4 : 0); }   // stored planes
int mask_k(int m) { return ((m & 1) ? 20 : 0) + ((m & 2) ? 6 : 0) + ((m & 4) ? 8 : 0); }

size_t y_elem(int dt) { return dt == PB200_Y_F64 ? 8 : 4; }

}  // namespace

extern "C" {

PB200_API void pb200_default_options(pb200_options* o) {
    if (!o) return;
    memset(o, 0, sizeof *o);
    o->abi_version = PB200_ABI_VERSION;
    o->growth = PB200_GROWTH_LOGISTIC;       // prophet_modeler.py:65
    o->multiplicative = 1;                   // prophet_modeler.py:65
    o->n_changepoints = 25;
    o->changepoint_range = 0.8;
    o->changepoint_prior_scale = 0.05;
    o->seasonality_prior_scale = 10.0;
    o->yearly = o->weekly = o->daily = PB200_SEAS_AUTO;
    o->max_iter = 10000;
    o->history_size = 5;
    o->init_alpha = 1e-3;
    o->tol_obj = 1e-12;
    o->tol_rel_obj = 1e4;
    o->tol_grad = 1e-8;
    o->tol_rel_grad = 1e7;
    o->tol_param = 1e-8;
    o->interval_width = 0.8;
    o->uncertainty_samples = 1000;
}

PB200_API int pb200_get_layout(const pb200_options* o, pb200_layout* out) {
    int rc = check_opts(o);
    if (rc) return rc;
    if (!out) return fail(PB200_E_ARG, "layout is null");
    out->smax = o->n_changepoints > 0 ? o->n_changepoints : 1;
    int k = 0;
    if (o->yearly != 0) k += 20;
    if (o->weekly != 0) k += 6;
    if (o->daily != 0) k += 8;
    out->kmax = k > 0 ? k : 1;
    out->pstride = 3 + out->smax + out->kmax;
    out->meta_i32_stride = 8;
    out->meta_i64_stride = 2;
    out->meta_f64_stride = 4;
    return PB200_OK;
}

PB200_API const char* pb200_last_error(void) { return g_err.c_str(); }

PB200_API pb200_ctx* pb200_create(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        fail(PB200_E_CUDA, "no CUDA device (this library has no CPU path)", e);
        return nullptr;
    }
    if (device < 0 || device >= n) {
        fail(PB200_E_ARG, "device index out of range");
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) {
        fail(PB200_E_CUDA, "cudaSetDevice");
        return nullptr;
    }
    pb200_ctx* c = new pb200_ctx();
    c->device = device;
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    c->sms = prop.multiProcessorCount;
    if (prop.major != 10) {
        fail(PB200_E_CUDA, "device is not sm_100 (this library is compiled for sm_100a only)");
        delete c;
        return nullptr;
    }
    bool ok = cudaEventCreateWithFlags(&c->fork_ev, cudaEventDisableTiming) == cudaSuccess;
    for (FitWs& w : c->ws) {
        ok = ok && cudaStreamCreateWithFlags(&w.stream, cudaStreamNonBlocking) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&w.ctl_ev, cudaEventDisableTiming) == cudaSuccess;
    }
    if (!ok) {
        fail(PB200_E_CUDA, "cudaStreamCreate / cudaEventCreate");
        for (FitWs& w : c->ws) {
            if (w.ctl_ev) cudaEventDestroy(w.ctl_ev);
            if (w.stream) cudaStreamDestroy(w.stream);
        }
        if (c->fork_ev) cudaEventDestroy(c->fork_ev);
        delete c;
        return nullptr;
    }
    c->stream = c->ws[0].stream;
    c->host_chunks = std::max(1, std::min(16, env_int("PB200_HOST_CHUNKS", 1)));
    c->lc_max[0] = env_int("PB200_LC0_MAX", 1 << 30);   // warp-per-series for every length
    c->lc_max[1] = env_int("PB200_LC1_MAX", 1 << 30);
    c->lc_max[2] = 1 << 30;
    c->lc_auto = !(getenv("PB200_LC0_MAX") || getenv("PB200_LC1_MAX"));
    c->tab_on = env_int("PB200_NO_TAB", 0) == 0;
    c->grp_g = env_int("PB200_GROUP", -1);
    if (c->grp_g != -1 && c->grp_g != 8 && c->grp_g != 16 && c->grp_g != 32) c->grp_g = 0;
    c->grp_min = env_int("PB200_GROUP_MIN", 16384);
    c->plain_grp = env_int("PB200_PLAIN_GROUP", 0) != 0;
    return c;
}

PB200_API void pb200_destroy(pb200_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (FitWs& w : c->ws) cudaStreamSynchronize(w.stream);
    for (DevBuf* b : {&c->d_ds, &c->d_y, &c->d_cap, &c->d_params, &c->d_tchange, &c->d_mi32, &c->d_mi64, &c->d_mf64, &c->d_fut,
                      &c->d_floor, &c->d_yhat, &c->d_lo, &c->d_hi, &c->d_yint, &c->d_mc, &c->d_trace, &c->d_vcount, &c->d_nq_all,
                      &c->d_offsets_full})
        b->release();
    for (FitWs& w : c->ws) {
        for (DevBuf* b : {&w.d_offsets, &w.d_order, &w.d_lenclass, &w.d_qitems, &w.d_qctl, &w.d_nq, &w.d_planes, &w.d_qkey, &w.d_qhist})
            b->release();
        w.h_ctl.release();
        cudaEventDestroy(w.ctl_ev);
        cudaStreamDestroy(w.stream);
    }
    cudaEventDestroy(c->fork_ev);
    delete c;
}

PB200_API void* pb200_stream(pb200_ctx* c) { return c ? (void*)c->stream : nullptr; }
PB200_API int64_t pb200_launch_count(pb200_ctx* c) { return c ? c->launches : 0; }

PB200_API int32_t pb200_tab_chunk(int32_t T, int32_t P) {
    if (T < 1 || P < 2) return -1;
    return pb200::tab_chunk(T, P);
}

PB200_API int pb200_last_fit_variant_counts(pb200_ctx* c, int32_t* h_counts) {
    if (!c || !h_counts) return fail(PB200_E_ARG, "null argument");
    static_assert(PB200_N_VARIANT_COUNTS == NQ, "variant count layout");
    for (int i = 0; i < NQ; ++i) h_counts[i] = 0;
    if (!c->d_vcount.p) return PB200_OK;      // no fit yet
    CK(cudaSetDevice(c->device));
    for (FitWs& w : c->ws) CK(cudaStreamSynchronize(w.stream));
    CK(cudaMemcpy(h_counts, c->d_vcount.p, NQ * 4, cudaMemcpyDeviceToHost));
    return PB200_OK;
}

PB200_API int pb200_synchronize(pb200_ctx* c) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    CK(cudaSetDevice(c->device));
    for (FitWs& w : c->ws) CK(cudaStreamSynchronize(w.stream));
    return PB200_OK;
}

}  // extern "C"

// zero the per-call variant counters (on workspace 0's stream; the other workspaces are ordered behind it)
static int begin_fit_call(pb200_ctx* c) {
    CK(c->d_vcount.reserve(NQ * 4));
    CK(cudaMemsetAsync(c->d_vcount.p, 0, NQ * 4, c->ws[0].stream));
    CK(cudaEventRecord(c->fork_ev, c->ws[0].stream));
    for (int i = 1; i < NWS; ++i) CK(cudaStreamWaitEvent(c->ws[i].stream, c->fork_ev, 0));
    return PB200_OK;
}

// newton_kernel over the queue {count, head, items...} at d_nq (16-warp CTAs with ~100 KB of shared memory: they do not
// fit beside a full house of fit CTAs, which is why the chunked host path runs them after all chunks, and only if needed)
static int launch_newton(pb200_ctx* c, cudaStream_t st, const pb200_options* opts, const int64_t* d_ds, const void* d_y,
                         int32_t y_dtype, const int64_t* d_offsets, int64_t n_series, int* d_nq, double* d_params,
                         double* d_tchange, int32_t* d_meta_i32, int64_t* d_meta_i64, double* d_meta_f64) {
    pb200_layout L;
    pb200_get_layout(opts, &L);
    if (opts->algorithm == PB200_ALG_LBFGS || L.pstride > pb200::nw::NW_PMAX) return PB200_OK;
    pb200::nw::NewtonArgs na;
    na.ds = (const long long*)d_ds;
    na.y = d_y;
    na.y_dtype = y_dtype;
    na.offsets = (const long long*)d_offsets;
    na.nq_count = d_nq;
    na.nq_head = d_nq + 1;
    na.nq_items = d_nq + 2;
    na.params = d_params;
    na.tchange = d_tchange;
    na.meta_i32 = d_meta_i32;
    na.meta_i64 = (const long long*)d_meta_i64;
    na.meta_f64 = d_meta_f64;
    na.smax = L.smax;
    na.kmax = L.kmax;
    na.pstride = L.pstride;
    na.o = to_dev(opts);
    const size_t nsm = pb200::nw::newton_smem_bytes(L.pstride);
    CK(cudaFuncSetAttribute(pb200::nw::newton_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)nsm));
    const int ngrid = (int)std::min<int64_t>(n_series, opts->algorithm == PB200_ALG_NEWTON ? (int64_t)c->sms * 2 : (int64_t)c->sms);
    pb200::nw::newton_kernel<<<ngrid, 32 * pb200::nw::NW_WARPS, nsm, st>>>(na);
    CK(cudaGetLastError());
    c->launches++;
    return PB200_OK;
}

static int fit_impl(pb200_ctx* c, FitWs& w, const pb200_options* opts, const int64_t* d_ds, const void* d_y, int32_t y_dtype,
                    const int64_t* h_offsets, int64_t n_series, double floor, double cap_multiplier,
                    const double* d_cap, double* d_params, double* d_tchange, int32_t* d_meta_i32,
                    int64_t* d_meta_i64, double* d_meta_f64, const double* d_theta_in, double* d_grad_out,
                    double* d_trace = nullptr, int trace_cap = 0, int64_t n_call = 0, int* ext_nq = nullptr) {
    // ext_nq (chunked host call): {count, head} of this chunk's Newton retry queue followed at ext_nq + 2 by its items;
    // the queue is then only FILLED here and the caller launches newton_kernel after all chunks (see pb200_fit_host)
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    int rc = check_opts(opts);
    if (rc) return rc;
    if (n_series < 0 || n_series > (1LL << 30)) return fail(PB200_E_ARG, "n_series");
    if (n_series == 0) return PB200_OK;
    if (!d_ds || !d_y || !h_offsets || !d_params || !d_tchange || !d_meta_i32 || !d_meta_i64 || !d_meta_f64)
        return fail(PB200_E_ARG, "null pointer");
    if (y_dtype < 0 || y_dtype > 2) return fail(PB200_E_ARG, "y_dtype");
    pb200_layout L;
    pb200_get_layout(opts, &L);
    CK(cudaSetDevice(c->device));
    const int N = (int)n_series;

    // ---- host: length classes and longest-first order (counting sort on T) ----
    size_t ctl_bytes = (size_t)(N + 1) * 8 + (size_t)N * 4 * 2;
    if (w.ctl_pending) {   // the pinned staging of the previous call must have been consumed
        CK(cudaEventSynchronize(w.ctl_ev));
        w.ctl_pending = false;
    }
    CK(w.h_ctl.reserve(ctl_bytes));
    int64_t* ho = (int64_t*)w.h_ctl.p;
    int* horder = (int*)(ho + N + 1);
    int* hlc = horder + N;
    memcpy(ho, h_offsets, (size_t)(N + 1) * 8);
    int lc_n[NLC] = {0, 0, 0}, lc_tmax[NLC] = {0, 0, 0};
    int64_t tmax_all = 0;
    for (int i = 0; i < N; ++i) {
        const int64_t T = ho[i + 1] - ho[i];
        if (T < 0) return fail(PB200_E_ARG, "offsets not monotone");
        if (T > tmax_all) tmax_all = T;
    }
    if (tmax_all > (1 << 24)) return fail(PB200_E_UNSUPPORTED, "series longer than 2^24 rows");
    {
        std::vector<int> cnt((size_t)tmax_all + 2, 0);
        for (int i = 0; i < N; ++i) cnt[(size_t)(ho[i + 1] - ho[i])]++;
        // descending T: position of length t = number of series with length > t
        std::vector<int> posv((size_t)tmax_all + 2, 0);
        int acc = 0;
        for (int64_t t = tmax_all; t >= 0; --t) { posv[(size_t)t] = acc; acc += cnt[(size_t)t]; }
        for (int i = 0; i < N; ++i) {
            const int T = (int)(ho[i + 1] - ho[i]);
            horder[posv[(size_t)T]++] = i;
            // CTA width: one warp per series fills the chip once there are >= ~8 series per SM; a small
            // batch of long series gets 4 warps per series instead (same kernels, NT = 128)
            int lc = 0;
            while (lc < NLC - 1 && T > c->lc_max[lc]) ++lc;
            if (c->lc_auto && N < c->sms * 8 && T >= 256) lc = NLC - 1;
            hlc[i] = lc;
            lc_n[lc]++;
            if (T > lc_tmax[lc]) lc_tmax[lc] = T;
        }
    }
    // ---- device control buffers ----
    CK(w.d_offsets.reserve((size_t)(N + 1) * 8));
    CK(w.d_order.reserve((size_t)N * 4));
    CK(w.d_lenclass.reserve((size_t)N * 4));
    CK(w.d_qitems.reserve((size_t)NLC * NQ * N * 4));
    CK(w.d_qctl.reserve((size_t)NLC * NQ * 2 * 4));
    CK(w.d_qkey.reserve((size_t)N * 4));
    CK(w.d_qhist.reserve((size_t)NLC * NQ * pb200::QBINS * 4));
    CK(cudaMemsetAsync(w.d_qkey.p, 0xff, (size_t)N * 4, w.stream));
    CK(cudaMemsetAsync(w.d_qhist.p, 0, (size_t)NLC * NQ * pb200::QBINS * 4, w.stream));
    int* nq = ext_nq;
    if (!nq) {
        CK(w.d_nq.reserve((size_t)(N + 2) * 4));             // count, head, items[N]
        nq = (int*)w.d_nq.p;
    }
    CK(cudaMemsetAsync(nq, 0, 8, w.stream));
    CK(cudaMemcpyAsync(w.d_offsets.p, ho, (size_t)(N + 1) * 8, cudaMemcpyHostToDevice, w.stream));
    CK(cudaMemcpyAsync(w.d_order.p, horder, (size_t)N * 4, cudaMemcpyHostToDevice, w.stream));
    CK(cudaMemcpyAsync(w.d_lenclass.p, hlc, (size_t)N * 4, cudaMemcpyHostToDevice, w.stream));
    CK(cudaEventRecord(w.ctl_ev, w.stream));
    w.ctl_pending = true;
    CK(cudaMemsetAsync(w.d_qctl.p, 0, (size_t)NLC * NQ * 2 * 4, w.stream));
    CK(cudaMemsetAsync(d_params, 0, (size_t)N * L.pstride * 8, w.stream));
    CK(cudaMemsetAsync(d_tchange, 0, (size_t)N * L.smax * 8, w.stream));
    int* q_count = (int*)w.d_qctl.p;
    int* q_head = q_count + NLC * NQ;

    const FitOptsDev od = to_dev(opts);
    // lanes per series of the grouped day-table kernel
    // (n_call: series of the whole API call when this is one chunk of it)
    const int grp_g = !c->tab_on ? 0 : (c->grp_g >= 0 ? c->grp_g : (std::max<int64_t>(N, n_call) >= c->grp_min ? 8 : 16));
    // ---- prep kernel ----
    {
        pb200::PrepArgs pa;
        pa.ds = (const long long*)d_ds;
        pa.y = d_y;
        pa.y_dtype = y_dtype;
        pa.offsets = (const long long*)w.d_offsets.p;
        pa.order = (const int*)w.d_order.p;
        pa.cap = d_cap;
        pa.floor = floor;
        pa.cap_multiplier = cap_multiplier;
        pa.n_series = N;
        pa.meta_i32 = d_meta_i32;
        pa.meta_i64 = (long long*)d_meta_i64;
        pa.meta_f64 = d_meta_f64;
        pa.lenclass = (const int*)w.d_lenclass.p;
        pa.q_items = (int*)w.d_qitems.p;
        pa.q_count = q_count;
        pa.o = od;
        pa.tab_lc_mask = 0;
        for (int lc = 0; lc < NLC; ++lc)
            if (c->tab_on && LC_NT[lc] == 32) pa.tab_lc_mask |= 1 << lc;
        pa.grp_g = grp_g;
        pa.grp_plain = (c->plain_grp && grp_g > 0) ? 1 : 0;
        { static const char* e = getenv("PB200_QKEY_CV"); pa.cv_weight = e ? atof(e) : 2.0; }
        pa.newton_only = (opts->algorithm == PB200_ALG_NEWTON && !d_theta_in) ? 1 : 0;
        pa.nq_count = nq;
        pa.nq_items = nq + 2;
        pa.vcount = (int*)c->d_vcount.p;
        pa.qkey = (int*)w.d_qkey.p;
        pa.qhist = (int*)w.d_qhist.p;
        const int warps_per_block = 8;
        int grid = (N + warps_per_block - 1) / warps_per_block;
        grid = std::min(grid, c->sms * 8);
        pb200::prep_kernel<<<grid, warps_per_block * 32, 0, w.stream>>>(pa);
        CK(cudaGetLastError());
        pb200::queue_scan_kernel<<<(NLC * NQ + 127) / 128, 128, 0, w.stream>>>((int*)w.d_qhist.p, NLC * NQ);
        CK(cudaGetLastError());
        pb200::queue_scatter_kernel<<<std::min((N + 255) / 256, c->sms * 8), 256, 0, w.stream>>>(
            (const int*)w.d_qkey.p, (int*)w.d_qhist.p, (int*)w.d_qitems.p, N);
        CK(cudaGetLastError());
        c->launches += 3;
    }
    // ---- fit kernels: one persistent launch per (length class, seasonality class) ----
    // pass 1: launch geometry and the planes workspace (one slice per resident CTA)
    struct Geo { int grid, Tp, ppad; size_t smem, slice, off; bool on, grouped; };
    Geo geo[NLC][NQ];       // [length class][variant * 8 + seasonality class]
    size_t planes_bytes = 0;
    for (int lc = 0; lc < NLC; ++lc)
        for (int rm = 0; rm < NQ; ++rm) {
            const int mask = rm & 7, reg = rm >> 3;
            Geo& g = geo[lc][rm];
            g.on = false;
            g.grouped = false;
            if (lc_n[lc] == 0) continue;
            const bool plain_grp = reg == 3 && mask == 0 && grp_g > 0 && c->plain_grp;   // grouped kernel's class without seasonality
            if (reg && mask == 0 && !plain_grp) continue;                // no Fourier features: nothing to regenerate
            if (reg >= 2 && ((mask != 6 && !plain_grp) || LC_NT[lc] != 32 || !c->tab_on)) continue;   // seasonal-table variants
            auto impossible = [&](int bit, int sw) { return (sw == 0 && (mask & bit)) || (sw == 1 && !(mask & bit)); };
            if (impossible(1, opts->yearly) || impossible(2, opts->weekly) || impossible(4, opts->daily)) continue;
            const int NT = LC_NT[lc];
            const int chunk = std::max((lc_tmax[lc] + NT - 1) / NT, 1);
            g.Tp = ((lc_tmax[lc] + chunk + pb200::TAB_CHUNK_SLACK + 1 + 7) / 8) * 8;   // the table variants may widen a chunk
            const int K = mask_k(mask);
            g.ppad = ((L.smax + (K > 0 ? K : 1) + 3) + 1) & ~1;
            const int nst = reg ? 0 : mask_nseas(mask);                    // stored feature planes
            const int nsa = (mask & 1) + ((mask >> 1) & 1) + ((mask >> 2) & 1);   // active seasonalities
            g.smem = pb200::fit_smem_bytes(NT, 1 + nst, g.ppad, reg == 1 ? nsa : (reg == 2 ? 1 : (reg == 3 ? 2 : 0)),
                                           reg == 2 ? pb200::PTAB_WEEK_MAX : (reg == 3 ? pb200::PTAB_DAY_MAX : 0));
            int occ = 0;
            FitArgs dummy{};
            g.slice = (size_t)(1 + nst) * g.Tp;                   // double2 elements
            g.off = planes_bytes;
            if (reg == 3 && grp_g > 0) {
                // grouped day-table kernel: one warp per CTA, 32 / grp_g series per warp, one workspace slot per series
                const int nser = 32 / grp_g;
                CK(pb200::launch_fit_group(grp_g, opts->growth, opts->multiplicative ? 1 : 0, mask != 0, dummy, 0, w.stream, &occ));
                if (occ < 1) return fail(PB200_E_UNSUPPORTED, "grouped fit kernel does not fit on an SM");
                g.grouped = true;
                g.slice = pb200::fit_group_plane_doubles(lc_tmax[lc], grp_g);           // doubles per slot
                g.grid = (int)std::min<int64_t>(((int64_t)lc_n[lc] + nser - 1) / nser, (int64_t)c->sms * occ);
                planes_bytes += (size_t)g.grid * nser * g.slice * 8;
                g.on = true;
                continue;
            }
            CK(LAUNCH[mask](NT, opts->growth, reg, dummy, 0, g.smem, w.stream, &occ));
            if (occ < 1) return fail(PB200_E_UNSUPPORTED, "fit kernel does not fit on an SM");
            g.grid = (int)std::min<int64_t>((int64_t)lc_n[lc], (int64_t)c->sms * occ);
            planes_bytes += (size_t)g.grid * g.slice * 16;
            g.on = true;
        }
    CK(w.d_planes.reserve(planes_bytes));
    for (int lc = 0; lc < NLC; ++lc) {
        if (lc_n[lc] == 0) continue;
        const int NT = LC_NT[lc];
        for (int rm = 0; rm < NQ; ++rm) {
            const int mask = rm & 7, reg = rm >> 3;
            const Geo& g = geo[lc][rm];
            if (!g.on) continue;
            const int Tp = g.Tp, ppad = g.ppad;
            const size_t smem = g.smem;
            FitArgs fa;
            fa.ds = (const long long*)d_ds;
            fa.y = d_y;
            fa.y_dtype = y_dtype;
            fa.offsets = (const long long*)w.d_offsets.p;
            const int q = lc * NQ + rm;
            fa.q_items = (const int*)w.d_qitems.p + (size_t)q * N;
            fa.q_count = q_count + q;
            fa.q_head = q_head + q;
            fa.params = d_params;
            fa.tchange = d_tchange;
            fa.meta_i32 = d_meta_i32;
            fa.meta_i64 = (long long*)d_meta_i64;
            fa.meta_f64 = d_meta_f64;
            fa.smax = L.smax;
            fa.kmax = L.kmax;
            fa.pstride = L.pstride;
            fa.Tp = Tp;
            fa.ppad = ppad;
            fa.planes = (double2*)((char*)w.d_planes.p + g.off);
            fa.nseas_stride = (int)g.slice;
            fa.theta_in = d_theta_in;
            fa.grad_out = d_grad_out;
            fa.trace = d_trace;
            fa.trace_cap = trace_cap;
            fa.nq_count = nq;
            fa.nq_items = opts->algorithm == PB200_ALG_LBFGS_NEWTON ? nq + 2 : nullptr;
            fa.o = od;
            if (g.grouped) {
                CK(pb200::launch_fit_group(grp_g, opts->growth, opts->multiplicative ? 1 : 0, mask != 0, fa, g.grid, w.stream, nullptr));
            } else {
                CK(LAUNCH[mask](NT, opts->growth, reg, fa, g.grid, smem, w.stream, nullptr));
            }
            c->launches++;
        }
    }
    // ---- fbprophet's Newton retry over the series whose L-BFGS failed its line search (normally an empty queue) ----
    if (!ext_nq && !d_theta_in)
        return launch_newton(c, w.stream, opts, d_ds, d_y, y_dtype, (const int64_t*)w.d_offsets.p, n_series, nq, d_params, d_tchange,
                             d_meta_i32, d_meta_i64, d_meta_f64);
    return PB200_OK;
}

extern "C" {

PB200_API int pb200_fit_device(pb200_ctx* c, const pb200_options* opts, const int64_t* d_ds, const void* d_y, int32_t y_dtype,
                     const int64_t* h_offsets, int64_t n_series, double floor, double cap_multiplier,
                     const double* d_cap, double* d_params, double* d_tchange, int32_t* d_meta_i32,
                     int64_t* d_meta_i64, double* d_meta_f64) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    CK(cudaSetDevice(c->device));
    int rc = begin_fit_call(c);
    if (rc) return rc;
    return fit_impl(c, c->ws[0], opts, d_ds, d_y, y_dtype, h_offsets, n_series, floor, cap_multiplier, d_cap, d_params, d_tchange,
                    d_meta_i32, d_meta_i64, d_meta_f64, nullptr, nullptr);
}

PB200_API int pb200_objective_host(pb200_ctx* c, const pb200_options* opts, const int64_t* h_ds, const void* h_y,
                                   int32_t y_dtype, const int64_t* h_offsets, int64_t n_series, double floor,
                                   double cap_multiplier, const double* h_theta, double* h_f, double* h_grad,
                                   int32_t* h_meta_i32) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    int rc = check_opts(opts);
    if (rc) return rc;
    if (n_series <= 0) return n_series == 0 ? PB200_OK : fail(PB200_E_ARG, "n_series");
    if (!h_ds || !h_y || !h_offsets || !h_theta || !h_f || !h_grad || !h_meta_i32) return fail(PB200_E_ARG, "null pointer");
    if (y_dtype < 0 || y_dtype > 2) return fail(PB200_E_ARG, "y_dtype");
    pb200_layout L;
    pb200_get_layout(opts, &L);
    CK(cudaSetDevice(c->device));
    const int64_t R = h_offsets[n_series];
    const size_t N = (size_t)n_series;
    CK(c->d_ds.reserve((size_t)R * 8));
    CK(c->d_y.reserve((size_t)R * y_elem(y_dtype)));
    CK(c->d_params.reserve(N * L.pstride * 8));
    CK(c->d_tchange.reserve(N * L.smax * 8));
    CK(c->d_mi32.reserve(N * 8 * 4));
    CK(c->d_mi64.reserve(N * 2 * 8));
    CK(c->d_mf64.reserve(N * 4 * 8));
    CK(c->d_yhat.reserve(N * L.pstride * 8));   // theta_in
    CK(c->d_lo.reserve(N * L.pstride * 8));     // grad_out
    CK(cudaMemcpyAsync(c->d_ds.p, h_ds, (size_t)R * 8, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->d_y.p, h_y, (size_t)R * y_elem(y_dtype), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->d_yhat.p, h_theta, N * L.pstride * 8, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(c->d_lo.p, 0, N * L.pstride * 8, c->stream));
    rc = begin_fit_call(c);
    if (rc) return rc;
    rc = fit_impl(c, c->ws[0], opts, (const int64_t*)c->d_ds.p, c->d_y.p, y_dtype, h_offsets, n_series, floor, cap_multiplier,
                  nullptr, (double*)c->d_params.p, (double*)c->d_tchange.p, (int32_t*)c->d_mi32.p,
                  (int64_t*)c->d_mi64.p, (double*)c->d_mf64.p, (const double*)c->d_yhat.p, (double*)c->d_lo.p);
    if (rc) return rc;
    std::vector<double> mf(N * 4);
    CK(cudaMemcpyAsync(h_grad, c->d_lo.p, N * L.pstride * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_meta_i32, c->d_mi32.p, N * 8 * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(mf.data(), c->d_mf64.p, N * 4 * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (size_t i = 0; i < N; ++i) h_f[i] = mf[i * 4 + 3];
    return PB200_OK;
}

PB200_API int pb200_fit_host(pb200_ctx* c, const pb200_options* opts, const int64_t* h_ds, const void* h_y, int32_t y_dtype,
                   const int64_t* h_offsets, int64_t n_series, double floor, double cap_multiplier, const double* h_cap,
                   double* h_params, double* h_tchange, int32_t* h_meta_i32, int64_t* h_meta_i64, double* h_meta_f64) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    int rc = check_opts(opts);
    if (rc) return rc;
    if (n_series <= 0) return n_series == 0 ? PB200_OK : fail(PB200_E_ARG, "n_series");
    if (!h_ds || !h_y || !h_offsets || !h_params || !h_tchange || !h_meta_i32 || !h_meta_i64 || !h_meta_f64)
        return fail(PB200_E_ARG, "null pointer");
    if (y_dtype < 0 || y_dtype > 2) return fail(PB200_E_ARG, "y_dtype");
    pb200_layout L;
    pb200_get_layout(opts, &L);
    CK(cudaSetDevice(c->device));
    const int64_t R = h_offsets[n_series];
    const size_t N = (size_t)n_series;
    CK(c->d_ds.reserve((size_t)R * 8));
    CK(c->d_y.reserve((size_t)R * y_elem(y_dtype)));
    CK(c->d_params.reserve(N * L.pstride * 8));
    CK(c->d_tchange.reserve(N * L.smax * 8));
    CK(c->d_mi32.reserve(N * 8 * 4));
    CK(c->d_mi64.reserve(N * 2 * 8));
    CK(c->d_mf64.reserve(N * 4 * 8));
    if (h_cap) CK(c->d_cap.reserve(N * 8));
    CK(c->d_nq_all.reserve((N + 2 * 16 + 2) * 4));
    CK(c->d_offsets_full.reserve((N + 1) * 8));
    rc = begin_fit_call(c);
    if (rc) return rc;
    CK(cudaMemcpyAsync(c->d_offsets_full.p, h_offsets, (N + 1) * 8, cudaMemcpyHostToDevice, c->ws[0].stream));
    // series chunks with (nearly) equal rows, alternating over the two workspaces / streams: copy in, fit, copy out
    int nch = c->host_chunks;
    if (n_series < 4096 * (int64_t)nch || R < (int64_t)nch * (1 << 20)) nch = 1;
    const size_t ye = y_elem(y_dtype);
    std::vector<int64_t> cut(nch + 1, 0), hoff;
    cut[nch] = n_series;
    for (int k = 1; k < nch; ++k)
        cut[k] = std::lower_bound(h_offsets, h_offsets + n_series + 1, R * k / nch) - h_offsets;
    for (int k = 0; k < nch; ++k) {
        const int64_t s0 = cut[k], s1 = cut[k + 1], nk = s1 - s0;
        if (nk <= 0) continue;
        FitWs& w = c->ws[k % NWS];
        const int64_t r0 = h_offsets[s0], rk = h_offsets[s1] - r0;
        CK(cudaMemcpyAsync((char*)c->d_ds.p + (size_t)r0 * 8, h_ds + r0, (size_t)rk * 8, cudaMemcpyHostToDevice, w.stream));
        CK(cudaMemcpyAsync((char*)c->d_y.p + (size_t)r0 * ye, (const char*)h_y + (size_t)r0 * ye, (size_t)rk * ye,
                           cudaMemcpyHostToDevice, w.stream));
        const double* dcap = nullptr;
        if (h_cap) {
            CK(cudaMemcpyAsync((double*)c->d_cap.p + s0, h_cap + s0, (size_t)nk * 8, cudaMemcpyHostToDevice, w.stream));
            dcap = (const double*)c->d_cap.p + s0;
        }
        hoff.resize((size_t)nk + 1);
        for (int64_t i = 0; i <= nk; ++i) hoff[(size_t)i] = h_offsets[s0 + i] - r0;
        rc = fit_impl(c, w, opts, (const int64_t*)c->d_ds.p + r0, (const char*)c->d_y.p + (size_t)r0 * ye, y_dtype, hoff.data(), nk,
                      floor, cap_multiplier, dcap, (double*)c->d_params.p + (size_t)s0 * L.pstride,
                      (double*)c->d_tchange.p + (size_t)s0 * L.smax, (int32_t*)c->d_mi32.p + (size_t)s0 * 8,
                      (int64_t*)c->d_mi64.p + (size_t)s0 * 2, (double*)c->d_mf64.p + (size_t)s0 * 4, nullptr, nullptr, nullptr, 0,
                      n_series, (int*)c->d_nq_all.p + s0 + 2 * k);
        if (rc) return rc;
    }
    // Newton retries, normally none: the per-chunk queue lengths are read back once every chunk's fit is done
    if (opts->algorithm != PB200_ALG_LBFGS) {
        for (FitWs& w : c->ws) CK(cudaStreamSynchronize(w.stream));
        for (int k = 0; k < nch; ++k) {
            const int64_t s0 = cut[k], nk = cut[k + 1] - s0;
            if (nk <= 0) continue;
            int* nq = (int*)c->d_nq_all.p + s0 + 2 * k;
            int cnt = 0;
            CK(cudaMemcpy(&cnt, nq, 4, cudaMemcpyDeviceToHost));
            if (cnt <= 0) continue;
            // chunk-local series indices, the call's un-rebased offsets: ds / y are passed whole
            rc = launch_newton(c, c->ws[k % NWS].stream, opts, (const int64_t*)c->d_ds.p, c->d_y.p, y_dtype,
                               (const int64_t*)c->d_offsets_full.p + s0, nk, nq, (double*)c->d_params.p + (size_t)s0 * L.pstride,
                               (double*)c->d_tchange.p + (size_t)s0 * L.smax, (int32_t*)c->d_mi32.p + (size_t)s0 * 8,
                               (int64_t*)c->d_mi64.p + (size_t)s0 * 2, (double*)c->d_mf64.p + (size_t)s0 * 4);
            if (rc) return rc;
        }
    }
    // results back, chunk by chunk, only after EVERY chunk is enqueued: a copy into pageable caller memory blocks the
    // host until its stream gets there, and issued inside the loop above it serialised the chunks (r2h: e2e / value 0.71)
    for (int k = 0; k < nch; ++k) {
        const int64_t s0 = cut[k], nk = cut[k + 1] - s0;
        if (nk <= 0) continue;
        FitWs& w = c->ws[k % NWS];
        const size_t n0 = (size_t)s0, nn = (size_t)nk;
        CK(cudaMemcpyAsync(h_params + n0 * L.pstride, (double*)c->d_params.p + n0 * L.pstride, nn * L.pstride * 8, cudaMemcpyDeviceToHost, w.stream));
        CK(cudaMemcpyAsync(h_tchange + n0 * L.smax, (double*)c->d_tchange.p + n0 * L.smax, nn * L.smax * 8, cudaMemcpyDeviceToHost, w.stream));
        CK(cudaMemcpyAsync(h_meta_i32 + n0 * 8, (int32_t*)c->d_mi32.p + n0 * 8, nn * 8 * 4, cudaMemcpyDeviceToHost, w.stream));
        CK(cudaMemcpyAsync(h_meta_i64 + n0 * 2, (int64_t*)c->d_mi64.p + n0 * 2, nn * 2 * 8, cudaMemcpyDeviceToHost, w.stream));
        CK(cudaMemcpyAsync(h_meta_f64 + n0 * 4, (double*)c->d_mf64.p + n0 * 4, nn * 4 * 8, cudaMemcpyDeviceToHost, w.stream));
    }
    for (FitWs& w : c->ws) CK(cudaStreamSynchronize(w.stream));
    return PB200_OK;
}

PB200_API int pb200_fit_trace_host(pb200_ctx* c, const pb200_options* opts, const int64_t* h_ds, const void* h_y, int32_t y_dtype,
                         const int64_t* h_offsets, int64_t n_series, double floor, double cap_multiplier, double* h_params,
                         double* h_tchange, int32_t* h_meta_i32, int64_t* h_meta_i64, double* h_meta_f64, double* h_trace,
                         int32_t trace_cap) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    int rc = check_opts(opts);
    if (rc) return rc;
    if (n_series <= 0) return n_series == 0 ? PB200_OK : fail(PB200_E_ARG, "n_series");
    if (!h_ds || !h_y || !h_offsets || !h_params || !h_tchange || !h_meta_i32 || !h_meta_i64 || !h_meta_f64 || !h_trace)
        return fail(PB200_E_ARG, "null pointer");
    if (y_dtype < 0 || y_dtype > 2) return fail(PB200_E_ARG, "y_dtype");
    if (trace_cap < 1 || (int64_t)trace_cap * n_series > (1LL << 26)) return fail(PB200_E_ARG, "trace_cap");
    pb200_layout L;
    pb200_get_layout(opts, &L);
    CK(cudaSetDevice(c->device));
    const int64_t R = h_offsets[n_series];
    const size_t N = (size_t)n_series, tbytes = N * (size_t)trace_cap * 4 * 8;
    CK(c->d_ds.reserve((size_t)R * 8));
    CK(c->d_y.reserve((size_t)R * y_elem(y_dtype)));
    CK(c->d_params.reserve(N * L.pstride * 8));
    CK(c->d_tchange.reserve(N * L.smax * 8));
    CK(c->d_mi32.reserve(N * 8 * 4));
    CK(c->d_mi64.reserve(N * 2 * 8));
    CK(c->d_mf64.reserve(N * 4 * 8));
    CK(c->d_trace.reserve(tbytes));
    CK(cudaMemcpyAsync(c->d_ds.p, h_ds, (size_t)R * 8, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->d_y.p, h_y, (size_t)R * y_elem(y_dtype), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(c->d_trace.p, 0, tbytes, c->stream));
    rc = begin_fit_call(c);
    if (rc) return rc;
    rc = fit_impl(c, c->ws[0], opts, (const int64_t*)c->d_ds.p, c->d_y.p, y_dtype, h_offsets, n_series, floor, cap_multiplier, nullptr,
                  (double*)c->d_params.p, (double*)c->d_tchange.p, (int32_t*)c->d_mi32.p, (int64_t*)c->d_mi64.p,
                  (double*)c->d_mf64.p, nullptr, nullptr, (double*)c->d_trace.p, trace_cap);
    if (rc) return rc;
    CK(cudaMemcpyAsync(h_params, c->d_params.p, N * L.pstride * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_tchange, c->d_tchange.p, N * L.smax * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_meta_i32, c->d_mi32.p, N * 8 * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_meta_i64, c->d_mi64.p, N * 2 * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_meta_f64, c->d_mf64.p, N * 4 * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_trace, c->d_trace.p, tbytes, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return PB200_OK;
}

PB200_API int pb200_make_future_device(pb200_ctx* c, const int64_t* d_last_ds, int64_t n_models, int32_t horizon, int64_t freq_ns,
                             int64_t* d_future_ds) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    if (n_models < 0 || horizon < 0) return fail(PB200_E_ARG, "sizes");
    if (n_models == 0 || horizon == 0) return PB200_OK;
    if (!d_last_ds || !d_future_ds) return fail(PB200_E_ARG, "null pointer");
    CK(cudaSetDevice(c->device));
    const int64_t n = n_models * horizon;
    const int grid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)c->sms * 16);
    pb200::make_future_kernel<<<grid, 256, 0, c->stream>>>((const long long*)d_last_ds, n_models, horizon, freq_ns,
                                                           (long long*)d_future_ds);
    CK(cudaGetLastError());
    c->launches++;
    return PB200_OK;
}

PB200_API int pb200_predict_device(pb200_ctx* c, const pb200_options* opts, const double* d_params, const double* d_tchange,
                         const int32_t* d_meta_i32, const int64_t* d_meta_i64, const double* d_meta_f64,
                         int64_t n_models, const int64_t* d_future_ds, int32_t horizon, const double* d_floor,
                         const double* d_cap, uint64_t seed, double* d_yhat, double* d_yhat_lower, double* d_yhat_upper,
                         int32_t* d_yhat_int) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    int rc = check_opts(opts);
    if (rc) return rc;
    if (n_models < 0 || horizon < 0 || n_models > (1LL << 30)) return fail(PB200_E_ARG, "sizes");
    if (n_models == 0 || horizon == 0) return PB200_OK;
    if (!d_params || !d_tchange || !d_meta_i32 || !d_meta_i64 || !d_meta_f64 || !d_future_ds || !d_floor || !d_cap ||
        !d_yhat || !d_yhat_int)
        return fail(PB200_E_ARG, "null pointer");
    pb200_layout L;
    pb200_get_layout(opts, &L);
    CK(cudaSetDevice(c->device));
    pb200::PredictArgs a;
    a.params = d_params;
    a.tchange = d_tchange;
    a.meta_i32 = d_meta_i32;
    a.meta_i64 = (const long long*)d_meta_i64;
    a.meta_f64 = d_meta_f64;
    a.future_ds = (const long long*)d_future_ds;
    a.floor = d_floor;
    a.cap = d_cap;
    a.n_models = (int)n_models;
    a.horizon = horizon;
    a.smax = L.smax;
    a.kmax = L.kmax;
    a.pstride = L.pstride;
    a.growth = opts->growth;
    a.mult = opts->multiplicative ? 1 : 0;
    a.yhat = d_yhat;
    a.trend = nullptr;
    a.yhat_int = d_yhat_int;
    {
        // one CTA per (model, 1024 future points): the per-model prologue (parameters, the serial gamma recurrence) is paid
        // once for config #5's 672 periods instead of three times
        dim3 grid((unsigned)n_models, (unsigned)std::min((horizon + 1023) / 1024, 64));
        pb200::predict_kernel<<<grid, 256, 0, c->stream>>>(a);
        CK(cudaGetLastError());
        c->launches++;
    }
    if (d_yhat_lower && d_yhat_upper && opts->uncertainty_samples > 0) {
        rc = pb200::launch_mc(c->stream, c->sms, a, opts->uncertainty_samples, opts->interval_width, seed, d_yhat_lower,
                              d_yhat_upper);
        if (rc == -1) return fail(PB200_E_UNSUPPORTED, "uncertainty_samples must be in [2, 1024]");
        if (rc) return fail(PB200_E_CUDA, "mc kernel launch", cudaGetLastError());
        c->launches++;
    }
    return PB200_OK;
}

PB200_API int pb200_predict_host(pb200_ctx* c, const pb200_options* opts, const double* h_params, const double* h_tchange,
                       const int32_t* h_meta_i32, const int64_t* h_meta_i64, const double* h_meta_f64, int64_t n_models,
                       const int64_t* h_future_ds, int32_t horizon, const double* h_floor, const double* h_cap,
                       uint64_t seed, double* h_yhat, double* h_yhat_lower, double* h_yhat_upper, int32_t* h_yhat_int) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    int rc = check_opts(opts);
    if (rc) return rc;
    if (n_models <= 0 || horizon <= 0) return (n_models == 0 || horizon == 0) ? PB200_OK : fail(PB200_E_ARG, "sizes");
    if (!h_params || !h_tchange || !h_meta_i32 || !h_meta_i64 || !h_meta_f64 || !h_future_ds || !h_floor || !h_cap ||
        !h_yhat || !h_yhat_int)
        return fail(PB200_E_ARG, "null pointer");
    pb200_layout L;
    pb200_get_layout(opts, &L);
    CK(cudaSetDevice(c->device));
    const size_t N = (size_t)n_models, NH = N * (size_t)horizon;
    const bool mc = h_yhat_lower && h_yhat_upper && opts->uncertainty_samples > 0;
    CK(c->d_params.reserve(N * L.pstride * 8));
    CK(c->d_tchange.reserve(N * L.smax * 8));
    CK(c->d_mi32.reserve(N * 8 * 4));
    CK(c->d_mi64.reserve(N * 2 * 8));
    CK(c->d_mf64.reserve(N * 4 * 8));
    CK(c->d_fut.reserve(NH * 8));
    CK(c->d_floor.reserve(N * 8));
    CK(c->d_cap.reserve(N * 8));
    CK(c->d_yhat.reserve(NH * 8));
    CK(c->d_yint.reserve(NH * 4));
    if (mc) {
        CK(c->d_lo.reserve(NH * 8));
        CK(c->d_hi.reserve(NH * 8));
    }
    cudaStream_t st = c->stream;
    CK(cudaMemcpyAsync(c->d_params.p, h_params, N * L.pstride * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_tchange.p, h_tchange, N * L.smax * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_mi32.p, h_meta_i32, N * 8 * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_mi64.p, h_meta_i64, N * 2 * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_mf64.p, h_meta_f64, N * 4 * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_fut.p, h_future_ds, NH * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_floor.p, h_floor, N * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_cap.p, h_cap, N * 8, cudaMemcpyHostToDevice, st));
    rc = pb200_predict_device(c, opts, (const double*)c->d_params.p, (const double*)c->d_tchange.p,
                              (const int32_t*)c->d_mi32.p, (const int64_t*)c->d_mi64.p, (const double*)c->d_mf64.p,
                              n_models, (const int64_t*)c->d_fut.p, horizon, (const double*)c->d_floor.p,
                              (const double*)c->d_cap.p, seed, (double*)c->d_yhat.p, mc ? (double*)c->d_lo.p : nullptr,
                              mc ? (double*)c->d_hi.p : nullptr, (int32_t*)c->d_yint.p);
    if (rc) return rc;
    CK(cudaMemcpyAsync(h_yhat, c->d_yhat.p, NH * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h_yhat_int, c->d_yint.p, NH * 4, cudaMemcpyDeviceToHost, st));
    if (mc) {
        CK(cudaMemcpyAsync(h_yhat_lower, c->d_lo.p, NH * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(h_yhat_upper, c->d_hi.p, NH * 8, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    return PB200_OK;
}

// ---- forecast CSV rows formatted on the device (csv_kernel.cuh) ----
static int csv_args(pb200::csv::CsvArgs& a, const int32_t* sid, const int32_t* did, const int64_t* ds, const int32_t* qty, int64_t n,
                    const char* created, int32_t created_len) {
    if (created_len < 0 || created_len > pb200::csv::MAX_CREATED) return fail(PB200_E_ARG, "created_timestamp longer than 64 bytes");
    if (created_len && !created) return fail(PB200_E_ARG, "null pointer");
    a.sid = sid; a.did = did; a.ds_ns = (const long long*)ds; a.qty = qty; a.n = n; a.created_len = created_len;
    memset(a.created, 0, sizeof(a.created));
    if (created_len) memcpy(a.created, created, (size_t)created_len);
    a.row_len = nullptr; a.row_off = nullptr; a.out = nullptr;
    return PB200_OK;
}

PB200_API int pb200_forecast_csv_lengths_device(pb200_ctx* c, const int32_t* d_series_id, const int32_t* d_dim_id,
                                                const int32_t* d_quantity, int64_t n_rows, int32_t created_len,
                                                int64_t* d_row_len) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    if (n_rows < 0) return fail(PB200_E_ARG, "sizes");
    if (n_rows == 0) return PB200_OK;
    if (!d_series_id || !d_dim_id || !d_quantity || !d_row_len) return fail(PB200_E_ARG, "null pointer");
    CK(cudaSetDevice(c->device));
    pb200::csv::CsvArgs a;
    char pad[pb200::csv::MAX_CREATED] = {0};
    int rc = csv_args(a, d_series_id, d_dim_id, nullptr, d_quantity, n_rows, pad, created_len);
    if (rc) return rc;
    a.row_len = (long long*)d_row_len;
    const int grid = (int)std::min<int64_t>((n_rows + 255) / 256, (int64_t)c->sms * 16);
    pb200::csv::csv_lengths_kernel<<<grid, 256, 0, c->stream>>>(a);
    CK(cudaGetLastError());
    c->launches++;
    return PB200_OK;
}

PB200_API int pb200_forecast_csv_rows_device(pb200_ctx* c, const int32_t* d_series_id, const int32_t* d_dim_id,
                                             const int64_t* d_ds_ns, const int32_t* d_quantity, int64_t n_rows,
                                             const char* h_created, int32_t created_len, const int64_t* d_row_off,
                                             uint8_t* d_out) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    if (n_rows < 0) return fail(PB200_E_ARG, "sizes");
    if (n_rows == 0) return PB200_OK;
    if (!d_series_id || !d_dim_id || !d_ds_ns || !d_quantity || !d_row_off || !d_out) return fail(PB200_E_ARG, "null pointer");
    CK(cudaSetDevice(c->device));
    pb200::csv::CsvArgs a;
    int rc = csv_args(a, d_series_id, d_dim_id, d_ds_ns, d_quantity, n_rows, h_created, created_len);
    if (rc) return rc;
    a.row_off = (const long long*)d_row_off;
    a.out = d_out;
    const int64_t warps = (n_rows + 31) / 32;
    const int grid = (int)std::min<int64_t>((warps + 3) / 4, (int64_t)c->sms * 8);
    pb200::csv::csv_rows_kernel<<<grid, 128, 0, c->stream>>>(a);
    CK(cudaGetLastError());
    c->launches++;
    return PB200_OK;
}

PB200_API int32_t pb200_forecast_csv_row_host(int32_t series_id, int32_t dim_id, int64_t ds_ns, int32_t quantity,
                                              const char* created, int32_t created_len, char* out) {
    if (created_len < 0 || created_len > pb200::csv::MAX_CREATED || !out || (created_len && !created)) return -1;
    char* e = pb200::csv::put_row(out, series_id, dim_id, ds_ns, quantity, created, created_len);
    const int n = (int)(e - out);
    return n == pb200::csv::row_len(series_id, dim_id, quantity, created_len) ? n : -1;
}

// ---- modeler input CSV parsed on the device (csv_reader.cuh) ----
static_assert(PB200_INPUT_CSV_TILE == pb200::csvin::TILE, "tile size of the count / index passes");

static int input_args(pb200::csvin::InArgs& a, const uint8_t* text, int64_t n_bytes) {
    memset(&a, 0, sizeof a);
    if (n_bytes < 0) return fail(PB200_E_ARG, "sizes");
    if (n_bytes && !text) return fail(PB200_E_ARG, "null pointer");
    if ((uintptr_t)text % 16) return fail(PB200_E_ARG, "d_text must be 16-byte aligned");
    a.text = text;
    a.n_bytes = n_bytes;
    return PB200_OK;
}

static int input_tile_grid(const pb200_ctx* c, int64_t n_bytes) {
    const int64_t tiles = (n_bytes + pb200::csvin::TILE - 1) / pb200::csvin::TILE;
    return (int)std::min<int64_t>((tiles + 7) / 8, (int64_t)c->sms * 8);
}

PB200_API int pb200_input_csv_count_device(pb200_ctx* c, const uint8_t* d_text, int64_t n_bytes, int64_t* d_tile_count) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    pb200::csvin::InArgs a;
    int rc = input_args(a, d_text, n_bytes);
    if (rc) return rc;
    if (n_bytes == 0) return PB200_OK;
    if (!d_tile_count) return fail(PB200_E_ARG, "null pointer");
    CK(cudaSetDevice(c->device));
    a.tile_count = (long long*)d_tile_count;
    pb200::csvin::input_count_kernel<<<input_tile_grid(c, n_bytes), 256, 0, c->stream>>>(a);
    CK(cudaGetLastError());
    c->launches++;
    return PB200_OK;
}

PB200_API int pb200_input_csv_index_device(pb200_ctx* c, const uint8_t* d_text, int64_t n_bytes, const int64_t* d_tile_off,
                                           int64_t* d_row_end) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    pb200::csvin::InArgs a;
    int rc = input_args(a, d_text, n_bytes);
    if (rc) return rc;
    if (n_bytes == 0) return PB200_OK;
    if (!d_tile_off || !d_row_end) return fail(PB200_E_ARG, "null pointer");
    CK(cudaSetDevice(c->device));
    a.tile_off = (const long long*)d_tile_off;
    a.row_end = (long long*)d_row_end;
    pb200::csvin::input_index_kernel<<<input_tile_grid(c, n_bytes), 256, 0, c->stream>>>(a);
    CK(cudaGetLastError());
    c->launches++;
    return PB200_OK;
}

PB200_API int pb200_input_csv_parse_device(pb200_ctx* c, const uint8_t* d_text, const int64_t* d_row_end, int64_t n_rows,
                                           const int64_t* d_file_start, const int32_t* d_file_sid, int32_t n_files,
                                           int32_t* d_series_id, int32_t* d_dim_id, int64_t* d_ds_ns, int32_t* d_quantity,
                                           uint8_t* d_quantity_valid, int64_t* d_refused) {
    if (!c) return fail(PB200_E_ARG, "ctx is null");
    if (n_rows < 0 || n_files < 0 || (n_rows > 0 && n_files == 0)) return fail(PB200_E_ARG, "sizes");
    if (!d_refused) return fail(PB200_E_ARG, "null pointer");
    CK(cudaSetDevice(c->device));
    CK(cudaMemsetAsync(d_refused, 0, 8, c->stream));
    CK(cudaMemsetAsync(d_refused + 1, 0xFF, 8, c->stream));
    if (n_rows == 0) return PB200_OK;
    if (!d_row_end || !d_file_start || !d_file_sid || !d_series_id || !d_dim_id || !d_ds_ns || !d_quantity || !d_quantity_valid)
        return fail(PB200_E_ARG, "null pointer");
    pb200::csvin::InArgs a;
    int rc = input_args(a, d_text, 1);
    if (rc) return rc;
    a.row_end = (long long*)d_row_end;
    a.n_rows = n_rows;
    a.file_start = (const long long*)d_file_start;
    a.file_sid = d_file_sid;
    a.n_files = n_files;
    a.sid = d_series_id;
    a.dim = d_dim_id;
    a.ds = (long long*)d_ds_ns;
    a.qty = d_quantity;
    a.qty_valid = d_quantity_valid;
    a.refused = (unsigned long long*)d_refused;
    const int64_t warps = (n_rows + 31) / 32;
    const int grid = (int)std::min<int64_t>((warps + 3) / 4, (int64_t)c->sms * 16);
    pb200::csvin::input_parse_kernel<<<grid, 128, 0, c->stream>>>(a);
    CK(cudaGetLastError());
    c->launches++;
    return PB200_OK;
}

PB200_API int32_t pb200_input_csv_row_host(const char* line, int64_t len, int32_t* dim_id, int64_t* ds_ns, int32_t* quantity,
                                           int32_t* quantity_valid) {
    if (len < 0 || (len && !line) || !dim_id || !ds_ns || !quantity || !quantity_valid) return -1;
    const unsigned char* p = (const unsigned char*)line;
    bool qv = false;
    const bool ok = pb200::csvin::parse_row(p, p + len, *dim_id, *ds_ns, *quantity, qv);
    *quantity_valid = ok && qv;
    return ok ? 1 : 0;
}

}  // extern "C"
