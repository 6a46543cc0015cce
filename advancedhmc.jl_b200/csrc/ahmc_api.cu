// ahmc_api.cu -- the C ABI of libahmc_b200 (include/ahmc_b200.h): context, models, argument
// validation, host-buffer staging and kernel dispatch.  No torch types, no exceptions across the ABI.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <new>
#include <string>
#include <vector>

// defaults of the host-buffer lane (see leapfrog_host_pipelined), chosen by measurement on B200 (profiles/README.md,
// "host-buffer lane"): page-locked buffers are read and written by the kernel directly in ONE launch whose residency
// is capped at one CTA per SM, so the grid runs in staggered waves and uploads overlap downloads (0.36 ms against
// 0.48 ms uncapped and 0.45-0.50 ms for the best copy-engine pipeline at 4096 x 128); pageable buffers go through
// the copy engines in two chunks.
#define AHMC_PIPE_DIRECT_CHUNKS 1
#define AHMC_PIPE_CE_CHUNKS 2
#define AHMC_PIPE_DIRECT_OCC 1  // resident CTAs per SM of a direct-access launch (0 = no cap)

#include "ahmc_kernels.cuh"

using namespace ahmc;

struct DevBuf {  // grow-only device buffer (see grow())
    char* p = nullptr;
    size_t bytes = 0;
};

struct ahmc_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    int64_t launches = 0;
    int* d_min_break = nullptr;   // device int for COMPAT_BREAK_ALL
    DevBuf arena;          // HOST_BUFFERS staging
    DevBuf nuts_scratch;   // per-chain NUTS tree workspace
    DevBuf adapt_scratch;  // adaptor statistics: last-block counter, per-block partials
    DevBuf mn_scratch;     // multinomial-static per-chain energy tape
    DevBuf dense_scratch;  // K4: padded Minv, norms, per-chain fallback mask
    DevBuf coop_scratch;   // cooperative NUTS products: Minv and cholU with padded columns (coop_lds)
    DevBuf split_scratch;  // callback (split-step) mode workspace
    // host-buffer pipeline: H2D stream, compute stream (= stream), D2H stream, one event pair per chunk
    static constexpr int kMaxPipeChunks = 32, kPipeStreams = 5;  // 3 upload, 1 download, 1 second compute
    cudaStream_t pipe[kPipeStreams] = {};
    cudaEvent_t ev_a = nullptr, ev_join[kPipeStreams] = {};
    cudaEvent_t ev_in[kMaxPipeChunks][3] = {}, ev_k[kMaxPipeChunks] = {};
    // transport choice of the host-buffer lane, measured per problem shape on its first calls (leapfrog_host_pipelined)
    struct PipeTune {
        int64_t N;
        int32_t D;
        int key;       // has_g | has_dr << 1 | per-chain eps << 2 | per-chain Minv << 3
        int calls;     // trial calls made so far
        int chosen;    // -1 while measuring
        double best_ms[8];
    };
    std::vector<PipeTune> tune;
    std::string transport = "none";  // what the last host-buffer call used (ahmc_last_transport)
};

struct ahmc_model {
    int kind = 0;
    int D = 0;
    double* d_p0 = nullptr;
    double* d_p1 = nullptr;
    double* d_p1_pad = nullptr;  // DENSE_GAUSS: precision zero-padded to Dp x Dp (K4), followed by |P|_inf
    double* d_p1_coop = nullptr; // DENSE_GAUSS: precision with columns padded to coop_lds(D) (cooperative NUTS products)
    int Dp = 0;
    double c0 = 0.0;
    ahmc_logp_grad_fn fn = nullptr;
    void* user = nullptr;
    UserModule* rtc = nullptr;  // AHMC_MODEL_USER: run-time compiled kernels
};

namespace {

int fail(ahmc_ctx* ctx, int code, const char* fmt, ...) {
    if (ctx) {
        char buf[4096];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        ctx->err = buf;
    }
    return code;
}

#define CU(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e__ = (call);                                                                      \
        if (e__ != cudaSuccess) {                                                                      \
            std::string ue__ = user_thread_error();                                                    \
            user_thread_error_clear();                                                                 \
            return fail(ctx, AHMC_ERR_CUDA, "%s failed: %s (%s:%d)%s%s", #call, cudaGetErrorString(e__), __FILE__, \
                        __LINE__, ue__.empty() ? "" : " -- ", ue__.c_str());                           \
        }                                                                                              \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
        cudaGetLastError();  // a stale error left by another library on this thread must not be blamed on our launches
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

constexpr size_t al256(size_t b) { return (b + 255) & ~(size_t)255; }

// Grows `b` to at least `need` bytes (allocating `cap` >= need, default need).  Queued work may still use the old
// allocation, so every stream of the context is drained before it is freed.
int grow(ahmc_ctx* ctx, DevBuf& b, size_t need, const char* what, size_t cap = 0) {
    if (need <= b.bytes) return AHMC_OK;
    if (b.p) {
        CU(cudaStreamSynchronize(ctx->stream));
        for (cudaStream_t s : ctx->pipe)
            if (s) CU(cudaStreamSynchronize(s));
        CU(cudaFree(b.p));
        b.p = nullptr;
        b.bytes = 0;
    }
    if (cap < need) cap = need;
    if (cudaMalloc((void**)&b.p, cap) != cudaSuccess) {
        b.p = nullptr;
        return fail(ctx, AHMC_ERR_NOMEM, "cudaMalloc(%zu) for the %s failed", cap, what);
    }
    b.bytes = cap;
    return AHMC_OK;
}

// Maps caller arrays to device arrays.  Device-pointer mode: identity, set at once (nothing is recorded, so that path
// never allocates).  HOST_BUFFERS mode: in / out / inout record the array; commit() carves every recorded array from
// the context arena, sets the device pointers and copies the inputs host->device on the context stream; finish()
// copies the outputs device->host.  Staged device pointers exist only after commit().
class Stager {
public:
    Stager(ahmc_ctx* c, bool host) : ctx_(c), host_(host) {}
    template <class T>
    void in(const T* h, size_t count, const T** d) { add(h, count * sizeof(T), d, true, false); }
    template <class T>
    void out(T* h, size_t count, T** d) { add(h, count * sizeof(T), d, false, true); }
    template <class T>
    void inout(T* h, size_t count, T** d) { add(h, count * sizeof(T), d, true, true); }
    int commit() {
        if (reqs_.empty()) return AHMC_OK;
        ahmc_ctx* ctx = ctx_;
        size_t need = 0;
        for (const Req& r : reqs_) need += al256(r.bytes);
        int rc = grow(ctx, ctx->arena, need, "staging arena", need + need / 4);
        if (rc) return rc;
        char* p = ctx->arena.p;
        for (Req& r : reqs_) {
            r.dev = p;
            set(r.slot, p);
            if (r.in) CU(cudaMemcpyAsync(p, r.h, r.bytes, cudaMemcpyHostToDevice, ctx->stream));
            p += al256(r.bytes);
        }
        return AHMC_OK;
    }
    int finish() {
        ahmc_ctx* ctx = ctx_;
        for (const Req& r : reqs_)
            if (r.out) CU(cudaMemcpyAsync((void*)r.h, r.dev, r.bytes, cudaMemcpyDeviceToHost, ctx->stream));
        return AHMC_OK;
    }
    bool host() const { return host_; }

private:
    struct Req {
        const void* h;
        size_t bytes;
        void* slot;  // the caller's T* that receives the device pointer
        bool in, out;
        void* dev;
    };
    // the slot is a T* of the caller's type: written bytewise, not through a void* lvalue
    static void set(void* slot, const void* p) { memcpy(slot, &p, sizeof p); }
    void add(const void* h, size_t bytes, void* slot, bool in, bool out) {
        if (!h || !host_) set(slot, h);
        else reqs_.push_back({h, bytes, slot, in, out, nullptr});
    }
    ahmc_ctx* ctx_;
    bool host_;
    std::vector<Req> reqs_;
};

int check_common(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N, bool streaming_ok = false) {
    if (!ctx) return AHMC_ERR_INVALID;
    if (D < 1) return fail(ctx, AHMC_ERR_INVALID, "D must be >= 1 (got %d)", D);
    if (N < 0) return fail(ctx, AHMC_ERR_INVALID, "N must be >= 0 (got %lld)", (long long)N);
    if (model) {
        if (model->D != D)
            return fail(ctx, AHMC_ERR_INVALID, "AxesMismatch: model has dimension %d but theta has %d rows", model->D, D);
    }
    if (metric) {
        if (metric->kind < AHMC_METRIC_UNIT || metric->kind > AHMC_METRIC_DENSE)
            return fail(ctx, AHMC_ERR_INVALID, "unknown metric kind %d", metric->kind);
        if (metric->kind != AHMC_METRIC_UNIT && !metric->Minv)
            return fail(ctx, AHMC_ERR_INVALID, "metric.Minv is NULL for a Diag/Dense metric");
        if (metric->kind == AHMC_METRIC_DIAG && metric->chain_stride != 0 && metric->chain_stride < D)
            return fail(ctx, AHMC_ERR_INVALID, "AxesMismatch: per-chain Minv stride %lld < D=%d (hamiltonian.jl:53-57)",
                        (long long)metric->chain_stride, D);
    }
    int G, E;
    if (!pick_layout(D, &G, &E)) {
        // D > 512: `step` and `phasepoint` stream the chain through registers tile by tile (ahmc_bigd.cu) for the separable
        // targets and the funnel with Unit / Diag metrics; everything else is register-resident and stops at 512
        if (streaming_ok && model && metric && bigd_supported(model->kind, metric->kind)) return AHMC_OK;
        return fail(ctx, AHMC_ERR_UNSUPPORTED,
                    "D=%d: this entry point / target / metric combination is register-resident (D <= 512); D > 512 is supported by "
                    "ahmc_leapfrog_f64 and ahmc_phasepoint_f64 for std-normal, diagonal-Gaussian and funnel targets with Unit / Diag metrics", D);
    }
    return AHMC_OK;
}

int check_pp(ahmc_ctx* ctx, const ahmc_phasepoint* z, int32_t D, const char* name, bool need_cache, int64_t N) {
    if (!z) return fail(ctx, AHMC_ERR_INVALID, "%s is NULL", name);
    if (N == 0) return AHMC_OK;  // empty batch: nothing is dereferenced
    if (!z->theta || !z->r) return fail(ctx, AHMC_ERR_INVALID, "%s.theta / %s.r is NULL", name, name);
    if (need_cache && (!z->lp_value || !z->lp_gradient || !z->lk_value))
        return fail(ctx, AHMC_ERR_INVALID, "%s.lp_value / lp_gradient / lk_value is NULL", name);
    if (z->ld < D)
        return fail(ctx, AHMC_ERR_INVALID, "%s.ld=%lld < D=%d: length(theta)==length(r)==length(gradient) violated (hamiltonian.jl:94)",
                    name, (long long)z->ld, D);
    return AHMC_OK;
}

size_t metric_minv_count(const ahmc_metric* m, int32_t D, int64_t N) {
    if (m->kind == AHMC_METRIC_DIAG) return m->chain_stride ? (size_t)m->chain_stride * (size_t)N : (size_t)D;
    if (m->kind == AHMC_METRIC_DENSE) return (size_t)D * D;
    return 0;
}

ModelDev model_dev(const ahmc_model* m) { return ModelDev{m->kind, m->D, m->d_p0, m->d_p1, m->c0, m->rtc, m->d_p1_coop}; }

// stage the metric descriptor (device or host pointers) into a MetricDev
void stage_metric(Stager& st, const ahmc_metric* m, int32_t D, int64_t N, MetricDev* out) {
    out->kind = m->kind;
    out->chain_stride = m->kind == AHMC_METRIC_DIAG ? m->chain_stride : 0;
    out->Minv_coop = nullptr;
    out->cholU_coop = nullptr;
    st.in(m->Minv, metric_minv_count(m, D, N), &out->Minv);
    st.in(m->kind == AHMC_METRIC_DENSE ? m->cholU : (const double*)nullptr, (size_t)D * D, &out->cholU);
}

int finish_call(ahmc_ctx* ctx, Stager& st, uint32_t flags) {
    int rc = st.finish();
    if (rc) return rc;
    if (!(flags & AHMC_FLAG_ASYNC) || st.host()) CU(cudaStreamSynchronize(ctx->stream));
    return AHMC_OK;
}


// ---- split-step (callback) mode --------------------------------------------------------------------------------
struct SplitWork {
    double* cb_lp;
    double* cb_grad;
    double* r0;
    double* lk0;
    uint32_t* status;
    int32_t* steps;
    int* flag;
};

int split_workspace(ahmc_ctx* ctx, int32_t D, int64_t N, int64_t ld, SplitWork* w) {
    const size_t need = al256((size_t)N * 8) + al256((size_t)ld * N * 8) + al256((size_t)D * N * 8) + al256((size_t)N * 8) +
                        al256((size_t)N * 4) * 2 + 256;
    int rc = grow(ctx, ctx->split_scratch, need, "split-step workspace");
    if (rc) return rc;
    char* p = ctx->split_scratch.p;
    w->cb_lp = (double*)p; p += al256((size_t)N * 8);
    w->cb_grad = (double*)p; p += al256((size_t)ld * N * 8);
    w->r0 = (double*)p; p += al256((size_t)D * N * 8);
    w->lk0 = (double*)p; p += al256((size_t)N * 8);
    w->status = (uint32_t*)p; p += al256((size_t)N * 4);
    w->steps = (int32_t*)p; p += al256((size_t)N * 4);
    w->flag = (int*)p;
    return AHMC_OK;
}

// user closure on the context stream: lp[N], grad[D x N] <- theta
int call_user(ahmc_ctx* ctx, const ahmc_model* model, const double* th, double* lp, double* grad, int32_t D, int64_t N,
              int64_t ld) {
    int rc = model->fn(model->user, th, lp, grad, D, N, ld, (void*)ctx->stream);
    if (rc != 0) return fail(ctx, AHMC_ERR_CALLBACK, "user gradient callback returned %d", rc);
    return AHMC_OK;
}

// n leapfrog steps in split mode on DEVICE work arrays (th, r, g, lp, lk[, dr]); status/steps are device arrays
int split_trajectory(ahmc_ctx* ctx, const ahmc_model* model, const MetricDev& md, int32_t D, int64_t N, double eps,
                     const double* eps_chain, int n_abs, int fwd, double temper_alpha, double* th, double* r, double* g,
                     double* lp, double* lk, double* dr, int64_t ld, uint32_t* status, int32_t* steps, const SplitWork& w,
                     bool compat, int* nl) {
    CU(cudaMemsetAsync(status, 0, (size_t)N * 4, ctx->stream));
    if (steps) CU(cudaMemsetAsync(steps, 0, (size_t)N * 4, ctx->stream));
    CU(cudaMemsetAsync(w.flag, 0, sizeof(int), ctx->stream));
    const double sa = temper_alpha > 0.0 ? sqrt(temper_alpha) : 1.0;
    for (int i = 1; i <= n_abs; ++i) {
        SplitArgs a{};
        a.metric = md;
        a.D = D;
        a.N = N;
        a.eps = eps;
        a.eps_chain = eps_chain;
        a.fwd = fwd;
        a.mul = temper_alpha > 0.0 ? ((2 * (i - 1) + 1 <= n_abs) ? sa : 1.0 / sa) : 1.0;
        a.step_index = i;
        a.th = th; a.r = r; a.g = g; a.lp = lp; a.lk = lk; a.dr = dr;
        a.cb_lp = w.cb_lp; a.cb_grad = w.cb_grad;
        a.ld = ld;
        a.status = status; a.steps_done = steps; a.any_nonfinite = w.flag;
        CU(launch_kick_drift(a, ctx->stream, nl));
        int rc = call_user(ctx, model, th, w.cb_lp, w.cb_grad, D, N, ld);
        if (rc) return rc;
        a.mul = temper_alpha > 0.0 ? ((2 * (i - 1) + 2 <= n_abs) ? sa : 1.0 / sa) : 1.0;
        CU(launch_kick_energy(a, ctx->stream, nl));
        if (compat) {  // reference quirk Q1: first non-finite chain stops everyone (hamiltonian.jl:141-142)
            int f = 0;
            CU(cudaMemcpyAsync(&f, w.flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaStreamSynchronize(ctx->stream));
            if (f) break;
        }
    }
    return AHMC_OK;
}

// K4 (tiled DMMA trajectory) takes GEMM-shaped operators: a Gaussian target, a metric shared by all chains, a dense
// matrix on either side, a tile shape for D, and neither exact checks, tempering nor COMPAT_BREAK_ALL.
bool dense_eligible(const ahmc_model* model, const MetricDev& metric, uint32_t flags, double temper_alpha, bool compat,
                    bool has_g, int32_t D) {
    const bool gauss = model->kind == AHMC_MODEL_STD_NORMAL || model->kind == AHMC_MODEL_DIAG_GAUSS ||
                       model->kind == AHMC_MODEL_DENSE_GAUSS;
    const bool metric_ok = metric.kind != AHMC_METRIC_DIAG || metric.chain_stride == 0;
    const bool has_dense = model->kind == AHMC_MODEL_DENSE_GAUSS || metric.kind == AHMC_METRIC_DENSE;
    int Dp, RB, CB;
    return gauss && metric_ok && has_dense && !compat && has_g && !(flags & AHMC_FLAG_EXACT_CHECKS) && !(temper_alpha > 0.0) &&
           dense_tile_shape(D, &Dp, &RB, &CB) && (model->kind != AHMC_MODEL_DENSE_GAUSS || model->d_p1_pad);
}

// K4 trajectory of a dense_eligible configuration; chains of tiles it declines (magnitude proof not met) are redone by
// the exact warp-per-chain kernel from the untouched inputs.  `a` holds DEVICE pointers.
int dense_trajectory(ahmc_ctx* ctx, const ahmc_model* model, const LeapfrogArgs& a, int n_abs, double eps, int* nl) {
    const int D = a.D;
    const long long N = a.N;
    int Dp, RB, CB;
    dense_tile_shape(D, &Dp, &RB, &CB);
    const size_t need = al256(dense_mat_doubles(Dp) * 8) + al256(16) + al256((size_t)N);
    int rc = grow(ctx, ctx->dense_scratch, need, "dense workspace");
    if (rc) return rc;
    double* Mpad = (double*)ctx->dense_scratch.p;
    double* norms = (double*)(ctx->dense_scratch.p + al256(dense_mat_doubles(Dp) * 8));
    uint8_t* mask = (uint8_t*)(ctx->dense_scratch.p + al256(dense_mat_doubles(Dp) * 8) + al256(16));
    DenseTrajHost h{};
    h.D = D; h.Dp = Dp; h.N = N; h.c0 = model->c0;
    h.mu = (model->kind == AHMC_MODEL_STD_NORMAL) ? nullptr : model->d_p0;
    if (model->kind == AHMC_MODEL_DENSE_GAUSS) {
        h.P = model->d_p1_pad;
        CU(cudaMemcpyAsync(norms + 1, model->d_p1_pad + dense_mat_doubles(Dp), 8, cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
        h.w = (model->kind == AHMC_MODEL_DIAG_GAUSS) ? model->d_p1 : nullptr;
        CU(launch_vec_norm(h.w, D, norms + 1, ctx->stream));
        *nl += 1;
    }
    if (a.metric.kind == AHMC_METRIC_DENSE) {
        CU(launch_pad_norm(a.metric.Minv, D, Dp, Mpad, norms, ctx->stream));
        h.Minv = Mpad;
    } else {
        h.Mdiag = (a.metric.kind == AHMC_METRIC_DIAG) ? a.metric.Minv : nullptr;
        CU(launch_vec_norm(h.Mdiag, D, norms, ctx->stream));
    }
    *nl += 1;
    h.norms = norms;
    h.eps = eps; h.eps_chain = a.eps_chain; h.n_steps = n_abs; h.fwd = a.fwd;
    h.th_in = a.th_in; h.r_in = a.r_in; h.g_in = a.g_in; h.ld_in = a.ld_in;
    h.th_out = a.th_out; h.r_out = a.r_out; h.g_out = a.g_out; h.dr_out = a.dr_out;
    h.lp_out = a.lp_out; h.lk_out = a.lk_out; h.ld_out = a.ld_out;
    h.status = a.status; h.steps_done = a.steps_done; h.need_exact = mask;
    CU(launch_dense_traj(h, ctx->stream, nl));
    LeapfrogArgs b = a;
    b.n_steps = n_abs;
    b.only_mask = mask;
    b.min_break = nullptr;
    CU(launch_leapfrog(b, ctx->stream, nl));
    return AHMC_OK;
}

// D x N column block copy between arrays of leading dimensions ldd / lds (nothing to do in place)
int copy_cols(ahmc_ctx* ctx, double* dst, int64_t ldd, const double* src, int64_t lds, int32_t D, int64_t N,
              cudaMemcpyKind kind = cudaMemcpyDeviceToDevice) {
    if (!dst || !src || dst == src) return AHMC_OK;
    CU(cudaMemcpy2DAsync(dst, (size_t)ldd * 8, src, (size_t)lds * 8, (size_t)D * 8, (size_t)N, kind, ctx->stream));
    return AHMC_OK;
}

int check_rng_alphas(ahmc_ctx* ctx, const ahmc_rng* rng) {
    if (!(rng->partial_refresh_alpha > -1.0 && rng->partial_refresh_alpha < 1.0))
        return fail(ctx, AHMC_ERR_INVALID, "partial_refresh_alpha must be in (-1, 1)");
    if (!(rng->temper_alpha >= 0.0) || std::isinf(rng->temper_alpha))
        return fail(ctx, AHMC_ERR_INVALID, "temper_alpha must be 0 (plain Leapfrog) or a finite alpha > 0 (TemperedLeapfrog)");
    return AHMC_OK;
}

int check_transition_output(ahmc_ctx* ctx, const ahmc_metric* metric, const ahmc_phasepoint* z_out, uint32_t flags) {
    if (metric->kind == AHMC_METRIC_DENSE && !metric->cholU && !(flags & AHMC_FLAG_NO_REFRESH))
        return fail(ctx, AHMC_ERR_INVALID, "Dense metric needs cholU for the momentum refresh (metric.jl:311-320)");
    if (z_out->lk_gradient)
        return fail(ctx, AHMC_ERR_UNSUPPORTED, "transition entry points do not emit lk_gradient; call ahmc_phasepoint_f64 if needed");
    return AHMC_OK;
}

// a transition reads (theta, r, -grad lp, lp) of z_in and writes (theta, r, -grad lp, lp, lk) of z_out; `Args` is any
// argument block with these fields (LeapfrogArgs, NutsArgs, MultinomialArgs)
template <class Args>
void stage_transition_pp(Stager& st, const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out, int64_t N, Args& a) {
    const size_t cin = (size_t)z_in->ld * N, cout = (size_t)z_out->ld * N;
    a.ld_in = z_in->ld;
    a.ld_out = z_out->ld;
    st.in((const double*)z_in->theta, cin, &a.th_in);
    st.in((const double*)z_in->r, cin, &a.r_in);
    st.in((const double*)z_in->lp_gradient, cin, &a.g_in);
    st.in((const double*)z_in->lp_value, (size_t)N, &a.lp_in);
    st.out(z_out->theta, cout, &a.th_out);
    st.out(z_out->r, cout, &a.r_out);
    st.out(z_out->lp_gradient, cout, &a.g_out);
    st.out(z_out->lp_value, (size_t)N, &a.lp_out);
    st.out(z_out->lk_value, (size_t)N, &a.lk_out);
}

void stage_stats(Stager& st, const ahmc_stats* s, int64_t N, StatsDev* d) {
    memset(d, 0, sizeof *d);
    if (!s) return;
    st.out(s->n_steps, (size_t)N, &d->n_steps);
    st.out(s->is_accept, (size_t)N, &d->is_accept);
    st.out(s->acceptance_rate, (size_t)N, &d->acceptance_rate);
    st.out(s->log_density, (size_t)N, &d->log_density);
    st.out(s->hamiltonian_energy, (size_t)N, &d->hamiltonian_energy);
    st.out(s->hamiltonian_energy_error, (size_t)N, &d->hamiltonian_energy_error);
    st.out(s->max_hamiltonian_energy_error, (size_t)N, &d->max_hamiltonian_energy_error);
    st.out(s->tree_depth, (size_t)N, &d->tree_depth);
    st.out(s->numerical_error, (size_t)N, &d->numerical_error);
}

void stage_rng(Stager& st, const ahmc_rng* r, int32_t D, int64_t N, bool nuts, RngDev* d) {
    d->seed = r->seed;
    d->offset = r->offset;
    d->partial_alpha = r->partial_refresh_alpha;
    d->temper_alpha = r->temper_alpha > 0.0 ? r->temper_alpha : 0.0;
    d->exp_stride = nuts ? r->exp_stride : 1;
    d->dir_stride = r->dir_stride;
    st.in(r->normal_tape, (size_t)D * N, &d->normal_tape);
    st.in(r->exp_tape, (size_t)(nuts ? r->exp_stride : 1) * N, &d->exp_tape);
    st.in(nuts ? r->dir_tape : (const uint8_t*)nullptr, (size_t)r->dir_stride * N, &d->dir_tape);
}

// adaptor-statistics workspace: [last-block counter (as 2 doubles)] [per-block partials].  Zeroed whenever it is
// (re)allocated; after that the kernel re-arms the counter at the end of every launch.
int adapt_workspace(ahmc_ctx* ctx, int32_t D, int64_t N, int* blocks) {
    *blocks = (int)(N < 148 ? N : 148);
    const size_t need = ((size_t)*blocks * (D + 1) + 2) * sizeof(double);
    if (need <= ctx->adapt_scratch.bytes) return AHMC_OK;
    int rc = grow(ctx, ctx->adapt_scratch, need, "adaptor workspace");
    if (rc) return rc;
    CU(cudaMemsetAsync(ctx->adapt_scratch.p, 0, need, ctx->stream));
    return AHMC_OK;
}
}  // namespace

// =================================================================================================
extern "C" {

const char* ahmc_version(void) { return "ahmc_b200 0.1.0 (sm_100a)"; }

int ahmc_create(ahmc_ctx** out, int32_t device, void* cuda_stream) {
    if (!out) return AHMC_ERR_INVALID;
    *out = nullptr;
    ahmc_ctx* ctx = new (std::nothrow) ahmc_ctx();
    if (!ctx) return AHMC_ERR_NOMEM;
    ctx->device = device;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || device < 0 || device >= ndev) {
        // no silent CPU fallback: the product path needs the GPU
        fprintf(stderr, "ahmc_create: no usable CUDA device %d (%s)\n", device, e != cudaSuccess ? cudaGetErrorString(e) : "out of range");
        delete ctx;
        return AHMC_ERR_CUDA;
    }
    DeviceGuard g(device);
    if (cuda_stream) {
        ctx->stream = (cudaStream_t)cuda_stream;
    } else {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete ctx;
            return AHMC_ERR_CUDA;
        }
        ctx->own_stream = true;
    }
    if (cudaMalloc((void**)&ctx->d_min_break, sizeof(int)) != cudaSuccess) {
        if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
        delete ctx;
        return AHMC_ERR_NOMEM;
    }
    *out = ctx;
    return AHMC_OK;
}

int ahmc_destroy(ahmc_ctx* ctx) {
    if (!ctx) return AHMC_OK;
    DeviceGuard g(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->d_min_break);
    for (DevBuf* b : {&ctx->arena, &ctx->nuts_scratch, &ctx->adapt_scratch, &ctx->mn_scratch, &ctx->dense_scratch,
                      &ctx->coop_scratch, &ctx->split_scratch})
        cudaFree(b->p);
    for (int i = 0; i < ahmc_ctx::kPipeStreams; ++i) {
        if (ctx->pipe[i]) cudaStreamDestroy(ctx->pipe[i]);
        if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]);
    }
    for (int i = 0; i < ahmc_ctx::kMaxPipeChunks; ++i) {
        for (int j = 0; j < 3; ++j)
            if (ctx->ev_in[i][j]) cudaEventDestroy(ctx->ev_in[i][j]);
        if (ctx->ev_k[i]) cudaEventDestroy(ctx->ev_k[i]);
    }
    if (ctx->ev_a) cudaEventDestroy(ctx->ev_a);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return AHMC_OK;
}

const char* ahmc_last_error(const ahmc_ctx* ctx) { return ctx ? ctx->err.c_str() : "ahmc: NULL context"; }

int ahmc_synchronize(ahmc_ctx* ctx) {
    if (!ctx) return AHMC_ERR_INVALID;
    DeviceGuard g(ctx->device);
    CU(cudaStreamSynchronize(ctx->stream));
    return AHMC_OK;
}

void* ahmc_stream(const ahmc_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
int64_t ahmc_launch_count(const ahmc_ctx* ctx) { return ctx ? ctx->launches : 0; }
const char* ahmc_last_transport(const ahmc_ctx* ctx) { return ctx ? ctx->transport.c_str() : "none"; }

// ---------------------------------------------------------------------------------------------- models
int ahmc_model_create(ahmc_ctx* ctx, int32_t kind, int32_t D, const double* p0, const double* p1, double c0,
                      ahmc_model** out) {
    if (!ctx || !out) return AHMC_ERR_INVALID;
    *out = nullptr;
    if (D < 1) return fail(ctx, AHMC_ERR_INVALID, "model dimension must be >= 1");
    if (kind < AHMC_MODEL_STD_NORMAL || kind > AHMC_MODEL_FUNNEL)
        return fail(ctx, AHMC_ERR_INVALID, "unknown built-in model kind %d", kind);
    if ((kind == AHMC_MODEL_DIAG_GAUSS || kind == AHMC_MODEL_DENSE_GAUSS) && (!p0 || !p1))
        return fail(ctx, AHMC_ERR_INVALID, "model kind %d needs p0 and p1", kind);
    DeviceGuard g(ctx->device);
    ahmc_model* m = new (std::nothrow) ahmc_model();
    if (!m) return AHMC_ERR_NOMEM;
    m->kind = kind;
    m->D = D;
    m->c0 = c0;
    if (kind == AHMC_MODEL_DIAG_GAUSS) {
        std::vector<double> w((size_t)D);
        for (int d = 0; d < D; ++d) w[d] = 1.0 / (p1[d] * p1[d]);  // 1/s^2
        if (cudaMalloc((void**)&m->d_p0, sizeof(double) * D) != cudaSuccess ||
            cudaMalloc((void**)&m->d_p1, sizeof(double) * D) != cudaSuccess) {
            ahmc_model_destroy(ctx, m);
            return fail(ctx, AHMC_ERR_NOMEM, "cudaMalloc for model parameters failed");
        }
        cudaMemcpy(m->d_p0, p0, sizeof(double) * D, cudaMemcpyHostToDevice);
        cudaMemcpy(m->d_p1, w.data(), sizeof(double) * D, cudaMemcpyHostToDevice);
    } else if (kind == AHMC_MODEL_DENSE_GAUSS) {
        if (cudaMalloc((void**)&m->d_p0, sizeof(double) * D) != cudaSuccess ||
            cudaMalloc((void**)&m->d_p1, sizeof(double) * (size_t)D * D) != cudaSuccess) {
            ahmc_model_destroy(ctx, m);
            return fail(ctx, AHMC_ERR_NOMEM, "cudaMalloc for model parameters failed");
        }
        cudaMemcpy(m->d_p0, p0, sizeof(double) * D, cudaMemcpyHostToDevice);
        cudaMemcpy(m->d_p1, p1, sizeof(double) * (size_t)D * D, cudaMemcpyHostToDevice);
        int RB, CB;
        if (dense_tile_shape(D, &m->Dp, &RB, &CB)) {  // padded copy + infinity norm for the tiled DMMA kernel
            if (cudaMalloc((void**)&m->d_p1_pad, sizeof(double) * (dense_mat_doubles(m->Dp) + 2)) != cudaSuccess) {
                ahmc_model_destroy(ctx, m);
                return fail(ctx, AHMC_ERR_NOMEM, "cudaMalloc for the padded precision failed");
            }
            launch_pad_norm(m->d_p1, D, m->Dp, m->d_p1_pad, m->d_p1_pad + dense_mat_doubles(m->Dp), ctx->stream);
            cudaStreamSynchronize(ctx->stream);
        }
        if (D > 16 && D <= 512) {  // the layouts the cooperative NUTS form runs on (one chain per warp)
            if (cudaMalloc((void**)&m->d_p1_coop, sizeof(double) * coop_padded_doubles(D)) != cudaSuccess) {
                ahmc_model_destroy(ctx, m);
                return fail(ctx, AHMC_ERR_NOMEM, "cudaMalloc for the column-padded precision failed");
            }
            launch_pad_columns(m->d_p1, D, m->d_p1_coop, ctx->stream);
            cudaStreamSynchronize(ctx->stream);
        }
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        ahmc_model_destroy(ctx, m);
        return fail(ctx, AHMC_ERR_CUDA, "copying model parameters failed: %s", cudaGetErrorString(e));
    }
    *out = m;
    return AHMC_OK;
}

int ahmc_model_create_callback(ahmc_ctx* ctx, int32_t D, ahmc_logp_grad_fn fn, void* user, ahmc_model** out) {
    if (!ctx || !out) return AHMC_ERR_INVALID;
    *out = nullptr;
    if (D < 1 || !fn) return fail(ctx, AHMC_ERR_INVALID, "callback model needs D >= 1 and a function");
    ahmc_model* m = new (std::nothrow) ahmc_model();
    if (!m) return AHMC_ERR_NOMEM;
    m->kind = AHMC_MODEL_CALLBACK;
    m->D = D;
    m->fn = fn;
    m->user = user;
    *out = m;
    return AHMC_OK;
}

int ahmc_model_create_user(ahmc_ctx* ctx, int32_t D, const char* cuda_src, const double* params, int32_t n_params, double c0,
                           ahmc_model** out) {
    if (!ctx || !cuda_src || !out) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/source/out");
    if (D < 1 || n_params < 0 || (n_params > 0 && !params)) return fail(ctx, AHMC_ERR_INVALID, "need D >= 1 and params for n_params > 0");
    if (!strstr(cuda_src, "ahmc_user_logp_grad") && !strstr(cuda_src, "ahmc_user_coord"))
        return fail(ctx, AHMC_ERR_INVALID, "the source must define ahmc_user_logp_grad(theta, grad, D, params) or, with "
                                           "#define AHMC_USER_COORDWISE, ahmc_user_coord(d, theta_d, params, grad_d)");
    DeviceGuard g(ctx->device);
    char why[256];
    UserModule* um = user_module_create(cuda_src, why, sizeof why);
    if (!um) return fail(ctx, AHMC_ERR_UNSUPPORTED, "run-time compilation is unavailable: %s", why);
    ahmc_model* m = new (std::nothrow) ahmc_model;
    if (!m) {
        user_module_destroy(um);
        return fail(ctx, AHMC_ERR_NOMEM, "out of host memory");
    }
    m->kind = AHMC_MODEL_USER;
    m->D = D;
    m->c0 = c0;
    m->rtc = um;
    if (n_params > 0) {
        if (cudaMalloc((void**)&m->d_p0, (size_t)n_params * 8) != cudaSuccess) {
            user_module_destroy(um);
            delete m;
            return fail(ctx, AHMC_ERR_NOMEM, "cudaMalloc for the user parameters failed");
        }
        CU(cudaMemcpy(m->d_p0, params, (size_t)n_params * 8, cudaMemcpyHostToDevice));
    }
    *out = m;
    return AHMC_OK;
}

int ahmc_user_source_check(const char* cuda_src, int32_t kernel, int32_t metric_kind, int32_t D, char* log, int64_t log_len) {
    if (!cuda_src || kernel < 0 || kernel > 4 || metric_kind < 0 || metric_kind > 2 || D < 1) return AHMC_ERR_INVALID;
    int rc = user_source_check(cuda_src, kernel, metric_kind, D, log, log_len > 0 ? (size_t)log_len : 0);
    return rc == 0 ? AHMC_OK : (rc == -3 ? AHMC_ERR_UNSUPPORTED : AHMC_ERR_INVALID);
}

int ahmc_model_destroy(ahmc_ctx* ctx, ahmc_model* m) {
    if (!m) return AHMC_OK;
    if (ctx) {
        DeviceGuard g(ctx->device);
        cudaFree(m->d_p0);
        cudaFree(m->d_p1);
        cudaFree(m->d_p1_pad);
        cudaFree(m->d_p1_coop);
        if (m->rtc) {
            cudaStreamSynchronize(ctx->stream);
            user_module_destroy(m->rtc);
        }
    }
    delete m;
    return AHMC_OK;
}

// ---------------------------------------------------------------------------------------------- phasepoint
int ahmc_phasepoint_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                        const ahmc_phasepoint* z, uint32_t flags) {
    if (!ctx || !model || !metric) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/model/metric");
    int rc = check_common(ctx, model, metric, D, N, true);
    if (rc) return rc;
    if ((rc = check_pp(ctx, z, D, "z", true, N))) return rc;
    if (N == 0) return AHMC_OK;
    DeviceGuard g(ctx->device);
    Stager st(ctx, flags & AHMC_FLAG_HOST_BUFFERS);
    PhasepointArgs a{};
    a.model = model_dev(model);
    stage_metric(st, metric, D, N, &a.metric);
    a.D = D;
    a.N = N;
    a.ld = z->ld;
    st.in((const double*)z->theta, (size_t)z->ld * N, &a.th);
    st.in((const double*)z->r, (size_t)z->ld * N, &a.r);
    st.out(z->lp_value, (size_t)N, &a.lp);
    st.out(z->lp_gradient, (size_t)z->ld * N, &a.g);
    st.out(z->lk_value, (size_t)N, &a.lk);
    st.out(z->lk_gradient, (size_t)z->ld * N, &a.dr);
    if ((rc = st.commit())) return rc;
    int nl = 0;
    if (model->kind == AHMC_MODEL_CALLBACK) {  // user closure, then the metric half of phasepoint
        SplitWork w;
        if ((rc = split_workspace(ctx, D, N, z->ld, &w))) return rc;
        if ((rc = call_user(ctx, model, a.th, w.cb_lp, w.cb_grad, D, N, z->ld))) return rc;
        SplitArgs sa{};
        sa.metric = a.metric; sa.D = D; sa.N = N; sa.fwd = 1; sa.mul = 1.0; sa.no_kick = 1;
        sa.r = const_cast<double*>(a.r); sa.g = a.g; sa.lp = a.lp; sa.lk = a.lk; sa.dr = a.dr;
        sa.cb_lp = w.cb_lp; sa.cb_grad = w.cb_grad; sa.ld = z->ld;
        CU(launch_kick_energy(sa, ctx->stream, &nl));
    } else {
        CU(launch_phasepoint(a, ctx->stream, &nl));
    }
    ctx->launches += nl;
    return finish_call(ctx, st, flags);
}

// ---------------------------------------------------------------------------------------------- leapfrog
static int copy_pp_device(ahmc_ctx* ctx, int32_t D, int64_t N, const ahmc_phasepoint* a, const ahmc_phasepoint* b,
                          cudaMemcpyKind kind) {
    int rc;
    if ((rc = copy_cols(ctx, b->theta, b->ld, a->theta, a->ld, D, N, kind))) return rc;
    if ((rc = copy_cols(ctx, b->r, b->ld, a->r, a->ld, D, N, kind))) return rc;
    if ((rc = copy_cols(ctx, b->lp_gradient, b->ld, a->lp_gradient, a->ld, D, N, kind))) return rc;
    if ((rc = copy_cols(ctx, b->lk_gradient, b->ld, a->lk_gradient, a->ld, D, N, kind))) return rc;
    if ((rc = copy_cols(ctx, b->lp_value, 1, a->lp_value, 1, 1, N, kind))) return rc;
    return copy_cols(ctx, b->lk_value, 1, a->lk_value, 1, 1, N, kind);
}

// device alias of a page-locked, device-mapped host pointer (cudaHostAlloc / cudaHostRegister memory under unified
// addressing), or nullptr for pageable memory
static void* pinned_alias(const void* p) {
    if (!p) return nullptr;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
    return at.devicePointer;
}

static int pipe_resources(ahmc_ctx* ctx) {
    if (ctx->pipe[0]) return AHMC_OK;
    for (int i = 0; i < ahmc_ctx::kPipeStreams; ++i) CU(cudaStreamCreateWithFlags(&ctx->pipe[i], cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&ctx->ev_a, cudaEventDisableTiming));
    for (int i = 0; i < ahmc_ctx::kPipeStreams; ++i) CU(cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming));
    for (int i = 0; i < ahmc_ctx::kMaxPipeChunks; ++i) {
        for (int j = 0; j < 3; ++j) CU(cudaEventCreateWithFlags(&ctx->ev_in[i][j], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->ev_k[i], cudaEventDisableTiming));
    }
    return AHMC_OK;
}

// HOST_BUFFERS fast lane.  The chain axis is cut into chunks (chains are independent, so a chunk is a complete
// sub-problem) that flow upload -> kernel -> download through separate streams linked chunk by chunk with events, so
// the upload of chunk i+1 overlaps the kernel and the download of chunk i (PCIe is full duplex): the call costs about
// max(H2D, D2H) + one chunk instead of their sum.  Same kernels, bit-identical results to the one-shot path.
//   upload   : copy engines, theta / r / gradient on one stream or on one stream each (their fixed per-copy latencies
//              overlap), or -- page-locked buffers only -- none at all: the kernel loads from host memory directly;
//   download : copy engines on a third stream, or -- page-locked buffers only -- none: the kernel's stores go straight
//              to host memory as posted PCIe writes.
// Pageable buffers always take the copy-engine form.  Knobs for A/B measurements: AHMC_PIPE_CHUNKS (chunk count),
// AHMC_PIPE_UP = ce1 | ce3 | direct, AHMC_PIPE_DOWN = ce | direct, AHMC_PIPE_TRACE=1 (event timeline on stderr).
static int leapfrog_host_pipelined(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D,
                                   int64_t N, double eps, const double* eps_chain, int32_t n_steps,
                                   double temper_alpha, const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out,
                                   uint32_t* status, int32_t* steps_done, uint32_t flags) {
    const auto t_enter = std::chrono::steady_clock::now();
    auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_enter).count(); };
    int rc = pipe_resources(ctx);
    if (rc) return rc;
    const char* ev;
    const bool per_chain_minv = metric->kind == AHMC_METRIC_DIAG && metric->chain_stride != 0;

    // which buffers can the device address directly?
    bool in_pinned = true, out_pinned = true;
    auto alias = [](const void* p, bool& all) -> void* {
        if (!p) return nullptr;
        void* d = pinned_alias(p);
        if (!d) all = false;
        return d;
    };
    const double* a_th = (const double*)alias(z_in->theta, in_pinned);
    const double* a_r = (const double*)alias(z_in->r, in_pinned);
    const double* a_g = (const double*)alias(z_in->lp_gradient, in_pinned);
    const double* a_eps = (const double*)alias(eps_chain, in_pinned);
    const double* a_minv = per_chain_minv ? (const double*)alias(metric->Minv, in_pinned) : nullptr;
    double* b_th = (double*)alias(z_out->theta, out_pinned);
    double* b_r = (double*)alias(z_out->r, out_pinned);
    double* b_g = (double*)alias(z_out->lp_gradient, out_pinned);
    double* b_dr = (double*)alias(z_out->lk_gradient, out_pinned);
    double* b_lp = (double*)alias(z_out->lp_value, out_pinned);
    double* b_lk = (double*)alias(z_out->lk_value, out_pinned);
    uint32_t* b_st = (uint32_t*)alias(status, out_pinned);
    int32_t* b_sd = (int32_t*)alias(steps_done, out_pinned);

    const double t_attr = since();
    enum { UP_CE1, UP_CE3, UP_DIRECT };
    const bool has_g = z_in->lp_gradient != nullptr;
    int up = in_pinned ? UP_DIRECT : UP_CE1;
    bool down_direct = out_pinned;
    int occ_cap = AHMC_PIPE_DIRECT_OCC;
    int nchunk = 0;
    // ---- transport choice.  Page-locked buffers can be moved in several ways whose ranking depends on the HOST (the
    // zero-copy lane measured 0.36 ms on one box and 3.8 ms on another: SM-issued reads of system memory are at the mercy
    // of the platform's read-completion latency, copy engines are not), so the first calls of a given shape try each
    // candidate in turn -- results are bit-identical in every mode, nothing extra is executed -- and the fastest is kept
    // for the life of the context.  Candidates: {direct loads + direct stores, 1 CTA/SM}, {copy engines, 2 / 4 chunks},
    // {copy-engine upload, direct stores, 4 chunks}.  The AHMC_PIPE_* variables pin the choice (A/B runs).
    struct Cand { int up; bool down_direct; int chunks; int occ; };
    static const Cand kCands[] = {{UP_DIRECT, true, 1, 1}, {UP_CE1, false, 2, 0}, {UP_CE1, false, 4, 0}, {UP_CE1, true, 4, 1}};
    constexpr int kNCand = 4, kRounds = 3;  // round 0 warms every candidate up (arena growth, first-touch), rounds 1.. are timed
    const bool pinned_env = getenv("AHMC_PIPE_UP") || getenv("AHMC_PIPE_DOWN") || getenv("AHMC_PIPE_CHUNKS") || getenv("AHMC_PIPE_OCC");
    const bool tunable = in_pinned && out_pinned && !pinned_env && N >= 1024 && !((ev = getenv("AHMC_PIPE_AUTOTUNE")) && atoi(ev) == 0);
    ahmc_ctx::PipeTune* tune = nullptr;
    int trial = -1;
    if (tunable) {
        const int key = (has_g ? 1 : 0) | (z_out->lk_gradient ? 2 : 0) | (eps_chain ? 4 : 0) | (per_chain_minv ? 8 : 0);
        for (auto& t : ctx->tune)
            if (t.N == N && t.D == D && t.key == key) tune = &t;
        if (!tune) {
            ahmc_ctx::PipeTune t{};
            t.N = N; t.D = D; t.key = key; t.calls = 0; t.chosen = -1;
            for (double& b : t.best_ms) b = 1e30;
            ctx->tune.push_back(t);
            tune = &ctx->tune.back();
        }
        int c = tune->chosen;
        if (c < 0) {
            trial = tune->calls % kNCand;
            c = trial;
        }
        up = kCands[c].up; down_direct = kCands[c].down_direct; nchunk = kCands[c].chunks; occ_cap = kCands[c].occ;
    }
    if ((ev = getenv("AHMC_PIPE_UP"))) up = !strcmp(ev, "direct") ? UP_DIRECT : !strcmp(ev, "ce3") ? UP_CE3 : UP_CE1;
    if ((ev = getenv("AHMC_PIPE_DOWN"))) down_direct = !strcmp(ev, "direct");
    if (!in_pinned && up == UP_DIRECT) up = UP_CE3;
    if (!out_pinned) down_direct = false;
    const bool trace = (ev = getenv("AHMC_PIPE_TRACE")) && atoi(ev) != 0;
    if ((ev = getenv("AHMC_PIPE_OCC"))) occ_cap = atoi(ev);
    if ((ev = getenv("AHMC_PIPE_CHUNKS"))) nchunk = atoi(ev);
    if (nchunk <= 0) {
        if (up == UP_DIRECT) {
            nchunk = AHMC_PIPE_DIRECT_CHUNKS;
        } else {
            nchunk = N >= 1024 ? AHMC_PIPE_CE_CHUNKS : 1;
        }
        if (nchunk < 1) nchunk = 1;
    }
    if (nchunk > ahmc_ctx::kMaxPipeChunks) nchunk = ahmc_ctx::kMaxPipeChunks;
    int64_t chunk = (N + nchunk - 1) / nchunk;
    chunk = (chunk + 3) & ~(int64_t)3;

    // device staging for whatever is not addressed directly
    const int64_t ldi = z_in->ld, ldo = z_out->ld;
    const size_t nMinv = metric_minv_count(metric, D, N);
    const bool stage_in = up != UP_DIRECT, stage_out = !down_direct;
    const bool hasU = metric->kind == AHMC_METRIC_DENSE && metric->cholU;
    size_t need = (per_chain_minv && !stage_in ? 0 : al256(nMinv * 8)) + (hasU ? al256((size_t)D * D * 8) : 0);
    if (stage_in) need += al256((size_t)N * 8) + (has_g ? 3 : 2) * al256((size_t)ldi * N * 8);
    if (stage_out) need += 4 * al256((size_t)ldo * N * 8) + 2 * al256((size_t)N * 8) + 2 * al256((size_t)N * 4);
    if ((rc = grow(ctx, ctx->arena, need, "staging arena", need + need / 4))) return rc;
    size_t off = 0;
    auto carve = [&](bool want, size_t bytes) -> char* {
        if (!want || !bytes) return nullptr;
        char* p = ctx->arena.p + off;
        off += al256(bytes);
        return p;
    };
    double* dMinv = (double*)carve(!(per_chain_minv && !stage_in), nMinv * 8);
    double* dU = (double*)carve(hasU, (size_t)D * D * 8);
    double* dEps = (double*)carve(stage_in, (size_t)N * 8);
    double* dTh = (double*)carve(stage_in, (size_t)ldi * N * 8);
    double* dR = (double*)carve(stage_in, (size_t)ldi * N * 8);
    double* dG = (double*)carve(stage_in && has_g, (size_t)ldi * N * 8);
    double* oTh = (double*)carve(stage_out, (size_t)ldo * N * 8);
    double* oR = (double*)carve(stage_out, (size_t)ldo * N * 8);
    double* oG = (double*)carve(stage_out, (size_t)ldo * N * 8);
    double* oDr = (double*)carve(stage_out, (size_t)ldo * N * 8);
    double* oLp = (double*)carve(stage_out, (size_t)N * 8);
    double* oLk = (double*)carve(stage_out, (size_t)N * 8);
    uint32_t* oSt = (uint32_t*)carve(stage_out, (size_t)N * 4);
    int32_t* oSd = (int32_t*)carve(stage_out, (size_t)N * 4);

    cudaStream_t s_cmp = ctx->stream;
    cudaStream_t s_up[3] = {ctx->pipe[0], up == UP_CE3 ? ctx->pipe[1] : ctx->pipe[0], up == UP_CE3 ? ctx->pipe[2] : ctx->pipe[0]};
    cudaStream_t s_down = ctx->pipe[3];
    const int n_up = up == UP_CE3 ? 3 : 1;

    // everything is ordered after earlier work on the context stream; shared parameters (re-read by every chain, so
    // always staged) go first on the compute stream itself
    CU(cudaEventRecord(ctx->ev_a, s_cmp));
    if (stage_in)
        for (int j = 0; j < n_up; ++j) CU(cudaStreamWaitEvent(s_up[j], ctx->ev_a, 0));
    if (nMinv && !per_chain_minv) CU(cudaMemcpyAsync(dMinv, metric->Minv, nMinv * 8, cudaMemcpyHostToDevice, s_cmp));
    if (hasU) CU(cudaMemcpyAsync(dU, metric->cholU, (size_t)D * D * 8, cudaMemcpyHostToDevice, s_cmp));
    if (!stage_in) {  // the second compute stream starts after the shared parameters have landed
        CU(cudaEventRecord(ctx->ev_join[0], s_cmp));
        CU(cudaStreamWaitEvent(ctx->pipe[4], ctx->ev_join[0], 0));
    }

    std::vector<cudaEvent_t> tr;  // optional timeline (timing events are created only when tracing)
    auto mark = [&](cudaStream_t st) {
        if (!trace) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        tr.push_back(e);
    };
    mark(s_cmp);

    const int n_abs = n_steps < 0 ? -n_steps : n_steps;
    int nl = 0, k = 0;
    for (int64_t c0 = 0; c0 < N; c0 += chunk, ++k) {
        const int64_t n = (c0 + chunk <= N) ? chunk : N - c0;
        if (stage_in) {
            CU(cudaMemcpyAsync(dTh + ldi * c0, z_in->theta + ldi * c0, (size_t)ldi * n * 8, cudaMemcpyHostToDevice, s_up[0]));
            if (eps_chain) CU(cudaMemcpyAsync(dEps + c0, eps_chain + c0, (size_t)n * 8, cudaMemcpyHostToDevice, s_up[0]));
            CU(cudaMemcpyAsync(dR + ldi * c0, z_in->r + ldi * c0, (size_t)ldi * n * 8, cudaMemcpyHostToDevice, s_up[1]));
            if (per_chain_minv)
                CU(cudaMemcpyAsync(dMinv + metric->chain_stride * c0, metric->Minv + metric->chain_stride * c0,
                                   (size_t)metric->chain_stride * n * 8, cudaMemcpyHostToDevice, s_up[1]));
            if (has_g) CU(cudaMemcpyAsync(dG + ldi * c0, z_in->lp_gradient + ldi * c0, (size_t)ldi * n * 8, cudaMemcpyHostToDevice, s_up[2]));
            for (int j = 0; j < n_up; ++j) {
                CU(cudaEventRecord(ctx->ev_in[k][j], s_up[j]));
                CU(cudaStreamWaitEvent(s_cmp, ctx->ev_in[k][j], 0));
            }
            mark(s_up[n_up - 1]);
        }
        LeapfrogArgs a{};
        a.model = model_dev(model);
        const double* minv_k = !nMinv ? nullptr
                               : !per_chain_minv ? dMinv
                               : stage_in ? dMinv + metric->chain_stride * c0 : a_minv + metric->chain_stride * c0;
        a.metric = MetricDev{metric->kind, minv_k, per_chain_minv ? metric->chain_stride : 0, hasU ? dU : nullptr};
        a.D = D;
        a.N = n;
        a.eps = eps;
        a.eps_chain = !eps_chain ? nullptr : stage_in ? dEps + c0 : a_eps + c0;
        a.n_steps = n_abs;
        a.fwd = n_steps > 0;
        a.temper_alpha = temper_alpha;
        a.th_in = (stage_in ? dTh : a_th) + ldi * c0;
        a.r_in = (stage_in ? dR : a_r) + ldi * c0;
        a.g_in = !has_g ? nullptr : (stage_in ? dG : a_g) + ldi * c0;
        a.ld_in = ldi;
        a.th_out = (stage_out ? oTh : b_th) + ldo * c0;
        a.r_out = (stage_out ? oR : b_r) + ldo * c0;
        a.g_out = (stage_out ? oG : b_g) + ldo * c0;
        a.dr_out = !z_out->lk_gradient ? nullptr : (stage_out ? oDr : b_dr) + ldo * c0;
        a.lp_out = (stage_out ? oLp : b_lp) + c0;
        a.lk_out = (stage_out ? oLk : b_lk) + c0;
        a.ld_out = ldo;
        a.status = !status ? nullptr : (stage_out ? oSt : b_st) + c0;
        a.steps_done = !steps_done ? nullptr : (stage_out ? oSd : b_sd) + c0;
        a.flags = flags;
        a.resident_blocks_per_sm = (!stage_in || !stage_out) ? occ_cap : 0;
        // with direct loads the kernels of different chunks may run side by side: alternate two streams
        cudaStream_t s_k = (!stage_in && (k & 1)) ? ctx->pipe[4] : s_cmp;
        CU(launch_leapfrog(a, s_k, &nl));
        mark(s_k);
        if (stage_out) {
            CU(cudaEventRecord(ctx->ev_k[k], s_k));
            CU(cudaStreamWaitEvent(s_down, ctx->ev_k[k], 0));
            CU(cudaMemcpyAsync(z_out->theta + ldo * c0, a.th_out, (size_t)ldo * n * 8, cudaMemcpyDeviceToHost, s_down));
            CU(cudaMemcpyAsync(z_out->r + ldo * c0, a.r_out, (size_t)ldo * n * 8, cudaMemcpyDeviceToHost, s_down));
            CU(cudaMemcpyAsync(z_out->lp_gradient + ldo * c0, a.g_out, (size_t)ldo * n * 8, cudaMemcpyDeviceToHost, s_down));
            if (a.dr_out) CU(cudaMemcpyAsync(z_out->lk_gradient + ldo * c0, a.dr_out, (size_t)ldo * n * 8, cudaMemcpyDeviceToHost, s_down));
            mark(s_down);
        }
    }
    ctx->launches += nl;
    if (stage_out) {
        // the per-chain scalars of all chunks go back in one copy each (stream order puts them after the last kernel)
        CU(cudaMemcpyAsync(z_out->lp_value, oLp, (size_t)N * 8, cudaMemcpyDeviceToHost, s_down));
        CU(cudaMemcpyAsync(z_out->lk_value, oLk, (size_t)N * 8, cudaMemcpyDeviceToHost, s_down));
        if (status) CU(cudaMemcpyAsync(status, oSt, (size_t)N * 4, cudaMemcpyDeviceToHost, s_down));
        if (steps_done) CU(cudaMemcpyAsync(steps_done, oSd, (size_t)N * 4, cudaMemcpyDeviceToHost, s_down));
        mark(s_down);
        CU(cudaEventRecord(ctx->ev_join[3], s_down));
        CU(cudaStreamWaitEvent(s_cmp, ctx->ev_join[3], 0));
    }
    if (!stage_in && k > 1) {
        CU(cudaEventRecord(ctx->ev_join[4], ctx->pipe[4]));
        CU(cudaStreamWaitEvent(s_cmp, ctx->ev_join[4], 0));
    }
    // host buffers are valid once everything joined into the context stream has retired
    const double t_issued = since();
    CU(cudaStreamSynchronize(s_cmp));
    {
        char buf[96];
        snprintf(buf, sizeof buf, "up=%s down=%s chunks=%d%s%s", up == UP_DIRECT ? "direct" : up == UP_CE3 ? "ce3" : "ce1",
                 down_direct ? "direct" : "ce", k, (!stage_in || !stage_out) && occ_cap > 0 ? " occ=1" : "",
                 tune ? (tune->chosen >= 0 ? " (autotuned)" : " (autotune trial)") : "");
        ctx->transport = buf;
    }
    if (tune && trial >= 0) {
        const double ms = since();
        if (tune->calls >= kNCand && ms < tune->best_ms[trial]) tune->best_ms[trial] = ms;
        if (++tune->calls >= kNCand * kRounds) {
            int best = 0;
            for (int c = 1; c < kNCand; ++c)
                if (tune->best_ms[c] < tune->best_ms[best]) best = c;
            tune->chosen = best;
            if (trace)
                fprintf(stderr, "[ahmc pipe] autotune N=%lld D=%d: %.3f %.3f %.3f %.3f ms -> candidate %d\n", (long long)N, D,
                        tune->best_ms[0], tune->best_ms[1], tune->best_ms[2], tune->best_ms[3], best);
        }
    }
    if (trace)
        fprintf(stderr, "[ahmc pipe] host ms: pointer queries %.3f, everything issued %.3f, synchronised %.3f\n", t_attr,
                t_issued, since());
    if (trace && !tr.empty()) {
        fprintf(stderr, "[ahmc pipe] up=%s down=%s chunks=%d x %lld chains; ms after the first mark, per chunk [upload] kernel [download]:\n ",
                up == UP_DIRECT ? "direct" : up == UP_CE3 ? "ce3" : "ce1", down_direct ? "direct" : "ce", k, (long long)chunk);
        const int per = 1 + (stage_in ? 1 : 0) + (stage_out ? 1 : 0);
        for (size_t i = 1; i < tr.size(); ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, tr[0], tr[i]);
            fprintf(stderr, "%s%.3f", (i - 1) % per == 0 ? " | " : " ", ms);
        }
        fprintf(stderr, "\n");
        for (cudaEvent_t e : tr) cudaEventDestroy(e);
    }
    return AHMC_OK;
}

int ahmc_leapfrog_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                      double eps, const double* eps_chain, int32_t n_steps, double temper_alpha,
                      const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out, uint32_t* status,
                      int32_t* steps_done, uint32_t flags) {
    if (!ctx || !model || !metric) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/model/metric");
    int rc = check_common(ctx, model, metric, D, N, true);
    if (!rc && D > 512 && temper_alpha > 0.0) rc = fail(ctx, AHMC_ERR_UNSUPPORTED, "TemperedLeapfrog at D > 512 is not built");
    if (rc) return rc;
    // z_in: only theta and r are required.  The cached energies are not read, and a NULL z_in->lp_gradient means "not
    // cached": built-in targets recompute dH/dtheta at the start point on the device (bit-identical to the value
    // phasepoint / a previous step produced), which saves a third of the upload of a host-buffer call.
    if ((rc = check_pp(ctx, z_in, D, "z_in", false, N))) return rc;
    if ((rc = check_pp(ctx, z_out, D, "z_out", true, N))) return rc;
    if (N == 0) return AHMC_OK;
    if (!z_in->lp_gradient && model->kind == AHMC_MODEL_CALLBACK)
        return fail(ctx, AHMC_ERR_INVALID, "z_in.lp_gradient is NULL: a callback target needs the cached gradient (call ahmc_phasepoint_f64 first)");
    DeviceGuard g(ctx->device);
    const bool host = flags & AHMC_FLAG_HOST_BUFFERS;
    const int n_abs = n_steps < 0 ? -n_steps : n_steps;
    if (n_abs == 0 && !z_in->lp_gradient)
        return fail(ctx, AHMC_ERR_INVALID, "n_steps == 0 returns z unchanged and needs z_in.lp_gradient");
    if (n_abs == 0) {  // the loop body never runs: z is returned unchanged (integrator.jl:233)
        rc = copy_pp_device(ctx, D, N, z_in, z_out, host ? cudaMemcpyHostToHost : cudaMemcpyDeviceToDevice);
        if (rc) return rc;
        CU(cudaStreamSynchronize(ctx->stream));
        if (host) {
            if (status) memset(status, 0, sizeof(uint32_t) * (size_t)N);
            if (steps_done) memset(steps_done, 0, sizeof(int32_t) * (size_t)N);
        } else {
            if (status) CU(cudaMemsetAsync(status, 0, sizeof(uint32_t) * (size_t)N, ctx->stream));
            if (steps_done) CU(cudaMemsetAsync(steps_done, 0, sizeof(int32_t) * (size_t)N, ctx->stream));
            if (!(flags & AHMC_FLAG_ASYNC)) CU(cudaStreamSynchronize(ctx->stream));
        }
        return AHMC_OK;
    }
    // dense targets / metrics go through the staged lane below, which can pick the tiled kernel
    const bool host_fast = host && !(flags & AHMC_FLAG_COMPAT_BREAK_ALL) && model->kind != AHMC_MODEL_CALLBACK &&
                           model->kind != AHMC_MODEL_DENSE_GAUSS && metric->kind != AHMC_METRIC_DENSE;
    if (host_fast && N >= 256)
        return leapfrog_host_pipelined(ctx, model, metric, D, N, eps, eps_chain, n_steps, temper_alpha, z_in, z_out,
                                       status, steps_done, flags);
    Stager st(ctx, host);
    const size_t cin = (size_t)z_in->ld * N, cout = (size_t)z_out->ld * N;
    LeapfrogArgs a{};
    a.model = model_dev(model);
    stage_metric(st, metric, D, N, &a.metric);
    a.D = D;
    a.N = N;
    a.eps = eps;
    st.in(eps_chain, (size_t)N, &a.eps_chain);
    a.n_steps = n_abs;
    a.fwd = n_steps > 0;
    a.temper_alpha = temper_alpha;
    a.ld_in = z_in->ld;
    a.ld_out = z_out->ld;
    st.in((const double*)z_in->theta, cin, &a.th_in);
    st.in((const double*)z_in->r, cin, &a.r_in);
    st.in((const double*)z_in->lp_gradient, cin, &a.g_in);
    st.out(z_out->theta, cout, &a.th_out);
    st.out(z_out->r, cout, &a.r_out);
    st.out(z_out->lp_gradient, cout, &a.g_out);
    st.out(z_out->lk_gradient, cout, &a.dr_out);
    st.out(z_out->lp_value, (size_t)N, &a.lp_out);
    st.out(z_out->lk_value, (size_t)N, &a.lk_out);
    st.out(status, (size_t)N, &a.status);
    st.out(steps_done, (size_t)N, &a.steps_done);
    if ((rc = st.commit())) return rc;
    a.flags = flags;
    const bool compat = flags & AHMC_FLAG_COMPAT_BREAK_ALL;
    if (dense_eligible(model, a.metric, flags, temper_alpha, compat, a.g_in, D)) {
        int nl = 0;
        if ((rc = dense_trajectory(ctx, model, a, n_abs, eps, &nl))) return rc;
        ctx->launches += nl;
        return finish_call(ctx, st, flags);
    }
    if (model->kind == AHMC_MODEL_CALLBACK) {
        // split-step mode: the work state is the OUTPUT phase point; two small kernels + the user closure per step
        SplitWork w;
        if ((rc = split_workspace(ctx, D, N, z_out->ld, &w))) return rc;
        if ((rc = copy_cols(ctx, a.th_out, a.ld_out, a.th_in, a.ld_in, D, N))) return rc;
        if ((rc = copy_cols(ctx, a.r_out, a.ld_out, a.r_in, a.ld_in, D, N))) return rc;
        if ((rc = copy_cols(ctx, a.g_out, a.ld_out, a.g_in, a.ld_in, D, N))) return rc;
        int nl = 0;
        rc = split_trajectory(ctx, model, a.metric, D, N, eps, a.eps_chain, n_abs, a.fwd, temper_alpha, a.th_out, a.r_out,
                              a.g_out, a.lp_out, a.lk_out, a.dr_out, a.ld_out, a.status ? a.status : w.status,
                              a.steps_done, w, compat, &nl);
        ctx->launches += nl;
        if (rc) return rc;
        return finish_call(ctx, st, flags);
    }
    if (compat) {
        const int big = 0x7fffffff;
        CU(cudaMemcpyAsync(ctx->d_min_break, &big, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        a.min_break = ctx->d_min_break;
    }
    int nl = 0;
    CU(launch_leapfrog(a, ctx->stream, &nl));
    if (compat) {
        // reference quirk Q1: `isfinite(z)` is all(...) over every chain, so the first non-finite step
        // stops ALL chains.  Re-run everyone for exactly that many steps (inputs are untouched unless
        // the caller aliased z_out = z_in, which COMPAT mode therefore forbids).
        int mb = 0;
        CU(cudaMemcpyAsync(&mb, ctx->d_min_break, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        if (mb < n_abs) {
            if (!host && z_in->theta == z_out->theta)
                return fail(ctx, AHMC_ERR_INVALID, "COMPAT_BREAK_ALL cannot re-run an in-place call (z_out aliases z_in)");
            a.n_steps = mb;
            a.min_break = nullptr;
            a.flags |= AHMC_FLAG_EXACT_CHECKS;
            CU(launch_leapfrog(a, ctx->stream, &nl));
        }
    }
    ctx->launches += nl;
    return finish_call(ctx, st, flags);
}

// ---------------------------------------------------------------------------------------------- rand_momentum
int ahmc_rand_momentum_f64(ahmc_ctx* ctx, const ahmc_metric* metric, int32_t D, int64_t N, const ahmc_rng* rng,
                           double* r, int64_t ld, uint32_t flags) {
    if (!ctx || !metric || !rng || !r) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/metric/rng/r");
    int rc = check_common(ctx, nullptr, metric, D, N);
    if (rc) return rc;
    if (ld < D) return fail(ctx, AHMC_ERR_INVALID, "ld < D");
    if (metric->kind == AHMC_METRIC_DENSE && !metric->cholU)
        return fail(ctx, AHMC_ERR_INVALID, "Dense metric needs cholU for rand_momentum (metric.jl:311-320)");
    if (N == 0) return AHMC_OK;
    DeviceGuard g(ctx->device);
    Stager st(ctx, flags & AHMC_FLAG_HOST_BUFFERS);
    MomentumArgs a{};
    stage_metric(st, metric, D, N, &a.metric);
    a.D = D;
    a.N = N;
    a.seed = rng->seed;
    a.offset = rng->offset;
    st.in(rng->normal_tape, (size_t)D * N, &a.normal_tape);
    st.out(r, (size_t)ld * N, &a.r);
    if ((rc = st.commit())) return rc;
    a.ld = ld;
    int nl = 0;
    CU(launch_rand_momentum(a, ctx->stream, &nl));
    ctx->launches += nl;
    return finish_call(ctx, st, flags);
}

// ---------------------------------------------------------------------------------------------- transitions
static int hmc_impl(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                    double eps, const double* eps_chain, int32_t n_steps, int32_t n_transitions, const ahmc_rng* rng,
                    const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out, double* draws, const ahmc_stats* stats,
                    uint32_t flags) {
    if (!ctx || !model || !metric || !rng) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/model/metric/rng");
    if (n_transitions < 1) return fail(ctx, AHMC_ERR_INVALID, "n_transitions must be >= 1");
    if (n_transitions > 1 && (rng->normal_tape || rng->exp_tape))
        return fail(ctx, AHMC_ERR_INVALID, "random tapes describe ONE transition; multi-transition sampling uses the Philox streams");
    if (n_transitions > 1 && model->kind == AHMC_MODEL_CALLBACK)
        return fail(ctx, AHMC_ERR_UNSUPPORTED, "multi-transition sampling needs a device-resident target");
    if (rng->partial_refresh_alpha != 0.0 && model->kind == AHMC_MODEL_CALLBACK)
        return fail(ctx, AHMC_ERR_UNSUPPORTED, "partial momentum refreshment is not wired into the split-step path");
    int rc = check_rng_alphas(ctx, rng);
    if (rc) return rc;
    if ((rc = check_common(ctx, model, metric, D, N))) return rc;
    if ((rc = check_pp(ctx, z_in, D, "z_in", true, N))) return rc;
    if ((rc = check_pp(ctx, z_out, D, "z_out", true, N))) return rc;
    if (n_steps < 1) return fail(ctx, AHMC_ERR_INVALID, "n_steps must be >= 1 (nsteps(tau) = max(1, ...), trajectory.jl:240-243)");
    if (flags & AHMC_FLAG_COMPAT_BREAK_ALL)
        return fail(ctx, AHMC_ERR_UNSUPPORTED, "COMPAT_BREAK_ALL is only available on ahmc_leapfrog_f64");
    if ((rc = check_transition_output(ctx, metric, z_out, flags))) return rc;
    if (N == 0) return AHMC_OK;
    DeviceGuard g(ctx->device);
    Stager st(ctx, flags & AHMC_FLAG_HOST_BUFFERS);
    HmcArgs h{};
    LeapfrogArgs& a = h.lf;
    a.model = model_dev(model);
    stage_metric(st, metric, D, N, &a.metric);
    a.D = D;
    a.N = N;
    a.eps = eps;
    st.in(eps_chain, (size_t)N, &a.eps_chain);
    a.n_steps = n_steps;
    a.fwd = 1;
    a.temper_alpha = 0.0;
    stage_transition_pp(st, z_in, z_out, N, a);
    a.flags = flags;
    stage_rng(st, rng, D, N, false, &h.rng);
    stage_stats(st, stats, N * n_transitions, &h.st);
    st.out(draws, (size_t)D * N * n_transitions, &h.draws);
    if ((rc = st.commit())) return rc;
    h.n_transitions = n_transitions;
    h.refresh = (flags & AHMC_FLAG_NO_REFRESH) ? 0 : 1;
    int nl = 0;
    // Callback targets, and GEMM-shaped operators of a single plain transition that the tiled K4 trajectory takes, run
    // unfused with hmc_kernel's semantics: refresh -> kinetic energy -> start point copied to z_out -> trajectory in
    // place on z_out -> MH select.  Everything else is one fused launch.
    const bool callback = model->kind == AHMC_MODEL_CALLBACK;
    const bool k4 = !callback && n_transitions == 1 && a.th_out != a.th_in && h.rng.partial_alpha == 0.0 && !draws &&
                    dense_eligible(model, a.metric, flags, h.rng.temper_alpha, false, a.g_out, D);
    if (!callback && !k4) {
        CU(launch_hmc(h, ctx->stream, &nl));
        ctx->launches += nl;
        return finish_call(ctx, st, flags);
    }
    if (callback && a.th_out == a.th_in)
        return fail(ctx, AHMC_ERR_INVALID, "callback-mode transitions need z_out distinct from z_in (the start point is re-read on rejection)");
    SplitWork w;
    if ((rc = split_workspace(ctx, D, N, z_out->ld, &w))) return rc;
    if (h.refresh) {
        MomentumArgs ma{};
        ma.metric = a.metric; ma.D = D; ma.N = N; ma.seed = h.rng.seed; ma.offset = h.rng.offset;
        ma.normal_tape = h.rng.normal_tape; ma.r = w.r0; ma.ld = D;
        CU(launch_rand_momentum(ma, ctx->stream, &nl));
    } else if ((rc = copy_cols(ctx, w.r0, D, a.r_in, a.ld_in, D, N))) {
        return rc;
    }
    SplitArgs k0{};  // lk0 = neg kinetic energy of the refreshed momentum
    k0.metric = a.metric; k0.D = D; k0.N = N; k0.fwd = 1; k0.mul = 1.0; k0.no_kick = 1;
    k0.r = w.r0; k0.lk = w.lk0; k0.ld = D;
    CU(launch_kick_energy(k0, ctx->stream, &nl));
    if ((rc = copy_cols(ctx, a.th_out, a.ld_out, a.th_in, a.ld_in, D, N))) return rc;
    if ((rc = copy_cols(ctx, a.g_out, a.ld_out, a.g_in, a.ld_in, D, N))) return rc;
    if ((rc = copy_cols(ctx, a.r_out, a.ld_out, w.r0, D, D, N))) return rc;
    if (callback) {
        rc = split_trajectory(ctx, model, a.metric, D, N, eps, a.eps_chain, n_steps, 1, h.rng.temper_alpha, a.th_out, a.r_out,
                              a.g_out, a.lp_out, a.lk_out, nullptr, a.ld_out, w.status, w.steps, w, false, &nl);
    } else {
        LeapfrogArgs t = a;
        t.th_in = a.th_out; t.r_in = a.r_out; t.g_in = a.g_out; t.ld_in = a.ld_out;
        t.status = nullptr; t.steps_done = nullptr;
        rc = dense_trajectory(ctx, model, t, n_steps, eps, &nl);
    }
    if (rc) return rc;
    MhArgs m{};
    m.D = D; m.N = N; m.n_steps = n_steps;
    m.th0 = a.th_in; m.g0 = a.g_in; m.lp0 = a.lp_in; m.ld0 = a.ld_in;
    m.r0 = w.r0; m.lk0 = w.lk0;
    m.th = a.th_out; m.r = a.r_out; m.g = a.g_out; m.lp = a.lp_out; m.lk = a.lk_out; m.ld = a.ld_out;
    m.rng = h.rng; m.st = h.st;
    CU(launch_mh_select(m, ctx->stream, &nl));
    ctx->launches += nl;
    return finish_call(ctx, st, flags);
}

static int nuts_impl(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                     double eps, const double* eps_chain, int32_t max_depth, double delta_max, int32_t n_transitions,
                     const ahmc_rng* rng, const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out, double* draws,
                     const ahmc_stats* stats, uint32_t flags, const ahmc_adapt_cfg* cfg = nullptr) {
    if (!ctx || !model || !metric || !rng) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/model/metric/rng");
    if (n_transitions < 1) return fail(ctx, AHMC_ERR_INVALID, "n_transitions must be >= 1");
    if (cfg) {
        if (metric->kind != AHMC_METRIC_DIAG)
            return fail(ctx, AHMC_ERR_UNSUPPORTED, "in-launch adaptation needs the Diag metric (per-chain diagonal M^-1)");
        if (flags & (AHMC_FLAG_NUTS_SLICE_TS | AHMC_FLAG_NUTS_CLASSIC | AHMC_FLAG_NUTS_STRICT))
            return fail(ctx, AHMC_ERR_UNSUPPORTED, "in-launch adaptation is built for MultinomialTS + GeneralisedNoUTurn");
        if (rng->normal_tape || rng->exp_tape || rng->dir_tape)
            return fail(ctx, AHMC_ERR_INVALID, "in-launch adaptation draws from the Philox streams (no tapes)");
        if (cfg->n_adapts < 0 || cfg->n_adapts > n_transitions)
            return fail(ctx, AHMC_ERR_INVALID, "need 0 <= n_adapts <= n_transitions");
        if (!cfg->eps_chain) return fail(ctx, AHMC_ERR_INVALID, "cfg.eps_chain (N, in/out) is required");
        if (cfg->adapt_metric && !cfg->Minv_chain)
            return fail(ctx, AHMC_ERR_INVALID, "cfg.Minv_chain (N x D, out) is required with adapt_metric");
        if (cfg->init_buffer < 0 || cfg->term_buffer < 0 || cfg->window_size < 1)
            return fail(ctx, AHMC_ERR_INVALID, "need init_buffer >= 0, term_buffer >= 0, window_size >= 1");
        if (!(cfg->gamma > 0.0) || !(cfg->t0 >= 0.0) || !(cfg->delta > 0.0 && cfg->delta < 1.0))
            return fail(ctx, AHMC_ERR_INVALID, "need gamma > 0, t0 >= 0, 0 < delta < 1");
    }
    if (n_transitions > 1 && (rng->normal_tape || rng->exp_tape || rng->dir_tape))
        return fail(ctx, AHMC_ERR_INVALID, "random tapes describe ONE transition; multi-transition sampling uses the Philox streams");
    int rc = check_rng_alphas(ctx, rng);
    if (rc) return rc;
    if ((rc = check_common(ctx, model, metric, D, N))) return rc;
    if ((rc = check_pp(ctx, z_in, D, "z_in", true, N))) return rc;
    if ((rc = check_pp(ctx, z_out, D, "z_out", true, N))) return rc;
    if (max_depth < 0 || max_depth > 20) return fail(ctx, AHMC_ERR_INVALID, "max_depth must be in 0..20");
    if (cfg && max_depth == 0)  // no leaf is ever built: acceptance_rate = 0/0 (as in the reference) would poison dual averaging
        return fail(ctx, AHMC_ERR_INVALID, "in-launch adaptation needs max_depth >= 1");
    if ((flags & AHMC_FLAG_NUTS_CLASSIC) && (flags & AHMC_FLAG_NUTS_STRICT))
        return fail(ctx, AHMC_ERR_INVALID, "AHMC_FLAG_NUTS_CLASSIC and AHMC_FLAG_NUTS_STRICT are mutually exclusive");
    if (model->kind == AHMC_MODEL_CALLBACK)
        return fail(ctx, AHMC_ERR_UNSUPPORTED, "NUTS needs a device-resident target: callback (split-step) models are supported by ahmc_leapfrog_f64 / ahmc_hmc_transition_f64 / ahmc_phasepoint_f64 only; express the target as CUDA source (ahmc_model_create_user) to run NUTS on it");
    if (model->kind == AHMC_MODEL_USER && (cfg || (flags & (AHMC_FLAG_NUTS_SLICE_TS | AHMC_FLAG_NUTS_CLASSIC | AHMC_FLAG_NUTS_STRICT))))
        return fail(ctx, AHMC_ERR_UNSUPPORTED, "run-time compiled targets: MultinomialTS + GeneralisedNoUTurn without in-launch adaptation");
    if ((rc = check_transition_output(ctx, metric, z_out, flags))) return rc;
    if (rng->exp_tape && rng->exp_stride < 1) return fail(ctx, AHMC_ERR_INVALID, "exp_tape needs exp_stride >= 1");
    if (rng->dir_tape && rng->dir_stride < max_depth) return fail(ctx, AHMC_ERR_INVALID, "dir_tape needs dir_stride >= max_depth");
    if (N == 0) return AHMC_OK;
    DeviceGuard g(ctx->device);
    Stager st(ctx, flags & AHMC_FLAG_HOST_BUFFERS);
    NutsArgs a{};
    a.model = model_dev(model);
    stage_metric(st, metric, D, N, &a.metric);
    if (cfg) {
        st.inout(cfg->eps_chain, (size_t)N, &a.ad.eps);
        st.out(cfg->Minv_chain, (size_t)N * D, &a.ad.minv);
        st.out(cfg->eps_trace, (size_t)N * n_transitions, &a.ad.eps_trace);
    } else {
        st.in(eps_chain, (size_t)N, &a.eps_chain);
    }
    stage_transition_pp(st, z_in, z_out, N, a);
    stage_rng(st, rng, D, N, true, &a.rng);
    stage_stats(st, stats, N * n_transitions, &a.st);
    st.out(draws, (size_t)D * N * n_transitions, &a.draws);
    if ((rc = st.commit())) return rc;
    int n_prep = 0;
    if (a.metric.kind == AHMC_METRIC_DENSE && D > 16 && D <= 512) {
        // the cooperative form streams Minv / cholU in chunks of columns: hand it copies whose columns are padded to the
        // shared-memory leading dimension, so that a chunk is one bulk copy (two small kernels per call, on the stream)
        const size_t per = coop_padded_doubles(D);
        if ((rc = grow(ctx, ctx->coop_scratch, 2 * per * sizeof(double), "column-padded metric"))) return rc;
        double* coop = (double*)ctx->coop_scratch.p;
        CU(launch_pad_columns(a.metric.Minv, D, coop, ctx->stream));
        a.metric.Minv_coop = coop;
        ++n_prep;
        if (a.metric.cholU) {
            CU(launch_pad_columns(a.metric.cholU, D, coop + per, ctx->stream));
            a.metric.cholU_coop = coop + per;
            ++n_prep;
        }
    }
    ctx->launches += n_prep;
    a.D = D;
    a.N = N;
    a.eps = eps;
    if (cfg) {
        AdaptDev& ad = a.ad;
        ad.enabled = 1;
        ad.n_adapts = cfg->n_adapts;
        ad.delta = cfg->delta;
        ad.gamma = cfg->gamma;
        ad.t0 = cfg->t0;
        ad.kappa = cfg->kappa;
        ad.adapt_metric = cfg->adapt_metric ? 1 : 0;
        ad.n_min = cfg->n_min > 0 ? cfg->n_min : 10;
        if (!stan_window_schedule(ad, cfg->init_buffer, cfg->term_buffer, cfg->window_size, cfg->n_adapts))
            return fail(ctx, AHMC_ERR_UNSUPPORTED, "the window schedule (stan_adaptor.jl:13-50) needs more than %d splits",
                        (int)(sizeof(ad.splits) / sizeof(ad.splits[0])));
        a.eps_chain = ad.eps;
    }
    a.max_depth = max_depth;
    a.delta_max = delta_max;
    a.sampler = (flags & AHMC_FLAG_NUTS_SLICE_TS) ? 1 : 0;
    a.criterion = (flags & AHMC_FLAG_NUTS_STRICT) ? 2 : (flags & AHMC_FLAG_NUTS_CLASSIC) ? 1 : 0;
    a.refresh = (flags & AHMC_FLAG_NO_REFRESH) ? 0 : 1;
    a.n_transitions = n_transitions;
    // per-chain tree workspace
    a.scratch_stride = nuts_scratch_doubles_per_chain(D, max_depth, cfg != nullptr);
    if ((rc = grow(ctx, ctx->nuts_scratch, (size_t)a.scratch_stride * (size_t)N * sizeof(double), "NUTS workspace"))) return rc;
    a.scratch = (double*)ctx->nuts_scratch.p;
    int nl = 0;
    CU(launch_nuts(a, ctx->stream, &nl));
    ctx->launches += nl;
    return finish_call(ctx, st, flags);
}

int ahmc_leapfrog_trajectory_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D,
                                 int64_t N, double eps, const double* eps_chain, int32_t n_steps, double temper_alpha,
                                 const ahmc_phasepoint* z_in, const ahmc_phasepoint* traj, int64_t step_stride,
                                 int32_t* steps_done, uint32_t flags) {
    if (!ctx || !model || !metric) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/model/metric");
    int rc = check_common(ctx, model, metric, D, N);
    if (rc) return rc;
    if ((rc = check_pp(ctx, z_in, D, "z_in", true, N))) return rc;
    const int n_abs = n_steps < 0 ? -n_steps : n_steps;
    if (n_abs == 0 || N == 0) return AHMC_OK;  // res = Vector{P}(undef, 0)
    if ((rc = check_pp(ctx, traj, D, "traj", true, N))) return rc;
    if (step_stride < traj->ld * N) return fail(ctx, AHMC_ERR_INVALID, "step_stride must be >= ld*N");
    if (model->kind == AHMC_MODEL_CALLBACK || model->kind == AHMC_MODEL_USER)
        return fail(ctx, AHMC_ERR_UNSUPPORTED, "full_trajectory: built-in targets only (callback / run-time compiled targets: loop over ahmc_leapfrog_f64)");
    DeviceGuard g(ctx->device);
    Stager st(ctx, flags & AHMC_FLAG_HOST_BUFFERS);
    const size_t cin = (size_t)z_in->ld * N, ctraj = (size_t)step_stride * n_abs;
    TrajArgs a{};
    a.model = model_dev(model);
    stage_metric(st, metric, D, N, &a.metric);
    a.D = D; a.N = N; a.eps = eps;
    st.in(eps_chain, (size_t)N, &a.eps_chain);
    a.n_steps = n_abs; a.fwd = n_steps > 0; a.temper_alpha = temper_alpha;
    a.ld_in = z_in->ld; a.ld_out = traj->ld; a.step_stride = step_stride;
    st.in((const double*)z_in->theta, cin, &a.th_in);
    st.in((const double*)z_in->r, cin, &a.r_in);
    st.in((const double*)z_in->lp_gradient, cin, &a.g_in);
    st.out(traj->theta, ctraj, &a.th_out);
    st.out(traj->r, ctraj, &a.r_out);
    st.out(traj->lp_gradient, ctraj, &a.g_out);
    st.out(traj->lk_gradient, ctraj, &a.dr_out);
    st.out(traj->lp_value, (size_t)N * n_abs, &a.lp_out);
    st.out(traj->lk_value, (size_t)N * n_abs, &a.lk_out);
    st.out(steps_done, (size_t)N, &a.steps_done);
    if ((rc = st.commit())) return rc;
    int nl = 0;
    CU(launch_trajectory(a, ctx->stream, &nl));
    ctx->launches += nl;
    return finish_call(ctx, st, flags);
}

int ahmc_hmc_multinomial_transition_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D,
                                        int64_t N, double eps, const double* eps_chain, int32_t n_steps,
                                        int32_t n_steps_fwd, const ahmc_rng* rng, const ahmc_phasepoint* z_in,
                                        const ahmc_phasepoint* z_out, const ahmc_stats* stats, uint32_t flags) {
    if (!ctx || !model || !metric || !rng) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/model/metric/rng");
    int rc = check_common(ctx, model, metric, D, N);
    if (rc) return rc;
    if ((rc = check_pp(ctx, z_in, D, "z_in", true, N))) return rc;
    if ((rc = check_pp(ctx, z_out, D, "z_out", true, N))) return rc;
    if (n_steps < 1 || n_steps_fwd < 0 || n_steps_fwd > n_steps)
        return fail(ctx, AHMC_ERR_INVALID, "need n_steps >= 1 and 0 <= n_steps_fwd <= n_steps (rand(0:n_steps), trajectory.jl:373)");
    if (model->kind == AHMC_MODEL_CALLBACK || model->kind == AHMC_MODEL_USER)
        return fail(ctx, AHMC_ERR_UNSUPPORTED, "MultinomialTS static transitions: built-in targets only");
    if ((rc = check_transition_output(ctx, metric, z_out, flags))) return rc;
    if ((rc = check_rng_alphas(ctx, rng))) return rc;
    if (N == 0) return AHMC_OK;
    DeviceGuard g(ctx->device);
    Stager st(ctx, flags & AHMC_FLAG_HOST_BUFFERS);
    MultinomialArgs a{};
    a.model = model_dev(model);
    stage_metric(st, metric, D, N, &a.metric);
    a.D = D; a.N = N; a.eps = eps;
    st.in(eps_chain, (size_t)N, &a.eps_chain);
    a.n_steps = n_steps; a.n_fwd = n_steps_fwd;
    a.refresh = (flags & AHMC_FLAG_NO_REFRESH) ? 0 : 1;
    stage_transition_pp(st, z_in, z_out, N, a);
    stage_rng(st, rng, D, N, false, &a.rng);
    stage_stats(st, stats, N, &a.st);
    if ((rc = st.commit())) return rc;
    if ((rc = grow(ctx, ctx->mn_scratch, (size_t)(n_steps + 1) * (size_t)N * sizeof(double), "multinomial energy tape"))) return rc;
    a.energies = (double*)ctx->mn_scratch.p;
    int nl = 0;
    CU(launch_multinomial(a, ctx->stream, &nl));
    ctx->launches += nl;
    return finish_call(ctx, st, flags);
}

int ahmc_hmc_transition_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                            double eps, const double* eps_chain, int32_t n_steps, const ahmc_rng* rng,
                            const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out, const ahmc_stats* stats,
                            uint32_t flags) {
    return hmc_impl(ctx, model, metric, D, N, eps, eps_chain, n_steps, 1, rng, z_in, z_out, nullptr, stats, flags);
}

int ahmc_nuts_transition_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                             double eps, const double* eps_chain, int32_t max_depth, double delta_max,
                             const ahmc_rng* rng, const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out,
                             const ahmc_stats* stats, uint32_t flags) {
    return nuts_impl(ctx, model, metric, D, N, eps, eps_chain, max_depth, delta_max, 1, rng, z_in, z_out, nullptr, stats,
                     flags);
}

int ahmc_hmc_sample_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                        double eps, const double* eps_chain, int32_t n_steps, int32_t n_transitions, const ahmc_rng* rng,
                        const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out, double* draws,
                        const ahmc_stats* stats, uint32_t flags) {
    return hmc_impl(ctx, model, metric, D, N, eps, eps_chain, n_steps, n_transitions, rng, z_in, z_out, draws, stats, flags);
}

int ahmc_nuts_sample_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                         double eps, const double* eps_chain, int32_t max_depth, double delta_max, int32_t n_transitions,
                         const ahmc_rng* rng, const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out, double* draws,
                         const ahmc_stats* stats, uint32_t flags) {
    return nuts_impl(ctx, model, metric, D, N, eps, eps_chain, max_depth, delta_max, n_transitions, rng, z_in, z_out,
                     draws, stats, flags);
}

int ahmc_nuts_adapt_sample_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                               int32_t max_depth, double delta_max, int32_t n_transitions, const ahmc_adapt_cfg* cfg,
                               const ahmc_rng* rng, const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out,
                               double* draws, const ahmc_stats* stats, uint32_t flags) {
    if (!cfg) return fail(ctx, AHMC_ERR_INVALID, "NULL cfg");
    return nuts_impl(ctx, model, metric, D, N, 0.0, nullptr, max_depth, delta_max, n_transitions, rng, z_in, z_out, draws,
                     stats, flags, cfg);
}

// ---------------------------------------------------------------------------------------------- adaptor stats
int ahmc_adapt_summary_f64(ahmc_ctx* ctx, int32_t D, int64_t N, const double* theta, int64_t ld,
                           const double* acceptance_rate, double* out, uint32_t flags) {
    if (!ctx || !theta || !out) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/theta/out");
    if (D < 1 || N < 1 || ld < D) return fail(ctx, AHMC_ERR_INVALID, "need D >= 1, N >= 1, ld >= D");
    DeviceGuard g(ctx->device);
    int blocks;
    int rc = adapt_workspace(ctx, D, N, &blocks);
    if (rc) return rc;
    Stager st(ctx, flags & AHMC_FLAG_HOST_BUFFERS);
    const double *d_theta, *d_alpha;
    double* d_out;
    st.in(theta, (size_t)ld * N, &d_theta);
    st.in(acceptance_rate, (size_t)N, &d_alpha);
    st.out(out, (size_t)(2 + 2 * D), &d_out);
    if ((rc = st.commit())) return rc;
    double* ws = (double*)ctx->adapt_scratch.p;
    int nl = 0;
    CU(launch_adapt_summary(D, N, d_theta, ld, d_alpha, d_out, ws + 2, (unsigned*)ws, blocks, ctx->stream, &nl));
    ctx->launches += nl;
    return finish_call(ctx, st, flags);
}

int ahmc_adapt_cov_f64(ahmc_ctx* ctx, int32_t D, int64_t N, const double* theta, int64_t ld, const double* mean,
                       double* out, uint32_t flags) {
    if (!ctx || !theta || !mean || !out) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/theta/mean/out");
    if (D < 1 || N < 1 || ld < D) return fail(ctx, AHMC_ERR_INVALID, "need D >= 1, N >= 1, ld >= D");
    DeviceGuard g(ctx->device);
    Stager st(ctx, flags & AHMC_FLAG_HOST_BUFFERS);
    const double *d_theta, *d_mean;
    double* d_out;
    st.in(theta, (size_t)ld * N, &d_theta);
    st.in(mean, (size_t)D, &d_mean);
    st.out(out, (size_t)D * D, &d_out);
    int rc = st.commit();
    if (rc) return rc;
    int nl = 0;
    CU(launch_adapt_cov(D, N, d_theta, ld, d_mean, d_out, ctx->stream, &nl));
    ctx->launches += nl;
    return finish_call(ctx, st, flags);
}

int ahmc_find_good_stepsize_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                                const ahmc_phasepoint* z, const ahmc_rng* rng, double initial_step_size, int32_t max_n_iters,
                                double* eps_out, double* r_out, uint32_t flags) {
    if (!ctx || !model || !metric || !rng || !eps_out) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/model/metric/rng/eps_out");
    int rc = check_common(ctx, model, metric, D, N);
    if (rc) return rc;
    if (!z || (N > 0 && (!z->theta || !z->lp_value || !z->lp_gradient)))
        return fail(ctx, AHMC_ERR_INVALID, "z.theta / lp_value / lp_gradient is NULL (call ahmc_phasepoint_f64 first)");
    if (N > 0 && z->ld < D) return fail(ctx, AHMC_ERR_INVALID, "z.ld < D");
    if (!(initial_step_size > 0.0) || max_n_iters < 0) return fail(ctx, AHMC_ERR_INVALID, "need initial_step_size > 0, max_n_iters >= 0");
    if (model->kind == AHMC_MODEL_CALLBACK)
        return fail(ctx, AHMC_ERR_UNSUPPORTED, "find_good_stepsize in one launch needs the gradient inside the kernel (built-in targets)");
    if (N == 0) return AHMC_OK;
    DeviceGuard g(ctx->device);
    Stager st(ctx, flags & AHMC_FLAG_HOST_BUFFERS);
    const size_t cin = (size_t)z->ld * N;
    FindEpsArgs a{};
    a.model = model_dev(model);
    stage_metric(st, metric, D, N, &a.metric);
    a.D = D;
    a.N = N;
    a.ld = z->ld;
    st.in((const double*)z->theta, cin, &a.th);
    st.in((const double*)z->lp_gradient, cin, &a.g);
    st.in((const double*)z->lp_value, (size_t)N, &a.lp);
    st.in(rng->normal_tape, (size_t)D * N, &a.normal_tape);
    a.seed = rng->seed;
    a.offset = rng->offset;
    a.eps0 = initial_step_size;
    a.max_iters = max_n_iters;
    st.out(eps_out, (size_t)N, &a.eps_out);
    st.out(r_out, cin, &a.r_out);
    if ((rc = st.commit())) return rc;
    int nl = 0;
    CU(launch_find_eps(a, ctx->stream, &nl));
    ctx->launches += nl;
    return finish_call(ctx, st, flags);
}

// ------------------------------------------------------------------------------------------ comm + pooled adaptor
struct ahmc_comm {
    void* nccl = nullptr;
    int nranks = 1, rank = 0;
    bool owned = false;
};
struct ahmc_pooled {
    int D = 0;
    int64_t N = 0;
    char* dev = nullptr;  // one allocation: state | eps_chain | minv | w_mu | w_M2 | record | merged (dense: see _create_dense)
    void* state = nullptr;
    double *eps_chain = nullptr, *minv = nullptr, *w_mu = nullptr, *w_M2 = nullptr, *record = nullptr, *merged = nullptr;
    DevBuf gathered;  // R records of the last multi-rank exchange (grown on demand)
    // dense adaptor (pooled WelfordCov): minv and cholU are D x D column-major; w_M the window's D x D accumulator, cand the
    // candidate estimate, work the factorisation's workspace.  The host follows the schedule to launch the factorisation
    // only at window splits.
    bool dense = false;
    int adapt_metric = 0;
    int calls = 0;  // exchanges so far
    AdaptDev sched{};
    double *cholU = nullptr, *w_M = nullptr, *cand = nullptr, *work = nullptr;
    size_t record_len() const { return (size_t)(2 + 2 * D) + (dense && adapt_metric ? (size_t)D * D : 0); }
};

int ahmc_comm_unique_id(ahmc_ctx* ctx, void* id128_out) {
    if (!ctx || !id128_out) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/id");
    if (const char* why = nccl_bind()) return fail(ctx, AHMC_ERR_UNSUPPORTED, "NCCL unavailable: %s", why);
    int rc = nccl_unique_id(id128_out);
    if (rc) return fail(ctx, AHMC_ERR_CUDA, "ncclGetUniqueId: %s", nccl_err(rc));
    return AHMC_OK;
}
int ahmc_comm_create(ahmc_ctx* ctx, const void* id128, int32_t nranks, int32_t rank, ahmc_comm** out) {
    if (!ctx || !id128 || !out) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/id/out");
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(ctx, AHMC_ERR_INVALID, "need 0 <= rank < nranks");
    if (const char* why = nccl_bind()) return fail(ctx, AHMC_ERR_UNSUPPORTED, "NCCL unavailable: %s", why);
    DeviceGuard g(ctx->device);
    void* c = nullptr;
    int rc = nccl_comm_init(&c, nranks, id128, rank);
    if (rc) return fail(ctx, AHMC_ERR_CUDA, "ncclCommInitRank: %s", nccl_err(rc));
    ahmc_comm* m = new (std::nothrow) ahmc_comm;
    if (!m) return fail(ctx, AHMC_ERR_NOMEM, "out of host memory");
    m->nccl = c; m->nranks = nranks; m->rank = rank; m->owned = true;
    *out = m;
    return AHMC_OK;
}
int ahmc_comm_from_nccl(ahmc_ctx* ctx, void* nccl_comm, int32_t nranks, int32_t rank, ahmc_comm** out) {
    if (!ctx || !nccl_comm || !out) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/comm/out");
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(ctx, AHMC_ERR_INVALID, "need 0 <= rank < nranks");
    if (const char* why = nccl_bind()) return fail(ctx, AHMC_ERR_UNSUPPORTED, "NCCL unavailable: %s", why);
    ahmc_comm* m = new (std::nothrow) ahmc_comm;
    if (!m) return fail(ctx, AHMC_ERR_NOMEM, "out of host memory");
    m->nccl = nccl_comm; m->nranks = nranks; m->rank = rank; m->owned = false;
    *out = m;
    return AHMC_OK;
}
int ahmc_comm_destroy(ahmc_ctx* ctx, ahmc_comm* comm) {
    if (!ctx) return AHMC_ERR_INVALID;
    if (!comm) return AHMC_OK;
    DeviceGuard g(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (comm->owned && comm->nccl) nccl_comm_destroy(comm->nccl);
    delete comm;
    return AHMC_OK;
}

int ahmc_adapt_allgather_f64(ahmc_ctx* ctx, ahmc_comm* comm, const double* record, int64_t n, double* out, uint32_t flags) {
    if (!ctx || !record || !out || n < 1) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/record/out or n < 1");
    if (flags & AHMC_FLAG_HOST_BUFFERS) return fail(ctx, AHMC_ERR_UNSUPPORTED, "the exchange takes device pointers");
    DeviceGuard g(ctx->device);
    if (!comm || comm->nranks == 1) {
        if (out != record) CU(cudaMemcpyAsync(out, record, (size_t)n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
        int rc = nccl_allgather_f64(record, out, (size_t)n, comm->nccl, ctx->stream);
        if (rc) return fail(ctx, AHMC_ERR_CUDA, "ncclAllGather: %s", nccl_err(rc));
    }
    if (!(flags & AHMC_FLAG_ASYNC)) CU(cudaStreamSynchronize(ctx->stream));
    return AHMC_OK;
}

namespace {
int pooled_check(ahmc_ctx* ctx, int32_t D, int64_t N, const ahmc_pooled_cfg* cfg, ahmc_pooled** out, AdaptDev* sched) {
    if (!ctx || !cfg || !out) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/cfg/out");
    if (D < 1 || N < 1) return fail(ctx, AHMC_ERR_INVALID, "need D >= 1, N >= 1");
    if (cfg->n_adapts < 0 || !(cfg->eps0 > 0.0)) return fail(ctx, AHMC_ERR_INVALID, "need n_adapts >= 0 and eps0 > 0");
    if (!stan_window_schedule(*sched, cfg->init_buffer, cfg->term_buffer, cfg->window_size, cfg->n_adapts))
        return fail(ctx, AHMC_ERR_UNSUPPORTED, "the window schedule has more than 12 window ends");
    return AHMC_OK;
}
}  // namespace

int ahmc_pooled_create(ahmc_ctx* ctx, int32_t D, int64_t N, const ahmc_pooled_cfg* cfg, const double* Minv0, ahmc_pooled** out) {
    AdaptDev sched{};
    if (int rc = pooled_check(ctx, D, N, cfg, out, &sched)) return rc;
    DeviceGuard g(ctx->device);
    ahmc_pooled* a = new (std::nothrow) ahmc_pooled;
    if (!a) return fail(ctx, AHMC_ERR_NOMEM, "out of host memory");
    a->D = D;
    a->N = N;
    const size_t rec = (size_t)(2 + 2 * D) * 8;
    const size_t total = al256(pooled_state_bytes()) + al256((size_t)N * 8) + 3 * al256((size_t)D * 8) + 2 * al256(rec);
    if (cudaMalloc((void**)&a->dev, total) != cudaSuccess) {
        delete a;
        return fail(ctx, AHMC_ERR_NOMEM, "cudaMalloc(%zu) for the pooled adaptor failed", total);
    }
    char* p = a->dev;
    a->state = p; p += al256(pooled_state_bytes());
    a->eps_chain = (double*)p; p += al256((size_t)N * 8);
    a->minv = (double*)p; p += al256((size_t)D * 8);
    a->w_mu = (double*)p; p += al256((size_t)D * 8);
    a->w_M2 = (double*)p; p += al256((size_t)D * 8);
    a->record = (double*)p; p += al256(rec);
    a->merged = (double*)p;
    std::vector<char> img(pooled_state_bytes());
    pooled_state_init(img.data(), cfg->eps0, sched, cfg->delta, cfg->gamma, cfg->t0, cfg->kappa, cfg->n_adapts,
                      cfg->adapt_metric, cfg->n_min);
    CU(cudaMemcpyAsync(a->state, img.data(), img.size(), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemsetAsync(a->w_mu, 0, (size_t)D * 8, ctx->stream));
    CU(cudaMemsetAsync(a->w_M2, 0, (size_t)D * 8, ctx->stream));
    CU(cudaMemsetAsync(a->merged, 0, rec, ctx->stream));
    if (Minv0) CU(cudaMemcpyAsync(a->minv, Minv0, (size_t)D * 8, cudaMemcpyHostToDevice, ctx->stream));
    else CU(launch_fill(a->minv, D, 1.0, ctx->stream));
    CU(launch_fill(a->eps_chain, N, cfg->eps0, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));  // img / Minv0 are host memory of this frame
    *out = a;
    return AHMC_OK;
}
int ahmc_pooled_destroy(ahmc_ctx* ctx, ahmc_pooled* a) {
    if (!ctx) return AHMC_ERR_INVALID;
    if (!a) return AHMC_OK;
    DeviceGuard g(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(a->dev);
    cudaFree(a->gathered.p);
    delete a;
    return AHMC_OK;
}
int ahmc_pooled_create_dense(ahmc_ctx* ctx, int32_t D, int64_t N, const ahmc_pooled_cfg* cfg, const double* Minv0,
                             ahmc_pooled** out) {
    AdaptDev sched{};
    if (int rc = pooled_check(ctx, D, N, cfg, out, &sched)) return rc;
    if (D > 512) return fail(ctx, AHMC_ERR_UNSUPPORTED, "the dense pooled adaptor supports D <= 512 (got %d)", (int)D);
    DeviceGuard g(ctx->device);
    ahmc_pooled* a = new (std::nothrow) ahmc_pooled;
    if (!a) return fail(ctx, AHMC_ERR_NOMEM, "out of host memory");
    a->D = D;
    a->N = N;
    a->dense = true;
    a->adapt_metric = cfg->adapt_metric ? 1 : 0;
    a->sched = sched;
    const size_t dd = al256((size_t)D * D * 8), rec = al256(a->record_len() * 8), rec_full = al256(((size_t)(2 + 2 * D) + (size_t)D * D) * 8);
    const size_t total = al256(pooled_state_bytes()) + al256((size_t)N * 8) + 2 * al256((size_t)D * 8) + rec + rec_full + 5 * dd;
    if (cudaMalloc((void**)&a->dev, total) != cudaSuccess) {
        delete a;
        return fail(ctx, AHMC_ERR_NOMEM, "cudaMalloc(%zu) for the pooled adaptor failed", total);
    }
    char* p = a->dev;
    a->state = p; p += al256(pooled_state_bytes());
    a->eps_chain = (double*)p; p += al256((size_t)N * 8);
    a->w_mu = (double*)p; p += al256((size_t)D * 8);
    a->w_M2 = (double*)p; p += al256((size_t)D * 8);
    a->record = (double*)p; p += rec;
    a->merged = (double*)p; p += rec_full;
    a->minv = (double*)p; p += dd;
    a->cholU = (double*)p; p += dd;
    a->w_M = (double*)p; p += dd;
    a->cand = (double*)p; p += dd;
    a->work = (double*)p;
    auto undo = [&](int rc) {
        cudaStreamSynchronize(ctx->stream);
        cudaFree(a->dev);
        delete a;
        return rc;
    };
    std::vector<char> img(pooled_state_bytes());
    pooled_state_init(img.data(), cfg->eps0, sched, cfg->delta, cfg->gamma, cfg->t0, cfg->kappa, cfg->n_adapts, a->adapt_metric,
                      cfg->n_min);
    pooled_state_set_dense(img.data(), (int)a->record_len(), 0);
    cudaError_t e = cudaMemcpyAsync(a->state, img.data(), img.size(), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(a->w_mu, 0, (size_t)D * 8, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(a->w_M2, 0, (size_t)D * 8, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(a->merged, 0, rec_full, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(a->w_M, 0, (size_t)D * D * 8, ctx->stream);
    std::vector<double> eye;  // Minv0 == NULL: I
    if (!Minv0) {
        eye.assign((size_t)D * D, 0.0);
        for (int d = 0; d < D; ++d) eye[(size_t)d * (D + 1)] = 1.0;
    }
    // the candidate is factorised below and, when positive definite, committed to minv / cholU
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(a->cand, Minv0 ? Minv0 : eye.data(), (size_t)D * D * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = launch_fill(a->eps_chain, N, cfg->eps0, ctx->stream);
    int nl = 0;
    if (e == cudaSuccess) e = launch_pooled_chol(a->state, D, a->cand, a->work, a->minv, a->cholU, 1, ctx->stream, &nl);
    if (e == cudaSuccess) e = cudaMemcpyAsync(img.data(), a->state, img.size(), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);  // img / Minv0 / eye are host memory of this frame
    if (e != cudaSuccess) return undo(fail(ctx, AHMC_ERR_CUDA, "creating the dense pooled adaptor: %s", cudaGetErrorString(e)));
    ctx->launches += nl;
    int chol_failed = 0;
    pooled_state_read_dense(img.data(), nullptr, &chol_failed);
    if (chol_failed) return undo(fail(ctx, AHMC_ERR_INVALID, "Minv0 is not positive definite (Cholesky pivot <= 0 or NaN)"));
    *out = a;
    return AHMC_OK;
}

double* ahmc_pooled_eps(ahmc_pooled* a) { return a ? a->eps_chain : nullptr; }
double* ahmc_pooled_minv(ahmc_pooled* a) { return a ? a->minv : nullptr; }
double* ahmc_pooled_cholu(ahmc_pooled* a) { return a && a->dense ? a->cholU : nullptr; }

int ahmc_adapt_exchange_f64(ahmc_ctx* ctx, ahmc_comm* comm, ahmc_pooled* a, int32_t D, int64_t N, const double* theta,
                            int64_t ld, const double* acceptance_rate, double* eps_trace, uint32_t flags) {
    if (!ctx || !a || !theta || !acceptance_rate) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/adaptor/theta/acceptance_rate");
    if (flags & AHMC_FLAG_HOST_BUFFERS) return fail(ctx, AHMC_ERR_UNSUPPORTED, "the exchange takes device pointers");
    if (D != a->D || N != a->N || ld < D) return fail(ctx, AHMC_ERR_INVALID, "D / N differ from the adaptor's, or ld < D");
    DeviceGuard g(ctx->device);
    const int R = comm ? comm->nranks : 1;
    const size_t rec = a->record_len();
    const bool cov = a->dense && a->adapt_metric;  // the D x D part of the record is computed and merged
    int rc;
    if (R > 1 && (rc = grow(ctx, a->gathered, rec * 8 * (size_t)R, "gathered records"))) return rc;
    // K5 (+ K5b for a dense adaptor): this rank's record
    int blocks;
    if ((rc = adapt_workspace(ctx, D, N, &blocks))) return rc;
    double* ws = (double*)ctx->adapt_scratch.p;
    int nl = 0;
    CU(launch_adapt_summary(D, N, theta, ld, acceptance_rate, a->record, ws + 2, (unsigned*)ws, blocks, ctx->stream, &nl));
    if (cov) CU(launch_adapt_cov(D, N, theta, ld, a->record + 2, a->record + 2 + 2 * D, ctx->stream, &nl));
    const double* gathered = a->record;
    if (R > 1) {
        if ((rc = nccl_allgather_f64(a->record, (double*)a->gathered.p, rec, comm->nccl, ctx->stream)))
            return fail(ctx, AHMC_ERR_CUDA, "ncclAllGather: %s", nccl_err(rc));
        gathered = (double*)a->gathered.p;
    }
    // dense: the D x D merge / push reads the window's n and mean before pooled_update_kernel advances them
    if (cov) CU(launch_pooled_cov(a->state, gathered, R, D, a->w_mu, a->w_M, a->cand, a->merged, ctx->stream, &nl));
    CU(launch_pooled_update(a->state, gathered, R, D, a->w_mu, a->w_M2, a->dense ? nullptr : a->minv, a->eps_chain, N, eps_trace,
                            a->merged, ctx->stream, &nl));
    a->calls += 1;
    if (cov && pooled_chol_due(a->sched, a->adapt_metric, a->calls))
        CU(launch_pooled_chol(a->state, D, a->cand, a->work, a->minv, a->cholU, 0, ctx->stream, &nl));
    ctx->launches += nl;
    if (!(flags & AHMC_FLAG_ASYNC)) CU(cudaStreamSynchronize(ctx->stream));
    return AHMC_OK;
}

int ahmc_pooled_state(ahmc_ctx* ctx, ahmc_pooled* a, double* eps, double* Minv, int32_t* iteration, double* merged_record) {
    if (!ctx || !a) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/adaptor");
    if (a->dense) return fail(ctx, AHMC_ERR_INVALID, "dense pooled adaptor: read it with ahmc_pooled_state_dense");
    DeviceGuard g(ctx->device);
    std::vector<char> img(pooled_state_bytes());
    CU(cudaMemcpyAsync(img.data(), a->state, img.size(), cudaMemcpyDeviceToHost, ctx->stream));
    if (Minv) CU(cudaMemcpyAsync(Minv, a->minv, (size_t)a->D * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (merged_record) CU(cudaMemcpyAsync(merged_record, a->merged, (size_t)(2 + 2 * a->D) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    int it = 0;
    pooled_state_read(img.data(), eps, &it, nullptr, nullptr);
    if (iteration) *iteration = it;
    return AHMC_OK;
}

int ahmc_pooled_state_dense(ahmc_ctx* ctx, ahmc_pooled* a, double* eps, double* Minv, double* cholU, int32_t* iteration,
                            double* merged_record, int32_t* failed_iteration) {
    if (!ctx || !a) return fail(ctx, AHMC_ERR_INVALID, "NULL ctx/adaptor");
    if (!a->dense) return fail(ctx, AHMC_ERR_INVALID, "diagonal pooled adaptor: read it with ahmc_pooled_state");
    DeviceGuard g(ctx->device);
    const size_t dd = (size_t)a->D * a->D * 8;
    std::vector<char> img(pooled_state_bytes());
    CU(cudaMemcpyAsync(img.data(), a->state, img.size(), cudaMemcpyDeviceToHost, ctx->stream));
    if (Minv) CU(cudaMemcpyAsync(Minv, a->minv, dd, cudaMemcpyDeviceToHost, ctx->stream));
    if (cholU) CU(cudaMemcpyAsync(cholU, a->cholU, dd, cudaMemcpyDeviceToHost, ctx->stream));
    if (merged_record)
        CU(cudaMemcpyAsync(merged_record, a->merged, (size_t)(2 + 2 * a->D) * 8 + dd, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    int it = 0, failed = 0;
    pooled_state_read(img.data(), eps, &it, nullptr, nullptr);
    pooled_state_read_dense(img.data(), &failed, nullptr);
    if (iteration) *iteration = it;
    if (failed_iteration) *failed_iteration = failed;
    return AHMC_OK;
}

}  // extern "C"
