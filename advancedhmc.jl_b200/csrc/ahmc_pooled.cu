// ahmc_pooled.cu -- the path's one exchange, behind the C ABI and on the device (SURVEY 8e, DESIGN "K5c"):
// pooled (all chains of all ranks) step-size and mass-matrix adaptation with ZERO host synchronisation per warm-up
// iteration.  Per iteration, on the context stream:
//     K5 (ahmc_adapt.cu)      this rank's record  [N, sum min(1,alpha), mean_c theta, sum_c (theta - mean)^2]
//     ncclAllGather           (2 + 2D) doubles per rank -- latency only; skipped for a single rank
//     pooled_update_kernel    rank-ordered Chan merge (bit-identical on every rank), then the reference's adaptor
//                             arithmetic on the merged record: NesterovDualAveraging `adapt!` / `reset!` / `finalize!`
//                             (src/adaptation/stepsize.jl:38-62, 178-210), WelfordVar `push!` / `get_estimation`
//                             (massmatrix.jl:141-157, n_min :60-62), the Stan window schedule
//                             (stan_adaptor.jl:13-50, 137-159); eps and M^-1 are written straight into the device buffers
//                             the next transition reads (eps_chain[N], Minv[D]).
// A dense adaptor (pooled `WelfordCov`, massmatrix.jl:286-340) records (2 + 2D + D^2) doubles per rank (K5 + K5b), and
// runs, in this order:
//     pooled_cov_kernel       rank-ordered merge of the D x D blocks, push into the window's D x D accumulator and, at an
//                             update, the regularised estimate into a scratch candidate -- BEFORE pooled_update_kernel,
//                             which advances i, n and the window mean it reads
//     pooled_update_kernel    as above, with Minv == nullptr (the diagonal estimate is not written)
//     pooled_chol_kernel      only at window splits inside the metric window: factorises the candidate and, if every
//                             pivot is > 0, commits M^-1 and its upper factor U together; otherwise keeps both and
//                             records the iteration (`cholesky` throws PosDefException there, metric.jl:104-108).
// NCCL is bound at run time (dlopen): the library loads without it and a Julia host can hand over the communicator it
// already owns (NCCL.jl) or let ahmc_comm_create make one from a broadcast unique id.
#ifndef AHMC_SIMT_EMULATION
#include <dlfcn.h>
#endif

#include <cstdio>
#include <cstring>
#include <mutex>

#include "ahmc_kernels.cuh"

namespace ahmc {

// ---------------------------------------------------------------------------------------------- device state
struct PooledState {
    // dual averaging (stepsize.jl:25-36)
    double eps, mu, x_bar, H_bar;
    double delta, gamma, t0, kappa;
    int m;
    // Welford over chains x iterations of the current window (massmatrix.jl:86-101)
    double n;
    // schedule (stan_adaptor.jl:61-72)
    int i, n_adapts, window_start, window_end, n_splits;
    int splits[16];
    int adapt_metric, n_min;
    int finalized;
    // dense adaptor only (zero = diagonal adaptor)
    int record_len;        // doubles per rank in `gathered`; 0 = 2 + 2D
    int cand_ready;        // pooled_cov_kernel wrote a new estimate to the candidate; pooled_chol_kernel consumes it
    int chol_failed;       // the last factorisation found a pivot <= 0 or NaN
    int failed_iteration;  // first iteration whose factorisation failed (0 = never)
};

// schedule of iteration st->i + 1 (stan_adaptor.jl:137-159), shared by every kernel of one exchange
struct PooledStep {
    bool push, update, reset;
};
__device__ inline PooledStep pooled_schedule(const PooledState* st) {
    const int i = st->i + 1;
    bool split = false;
    for (int k = 0; k < st->n_splits; ++k) split |= (st->splits[k] == i);
    PooledStep s;
    s.push = st->adapt_metric && i >= st->window_start && i <= st->window_end;
    s.update = s.push && split;
    s.reset = split;
    return s;
}

// one CTA.  gathered: R records of st->record_len (default 2 + 2D) doubles in rank order.  Minv == nullptr: the estimate is
// not written (dense adaptor: pooled_cov_kernel owns M^-1).
__global__ void __launch_bounds__(256) pooled_update_kernel(PooledState* st, const double* __restrict__ gathered, int R, int D,
                                                            double* w_mu, double* w_M2, double* Minv, double* eps_chain,
                                                            long long N, double* eps_trace, double* merged_out) {
    __shared__ double s_n, s_alpha;
    __shared__ int s_push, s_update, s_reset;
    const int rec = st->record_len ? st->record_len : 2 + 2 * D;
    // ---- rank-ordered Chan merge of the R records (adaptation.py merge_records; fixed order => identical on all ranks)
    if (threadIdx.x == 0) {
        double n = gathered[0], a = gathered[1];
        for (int r = 1; r < R; ++r) {
            n += gathered[(size_t)r * rec];
            a = a + gathered[(size_t)r * rec + 1];
        }
        s_n = n;
        s_alpha = a;
        if (merged_out) {
            merged_out[0] = n;
            merged_out[1] = a;
        }
    }
    // schedule decisions of THIS iteration (stan_adaptor.jl:137-159)
    if (threadIdx.x == 0) {
        const PooledStep s = pooled_schedule(st);
        s_push = s.push;
        s_update = s.update;
        s_reset = s.reset;
    }
    __syncthreads();
    const bool push = s_push != 0, update = s_update != 0, reset = s_reset != 0;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        double n_a = gathered[0], mean = gathered[2 + d], M2 = gathered[2 + D + d];
        for (int r = 1; r < R; ++r) {
            const double* g = gathered + (size_t)r * rec;
            const double n_b = g[0], n = n_a + n_b, w = n_a * n_b / n;
            const double dl = g[2 + d] - mean;
            M2 += g[2 + D + d] + dl * dl * w;
            mean += dl * (n_b / n);
            n_a = n;
        }
        if (merged_out) {
            merged_out[2 + d] = mean;
            merged_out[2 + D + d] = M2;
        }
        if (push) {  // WelfordVar.push_record: Chan merge of the iteration's pooled record into the window's accumulator
            const double na = st->n, nb = s_n, n = na + nb;
            const double dl = mean - w_mu[d];
            double M = w_M2[d] + M2 + dl * dl * (na * nb / n);
            double mu = w_mu[d] + dl * (nb / n);
            if (Minv && update && n >= (double)st->n_min)  // get_estimation (massmatrix.jl:152-157)
                Minv[d] = n / ((n + 5.0) * (n - 1.0)) * M + 1e-3 * (5.0 / (n + 5.0));
            if (reset) {
                M = 0.0;
                mu = 0.0;
            }
            w_M2[d] = M;
            w_mu[d] = mu;
        } else if (reset) {
            w_M2[d] = 0.0;
            w_mu[d] = 0.0;
        }
    }
    __syncthreads();
    __shared__ double s_eps;
    if (threadIdx.x == 0) {
        const int i = st->i + 1;
        st->i = i;
        // NesterovDualAveraging.adapt (stepsize.jl:178-210) on the pooled mean of min(1, alpha)
        const double a = s_alpha / s_n;
        const int m = st->m + 1;
        const double eta_H = 1.0 / ((double)m + st->t0);
        const double H_bar = (1.0 - eta_H) * st->H_bar + eta_H * (st->delta - a);
        const double x = st->mu - H_bar * (sqrt((double)m) / st->gamma);
        const double eta_x = pow((double)m, -st->kappa);
        const double x_bar = (1.0 - eta_x) * st->x_bar + eta_x * x;
        const double eps = exp(x);
        if (finite_d(eps)) {  // stepsize.jl:199-203: a non-finite proposal keeps the previous state
            st->m = m;
            st->eps = eps;
            st->x_bar = x_bar;
            st->H_bar = H_bar;
        }
        if (push) st->n = reset ? 0.0 : st->n + s_n;
        else if (reset) st->n = 0.0;
        if (reset) {  // reset!(ssa) (stepsize.jl:38-44): restart dual averaging around the current step size
            st->m = 0;
            st->mu = log(10.0 * st->eps);
            st->x_bar = 0.0;
            st->H_bar = 0.0;
        }
        if (i == st->n_adapts) {  // finalize! (stepsize.jl:54-57)
            st->eps = exp(st->x_bar);
            st->finalized = 1;
        }
        s_eps = st->eps;
        if (eps_trace) eps_trace[i - 1] = st->eps;
    }
    __syncthreads();
    const double e = s_eps;
    for (long long c = threadIdx.x; c < N; c += blockDim.x) eps_chain[c] = e;
}

// Dense adaptor, step 1 of the exchange (before pooled_update_kernel).  Any grid; one thread per entry e = i + D*j of the
// column-major D x D blocks (coalesced).  gathered: R records [n, sum alpha, mean[D], M2diag[D], M2full[D*D]].
//   * rank-ordered Chan merge of the D x D blocks, the same arithmetic and order as adaptation.merge_records(.., "cov"): each
//     rank's step uses the running means BEFORE that rank is merged;
//   * WelfordCov push_record into w_M with the window's n and mean BEFORE this iteration (st->n, w_mu);
//   * at an update with n >= n_min, get_estimation (massmatrix.jl:335-340) into `cand`, and st->cand_ready = 1;
//   * at a split, w_M restarts from zero.
__global__ void __launch_bounds__(256) pooled_cov_kernel(PooledState* st, const double* __restrict__ gathered, int R, int D,
                                                         const double* __restrict__ w_mu, double* w_M, double* cand,
                                                         double* merged_out) {
    const int rec = st->record_len;
    const PooledStep s = pooled_schedule(st);
    double n_b = gathered[0];
    for (int r = 1; r < R; ++r) n_b += gathered[(size_t)r * rec];
    const double n_w = st->n, n = n_w + n_b;
    const bool update = s.update && n >= (double)st->n_min;
    if (blockIdx.x == 0 && threadIdx.x == 0) st->cand_ready = update;
    const long long DD = (long long)D * D;
    const double c = n / ((n + 5.0) * (n - 1.0)), reg = 1e-3 * (5.0 / (n + 5.0)), wt = n_w * n_b / n;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < DD; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e % D), j = (int)(e / D);
        const size_t off = 2 + 2 * (size_t)D + (size_t)e;
        double n_a = gathered[0], mi = gathered[2 + i], mj = gathered[2 + j], M = gathered[off];
        for (int r = 1; r < R; ++r) {
            const double* g = gathered + (size_t)r * rec;
            const double nb = g[0], nn = n_a + nb, w = n_a * nb / nn;
            const double di = g[2 + i] - mi, dj = g[2 + j] - mj;
            M += g[off] + di * dj * w;
            mi += di * (nb / nn);
            mj += dj * (nb / nn);
            n_a = nn;
        }
        if (merged_out) merged_out[off] = M;
        if (s.push) {
            const double di = mi - w_mu[i], dj = mj - w_mu[j];
            const double W = w_M[e] + M + di * dj * wt;
            if (update) cand[e] = c * W + (i == j ? reg : 0.0);
            w_M[e] = s.reset ? 0.0 : W;
        } else if (s.reset) {
            w_M[e] = 0.0;
        }
    }
}

// Dense adaptor, step 3 (window splits inside the metric window only; once at creation with force = 1).  One CTA, D <= 512.
// Consumes st->cand_ready.  Factorises cand = U^T U reading only its upper triangle (cholesky(Symmetric(M^-1)).U,
// metric.jl:104-108, 117) by the column Cholesky-Crout recurrence on L = U^T, kept column-major in `work` so that the
// threads (one per row) read it coalesced; every sum has a fixed order.  The pivot test is LAPACK potrf's: a pivot <= 0 or
// NaN fails.  On success cand -> Minv and U -> cholU (column-major, zero below the diagonal), both at once; on failure
// both keep their previous values and the first failing iteration is recorded.
constexpr int kCholThreads = 512;
__global__ void __launch_bounds__(kCholThreads) pooled_chol_kernel(PooledState* st, int D, const double* __restrict__ cand,
                                                                   double* work, double* Minv, double* cholU, int force) {
    __shared__ int s_go;
    __shared__ double s_piv;
    if (threadIdx.x == 0) {
        s_go = force || st->cand_ready;
        st->cand_ready = 0;
    }
    __syncthreads();
    if (!s_go) return;
    bool ok = true;
    for (int j = 0; j < D; ++j) {
        const double* Lj = work + j;  // row j of L: Lj[D * k]
        for (int i = threadIdx.x; i < D; i += blockDim.x) {
            if (i < j) continue;
            const double* Li = work + i;
            double d0 = 0.0, d1 = 0.0;
            int k = 0;
            for (; k + 1 < j; k += 2) {
                d0 = fma(Li[(size_t)D * k], Lj[(size_t)D * k], d0);
                d1 = fma(Li[(size_t)D * (k + 1)], Lj[(size_t)D * (k + 1)], d1);
            }
            if (k < j) d0 = fma(Li[(size_t)D * k], Lj[(size_t)D * k], d0);
            const double v = cand[j + (size_t)D * i] - (d0 + d1);  // A[j][i], j <= i: upper triangle
            if (i == j) s_piv = v;
            else work[i + (size_t)D * j] = v;
        }
        __syncthreads();
        const double piv = s_piv;
        if (!(piv > 0.0)) {  // the same value in every thread: the whole block leaves together
            ok = false;
            break;
        }
        const double ljj = sqrt(piv);
        for (int i = threadIdx.x; i < D; i += blockDim.x) {
            if (i < j) continue;
            work[i + (size_t)D * j] = i == j ? ljj : work[i + (size_t)D * j] / ljj;
        }
        __syncthreads();
    }
    if (ok) {
        const long long DD = (long long)D * D;
        for (long long e = threadIdx.x; e < DD; e += blockDim.x) {
            const int r = (int)(e % D), c = (int)(e / D);
            Minv[e] = cand[e];
            cholU[e] = r <= c ? work[c + (size_t)D * r] : 0.0;
        }
    }
    if (threadIdx.x == 0) {
        st->chol_failed = !ok;
        if (!ok && !force && st->failed_iteration == 0) st->failed_iteration = st->i;
    }
}

#ifndef AHMC_SIMT_EMULATION  // host launch code and the NCCL binding (skipped by the CPU SIMT emulation harness, tests/simt_emu/)
__global__ void fill_kernel(double* p, long long n, double v) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = v;
}

cudaError_t launch_pooled_update(void* state, const double* gathered, int R, int D, double* w_mu, double* w_M2, double* Minv,
                                 double* eps_chain, long long N, double* eps_trace, double* merged_out, cudaStream_t st,
                                 int* n_launches) {
    pooled_update_kernel<<<1, 256, 0, st>>>((PooledState*)state, gathered, R, D, w_mu, w_M2, Minv, eps_chain, N, eps_trace, merged_out);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}
cudaError_t launch_pooled_cov(void* state, const double* gathered, int R, int D, const double* w_mu, double* w_M, double* cand,
                              double* merged_out, cudaStream_t st, int* n_launches) {
    const long long DD = (long long)D * D;
    const unsigned blocks = (unsigned)((DD + 255) / 256 < 4096 ? (DD + 255) / 256 : 4096);
    pooled_cov_kernel<<<blocks, 256, 0, st>>>((PooledState*)state, gathered, R, D, w_mu, w_M, cand, merged_out);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}
cudaError_t launch_pooled_chol(void* state, int D, const double* cand, double* work, double* Minv, double* cholU, int force,
                               cudaStream_t st, int* n_launches) {
    const int threads = D >= kCholThreads ? kCholThreads : (D + 31) / 32 * 32;
    pooled_chol_kernel<<<1, threads, 0, st>>>((PooledState*)state, D, cand, work, Minv, cholU, force);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}
cudaError_t launch_fill(double* p, long long n, double v, cudaStream_t st) {
    fill_kernel<<<(unsigned)((n + 255) / 256 < 1024 ? (n + 255) / 256 : 1024), 256, 0, st>>>(p, n, v);
    return cudaGetLastError();
}
#endif  // AHMC_SIMT_EMULATION
size_t pooled_state_bytes() { return sizeof(PooledState); }

// host image of the state for creation / read-back
void pooled_state_init(void* host_image, double eps0, const AdaptDev& sched, double delta, double gamma, double t0, double kappa,
                       int n_adapts, int adapt_metric, int n_min) {
    PooledState s{};
    s.eps = eps0;
    s.mu = log(10.0 * eps0);  // stepsize.jl:38-44
    s.x_bar = 0.0;
    s.H_bar = 0.0;
    s.delta = delta; s.gamma = gamma; s.t0 = t0; s.kappa = kappa;
    s.m = 0;
    s.n = 0.0;
    s.i = 0;
    s.n_adapts = n_adapts;
    s.window_start = sched.window_start;
    s.window_end = sched.window_end;
    s.n_splits = sched.n_splits;
    for (int k = 0; k < sched.n_splits && k < 16; ++k) s.splits[k] = sched.splits[k];
    s.adapt_metric = adapt_metric;
    s.n_min = n_min;
    s.finalized = 0;
    memcpy(host_image, &s, sizeof s);
}
void pooled_state_set_dense(void* host_image, int record_len, int cand_ready) {
    PooledState s;
    memcpy(&s, host_image, sizeof s);
    s.record_len = record_len;
    s.cand_ready = cand_ready;
    memcpy(host_image, &s, sizeof s);
}
void pooled_state_read_dense(const void* host_image, int* failed_iteration, int* chol_failed) {
    PooledState s;
    memcpy(&s, host_image, sizeof s);
    if (failed_iteration) *failed_iteration = s.failed_iteration;
    if (chol_failed) *chol_failed = s.chol_failed;
}
// host-side schedule of the dense adaptor's factorisation: iteration i is a window split inside the metric window
bool pooled_chol_due(const AdaptDev& sched, int adapt_metric, int i) {
    if (!adapt_metric || i < sched.window_start || i > sched.window_end) return false;
    for (int k = 0; k < sched.n_splits; ++k)
        if (sched.splits[k] == i) return true;
    return false;
}
void pooled_state_read(const void* host_image, double* eps, int* iteration, int* m, double* n_window) {
    PooledState s;
    memcpy(&s, host_image, sizeof s);
    if (eps) *eps = s.eps;
    if (iteration) *iteration = s.i;
    if (m) *m = s.m;
    if (n_window) *n_window = s.n;
}

#ifndef AHMC_SIMT_EMULATION
// ---------------------------------------------------------------------------------------------- NCCL (bound at run time)
namespace {
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    char why[256] = {0};
};
NcclApi g_nccl;
bool g_nccl_tried = false;
std::mutex g_nccl_mutex;
}  // namespace

const char* nccl_bind() {  // nullptr on success, else a reason
    std::lock_guard<std::mutex> lock(g_nccl_mutex);
    if (g_nccl.lib) return nullptr;
    if (g_nccl_tried) return g_nccl.why;
    g_nccl_tried = true;
    const char* env = getenv("AHMC_NCCL_LIB");
    const char* names[] = {env, "libnccl.so.2", "libnccl.so", "/usr/lib/x86_64-linux-gnu/libnccl.so.2"};
    for (const char* n : names) {
        if (!n) continue;
        g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.lib) break;
    }
    if (!g_nccl.lib) {
        snprintf(g_nccl.why, sizeof g_nccl.why, "libnccl.so.2 not found (set AHMC_NCCL_LIB): %s", dlerror());
        return g_nccl.why;
    }
    g_nccl.GetUniqueId = (int (*)(void*))dlsym(g_nccl.lib, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(g_nccl.lib, "ncclCommInitRank");
    g_nccl.CommDestroy = (int (*)(void*))dlsym(g_nccl.lib, "ncclCommDestroy");
    g_nccl.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(g_nccl.lib, "ncclAllGather");
    g_nccl.GetErrorString = (const char* (*)(int))dlsym(g_nccl.lib, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.AllGather) {
        snprintf(g_nccl.why, sizeof g_nccl.why, "NCCL library lacks ncclGetUniqueId / ncclCommInitRank / ncclAllGather");
        g_nccl.lib = nullptr;
        return g_nccl.why;
    }
    return nullptr;
}
const char* nccl_err(int rc) { return g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "nccl error"; }
int nccl_unique_id(void* out128) { return g_nccl.GetUniqueId(out128); }
int nccl_comm_init(void** comm, int nranks, const void* id128, int rank) {
    NcclId id;
    memcpy(id.internal, id128, 128);
    return g_nccl.CommInitRank(comm, nranks, id, rank);
}
int nccl_comm_destroy(void* comm) { return g_nccl.CommDestroy(comm); }
int nccl_allgather_f64(const double* send, double* recv, size_t count, void* comm, cudaStream_t st) {
    return g_nccl.AllGather(send, recv, count, 8 /* ncclFloat64 */, comm, st);
}
#endif  // AHMC_SIMT_EMULATION

}  // namespace ahmc
