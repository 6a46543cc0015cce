// pooled_dense_emu.cpp -- the dense pooled adaptor's kernels (advancedhmc.jl_b200/csrc/ahmc_pooled.cu `pooled_cov_kernel`,
// `pooled_update_kernel`, `pooled_chol_kernel`, unmodified) under the CPU SIMT emulator, launched in the order and on the
// schedule ahmc_adapt_exchange_f64 uses for a dense adaptor: the rank-ordered D x D merge, WelfordCov, the Stan windows and
// the device Cholesky, checkable without a GPU or NCCL.  TEST INFRASTRUCTURE ONLY.
#define AHMC_SIMT_EMULATION 1
#define __shared__ static  // static shared variables only; one block at a time
#include <cstdlib>
#include <vector>

#include "ahmc_pooled.cu"

void emu_launch(void (*kernel)(const void*), const void* args, int blocks, int threads);
using namespace ahmc;

namespace {
struct CovArgs {
    PooledState* st;
    const double* gathered;
    int R, D;
    const double* w_mu;
    double *w_M, *cand, *merged;
};
void cov_thunk(const void* p) {
    const CovArgs& a = *static_cast<const CovArgs*>(p);
    pooled_cov_kernel(a.st, a.gathered, a.R, a.D, a.w_mu, a.w_M, a.cand, a.merged);
}
struct UpdArgs {
    PooledState* st;
    const double* gathered;
    int R, D;
    double *w_mu, *w_M2, *eps_chain;
    long long N;
    double* merged;
};
void upd_thunk(const void* p) {
    const UpdArgs& a = *static_cast<const UpdArgs*>(p);
    pooled_update_kernel(a.st, a.gathered, a.R, a.D, a.w_mu, a.w_M2, nullptr, a.eps_chain, a.N, nullptr, a.merged);
}
struct CholArgs {
    PooledState* st;
    int D;
    const double* cand;
    double *work, *Minv, *cholU;
    int force;
};
void chol_thunk(const void* p) {
    const CholArgs& a = *static_cast<const CholArgs*>(p);
    pooled_chol_kernel(a.st, a.D, a.cand, a.work, a.Minv, a.cholU, a.force);
}

// emulated grids are small (every CUDA thread is a host thread): the kernels' grid-stride loops cover the rest
constexpr int kCovBlocks = 3, kThreads = 64;

struct EmuDense {
    std::vector<char> state;
    std::vector<double> w_mu, w_M2, w_M, cand, work, Minv, cholU, eps_chain, merged;
    AdaptDev sched{};
    int D = 0, adapt_metric = 0, calls = 0;
    long long N = 0;
    PooledState* st() { return reinterpret_cast<PooledState*>(state.data()); }
};
void chol(EmuDense* e, int force) {
    CholArgs a{e->st(), e->D, e->cand.data(), e->work.data(), e->Minv.data(), e->cholU.data(), force};
    emu_launch(chol_thunk, &a, 1, kThreads);
}
}  // namespace

// Minv0: D x D column-major (NULL = I).  Returns NULL if the schedule is unsupported or Minv0's factorisation fails.
extern "C" void* emu_pd_create(int D, long long N, int n_adapts, int init_buffer, int term_buffer, int window_size, double eps0,
                               double delta, int adapt_metric, int n_min, const double* Minv0) {
    AdaptDev sched{};
    if (!stan_window_schedule(sched, init_buffer, term_buffer, window_size, n_adapts)) return nullptr;
    EmuDense* e = new EmuDense;
    const size_t DD = (size_t)D * D;
    e->D = D;
    e->N = N;
    e->sched = sched;
    e->adapt_metric = adapt_metric;
    e->state.resize(pooled_state_bytes());
    pooled_state_init(e->state.data(), eps0, sched, delta, 0.05, 10.0, 0.75, n_adapts, adapt_metric, n_min);
    pooled_state_set_dense(e->state.data(), 2 + 2 * D + (adapt_metric ? D * D : 0), 0);
    e->w_mu.assign(D, 0.0);
    e->w_M2.assign(D, 0.0);
    e->w_M.assign(DD, 0.0);
    e->work.assign(DD, 0.0);
    e->Minv.assign(DD, 0.0);
    e->cholU.assign(DD, 0.0);
    e->cand.assign(DD, 0.0);
    for (size_t k = 0; k < DD; ++k) e->cand[k] = Minv0 ? Minv0[k] : (k % (D + 1) == 0 ? 1.0 : 0.0);
    e->eps_chain.assign(N, eps0);
    e->merged.assign(2 + 2 * D + DD, 0.0);
    chol(e, 1);
    int failed = 0;
    pooled_state_read_dense(e->state.data(), nullptr, &failed);
    if (failed) {
        delete e;
        return nullptr;
    }
    return e;
}

// one exchange: `gathered` = R records of (2 + 2D + D*D) doubles (2 + 2D with adapt_metric = 0) in rank order.
// Outputs: eps, Minv / cholU (column-major), the merged record (2 + 2D + D*D), the failed iteration.  Returns the
// iteration, or -1 if eps_chain is not uniformly eps.
extern "C" int emu_pd_update(void* h, const double* gathered, int R, double* eps_out, double* minv_out, double* cholu_out,
                             double* merged_out, int* failed_out) {
    EmuDense* e = static_cast<EmuDense*>(h);
    const int D = e->D;
    if (e->adapt_metric) {
        CovArgs c{e->st(), gathered, R, D, e->w_mu.data(), e->w_M.data(), e->cand.data(), e->merged.data()};
        emu_launch(cov_thunk, &c, kCovBlocks, kThreads);
    }
    UpdArgs u{e->st(), gathered, R, D, e->w_mu.data(), e->w_M2.data(), e->eps_chain.data(), e->N, e->merged.data()};
    emu_launch(upd_thunk, &u, 1, 256);
    e->calls += 1;
    if (e->adapt_metric && pooled_chol_due(e->sched, e->adapt_metric, e->calls)) chol(e, 0);
    int it = 0;
    pooled_state_read(e->state.data(), eps_out, &it, nullptr, nullptr);
    pooled_state_read_dense(e->state.data(), failed_out, nullptr);
    for (size_t k = 0; k < (size_t)D * D; ++k) {
        minv_out[k] = e->Minv[k];
        cholu_out[k] = e->cholU[k];
    }
    for (size_t k = 0; k < e->merged.size(); ++k) merged_out[k] = e->merged[k];
    for (long long c = 0; c < e->N; ++c)
        if (e->eps_chain[c] != *eps_out) return -1;
    return it;
}
extern "C" void emu_pd_destroy(void* h) { delete static_cast<EmuDense*>(h); }

// the factorisation alone, as at a window split of iteration `iteration`: A (column-major, only its upper triangle is
// read) is the candidate; Minv / cholU hold the committed values and are replaced only on success.  Returns the failed
// iteration (0 = success).
extern "C" int emu_pd_chol(int D, const double* A, double* Minv, double* cholU, int iteration) {
    EmuDense e;
    e.D = D;
    e.state.assign(pooled_state_bytes(), 0);
    AdaptDev sched{};
    pooled_state_init(e.state.data(), 0.1, sched, 0.8, 0.05, 10.0, 0.75, 0, 1, 1);
    pooled_state_set_dense(e.state.data(), 2 + 2 * D + D * D, 1);
    e.st()->i = iteration;
    e.cand.assign(A, A + (size_t)D * D);
    e.work.assign((size_t)D * D, -7.0);
    e.Minv.assign(Minv, Minv + (size_t)D * D);
    e.cholU.assign(cholU, cholU + (size_t)D * D);
    chol(&e, 0);
    std::copy(e.Minv.begin(), e.Minv.end(), Minv);
    std::copy(e.cholU.begin(), e.cholU.end(), cholU);
    int failed = 0;
    pooled_state_read_dense(e.state.data(), &failed, nullptr);
    return failed;
}

#ifdef RACE_MAIN  // ThreadSanitizer build: the three kernels over a few exchanges, one of them a window split
#include <cstdio>
int main() {
    const int D = 13, R = 2, n_adapts = 12;
    const int rec = 2 + 2 * D + D * D;
    void* h = emu_pd_create(D, 8, n_adapts, 1, 1, 2, 0.2, 0.8, 1, 3, nullptr);  // window split at 3
    if (!h) return 1;
    std::vector<double> g((size_t)R * rec), minv((size_t)D * D), U((size_t)D * D), merged(rec);
    unsigned s = 12345u;
    auto u01 = [&] { s = s * 1664525u + 1013904223u; return (s >> 8) * (1.0 / 16777216.0); };
    int rc = 0;
    for (int i = 1; i <= 6; ++i) {
        for (int r = 0; r < R; ++r) {
            double* x = g.data() + (size_t)r * rec;
            x[0] = 5 + r;
            x[1] = 2.5;
            for (int d = 0; d < D; ++d) x[2 + d] = u01() - 0.5;
            for (int a = 0; a < D; ++a)
                for (int b = 0; b <= a; ++b) {
                    const double v = (a == b) ? 3.0 + u01() : 0.1 * (u01() - 0.5);
                    x[2 + 2 * D + a + D * b] = x[2 + 2 * D + b + D * a] = v;
                }
            for (int d = 0; d < D; ++d) x[2 + D + d] = x[2 + 2 * D + d * (D + 1)];
        }
        double eps = 0.0;
        int failed = 0;
        const int it = emu_pd_update(h, g.data(), R, &eps, minv.data(), U.data(), merged.data(), &failed);
        printf("rc %d\n", it == i ? 0 : 1);
        rc |= it != i;
    }
    emu_pd_destroy(h);
    return rc;
}
#endif
