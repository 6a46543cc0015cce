// ahmc_kernels.cuh -- kernel argument blocks + launch dispatch declarations (host side sees only these).
#pragma once
#include "ahmc_device.cuh"

namespace ahmc {

struct LeapfrogArgs {
    ModelDev model;
    MetricDev metric;
    int D;
    long long N;
    double eps;               // scalar step size (used when eps_chain == nullptr), sign applied by `fwd`
    const double* eps_chain;  // per-chain step sizes or nullptr
    int n_steps;              // >= 1 (absolute)
    int fwd;                  // 1: forward, 0: backward (integrator.jl:221-226)
    double temper_alpha;      // <= 0: none
    const double *th_in, *r_in, *g_in, *lp_in, *lk_in;
    long long ld_in;
    double *th_out, *r_out, *g_out, *lp_out, *lk_out, *dr_out;
    long long ld_out;
    uint32_t* status;
    int32_t* steps_done;
    int* min_break;  // device int: atomicMin of the first non-finite step over all chains (COMPAT_BREAK_ALL)
    uint32_t flags;
    const uint8_t* only_mask;  // nullable: process only chains whose mask byte is non-zero (K4 exact fallback)
    int resident_blocks_per_sm;  // 0 = as many as fit; > 0 caps residency (the launch pads the dynamic shared memory)
};

struct PhasepointArgs {
    ModelDev model;
    MetricDev metric;
    int D;
    long long N;
    const double *th, *r;
    double *lp, *g, *lk, *dr;
    long long ld;
};

struct MomentumArgs {
    MetricDev metric;
    int D;
    long long N;
    uint64_t seed, offset;
    const double* normal_tape;  // D x N contiguous (ld = D) or nullptr
    double* r;
    long long ld;
};

// find_good_stepsize for every chain in ONE launch (trajectory.jl:753-837)
struct FindEpsArgs {
    ModelDev model;
    MetricDev metric;
    int D;
    long long N;
    const double *th, *g, *lp;  // positions and the cached (lp, -grad) of phasepoint
    long long ld;
    uint64_t seed, offset;
    const double* normal_tape;  // D x N standard normals or nullptr (Philox)
    double eps0;
    int max_iters;
    double* eps_out;            // N
    double* r_out;              // nullable, D x N (ld): the momentum each search used
};

struct StatsDev {
    int32_t* n_steps;
    uint8_t* is_accept;
    double* acceptance_rate;
    double* log_density;
    double* hamiltonian_energy;
    double* hamiltonian_energy_error;
    double* max_hamiltonian_energy_error;
    int32_t* tree_depth;
    uint8_t* numerical_error;
};

struct RngDev {
    uint64_t seed, offset;
    const double* normal_tape;
    const double* exp_tape;
    long long exp_stride;
    const uint8_t* dir_tape;
    long long dir_stride;
    double partial_alpha;  // 0: full refresh; else r' = alpha r + sqrt(1-alpha^2) xi (hamiltonian.jl:243-254)
    double temper_alpha;   // > 0: the transition integrates with TemperedLeapfrog(eps, alpha) (integrator.jl:174-209)
};

struct HmcArgs {
    LeapfrogArgs lf;  // th_in/r_in/g_in/lp_in = current phase point; outputs = new phase point
    RngDev rng;
    StatsDev st;          // arrays of n_transitions x N entries (transition-major)
    int refresh;          // 1: draw new momentum
    int n_transitions;    // >= 1: persistent sampling loop inside the kernel (sampler.jl:182 `for i in 1:n_samples`)
    double* draws;        // nullable: n_transitions x (D x N) positions, draw t of chain c at (t*N + c)*D
};

// in-kernel per-chain adaptation (K3 adaptive family): NesterovDualAveraging + windowed WelfordVar per chain
struct AdaptDev {
    int enabled;
    int n_adapts;                  // iterations 1..n_adapts adapt (sampler.jl:72-90)
    int window_start, window_end;  // stan_adaptor.jl:13-50
    int n_splits;
    int splits[12];
    double delta, gamma, t0, kappa;  // stepsize.jl:162-172
    int adapt_metric;                // 0: step size only
    int n_min;                       // massmatrix.jl:103-107
    double* eps;                     // N, out: adapted step size per chain (in: a.eps_chain / a.eps)
    double* minv;                    // N*D, out: adapted diagonal M^-1 per chain (nullable when !adapt_metric)
    double* eps_trace;               // nullable, n_transitions x N: step size used by each transition
};
// initialize!(StanHMCAdaptorState, init_buffer, term_buffer, window_size, n_adapts) (stan_adaptor.jl:13-50): the
// host side of the in-launch adaptation.  false: the schedule needs more window splits than AdaptDev holds.
inline bool stan_window_schedule(AdaptDev& ad, int init_buffer, int term_buffer, int window_size, int n_adapts) {
    constexpr int kMaxSplits = (int)(sizeof(ad.splits) / sizeof(ad.splits[0]));
    ad.window_start = init_buffer + 1;
    ad.window_end = n_adapts - term_buffer;
    ad.n_splits = 0;
    long long wsz = window_size, next = (long long)init_buffer + wsz;
    while (next <= ad.window_end) {
        if (next + 2 * wsz > ad.window_end) next = ad.window_end;  // the last window runs to the end of the slow phase
        if (ad.n_splits == kMaxSplits) return false;
        ad.splits[ad.n_splits++] = (int)next;
        wsz *= 2;
        next += wsz;
    }
    if (ad.n_splits > 0 && ad.splits[ad.n_splits - 1] == n_adapts) --ad.n_splits;  // "avoid updating in the end"
    return true;
}

struct NutsArgs {
    ModelDev model;
    MetricDev metric;
    int D;
    long long N;
    double eps;
    const double* eps_chain;
    int max_depth;
    double delta_max;
    int sampler;    // 0 MultinomialTS, 1 SliceTS
    int criterion;  // 0 GeneralisedNoUTurn, 1 ClassicNoUTurn, 2 StrictGeneralisedNoUTurn
    AdaptDev ad;
    RngDev rng;
    int refresh;
    const double *th_in, *r_in, *g_in, *lp_in;
    long long ld_in;
    double *th_out, *r_out, *g_out, *lp_out, *lk_out, *dr_out;
    long long ld_out;
    StatsDev st;              // arrays of n_transitions x N entries
    int n_transitions;
    double* draws;            // nullable: n_transitions x (D x N)
    double* scratch;          // per-chain tree workspace (see ahmc_nuts.cu)
    long long scratch_stride; // doubles per chain
};

// split-step mode (user gradient callback between the two half kicks): one leapfrog step = kick_drift kernel,
// the user's lp/grad evaluation on the same stream, kick_energy kernel.  State lives in the OUTPUT phase point.
struct SplitArgs {
    MetricDev metric;
    int D;
    long long N;
    double eps;
    const double* eps_chain;
    int fwd;
    double mul;                 // tempering multiplier for this half (1.0: none)
    int step_index;             // 1-based step number (kick_energy records it in steps_done)
    int no_kick;                // 1: phasepoint mode -- leave r alone, ignore status, only (g, lp, lk, dr)
    double *th, *r, *g;         // work state (D x N, ld)
    double *lp, *lk, *dr;       // energies (N) and optional dH/dr
    const double* cb_lp;        // callback outputs: lp[N], grad[D x N] (PLUS gradient)
    const double* cb_grad;
    long long ld;
    uint32_t* status;           // per-chain: non-zero = frozen (already non-finite)
    int32_t* steps_done;
    int* any_nonfinite;         // device flag, set when a chain turns non-finite in this step
};

struct MhArgs {  // accept / revert / flip + stats after a split-mode trajectory (trajectory.jl:271-300)
    int D;
    long long N;
    int n_steps;
    const double *th0, *g0, *lp0;  // start point (ld0)
    long long ld0;
    const double *r0, *lk0;        // refreshed momentum (ld = D) and its kinetic energy
    double *th, *r, *g, *lp, *lk;  // in: proposal; out: new phase point (ld)
    long long ld;
    RngDev rng;
    StatsDev st;
};

struct TrajArgs {  // step(...; full_trajectory = Val(true)) (integrator.jl:229,249-261)
    ModelDev model;
    MetricDev metric;
    int D;
    long long N;
    double eps;
    const double* eps_chain;
    int n_steps;  // absolute
    int fwd;
    double temper_alpha;
    const double *th_in, *r_in, *g_in;
    long long ld_in;
    double *th_out, *r_out, *g_out, *dr_out;  // point i (0-based) at i*step_stride + ld_out*chain
    double *lp_out, *lk_out;                   // point i at i*N + chain
    long long ld_out, step_stride;
    int32_t* steps_done;
};

struct MultinomialArgs {  // static transition with MultinomialTS (trajectory.jl:344-390)
    ModelDev model;
    MetricDev metric;
    int D;
    long long N;
    double eps;
    const double* eps_chain;
    int n_steps, n_fwd;
    int refresh;
    RngDev rng;  // exp_tape doubles as the per-chain UNIFORM tape of `randcat`
    const double *th_in, *r_in, *g_in, *lp_in;
    long long ld_in;
    double *th_out, *r_out, *g_out, *lp_out, *lk_out;
    long long ld_out;
    StatsDev st;
    double* energies;  // (n_steps + 1) doubles per chain
};

// K4 (ahmc_dense.cu): tiled DMMA trajectory for dense metric / dense-Gaussian target
struct DenseTrajHost {
    int D, Dp;
    long long N;
    const double* P;      // padded Dp x Dp precision or nullptr
    const double* w;      // 1/s^2 (DIAG_GAUSS) or nullptr
    const double* mu;
    double c0;
    const double* Minv;   // padded Dp x Dp or nullptr
    const double* Mdiag;  // D or nullptr
    const double* norms;  // device: [|Minv|_inf, |P|_inf]
    double eps;
    const double* eps_chain;
    int n_steps, fwd;
    const double *th_in, *r_in, *g_in;
    long long ld_in;
    double *th_out, *r_out, *g_out, *dr_out, *lp_out, *lk_out;
    long long ld_out;
    uint32_t* status;
    int32_t* steps_done;
    uint8_t* need_exact;
};
bool dense_tile_shape(int D, int* Dp, int* RB, int* CB);
// padded matrices (K4) are stored with the shared-memory stage's leading dimension: a 16-column chunk is one bulk copy
__host__ __device__ constexpr int dense_lda(int Dp) { return Dp + 4; }
__host__ __device__ constexpr size_t dense_mat_doubles(int Dp) { return (size_t)Dp * (size_t)dense_lda(Dp); }
#ifndef __CUDACC_RTC__
cudaError_t launch_dense_traj(const DenseTrajHost& h, cudaStream_t stream, int* n_launches);
cudaError_t launch_pad_norm(const double* A, int D, int Dp, double* Ap, double* norm, cudaStream_t st);
cudaError_t launch_vec_norm(const double* v, int D, double* norm, cudaStream_t st);
#endif

// choose (G, E) for a dimension: returns false if D is out of the register-resident range
bool pick_layout(int D, int* G, int* E);

#ifndef __CUDACC_RTC__  // host-side declarations (cudaError_t / cudaStream_t are unknown to NVRTC)
// launchers (defined in the .cu files); all enqueue on `stream` and return the cudaError_t of the launch
cudaError_t launch_leapfrog(const LeapfrogArgs& a, cudaStream_t stream, int* n_launches);
cudaError_t launch_phasepoint(const PhasepointArgs& a, cudaStream_t stream, int* n_launches);
cudaError_t launch_rand_momentum(const MomentumArgs& a, cudaStream_t stream, int* n_launches);
cudaError_t launch_hmc(const HmcArgs& a, cudaStream_t stream, int* n_launches);
cudaError_t launch_find_eps(const FindEpsArgs& a, cudaStream_t stream, int* n_launches);
// A (D x D column-major) -> out with leading dimension coop_lds(D), zero filled (the cooperative NUTS products fetch whole
// chunks of such columns with one bulk copy); coop_padded_doubles(D) doubles
size_t coop_padded_doubles(int D);
cudaError_t launch_pad_columns(const double* A, int D, double* out, cudaStream_t st);
// D > 512: streaming form of step / phasepoint (ahmc_bigd.cu)
bool bigd_supported(int model_kind, int metric_kind);
cudaError_t launch_leapfrog_big(const LeapfrogArgs& a, cudaStream_t st);
cudaError_t launch_phasepoint_big(const PhasepointArgs& a, cudaStream_t st);
cudaError_t launch_nuts(const NutsArgs& a, cudaStream_t stream, int* n_launches);
long long nuts_scratch_doubles_per_chain(int D, int max_depth, bool adaptive);
cudaError_t launch_trajectory(const TrajArgs& a, cudaStream_t stream, int* n_launches);
cudaError_t launch_multinomial(const MultinomialArgs& a, cudaStream_t stream, int* n_launches);
cudaError_t launch_kick_drift(const SplitArgs& a, cudaStream_t stream, int* n_launches);
cudaError_t launch_kick_energy(const SplitArgs& a, cudaStream_t stream, int* n_launches);
cudaError_t launch_mh_select(const MhArgs& a, cudaStream_t stream, int* n_launches);
cudaError_t launch_adapt_summary(int D, long long N, const double* theta, long long ld, const double* alpha,
                                 double* out, double* partial, unsigned* counter, int blocks, cudaStream_t st,
                                 int* n_launches);
cudaError_t launch_adapt_cov(int D, long long N, const double* theta, long long ld, const double* mean, double* out,
                             cudaStream_t st, int* n_launches);

// pooled adaptation on the device + NCCL bound at run time (ahmc_pooled.cu)
struct NcclId {
    char internal[128];
};
cudaError_t launch_pooled_update(void* state, const double* gathered, int R, int D, double* w_mu, double* w_M2, double* Minv,
                                 double* eps_chain, long long N, double* eps_trace, double* merged_out, cudaStream_t st,
                                 int* n_launches);
cudaError_t launch_pooled_cov(void* state, const double* gathered, int R, int D, const double* w_mu, double* w_M, double* cand,
                              double* merged_out, cudaStream_t st, int* n_launches);
cudaError_t launch_pooled_chol(void* state, int D, const double* cand, double* work, double* Minv, double* cholU, int force,
                               cudaStream_t st, int* n_launches);
cudaError_t launch_fill(double* p, long long n, double v, cudaStream_t st);
size_t pooled_state_bytes();
void pooled_state_set_dense(void* host_image, int record_len, int cand_ready);
void pooled_state_read_dense(const void* host_image, int* failed_iteration, int* chol_failed);
bool pooled_chol_due(const AdaptDev& sched, int adapt_metric, int i);
void pooled_state_init(void* host_image, double eps0, const AdaptDev& sched, double delta, double gamma, double t0, double kappa,
                       int n_adapts, int adapt_metric, int n_min);
void pooled_state_read(const void* host_image, double* eps, int* iteration, int* m, double* n_window);
const char* nccl_bind();
const char* nccl_err(int rc);
int nccl_unique_id(void* out128);
int nccl_comm_init(void** comm, int nranks, const void* id128, int rank);
int nccl_comm_destroy(void* comm);
int nccl_allgather_f64(const double* send, double* recv, size_t count, void* comm, cudaStream_t st);

// user targets compiled at run time (ahmc_user.cu): NVRTC + the driver API, both bound with dlopen
enum UserKernel { UK_PHASEPOINT = 0, UK_LEAPFROG = 1, UK_HMC = 2, UK_NUTS = 3, UK_FIND_EPS = 4 };
struct UserModule;  // per-model cache of compiled kernels
UserModule* user_module_create(const char* cuda_src, char* err, size_t err_len);
void user_module_destroy(UserModule* m);
// compile (first use) and launch kernel `which` of the user module for (metric, G, E); args = the kernel's argument block
cudaError_t user_launch(UserModule* m, int which, int metric_kind, int G, int E, const void* args, unsigned blocks, size_t smem,
                        cudaStream_t st);
const char* user_last_error(const UserModule* m);
int user_source_check(const char* cuda_src, int which, int metric_kind, int D, char* log, size_t log_len);
const char* user_thread_error();  // message of the last failed user_launch on this thread ("" if none)
void user_thread_error_clear();

#endif  // __CUDACC_RTC__

constexpr int kBlockThreads = 128;

// dynamic shared memory needed by the dense paths: one D-double slab per group
inline size_t smem_bytes(int model_kind, int metric_kind, int D, int G) {
    bool dense = (model_kind == AHMC_MODEL_DENSE_GAUSS) || (metric_kind == AHMC_METRIC_DENSE) || (model_kind == AHMC_MODEL_USER);
    return dense ? (size_t)(kBlockThreads / G) * (size_t)(model_kind == AHMC_MODEL_USER ? 2 : 1) * (size_t)D * sizeof(double) : 0;
}

}  // namespace ahmc
