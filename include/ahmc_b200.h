/*
 * ahmc_b200.h -- C ABI of libahmc_b200: the B200-native (sm_100a) many-chain leapfrog / HMC / NUTS
 * engine that slots under AdvancedHMC.jl's `AbstractIntegrator` / `Hamiltonian` / `AbstractMetric`
 * plugin surface (see INTEGRATION.md for the Julia `ccall` shim that binds every entry point).
 *
 * Conventions
 *  - All entry points are `extern "C"`, return an `int` status (AHMC_OK or a negative AHMC_ERR_*),
 *    never throw; the message of the last failure is `ahmc_last_error(ctx)`.  Numerical trouble is
 *    DATA, never an error: non-finite energies are mapped to -Inf exactly like the PhasePoint
 *    constructor (src/hamiltonian.jl:95-104) and reported in per-chain status/statistics.
 *  - Arrays are Julia column-major D x N: element (d, chain c) at `d + ld*c` (each chain contiguous).
 *    Unless AHMC_FLAG_HOST_BUFFERS is passed every array pointer is a DEVICE pointer (e.g. the
 *    `pointer(::CuArray)` of the reference's CUDA extension, ext/AdvancedHMCCUDAExt.jl).
 *    With AHMC_FLAG_HOST_BUFFERS they are host pointers; the library stages them through pinned
 *    memory on the context stream (host->device, kernels, device->host inside the call).
 *  - The caller owns every buffer; the library neither frees nor retains pointers past the call
 *    (model / metric parameter arrays are copied at creation).  Outputs may alias inputs
 *    (z_out == z_in works: every element is read and written by the same thread).
 *  - A context is bound to one device and one stream and is not thread-safe; calls synchronise the
 *    stream before returning unless AHMC_FLAG_ASYNC is passed.
 *  - `lp_gradient` holds MINUS grad log pi, which is what PhasePoint.lp.gradient caches in the
 *    reference (`dH/dtheta` returns DualValue(lp, -grad), src/hamiltonian.jl:45-48).
 *
 * All `file:line` citations are relative to the reference checkout (AdvancedHMC.jl v0.8.6).
 */
#ifndef AHMC_B200_H
#define AHMC_B200_H

#ifndef __CUDACC_RTC__ /* (the header is also seen by NVRTC when user-target kernels are compiled at run time) */
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define AHMC_OK 0
#define AHMC_ERR_INVALID (-1)     /* bad argument: the ArgumentError / @argcheck analogue (hamiltonian.jl:55-57,94) */
#define AHMC_ERR_CUDA (-2)        /* CUDA runtime failure */
#define AHMC_ERR_UNSUPPORTED (-3) /* valid request this build has no kernel for */
#define AHMC_ERR_NOMEM (-4)
#define AHMC_ERR_CALLBACK (-5)    /* user gradient callback returned non-zero */

/* metric kinds -- src/metric.jl:17-35 (Unit), :52-72 (Diag), :89-120 (Dense) */
#define AHMC_METRIC_UNIT 0
#define AHMC_METRIC_DIAG 1
#define AHMC_METRIC_DENSE 2

/* built-in log-density models (the `lp` / `dlp/dtheta` closures of `Hamiltonian`, src/hamiltonian.jl:1-6) */
#define AHMC_MODEL_STD_NORMAL 0  /* lp = c0 - sum(th^2)/2 */
#define AHMC_MODEL_DIAG_GAUSS 1  /* p0 = mean[D], p1 = std[D]; lp = c0 - sum(((th-m)/s)^2)/2 (test/common.jl:35-77) */
#define AHMC_MODEL_DENSE_GAUSS 2 /* p0 = mean[D], p1 = precision[DxD] col-major; lp = c0 - (th-mu)'P(th-mu)/2 */
#define AHMC_MODEL_FUNNEL 3      /* Neal's funnel: v=th[0]; lp = c0 - v^2/18 - sum_{i>=1}(th_i^2 e^{-v} + v)/2 */
#define AHMC_MODEL_CALLBACK 4    /* user-supplied gradient callback (split-step mode) */
#define AHMC_MODEL_USER 5        /* user-supplied CUDA device function, compiled at run time INTO the fused kernels */

/* flags */
#define AHMC_FLAG_HOST_BUFFERS 0x1u    /* array arguments are host pointers (staged by the library) */
#define AHMC_FLAG_COMPAT_BREAK_ALL 0x2u /* mirror the reference's matrix-mode quirk: the first non-finite chain
                                           stops ALL chains at that step (hamiltonian.jl:141-142 + integrator.jl:252-258).
                                           Default: each chain stops on its own. */
#define AHMC_FLAG_ASYNC 0x4u           /* do not synchronise the context stream before returning */
#define AHMC_FLAG_EXACT_CHECKS 0x8u    /* force the per-step energy/finiteness path (disables the fused fast path) */
#define AHMC_FLAG_NO_REFRESH 0x10u     /* transitions: keep z_in.r instead of drawing a new momentum */
/* NUTS variants (ahmc_nuts_transition_f64 / ahmc_nuts_sample_f64 only; default = MultinomialTS + GeneralisedNoUTurn) */
#define AHMC_FLAG_NUTS_SLICE_TS 0x20u  /* `SliceTS` trajectory sampler (src/trajectory.jl:102-109, 144-189, 202) */
#define AHMC_FLAG_NUTS_CLASSIC 0x40u   /* `ClassicNoUTurn` criterion (src/trajectory.jl:551-557) */
#define AHMC_FLAG_NUTS_STRICT 0x80u    /* `StrictGeneralisedNoUTurn` criterion (src/trajectory.jl:579-613) */

/* per-chain status bits */
#define AHMC_STATUS_NONFINITE 0x1u /* !isfinite(z) hit (integrator.jl:252-258) */

typedef struct ahmc_ctx ahmc_ctx;
typedef struct ahmc_model ahmc_model;

/* Metric descriptor.  `Minv`: Diag -> D entries (chain_stride 0) or D x N per-chain (chain_stride = D,
 * metric.jl:64); Dense -> D x D column-major.  `cholU`: Dense only, upper factor of cholesky(Minv)
 * (metric.jl:104-109), needed by ahmc_rand_momentum_f64 and the transition kernels.  Device pointers
 * (host pointers with AHMC_FLAG_HOST_BUFFERS). */
typedef struct ahmc_metric {
    int32_t kind;
    const double* Minv;
    int64_t chain_stride;
    const double* cholU;
} ahmc_metric;

/* PhasePoint (src/hamiltonian.jl:88-107) as a struct of arrays. */
typedef struct ahmc_phasepoint {
    double* theta;       /* D x N */
    double* r;           /* D x N */
    double* lp_value;    /* N   : log pi(theta)              (PhasePoint.lp.value)    */
    double* lp_gradient; /* D x N: MINUS grad log pi(theta)  (PhasePoint.lp.gradient) */
    double* lk_value;    /* N   : minus kinetic energy       (PhasePoint.lk.value)    */
    double* lk_gradient; /* D x N or NULL: dH/dr             (PhasePoint.lk.gradient) */
    int64_t ld;          /* leading dimension, >= D */
} ahmc_phasepoint;

/* Per-chain transition statistics = the `stat` NamedTuple of src/trajectory.jl:286-298 (static) and
 * :726-739 (NUTS).  Any pointer may be NULL. */
typedef struct ahmc_stats {
    int32_t* n_steps;
    uint8_t* is_accept;
    double* acceptance_rate;
    double* log_density;
    double* hamiltonian_energy;
    double* hamiltonian_energy_error;
    double* max_hamiltonian_energy_error; /* NUTS only */
    int32_t* tree_depth;                  /* NUTS only */
    uint8_t* numerical_error;
} ahmc_stats;

/* Random inputs of one transition.  Tapes (device pointers, or host with HOST_BUFFERS) make a
 * transition a pure function, which is how parity with the CPU oracle is defined (the reference's
 * MersenneTwister/Xoshiro streams are not reproducible off-Julia, SURVEY 8c).  Where a tape is NULL
 * the value comes from the built-in counter-based Philox4x32-10 generator keyed by (seed, chain, draw). */
typedef struct ahmc_rng {
    uint64_t seed;
    uint64_t offset;           /* transition counter: advance by 1 per transition call */
    const double* normal_tape; /* D x N standard normals for rand_momentum (metric.jl:290-320) */
    const double* exp_tape;    /* static: N; NUTS: exp_stride x N, consumed in the reference's order */
    int64_t exp_stride;
    const uint8_t* dir_tape;   /* NUTS: dir_stride x N direction bits (`rand(rng,Bool)`, trajectory.jl:693) */
    int64_t dir_stride;
    double partial_refresh_alpha; /* 0: FullMomentumRefreshment; else PartialMomentumRefreshment(alpha):
                                     r' = alpha*r + sqrt(1-alpha^2)*rand_momentum (hamiltonian.jl:222-254) */
    double temper_alpha;          /* 0: the transition integrates with Leapfrog; > 0: with TemperedLeapfrog(eps, alpha)
                                     (integrator.jl:174-209) -- every `step` the reference's transition makes tempers by its own
                                     n_steps: the static trajectory, each leg of the multinomial one, each NUTS leaf (n = 1) */
} ahmc_rng;

/* User gradient callback for AHMC_MODEL_CALLBACK (replaces the Julia closure h.dlp/dth, hamiltonian.jl:45-48).
 * Must enqueue, on `stream`, work that fills lp[N] and grad[D x N] (PLUS gradient of log pi, column-major,
 * leading dimension ld) from theta (device pointers).  Return 0 on success. */
typedef int (*ahmc_logp_grad_fn)(void* user, const double* theta, double* lp, double* grad, int32_t D, int64_t N,
                                 int64_t ld, void* stream);

/* ---- context --------------------------------------------------------------------------------- */
const char* ahmc_version(void);
int ahmc_create(ahmc_ctx** out, int32_t device, void* cuda_stream /* cudaStream_t or NULL = new stream */);
int ahmc_destroy(ahmc_ctx* ctx);
const char* ahmc_last_error(const ahmc_ctx* ctx);
int ahmc_synchronize(ahmc_ctx* ctx);
/* the cudaStream_t every call of this context enqueues on (the one given to ahmc_create, or the context's own).  A host
 * that passes AHMC_FLAG_ASYNC must order its own work -- and the lifetime of the buffers it hands over -- on this stream. */
void* ahmc_stream(const ahmc_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches evidence) */
int64_t ahmc_launch_count(const ahmc_ctx* ctx);
/* how the last AHMC_FLAG_HOST_BUFFERS call of ahmc_leapfrog_f64 moved its buffers, e.g. "up=direct down=direct chunks=1
 * occ=1 (autotuned)": page-locked buffers are moved by whichever of {kernel loads/stores of host memory, copy-engine
 * pipelines of 2 / 4 chunks} measured fastest on the first calls of that shape (results are bit-identical in every mode) */
const char* ahmc_last_transport(const ahmc_ctx* ctx);

/* ---- models ---------------------------------------------------------------------------------- */
/* p0/p1 are HOST pointers (copied to the device at creation); meaning per AHMC_MODEL_*. */
int ahmc_model_create(ahmc_ctx* ctx, int32_t kind, int32_t D, const double* p0, const double* p1, double c0,
                      ahmc_model** out);
int ahmc_model_create_callback(ahmc_ctx* ctx, int32_t D, ahmc_logp_grad_fn fn, void* user, ahmc_model** out);
/* A user-supplied log pi / grad log pi FUSED into the kernels (the `h.dlp/dtheta` closure of src/hamiltonian.jl:45-48 as a CUDA
 * device function): `cuda_src` is CUDA C++ source that defines ONE of
 *     __device__ double ahmc_user_logp_grad(const double* theta, double* grad, int D, const double* params);
 *         log pi of one chain; writes the PLUS gradient into grad[0..D) (theta / grad: D-vectors in shared memory)
 *     #define AHMC_USER_COORDWISE
 *     __device__ double ahmc_user_coord(int d, double theta_d, const double* params, double* grad_d);
 *         for targets that are a sum over coordinates: term d and its derivative (every lane evaluates its own coordinates)
 * It is compiled at run time (NVRTC, sm_100a) together with the library's own kernel sources on first use of each kernel, so
 * phasepoint, the fused trajectory, the static HMC transition, NUTS (MultinomialTS + GeneralisedNoUTurn) and
 * find_good_stepsize run on it exactly as on a built-in target: no host round trip per step.  params[n_params] (host) is
 * copied to the device and handed to the function; lp = c0 + the function's value.  Compilation errors come back through
 * ahmc_last_error of the first call that needs the kernel.  Needs libnvrtc + the driver library at run time (dlopen). */
int ahmc_model_create_user(ahmc_ctx* ctx, int32_t D, const char* cuda_src, const double* params, int32_t n_params, double c0,
                           ahmc_model** out);
/* Compile-only check of a user target (no device, no context needed): kernel 0 phasepoint, 1 trajectory, 2 static HMC,
 * 3 NUTS, 4 find_good_stepsize; the layout follows from D.  AHMC_OK, or AHMC_ERR_INVALID with the NVRTC log in `log`. */
int ahmc_user_source_check(const char* cuda_src, int32_t kernel, int32_t metric_kind, int32_t D, char* log, int64_t log_len);
int ahmc_model_destroy(ahmc_ctx* ctx, ahmc_model* model);

/* ---- hot path -------------------------------------------------------------------------------- */
/* phasepoint(h, theta, r)  (src/hamiltonian.jl:115-119): fills z->lp_value, lp_gradient, lk_value
 * (and lk_gradient if non-NULL) from z->theta, z->r. */
int ahmc_phasepoint_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                        const ahmc_phasepoint* z, uint32_t flags);

/* step(lf, h, z, n_steps)  (src/integrator.jl:216-265) for Leapfrog / TemperedLeapfrog
 * (JitteredLeapfrog = caller passes the jittered per-chain eps, integrator.jl:140-156).
 *   eps_chain == NULL -> scalar step size `eps`; else per-chain eps_chain[N] (`AbstractScalarOrVec`).
 *   n_steps < 0 integrates backward (integrator.jl:221-226).  temper_alpha <= 0: no tempering.
 *   status[N] / steps_done[N] may be NULL.  z_in->lp_gradient may be NULL ("not cached": recomputed on the device).
 *   D <= 512: every target x metric, chain state register-resident.  D > 512: std-normal / diagonal-Gaussian / funnel
 *   targets with Unit / Diag metrics (the chain is streamed through registers tile by tile); same for ahmc_phasepoint_f64. */
int ahmc_leapfrog_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                      double eps, const double* eps_chain, int32_t n_steps, double temper_alpha,
                      const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out, uint32_t* status,
                      int32_t* steps_done, uint32_t flags);

/* step(lf, h, z, n_steps; full_trajectory = Val(true))  (src/integrator.jl:229,249-261): every intermediate phase
 * point is returned.  `traj` arrays hold |n_steps| phase points: point i (0-based) of theta/r/lp_gradient/lk_gradient
 * at `i*step_stride + ld*c`, of lp_value/lk_value at `i*N + c`.  A chain that turns non-finite at step k fills k
 * points (the non-finite one included, like `resize!(res, i)`); steps_done[c] = k. */
int ahmc_leapfrog_trajectory_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D,
                                 int64_t N, double eps, const double* eps_chain, int32_t n_steps, double temper_alpha,
                                 const ahmc_phasepoint* z_in, const ahmc_phasepoint* traj, int64_t step_stride,
                                 int32_t* steps_done, uint32_t flags);

/* rand_momentum(rng, metric, kinetic, theta)  (src/metric.jl:290-320): r[D x N] from normals (tape or Philox). */
int ahmc_rand_momentum_f64(ahmc_ctx* ctx, const ahmc_metric* metric, int32_t D, int64_t N, const ahmc_rng* rng,
                           double* r, int64_t ld, uint32_t flags);

/* One static-HMC transition for all chains: refresh (src/sampler.jl:48-58, hamiltonian.jl:213-220) +
 * `transition(rng, h, Trajectory{EndPointTS,...,FixedNSteps}, z)` (src/trajectory.jl:271-300,336-340)
 * + `mh_accept_ratio` (:863-880) + `accept_phasepoint!` (:312-332) + momentum flip (:283). */
int ahmc_hmc_transition_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                            double eps, const double* eps_chain, int32_t n_steps, const ahmc_rng* rng,
                            const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out, const ahmc_stats* stats,
                            uint32_t flags);

/* Static transition with `MultinomialTS` (src/trajectory.jl:344-390): n_steps_fwd forward and
 * n_steps - n_steps_fwd backward steps from z, new point ~ softmax(-H) over the whole trajectory by inverse CDF
 * (`randcat`, src/utilities.jl:92-103), is_accept = true, acceptance_rate = mean_i min(1, exp(H0 - H_i)).
 * The caller draws n_steps_fwd ~ U{0..n_steps} ONCE for all chains, as the reference does (`rand_coupled`,
 * trajectory.jl:371-373).  rng->exp_tape (if given) is the per-chain UNIFORM tape u[N] of `randcat`.
 * stats->tree_depth (if given) receives the signed offset of the drawn point from z. */
int ahmc_hmc_multinomial_transition_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D,
                                        int64_t N, double eps, const double* eps_chain, int32_t n_steps,
                                        int32_t n_steps_fwd, const ahmc_rng* rng, const ahmc_phasepoint* z_in,
                                        const ahmc_phasepoint* z_out, const ahmc_stats* stats, uint32_t flags);

/* One NUTS transition per chain (MultinomialTS + GeneralisedNoUTurn = what `NUTS(delta)` builds,
 * src/abstractmcmc.jl:415-419): src/trajectory.jl:626-742, run one chain per warp-group.
 * AHMC_FLAG_NUTS_SLICE_TS / _CLASSIC / _STRICT select the reference's other trajectory sampler and termination
 * criteria (`HMCKernel(Trajectory{SliceTS}(integrator, ClassicNoUTurn()))` etc.).  With SliceTS the random tape
 * rng->exp_tape holds, per chain, [randexp for the slice variable, then the rand() uniforms of each combine / mh_accept]. */
int ahmc_nuts_transition_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                             double eps, const double* eps_chain, int32_t max_depth, double delta_max,
                             const ahmc_rng* rng, const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out,
                             const ahmc_stats* stats, uint32_t flags);

/* n_transitions transitions per chain in ONE launch: the body of `sample(rng, h, kappa, theta, n_samples)` without
 * adaptation (`for i in 1:n_samples; t = transition(rng, h, kappa, t.z); thetas[i] = t.z.theta`, src/sampler.jl:182-228).
 * Each chain advances at its own pace (no cross-chain barrier between transitions: divergent NUTS tree sizes do
 * not idle the other chains).  Randomness: Philox streams (seed, offset + i); tapes are rejected for n_transitions > 1.
 *   draws  : nullable, n_transitions x (D x N) doubles -- draw i of chain c at ((i*N + c)*D)
 *   stats  : arrays of n_transitions x N entries (entry i*N + c); z_out = phase point after the last transition. */
int ahmc_hmc_sample_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                        double eps, const double* eps_chain, int32_t n_steps, int32_t n_transitions, const ahmc_rng* rng,
                        const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out, double* draws,
                        const ahmc_stats* stats, uint32_t flags);
int ahmc_nuts_sample_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                         double eps, const double* eps_chain, int32_t max_depth, double delta_max, int32_t n_transitions,
                         const ahmc_rng* rng, const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out, double* draws,
                         const ahmc_stats* stats, uint32_t flags);

/* Warm-up + sampling in ONE launch with the reference's VECTORISED adaptors: every chain owns a
 * `NesterovDualAveraging` state (src/adaptation/stepsize.jl:178-210: eps is a length-N vector and adapts per chain) and,
 * with adapt_metric, a windowed `WelfordVar` over its own draws (massmatrix.jl:141-157 with a D x N variance, i.e. a
 * per-chain diagonal M^-1), scheduled like `StanHMCAdaptor` (stan_adaptor.jl:13-50, 137-159: windows, reset of both
 * adaptors at each window end, `finalize!` eps = exp(x_bar) after iteration n_adapts).  Because nothing is pooled,
 * chains never wait for each other: iterations 1..n_adapts adapt, n_adapts+1..n_transitions sample with the final
 * eps / M^-1.  Requires the Diag metric (shared or per-chain M^-1 as the starting point), MultinomialTS +
 * GeneralisedNoUTurn, Philox randomness (no tapes).  Deviation from the reference: a non-finite eps proposal reverts
 * that chain only (the reference reverts every chain, "buggy for batch mode" by its own comment, stepsize.jl:199-203). */
typedef struct ahmc_adapt_cfg {
    int32_t n_adapts;                             /* 0 <= n_adapts <= n_transitions */
    int32_t init_buffer, term_buffer, window_size; /* Stan defaults 75 / 50 / 25; a schedule with more than 12 window
                                                      ends (tiny window_size, huge n_adapts) -> AHMC_ERR_UNSUPPORTED */
    double delta, gamma, t0, kappa;               /* 0.8, 0.05, 10, 0.75 (stepsize.jl:162-172) */
    int32_t adapt_metric;                         /* 0: step size only; 1: + per-chain WelfordVar */
    int32_t n_min;                                /* WelfordVar n_min, 10 (massmatrix.jl:103-107) */
    double* eps_chain;  /* N, in: initial step size per chain; out: adapted step size per chain */
    double* Minv_chain; /* N x D, out: adapted diagonal M^-1 per chain (required iff adapt_metric) */
    double* eps_trace;  /* nullable, n_transitions x N: the step size each transition used (`step_size` stat) */
} ahmc_adapt_cfg;
int ahmc_nuts_adapt_sample_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                               int32_t max_depth, double delta_max, int32_t n_transitions, const ahmc_adapt_cfg* cfg,
                               const ahmc_rng* rng, const ahmc_phasepoint* z_in, const ahmc_phasepoint* z_out,
                               double* draws, const ahmc_stats* stats, uint32_t flags);

/* `find_good_stepsize(rng, h, theta)` (src/trajectory.jl:768-837) for N chains at once, each running its own search, in
 * ONE launch: momentum draw (rng->normal_tape or Philox), the direction probe, the crossing loop and the bisection, every
 * probe `A(h, z, eps)` (:753-757) one leapfrog step.  z: theta + the cached lp_value / lp_gradient (ahmc_phasepoint_f64);
 * eps_out[N]; r_out (nullable, D x N with z->ld) receives the momenta used.  No host round trip. */
int ahmc_find_good_stepsize_f64(ahmc_ctx* ctx, const ahmc_model* model, const ahmc_metric* metric, int32_t D, int64_t N,
                                const ahmc_phasepoint* z, const ahmc_rng* rng, double initial_step_size, int32_t max_n_iters,
                                double* eps_out, double* r_out, uint32_t flags);

/* ---- the one exchange: pooled adaptation across ranks, on the device (SURVEY 8e) ------------------ */
/* Communicator over the GPUs that share one adaptation (one rank per GPU).  NCCL is bound at run time (dlopen of
 * libnccl.so.2, override with AHMC_NCCL_LIB); without it these calls return AHMC_ERR_UNSUPPORTED and single-rank use
 * (comm == NULL) still works.
 *   ahmc_comm_unique_id : rank 0 fills 128 bytes, the host broadcasts them (MPI.jl / Distributed / torch.distributed ...)
 *   ahmc_comm_create    : collective over all ranks -> ncclCommInitRank
 *   ahmc_comm_from_nccl : wrap a communicator the host already owns (NCCL.jl's `Communicator` handle); not destroyed by us */
typedef struct ahmc_comm ahmc_comm;
int ahmc_comm_unique_id(ahmc_ctx* ctx, void* id128_out);
int ahmc_comm_create(ahmc_ctx* ctx, const void* id128, int32_t nranks, int32_t rank, ahmc_comm** out);
int ahmc_comm_from_nccl(ahmc_ctx* ctx, void* nccl_comm /* ncclComm_t */, int32_t nranks, int32_t rank, ahmc_comm** out);
int ahmc_comm_destroy(ahmc_ctx* ctx, ahmc_comm* comm);

/* All-gather of a small per-rank record of n doubles on the context stream (ncclAllGather; comm == NULL: one rank, a
 * device copy).  record / out are device pointers (out: nranks * n doubles, rank order).  No host synchronisation with
 * AHMC_FLAG_ASYNC. */
int ahmc_adapt_allgather_f64(ahmc_ctx* ctx, ahmc_comm* comm, const double* record, int64_t n, double* out, uint32_t flags);

/* Pooled Stan-style adaptor living on the device: one shared step size (dual averaging on the mean of min(1, alpha)
 * over ALL chains of ALL ranks, src/adaptation/stepsize.jl:178-210) and one shared diagonal M^-1 (`WelfordVar` over
 * chains x iterations of a window, massmatrix.jl:141-157), scheduled by `StanHMCAdaptor` (stan_adaptor.jl:13-50,
 * 137-159).  The reference never pools (`Adaptation.jl:52` TODO); with one chain on one rank this is its scalar path.
 * The adaptor owns two device buffers the transition calls read directly:
 *   ahmc_pooled_eps(a)  : eps_chain[N] (every entry the shared step size)  -> pass as `eps_chain`
 *   ahmc_pooled_minv(a) : Minv[D]                                          -> pass as ahmc_metric.Minv (Diag, stride 0) */
typedef struct ahmc_pooled_cfg {
    int32_t n_adapts;
    int32_t init_buffer, term_buffer, window_size; /* 75 / 50 / 25 */
    double delta, gamma, t0, kappa;               /* 0.8, 0.05, 10, 0.75 */
    double eps0;                                  /* initial step size */
    int32_t adapt_metric;                         /* 0: step size only; 1: + pooled WelfordVar */
    int32_t n_min;                                /* 10 */
} ahmc_pooled_cfg;
typedef struct ahmc_pooled ahmc_pooled;
int ahmc_pooled_create(ahmc_ctx* ctx, int32_t D, int64_t N, const ahmc_pooled_cfg* cfg,
                       const double* Minv0 /* host, D doubles, NULL = ones */, ahmc_pooled** out);
int ahmc_pooled_destroy(ahmc_ctx* ctx, ahmc_pooled* a);
double* ahmc_pooled_eps(ahmc_pooled* a);
double* ahmc_pooled_minv(ahmc_pooled* a);
/* `adapt!(adaptor, theta, alpha)` of iteration i = (calls so far) + 1 (sampler.jl:72-90 glue), entirely on the context
 * stream: K5 record of this rank's N chains -> all-gather over `comm` (NULL: single rank) -> rank-ordered Chan merge,
 * dual averaging, window logic, `finalize!` at i == n_adapts; eps / M^-1 land in the buffers above before the next
 * transition (same stream) starts.  theta[D x N] (ld), acceptance_rate[N]: device pointers.  Nothing is copied to the
 * host and, with AHMC_FLAG_ASYNC, nothing is waited for.  eps_trace (nullable, device, n_adapts doubles) receives the
 * step size after each iteration. */
int ahmc_adapt_exchange_f64(ahmc_ctx* ctx, ahmc_comm* comm, ahmc_pooled* a, int32_t D, int64_t N, const double* theta,
                            int64_t ld, const double* acceptance_rate, double* eps_trace, uint32_t flags);
/* synchronising read-back of the adaptor (host outputs, each nullable): current eps, Minv[D], iterations done,
 * the merged record [n, sum alpha, mean[D], M2[D]] of the last exchange.  A dense adaptor -> AHMC_ERR_INVALID
 * (use ahmc_pooled_state_dense). */
int ahmc_pooled_state(ahmc_ctx* ctx, ahmc_pooled* a, double* eps, double* Minv, int32_t* iteration, double* merged_record);

/* StanHMCAdaptor(WelfordCov, NesterovDualAveraging) pooled over all chains of all ranks, on the device (massmatrix.jl:286-340).
 * Minv0: host, D x D column-major, symmetric positive definite; NULL = I.  1 <= D <= 512 (the dense operators' bound):
 * D > 512 -> AHMC_ERR_UNSUPPORTED; a Minv0 whose Cholesky factorisation fails -> AHMC_ERR_INVALID (creation synchronises).
 *   ahmc_pooled_minv(a)  : Minv[D x D] column-major     -> ahmc_metric{AHMC_METRIC_DENSE, Minv, 0, cholU}
 *   ahmc_pooled_cholu(a) : cholU[D x D] column-major upper factor, U'U = Minv (NULL for a diagonal adaptor)
 * ahmc_adapt_exchange_f64 records [n, sum alpha, mean[D], M2diag[D], M2full[D*D]] (K5 + K5b, adapt_metric = 1) or the
 * diagonal record (adapt_metric = 0: step size only, Minv0 and its factor are never touched).  Minv changes only at a window
 * split inside the metric window with n >= n_min, to n/((n+5)(n-1)) M + 1e-3 (5/(n+5)) I, and cholU with it: the new
 * estimate is factorised on the device (upper triangle only) and committed with its factor only if every pivot is > 0;
 * otherwise both keep their previous values and the iteration is recorded as `failed_iteration` (first failure only). */
int ahmc_pooled_create_dense(ahmc_ctx* ctx, int32_t D, int64_t N, const ahmc_pooled_cfg* cfg, const double* Minv0,
                             ahmc_pooled** out);
double* ahmc_pooled_cholu(ahmc_pooled* a);
/* synchronising read-back of a dense adaptor (host outputs, each nullable): eps, Minv[D*D], cholU[D*D] (column-major),
 * iterations done, the merged record [n, sum alpha, mean[D], M2diag[D], M2full[D*D]] of the last exchange (the D x D part
 * stays zero with adapt_metric = 0), the first iteration whose factorisation failed (0 = never).  A diagonal adaptor ->
 * AHMC_ERR_INVALID. */
int ahmc_pooled_state_dense(ahmc_ctx* ctx, ahmc_pooled* a, double* eps, double* Minv, double* cholU, int32_t* iteration,
                            double* merged_record, int32_t* failed_iteration);

/* ---- adaptor statistics (src/adaptation) ------------------------------------------------------ */
/* Pooled summary of one iteration over this GPU's N chains, written to a small device/host record that
 * the host all-gathers across ranks (one NCCL all-gather, SURVEY 8e) and merges in rank order:
 *   out[0] = N, out[1] = sum_c min(1, alpha_c)                       (dual averaging, stepsize.jl:178-210)
 *   out[2 .. 2+D)   = mean_c theta[:,c]        out[2+D .. 2+2D) = sum_c (theta[:,c]-mean)^2
 * (the (n, mu, M2) Welford partial of massmatrix.jl:141-149 over the chain axis). */
int ahmc_adapt_summary_f64(ahmc_ctx* ctx, int32_t D, int64_t N, const double* theta, int64_t ld,
                           const double* acceptance_rate, double* out /* 2+2D */, uint32_t flags);

/* Dense companion of the record above, for the pooled `WelfordCov` (src/adaptation/massmatrix.jl:286-340):
 *   out[i + D*j] = sum_c (theta[i,c] - mean[i]) * (theta[j,c] - mean[j])      (D x D, symmetric)
 * with `mean` = out[2 .. 2+D) of ahmc_adapt_summary_f64 on the same theta.  Records (n, mean, M2) of different
 * ranks / iterations merge exactly (Chan): M2 = M2_a + M2_b + (n_a n_b / n) dd', d = mean_b - mean_a. */
int ahmc_adapt_cov_f64(ahmc_ctx* ctx, int32_t D, int64_t N, const double* theta, int64_t ld, const double* mean,
                       double* out /* D*D */, uint32_t flags);

#ifdef __cplusplus
}
#endif
#endif /* AHMC_B200_H */
