/*
 * pn_b200.h -- C ABI of the B200-native adaptive probabilistic IVP solver.
 *
 * The reference (pnkraemer/code-adaptive-prob-ode-solvers) has no FFI: its boundary is the
 * Python call `odecheckpts.ivpsolvers.solve(...)` -> `solve_(u0, p)`
 * (src/odecheckpts/ivpsolvers.py:14-91), which builds a probdiffeq solver and calls
 * `ivpsolve.solve_adaptive_save_at` (ivpsolvers.py:71-77) followed by
 * `stats.markov_marginals(reverse=True)` (ivpsolvers.py:80-81).  The entry points below are
 * what a jax.ffi / ctypes binding for that path binds: plain pointers and sizes, a POD
 * descriptor, a CUDA stream.  No torch/jax types.  See INTEGRATION.md for the binding stubs.
 *
 * Ownership: the caller owns every buffer.  `pn_b200_solve_save_at` takes DEVICE pointers, is
 * stream-ordered and asynchronous, and is re-entrant across streams and threads as long as each
 * call has its own workspace.  Process-wide state is limited to immutable constant tables, a cache
 * of launch geometry per (device, kernel), and -- for `pn_b200_solve_save_at_host` only -- one
 * private stream-ordered memory pool per device that keeps its blocks between calls (release them
 * with `pn_b200_trim`).  The host entry restores the caller's current device before it returns.
 * The optional kernel timing (`pn_b200_set_profiling`) is per calling thread.
 * Per-member numerical failure never aborts the batch: it is reported in status[b].
 */
#ifndef PN_B200_H
#define PN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* problem ids: the IVP zoo of src/odecheckpts/ivps.py (device functors) */
enum {
  PN_B200_LOGISTIC = 0,       /* ivps.py:8-17    d=1  q=1 params (a, b)      */
  PN_B200_RIGID_BODY = 1,     /* ivps.py:20-29   d=3  q=1 params (a, b, c)   */
  PN_B200_THREE_BODY = 2,     /* ivps.py:32-41   d=2  q=2 params (mu)        */
  PN_B200_PLEIADES = 3,       /* ivps.py:59-99   d=14 q=2 no params          */
  PN_B200_BRUSSELATOR = 4,    /* ivps.py:124-156 d=2N q=1 params (alpha)     */
  PN_B200_VAN_DER_POL = 5,    /* ivps.py:159-167 d=1  q=2 params (mu)        */
  PN_B200_LOTKA_VOLTERRA = 6  /* diffeqzoo       d=2  q=1 params (a,b,c,d)   */
};
enum { PN_B200_ISOTROPIC = 0, PN_B200_BLOCKDIAG = 1, PN_B200_DENSE = 2 }; /* impl.select, ivpsolvers.py:33 */
enum { PN_B200_TS0 = 0, PN_B200_TS1 = 1 };            /* correction_ts0/ts1, ivpsolvers.py:37; vdp.py:64 */
enum { PN_B200_FILTER = 0, PN_B200_FIXEDPOINT = 1 };  /* strategy_*, ivpsolvers.py:43; vdp.py:65          */
enum {
  PN_B200_CALIB_NONE = 0,    /* ivpsolvers.solver,         ivpsolvers.py:48 */
  PN_B200_CALIB_DYNAMIC = 1, /* ivpsolvers.solver_dynamic, ivpsolvers.py:46 */
  PN_B200_CALIB_MLE = 2      /* ivpsolvers.solver_mle (no call site in the reference): the solve uses output_scale0; the
                                running quasi-MLE sqrt(mean over accepted steps of z^T S^-1 z / d) is reported in
                                output_scale and its final value scales u_std / marg_chol; thread-per-IVP kernels */
};
enum { PN_B200_OK = 0, PN_B200_NAN = 1, PN_B200_MAX_ATTEMPTS = 2 };  /* status[b] */
enum {
  PN_B200_FLAG_FIXED_GRID = 1, /* solve_fixed_grid (vdp.py:88-91): steps = diff(save_at), no rejection */
  PN_B200_FLAG_RECORD = 2,     /* solve_adaptive_save_every_step (vdp.py:77-79): record accepted steps */
  PN_B200_FLAG_MEMBER_GRIDS = 4 /* save_at is [B][K]: row b is member b's grid (jax.vmap over save_at / t0 / t1) */
};

/* return codes of the entry points */
enum {
  PN_B200_SUCCESS = 0,
  PN_B200_ERR_UNSUPPORTED = -1,  /* no kernel for this (problem, nu, factorisation, ...) */
  PN_B200_ERR_ARGUMENT = -2,
  PN_B200_ERR_WORKSPACE = -3,
  PN_B200_ERR_CUDA = -4
};

/* Mirrors the solver construction of ivpsolvers.py:14-53. */
typedef struct {
  int32_t problem, d, nu, ode_order;
  int32_t factorisation, correction, strategy, calibration;
  double atol, rtol, dt0;                 /* ivpsolve.adaptive(atol=, rtol=), dt0    ivpsolvers.py:53,75 */
  double safety, factor_min, factor_max;  /* control_proportional_integral() defaults 0.95, 0.2, 10 */
  double power_integral, power_proportional; /* 0.3, 0.4 (divided by nu+1 inside)                    */
  int64_t batch;                          /* ensemble members B                                     */
  int64_t num_save_at;                    /* K checkpoints, save_at[0] = t0          ivpsolvers.py:63 */
  int64_t max_attempts;                   /* per member; <= 0: unlimited                            */
  int32_t num_params;                     /* P parameters per member                                */
  int32_t flags;                          /* PN_B200_FLAG_*                                         */
  int64_t traj_capacity;                  /* PN_B200_FLAG_RECORD: grid points kept per member       */
} pn_b200_desc;

/* 0 if a kernel exists for this descriptor, else PN_B200_ERR_UNSUPPORTED / _ARGUMENT. */
int pn_b200_supported(const pn_b200_desc* desc);

/* Device scratch the solve needs (the K backward conditionals per member: O(K), not O(#steps)). */
size_t pn_b200_workspace_bytes(const pn_b200_desc* desc);

/* Element counts of every output buffer of pn_b200_solve_save_at for `desc` (doubles, except
 * n_accepted / n_rejected / traj_len: int64 and status: int32).  Callers size their buffers from
 * this instead of deriving shapes by hand (marg_chol depends on the factorisation, see below). */
typedef struct {
  size_t u, u_std;                 /* B*K*d each                                             */
  size_t marg_mean, marg_chol;     /* optional outputs                                       */
  size_t output_scale;             /* B*K, blockdiag: B*K*d                                  */
  size_t n_accepted, n_rejected, status;
  size_t traj_t, traj_u, traj_std, traj_len; /* 0 unless PN_B200_FLAG_RECORD                 */
} pn_b200_sizes;
int pn_b200_output_sizes(const pn_b200_desc* desc, pn_b200_sizes* sizes);

/*
 * solve_adaptive_save_at + backward marginalisation for a whole ensemble (DEVICE pointers).
 *   u0            [B][q][d]     initial values (u, u', ...)
 *   params        [B][P]        vector-field parameters (may be NULL if P == 0)
 *   tol           [B][2] | NULL per-member (atol, rtol); NULL: desc->atol/rtol for all
 *   save_at       [K]           checkpoints, strictly increasing, save_at[0] = t0 (a precondition: not checked)
 *                 [B][K]        with PN_B200_FLAG_MEMBER_GRIDS: row-major, row b is member b's grid, each row
 *                               strictly increasing (not checked), save_at[b][0] = t0 of member b; K is the same
 *                               for every member.  Combined with PN_B200_FLAG_FIXED_GRID row b is member b's
 *                               step grid; with PN_B200_FLAG_RECORD (K = 2) row b is [t0_b, t1_b] and the
 *                               recording semantics below hold per member (the last point is at t1_b).  The flag
 *                               changes no output size, no workspace size and no supported configuration;
 *                               sampling and the likelihood take no times (they read the finished solve's
 *                               workspace), so they need no per-member argument.
 *   output_scale0 [B] | NULL    initial output scale (ivpsolvers.py:55,68); NULL: 1.0
 *   u, u_std      [B][K][d]     smoothed checkpoint means / marginal standard deviations
 *   marg_mean     [B][K][n][d] | NULL   full marginal means (n = nu+1; for the dense factorisation this
 *                 is the flat state vector of length D = n*d, derivative-major index i*d + l)
 *   marg_chol     | NULL                full marginal square-root factors, shape by factorisation:
 *                 isotropic, and dense with d == 1:  [B][K][n][n]
 *                 blockdiag with d > 1:              [B][K][d][n][n]   (one factor per dimension)
 *                 dense with d > 1:                  [B][K][D][D], D = n*d, derivative-major
 *                 -- size the buffer with pn_b200_output_sizes(), never by hand
 *   output_scale  [B][K] | NULL the output scale every checkpoint carries (solution.output_scale:
 *                 the calibrated sigma of the accepted step that reached or crossed it; entry 0 is
 *                 output_scale0); blockdiag: [B][K][d], one scale per dimension
 *   n_accepted    [B][K]        cumulative accepted steps when checkpoint k was emitted
 *   n_rejected    [B], status [B]
 *   traj_*        PN_B200_FLAG_RECORD only (filter strategy): traj_t [cap][B], traj_u [cap][d][B],
 *                 traj_std [cap][B] (one std for all dimensions), or [cap][d][B] for the dense
 *                 factorisation with d > 1 (per dimension: sqrt of the diagonal of L L^T), traj_len [B];
 *                 NULL otherwise.  Point 0 is t0 (std 0), then one point per accepted step; a step that
 *                 crosses checkpoints is recorded at the last of them, so the last point is at
 *                 save_at[K-1] (save_at[b][K-1] with PN_B200_FLAG_MEMBER_GRIDS).  traj_len = min(accepted steps + 1, cap): later points are dropped
 */
int pn_b200_solve_save_at(const pn_b200_desc* desc, const double* u0, const double* params,
                          const double* tol, const double* save_at, const double* output_scale0,
                          double* u, double* u_std, double* marg_mean, double* marg_chol,
                          double* output_scale, int64_t* n_accepted, int64_t* n_rejected, int32_t* status, double* traj_t,
                          double* traj_u, double* traj_std, int64_t* traj_len, void* workspace,
                          size_t workspace_bytes, void* cuda_stream);

/*
 * The same call with HOST buffers (what a CPU caller such as the reference's experiment
 * scripts holds): allocates device memory, copies in, solves, copies out, synchronises.
 * `device` is the CUDA device ordinal.  With PN_B200_FLAG_MEMBER_GRIDS it copies B*K grid points
 * and returns PN_B200_ERR_ARGUMENT when a row is not strictly increasing.
 */
int pn_b200_solve_save_at_host(const pn_b200_desc* desc, const double* u0, const double* params,
                               const double* tol, const double* save_at, const double* output_scale0,
                               double* u, double* u_std, double* marg_mean, double* marg_chol,
                               double* output_scale, int64_t* n_accepted, int64_t* n_rejected, int32_t* status, double* traj_t,
                               double* traj_u, double* traj_std, int64_t* traj_len, int device);

/* Returns the device memory cached by pn_b200_solve_save_at_host on `device` to the driver. */
int pn_b200_trim(int device);

/*
 * Joint samples from the checkpoint Markov sequence of a FINISHED fixed-point solve:
 * stats.markov_sample(key, posterior, shape=(S,), reverse=True), experiments/5_vs_interpolation/measure.py:69-77.
 * `workspace` / `status` are the buffers the solve call used (the K backward conditionals are read
 * from the workspace); samples: [B][S][K][d] draws of the ODE solution at the checkpoints (DEVICE).
 * Random numbers are Philox4x32-10 + Box-Muller keyed by `seed`: same distribution as the reference,
 * not the same bits as jax.random.  Every kernel family (isotropic / blockdiag / dense, any dimension).
 */
int pn_b200_markov_sample(const pn_b200_desc* desc, const void* workspace, size_t workspace_bytes,
                          const int32_t* status, uint64_t seed, int64_t num_samples, double* samples,
                          void* cuda_stream);

/*
 * Log marginal likelihood of observations of the ODE solution at the checkpoints, from a FINISHED
 * fixed-point solve: stats.log_marginal_likelihood(u, standard_deviation=, posterior=),
 * src/odecheckpts/train_util.py:22-24 (the parameter-inference loss, forward value only).
 * `workspace` / `status` are the buffers the solve call used.  data: [B][K][d] observed values of u
 * at save_at[0..K-1] (member b's row save_at[b][0..K-1] with PN_B200_FLAG_MEMBER_GRIDS); obs_std: [B][K] observation noise standard deviations (> 0); lml: [B] (all
 * DEVICE pointers).  lml[b] is the running mean over the K data points of
 * log p(y_k | y_{k+1}, ..., y_{K-1}) -- probdiffeq's reverse Kalman-filter estimator -- i.e. the joint
 * log density divided by K; NaN for failed members.  Isotropic and blockdiag factorisations of any dimension and the
 * dense factorisation with d == 1 (PN_B200_ERR_UNSUPPORTED for dense with d > 1).
 */
int pn_b200_log_marginal_likelihood(const pn_b200_desc* desc, const void* workspace, size_t workspace_bytes,
                                    const int32_t* status, const double* data, const double* obs_std,
                                    double* lml, void* cuda_stream);

/* Launch geometry and compiled resource usage of the kernel that serves `desc` (for reports). */
typedef struct {
  int32_t threads_per_cta, ctas_per_sm, num_sms, grid;
  int32_t registers_per_thread, static_smem_bytes, dynamic_smem_bytes, local_bytes_per_thread;
} pn_b200_kernel_info;
int pn_b200_get_kernel_info(const pn_b200_desc* desc, pn_b200_kernel_info* info);

/* Register-resident DFMA-chain microbenchmark: measured fp64 FMA peak of the current device in
 * TFLOP/s (the roofline denominator; MEASURED_PEAKS.json carries no fp64 entry). */
int pn_b200_measure_fp64_peak(double* tflops, void* cuda_stream);

/* Optional per-kernel timing for reports: when enabled, pn_b200_solve_save_at brackets its two
 * kernels (the persistent solver loop and the smoothing sweep) with CUDA events on the caller's
 * stream; pn_b200_get_last_timing waits for them and returns their durations in milliseconds. */
int pn_b200_set_profiling(int enable);
int pn_b200_get_last_timing(float* solve_ms, float* smooth_ms);

/*
 * User-defined vector fields, compiled at run time (NVRTC) into the same kernels the built-in problems use.
 *
 * `source` is CUDA C++ in one of two forms:
 *   PN_B200_FORM_SIMPLE  template <class T> PN_DEV void vf(const T* u, const double* p, T* f)
 *                        u = (u, u', ...)[ode_order * d], p[num_params], f[d]; T is double or pn::Jet<N> (truncated
 *                        Taylor series).  Optionally  PN_DEV void jac(const double* u, const double* p, double* J)
 *                        with J[d][ode_order * d]; without it the Jacobian is derived from vf on pn::Jet<2>.
 *   PN_B200_FORM_FULL    struct Problem with the interface of the built-in functors (csrc/pn_problems.cuh):
 *                        D, Q, P, HAS_JAC, vf, jac, vf_jet<N>.
 * OR-ed into `form`, PN_B200_FORM_TIME_DEPENDENT registers a non-autonomous field, whose functions take the time
 * after the state:
 *   simple               template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f), and
 *                        optionally  PN_DEV void jac(const double* u, double t, const double* p, double* J).  In the
 *                        Taylor-mode initialisation t is the series (t0, 1, 0, ...), so the coefficients are the
 *                        exact derivatives u^(k)(t0).
 *   full                 struct Problem with  static constexpr bool TIME = true,  vf(u, t, p, f), jac(u, t, p, J)
 *                        and vf_jet<N>(U, Tc, p, F), Tc[N] the time's normalised Taylor coefficients.
 * The solver evaluates the field (and the Jacobian) of an attempted step at its end, t + dt, or at the checkpoint
 * it is aimed at: the time the step commits when it is accepted.  The flag is part of the registration: the same
 * name and source with and without it are two problems.
 * Registration compiles a check kernel: a compile error returns PN_B200_ERR_ARGUMENT, and pn_b200_last_error()
 * holds the whole compiler log, whose line numbers are the lines of `source` under the file name `name`
 * ([A-Za-z0-9_.-], at most 128 characters).  Registering the same (name, source, form, sizes) again returns the
 * same id.  d in 1 .. 32, ode_order 1 or 2, num_params 0 .. 64.  The source lives in a namespace of its own in
 * which the names Prob, PnSource, PN_HAS_JAC and pn_no_jac are taken.  Ids are handed out in registration order,
 * so processes that register the same problems in the same order (the ranks of a multi-GPU run) share ids.
 *
 * A user problem id (>= PN_B200_USER_PROBLEM_BASE) goes into pn_b200_desc.problem like a built-in one.  Its kernels
 * are compiled on first use per (kernel family, nu, strategy) and cached for the life of the process: the first
 * solve, pn_b200_get_kernel_info or pn_b200_compile of a configuration compiles, pn_b200_supported and
 * pn_b200_workspace_bytes never do.  Builds: the thread-per-IVP kernels (d <= 3; the small-ensemble build for the
 * fixed-point strategy with d <= 2), the lane-per-dimension kernels (isotropic and blockdiag, d <= 32) and the
 * dense register-column kernel ((nu + 1) d <= 32).
 */
enum { PN_B200_USER_PROBLEM_BASE = 1024 };
enum { PN_B200_FORM_SIMPLE = 0, PN_B200_FORM_FULL = 1, PN_B200_FORM_TIME_DEPENDENT = 2 };
int pn_b200_register_problem(const char* name, const char* source, int form, int32_t d, int32_t ode_order,
                             int32_t num_params, int32_t* problem_id);

/* Compiles (and loads) the kernels that serve `desc` now, so that a later timed solve does not include the
 * compilation.  A no-op for built-in problems. */
int pn_b200_compile(const pn_b200_desc* desc);

/*
 * Evaluates a problem's functor for n states (DEVICE pointers, stream-ordered): u0 [n][ode_order][d],
 * params [n][P] (P: the problem's parameter count); outputs, each optional (NULL: not computed):
 *   f      [n][d]              the vector field at u0
 *   taylor [n][nu + 1][d]      the Taylor coefficients u^(k)(t0), k = 0 .. nu, the solver's initialisation
 *   jac    [n][d][ode_order d] the Jacobian (PN_B200_ERR_UNSUPPORTED for a problem without one)
 * For user problems and for the built-in problems of fixed size (all but the Brusselator), whose functors are
 * compiled for this the same way.
 */
int pn_b200_problem_evaluate(int32_t problem, int32_t nu, int64_t n, const double* u0, const double* params, double* f,
                             double* taylor, double* jac, void* cuda_stream);
/* The same at per-state times t [n] (DEVICE; NULL: 0), for time-dependent problems: f and jac at (t, u0), taylor the
 * coefficients u^(k)(t).  An autonomous problem ignores t. */
int pn_b200_problem_evaluate_at(int32_t problem, int32_t nu, int64_t n, const double* t, const double* u0,
                                const double* params, double* f, double* taylor, double* jac, void* cuda_stream);

/* Human-readable description of the last error on the calling thread. */
const char* pn_b200_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
