// pn_scalar_kernel.cuh -- thread-per-IVP persistent solver kernel (sm_100a, fp64).
//
// One CUDA thread owns one IVP of the ensemble and runs the whole adaptive time loop of
// probdiffeq's `ivpsolve.solve_adaptive_save_at` (called at
// src/odecheckpts/ivpsolvers.py:71-77, experiments/4_brusselator/run.py:122-129,
// experiments/5_vs_interpolation/measure.py:66-68) for state-space models whose square-root
// factors are n x n (n = nu+1):
//   * isotropic factorisation (impl.select("isotropic"), ivpsolvers.py:32-33) with EKF0
//     (correction_ts0) for small ODE dimension D (mean n x D in registers), and
//   * dense factorisation with D == 1 (experiments/1_van_der_pol/vdp.py:61-66) with EKF0/EKF1.
// The algorithm is SURVEY.md Appendix A: IWP prior in preconditioned coordinates (A.1),
// one attempted step = predict mean -> linearise -> calibrate + local error -> predict
// sqrt-covariance by Householder QR of the stacked factors (fixed-point strategy: 2n x 2n block
// QR + triangular solve -> backward conditional, merged into the running conditional) ->
// sqrt correction -> scaled error norm -> PI controller (A.3, A.4); checkpoints by
// interpolation with an identity-reset backward model (A.5).
//
// Design (B200-first, not a translation of the JAX control flow):
//   * All lanes of a warp always execute the SAME straight-line "uber step": a lane is either
//     attempting a step (MODE_STEP) or doing one of the two extra predictions a checkpoint
//     needs (MODE_INTERP_A: previous state -> checkpoint, MODE_INTERP_B: checkpoint -> accepted
//     state).  Accept/reject and checkpoint handling only change which results a lane commits,
//     so per-member step control costs predicated moves, not divergent code.
//   * The step's working set (block-QR workspace, reflectors, new conditional) lives in registers;
//     everything only read at the start of a step or written at commit -- hidden state (mean,
//     Cholesky factor), running backward conditional (G, g, Lam), and the accepted-but-uncommitted
//     state of a lane that is interpolating -- is parked in shared memory ([element][thread],
//     conflict free).
//   * Only the first n columns of the 2n x 2n fixed-point block matrix are triangularised; the
//     lower-right block is used as a full square-root factor and the merge re-triangularises.
//   * Lanes pull members from a global atomic ticket, so differing step counts (tolerance
//     sweeps) never idle a lane while work remains; members that carry their own tolerances are
//     handed out tightest first (SolveArgs::order).
//   * SLICE = 1 instances time-slice the members (see SolveArgs::slice_mask and the slice_* helpers):
//     a member is parked after a quantum of attempted steps when a more lagging one is ready, so all
//     members finish together and an ensemble of 1.73 x the resident lanes does not end on a
//     half-empty wave.  The helpers are out of line: the step's register allocation is untouched.
//   * HBM traffic: inputs once per member; per checkpoint one backward conditional into the
//     member-major workspace [member][checkpoint][element] (a lane's slot is contiguous, so its
//     stores fill whole sectors even when the lanes of a warp cross checkpoints at different times).
//   * The O(K) backward marginalisation (stats.markov_marginals(reverse=True),
//     ivpsolvers.py:80-81) runs as a second, fully convergent kernel (pn_smooth_kernel).
//   * GROUP > 1 / WIDE = 1 reuse the same step for lane-per-dimension and CTA-per-IVP mappings.
//
// Arithmetic order follows oracle/pn_solver.c exactly, skipping structural zeros only (which is
// exact), so results are comparable bit for bit.
#pragma once
#include "pn_math.cuh"
#include "pn_problems.cuh"

namespace pn {

enum : int { MODE_STEP = 0, MODE_INTERP_A = 1, MODE_INTERP_B = 2 };
enum : int { FLAG_FIXED_GRID = 1, FLAG_RECORD = 2, FLAG_MEMBER_GRIDS = 4 };

struct SolveArgs {
  int32_t correction;   // 0 ts0, 1 ts1 (D == 1 only)
  int32_t calibration;  // 0 none, 1 dynamic, 2 running quasi-MLE (solver_mle; thread-per-IVP kernels)
  int32_t flags;
  int32_t num_params;
  double atol, rtol, dt0;
  double safety, factor_min, factor_max, pow_i, pow_p;  // pow_* already divided by n
  long long B, K, max_attempts;
  const double* u0;       // [B][Q*D]
  const double* params;   // [B][P]
  const double* tol;      // nullable [B][2]
  const double* save_at;  // [K], or [B][K] (FLAG_MEMBER_GRIDS): read through grid_row()
  const double* sigma0;   // nullable [B]
  double* cond;           // workspace [B*dv][K][SLOT] (member-major: a lane's slot is contiguous, so its
                          // stores fill whole 32-byte sectors); slot 0 = terminal state
  long long* n_accepted;  // [B][K]
  long long* n_rejected;  // [B]
  int32_t* status;        // [B]
  unsigned long long* ticket;
  // nullable [B]: ticket -> member.  The host entry fills it (smallest tolerance first) when members
  // carry their own tolerances, so the members with the most steps start first and the launch does
  // not end on a tail of a few long solves.
  const long long* order;
  // Time-sliced scheduling (SLICE = 1 instances of the thread-per-IVP kernel, uniform tolerances): a
  // lane runs a member for a quantum of attempted steps, then parks it (state -> ctx) in the ready queue
  // of the checkpoint interval it is in and takes the most lagging ready member instead.  All members
  // then move through the checkpoints roughly in lockstep and finish together, so an ensemble that is a
  // non-integer multiple of the resident lanes no longer ends on a half-empty wave.  Scheduling only:
  // the arithmetic of a member is unchanged.  Fresh members (plain ticket) go before every parked one.
  //   squeue [G][B]  rings of parked member ids, one per queue group g = (k_next - 1) >> slice_shift
  //                  (-1 = position taken, id not stored yet); G <= 63
  //   sq     [2 g]   pop counter, [2 g + 1] push counter of group g
  //   sw     [0]     bit g: queue g may be non-empty; bit 63: no fresh member left;  [1] finished members
  //   ctx    [B][CTX] parked states
  long long slice_mask;  // quantum - 1 (quantum: attempted steps between two scheduling decisions, a power of two)
  int32_t slice_shift;
  int32_t* squeue;
  unsigned* sq;
  unsigned long long* sw;
  double* ctx;
  // calibration == 2 (solver_mle): [B] the final quasi-MLE factor sqrt(mean over accepted steps of z^T S^-1 z / d)
  // that the smoothing kernel applies to the marginal standard deviations / factors (nullable otherwise)
  double* mle_scale;
  // nullable [B][K][S]: the output scale carried by every checkpoint (solution.output_scale);
  // S = d for the blockdiag factorisation (one scale per dimension), else 1
  double* out_scale;
  // optional trajectory recording (solve_adaptive_save_every_step, vdp.py:77-79)
  double* traj_t;    // [cap][B]
  double* traj_u;    // [cap][D][B]
  double* traj_std;  // [cap][B]   (isotropic: one std for all dimensions)
  long long traj_cap;
  long long* traj_len;  // [B]
  // wide (CTA-per-IVP) kernel only: runtime ODE dimension and the per-member mean arrays
  // [B][3][n][d] (state mean, backward-conditional offset g, pending mean) in global memory
  int wide_d;
  int wide_smem_means;  // how many of the member's mean arrays (state mean, conditional offset g, pending mean -- in
                        // that order) live in shared memory instead of wide_mean: few members, as many as fit
  double* wide_mean;
  // Prior constant (SURVEY A.1): lower Cholesky factor of the flipped Hilbert matrix, row-major
  // n x n, computed by the host (pn_capi.cu).  Kernel parameters live in the constant bank, so
  // DFMA reads these entries as immediate constant operands.
  double lq[100];
  // row stride of save_at: 0 (one grid for all members) or K (FLAG_MEMBER_GRIDS).  Last, so that the fields above
  // keep their parameter offsets.
  long long save_stride;
};

// Member b's checkpoint grid, derived from b where it is read (member fetch, emitted checkpoints, the dense kernels), so
// that no per-lane row pointer stays live through a step loop.  The step loop of pn_scalar_kernel reads the time of
// checkpoint k_next from its shared-memory slot instead (ck_cached / set_ck).
PN_DEV const double* grid_row(const SolveArgs& a, long long b) { return a.save_at + b * a.save_stride; }

// ---- time-sliced scheduling: cold paths, kept out of line so that they do not disturb the register
// allocation of the step -----------------------------------------------------------------------
// Default number of attempted steps between two scheduling decisions.  One park + take-over costs the
// WARP about nine step iterations (cold code, L2 / DRAM round trips), so the quantum is long: two to
// four slices per member are enough to fill the last wave (measured: 8192 -> 179 ms, 2048 -> 193 ms,
// unsliced 208 ms on the 65,536-member Van der Pol ensemble).
constexpr int SLICE_QUANTUM = 8192;
constexpr unsigned long long SLICE_FRESH_GONE = 1ULL << 63;
// doubles one parked member occupies: running conditional + hidden state + 8 scalars, padded to 16 bytes
__host__ __device__ constexpr int slice_ctx_doubles(int nbw, int nstate) { return (nbw + nstate + 8 + 1) & ~1; }
struct SliceScalars {
  double t, dt_next, le_prev, sigma_state;
  long long k_next, n_acc, n_rej, n_att;
};

// after a pop that may have emptied queue g (or found it empty): clear its bit, then repair the bit if
// a push slipped in between (a pusher sets the bit itself after it has taken its position)
static __device__ __forceinline__ void slice_mark_empty(const SolveArgs* a, int g) {
  atomicAnd(a->sw, ~(1ULL << g));
  __threadfence();  // the re-read must not overtake the clear: a push + set in between would be wiped out
  const uint2 ht = __ldcg((const uint2*)(a->sq + 2 * g));
  if (ht.x < ht.y) atomicOr(a->sw, 1ULL << g);
}

// Safety net, run by warps that have nothing to do: rebuild the "may be non-empty" bits from the
// counters themselves, so that a parked member can never stay invisible (stale set bits are harmless,
// the next taker clears them).
static __device__ __noinline__ void slice_repair(const SolveArgs* a, int groups) {
  for (int g = 0; g < groups; ++g) {
    const uint2 ht = __ldcg((const uint2*)(a->sq + 2 * g));
    if (ht.x < ht.y) atomicOr(a->sw, 1ULL << g);
  }
}

// Take the most lagging ready member: a fresh one while tickets last, else the head of the lowest
// non-empty ready queue.  Returns the member or -1; *resume = 1 if it has a parked state.
static __device__ __noinline__ long long slice_claim(const SolveArgs* a, int* resume, int* exhausted) {
  const unsigned long long Bu = (unsigned long long)a->B;
  *resume = 0;
  const ulonglong2 w = __ldcg((const ulonglong2*)a->sw);  // (queue mask | fresh-gone flag, finished members)
  unsigned long long m = w.x;
  if (!(m & SLICE_FRESH_GONE)) {
    const unsigned long long h = atomicAdd(a->ticket, 1ULL);
    if (h < Bu) return (long long)h;
    atomicOr(a->sw, SLICE_FRESH_GONE);
  }
  m &= ~SLICE_FRESH_GONE;
  for (int tries = 0; m != 0 && tries < 6; ++tries) {
    const int g = __ffsll((long long)m) - 1;
    const uint2 ht = __ldcg((const uint2*)(a->sq + 2 * g));
    if (ht.x >= ht.y) {  // stale bit
      slice_mark_empty(a, g);
      m &= ~(1ULL << g);
      continue;
    }
    // Look before taking: a position whose id is not stored yet (its pusher sits between its two
    // stores, possibly in this very warp) is treated as not ready -- nobody ever waits for anybody.
    int* slot = a->squeue + (size_t)g * a->B + (ht.x % (unsigned)a->B);
    const int c = __ldcg(slot);
    if (c < 0) {
      m &= ~(1ULL << g);
      continue;
    }
    if (atomicCAS(a->sq + 2 * g, ht.x, ht.x + 1u) != ht.x) continue;  // somebody else took it: look again
    *(volatile int*)slot = -1;  // the queues are rings: at most B members are parked at any time
    if (ht.x + 1u >= ht.y) slice_mark_empty(a, g);
    *resume = 1;
    return (long long)c;
  }
  if (w.y >= Bu) *exhausted = 1;
  return -1;
}

// Parked state -> shared memory + scalars.  All loads are issued before the first use: the parked
// states are long out of L2 by the time they are needed again, so the latency must be paid once.
template <int NBW, int NSTATE>
static __device__ __noinline__ void slice_restore(const SolveArgs* a, long long b, double* sm_bw, double* sm_state, int stride,
                                                  SliceScalars* io) {
  __threadfence();
  constexpr int TOT = slice_ctx_doubles(NBW, NSTATE);
  const double2* cx = (const double2*)(a->ctx + (size_t)b * TOT);
  double buf[TOT];
#pragma unroll
  for (int e = 0; e < TOT / 2; ++e) {
    const double2 v = __ldcg(cx + e);
    buf[2 * e] = v.x;
    buf[2 * e + 1] = v.y;
  }
#pragma unroll
  for (int e = 0; e < NBW; ++e) sm_bw[e * stride] = buf[e];
#pragma unroll
  for (int e = 0; e < NSTATE; ++e) sm_state[e * stride] = buf[NBW + e];
  io->t = buf[NBW + NSTATE];
  io->dt_next = buf[NBW + NSTATE + 1];
  io->le_prev = buf[NBW + NSTATE + 2];
  io->sigma_state = buf[NBW + NSTATE + 3];
  io->k_next = __double_as_longlong(buf[NBW + NSTATE + 4]);
  io->n_acc = __double_as_longlong(buf[NBW + NSTATE + 5]);
  io->n_rej = __double_as_longlong(buf[NBW + NSTATE + 6]);
  io->n_att = __double_as_longlong(buf[NBW + NSTATE + 7]);
}

// A member has used up its quantum of attempted steps while in queue group g (its checkpoint interval,
// coarsened to at most 63 groups).  If a fresh member or a ready member of a group <= g is waiting, park
// this one and report 1 (the lane then takes the waiting one); else the lane keeps it.
static __device__ __noinline__ int slice_park_if_waiting(const SolveArgs* a, long long b, int g, const double* sm_bw, int nbw,
                                                         const double* sm_state, int nstate, int stride,
                                                         const SliceScalars* io) {
  const unsigned long long m = __ldcg(a->sw);
  const unsigned long long upto = (g >= 62) ? ~SLICE_FRESH_GONE : ((2ULL << g) - 1ULL);
  if ((m & SLICE_FRESH_GONE) && !(m & upto)) return 0;
  double* cx = a->ctx + (size_t)b * slice_ctx_doubles(nbw, nstate);
  for (int e = 0; e < nbw; ++e) cx[e] = sm_bw[e * stride];
  for (int e = 0; e < nstate; ++e) cx[nbw + e] = sm_state[e * stride];
  cx += nbw + nstate;
  cx[0] = io->t;
  cx[1] = io->dt_next;
  cx[2] = io->le_prev;
  cx[3] = io->sigma_state;
  long long* ci = (long long*)cx + 4;
  ci[0] = io->k_next;
  ci[1] = io->n_acc;
  ci[2] = io->n_rej;
  ci[3] = io->n_att;
  __threadfence();
  const unsigned pos = atomicAdd(a->sq + 2 * g + 1, 1u);
  *(volatile int*)(a->squeue + (size_t)g * a->B + (pos % (unsigned)a->B)) = (int)b;
  __threadfence();
  atomicOr(a->sw, 1ULL << g);
  return 1;
}

// Long members: keep the number of hand-overs per member bounded (about eight) whatever its length.
// The total number of attempted steps is extrapolated from the part of [t0, t1] covered so far and
// the quantum grows to about an eighth of it (a finer one was measured slower: every hand-over stalls
// the warp).  Evaluated at multiples of the base quantum only.
static __device__ __noinline__ bool slice_quantum_reached(const SolveArgs& a, double t, long long n_att, long long b) {
  const double* ts = grid_row(a, b);
  const double t0 = ts[0], t1 = ts[a.K - 1];
  const double frac = fmax((t - t0) / (t1 - t0), 1e-3);
  const double target = 0.125 * (double)n_att / frac;
  long long q = a.slice_mask + 1;
  while ((double)q < target && q < (1LL << 40)) q <<= 1;
  return ((n_att + b * 7919LL) & (q - 1)) == 0;
}

template <int V>
struct IntTag {
  static constexpr int value = V;
};

template <int N>
struct Binom {
  // flipped Pascal matrix A1[i][j] = C(nu-i, nu-j)
  __host__ __device__ static constexpr double at(int i, int j) {
    int a = N - 1 - i, b = N - 1 - j;
    if (b < 0 || b > a) return 0.0;
    double c = 1.0;
    for (int k = 1; k <= b; ++k) c = c * (double)(a - b + k) / (double)k;
    return c;
  }
};

__host__ __device__ constexpr double factorial(int k) {
  double f = 1.0;
  for (int i = 2; i <= k; ++i) f *= (double)i;
  return f;
}

// number of doubles one backward conditional / one marginal occupies
template <int N, int D>
struct Layout {
  static constexpr int NT = N * (N + 1) / 2;
  static constexpr int BW = N * N + N * D + NT;   // G (full), g, Lam (lower, packed)
  static constexpr int MARG = N * D + NT;         // mean, chol (lower, packed)
  static constexpr int PEND = MARG + 3;           // + t1, sigma1, time of checkpoint k_next (see ck_cached)
  static constexpr int SLOT_FIX = BW + MARG;      // fixed-point slot: cond (+ terminal marginal in slot 0)
  static constexpr int SLOT_FILT = MARG;          // filter slot: the marginal itself
  __host__ __device__ static constexpr int tri(int i, int j) { return i * (i + 1) / 2 + j; }  // j <= i
};

// butterfly sum over the GROUP lanes of one IVP (all lanes end with the same bits)
template <int GROUP>
PN_DEV double group_sum(double v, unsigned gmask) {
#pragma unroll
  for (int off = GROUP / 2; off >= 1; off >>= 1) v = v + __shfl_xor_sync(gmask, v, off);
  return v;
}

// Vector field for the lane-per-dimension kernels: every lane holds ITS dimension's predicted
// (u, u', ...) and gets back ITS component of f.  Default: gather everything with shuffles,
// evaluate the whole field, select the own component.  t: the time of the evaluation (read by
// time-dependent problems only).
template <class Prob, int GROUP>
struct GroupVf {
  PN_DEV static double eval(const double* own /*[Q]*/, int sub, int base, unsigned gmask, double t, const double* par) {
    constexpr int DT = Prob::D, Q = Prob::Q;
    double u[Q * DT], f[DT];
#pragma unroll
    for (int k = 0; k < Q; ++k)
#pragma unroll
      for (int c = 0; c < DT; ++c) u[k * DT + c] = __shfl_sync(gmask, own[k], base + c);
    vf_at<Prob>(u, t, par, f);
    double r = f[0];
#pragma unroll
    for (int c = 1; c < DT; ++c) r = (sub == c) ? f[c] : r;
    return r;
  }
};

// Pleiades: lane c < 7 owns x_c, lane 7 + i owns y_i; each lane sums its 6 pair terms.
template <int GROUP>
struct GroupVf<Pleiades, GROUP> {
  PN_DEV static double eval(const double* own, int sub, int base, unsigned gmask, double, const double*) {
    const int i = (sub < 7) ? sub : ((sub < 14) ? sub - 7 : 0);
    const bool isx = sub < 7;
    const double xi = __shfl_sync(gmask, own[0], base + i);
    const double yi = __shfl_sync(gmask, own[0], base + 7 + i);
    double acc = 0.0;
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      const double xj = __shfl_sync(gmask, own[0], base + j);
      const double yj = __shfl_sync(gmask, own[0], base + 7 + j);
      const double dx = xj - xi, dy = yj - yi;
      const double pw = inv_pow32(fma(dy, dy, dx * dx));
      const double term = fma((double)(j + 1), pw * (isx ? dx : dy), acc);
      acc = (j == i) ? acc : term;  // nan_to_num(0/0) = 0 (ivps.py:95-96)
    }
    return acc;
  }
};

// Brusselator: lane i < N owns u_i, lane N + i owns v_i; nearest-neighbour stencil by shuffles.
template <int NPTS, int GROUP>
struct GroupVf<Brusselator<NPTS>, GROUP> {
  PN_DEV static double eval(const double* own, int sub, int base, unsigned gmask, double, const double* par) {
    const bool isu = sub < NPTS;
    const int i = isu ? sub : sub - NPTS;
    const double c = par[0] * (double)((NPTS + 1) * (NPTS + 1));
    const double me = own[0];
    const double lft = __shfl_sync(gmask, me, base + ((sub > 0) ? sub - 1 : 0));
    const double rgt = __shfl_sync(gmask, me, base + ((sub + 1 < GROUP) ? sub + 1 : GROUP - 1));
    const double oth = __shfl_sync(gmask, me, base + (isu ? ((sub + NPTS < GROUP) ? sub + NPTS : sub) : sub - NPTS));
    const double pad = isu ? 1.0 : 3.0;
    const double l = (i == 0) ? pad : lft;
    const double r = (i == NPTS - 1) ? pad : rgt;
    const double ui = isu ? me : oth, vi = isu ? oth : me;
    const double uuv = (ui * ui) * vi;
    const double lap = fma(-2.0, me, l + r);
    return isu ? fma(c, lap, fma(-4.0, ui, 1.0 + uuv)) : fma(c, lap, fma(3.0, ui, -uuv));
  }
};


// ---- PIPE = 1 (CTA-per-IVP kernel, fixed-point strategy, at most one member per SM): a fifth warp owns the
// running backward conditional.  The n x n factor arithmetic of one attempted step is a single dependent chain
// (every thread of the CTA replicates it), and two fifths of that chain -- the right block of the predict QR,
// the back substitution for the smoothing gain, the merge products and the merge QR -- are not needed by the
// NEXT step at all.  The main warps (THREADS threads) keep the filter path: predict the mean, residual, left
// block of the predict QR, correction, error norm, controller.  Once per iteration they publish the reflectors
// of the predict QR; the backward warp applies them to the right block, solves for X (which the main warps need
// for the offset g of the conditional: ready before their pass 3), merges with the running conditional while
// the main warps are already in the next step, and carries out what the bookkeeping decided (commit / reset /
// emit to a checkpoint slot) from a small op list.  Hand-over through shared memory + named barriers
// (producer: bar.arrive, consumer: bar.sync).  Every quantity is computed by the same operations in the same
// order as in the PIPE = 0 kernel: results are bit-identical.
namespace pipe {
constexpr int BAR_JOB = 1, BAR_X = 2, BAR_ACT = 3, BAR_MAIN = 4;
enum : int { OP_COMMIT = 1, OP_RESET = 2, OP_STORE_MERGED = 3, OP_STORE_RUNNING = 4, OP_STORE_IDENTITY = 5 };
constexpr int MAX_OPS = 24;
PN_DEV void bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
// (shared-memory stores of the arriving thread are ordered before the completion of the barrier: the
// producer / consumer use of named barriers, no fence needed)
PN_DEV void bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
template <int N>
struct Mail {
  static constexpr int NT = N * (N + 1) / 2;
  // job: main warps -> backward warp (written before BAR_JOB)
  double BL[N * N];        // [i][j]: row i of the bottom-left block after the QR = tail of reflector j
  double v0[N], g[N];      // reflector scalars
  double RY[N * N];        // R factor (upper triangle)
  double Lp[NT];           // preconditioned state factor L_p (lower, packed): the right block starts as L_p^T
  double p[N], pinv[N];
  int reset, exit_;
  // backward warp -> main warps (written before BAR_X)
  double X[N * N];         // X = RY^{-1} R12
  int cur;                 // which buffer of R holds the running conditional
  double R[2][N * N + NT]; // running conditional [G | Lam packed]; the other buffer receives the merged one
  double gain[N];          // main warp 0 -> the other main warps
  unsigned long long* stats;  // PN_PIPE_STATS builds: the workspace header's statistics words
  double red[2][8];        // main warps: warp sums of a CTA reduction, double-buffered (one barrier per reduction)
  // bookkeeping: main warps -> backward warp (written before BAR_ACT)
  int nops;
  int op[MAX_OPS];
  double* dst[MAX_OPS];
};
template <int N>
PN_DEV Mail<N>& mail() {
  __shared__ Mail<N> m;
  return m;
}

template <int N>
__device__ __noinline__ void backward_warp(Mail<N>& M, const int nmain) {
  using Lay = Layout<N, 1>;
  constexpr int NT = Mail<N>::NT, OFF_LAM = N * N + N;
  const int lane = threadIdx.x & 31, total = nmain + 32;
  int cur = 0;
  auto set_identity = [&](double* R) {
    for (int e = lane; e < N * N + NT; e += 32) R[e] = (e < N * N && (e / N) == (e % N)) ? 1.0 : 0.0;
    __syncwarp();
  };
  // slot factor part: [G (n x n) | n zeros | Lam (packed)]
  auto store_factor = [&](double* dst, const double* R) {
    for (int e = lane; e < N * N + N + NT; e += 32)
      dst[e] = (R == nullptr) ? ((e < N * N && (e / N) == (e % N)) ? 1.0 : 0.0)
                              : ((e < N * N) ? R[e] : ((e < OFF_LAM) ? 0.0 : R[N * N + (e - OFF_LAM)]));
  };
#ifdef PN_PIPE_STATS
  long long st_job = 0, st_act = 0, st_c0 = 0, st_x = 0, st_merge = 0;
#define PN_PIPE_T0() st_c0 = clock64()
#define PN_PIPE_T1(acc) acc += clock64() - st_c0
#else
#define PN_PIPE_T0()
#define PN_PIPE_T1(acc)
#endif
  for (;;) {
    PN_PIPE_T0();
    bar_sync(BAR_JOB, total);
    PN_PIPE_T1(st_job);
#ifdef PN_PIPE_STATS
    if (M.exit_ && lane == 0 && M.stats) {
      atomicAdd(M.stats + 9, (unsigned long long)st_job);
      atomicAdd(M.stats + 10, (unsigned long long)st_act);
      atomicAdd(M.stats + 12, (unsigned long long)st_x);
      atomicAdd(M.stats + 13, (unsigned long long)st_merge);
    }
#endif
    if (M.exit_) return;
    if (M.reset) set_identity(M.R[cur]);
    PN_PIPE_T0();
    double BL[N][N], BR[N][N], R12[N][N], RY[N][N], v0[N], gg[N], p[N], pinv[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      v0[i] = M.v0[i];
      gg[i] = M.g[i];
      p[i] = M.p[i];
      pinv[i] = M.pinv[i];
#pragma unroll
      for (int j = 0; j < N; ++j) {
        BL[i][j] = M.BL[i * N + j];
        RY[i][j] = (j >= i) ? M.RY[i * N + j] : 0.0;
        BR[i][j] = (i <= j) ? M.Lp[Lay::tri(j, i)] : 0.0;  // L_p^T (upper)
      }
    }
    // the reflectors of the predict QR applied to the right block [0 ; L_p^T] (pn_scalar_kernel: "right block columns")
#pragma unroll
    for (int j = 0; j < N; ++j) {
#pragma unroll
      for (int c = 0; c < N; ++c) {
        double w = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) {
          if (j == 0 && i > c) continue;  // still structurally zero
          w = fma(BL[i][j], BR[i][c], w);
        }
        const double f = w * gg[j];
        R12[j][c] = fma(f, v0[j], 0.0);
#pragma unroll
        for (int i = 0; i < N; ++i) BR[i][c] = fma(f, BL[i][j], BR[i][c]);
      }
    }
    // X = RY^{-1} R12 (back substitution); G_p = X^T
    double X[N][N];
#pragma unroll
    for (int i = N - 1; i >= 0; --i) {
      const double inv = rcp_raw(RY[i][i]);
#pragma unroll
      for (int c = 0; c < N; ++c) {
        double acc = R12[i][c];
#pragma unroll
        for (int k = i + 1; k < N; ++k) acc = fma(-RY[i][k], X[k][c], acc);
        X[i][c] = acc * inv;
      }
    }
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int c = 0; c < N; ++c) M.X[i * N + c] = X[i][c];
      M.cur = cur;
    }
    bar_arrive(BAR_X, total);
    PN_PIPE_T1(st_x);
    PN_PIPE_T0();
    // new conditional (un-preconditioned) and the merge with the running one (A.4)
    double Gn[N][N], Ln[N][N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
      for (int j = 0; j < N; ++j) Gn[i][j] = (p[i] * X[j][i]) * pinv[j];
#pragma unroll
      for (int j = 0; j < N; ++j) Ln[i][j] = p[i] * BR[j][i];
    }
    const double* Rc = M.R[cur];
    double* Rn = M.R[cur ^ 1];
    double G1[N][N], Mt[N][N], Mb[N][N];
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int j = 0; j < N; ++j) G1[i][j] = Rc[i * N + j];
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
      for (int j = 0; j < N; ++j) {
        double acc = G1[i][0] * Gn[0][j];
#pragma unroll
        for (int k = 1; k < N; ++k) acc = fma(G1[i][k], Gn[k][j], acc);
        if (lane == 0) Rn[i * N + j] = acc;  // merged G
      }
    }
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int j = 0; j < N; ++j) {
        double acc = G1[i][0] * Ln[0][j];
#pragma unroll
        for (int k = 1; k < N; ++k) acc = fma(G1[i][k], Ln[k][j], acc);
        Mt[j][i] = acc;
      }
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = 0; i < N; ++i) Mb[i][j] = (i <= j) ? Rc[N * N + Lay::tri(j, i)] : 0.0;
#pragma unroll
    for (int j = 0; j < N; ++j) {
      double sigma2 = 0.0;
#pragma unroll
      for (int i = j + 1; i < N; ++i) sigma2 = fma(Mt[i][j], Mt[i][j], sigma2);
#pragma unroll
      for (int i = 0; i <= j; ++i) sigma2 = fma(Mb[i][j], Mb[i][j], sigma2);
      const Reflector rf = make_reflector(Mt[j][j], sigma2);
#pragma unroll
      for (int c = j + 1; c < N; ++c) {
        double w = 0.0;
#pragma unroll
        for (int i = j + 1; i < N; ++i) w = fma(Mt[i][j], Mt[i][c], w);
#pragma unroll
        for (int i = 0; i <= j; ++i) w = fma(Mb[i][j], Mb[i][c], w);
        w = fma(rf.v0, Mt[j][c], w);
        const double f = w * rf.ng;
        Mt[j][c] = fma(f, rf.v0, Mt[j][c]);
#pragma unroll
        for (int i = j + 1; i < N; ++i) Mt[i][c] = fma(f, Mt[i][j], Mt[i][c]);
#pragma unroll
        for (int i = 0; i <= j; ++i) Mb[i][c] = fma(f, Mb[i][j], Mb[i][c]);
      }
      Mt[j][j] = rf.beta;
    }
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) Rn[N * N + Lay::tri(i, j)] = Mt[j][i];  // merged Lam (lower)
    }
    __syncwarp();
    PN_PIPE_T1(st_merge);
    // what the bookkeeping of this iteration decided
    PN_PIPE_T0();
    bar_sync(BAR_ACT, total);
    PN_PIPE_T1(st_act);
    const int nops = M.nops;
    for (int o = 0; o < nops; ++o) {
      const int op = M.op[o];
      double* dst = M.dst[o];
      if (op == OP_COMMIT) {
        cur ^= 1;
      } else if (op == OP_RESET) {
        set_identity(M.R[cur]);
      } else if (op == OP_STORE_MERGED) {
        store_factor(dst, M.R[cur ^ 1]);
      } else if (op == OP_STORE_RUNNING) {
        store_factor(dst, M.R[cur]);
      } else if (op == OP_STORE_IDENTITY) {
        store_factor(dst, nullptr);
      }
    }
    __syncwarp();
  }
}
}  // namespace pipe


// ---- PAIR = 1 (thread-per-IVP kernels, fixed-point strategy, small ensembles): the backward warp idea of the
// PIPE build, lane by lane.  Below ~19k members every SM sub-partition holds at most one warp of the
// thread-per-IVP kernel and the launch takes 16k steps x the latency of ONE step whatever the ensemble size
// (DESIGN 3.6).  Here a CTA is THREADS "filter" lanes + THREADS "backward" lanes: lane l of filter warp w and
// lane l of backward warp w serve the same IVP.  The filter lane keeps predict mean / left block of the predict
// QR / correction / error norm / controller and the state; once per iteration it leaves the reflectors of the
// predict QR and what its bookkeeping decided (a short op list) in a per-lane mailbox in shared memory.  The
// backward lane -- one iteration behind -- applies the reflectors to the right block, solves for the smoothing
// gain, forms the new conditional, merges it into the running one (which it owns) and executes the ops.  Two
// named barriers per warp pair and iteration (job ready: filter arrives / backward waits; mailbox free: the
// other way round).  Same operations in the same order as the PAIR = 0 kernel: bit-identical results.
namespace pair {
constexpr int MAX_OPS = 8;
template <int N, int D>
struct Mailbox {
  static constexpr int NT = N * (N + 1) / 2;
  // doubles per lane
  static constexpr int O_BL = 0, O_V0 = O_BL + N * N, O_G = O_V0 + N, O_RY = O_G + N, O_LP = O_RY + NT, O_P = O_LP + NT,
                       O_PINV = O_P + N, O_MP = O_PINV + N, O_MEP = O_MP + N * D, JOB_RAW = O_MEP + N * D,
                       JOB = (JOB_RAW + 1) & ~1,  // the job travels as 16-byte pairs: [pair][lane][2]
                       O_DST = JOB,               // op destinations: 64-bit pointers in double-sized cells, [cell][lane]
                       DOUBLES = O_DST + 2 * MAX_OPS;
  // The op list is double-buffered (parity of the iteration): the backward lane reads it AFTER its merge, when
  // the filter lane may already be writing the next one; the job itself is taken out of the mailbox at once.
  // ints per lane: [0] reset-before flag (part of the job), then per parity [number of ops, op codes ...]
  static constexpr int INTS = 1 + 2 * (1 + MAX_OPS);
  __host__ __device__ static constexpr int i_nops(int q) { return 1 + q * (1 + MAX_OPS); }
  static constexpr int BYTES_PER_LANE = DOUBLES * 8 + INTS * 4;
};

template <int N, int D, int THREADS>
__device__ __noinline__ void backward_lanes(double* s_bw, double* s_job, int* s_int, const volatile int* s_exit) {
  using Lay = Layout<N, D>;
  using MB = Mailbox<N, D>;
  constexpr int OFF_G = 0, OFF_g = N * N, OFF_LAM = N * N + N * D;
  // backward warp pw serves filter warp (pw + NW / 2) mod NW: filter warp w issues from scheduler w mod 4, its
  // backward lanes from the scheduler opposite, so that a lone pair (small ensembles) does not share one
  constexpr int NW = THREADS / 32;
  const int lraw = threadIdx.x - THREADS;
  const int w = ((lraw >> 5) + NW / 2) % NW, l = w * 32 + (lraw & 31);
#define PBW(e) s_bw[(e) * THREADS + l]
#define PJ(e) s_job[(e) * THREADS + l]
#define PI(e) s_int[(e) * THREADS + l]
  int q = 0;  // parity of the job
  for (;;) {
    pipe::bar_sync(1 + w, 64);
    if (s_exit[w]) return;
    double BL[N][N], BR[N][N], R12[N][N], RY[N][N], v0[N], gg[N], p[N], pinv[N], m_p[N][D], m_ext_p[N][D];
    {
      double jb[MB::JOB];
#pragma unroll
      for (int e = 0; e < MB::JOB / 2; ++e) {
        const double2 v = reinterpret_cast<const double2*>(s_job)[e * THREADS + l];
        jb[2 * e] = v.x;
        jb[2 * e + 1] = v.y;
      }
#pragma unroll
      for (int i = 0; i < N; ++i) {
        v0[i] = jb[MB::O_V0 + i];
        gg[i] = jb[MB::O_G + i];
        p[i] = jb[MB::O_P + i];
        pinv[i] = jb[MB::O_PINV + i];
#pragma unroll
        for (int c = 0; c < D; ++c) {
          m_p[i][c] = jb[MB::O_MP + i * D + c];
          m_ext_p[i][c] = jb[MB::O_MEP + i * D + c];
        }
#pragma unroll
        for (int j = 0; j < N; ++j) {
          BL[i][j] = jb[MB::O_BL + i * N + j];
          RY[i][j] = (j >= i) ? jb[MB::O_RY + Lay::tri(j, i)] : 0.0;
          BR[i][j] = (i <= j) ? jb[MB::O_LP + Lay::tri(j, i)] : 0.0;  // L_p^T (upper)
        }
      }
    }
    const int reset = PI(0);
    pipe::bar_arrive(1 + THREADS / 32 + w, 64);  // mailbox free
    if (reset) {
#pragma unroll
      for (int e = 0; e < Lay::BW; ++e) PBW(e) = 0.0;
#pragma unroll
      for (int i = 0; i < N; ++i) PBW(OFF_G + i * N + i) = 1.0;
    }
    // right block of the predict QR
#pragma unroll
    for (int j = 0; j < N; ++j) {
#pragma unroll
      for (int c = 0; c < N; ++c) {
        double wv = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) {
          if (j == 0 && i > c) continue;  // still structurally zero
          wv = fma(BL[i][j], BR[i][c], wv);
        }
        const double f = wv * gg[j];
        R12[j][c] = fma(f, v0[j], 0.0);
#pragma unroll
        for (int i = 0; i < N; ++i) BR[i][c] = fma(f, BL[i][j], BR[i][c]);
      }
    }
    double X[N][N];
#pragma unroll
    for (int i = N - 1; i >= 0; --i) {
      const double inv = rcp_raw(RY[i][i]);
#pragma unroll
      for (int c = 0; c < N; ++c) {
        double acc = R12[i][c];
#pragma unroll
        for (int k = i + 1; k < N; ++k) acc = fma(-RY[i][k], X[k][c], acc);
        X[i][c] = acc * inv;
      }
    }
    double Gn[N][N], gn[N][D], Ln[N][N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
      for (int c = 0; c < D; ++c) {
        double acc = m_p[i][c];
#pragma unroll
        for (int k = 0; k < N; ++k) acc = fma(-X[k][i], m_ext_p[k][c], acc);
        gn[i][c] = p[i] * acc;
      }
#pragma unroll
      for (int j = 0; j < N; ++j) Gn[i][j] = (p[i] * X[j][i]) * pinv[j];
#pragma unroll
      for (int j = 0; j < N; ++j) Ln[i][j] = p[i] * BR[j][i];
    }
    // merge with the running conditional (A.4)
    double Gm[N][N], gm[N][D], Lm[N][N];
    {
      double G1[N][N];
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) G1[i][j] = PBW(OFF_G + i * N + j);
#pragma unroll
      for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = 0; j < N; ++j) {
          double acc = G1[i][0] * Gn[0][j];
#pragma unroll
          for (int k = 1; k < N; ++k) acc = fma(G1[i][k], Gn[k][j], acc);
          Gm[i][j] = acc;
        }
#pragma unroll
        for (int c = 0; c < D; ++c) {
          double acc = PBW(OFF_g + i * D + c);
#pragma unroll
          for (int k = 0; k < N; ++k) acc = fma(G1[i][k], gn[k][c], acc);
          gm[i][c] = acc;
        }
      }
      double Mt[N][N], Mb[N][N];
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) {
          double acc = G1[i][0] * Ln[0][j];
#pragma unroll
          for (int k = 1; k < N; ++k) acc = fma(G1[i][k], Ln[k][j], acc);
          Mt[j][i] = acc;
        }
#pragma unroll
      for (int j = 0; j < N; ++j)
#pragma unroll
        for (int i = 0; i < N; ++i) Mb[i][j] = (i <= j) ? PBW(OFF_LAM + Lay::tri(j, i)) : 0.0;
#pragma unroll
      for (int j = 0; j < N; ++j) {
        double sigma2 = 0.0;
#pragma unroll
        for (int i = j + 1; i < N; ++i) sigma2 = fma(Mt[i][j], Mt[i][j], sigma2);
#pragma unroll
        for (int i = 0; i <= j; ++i) sigma2 = fma(Mb[i][j], Mb[i][j], sigma2);
        const Reflector rf = make_reflector(Mt[j][j], sigma2);
#pragma unroll
        for (int c = j + 1; c < N; ++c) {
          double wv = 0.0;
#pragma unroll
          for (int i = j + 1; i < N; ++i) wv = fma(Mt[i][j], Mt[i][c], wv);
#pragma unroll
          for (int i = 0; i <= j; ++i) wv = fma(Mb[i][j], Mb[i][c], wv);
          wv = fma(rf.v0, Mt[j][c], wv);
          const double f = wv * rf.ng;
          Mt[j][c] = fma(f, rf.v0, Mt[j][c]);
#pragma unroll
          for (int i = j + 1; i < N; ++i) Mt[i][c] = fma(f, Mt[i][j], Mt[i][c]);
#pragma unroll
          for (int i = 0; i <= j; ++i) Mb[i][c] = fma(f, Mb[i][j], Mb[i][c]);
        }
        Mt[j][j] = rf.beta;
      }
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) Lm[i][j] = (j <= i) ? Mt[j][i] : 0.0;
    }
    // what the filter lane's bookkeeping decided (per lane: may diverge)
    const int nops = PI(MB::i_nops(q));
    for (int o = 0; o < nops; ++o) {
      {
        const int op = PI(MB::i_nops(q) + 1 + o);
        double* d_ = (double*)__double_as_longlong(PJ(MB::O_DST + q * MAX_OPS + o));
        if (op == pipe::OP_COMMIT) {
#pragma unroll
          for (int i = 0; i < N; ++i) {
#pragma unroll
            for (int j = 0; j < N; ++j) PBW(OFF_G + i * N + j) = Gm[i][j];
#pragma unroll
            for (int c = 0; c < D; ++c) PBW(OFF_g + i * D + c) = gm[i][c];
#pragma unroll
            for (int j = 0; j <= i; ++j) PBW(OFF_LAM + Lay::tri(i, j)) = Lm[i][j];
          }
        } else if (op == pipe::OP_RESET) {
#pragma unroll
          for (int e = 0; e < Lay::BW; ++e) PBW(e) = 0.0;
#pragma unroll
          for (int i = 0; i < N; ++i) PBW(OFF_G + i * N + i) = 1.0;
        } else if (op == pipe::OP_STORE_MERGED) {
#pragma unroll
          for (int i = 0; i < N; ++i) {
#pragma unroll
            for (int j = 0; j < N; ++j) d_[OFF_G + i * N + j] = Gm[i][j];
#pragma unroll
            for (int c = 0; c < D; ++c) d_[OFF_g + i * D + c] = gm[i][c];
#pragma unroll
            for (int j = 0; j <= i; ++j) d_[OFF_LAM + Lay::tri(i, j)] = Lm[i][j];
          }
        } else if (op == pipe::OP_STORE_RUNNING) {
#pragma unroll
          for (int e = 0; e < Lay::BW; ++e) d_[e] = PBW(e);
        } else if (op == pipe::OP_STORE_IDENTITY) {
#pragma unroll
          for (int e = 0; e < Lay::BW; ++e) d_[e] = 0.0;
#pragma unroll
          for (int i = 0; i < N; ++i) d_[OFF_G + i * N + i] = 1.0;
        }
      }
    }
    __syncwarp();
    q ^= 1;
  }
#undef PBW
#undef PJ
#undef PI
}
}  // namespace pair

#ifndef PN_MINBLOCKS
#define PN_MINBLOCKS 2
#endif
// GROUP = 1: one thread per IVP, the factor is shared by the Prob::D mean columns the thread holds.
// GROUP > 1: GROUP lanes per IVP, lane `sub` owns ODE dimension `sub` (one mean column) and a full
//            n x n factor set: per-dimension factors for BDIAG (blockdiag factorisation), replicated
//            identical factors for the isotropic factorisation.
// WIDE = 1: one CTA per IVP for isotropic problems with a large runtime dimension d (Brusselator,
//           d = 2N up to 2048).  Every thread carries the same n x n factor state and executes the
//           same factor arithmetic as a thread-per-IVP lane; the n x d mean arrays live in global
//           memory (L2 resident) and each thread owns the columns c = tid, tid + THREADS, ...;
//           norms are reduced over the CTA.  Prob::D is a dummy (1) in this mode.
template <class Prob, int NU, int STRAT, int GROUP, int BDIAG, int THREADS, int WIDE = 0, int SLICE = 0, int PIPE = 0, int PAIR = 0>
__global__ void __launch_bounds__(THREADS * (1 + PAIR) + 64 * PIPE, (PIPE || PAIR) ? 1 : PN_MINBLOCKS)
    pn_scalar_kernel(const __grid_constant__ SolveArgs a) {
  constexpr int N = NU + 1, DT = Prob::D, D = (GROUP > 1) ? 1 : DT, Q = Prob::Q, P = (Prob::P > 0 ? Prob::P : 1);
  constexpr int DV = (GROUP > 1) ? DT : 1;  // lanes ("virtual members") per IVP that own state
  static_assert(GROUP == 1 || (GROUP >= DT && (GROUP & (GROUP - 1)) == 0 && GROUP <= 32), "bad GROUP");
  static_assert(GROUP > 1 || BDIAG == 0, "blockdiag with one thread per IVP only makes sense for d == 1");
  using Lay = Layout<N, D>;
  constexpr bool FIX = (STRAT == 1);
  constexpr int SLOT = FIX ? Lay::SLOT_FIX : Lay::SLOT_FILT;
  constexpr double TIME_EPS = 10.0 * 2.220446049250313e-16;
  static_assert(!PIPE || (WIDE && STRAT == 1 && GROUP == 1), "PIPE: CTA-per-IVP kernel with the fixed-point strategy");
  if constexpr (PIPE) {
    // warps 0 .. THREADS/32 - 1: main; the next warp exits at once (warp w runs on sub-partition w mod 4: the
    // backward warp must not share the fp64 pipe of main warp 0, the one that carries the factor arithmetic);
    // the last warp is the backward warp
    if (threadIdx.x >= THREADS) {
      if (threadIdx.x >= THREADS + 32) pipe::backward_warp<N>(pipe::mail<N>(), THREADS);
      return;
    }
  }
  // PIPE: the n x n factor arithmetic of the filter path runs on main warp 0 only (the other main warps sweep
  // their mean columns and get the gain through shared memory): sub-partitions 1 .. 3 stay free for the
  // backward warp.  Otherwise every thread carries it.
  const bool pipe_F = !PIPE || (threadIdx.x < 32);
  // barrier over the threads that run the step (PIPE: the main warps only)
  auto cta_sync = [&]() {
    if constexpr (PIPE) pipe::bar_sync(pipe::BAR_MAIN, THREADS); else __syncthreads();
  };
  bool pipe_reset = false;  // PIPE: the next job is the first of a member
  int pipe_nops = 0;        // PIPE: ops queued for the backward warp in this iteration
  int pipe_red_phase = 0;   // PIPE: which reduction scratch buffer the next CTA reduction uses
  // PIPE: the checkpoint time the bookkeeping compares with, kept in a register between checkpoints (every
  // iteration asked global memory for it twice, in the middle of the serial part of the step)
  long long pipe_ck_k = -1;
  double pipe_ck_t = 0.0;
#ifdef PN_PIPE_STATS
  long long pipe_tm = clock64();
#define PN_MAIN_PHASE(w) do { if ((PIPE || PAIR) && tid == 0 && blockIdx.x == 0) { const long long now_ = clock64(); atomicAdd(a.ticket + (w), (unsigned long long)(now_ - pipe_tm)); pipe_tm = now_; } } while (0)
#else
#define PN_MAIN_PHASE(w) do { } while (0)
#endif
  // PIPE: preconditioner of the step the controller proposes, computed one iteration ahead (off the head of the chain)
  double pipe_spec_dt = __longlong_as_double(0x7ff8000000000000LL), pipe_spec_p[N], pipe_spec_pinv[N];

  int* pair_exit = nullptr;
  extern __shared__ double smem[];
  // [element][thread]
  double* s_bw = smem;                                       // BW * THREADS (fixed-point only)
  double* s_pend = smem + (FIX ? Lay::BW : 0) * THREADS;     // PEND * THREADS
  double* s_state = s_pend + Lay::PEND * THREADS;            // MARG * THREADS: hidden state (mean, factor)
  // PAIR: per-lane mailbox filter lane -> backward lane behind the state ([element][lane]); the running
  // conditional in s_bw belongs to the backward lanes
  static_assert(!PAIR || (GROUP == 1 && !WIDE && STRAT == 1 && !SLICE && !PIPE), "PAIR: thread-per-IVP fixed-point kernels");
  using PMB = pair::Mailbox<N, D>;
  double* s_job = s_state + Lay::MARG * THREADS;
  int* s_int = (int*)(s_job + PMB::DOUBLES * THREADS);
  if constexpr (PAIR) {
    __shared__ int s_pair_exit[THREADS / 32];
    if (threadIdx.x < THREADS / 32) s_pair_exit[threadIdx.x] = 0;
    __syncthreads();
    if (threadIdx.x >= THREADS) {
      pair::backward_lanes<N, D, THREADS>(s_bw, s_job, s_int, s_pair_exit);
      return;
    }
    pair_exit = s_pair_exit;
  }
  bool pair_started = false, pair_reset = false;
  int pair_nops = 0, pair_q = 1;
  const int tid = threadIdx.x;
#define SBW(e) s_bw[(e) * THREADS + tid]
#define SPEND(e) s_pend[(e) * THREADS + tid]
#define SCK SPEND(Lay::PEND - 1)
#define SM(i, c) s_state[((i) * D + (c)) * THREADS + tid]
#define SL(i, j) s_state[(N * D + Lay::tri(i, j)) * THREADS + tid]
  constexpr int OFF_G = 0, OFF_g = N * N, OFF_LAM = N * N + N * D;

  const double* LQ = a.lq;
  const double inv_sqrt_d = rcp(dsqrt((double)(WIDE ? a.wide_d : DT)));
  const int lane = threadIdx.x & 31;
  const int sub = (GROUP > 1) ? (lane & (GROUP - 1)) : 0;   // dimension owned by this lane
  const int base = lane - sub;                               // first lane of the group
  const unsigned gmask = (GROUP >= 32) ? 0xffffffffu : (((1u << GROUP) - 1u) << base);
  const bool real = WIDE ? false : (sub < DT);               // padding lanes carry no dimension; the wide
                                                             // mode has its own workspace stores
  const bool leader = WIDE ? (threadIdx.x == 0) : (sub == 0);  // writes the per-member counters
  const long long VB = WIDE ? 1 : a.B * DV;                  // (member, owned dimension) pairs; trajectory stride
  // ---- wide mode: dimensions, per-member arrays, shared staging buffers ---------------------
  const int wd = WIDE ? a.wide_d : 0;                        // runtime ODE dimension
  const int wN = wd / 2;                                     // Brusselator grid points
  constexpr int WSLOT = Lay::BW + Lay::NT;                   // factor part of a wide slot: (G, -, Lam) + L1
  const long long wslot = WIDE ? (long long)WSLOT + 2LL * N * wd : 0;  // + g [n][d] + m1 [n][d]
  double* s_ubuf = smem + ((FIX ? Lay::BW : 0) + Lay::PEND + Lay::MARG) * THREADS;  // [d] predicted u
  double* s_zbuf = s_ubuf + wd;                                                      // [d] residual z
  double* s_red = s_zbuf + wd;                                                       // [THREADS/32]
  double* s_means = s_red + THREADS / 32 + 2;                                        // [3][n][d] if wide_smem_means
  double* Wm = nullptr;    // state mean [n][d]
  double* Wg = nullptr;    // backward-conditional offset g [n][d]
  double* Wp = nullptr;    // pending (accepted, uncommitted) mean [n][d]
  double* wcond = nullptr; // this member's slots [K][wslot]
  auto block_sum = [&](double v) -> double {
    // fixed order: per-warp butterfly, then the warp sums added in warp order
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v = v + __shfl_xor_sync(0xffffffffu, v, off);
    if constexpr (PIPE) {
      // alternating scratch buffers: the barrier of the NEXT reduction separates this one's reads from the
      // writes of the one after it
      double* rb = pipe::mail<N>().red[pipe_red_phase];
      pipe_red_phase ^= 1;
      if ((tid & 31) == 0) rb[tid >> 5] = v;
      cta_sync();
      double r = rb[0];
#pragma unroll
      for (int w = 1; w < THREADS / 32; ++w) r = r + rb[w];
      return r;
    }
    cta_sync();
    if ((tid & 31) == 0) s_red[tid >> 5] = v;
    cta_sync();
    double r = s_red[0];
#pragma unroll
    for (int w = 1; w < THREADS / 32; ++w) r = r + s_red[w];
    return r;
  };

  // ---- per-lane persistent state --------------------------------------------------------
  bool have = false, exhausted = false, poll_now = true;
  static_assert(!SLICE || (GROUP == 1 && !WIDE), "time-sliced scheduling: thread-per-IVP kernels only");
  long long b = 0, vb = 0;
  double t = 0.0, dt_next = 0.0, le_prev = 0.0, sigma_state = 1.0, sigma0 = 1.0;
  double atol = a.atol, rtol = a.rtol;
  double par[P];
  int mode = MODE_STEP;
  long long k_next = 1, n_acc = 0, n_rej = 0, n_att = 0;
  // The time of checkpoint k_next (clamped to K - 1) in this member's grid.  PIPE / PAIR: cached in a register.
  // Otherwise in the lane's shared-memory slot SCK, which set_ck() rewrites whenever k_next or the member changes:
  // the step loop reads the slot and computes no row address (save_at + b * save_stride) of its own.
  auto set_ck = [&]() {
    if constexpr (!(PIPE || PAIR)) SCK = grid_row(a, b)[k_next < a.K ? k_next : a.K - 1];
  };
  auto ck_cached = [&]() -> double {
    if constexpr (PIPE || PAIR) {
      const long long kc = k_next < a.K ? k_next : a.K - 1;
      if (kc != pipe_ck_k) {
        pipe_ck_k = kc;
        pipe_ck_t = grid_row(a, b)[kc];
      }
      return pipe_ck_t;
    } else {
      return SCK;
    }
  };
  double mle_ss = 0.0;  // solver_mle: sum over the accepted steps of z^T S^-1 z / d
  // utilisation statistics (per warp, flushed once at exit): loop iterations, lane-iterations with
  // work, lane-iterations spent on checkpoint interpolation
  // (32-bit, per lane: three 64-bit warp-uniform counters fed by a ballot + popc each lived in local memory and
  // cost ~45 instructions and six local-memory round trips at the head of every iteration)
  unsigned stat_warp_iters = 0, stat_lane_iters = 0, stat_interp_iters = 0;
  const long long clk0 = clock64();

  // solution.output_scale at checkpoint k: one value per IVP, one per dimension for blockdiag
  auto emit_scale = [&](long long k, double v) {
    if (a.out_scale) {
      if (a.calibration == 2) v = sigma0 * ((n_acc > 0) ? dsqrt(mle_ss * rcp((double)n_acc)) : 1.0);  // running MLE
      if (BDIAG) {
        if (real) a.out_scale[(b * a.K + k) * DT + sub] = v;
      } else if (leader) {
        a.out_scale[b * a.K + k] = v;
      }
    }
  };

  for (;;) {
    if constexpr (PAIR) {
      // the job and the op list of the previous iteration are complete: hand them to the backward lanes
      __syncwarp();  // (lanes without a member come here early)
      if (pair_started) pipe::bar_arrive(1 + (tid >> 5), 64);
    }
    // ---- fetch a member ----------------------------------------------------------------
    // SLICE: a lane that has just lost its member looks for the next one at once; after an unsuccessful
    // look it only polls every eighth iteration (a poll is an L2 round trip that stalls the whole warp)
    if (!have && !exhausted && (!SLICE || poll_now || (stat_warp_iters & 7u) == 0)) {
      unsigned long long tk = 0;
      bool resume = false, claimed_none = false;
      if constexpr (SLICE) {
        int rs = 0, ex = 0;
        const long long c = slice_claim(&a, &rs, &ex);
        resume = rs != 0;
        exhausted = ex != 0;
        claimed_none = c < 0;
        poll_now = false;
        tk = claimed_none ? (unsigned long long)a.B : (unsigned long long)c;
      } else if constexpr (WIDE) {
        __shared__ unsigned long long s_ticket;
        cta_sync();
        if (tid == 0) s_ticket = atomicAdd(a.ticket, 1ULL);
        cta_sync();
        tk = s_ticket;
      } else {
        if (sub == 0) tk = atomicAdd(a.ticket, 1ULL);
        if (GROUP > 1) tk = __shfl_sync(gmask, tk, base);
      }
      if (tk < (unsigned long long)a.B) {
        b = (a.order && !SLICE) ? a.order[tk] : (long long)tk;
        vb = WIDE ? 0 : (b * DV + ((GROUP > 1 && real) ? sub : 0));
        have = true;
        double u0[Q * DT];
        if constexpr (!WIDE) {
#pragma unroll
          for (int i = 0; i < Q * DT; ++i) u0[i] = a.u0[b * (Q * DT) + i];
        }
#pragma unroll
        for (int i = 0; i < P; ++i) par[i] = (i < a.num_params) ? a.params[b * a.num_params + i] : 0.0;
        atol = a.tol ? a.tol[2 * b] : a.atol;
        rtol = a.tol ? a.tol[2 * b + 1] : a.rtol;
        sigma0 = a.sigma0 ? a.sigma0[b] : 1.0;
        if (!resume) {
        if constexpr (WIDE) {
          // state mean, backward-conditional offset and pending mean: shared memory when the launch has at
          // most one member per SM and they fit (each pass over the columns then saves an L2 round trip)
          Wm = a.wide_mean + (size_t)b * 3 * N * wd;
          Wg = Wm + (size_t)N * wd;
          Wp = Wg + (size_t)N * wd;
          if (a.wide_smem_means > 0) Wm = s_means;
          if (a.wide_smem_means > 1) Wg = s_means + (size_t)N * wd;
          if (a.wide_smem_means > 2) Wp = s_means + (size_t)2 * N * wd;
          wcond = a.cond + (size_t)b * a.K * wslot;
          // Taylor-mode initialisation of the Brusselator, one grid point per thread and order
          // (normalised coefficients C_k in Wm; the k-th coefficient of f only needs C_0..C_k)
          const double cc = par[0] * (double)((wN + 1) * (wN + 1));
          for (int c = tid; c < wd; c += THREADS) {
            Wm[c] = a.u0[b * wd + c];
            for (int i = 1; i < N; ++i) Wm[(size_t)i * wd + c] = 0.0;
            for (int i = 0; i < N; ++i) Wg[(size_t)i * wd + c] = 0.0;
          }
          cta_sync();
          for (int k = 0; k < NU; ++k) {
            for (int gi = tid; gi < wN; gi += THREADS) {
              double uj[N], vj[N], u2[N];
              for (int j = 0; j <= k; ++j) {
                uj[j] = Wm[(size_t)j * wd + gi];
                vj[j] = Wm[(size_t)j * wd + wN + gi];
              }
              for (int kk = 0; kk <= k; ++kk) {
                double acc = uj[0] * uj[kk];
                for (int j = 1; j <= kk; ++j) acc = fma(uj[j], uj[kk - j], acc);
                u2[kk] = acc;
              }
              double uuv = u2[0] * vj[k];
              for (int j = 1; j <= k; ++j) uuv = fma(u2[j], vj[k - j], uuv);
              const double padu = (k == 0) ? 1.0 : 0.0, padv = (k == 0) ? 3.0 : 0.0;
              const double ul = (gi == 0) ? padu : Wm[(size_t)k * wd + gi - 1];
              const double ur = (gi == wN - 1) ? padu : Wm[(size_t)k * wd + gi + 1];
              const double vl = (gi == 0) ? padv : Wm[(size_t)k * wd + wN + gi - 1];
              const double vr = (gi == wN - 1) ? padv : Wm[(size_t)k * wd + wN + gi + 1];
              const double lap_u = fma(-2.0, uj[k], ul + ur);
              const double lap_v = fma(-2.0, vj[k], vl + vr);
              const double fu = fma(cc, lap_u, fma(-4.0, uj[k], padu + uuv));
              const double fv = fma(cc, lap_v, fma(3.0, uj[k], -uuv));
              // row k+1 is not read by anybody during this sweep
              Wm[(size_t)(k + 1) * wd + gi] = fu / (double)(k + 1);
              Wm[(size_t)(k + 1) * wd + wN + gi] = fv / (double)(k + 1);
            }
            cta_sync();
          }
          {
            double fact = 1.0;
            for (int k = 0; k <= NU; ++k) {
              if (k > 0) fact *= (double)k;
              for (int c = tid; c < wd; c += THREADS) Wm[(size_t)k * wd + c] = fact * Wm[(size_t)k * wd + c];
            }
          }
          cta_sync();
#pragma unroll
          for (int i = 0; i < N; ++i) SM(i, 0) = 0.0;  // dummy register column
        } else {
          double tc[N][DT];
          taylor_init<Prob, NU>(u0, grid_row(a, b)[0], par, tc);
#pragma unroll
          for (int i = 0; i < N; ++i) {
            if constexpr (GROUP == 1) {
#pragma unroll
              for (int c = 0; c < D; ++c) SM(i, c) = tc[i][c];
            } else {
              double v = tc[i][0];
#pragma unroll
              for (int c = 1; c < DT; ++c) v = (sub == c) ? tc[i][c] : v;
              SM(i, 0) = v;
            }
          }
        }
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
          for (int j = 0; j <= i; ++j) SL(i, j) = 0.0;
        if (FIX && !PAIR) {
#pragma unroll
          for (int e = 0; e < Lay::BW; ++e) SBW(e) = 0.0;
#pragma unroll
          for (int i = 0; i < N; ++i) SBW(OFF_G + i * N + i) = 1.0;
        }
        pair_reset = true;  // PAIR: the backward lane resets its running conditional in front of the next job
        t = grid_row(a, b)[0];
        dt_next = a.dt0;
        le_prev = 0.0;
        sigma_state = sigma0;
        mode = MODE_STEP;
        k_next = 1;
        set_ck();
        pipe_reset = true;
        pipe_ck_k = -1;  // the cached checkpoint time belongs to the previous member's grid
        n_acc = n_rej = n_att = 0;
        mle_ss = 0.0;
        if (leader) a.n_accepted[b * a.K] = 0;
        emit_scale(0, sigma0);
        if (a.flags & FLAG_RECORD) {
          // trajectory layout: traj_t / traj_std [cap][B], traj_u [cap][d][B]; a lane of a lane-per-dimension
          // kernel writes its own dimension (a thread of the CTA-per-IVP kernel its own columns), the leader
          // the time and (its) standard deviation
          if (leader) {
            a.traj_t[b] = t;
            a.traj_std[b] = 0.0;
          }
          if constexpr (WIDE) {
            for (int c = tid; c < wd; c += THREADS) a.traj_u[(long long)c * a.B + b] = Wm[c];
          } else if (GROUP == 1) {
#pragma unroll
            for (int c = 0; c < D; ++c) a.traj_u[(long long)c * a.B + b] = SM(0, c);
          } else if (real) {
            a.traj_u[(long long)sub * a.B + b] = SM(0, 0);
          }
        }
        if constexpr (WIDE) {
          if (!FIX) {  // filter: slot 0 holds the initial marginal (factor part zero)
            for (int e = tid; e < WSLOT; e += THREADS) wcond[e] = 0.0;
            for (int e = tid; e < N * wd; e += THREADS) wcond[WSLOT + (size_t)N * wd + e] = Wm[e];
          }
        } else if (!FIX && real) {
          // filter: slot 0 holds the initial marginal
#pragma unroll
          for (int i = 0; i < N; ++i) {
#pragma unroll
            for (int c = 0; c < D; ++c) a.cond[(long long)vb * a.K * SLOT + i * D + c] = SM(i, c);
#pragma unroll
            for (int j = 0; j <= i; ++j) a.cond[(long long)vb * a.K * SLOT + N * D + Lay::tri(i, j)] = 0.0;
          }
        }
        } else if constexpr (SLICE) {
          // take over a member another lane parked at a checkpoint
          SliceScalars io;
          slice_restore<(FIX ? Lay::BW : 0), Lay::MARG>(&a, b, s_bw + tid, s_state + tid, THREADS, &io);
          t = io.t;
          dt_next = io.dt_next;
          le_prev = io.le_prev;
          sigma_state = io.sigma_state;
          k_next = io.k_next;
          set_ck();
          n_acc = io.n_acc;
          n_rej = io.n_rej;
          n_att = io.n_att;
          mode = MODE_STEP;
        }
      } else if (!claimed_none) {
        exhausted = true;
      }
    }
    // warp-level vote keeps the loop convergent; the lane counts feed the utilisation statistics
    const unsigned active = __ballot_sync(0xffffffffu, have);
    if constexpr (PAIR) {
      if (active == 0u) {
        // the backward lanes must have taken the last job out of the mailbox (and passed their exit check)
        // before the exit flag goes up
        if (pair_started) pipe::bar_sync(1 + THREADS / 32 + (tid >> 5), 64);
        if ((tid & 31) == 0) pair_exit[tid >> 5] = 1;
        __syncwarp();
        pipe::bar_arrive(1 + (tid >> 5), 64);
      }
      pair_q ^= 1;  // (0 for the first job)
      pair_nops = 0;
    }
    if (active == 0u) {
      if constexpr (PIPE) {  // (have is uniform over the CTA in this mode: every main warp leaves here)
        if (tid == 0) pipe::mail<N>().exit_ = 1;
        pipe::bar_arrive(pipe::BAR_JOB, THREADS + 32);
      }
      if (!SLICE || __all_sync(0xffffffffu, exhausted)) break;
      if ((threadIdx.x & 31) == 0) slice_repair(&a, (int)((a.K - 2) >> a.slice_shift) + 1);
      __nanosleep(5000);  // members are still running elsewhere and may yet be parked
      poll_now = true;    // (this warp's iteration counter stands still while it has no member)
      continue;
    }
    stat_warp_iters += 1;
    PN_MAIN_PHASE(14);  // end of the previous iteration's tail / member fetch
#ifdef PN_PIPE_STATS
    if (PAIR && tid == 0 && blockIdx.x == 0) atomicAdd(a.ticket + 11, 1ULL);
#endif
    if constexpr (SLICE) {
      // belt and braces: every warp re-derives the queue mask from the counters once in a while, so a
      // parked member could not stay invisible even if no warp ever ran completely out of work
      if ((stat_warp_iters & 4095u) == 0 && (threadIdx.x & 31) == 0)
        slice_repair(&a, (int)((a.K - 2) >> a.slice_shift) + 1);
    }
    stat_lane_iters += have ? 1u : 0u;
    stat_interp_iters += (have && mode != MODE_STEP) ? 1u : 0u;
    if constexpr (!PAIR) {
      if (!have) continue;  // idle lane
    }
    // (PAIR: idle lanes walk through the step on whatever their registers hold -- the named barriers inside it
    // need the whole warp -- and leave in front of the bookkeeping)

    // ---- choose this iteration's prediction --------------------------------------------
    double t_ck = ck_cached();
    double dt, sigma_given;
    if (mode == MODE_STEP) {
      dt = (a.flags & FLAG_FIXED_GRID) ? (t_ck - t) : dt_next;
      sigma_given = sigma0;
    } else if (mode == MODE_INTERP_A) {
      dt = t_ck - t;
      sigma_given = SPEND(1);
    } else {
      dt = SPEND(0) - t;
      sigma_given = SPEND(1);
    }

    // ==================== uber step (straight-line, identical for all lanes) ============
    // A.1 preconditioner
    double p[N], pinv[N];
    auto precondition = [&](double dt_, double (&p_)[N], double (&pinv_)[N]) {
      double adt = fabs(dt_);
      // |dt| of a step that matters is a positive normal number (a step or an interpolation interval longer than
      // TIME_EPS): the unguarded fast paths are exact; the 0 / inf selects of rcp() / dsqrt() were ~8 instructions
      // per call of an instruction-fetch-bound step (DESIGN 3.1)
      double sq = dsqrt_raw(adt);
      double isq = rcp_raw(sq), idt = rcp_raw(adt);
      double dtp = 1.0, idtp = 1.0;
#pragma unroll
      for (int k = 0; k <= NU; ++k) {
        const int i = NU - k;
        p_[i] = (sq * dtp) * (1.0 / factorial(k));
        pinv_[i] = (isq * idtp) * factorial(k);
        dtp *= adt;
        idtp *= idt;
      }
    };
    if constexpr (PIPE) {
      // the previous iteration has already worked this out beside its controller chain if it guessed the step right
      if (dt == pipe_spec_dt) {
#pragma unroll
        for (int i = 0; i < N; ++i) {
          p[i] = pipe_spec_p[i];
          pinv[i] = pipe_spec_pinv[i];
        }
      } else {
        precondition(dt, p, pinv);
      }
    } else {
      precondition(dt, p, pinv);
    }
    // predicted mean
    double m_p[N][D], m_ext_p[N][D], m_ext[N][D];
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int c = 0; c < D; ++c) m_p[i][c] = pinv[i] * SM(i, c);
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int c = 0; c < D; ++c) {
        double acc = m_p[i][c];
#pragma unroll
        for (int j = i + 1; j < N; ++j) acc = fma(Binom<N>::at(i, j), m_p[j][c], acc);
        m_ext_p[i][c] = acc;
        m_ext[i][c] = p[i] * acc;
      }
    // linearise at the predicted mean, at the time this iteration's prediction reaches (for a time-dependent
    // problem; the same double an accepted step or a checkpoint commits as the new time)
    double t_vf = 0.0;
    if constexpr (TimeDependent<Prob>::value) {
      if (mode == MODE_STEP)
        t_vf = (a.flags & FLAG_FIXED_GRID) ? t_ck : (t + dt);
      else
        t_vf = (mode == MODE_INTERP_A) ? t_ck : SPEND(0);
    }
    double z[D], h[Q + 1];
    if (GROUP > 1) {
      double own[Q];
#pragma unroll
      for (int k = 0; k < Q; ++k) own[k] = m_ext[k][0];
      const double f_own = GroupVf<Prob, GROUP>::eval(own, sub, base, gmask, t_vf, par);
      z[0] = m_ext[Q][0] - f_own;
#pragma unroll
      for (int k = 0; k < Q; ++k) h[k] = 0.0;
      h[Q] = 1.0;
    } else {
      double uarg[Q * D], f[D];
#pragma unroll
      for (int k = 0; k < Q; ++k)
#pragma unroll
        for (int c = 0; c < D; ++c) uarg[k * D + c] = m_ext[k][c];
      vf_at<Prob>(uarg, t_vf, par, f);
#pragma unroll
      for (int c = 0; c < D; ++c) z[c] = m_ext[Q][c] - f[c];
#pragma unroll
      for (int k = 0; k < Q; ++k) h[k] = 0.0;
      h[Q] = 1.0;
      if (D == 1 && Prob::HAS_JAC && a.correction == 1) {
        double J[Q * D * D];
        jac_at<Prob>(uarg, t_vf, par, J);
#pragma unroll
        for (int k = 0; k < Q; ++k) h[k] = -J[k];
      }
    }
    if constexpr (PAIR) PN_MAIN_PHASE(15);  // precondition + predicted mean + vector field
    // wide mode, pass 1: per owned column predict the mean, stage u = m_ext[0] for the stencil,
    // form the residual z (kept in shared memory) and the CTA-wide sum of squares
    double wide_zz = 0.0;
    if constexpr (WIDE) {
      {
        // (PIPE: two columns at a time, loads first -- see pass 3)
        auto cols = [&](auto nc_tag, int c0) {
          constexpr int NC = decltype(nc_tag)::value;
          double mo[NC][N];
#pragma unroll
          for (int u = 0; u < NC; ++u)
#pragma unroll
            for (int i = 0; i < N; ++i) mo[u][i] = Wm[(size_t)i * wd + c0 + u * THREADS];
#pragma unroll
          for (int u = 0; u < NC; ++u) {
            double mp[N];
#pragma unroll
            for (int i = 0; i < N; ++i) mp[i] = pinv[i] * mo[u][i];
            double e0 = mp[0], e1 = mp[1];
#pragma unroll
            for (int j = 1; j < N; ++j) e0 = fma(Binom<N>::at(0, j), mp[j], e0);
#pragma unroll
            for (int j = 2; j < N; ++j) e1 = fma(Binom<N>::at(1, j), mp[j], e1);
            s_ubuf[c0 + u * THREADS] = p[0] * e0;
            s_zbuf[c0 + u * THREADS] = p[1] * e1;  // m_ext[q = 1][c] for now
          }
        };
        int c = tid;
        if constexpr (PIPE) {
          for (; c + THREADS < wd; c += 2 * THREADS) cols(IntTag<2>{}, c);
        }
        for (; c < wd; c += THREADS) cols(IntTag<1>{}, c);
      }
      cta_sync();
      const double cc = par[0] * (double)((wN + 1) * (wN + 1));
      double acc = 0.0;
      for (int c = tid; c < wd; c += THREADS) {
        const bool isu = c < wN;
        const int gi = isu ? c : c - wN;
        const double me = s_ubuf[c];
        const double pad = isu ? 1.0 : 3.0;
        const double l = (gi == 0) ? pad : s_ubuf[c - 1];
        const double r = (gi == wN - 1) ? pad : s_ubuf[c + 1];
        const double ui = s_ubuf[gi], vi = s_ubuf[wN + gi];
        const double uuv = (ui * ui) * vi;
        const double lap = fma(-2.0, me, l + r);
        const double f = isu ? fma(cc, lap, fma(-4.0, ui, 1.0 + uuv)) : fma(cc, lap, fma(3.0, ui, -uuv));
        const double zc = s_zbuf[c] - f;
        acc = fma(zc, zc, acc);
        s_zbuf[c] = zc;  // own column only: no hazard
      }
      wide_zz = block_sum(acc);
      PN_MAIN_PHASE(15);  // preconditioner + pass 1
    }
    // local calibration + error estimate from the process noise
    double err, sigma;
    double mle_zz = 0.0, mle_invS = 0.0;  // solver_mle: the two ingredients of z^T S^-1 z
    {
      double s2 = 0.0;
#pragma unroll
      for (int j = 0; j <= Q; ++j) {
        double acc = 0.0;
#pragma unroll
        for (int i = j; i <= Q; ++i) acc = fma(h[i] * p[i], LQ[i * N + j], acc);
        s2 = fma(acc, acc, s2);
      }
      double s = dsqrt_raw(s2);  // s2 >= (p_q LQ_qq)^2 > 0
      double zz = 0.0;
      if constexpr (WIDE) {
        zz = wide_zz;
      } else if (GROUP == 1) {
#pragma unroll
        for (int c = 0; c < D; ++c) zz = fma(z[c], z[c], zz);
      } else {
        zz = real ? fma(z[0], z[0], 0.0) : 0.0;
        if (!BDIAG) zz = group_sum<GROUP>(zz, gmask);
      }
      mle_zz = zz;
      double sigma_hat = dsqrt(zz) * rcp_raw(s);
      sigma_hat = BDIAG ? sigma_hat : sigma_hat * inv_sqrt_d;
      err = (fabs(dt) * sigma_hat) * s;
      sigma = (mode == MODE_STEP) ? ((a.calibration == 1) ? sigma_hat : sigma_given) : sigma_given;
    }
    // predict the square-root covariance
    double L_ext[N][N];         // lower
    double Gn[N][N], gn[N][D];  // new conditional (un-preconditioned); Lam_n lower
    double Ln[N][N];
    double X[N][N];             // RY^{-1} R12 (fixed-point); G_p = X^T
    if (pipe_F) {
      double L_p[N][N];  // lower
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) L_p[i][j] = pinv[i] * SL(i, j);
      // BL[i][j] = (A L_p)[j][i]
      double BL[N][N];
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) {
          const int k0 = (i > j) ? i : j;
          double acc = (k0 == i) ? L_p[i][j] : Binom<N>::at(i, k0) * L_p[k0][j];
#pragma unroll
          for (int k = k0 + 1; k < N; ++k) acc = fma(Binom<N>::at(i, k), L_p[k][j], acc);
          BL[j][i] = acc;
        }
      // top-left block rows: TL[j][c] = sigma * LQ[c][j] (c >= j), materialised when row j is used
      double RY[N][N];   // upper
      double R12[N][N];  // full (fixed-point)
      double BR[N][N];   // bottom-right block, starts as L_p^T (upper), fills in (fixed-point)
      if (FIX && !PIPE && !PAIR) {
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
          for (int c = 0; c < N; ++c) BR[i][c] = (i <= c) ? L_p[c][i] : 0.0;
      }
      double pipe_v0[N], pipe_g[N];  // PIPE: the reflector scalars go to the backward warp
#pragma unroll
      for (int j = 0; j < N; ++j) {
        double sigma2 = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) sigma2 = fma(BL[i][j], BL[i][j], sigma2);
        const double alpha = sigma * LQ[j * N + j];
        Reflector rf = make_reflector(alpha, sigma2);
        RY[j][j] = rf.beta;
        if constexpr (PIPE || PAIR) {
          pipe_v0[j] = rf.v0;
          pipe_g[j] = rf.ng;  // the NEGATED 2 / v^T v (see Reflector)
        }
        // left block columns c > j
#pragma unroll
        for (int c = j + 1; c < N; ++c) {
          double top = sigma * LQ[c * N + j];
          double w = 0.0;
#pragma unroll
          for (int i = 0; i < N; ++i) w = fma(BL[i][j], BL[i][c], w);
          w = fma(rf.v0, top, w);
          double f = w * rf.ng;
          RY[j][c] = fma(f, rf.v0, top);
#pragma unroll
          for (int i = 0; i < N; ++i) BL[i][c] = fma(f, BL[i][j], BL[i][c]);
        }
        if (FIX && !PIPE && !PAIR) {
          // right block columns: top entry starts at 0
#pragma unroll
          for (int c = 0; c < N; ++c) {
            double w = 0.0;  // the v0 term multiplies the (still zero) top-right entry
#pragma unroll
            for (int i = 0; i < N; ++i) {
              if (j == 0 && i > c) continue;  // still structurally zero
              w = fma(BL[i][j], BR[i][c], w);
            }
            double f = w * rf.ng;
            R12[j][c] = fma(f, rf.v0, 0.0);
#pragma unroll
            for (int i = 0; i < N; ++i) BR[i][c] = fma(f, BL[i][j], BR[i][c]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) L_ext[i][j] = p[i] * RY[j][i];
      if constexpr (PIPE) {
        // hand the reflectors to the backward warp (one main warp writes: every thread holds the same values)
        {
          pipe::Mail<N>& M = pipe::mail<N>();
#pragma unroll
          for (int i = 0; i < N; ++i) {
            M.v0[i] = pipe_v0[i];
            M.g[i] = pipe_g[i];
            M.p[i] = p[i];
            M.pinv[i] = pinv[i];
#pragma unroll
            for (int j = 0; j < N; ++j) M.BL[i * N + j] = BL[i][j];
#pragma unroll
            for (int j = i; j < N; ++j) M.RY[i * N + j] = RY[i][j];
#pragma unroll
            for (int j = 0; j <= i; ++j) M.Lp[Lay::tri(i, j)] = L_p[i][j];
          }
          M.reset = pipe_reset ? 1 : 0;
          M.exit_ = 0;
          M.stats = a.ticket;
        }
      }
      if constexpr (PAIR) {
        // the backward lanes took the previous job out of the mailbox long ago (they arrive at this barrier as
        // soon as they have loaded it): no waiting here in the steady state
        if (pair_started) pipe::bar_sync(1 + THREADS / 32 + (tid >> 5), 64);
        pair_started = true;
        // (the backward lane has loaded the previous job, so it is done with the op list of the job before that,
        // which is the buffer this iteration writes: no ops until the bookkeeping says otherwise)
        s_int[PMB::i_nops(pair_q) * THREADS + tid] = 0;
        // the lane's mailbox: reflectors of the predict QR, R factor, L_p, preconditioner, predicted means
        {
          double jb[PMB::JOB];
          jb[PMB::JOB - 1] = 0.0;  // (padding of an odd job)
#pragma unroll
          for (int i = 0; i < N; ++i) {
            jb[PMB::O_V0 + i] = pipe_v0[i];
            jb[PMB::O_G + i] = pipe_g[i];
            jb[PMB::O_P + i] = p[i];
            jb[PMB::O_PINV + i] = pinv[i];
#pragma unroll
            for (int c = 0; c < D; ++c) {
              jb[PMB::O_MP + i * D + c] = m_p[i][c];
              jb[PMB::O_MEP + i * D + c] = m_ext_p[i][c];
            }
#pragma unroll
            for (int j = 0; j < N; ++j) jb[PMB::O_BL + i * N + j] = BL[i][j];
#pragma unroll
            for (int j = i; j < N; ++j) jb[PMB::O_RY + Lay::tri(j, i)] = RY[i][j];
#pragma unroll
            for (int j = 0; j <= i; ++j) jb[PMB::O_LP + Lay::tri(i, j)] = L_p[i][j];
          }
#pragma unroll
          for (int e = 0; e < PMB::JOB / 2; ++e)
            reinterpret_cast<double2*>(s_job)[e * THREADS + tid] = make_double2(jb[2 * e], jb[2 * e + 1]);
        }
        s_int[0 * THREADS + tid] = pair_reset ? 1 : 0;
        pair_reset = false;
        PN_MAIN_PHASE(16);  // calibration + left block of the predict QR + mailbox
      }
      if (FIX && !PIPE && !PAIR) {
        // The lower-right block BR is NOT triangularised: BR^T is already a valid square-root factor
        // of the backward noise (BR^T BR = R_XY^T R_XY) and the merge below re-triangularises anyway.
        // That removes n-1 serial Householder chains per step.
        // X = RY^{-1} R12 (back substitution); G_p = X^T
#pragma unroll
        for (int i = N - 1; i >= 0; --i) {
          double inv = rcp_raw(RY[i][i]);  // a zero pivot (sigma = 0 and L = 0) poisons X with NaN either way (0 * inf)
#pragma unroll
          for (int c = 0; c < N; ++c) {
            double acc = R12[i][c];
#pragma unroll
            for (int k = i + 1; k < N; ++k) acc = fma(-RY[i][k], X[k][c], acc);
            X[i][c] = acc * inv;
          }
        }
#pragma unroll
        for (int i = 0; i < N; ++i) {
#pragma unroll
          for (int c = 0; c < D; ++c) {
            double acc = m_p[i][c];
#pragma unroll
            for (int k = 0; k < N; ++k) acc = fma(-X[k][i], m_ext_p[k][c], acc);
            gn[i][c] = p[i] * acc;
          }
#pragma unroll
          for (int j = 0; j < N; ++j) Gn[i][j] = (p[i] * X[j][i]) * pinv[j];
#pragma unroll
          for (int j = 0; j < N; ++j) Ln[i][j] = p[i] * BR[j][i];
        }
      }
    }
    if constexpr (PIPE) {
      pipe_reset = false;
      pipe::bar_arrive(pipe::BAR_JOB, THREADS + 32);  // (all main threads arrive; warp 0 wrote the job)
      PN_MAIN_PHASE(16);  // calibration + predict QR + publish
    }
    // Program order of the two blocks that are off the step-size chain (merge of the backward conditional,
    // QR of the corrected factor).  Thread-per-IVP kernels run them AFTER the error norm and the PI
    // controller: the controller's serial sqrt -> log -> exp chain then overlaps with their independent
    // work (-2 % on the headline kernel).  The lane-per-dimension and CTA-per-IVP instances keep the
    // original order (the late order costs them registers: Brusselator N = 16 was 1.5x slower).
    constexpr bool LATE_BLOCKS = (GROUP == 1 && !WIDE);
    // merge with the running conditional (A.4); running conditional lives in shared memory
    double Gm[N][N], gm[N][D], Lm[N][N];
    auto merge_running_conditional = [&]() {
    if (FIX && !PIPE && !PAIR) {
      double G1[N][N];
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) G1[i][j] = SBW(OFF_G + i * N + j);
#pragma unroll
      for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = 0; j < N; ++j) {
          double acc = G1[i][0] * Gn[0][j];
#pragma unroll
          for (int k = 1; k < N; ++k) acc = fma(G1[i][k], Gn[k][j], acc);
          Gm[i][j] = acc;
        }
#pragma unroll
        for (int c = 0; c < D; ++c) {
          double acc = SBW(OFF_g + i * D + c);
#pragma unroll
          for (int k = 0; k < N; ++k) acc = fma(G1[i][k], gn[k][c], acc);
          gm[i][c] = acc;
        }
      }
      // T = G1 Lam_n ; M = [T^T ; Lam_run^T]
      double Mt[N][N];  // Mt[i][j] = T[j][i]
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) {
          double acc = G1[i][0] * Ln[0][j];
#pragma unroll
          for (int k = 1; k < N; ++k) acc = fma(G1[i][k], Ln[k][j], acc);
          Mt[j][i] = acc;
        }
      double Mb[N][N];  // Mb[i][j] = Lam_run[j][i], nonzero for i <= j
#pragma unroll
      for (int j = 0; j < N; ++j)
#pragma unroll
        for (int i = 0; i <= j; ++i) Mb[i][j] = SBW(OFF_LAM + Lay::tri(j, i));
#pragma unroll
      for (int j = 0; j < N; ++j) {
        double sigma2 = 0.0;
#pragma unroll
        for (int i = j + 1; i < N; ++i) sigma2 = fma(Mt[i][j], Mt[i][j], sigma2);
#pragma unroll
        for (int i = 0; i <= j; ++i) sigma2 = fma(Mb[i][j], Mb[i][j], sigma2);
        Reflector rf = make_reflector(Mt[j][j], sigma2);
#pragma unroll
        for (int c = j + 1; c < N; ++c) {
          double w = 0.0;
#pragma unroll
          for (int i = j + 1; i < N; ++i) w = fma(Mt[i][j], Mt[i][c], w);
#pragma unroll
          for (int i = 0; i <= j; ++i) w = fma(Mb[i][j], Mb[i][c], w);
          w = fma(rf.v0, Mt[j][c], w);
          double f = w * rf.ng;
          Mt[j][c] = fma(f, rf.v0, Mt[j][c]);
#pragma unroll
          for (int i = j + 1; i < N; ++i) Mt[i][c] = fma(f, Mt[i][j], Mt[i][c]);
#pragma unroll
          for (int i = 0; i <= j; ++i) Mb[i][c] = fma(f, Mb[i][j], Mb[i][c]);
        }
        Mt[j][j] = rf.beta;
      }
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) Lm[i][j] = Mt[j][i];
    }
    };
    if constexpr (!LATE_BLOCKS) merge_running_conditional();
    // correction (noise-free observation, sqrt form)
    double m_new[N][D], L_new[N][N];
    double gain[N];
    double e_norm;
    double hL[Q + 1];
    auto corrected_factor = [&]() {
    // Mc[j][i] = L_ext[i][j] - hL[j] gain[i]; rows j > Q are untouched rows of L_ext^T
    double Mc[Q + 1][N];
#pragma unroll
    for (int j = 0; j <= Q; ++j)
#pragma unroll
      for (int i = 0; i < N; ++i) Mc[j][i] = fma(-hL[j], gain[i], (j <= i) ? L_ext[i][j] : 0.0);
#pragma unroll
    for (int c0 = 0; c0 < Q; ++c0) {
      double sigma2 = 0.0;
#pragma unroll
      for (int i = c0 + 1; i <= Q; ++i) sigma2 = fma(Mc[i][c0], Mc[i][c0], sigma2);
      Reflector rf = make_reflector(Mc[c0][c0], sigma2);
#pragma unroll
      for (int c = c0 + 1; c < N; ++c) {
        double w = 0.0;
#pragma unroll
        for (int i = c0 + 1; i <= Q; ++i) w = fma(Mc[i][c0], Mc[i][c], w);
        w = fma(rf.v0, Mc[c0][c], w);
        double f = w * rf.ng;
        Mc[c0][c] = fma(f, rf.v0, Mc[c0][c]);
#pragma unroll
        for (int i = c0 + 1; i <= Q; ++i) Mc[i][c] = fma(f, Mc[i][c0], Mc[i][c]);
      }
      Mc[c0][c0] = rf.beta;
    }
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int j = 0; j <= i; ++j) L_new[i][j] = (j <= Q) ? Mc[j][i] : L_ext[i][j];
    };
    {
      if (pipe_F) {
      double S = 0.0;
#pragma unroll
      for (int j = 0; j <= Q; ++j) {
        double acc = 0.0;
#pragma unroll
        for (int i = j; i <= Q; ++i) acc = fma(h[i], L_ext[i][j], acc);
        hL[j] = acc;
        S = fma(acc, acc, S);
      }
      double invS = rcp_raw(S);  // S = 0 (no predicted variance at all): the gain is NaN either way (0 * inf)
      mle_invS = invS;
#pragma unroll
      for (int i = 0; i < N; ++i) {
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j <= ((i < Q) ? i : Q); ++j) acc = fma(L_ext[i][j], hL[j], acc);
        gain[i] = acc * invS;
      }
      }
      if constexpr (PIPE) {
        // main warp 0 -> the other main warps: the gain (all they need of the factor arithmetic)
        pipe::Mail<N>& M = pipe::mail<N>();
        if (pipe_F) {
#pragma unroll
          for (int i = 0; i < N; ++i) M.gain[i] = gain[i];
        }
        cta_sync();
#pragma unroll
        for (int i = 0; i < N; ++i) gain[i] = M.gain[i];
      }
      if constexpr (!LATE_BLOCKS && !PIPE) corrected_factor();
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int c = 0; c < D; ++c) m_new[i][c] = fma(-gain[i], z[c], m_ext[i][c]);
      double acc = 0.0;
      if constexpr (WIDE) {
        // pass 2: proposed u = m_new[0][c] = m_ext[0][c] - gain[0] z[c] per owned column
        double part = 0.0;
        {
          int c = tid;
          if constexpr (PIPE) {
            // two reciprocal chains in flight; the partial sum still takes the columns in ascending order
            for (; c + THREADS < wd; c += 2 * THREADS) {
              const double ua = fma(-gain[0], s_zbuf[c], s_ubuf[c]);
              const double ub = fma(-gain[0], s_zbuf[c + THREADS], s_ubuf[c + THREADS]);
              const double ra = err * rcp(fma(rtol, fabs(ua), atol));
              const double rb = err * rcp(fma(rtol, fabs(ub), atol));
              part = fma(ra, ra, part);
              part = fma(rb, rb, part);
            }
          }
          for (; c < wd; c += THREADS) {
            const double u_new = fma(-gain[0], s_zbuf[c], s_ubuf[c]);
            const double ratio = err * rcp(fma(rtol, fabs(u_new), atol));
            part = fma(ratio, ratio, part);
          }
        }
        acc = block_sum(part);
        PN_MAIN_PHASE(17);  // correction + gain broadcast + pass 2
      } else if (GROUP == 1) {
#pragma unroll
        for (int c = 0; c < D; ++c) {
          double ratio = err * rcp(fma(rtol, fabs(m_new[0][c]), atol));
          acc = fma(ratio, ratio, acc);
        }
      } else {
        // (guarded reciprocal: atol = 0 and a proposed u of exactly 0 must give an infinite error norm -- a rejected
        // step, as in the oracle's division -- not a NaN, which would retire the member)
        double ratio = err * rcp(fma(rtol, fabs(m_new[0][0]), atol));
        acc = group_sum<GROUP>(real ? fma(ratio, ratio, 0.0) : 0.0, gmask);
      }
      e_norm = dsqrt(acc) * inv_sqrt_d;
    }
    // PIPE: the corrected factor's Householder chain sits beside the controller's sqrt -> log -> exp chain (two
    // independent serial chains in one basic block) instead of in front of the error norm's CTA reduction
    if constexpr (PIPE) {
      if (pipe_F) corrected_factor();
    }
    if constexpr (PAIR) PN_MAIN_PHASE(17);  // correction + error norm
    // PI controller
    double fac, le_now;
    {
      // safety (1/e)^n1 (e_prev/e)^n2 = safety exp(n2 ln e_prev - (n1 + n2) ln e); ln e_prev is cached
      le_now = det_log(e_norm < 2.2250738585072014e-308 ? 2.2250738585072014e-308 : e_norm);
      le_now = (e_norm == 0.0) ? -745.0 : le_now;
      fac = a.safety * det_exp(fma(a.pow_p, le_prev, -((a.pow_i + a.pow_p) * le_now)));
      fac = (e_norm == 0.0) ? a.factor_max : fac;
      fac = (e_norm != e_norm) ? e_norm : fac;
      fac = (fac < a.factor_max) ? fac : a.factor_max;
      fac = (fac > a.factor_min) ? fac : a.factor_min;
    }
    if constexpr (LATE_BLOCKS) {
      corrected_factor();
      merge_running_conditional();
    }
    if constexpr (PAIR) PN_MAIN_PHASE(18);  // controller + corrected factor
    if constexpr (PIPE) {
      pipe_spec_dt = fac * dt;  // = dt_next of an attempted step (the bookkeeping below forms the same product)
      precondition(pipe_spec_dt, pipe_spec_p, pipe_spec_pinv);
    }
    // ==================== per-lane bookkeeping (cheap, may diverge) =====================
    // helpers -------------------------------------------------------------------------
    // PIPE: the backward warp has published X by now (it is busy with the merge); the running G the offset
    // update needs is the buffer it is NOT writing.  Everything the bookkeeping below wants done to the
    // running conditional is queued as an op and handed over in one piece (BAR_ACT).
    if constexpr (PAIR) {
      if (!have) continue;  // idle lane (its mailbox carries no ops)
    }
    const double* pipe_G1 = nullptr;  // PIPE: the running G (before this step's merge) and X, in shared memory
    const double* pipe_X = nullptr;
    if constexpr (PIPE) {
      PN_MAIN_PHASE(18);  // error norm + corrected factor + controller
#ifdef PN_PIPE_STATS
      const long long pipe_c0 = clock64();
#endif
      pipe::bar_sync(pipe::BAR_X, THREADS + 32);
#ifdef PN_PIPE_STATS
      if (tid == 0) {
        atomicAdd(a.ticket + 8, (unsigned long long)(clock64() - pipe_c0));
        atomicAdd(a.ticket + 11, 1ULL);
      }
#endif
      const pipe::Mail<N>& M = pipe::mail<N>();
      pipe_X = M.X;
      pipe_G1 = M.R[M.cur];
      pipe_nops = 0;
      PN_MAIN_PHASE(20);  // X wait + load
    }
    auto pipe_op = [&](int code, double* dst) {
      if constexpr (PAIR) {
        if (pair_nops < pair::MAX_OPS) {
          s_int[(PMB::i_nops(pair_q) + 1 + pair_nops) * THREADS + tid] = code;
          s_job[(PMB::O_DST + pair_q * pair::MAX_OPS + pair_nops) * THREADS + tid] = __longlong_as_double((long long)dst);
          pair_nops += 1;
          s_int[PMB::i_nops(pair_q) * THREADS + tid] = pair_nops;
        }
      }
      if constexpr (PIPE) {
        if (tid == 0 && pipe_nops < pipe::MAX_OPS) {
          pipe::Mail<N>& M = pipe::mail<N>();
          M.op[pipe_nops] = code;
          M.dst[pipe_nops] = dst;
        }
        pipe_nops += 1;
      }
    };
    // wide mode, pass 3: everything the bookkeeping below does to the n x d mean arrays, in ONE
    // sweep over the owned columns (reads the old state, writes the new one).
    //   mw: what becomes the state mean   (0 keep, 1 m_new, 2 m_ext, 3 pending mean)
    //   gw: what becomes the running g    (0 keep, 1 merged gm, 2 zero)
    //   pw: pending mean <- m_new
    //   eg / em: global destinations [n][d] for the merged g / a mean to emit (nullptr: none)
    //   em_src: 2 m_ext, 3 pending mean
    auto wide_pass3 = [&](int mw, int gw, bool pw, double* eg, double* em, int em_src) {
      if constexpr (WIDE) {
        // NC columns at a time: all loads first, then the arithmetic, then the stores -- the arrays may alias as
        // far as the compiler knows, so a column-by-column loop serialises on its own stores (PIPE build: 2)
        auto cols = [&](auto nc_tag, int c0) {
          constexpr int NC = decltype(nc_tag)::value;
          double mo[NC][N], wg[NC][N], pend_old[NC][N], zc[NC];
#pragma unroll
          for (int u = 0; u < NC; ++u) {
            const int c = c0 + u * THREADS;
            zc[u] = s_zbuf[c];
#pragma unroll
            for (int i = 0; i < N; ++i) {
              mo[u][i] = Wm[(size_t)i * wd + c];
              wg[u][i] = (FIX && (gw == 1 || eg != nullptr)) ? Wg[(size_t)i * wd + c] : 0.0;
              pend_old[u][i] = (mw == 3 || em_src == 3) ? Wp[(size_t)i * wd + c] : 0.0;
            }
          }
          double mext[NC][N], gmc[NC][N], mn[NC][N];
#pragma unroll
          for (int u = 0; u < NC; ++u) {
            double mp[N], mep[N];
#pragma unroll
            for (int i = 0; i < N; ++i) mp[i] = pinv[i] * mo[u][i];
#pragma unroll
            for (int i = 0; i < N; ++i) {
              double acc = mp[i];
#pragma unroll
              for (int j = i + 1; j < N; ++j) acc = fma(Binom<N>::at(i, j), mp[j], acc);
              mep[i] = acc;
              mext[u][i] = p[i] * acc;
            }
            if (FIX && (gw == 1 || eg != nullptr)) {
              double gnc[N];
#pragma unroll
              for (int i = 0; i < N; ++i) {
                double acc = mp[i];
#pragma unroll
                for (int k = 0; k < N; ++k) acc = fma(PIPE ? -pipe_X[k * N + i] : -X[k][i], mep[k], acc);
                gnc[i] = p[i] * acc;
              }
#pragma unroll
              for (int i = 0; i < N; ++i) {
                double acc = wg[u][i];
#pragma unroll
                for (int k = 0; k < N; ++k) acc = fma(PIPE ? pipe_G1[i * N + k] : SBW(OFF_G + i * N + k), gnc[k], acc);
                gmc[u][i] = acc;
              }
            }
#pragma unroll
            for (int i = 0; i < N; ++i) mn[u][i] = fma(-gain[i], zc[u], mext[u][i]);
          }
#pragma unroll
          for (int u = 0; u < NC; ++u) {
            const int c = c0 + u * THREADS;
#pragma unroll
            for (int i = 0; i < N; ++i) {
              if (pw) Wp[(size_t)i * wd + c] = mn[u][i];
              if (mw == 1) Wm[(size_t)i * wd + c] = mn[u][i];
              if (mw == 2) Wm[(size_t)i * wd + c] = mext[u][i];
              if (mw == 3) Wm[(size_t)i * wd + c] = pend_old[u][i];
              if (FIX && gw == 1) Wg[(size_t)i * wd + c] = gmc[u][i];
              if (FIX && gw == 2) Wg[(size_t)i * wd + c] = 0.0;
              if (FIX && eg != nullptr) eg[(size_t)i * wd + c] = gmc[u][i];
              if (em != nullptr) em[(size_t)i * wd + c] = (em_src == 2) ? mext[u][i] : pend_old[u][i];
            }
          }
        };
        int c = tid;
        if constexpr (PIPE) {
          for (; c + THREADS < wd; c += 2 * THREADS) cols(IntTag<2>{}, c);
        }
        for (; c < wd; c += THREADS) cols(IntTag<1>{}, c);
        cta_sync();
      }
    };
    // wide slot layout: [G | (unused n) | Lam | L1 | g (n x d) | m1 (n x d)]; src 0: merged result of
    // this step, 1: identity, 2: the committed running conditional (shared memory)
    auto wide_store_factor = [&](double* dst, int src) {
      if constexpr (PIPE) {
        pipe_op(src == 0 ? pipe::OP_STORE_MERGED : (src == 1 ? pipe::OP_STORE_IDENTITY : pipe::OP_STORE_RUNNING), dst);
      } else if constexpr (WIDE) {
        if (tid == 0) {
#pragma unroll
          for (int i = 0; i < N; ++i) {
#pragma unroll
            for (int j = 0; j < N; ++j)
              dst[OFF_G + i * N + j] = (src == 1) ? ((i == j) ? 1.0 : 0.0) : ((src == 2) ? SBW(OFF_G + i * N + j) : Gm[i][j]);
            dst[OFF_g + i] = 0.0;
#pragma unroll
            for (int j = 0; j <= i; ++j)
              dst[OFF_LAM + Lay::tri(i, j)] = (src == 1) ? 0.0 : ((src == 2) ? SBW(OFF_LAM + Lay::tri(i, j)) : Lm[i][j]);
          }
        }
      }
    };
    // L1 part of a wide slot; src 0: committed factor, 1: pending factor, 2: L_ext of this step
    auto wide_store_L1 = [&](double* dst, int src) {
      if constexpr (WIDE) {
        if (tid == 0) {
#pragma unroll
          for (int i = 0; i < N; ++i)
#pragma unroll
            for (int j = 0; j <= i; ++j)
              dst[Lay::BW + Lay::tri(i, j)] = (src == 0) ? SL(i, j) : ((src == 1) ? SPEND(2 + N * D + Lay::tri(i, j)) : L_ext[i][j]);
        }
      }
    };
    auto wide_copy = [&](double* dst, const double* src, bool zero_src) {  // [n][d] arrays
      if constexpr (WIDE) {
        for (int e = tid; e < N * wd; e += THREADS) dst[e] = zero_src ? 0.0 : src[e];
        cta_sync();
      }
    };

    auto store_cond = [&](double* dst /* element stride VB */) {
      if (!real) return;
      if constexpr (PAIR) {
        pipe_op(pipe::OP_STORE_MERGED, dst);
        return;
      }
#pragma unroll
      for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = 0; j < N; ++j) dst[OFF_G + i * N + j] = Gm[i][j];
#pragma unroll
        for (int c = 0; c < D; ++c) dst[OFF_g + i * D + c] = gm[i][c];
#pragma unroll
        for (int j = 0; j <= i; ++j) dst[OFF_LAM + Lay::tri(i, j)] = Lm[i][j];
      }
    };
    auto store_identity_cond = [&](double* dst) {
      if (!real) return;
      if constexpr (PAIR) {
        pipe_op(pipe::OP_STORE_IDENTITY, dst);
        return;
      }
#pragma unroll
      for (int e = 0; e < Lay::BW; ++e) dst[e] = 0.0;
#pragma unroll
      for (int i = 0; i < N; ++i) dst[OFF_G + i * N + i] = 1.0;
    };
    auto bw_commit = [&]() {  // running conditional <- merged result
      if constexpr (PIPE || PAIR) {
        pipe_op(pipe::OP_COMMIT, nullptr);
        return;
      }
#pragma unroll
      for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = 0; j < N; ++j) SBW(OFF_G + i * N + j) = Gm[i][j];
#pragma unroll
        for (int c = 0; c < D; ++c) SBW(OFF_g + i * D + c) = gm[i][c];
#pragma unroll
        for (int j = 0; j <= i; ++j) SBW(OFF_LAM + Lay::tri(i, j)) = Lm[i][j];
      }
    };
    auto bw_reset = [&]() {  // running conditional <- identity (A.2)
      if constexpr (PIPE || PAIR) {
        pipe_op(pipe::OP_RESET, nullptr);
        return;
      }
#pragma unroll
      for (int e = 0; e < Lay::BW; ++e) SBW(e) = 0.0;
#pragma unroll
      for (int i = 0; i < N; ++i) SBW(OFF_G + i * N + i) = 1.0;
    };
    auto store_marg = [&](double* dst, const double (&mm)[N][D], const double (&LL)[N][N]) {
      if (!real) return;
#pragma unroll
      for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int c = 0; c < D; ++c) dst[i * D + c] = mm[i][c];
#pragma unroll
        for (int j = 0; j <= i; ++j) dst[N * D + Lay::tri(i, j)] = LL[i][j];
      }
    };
    auto store_state = [&](double* dst) {  // committed hidden state (shared memory) -> workspace
      if (!real) return;
#pragma unroll
      for (int e = 0; e < Lay::MARG; ++e) dst[e] = s_state[e * THREADS + tid];
    };
    auto record = [&](double tt, const double (&mm)[N][D], const double (&LL)[N][N]) {
      if ((a.flags & FLAG_RECORD) && n_acc < a.traj_cap) {
        if constexpr (WIDE) {
          // pass 3 has just moved the recorded mean into the state array (row 0 = u)
          if (leader) {
            a.traj_t[n_acc * a.B + b] = tt;
            a.traj_std[n_acc * a.B + b] = dsqrt(fma(LL[0][0], LL[0][0], 0.0));
          }
          for (int c = tid; c < wd; c += THREADS) a.traj_u[((long long)n_acc * wd + c) * a.B + b] = Wm[c];
        } else if (GROUP == 1) {
          a.traj_t[n_acc * VB + vb] = tt;
#pragma unroll
          for (int c = 0; c < D; ++c) a.traj_u[(n_acc * D + c) * VB + vb] = mm[0][c];
          a.traj_std[n_acc * VB + vb] = dsqrt(fma(LL[0][0], LL[0][0], 0.0));
        } else {
          if (leader) {
            a.traj_t[n_acc * a.B + b] = tt;
            a.traj_std[n_acc * a.B + b] = dsqrt(fma(LL[0][0], LL[0][0], 0.0));
          }
          if (real) a.traj_u[(n_acc * DT + sub) * a.B + b] = mm[0][0];
        }
      }
    };
    // exact hits on checkpoints by the committed state (m, L, running conditional): emit, reset
    auto resolve_hits = [&](bool& fin) {
      while (k_next < a.K && !(t + TIME_EPS < ck_cached())) {
        double* slot = a.cond + ((long long)vb * a.K + k_next) * SLOT;
        if constexpr (WIDE) {
          double* ws = wcond + (size_t)k_next * wslot;
          if (FIX) {
            wide_store_factor(ws, 2);
            wide_copy(ws + WSLOT, Wg, false);
            if (k_next == a.K - 1) {
              wide_store_factor(wcond, 1);
              wide_store_L1(wcond, 0);
              wide_copy(wcond + WSLOT, nullptr, true);
              wide_copy(wcond + WSLOT + (size_t)N * wd, Wm, false);
            }
            wide_copy(Wg, nullptr, true);
          } else {
            wide_store_L1(ws, 0);
            wide_copy(ws + WSLOT + (size_t)N * wd, Wm, false);
          }
        }
        if (FIX) {
          if constexpr (PAIR) {
            pipe_op(pipe::OP_STORE_RUNNING, slot);
          } else if (real) {
#pragma unroll
            for (int e = 0; e < Lay::BW; ++e) slot[e] = SBW(e);
          }
          if (k_next == a.K - 1) {
            store_identity_cond(a.cond + (long long)vb * a.K * SLOT);
            store_state(a.cond + (long long)vb * a.K * SLOT + Lay::BW);
          }
          bw_reset();
        } else {
          store_state(slot);
        }
        if (leader) a.n_accepted[b * a.K + k_next] = n_acc;
        emit_scale(k_next, sigma_state);
        k_next += 1;
        set_ck();
      }
      if (k_next >= a.K) fin = true;
    };
    auto commit_pending = [&]() {
      t = SPEND(0);
      sigma_state = SPEND(1);
#pragma unroll
      for (int e = 0; e < Lay::MARG; ++e) s_state[e * THREADS + tid] = SPEND(2 + e);
    };
    // after a checkpoint was emitted while the accepted state waits in s_pend
    auto after_checkpoint = [&](bool& fin) {
      const double t1 = SPEND(0);
      if (k_next < a.K && t1 > ck_cached() + TIME_EPS) {
        mode = MODE_INTERP_A;  // the next checkpoint lies inside the same step
      } else {
        commit_pending();
        if (FIX) bw_commit();
        if (WIDE && !FIX) wide_copy(Wm, Wp, false);  // fixed-point: done by pass 3 of prediction B
        mode = MODE_STEP;
        resolve_hits(fin);
      }
    };

    bool finished = false;
    int st = 0;
    const bool fixed_grid = (a.flags & FLAG_FIXED_GRID) != 0;
    const bool attempted = (mode == MODE_STEP);
    if (mode == MODE_STEP) {
      n_att += 1;
      if (e_norm != e_norm && !fixed_grid) {
        finished = true;
        st = 1;
      } else {
        dt_next = fac * dt;
        if (e_norm <= 1.0 || fixed_grid) {
          if (!fixed_grid) {
            le_prev = le_now;
          }
          n_acc += 1;
          if (GROUP == 1 && !WIDE && a.calibration == 2) mle_ss = mle_ss + (mle_zz * mle_invS) * (1.0 / (double)DT);
          const double t1 = fixed_grid ? t_ck : (t + dt);
          const bool overshoot = (k_next < a.K) && (t1 > t_ck + TIME_EPS);
          if (overshoot) {
            // keep the accepted state aside; interpolate from the (unchanged) previous state
            SPEND(0) = t1;
            SPEND(1) = sigma;
#pragma unroll
            for (int i = 0; i < N; ++i) {
#pragma unroll
              for (int c = 0; c < D; ++c) SPEND(2 + i * D + c) = m_new[i][c];
#pragma unroll
              for (int j = 0; j <= i; ++j) SPEND(2 + N * D + Lay::tri(i, j)) = L_new[i][j];
            }
            wide_pass3(0, 0, true, nullptr, nullptr, 0);
            mode = MODE_INTERP_A;
          } else {
            wide_pass3(1, FIX ? 1 : 0, false, nullptr, nullptr, 0);  // before bw_commit: needs the old G
            PN_MAIN_PHASE(21);  // pass 3 of an accepted step
            t = t1;
            sigma_state = sigma;
#pragma unroll
            for (int i = 0; i < N; ++i) {
#pragma unroll
              for (int c = 0; c < D; ++c) SM(i, c) = m_new[i][c];
#pragma unroll
              for (int j = 0; j <= i; ++j) SL(i, j) = L_new[i][j];
            }
            PN_MAIN_PHASE(22);  // state parked
            PN_MAIN_PHASE(23);  // (empty: the cost of a marker)
            if (FIX) bw_commit();
            record(t1, m_new, L_new);
            PN_MAIN_PHASE(24);  // commit op + record
            resolve_hits(finished);
            PN_MAIN_PHASE(25);  // resolve_hits
          }
        } else {
          n_rej += 1;
        }
        if (!finished && mode == MODE_STEP && a.max_attempts > 0 && n_att >= a.max_attempts) {
          finished = true;
          st = 2;
        }
      }
    } else if (mode == MODE_INTERP_A) {
      // prediction "previous state -> checkpoint": fixed-point emits the merged conditional
      // "t_c -> previous checkpoint" and continues from (t_c, m_t, L_t, identity); the filter emits
      // the extrapolated marginal.
      double* slot = a.cond + ((long long)vb * a.K + k_next) * SLOT;
      if constexpr (WIDE) {
        double* ws = wcond + (size_t)k_next * wslot;
        if (FIX) {
          wide_store_factor(ws, 0);
          wide_pass3(2, 2, false, ws + WSLOT, nullptr, 0);  // before bw_reset: needs the running G
        } else {
          wide_store_L1(ws, 2);
          wide_pass3(2, 0, false, nullptr, ws + WSLOT + (size_t)N * wd, 2);
        }
      }
      if (FIX) {
        store_cond(slot);
        bw_reset();
      } else {
        store_marg(slot, m_ext, L_ext);
        record(t_ck, m_ext, L_ext);
      }
      t = t_ck;
#pragma unroll
      for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int c = 0; c < D; ++c) SM(i, c) = m_ext[i][c];
#pragma unroll
        for (int j = 0; j <= i; ++j) SL(i, j) = L_ext[i][j];
      }
      if (leader) a.n_accepted[b * a.K + k_next] = n_acc;
      emit_scale(k_next, sigma_given);
      if (FIX) {
        mode = MODE_INTERP_B;
      } else {
        k_next += 1;
        set_ck();
        after_checkpoint(finished);
      }
    } else {
      // MODE_INTERP_B (fixed-point): the merged result (running conditional was the identity) is
      // the conditional "accepted state -> checkpoint"; it becomes the accepted state's backward
      // model.  At the last checkpoint the terminal marginal marginalise((m1, L1), bw_1t) is
      // left to the smoothing kernel: store its two ingredients in slot 0.
      if constexpr (WIDE) {
        const bool term = (k_next == a.K - 1);
        const double t1p = SPEND(0);
        const bool again = (k_next + 1 < a.K) && (t1p > grid_row(a, b)[k_next + 1] + TIME_EPS);
        if (term) {
          wide_store_factor(wcond, 0);
          wide_store_L1(wcond, 1);
        }
        wide_pass3(again ? 0 : 3, again ? 0 : 1, false, term ? wcond + WSLOT : nullptr,
                   term ? wcond + WSLOT + (size_t)N * wd : nullptr, 3);
      }
      if (k_next == a.K - 1) {
        store_cond(a.cond + (long long)vb * a.K * SLOT);
        if (real) {
#pragma unroll
          for (int e = 0; e < Lay::MARG; ++e) a.cond[(long long)vb * a.K * SLOT + Lay::BW + e] = SPEND(2 + e);
        }
      }
      k_next += 1;
      set_ck();
      after_checkpoint(finished);
    }
    if constexpr (PAIR) PN_MAIN_PHASE(19);  // bookkeeping
    if constexpr (PIPE) {
      if (tid == 0) pipe::mail<N>().nops = (pipe_nops < pipe::MAX_OPS) ? pipe_nops : pipe::MAX_OPS;
      pipe::bar_arrive(pipe::BAR_ACT, THREADS + 32);
      PN_MAIN_PHASE(19);  // X wait + pass 3 + bookkeeping
    }
    if constexpr (SLICE) {
      // the quantum boundaries of different members are staggered (b * 7919): lanes that started together
      // would otherwise all reach the queues in the same iteration
      if (!finished && attempted && mode == MODE_STEP && ((n_att + b * 7919LL) & a.slice_mask) == 0 &&
          slice_quantum_reached(a, t, n_att, b)) {
        const SliceScalars io = {t, dt_next, le_prev, sigma_state, k_next, n_acc, n_rej, n_att};
        if (slice_park_if_waiting(&a, b, (int)(k_next - 1) >> a.slice_shift, s_bw + tid, FIX ? Lay::BW : 0, s_state + tid,
                                  Lay::MARG, THREADS, &io)) {
          have = false;
          poll_now = true;
        }
      }
      if (finished) {
        atomicAdd(a.sw + 1, 1ULL);
        poll_now = true;
      }
    }
    if (finished) {
      if (leader) {
        a.n_rejected[b] = n_rej;
        a.status[b] = st;
        if (a.mle_scale) a.mle_scale[b] = (a.calibration == 2 && n_acc > 0) ? dsqrt(mle_ss * rcp((double)n_acc)) : 1.0;
        if (st != 0)
          for (long long kk = k_next; kk < a.K; ++kk) a.n_accepted[b * a.K + kk] = n_acc;
      }
      if (leader && (a.flags & FLAG_RECORD)) a.traj_len[b] = (n_acc + 1 < a.traj_cap) ? (n_acc + 1) : a.traj_cap;
      have = false;
    }
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(a.ticket + 1, (unsigned long long)stat_warp_iters);
    atomicMax((long long*)a.ticket + 4, (long long)(clock64() - clk0));
  }
  if (stat_lane_iters) atomicAdd(a.ticket + 2, (unsigned long long)stat_lane_iters);  // once per lane, at exit
  if (stat_interp_iters) atomicAdd(a.ticket + 3, (unsigned long long)stat_interp_iters);
#undef SBW
#undef SPEND
#undef SCK
#undef SM
#undef SL
  (void)sigma_state;
}

}  // namespace pn
