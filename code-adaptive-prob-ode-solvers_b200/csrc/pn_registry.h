// pn_registry.h -- table of compiled kernel instances (one per problem functor x nu x strategy).
// An entry names only kernels the library launches from it: what several builds share lives in *Slots helpers
// that name no solve kernel, and each *Instance adds its own solve kernel(s).
#pragma once
#include <cuda_runtime.h>

#include "pn_dense_cta_kernel.cuh"
#include "pn_dense_kernel.cuh"
#include "pn_dense_rows_kernel.cuh"
#include "pn_lml_kernel.cuh"
#include "pn_sample_kernel.cuh"
#include "pn_scalar_kernel.cuh"
#include "pn_smooth_kernel.cuh"

namespace pn {

enum : int {
  FAMILY_SCALAR = 0,      // thread per IVP, one n x n factor shared by all mean columns
  FAMILY_GROUP_ISO = 1,   // lane per dimension, identical factors (isotropic)
  FAMILY_GROUP_BDIAG = 2, // lane per dimension, per-dimension factors (blockdiag)
  FAMILY_DENSE = 3,       // warp per IVP, D x D factors in shared memory (dense, d > 1)
  FAMILY_WIDE = 4,        // CTA per IVP, isotropic, runtime dimension (Brusselator d = 2N up to 4096)
  FAMILY_DENSE_ROWS = 5,  // 16 or 32 lanes per IVP, register-resident Householder columns (dense, D <= 32)
  FAMILY_DENSE_CTA = 6,   // CTA per IVP, dense with a large runtime dimension, blocked QR on the FP64 tensor path
  FAMILY_PAIR = 8         // thread per IVP + a backward lane per IVP in a partner warp (fixed-point, small ensembles)
};
inline bool family_is_dense(int family) { return family == FAMILY_DENSE || family == FAMILY_DENSE_ROWS; }

struct KernelEntry {
  int family, problem, nu, strategy;
  int N, D, Q, P;
  int slot_doubles;   // workspace doubles per (checkpoint, member)
  int smem_doubles;   // dynamic shared memory doubles per thread
  int threads;
  int extra_threads = 0;  // threads of the CTA beyond `threads` that do not run the step (CTA-per-IVP PIPE build: the backward warp)
  int group;          // lanes per IVP (1: thread per IVP)
  int dv;             // lanes per IVP that own state (workspace entries per member)
  int ctx_doubles = 0;  // doubles one parked member occupies (time-sliced scheduling); 0: not supported
  bool has_jac;
  const void* solve_func;
  const void* solve_func_sliced = nullptr;  // time-sliced variant of the same kernel (nullptr: none)
  cudaError_t (*launch_solve)(const SolveArgs&, int grid, size_t smem, cudaStream_t);
  cudaError_t (*launch_solve_sliced)(const SolveArgs&, int grid, size_t smem, cudaStream_t) = nullptr;
  cudaError_t (*launch_smooth)(const SmoothArgs&, cudaStream_t);
  cudaError_t (*launch_sample)(const SampleArgs&, cudaStream_t) = nullptr;  // nullptr: family has no sampler yet
  cudaError_t (*launch_lml)(const LmlArgs&, cudaStream_t) = nullptr;        // nullptr: no likelihood kernel for this family
  // run-time compiled builds of user problems (pn_jit.cu): the launch_* pointers stay null; the kernels are library
  // handles, set once jit_load has compiled the module, and are launched with cudaLaunchKernel (jit_launch_*)
  bool jit = false;
  const void* smooth_func = nullptr;
  const void* sample_func = nullptr;  // nullptr: no sampler
  const void* lml_func = nullptr;     // likelihood sweep; nullptr: no likelihood kernel
};

void register_kernel(const KernelEntry& e);
const KernelEntry* find_kernel(int family, int problem, int nu, int strategy, int d);

// what the thread-per-IVP and lane-per-dimension builds of one (problem, nu, strategy) share: slots, shared-memory
// state, smoothing / sampling / likelihood kernels
template <class Prob, int NU, int STRAT, int GROUP, int BDIAG>
struct ScalarSlots {
  static constexpr int DL = (GROUP > 1) ? 1 : Prob::D;  // mean columns per lane
  static constexpr int DV = (GROUP > 1) ? Prob::D : 1;
  using Lay = Layout<NU + 1, DL>;
  static cudaError_t launch_smooth(const SmoothArgs& a, cudaStream_t s) {
    int grid = (int)((a.B * a.dv + 127) / 128);
    pn_smooth_kernel<NU + 1, DL, STRAT><<<grid, 128, 0, s>>>(a);
    return cudaGetLastError();
  }
  static cudaError_t launch_sample(const SampleArgs& a, cudaStream_t s) {
    const long long total = a.B * a.dv * a.S;
    pn_sample_kernel<NU + 1, DL><<<(unsigned)((total + 127) / 128), 128, 0, s>>>(a);
    return cudaGetLastError();
  }
  static cudaError_t launch_lml(const LmlArgs& a, cudaStream_t s) {
    pn_lml_sweep_kernel<NU + 1, DL><<<(unsigned)((a.B * a.dv + 127) / 128), 128, 0, s>>>(a);
    pn_lml_reduce_kernel<0><<<(unsigned)((a.B + 127) / 128), 128, 0, s>>>(a);
    return cudaGetLastError();
  }
  static KernelEntry entry() {
    KernelEntry e;
    e.launch_sample = (STRAT == 1) ? &launch_sample : nullptr;
    e.launch_lml = (STRAT == 1) ? &launch_lml : nullptr;
    e.family = (GROUP == 1) ? FAMILY_SCALAR : (BDIAG ? FAMILY_GROUP_BDIAG : FAMILY_GROUP_ISO);
    e.group = GROUP;
    e.dv = DV;
    e.problem = Prob::ID;
    e.nu = NU;
    e.strategy = STRAT;
    e.N = NU + 1;
    e.D = Prob::D;
    e.Q = Prob::Q;
    e.P = Prob::P;
    e.slot_doubles = (STRAT == 1) ? Lay::SLOT_FIX : Lay::SLOT_FILT;
    e.smem_doubles = ((STRAT == 1) ? Lay::BW : 0) + Lay::PEND + Lay::MARG;
    e.has_jac = Prob::HAS_JAC;
    e.launch_smooth = &launch_smooth;
    return e;
  }
};

template <class Prob, int NU, int STRAT, int GROUP, int BDIAG, int THREADS>
struct ScalarInstance {
  using Slots = ScalarSlots<Prob, NU, STRAT, GROUP, BDIAG>;
  static cudaError_t launch_solve(const SolveArgs& a, int grid, size_t smem, cudaStream_t s) {
    pn_scalar_kernel<Prob, NU, STRAT, GROUP, BDIAG, THREADS><<<grid, THREADS, smem, s>>>(a);
    return cudaGetLastError();
  }
  // time-sliced scheduling: compiled for the thread-per-IVP fixed-point kernels (the checkpoint solver)
  static constexpr bool SLICED = (GROUP == 1 && STRAT == 1);
  static cudaError_t launch_solve_sliced(const SolveArgs& a, int grid, size_t smem, cudaStream_t s) {
    pn_scalar_kernel<Prob, NU, STRAT, GROUP, BDIAG, THREADS, 0, 1><<<grid, THREADS, smem, s>>>(a);
    return cudaGetLastError();
  }
  static KernelEntry entry() {
    KernelEntry e = Slots::entry();
    e.threads = THREADS;
    e.solve_func = (const void*)&pn_scalar_kernel<Prob, NU, STRAT, GROUP, BDIAG, THREADS>;
    e.launch_solve = &launch_solve;
    if constexpr (SLICED) {
      e.ctx_doubles = slice_ctx_doubles(Slots::Lay::BW, Slots::Lay::MARG);
      e.solve_func_sliced = (const void*)&pn_scalar_kernel<Prob, NU, STRAT, GROUP, BDIAG, THREADS, 0, 1>;
      e.launch_solve_sliced = &launch_solve_sliced;
    }
    return e;
  }
};

// posterior sampling for the dense families (row-major or transposed slots): one warp per (member, sample)
inline cudaError_t launch_dense_sample(const SampleArgs& a, int Dn, int transposed, cudaStream_t s) {
  constexpr int WARPS = 4;
  DenseSampleArgs w;
  w.B = a.B; w.K = a.K; w.S = a.S; w.Dn = Dn; w.d = a.d; w.transposed = transposed; w.seed = a.seed;
  w.cond = a.cond; w.status = a.status; w.samples = a.samples;
  const size_t smem = (size_t)WARPS * 3 * Dn * sizeof(double);
  auto kern = pn_dense_sample_kernel<WARPS>;
  if (smem > 48 * 1024) {
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return ce;
  }
  const long long warps = a.B * a.S;
  kern<<<(unsigned)((warps + WARPS - 1) / WARPS), 32 * WARPS, smem, s>>>(w);
  return cudaGetLastError();
}

// what the dense builds with d > 1 and WARPS warps per CTA share: slots, smoothing and sampling kernels
template <class Prob, int NU, int STRAT, int WARPS>
struct DenseSlots {
  using Lay = DenseLayout<NU + 1, Prob::D>;
  static cudaError_t launch_smooth(const SmoothArgs& a, cudaStream_t s) {
    const size_t smem = (size_t)WARPS * Lay::SMEM_SMOOTH * sizeof(double);
    auto kern = pn_dense_smooth_kernel<NU + 1, Prob::D, STRAT, WARPS>;
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return ce;
    int grid = (int)((a.B + WARPS - 1) / WARPS);
    kern<<<grid, 32 * WARPS, smem, s>>>(a);
    return cudaGetLastError();
  }
  static cudaError_t launch_sample(const SampleArgs& a, cudaStream_t s) {
    return launch_dense_sample(a, (NU + 1) * Prob::D, 0, s);
  }
  static KernelEntry entry() {
    KernelEntry e;
    e.launch_sample = (STRAT == 1) ? &launch_sample : nullptr;
    e.dv = 1;
    e.problem = Prob::ID;
    e.nu = NU;
    e.strategy = STRAT;
    e.N = NU + 1;
    e.D = Prob::D;
    e.Q = Prob::Q;
    e.P = Prob::P;
    e.slot_doubles = (STRAT == 1) ? Lay::SLOT_FIX : Lay::SLOT_FILT;
    e.threads = 32 * WARPS;
    e.has_jac = Prob::HAS_JAC;
    e.launch_smooth = &launch_smooth;
    return e;
  }
};

// dense factorisation with d > 1: warp per IVP, D x D factors in shared memory
template <class Prob, int NU, int STRAT, int WARPS>
struct DenseInstance {
  using Slots = DenseSlots<Prob, NU, STRAT, WARPS>;
  static cudaError_t launch_solve(const SolveArgs& a, int grid, size_t smem, cudaStream_t s) {
    pn_dense_kernel<Prob, NU, STRAT, WARPS><<<grid, 32 * WARPS, smem, s>>>(a);
    return cudaGetLastError();
  }
  static KernelEntry entry() {
    KernelEntry e = Slots::entry();
    e.family = FAMILY_DENSE;
    e.group = 32;
    e.smem_doubles = Slots::Lay::SMEM;  // per warp (= per 32 threads), see make_plan
    e.solve_func = (const void*)&pn_dense_kernel<Prob, NU, STRAT, WARPS>;
    e.launch_solve = &launch_solve;
    return e;
  }
};

// dense factorisation with d > 1 and D <= 32: LANES lanes per IVP, columns in registers
template <class Prob, int NU, int STRAT, int LANES, int WARPS>
struct DenseRowsInstance {
  using RL = DenseRowsLayout<NU + 1, Prob::D>;
  static cudaError_t launch_solve(const SolveArgs& a, int grid, size_t smem, cudaStream_t s) {
    pn_dense_rows_kernel<Prob, NU, STRAT, LANES, WARPS><<<grid, 32 * WARPS, smem, s>>>(a);
    return cudaGetLastError();
  }
  static KernelEntry entry() {
    KernelEntry e = DenseSlots<Prob, NU, STRAT, WARPS>::entry();
    e.family = FAMILY_DENSE_ROWS;
    e.group = LANES;
    e.smem_doubles = (32 / LANES) * RL::SMEM_SLOT + (RL::TABLES + WARPS - 1) / WARPS;  // per warp (the tables exist once per CTA), see make_plan
    e.solve_func = (const void*)&pn_dense_rows_kernel<Prob, NU, STRAT, LANES, WARPS>;
    e.launch_solve = &launch_solve;
    return e;
  }
};

// isotropic problems with a large runtime dimension: CTA per IVP
template <class Prob, int NU, int STRAT, int THREADS, int PIPE = 0>
struct WideInstance {
  using Lay = Layout<NU + 1, 1>;
  static cudaError_t launch_solve(const SolveArgs& a, int grid, size_t smem, cudaStream_t s) {
    pn_scalar_kernel<Prob, NU, STRAT, 1, 0, THREADS, 1, 0, PIPE><<<grid, THREADS + 64 * PIPE, smem, s>>>(a);
    return cudaGetLastError();
  }
  static cudaError_t launch_smooth(const SmoothArgs& a, cudaStream_t s) {
    WideSmoothArgs w;
    w.B = a.B; w.K = a.K; w.d = a.wide_d; w.cond = a.cond; w.mean = a.wide_mean; w.status = a.status;
    w.u = a.u; w.u_std = a.u_std; w.marg_mean = a.marg_mean; w.marg_chol = a.marg_chol;
    pn_wide_smooth_kernel<NU + 1, STRAT, THREADS><<<(int)a.B, THREADS, 0, s>>>(w);
    return cudaGetLastError();
  }
  static cudaError_t launch_sample(const SampleArgs& a, cudaStream_t s) {
    WideSampleArgs w;
    w.B = a.B; w.K = a.K; w.S = a.S; w.d = a.d; w.seed = a.seed; w.cond = a.cond; w.status = a.status; w.samples = a.samples;
    const long long total = a.B * a.S * a.d;
    pn_wide_sample_kernel<NU + 1><<<(unsigned)((total + 127) / 128), 128, 0, s>>>(w);
    return cudaGetLastError();
  }
  // the caller passes dv = d, D = 1: the scratch layout and the reduction of the lane-per-dimension isotropic kernels
  static cudaError_t launch_lml(const LmlArgs& a, cudaStream_t s) {
    WideLmlArgs w;
    w.B = a.B; w.K = a.K; w.d = a.dv; w.cond = a.cond; w.data = a.data; w.obs_std = a.obs_std; w.w = a.w; w.logs = a.logs;
    pn_wide_lml_sweep_kernel<NU + 1><<<(unsigned)((a.B * a.dv + 127) / 128), 128, 0, s>>>(w);
    pn_lml_reduce_kernel<0><<<(unsigned)((a.B + 127) / 128), 128, 0, s>>>(a);
    return cudaGetLastError();
  }
  static KernelEntry entry() {
    KernelEntry e;
    e.launch_sample = (STRAT == 1) ? &launch_sample : nullptr;
    e.launch_lml = (STRAT == 1) ? &launch_lml : nullptr;
    e.family = FAMILY_WIDE;
    e.group = THREADS;
    e.dv = 1;
    e.problem = Prob::ID;
    e.nu = NU;
    e.strategy = STRAT;
    e.N = NU + 1;
    // runtime dimension; -32: the one-warp-per-IVP build for large ensembles; -160: the build with a backward warp (PIPE)
    e.D = PIPE ? -(THREADS + 32) : ((THREADS == 128) ? 0 : -THREADS);
    e.extra_threads = 64 * PIPE;  // an idle warp (keeps the backward warp off main warp 0's sub-partition) + the backward warp
    e.Q = Prob::Q;
    e.P = Prob::P;
    e.slot_doubles = Lay::BW + Lay::NT;  // factor part of a slot; + 2 n d per slot and 3 n d per member at run time
    e.smem_doubles = ((STRAT == 1) ? Lay::BW : 0) + Lay::PEND + Lay::MARG;  // per thread; + 2 d + warps per CTA
    e.threads = THREADS;
    e.has_jac = false;
    e.solve_func = (const void*)&pn_scalar_kernel<Prob, NU, STRAT, 1, 0, THREADS, 1, 0, PIPE>;
    e.launch_solve = &launch_solve;
    e.launch_smooth = &launch_smooth;
    return e;
  }
};

// thread-per-IVP kernels for small ensembles: THREADS filter lanes + THREADS backward lanes per CTA (PAIR = 1);
// same slots / smoothing / sampling / likelihood kernels as the thread-per-IVP family
template <class Prob, int NU, int THREADS>
struct PairInstance {
  using MB = pair::Mailbox<NU + 1, Prob::D>;
  static cudaError_t launch_solve(const SolveArgs& a, int grid, size_t smem, cudaStream_t s) {
    pn_scalar_kernel<Prob, NU, 1, 1, 0, THREADS, 0, 0, 0, 1><<<grid, 2 * THREADS, smem, s>>>(a);
    return cudaGetLastError();
  }
  static KernelEntry entry() {
    KernelEntry e = ScalarSlots<Prob, NU, 1, 1, 0>::entry();
    e.family = FAMILY_PAIR;
    e.threads = THREADS;
    e.extra_threads = THREADS;
    e.smem_doubles += MB::DOUBLES + (MB::INTS + 1) / 2;  // per filter lane: its thread-per-IVP state + the mailbox
    e.solve_func = (const void*)&pn_scalar_kernel<Prob, NU, 1, 1, 0, THREADS, 0, 0, 0, 1>;
    e.launch_solve = &launch_solve;
    return e;
  }
};

// dense factorisation with a large runtime dimension: CTA per IVP, blocked Householder QR + DMMA products
template <class Prob, int NU, int STRAT, int NB, int MINB>
struct DenseCtaInstance {
  static cudaError_t launch_solve(const SolveArgs& a, int grid, size_t smem, cudaStream_t s) {
    cta::pn_dense_cta_kernel<Prob, NU, STRAT, NB, MINB><<<grid, cta::T, smem, s>>>(a);
    return cudaGetLastError();
  }
  static cudaError_t launch_smooth(const SmoothArgs& a, cudaStream_t s) {
    cta::CtaSmoothArgs w;
    w.B = a.B; w.K = a.K; w.d = a.wide_d; w.n = NU + 1; w.cond = a.cond; w.scratch = a.wide_mean; w.status = a.status;
    w.u = a.u; w.u_std = a.u_std; w.marg_mean = a.marg_mean; w.marg_chol = a.marg_chol;
    const size_t smem = cta::smem_doubles<NB>((NU + 1) * a.wide_d) * sizeof(double);
    auto kern = cta::pn_dense_cta_smooth_kernel<STRAT, NB>;
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return ce;
    const int grid = (int)(a.B < a.wide_ctas ? a.B : a.wide_ctas);
    kern<<<grid, cta::T, smem, s>>>(w);
    return cudaGetLastError();
  }
  static cudaError_t launch_sample(const SampleArgs& a, cudaStream_t s) {
    return launch_dense_sample(a, (NU + 1) * a.d, 1, s);  // kernel-native transposed slots
  }
  static KernelEntry entry() {
    KernelEntry e;
    e.launch_sample = (STRAT == 1) ? &launch_sample : nullptr;
    e.family = FAMILY_DENSE_CTA;
    e.group = cta::T;
    e.dv = 1;
    e.problem = Prob::ID;
    e.nu = NU;
    e.strategy = STRAT;
    e.N = NU + 1;
    e.D = (MINB == 2) ? -2 : 0;  // runtime dimension; -2 marks the two-CTAs-per-SM build
    e.Q = Prob::Q;
    e.P = Prob::P;
    e.slot_doubles = 0;  // runtime: cta::slot_doubles
    e.smem_doubles = NB; // runtime: cta::smem_doubles<NB>; this field carries the panel width
    e.threads = cta::T;
    e.has_jac = Prob::HAS_JAC;
    e.solve_func = (const void*)&cta::pn_dense_cta_kernel<Prob, NU, STRAT, NB, MINB>;
    e.launch_solve = &launch_solve;
    e.launch_smooth = &launch_smooth;
    return e;
  }
};

struct Registrar {
  explicit Registrar(const KernelEntry& e) { register_kernel(e); }
};

#define PN_CAT2(a, b) a##b
#define PN_CAT(a, b) PN_CAT2(a, b)
#ifndef PN_SCALAR_THREADS
#define PN_SCALAR_THREADS 128
#endif
#define PN_REGISTER_SCALAR(Prob, NU, STRAT) \
  static ::pn::Registrar PN_CAT(pn_reg_, __COUNTER__)(::pn::ScalarInstance<::pn::Prob, NU, STRAT, 1, 0, PN_SCALAR_THREADS>::entry())
#define PN_REGISTER_DENSE(Prob, NU, STRAT, WARPS) \
  static ::pn::Registrar PN_CAT(pn_reg_, __COUNTER__)(::pn::DenseInstance<::pn::Prob, NU, STRAT, WARPS>::entry())
#define PN_REGISTER_DENSE_ROWS(Prob, NU, STRAT, LANES, WARPS) \
  static ::pn::Registrar PN_CAT(pn_reg_, __COUNTER__)(::pn::DenseRowsInstance<::pn::Prob, NU, STRAT, LANES, WARPS>::entry())
#define PN_REGISTER_PAIR(Prob, NU) \
  static ::pn::Registrar PN_CAT(pn_reg_, __COUNTER__)(::pn::PairInstance<::pn::Prob, NU, 128>::entry())
#define PN_REGISTER_DENSE_CTA(Prob, NU, STRAT, NB, MINB) \
  static ::pn::Registrar PN_CAT(pn_reg_, __COUNTER__)(::pn::DenseCtaInstance<::pn::cta::Prob, NU, STRAT, NB, MINB>::entry())
#define PN_REGISTER_WIDE(Prob, NU, STRAT) \
  static ::pn::Registrar PN_CAT(pn_reg_, __COUNTER__)(::pn::WideInstance<::pn::Prob, NU, STRAT, 128>::entry())
#define PN_REGISTER_WIDE_PIPE(Prob, NU, STRAT) \
  static ::pn::Registrar PN_CAT(pn_reg_, __COUNTER__)(::pn::WideInstance<::pn::Prob, NU, STRAT, 128, 1>::entry())
#define PN_REGISTER_WIDE_T(Prob, NU, STRAT, THREADS) \
  static ::pn::Registrar PN_CAT(pn_reg_, __COUNTER__)(::pn::WideInstance<::pn::Prob, NU, STRAT, THREADS>::entry())
#define PN_REGISTER_SCALAR_T(Prob, NU, STRAT, THREADS) \
  static ::pn::Registrar PN_CAT(pn_reg_, __COUNTER__)(::pn::ScalarInstance<::pn::Prob, NU, STRAT, 1, 0, THREADS>::entry())
#define PN_REGISTER_GROUP_T(Prob, NU, STRAT, GROUP, BDIAG, THREADS) \
  static ::pn::Registrar PN_CAT(pn_reg_, __COUNTER__)(::pn::ScalarInstance<::pn::Prob, NU, STRAT, GROUP, BDIAG, THREADS>::entry())
// lane-per-dimension kernels: GROUP lanes per IVP, BDIAG = 1 blockdiag / 0 isotropic
#define PN_REGISTER_GROUP(Prob, NU, STRAT, GROUP, BDIAG) \
  static ::pn::Registrar PN_CAT(pn_reg_, __COUNTER__)(::pn::ScalarInstance<::pn::Prob, NU, STRAT, GROUP, BDIAG, 128>::entry())

}  // namespace pn
