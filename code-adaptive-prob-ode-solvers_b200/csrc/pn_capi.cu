// pn_capi.cu -- C ABI (include/pn_b200.h) over the compiled kernel instances.
//
// What this replaces in the reference: the Python closure `solve_(u0, p)` of
// src/odecheckpts/ivpsolvers.py:55-91 (Taylor initialisation :63-68, solve_adaptive_save_at
// :71-77, backward marginalisation :80-81, QOI selection :84-89), batched over an ensemble.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/pn_b200.h"
#include "pn_jit.h"
#include "pn_registry.h"

namespace pn {

static std::vector<KernelEntry>& table() {
  static std::vector<KernelEntry> t;
  return t;
}
void register_kernel(const KernelEntry& e) { table().push_back(e); }
const KernelEntry* find_kernel(int family, int problem, int nu, int strategy, int d) {
  if (jit_is_user_problem(problem)) return jit_find(family, problem, nu, strategy, d);
  for (const auto& e : table())
    if (e.family == family && e.problem == problem && e.nu == nu && e.strategy == strategy && e.D == d) return &e;
  return nullptr;
}

static thread_local std::string g_err;
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

// Prior constant: lower Cholesky factor of the flipped Hilbert matrix Q1[i][j] = 1/(2nu-i-j+1)
// (SURVEY A.1).  Factorised in extended precision and rounded once, so the table does not
// depend on host compiler flags.
static void prior_lq(int nu, double* lq /* n*n row-major */) {
  const int n = nu + 1;
  std::vector<long double> Lc((size_t)n * n, 0.0L);
  for (int j = 0; j < n; ++j) {
    long double s = 1.0L / (long double)(2 * nu - 2 * j + 1);
    for (int k = 0; k < j; ++k) s -= Lc[j * n + k] * Lc[j * n + k];
    long double djj = sqrtl(s);
    Lc[j * n + j] = djj;
    for (int i = j + 1; i < n; ++i) {
      long double t = 1.0L / (long double)(2 * nu - i - j + 1);
      for (int k = 0; k < j; ++k) t -= Lc[i * n + k] * Lc[j * n + k];
      Lc[i * n + j] = t / djj;
    }
  }
  for (int i = 0; i < n * n; ++i) lq[i] = (double)Lc[i];
}

// optional kernel timing (pn_b200_set_profiling)
// State is per calling thread (the report that asked for timing reads its own events back) and the
// events are re-created when the thread moves to another device.
static thread_local bool g_profiling = false;
static thread_local cudaEvent_t g_ev[4];
static thread_local int g_ev_dev = -1;
static thread_local bool g_ev_recorded = false;

struct Geometry {
  int dev;
  const KernelEntry* k;
  size_t smem;
  int num_sms, ctas_per_sm;
};
static std::vector<Geometry> g_geom;
static std::mutex g_geom_mutex;
// Largest dynamic shared memory size a kernel's attribute has been raised to, per (device, kernel).  The
// attribute is ONE value per function: it is only ever raised, never set back to a smaller request (a
// kernel is launched with different sizes: the CTA-per-IVP kernels stage 2 d doubles and, for few
// members, their mean arrays).
struct SmemLimit {
  int dev;
  const void* func;
  size_t bytes;
};
static std::vector<SmemLimit> g_smem_limit;

static cudaError_t raise_smem_limit(int dev, const void* func, size_t bytes) {
  if (!func) return cudaSuccess;
  std::lock_guard<std::mutex> lock(g_geom_mutex);
  for (auto& l : g_smem_limit)
    if (l.dev == dev && l.func == func) {
      if (bytes <= l.bytes) return cudaSuccess;
      cudaError_t ce = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
      if (ce == cudaSuccess) l.bytes = bytes;
      return ce;
    }
  cudaError_t ce = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (ce == cudaSuccess) g_smem_limit.push_back({dev, func, bytes});
  return ce;
}

// private memory pool of the host entry point, one per device
struct HostPool {
  int dev;
  cudaMemPool_t pool;
};
static std::vector<HostPool> g_host_pools;
static cudaMemPool_t host_pool(int dev) {
  std::lock_guard<std::mutex> lock(g_geom_mutex);
  for (auto& hp : g_host_pools)
    if (hp.dev == dev) return hp.pool;
  cudaMemPoolProps props;
  memset(&props, 0, sizeof props);
  props.allocType = cudaMemAllocationTypePinned;
  props.handleTypes = cudaMemHandleTypeNone;
  props.location.type = cudaMemLocationTypeDevice;
  props.location.id = dev;
  cudaMemPool_t pool = nullptr;
  if (cudaMemPoolCreate(&pool, &props) != cudaSuccess) return nullptr;
  unsigned long long keep = ~0ULL;
  cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  g_host_pools.push_back({dev, pool});
  return pool;
}

struct Plan {
  const KernelEntry* k = nullptr;
  int grid = 0, ctas_per_sm = 0, num_sms = 0;
  size_t smem = 0;
  size_t ws_ticket = 256;  // header: work-queue ticket + stats (256 B), ordering histogram / cursors, order[B]
  size_t ws_cond = 0;      // bytes of conditionals
  size_t ws_wide = 0;      // wide kernels: per-member mean arrays
  int wide_smem_means = 0;  // wide kernels: how many mean arrays of the running member live in shared memory
  size_t ws_slice = 0;     // time-sliced scheduling: ready queues [G][B] + control words + parked states [B][ctx]
  int slice_shift = 0;     // queue group of a member = (k_next - 1) >> slice_shift, G <= 63 groups
  size_t ws_queue = 0;     // ... of which the ready queues (set to -1 before every launch)
  size_t ws_mle = 0;       // solver_mle: [B] final calibration factors
};

// ---------------------------------------------------------------------------------------
// Launch order for ragged ensembles: members that carry their own tolerances differ in step count
// by orders of magnitude (a 1e-3 ... 1e-10 sweep: ~25x at nu = 4).  A counting sort on the binary
// exponent of (atol + rtol) hands out the tightest tolerances first (longest-job-first), which
// removes most of the tail at the end of the persistent launch.  Scheduling only: results do not
// depend on it.
// ---------------------------------------------------------------------------------------
// control block of the time-sliced scheduler: sw[2] (queue mask, finished members) + 64 (pop, push) pairs
constexpr size_t SLICE_CONTROL_BYTES = 1024;
constexpr long long WIDE_SMEM_MAX_MEMBERS = 148;       // SMs of a B200: one CTA-per-IVP member per SM
constexpr size_t WIDE_SMEM_LIMIT_BYTES = 227 * 1024;   // dynamic shared memory per CTA on sm_100
constexpr int SLICE_MIN_CHECKPOINTS = 8;
constexpr size_t SLICE_MAX_QUEUE_BYTES = (size_t)512 << 20;
constexpr int ORDER_BUCKETS = 128;
constexpr size_t WS_HIST_OFFSET = 256, WS_CURSOR_OFFSET = WS_HIST_OFFSET + ORDER_BUCKETS * 4;
constexpr size_t WS_ORDER_OFFSET = WS_CURSOR_OFFSET + ORDER_BUCKETS * 4;
constexpr size_t WS_HEADER_CLEAR = WS_ORDER_OFFSET;

__device__ __forceinline__ int order_bucket(double atol, double rtol) {
  const double key = fabs(atol) + fabs(rtol);
  const int e = (int)((__double_as_longlong(key) >> 52) & 0x7ff);  // biased exponent; 0 for key == 0
  const int bk = e - (1023 - 100);                                 // 2^-100 ... 2^27
  return bk < 0 ? 0 : (bk >= ORDER_BUCKETS ? ORDER_BUCKETS - 1 : bk);
}
__global__ void pn_order_hist_kernel(const double* tol, long long B, unsigned* hist) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) atomicAdd(&hist[order_bucket(tol[2 * i], tol[2 * i + 1])], 1u);
}
__global__ void pn_order_scan_kernel(const unsigned* hist, unsigned* cursor) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    unsigned run = 0;
    for (int k = 0; k < ORDER_BUCKETS; ++k) {
      cursor[k] = run;
      run += hist[k];
    }
  }
}
__global__ void pn_order_scatter_kernel(const double* tol, long long B, unsigned* cursor, long long* order) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) order[atomicAdd(&cursor[order_bucket(tol[2 * i], tol[2 * i + 1])], 1u)] = i;
}

constexpr long long PAIR_MAX_MEMBERS = 148 * 128;  // thread-per-IVP PAIR build: one 128-lane CTA per SM
constexpr long long WIDE_WARP_MIN_BATCH = 592;  // CTA-per-IVP isotropic family: one warp per IVP from four members per SM on
constexpr long long DENSE_CTA_MAX_CTAS = 296;  // per-CTA scratch regions the workspace provides (2 per SM of a B200)
static size_t dense_cta_smem_bytes(const KernelEntry* k, const pn_b200_desc* d) {
  const int Dn = (d->nu + 1) * d->d;
  return (k->smem_doubles == 32 ? cta::smem_doubles<32>(Dn) : cta::smem_doubles<16>(Dn)) * sizeof(double);
}

static int resolve(const pn_b200_desc* d, const KernelEntry** out) {
  if (!d) return fail(PN_B200_ERR_ARGUMENT, "null descriptor");
  if (d->batch < 0 || d->num_save_at < 2) return fail(PN_B200_ERR_ARGUMENT, "need batch >= 0 and at least 2 save_at points");
  if (d->nu < 1 || d->nu > 8) return fail(PN_B200_ERR_UNSUPPORTED, "nu out of range");
  if (d->strategy != PN_B200_FILTER && d->strategy != PN_B200_FIXEDPOINT)
    return fail(PN_B200_ERR_ARGUMENT, "unknown strategy");
  if (d->correction != PN_B200_TS0 && d->correction != PN_B200_TS1)
    return fail(PN_B200_ERR_ARGUMENT, "unknown correction");
  if (d->calibration != PN_B200_CALIB_NONE && d->calibration != PN_B200_CALIB_DYNAMIC && d->calibration != PN_B200_CALIB_MLE)
    return fail(PN_B200_ERR_ARGUMENT, "unknown calibration");
  if ((d->flags & PN_B200_FLAG_RECORD) && d->strategy != PN_B200_FILTER)
    return fail(PN_B200_ERR_UNSUPPORTED, "trajectory recording is implemented for the filter strategy");
  const KernelEntry* k = nullptr;
  // thread-per-IVP family: isotropic EKF0 (any compiled d) and dense with d == 1
  bool scalar_ok = (d->factorisation == PN_B200_ISOTROPIC && d->correction == PN_B200_TS0) ||
                   (d->factorisation == PN_B200_DENSE && d->d == 1) ||
                   (d->factorisation == PN_B200_BLOCKDIAG && d->d == 1 && d->correction == PN_B200_TS0);
  if (scalar_ok) k = find_kernel(FAMILY_SCALAR, d->problem, d->nu, d->strategy, d->d);
  // Small ensembles of the thread-per-IVP family, fixed-point strategy: filter lane + backward lane per IVP
  // (PAIR build) while the members fit one filter warp per SM sub-partition (PN_B200_PAIR=0 switches it off;
  // results are bit-identical either way)
  if (k && k->family == FAMILY_SCALAR && d->strategy == PN_B200_FIXEDPOINT && d->calibration != PN_B200_CALIB_MLE &&
      !(d->flags & PN_B200_FLAG_RECORD)) {
    const char* pe = getenv("PN_B200_PAIR");
    if (!(pe && pe[0] == '0') && d->batch <= PAIR_MAX_MEMBERS) {
      const KernelEntry* kp = find_kernel(FAMILY_PAIR, d->problem, d->nu, d->strategy, d->d);
      if (kp) k = kp;
    }
  }
  // lane-per-dimension family: blockdiag EKF0, and isotropic EKF0 for problems too wide for one thread
  if (!k && d->correction == PN_B200_TS0 && d->factorisation == PN_B200_BLOCKDIAG)
    k = find_kernel(FAMILY_GROUP_BDIAG, d->problem, d->nu, d->strategy, d->d);
  if (!k && d->correction == PN_B200_TS0 && d->factorisation == PN_B200_ISOTROPIC)
    k = find_kernel(FAMILY_GROUP_ISO, d->problem, d->nu, d->strategy, d->d);
  // warp-per-IVP dense family: dense factorisation with d > 1, EKF0 or EKF1; the register-column kernel (D <= 32),
  // else the shared-memory kernel
  if (!k && d->factorisation == PN_B200_DENSE && d->d > 1) {
    k = find_kernel(FAMILY_DENSE_ROWS, d->problem, d->nu, d->strategy, d->d);
    if (!k) k = find_kernel(FAMILY_DENSE, d->problem, d->nu, d->strategy, d->d);
  }
  // CTA-per-IVP dense family: dense factorisation with a large runtime dimension (Brusselator N >= 5:
  // D = (nu+1) 2N > 40), blocked QR + DMMA products
  if (!k && d->factorisation == PN_B200_DENSE && d->d > 1 && (d->d % 2) == 0) {
    k = find_kernel(FAMILY_DENSE_CTA, d->problem, d->nu, d->strategy, 0);
    if (k && dense_cta_smem_bytes(k, d) > WIDE_SMEM_LIMIT_BYTES) k = nullptr;  // D too large for one CTA's panel
    // two CTAs per SM when their shared memory fits (+1 KB reserved per CTA) and there are members for them
    if (k && 2 * (dense_cta_smem_bytes(k, d) + 1024) <= WIDE_SMEM_LIMIT_BYTES && d->batch > 148) {
      const KernelEntry* k2 = find_kernel(FAMILY_DENSE_CTA, d->problem, d->nu, d->strategy, -2);
      if (k2) k = k2;
    }
  }
  // CTA-per-IVP wide family: isotropic EKF0 with a runtime dimension (Brusselator beyond the fixed sizes)
  if (!k && d->correction == PN_B200_TS0 && d->factorisation == PN_B200_ISOTROPIC && d->d >= 4 && d->d <= 4096 &&
      (d->d % 2) == 0)
  {
    k = find_kernel(FAMILY_WIDE, d->problem, d->nu, d->strategy, 0);
    // large ensembles: one warp per IVP (WIDE_WARP_MIN_BATCH members = four per SM; PN_B200_WIDE_WARP=0/1 forces)
    const char* ww = getenv("PN_B200_WIDE_WARP");
    const bool want_warp = ww ? (ww[0] == '1') : (d->batch >= WIDE_WARP_MIN_BATCH);
    if (k && want_warp) {
      const KernelEntry* k32 = find_kernel(FAMILY_WIDE, d->problem, d->nu, d->strategy, -32);
      if (k32) k = k32;
    } else if (k && d->strategy == PN_B200_FIXEDPOINT && d->batch <= WIDE_SMEM_MAX_MEMBERS) {
      // at most one member per SM: the build with a backward warp (PN_B200_WIDE_PIPE=0 switches it off for A/B runs)
      const char* wp = getenv("PN_B200_WIDE_PIPE");
      if (!(wp && wp[0] == '0')) {
        const KernelEntry* kp = find_kernel(FAMILY_WIDE, d->problem, d->nu, d->strategy, -160);
        if (kp) k = kp;
      }
    }
  }
  // trajectory recording: the dense factorisation with d > 1 records in the register-column kernel (D <= 32) and the
  // CTA-per-IVP dense kernel (the Brusselator's filter solves); the shared-memory dense kernel has no filter build
  if ((d->flags & PN_B200_FLAG_RECORD) &&
      ((k && k->family != FAMILY_SCALAR && k->family != FAMILY_GROUP_ISO && k->family != FAMILY_GROUP_BDIAG &&
        k->family != FAMILY_WIDE && k->family != FAMILY_DENSE_ROWS && k->family != FAMILY_DENSE_CTA) ||
       (!k && d->factorisation == PN_B200_DENSE && d->d > 1)))
    return fail(PN_B200_ERR_UNSUPPORTED, "trajectory recording is implemented for the thread-per-IVP, lane-per-dimension and "
                                         "CTA-per-IVP isotropic kernels and, for the dense factorisation with d > 1, the "
                                         "register-column kernel ((nu+1) d <= 32) and the CTA-per-IVP dense kernel");
  if (!k) {
    char buf[256];
    snprintf(buf, sizeof buf, "no kernel compiled for problem=%d nu=%d factorisation=%d correction=%d strategy=%d d=%d",
             d->problem, d->nu, d->factorisation, d->correction, d->strategy, d->d);
    return fail(PN_B200_ERR_UNSUPPORTED, buf);
  }
  if (d->calibration == PN_B200_CALIB_MLE && k->family != FAMILY_SCALAR)
    return fail(PN_B200_ERR_UNSUPPORTED, "solver_mle (running quasi-MLE calibration) is implemented for the thread-per-IVP kernels");
  if (k->Q != d->ode_order) return fail(PN_B200_ERR_ARGUMENT, "ode_order does not match the problem");
  if (d->correction == PN_B200_TS1 && !k->has_jac) return fail(PN_B200_ERR_UNSUPPORTED, "problem has no compiled Jacobian");
  if (d->num_params < 0 || d->num_params > (k->P > 0 ? k->P : 0)) return fail(PN_B200_ERR_ARGUMENT, "num_params exceeds the problem's parameter count");
  *out = k;
  return PN_B200_SUCCESS;
}

static int make_plan(const pn_b200_desc* d, Plan* p, bool need_device) {
  int rc = resolve(d, &p->k);
  if (rc) return rc;
  p->smem = family_is_dense(p->k->family)
                ? (size_t)p->k->smem_doubles * (p->k->threads / 32) * sizeof(double)  // per warp
                : (size_t)p->k->smem_doubles * p->k->threads * sizeof(double);        // per thread
  if (p->k->family == FAMILY_DENSE_CTA) p->smem = dense_cta_smem_bytes(p->k, d);
  if (p->k->family == FAMILY_WIDE) {
    p->smem += ((size_t)2 * d->d + p->k->threads / 32 + 2) * sizeof(double);
    // few members (at most one per SM: no occupancy to lose) whose mean arrays fit next to the rest
    const size_t one = (size_t)(d->nu + 1) * d->d * sizeof(double);
    if (d->batch <= WIDE_SMEM_MAX_MEMBERS) {
      while (p->wide_smem_means < 3 && p->smem + one <= WIDE_SMEM_LIMIT_BYTES) {
        p->smem += one;
        p->wide_smem_means += 1;
      }
    }
  }
  p->ws_ticket = (WS_ORDER_OFFSET + (size_t)d->batch * sizeof(long long) + 255) / 256 * 256;
  p->ws_cond = (size_t)d->num_save_at * p->k->slot_doubles * (size_t)d->batch * p->k->dv * sizeof(double);
  if (p->k->family == FAMILY_WIDE) {
    const size_t nd = (size_t)(d->nu + 1) * d->d;
    p->ws_cond = (size_t)d->batch * ((size_t)d->num_save_at * (p->k->slot_doubles + 2 * nd)) * sizeof(double);
    p->ws_wide = (size_t)d->batch * 3 * nd * sizeof(double);
  }
  if (p->k->family == FAMILY_DENSE_CTA) {
    const int Dn = (d->nu + 1) * d->d;
    const long long ctas = d->batch < DENSE_CTA_MAX_CTAS ? d->batch : DENSE_CTA_MAX_CTAS;
    p->ws_cond = (size_t)d->batch * d->num_save_at * cta::slot_doubles(Dn, d->strategy == PN_B200_FIXEDPOINT) * sizeof(double);
    p->ws_wide = (size_t)ctas * cta::scratch_doubles(Dn, d->d, d->ode_order) * sizeof(double);
  }
  if (d->calibration == PN_B200_CALIB_MLE) p->ws_mle = ((size_t)d->batch * sizeof(double) + 255) / 256 * 256;
  // time-sliced scheduling (pn_scalar_kernel.cuh: SolveArgs::slice): thread-per-IVP kernels, enough
  // checkpoints to slice at, bounded queue memory
  if (p->k->ctx_doubles > 0 && d->num_save_at >= SLICE_MIN_CHECKPOINTS && d->batch > 1 && d->batch < 0x7fffffffLL &&
      d->calibration != PN_B200_CALIB_MLE &&  // (the parked context does not carry the running MLE sum)
      !(d->flags & (PN_B200_FLAG_RECORD | PN_B200_FLAG_FIXED_GRID))) {
    int shift = 0;
    while (((d->num_save_at - 2) >> shift) > 62) ++shift;
    const size_t groups = (size_t)((d->num_save_at - 2) >> shift) + 1;
    const size_t queue = groups * d->batch * sizeof(int32_t);
    if (queue <= SLICE_MAX_QUEUE_BYTES) {
      p->slice_shift = shift;
      p->ws_queue = (queue + 255) / 256 * 256;
      p->ws_slice = p->ws_queue + SLICE_CONTROL_BYTES + (size_t)d->batch * p->k->ctx_doubles * sizeof(double);
    }
  }
  if (!need_device) return PN_B200_SUCCESS;
  if (p->k->jit) {
    rc = jit_load(p->k);
    if (rc) return rc;
  }
  int dev = 0;
  cudaError_t ce = cudaGetDevice(&dev);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
  // launch geometry is cached per (device, kernel): the attribute / occupancy queries are not free
  {
    std::lock_guard<std::mutex> lock(g_geom_mutex);
    for (const auto& g : g_geom)
      if (g.dev == dev && g.k == p->k && g.smem == p->smem) {
        p->num_sms = g.num_sms;
        p->ctas_per_sm = g.ctas_per_sm;
      }
  }
  if (p->ctas_per_sm == 0) {
    ce = cudaDeviceGetAttribute(&p->num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
    ce = raise_smem_limit(dev, p->k->solve_func, p->smem);
    if (ce == cudaSuccess) ce = raise_smem_limit(dev, p->k->solve_func_sliced, p->smem);
    if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(ce));
    int occ = 0;
    ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, p->k->solve_func, p->k->threads + p->k->extra_threads, p->smem);
    if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
    if (occ < 1) return fail(PN_B200_ERR_CUDA, "kernel does not fit on an SM");
    // the time-sliced instantiation is a different kernel (its own register count): the persistent grid must be
    // co-resident whichever of the two is launched
    if (p->k->solve_func_sliced) {
      int occ_sliced = 0;
      ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_sliced, p->k->solve_func_sliced, p->k->threads + p->k->extra_threads, p->smem);
      if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
      if (occ_sliced >= 1 && occ_sliced < occ) occ = occ_sliced;
    }
    p->ctas_per_sm = occ;
    std::lock_guard<std::mutex> lock(g_geom_mutex);
    g_geom.push_back({dev, p->k, p->smem, p->num_sms, occ});
  }
  const int occ = p->ctas_per_sm;
  long long per_cta = (p->k->family == FAMILY_WIDE) ? 1 : p->k->threads / p->k->group;  // IVPs per CTA
  long long want = (d->batch + per_cta - 1) / per_cta;
  long long cap = (long long)occ * p->num_sms;
  if (p->k->family == FAMILY_DENSE_CTA && cap > DENSE_CTA_MAX_CTAS) cap = DENSE_CTA_MAX_CTAS;
  p->grid = (int)(want < cap ? want : cap);
  if (p->grid < 1) p->grid = 1;
  return PN_B200_SUCCESS;
}

// ---------------------------------------------------------------------------------------
// fp64 peak microbenchmark: 16 independent DFMA chains per thread, fully register resident
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pn_dfma_peak_kernel(double* out, double a, double b, int iters) {
  double x[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) x[i] = (double)(threadIdx.x + i) * 1e-3;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 8; ++r) {
#pragma unroll
      for (int i = 0; i < 16; ++i) x[i] = fma(x[i], a, b);
    }
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += x[i];
  if (s == 123456.789) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

__global__ void pn_selftest_math_kernel(const double* x, const double* y, double* r, double* sq, double* pw, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  r[i] = rcp(x[i]);
  sq[i] = dsqrt(fabs(x[i]));
  pw[i] = det_pow(fabs(x[i]), y[i]);
}

// out[8 i ..]: (v0, beta, g, ng) of make_reflector, then of the plain composition sqrt -> reciprocal
__global__ void pn_selftest_reflector_kernel(const double* alpha, const double* sigma2, double* out, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Reflector a = make_reflector(alpha[i], sigma2[i]);
  const Reflector b = make_reflector_plain(alpha[i], sigma2[i]);
  double* o = out + 8 * i;
  o[0] = a.v0, o[1] = a.beta, o[2] = a.g, o[3] = a.ng;
  o[4] = b.v0, o[5] = b.beta, o[6] = b.g, o[7] = b.ng;
}

}  // namespace pn

using namespace pn;

extern "C" {

const char* pn_b200_last_error(void) { return g_err.c_str(); }

int pn_b200_supported(const pn_b200_desc* desc) {
  const KernelEntry* k = nullptr;
  return resolve(desc, &k);
}

size_t pn_b200_workspace_bytes(const pn_b200_desc* desc) {
  Plan p;
  if (make_plan(desc, &p, false)) return 0;
  return p.ws_ticket + p.ws_cond + p.ws_wide + p.ws_slice + p.ws_mle;
}

int pn_b200_compile(const pn_b200_desc* desc) {
  const KernelEntry* k = nullptr;
  int rc = resolve(desc, &k);
  if (rc == PN_B200_SUCCESS && k->jit) rc = jit_load(k);
  return rc;
}

int pn_b200_output_sizes(const pn_b200_desc* desc, pn_b200_sizes* sz) {
  const KernelEntry* k = nullptr;
  int rc = resolve(desc, &k);
  if (rc) return rc;
  if (!sz) return fail(PN_B200_ERR_ARGUMENT, "null sizes");
  const size_t B = (size_t)desc->batch, K = (size_t)desc->num_save_at, d = (size_t)desc->d, n = (size_t)desc->nu + 1;
  const bool bdiag = desc->factorisation == PN_B200_BLOCKDIAG && d > 1;
  const bool dense = desc->factorisation == PN_B200_DENSE && d > 1;
  const bool rec = (desc->flags & PN_B200_FLAG_RECORD) != 0;
  const size_t cap = rec ? (size_t)desc->traj_capacity : 0;
  memset(sz, 0, sizeof *sz);
  sz->u = sz->u_std = B * K * d;
  sz->marg_mean = B * K * n * d;
  sz->marg_chol = B * K * (bdiag ? d : (dense ? d * d : 1)) * n * n;
  sz->output_scale = B * K * (bdiag ? d : 1);
  sz->n_accepted = B * K;
  sz->n_rejected = B;
  sz->status = B;
  sz->traj_t = cap * B;
  sz->traj_u = cap * d * B;
  sz->traj_std = cap * (dense ? d : 1) * B;
  sz->traj_len = rec ? B : 0;
  return PN_B200_SUCCESS;
}

int pn_b200_get_kernel_info(const pn_b200_desc* desc, pn_b200_kernel_info* info) {
  Plan p;
  int rc = make_plan(desc, &p, true);
  if (rc) return rc;
  cudaFuncAttributes fa;
  cudaError_t ce = cudaFuncGetAttributes(&fa, p.k->solve_func);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
  info->threads_per_cta = p.k->threads + p.k->extra_threads;
  info->ctas_per_sm = p.ctas_per_sm;
  info->num_sms = p.num_sms;
  info->grid = p.grid;
  info->registers_per_thread = fa.numRegs;
  info->static_smem_bytes = (int32_t)fa.sharedSizeBytes;
  info->dynamic_smem_bytes = (int32_t)p.smem;
  info->local_bytes_per_thread = (int32_t)fa.localSizeBytes;
  return PN_B200_SUCCESS;
}

int pn_b200_solve_save_at(const pn_b200_desc* desc, const double* u0, const double* params,
                          const double* tol, const double* save_at, const double* output_scale0,
                          double* u, double* u_std, double* marg_mean, double* marg_chol,
                          double* output_scale, int64_t* n_accepted, int64_t* n_rejected, int32_t* status, double* traj_t,
                          double* traj_u, double* traj_std, int64_t* traj_len, void* workspace,
                          size_t workspace_bytes, void* cuda_stream) {
  Plan p;
  int rc = make_plan(desc, &p, true);
  if (rc) return rc;
  if (desc->batch == 0) return PN_B200_SUCCESS;
  if (!u0 || !save_at || !u || !u_std || !n_accepted || !n_rejected || !status)
    return fail(PN_B200_ERR_ARGUMENT, "null required buffer");
  if (desc->num_params > 0 && !params) return fail(PN_B200_ERR_ARGUMENT, "params is null but num_params > 0");
  if ((desc->flags & PN_B200_FLAG_RECORD) && (!traj_t || !traj_u || !traj_std || !traj_len || desc->traj_capacity < 2))
    return fail(PN_B200_ERR_ARGUMENT, "trajectory recording needs traj buffers and traj_capacity >= 2");
  if (!workspace || workspace_bytes < p.ws_ticket + p.ws_cond + p.ws_wide + p.ws_slice + p.ws_mle)
    return fail(PN_B200_ERR_WORKSPACE, "workspace too small");
  cudaStream_t stream = (cudaStream_t)cuda_stream;

  SolveArgs a;
  memset(&a, 0, sizeof a);
  a.correction = desc->correction;
  a.calibration = desc->calibration;
  a.flags = desc->flags;
  a.num_params = desc->num_params;
  a.atol = desc->atol;
  a.rtol = desc->rtol;
  a.dt0 = desc->dt0;
  a.safety = desc->safety;
  a.factor_min = desc->factor_min;
  a.factor_max = desc->factor_max;
  const double nn = (double)(desc->nu + 1);
  a.pow_i = desc->power_integral / nn;
  a.pow_p = desc->power_proportional / nn;
  a.B = desc->batch;
  a.K = desc->num_save_at;
  a.max_attempts = desc->max_attempts;
  a.u0 = u0;
  a.params = params;
  a.tol = tol;
  a.save_at = save_at;
  a.save_stride = (desc->flags & PN_B200_FLAG_MEMBER_GRIDS) ? desc->num_save_at : 0;
  a.sigma0 = output_scale0;
  a.ticket = (unsigned long long*)workspace;
  a.cond = (double*)((char*)workspace + p.ws_ticket);
  a.wide_d = (p.k->family == FAMILY_WIDE || p.k->family == FAMILY_DENSE_CTA) ? desc->d : 0;
  a.wide_smem_means = p.wide_smem_means;
  a.wide_mean = (double*)((char*)workspace + p.ws_ticket + p.ws_cond);
  a.out_scale = output_scale;
  a.mle_scale = p.ws_mle ? (double*)((char*)workspace + p.ws_ticket + p.ws_cond + p.ws_wide + p.ws_slice) : nullptr;
  a.n_accepted = (long long*)n_accepted;
  a.n_rejected = (long long*)n_rejected;
  a.status = status;
  a.traj_t = traj_t;
  a.traj_u = traj_u;
  a.traj_std = traj_std;
  a.traj_cap = desc->traj_capacity;
  a.traj_len = (long long*)traj_len;
  prior_lq(desc->nu, a.lq);

  cudaError_t ce = cudaMemsetAsync(workspace, 0, WS_HEADER_CLEAR, stream);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
  a.order = nullptr;
  if (tol && desc->batch > 1 && desc->batch < 0xffffffffLL) {
    unsigned* hist = (unsigned*)((char*)workspace + WS_HIST_OFFSET);
    unsigned* cursor = (unsigned*)((char*)workspace + WS_CURSOR_OFFSET);
    long long* order = (long long*)((char*)workspace + WS_ORDER_OFFSET);
    const unsigned blocks = (unsigned)((desc->batch + 255) / 256);
    pn_order_hist_kernel<<<blocks, 256, 0, stream>>>(tol, desc->batch, hist);
    pn_order_scan_kernel<<<1, 32, 0, stream>>>(hist, cursor);
    pn_order_scatter_kernel<<<blocks, 256, 0, stream>>>(tol, desc->batch, cursor, order);
    ce = cudaGetLastError();
    if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, std::string("ordering kernels: ") + cudaGetErrorString(ce));
    a.order = order;
  }
  // time-sliced scheduling: uniform tolerances only (ragged ensembles get the longest-first order
  // above instead), and only when the ensemble does not fit the resident lanes anyway
  bool sliced = false;
  if (p.ws_slice > 0 && p.k->solve_func_sliced && !tol && desc->batch > (int64_t)p.grid * p.k->threads &&
      !getenv("PN_B200_NO_SLICE")) {
    char* base = (char*)workspace + p.ws_ticket + p.ws_cond + p.ws_wide;
    ce = cudaMemsetAsync(base, 0xff, p.ws_queue, stream);
    if (ce == cudaSuccess) ce = cudaMemsetAsync(base + p.ws_queue, 0, SLICE_CONTROL_BYTES, stream);
    if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
    sliced = true;
    long long quantum = SLICE_QUANTUM;
    if (const char* q = getenv("PN_B200_SLICE_QUANTUM")) quantum = atoll(q);
    if (quantum < 1 || (quantum & (quantum - 1))) return fail(PN_B200_ERR_ARGUMENT, "PN_B200_SLICE_QUANTUM must be a power of two");
    a.slice_mask = quantum - 1;
    a.slice_shift = p.slice_shift;
    a.squeue = (int32_t*)base;
    a.sw = (unsigned long long*)(base + p.ws_queue);
    a.sq = (unsigned*)(a.sw + 2);
    a.ctx = (double*)(base + p.ws_queue + SLICE_CONTROL_BYTES);
  }
  const bool prof = g_profiling;
  if (prof) {
    int dev_now = 0;
    cudaGetDevice(&dev_now);
    if (g_ev_dev != dev_now) {
      if (g_ev_dev >= 0)
        for (auto& e : g_ev) cudaEventDestroy(e);
      for (auto& e : g_ev) cudaEventCreate(&e);
      g_ev_dev = dev_now;
      g_ev_recorded = false;
    }
  }
  if (prof) cudaEventRecord(g_ev[0], stream);
  if (p.k->jit)
    ce = jit_launch_solve(p.k, sliced, a, p.grid, p.smem, stream);
  else
    ce = sliced ? p.k->launch_solve_sliced(a, p.grid, p.smem, stream) : p.k->launch_solve(a, p.grid, p.smem, stream);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, std::string("solve kernel launch: ") + cudaGetErrorString(ce));
  if (prof) {
    cudaEventRecord(g_ev[1], stream);
    cudaEventRecord(g_ev[2], stream);
  }

  SmoothArgs s;
  s.B = desc->batch;
  s.K = desc->num_save_at;
  s.dv = p.k->dv;
  s.chol_per_dim = (p.k->family == FAMILY_GROUP_BDIAG) ? 1 : 0;
  s.wide_d = a.wide_d;
  s.wide_mean = a.wide_mean;
  s.wide_ctas = p.grid;
  s.cond = a.cond;
  s.mle_scale = a.mle_scale;
  s.status = status;
  s.u = u;
  s.u_std = u_std;
  s.marg_mean = marg_mean;
  s.marg_chol = marg_chol;
  ce = p.k->jit ? jit_launch_smooth(p.k, s, stream) : p.k->launch_smooth(s, stream);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, std::string("smoothing kernel launch: ") + cudaGetErrorString(ce));
  if (prof) {
    cudaEventRecord(g_ev[3], stream);
    g_ev_recorded = true;
  }
  return PN_B200_SUCCESS;
}

int pn_b200_markov_sample(const pn_b200_desc* desc, const void* workspace, size_t workspace_bytes,
                          const int32_t* status, uint64_t seed, int64_t num_samples, double* samples,
                          void* cuda_stream) {
  Plan p;
  int rc = make_plan(desc, &p, false);
  if (rc == PN_B200_SUCCESS && p.k->jit) rc = jit_load(p.k);
  if (rc) return rc;
  if (desc->strategy != PN_B200_FIXEDPOINT || !(p.k->launch_sample || p.k->sample_func))
    return fail(PN_B200_ERR_UNSUPPORTED, "posterior sampling needs a fixed-point solve");
  if (!workspace || workspace_bytes < p.ws_ticket + p.ws_cond || !samples || !status || num_samples < 1)
    return fail(PN_B200_ERR_ARGUMENT, "bad sampling arguments");
  if (desc->batch == 0) return PN_B200_SUCCESS;
  SampleArgs a;
  a.B = desc->batch;
  a.K = desc->num_save_at;
  a.S = num_samples;
  a.dv = p.k->dv;
  a.d = desc->d;
  a.seed = seed;
  a.cond = (const double*)((const char*)workspace + p.ws_ticket);
  a.status = status;
  a.samples = samples;
  cudaError_t ce = p.k->jit ? jit_launch_sample(p.k, a, (cudaStream_t)cuda_stream) : p.k->launch_sample(a, (cudaStream_t)cuda_stream);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, std::string("sampling kernel launch: ") + cudaGetErrorString(ce));
  return PN_B200_SUCCESS;
}

int pn_b200_log_marginal_likelihood(const pn_b200_desc* desc, const void* workspace, size_t workspace_bytes,
                                    const int32_t* status, const double* data, const double* obs_std,
                                    double* lml, void* cuda_stream) {
  Plan p;
  int rc = make_plan(desc, &p, false);
  if (rc == PN_B200_SUCCESS && p.k->jit) rc = jit_load(p.k);
  if (rc) return rc;
  if (desc->strategy != PN_B200_FIXEDPOINT || !(p.k->launch_lml || p.k->lml_func))
    return fail(PN_B200_ERR_UNSUPPORTED, "the log marginal likelihood needs a fixed-point solve of the thread-per-IVP, lane-per-dimension or CTA-per-IVP isotropic family");
  if (!workspace || workspace_bytes < p.ws_ticket + p.ws_cond || !status || !data || !obs_std || !lml)
    return fail(PN_B200_ERR_ARGUMENT, "bad likelihood arguments");
  if (desc->batch == 0) return PN_B200_SUCCESS;
  cudaStream_t stream = (cudaStream_t)cuda_stream;
  LmlArgs a;
  a.B = desc->batch;
  a.K = desc->num_save_at;
  // CTA-per-IVP isotropic family: one virtual member per column, as in the lane-per-dimension isotropic kernels
  const int lml_dv = (p.k->family == FAMILY_WIDE) ? desc->d : p.k->dv;
  a.dv = lml_dv;
  a.D = desc->d / lml_dv;
  a.per_dim = (p.k->family == FAMILY_GROUP_BDIAG) ? 1 : 0;
  a.cond = (const double*)((const char*)workspace + p.ws_ticket);
  a.status = status;
  a.data = data;
  a.obs_std = obs_std;
  a.lml = lml;
  // scratch: whitened residuals [B][K][d] + log|s| [B*dv][K], stream-ordered
  const size_t nw = (size_t)desc->batch * desc->num_save_at * desc->d, nl = (size_t)desc->batch * lml_dv * desc->num_save_at;
  double* scratch = nullptr;
  cudaError_t ce = cudaMallocAsync((void**)&scratch, (nw + nl) * sizeof(double), stream);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, std::string("cudaMallocAsync: ") + cudaGetErrorString(ce));
  a.w = scratch;
  a.logs = scratch + nw;
  ce = p.k->jit ? jit_launch_lml(p.k, a, stream) : p.k->launch_lml(a, stream);
  cudaFreeAsync(scratch, stream);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, std::string("likelihood kernel launch: ") + cudaGetErrorString(ce));
  return PN_B200_SUCCESS;
}

int pn_b200_set_profiling(int enable) {
  g_profiling = enable != 0;
  return PN_B200_SUCCESS;
}

int pn_b200_get_last_timing(float* solve_ms, float* smooth_ms) {
  if (!g_ev_recorded) return fail(PN_B200_ERR_ARGUMENT, "no profiled solve has been issued");
  cudaError_t ce = cudaEventSynchronize(g_ev[3]);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
  cudaEventElapsedTime(solve_ms, g_ev[0], g_ev[1]);
  cudaEventElapsedTime(smooth_ms, g_ev[2], g_ev[3]);
  return PN_B200_SUCCESS;
}

int pn_b200_solve_save_at_host(const pn_b200_desc* desc, const double* u0, const double* params,
                               const double* tol, const double* save_at, const double* output_scale0,
                               double* u, double* u_std, double* marg_mean, double* marg_chol,
                               double* output_scale, int64_t* n_accepted, int64_t* n_rejected, int32_t* status, double* traj_t,
                               double* traj_u, double* traj_std, int64_t* traj_len, int device) {
  pn_b200_sizes sz;
  int rc = pn_b200_output_sizes(desc, &sz);
  if (rc) return rc;
  if (desc->batch == 0) return PN_B200_SUCCESS;
  // per-member grids arrive in host memory here, so their precondition is checked: every row strictly increasing
  const bool member_grids = (desc->flags & PN_B200_FLAG_MEMBER_GRIDS) != 0;
  const size_t rows = member_grids ? (size_t)desc->batch : 1, nk = (size_t)desc->num_save_at;
  if (member_grids) {
    if (!save_at) return fail(PN_B200_ERR_ARGUMENT, "null required buffer");
    for (size_t r = 0; r < rows; ++r)
      for (size_t k = 1; k < nk; ++k)
        if (!(save_at[r * nk + k] > save_at[r * nk + k - 1])) {
          char buf[128];
          snprintf(buf, sizeof buf, "save_at row %zu is not strictly increasing at index %zu", r, k);
          return fail(PN_B200_ERR_ARGUMENT, buf);
        }
  }
  // the caller's current device is restored on every exit path
  struct DeviceGuard {
    int prev = -1;
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  } guard;
  cudaError_t ce = cudaGetDevice(&guard.prev);
  if (ce != cudaSuccess) guard.prev = -1;
  ce = cudaSetDevice(device);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
  const size_t B = (size_t)desc->batch, K = (size_t)desc->num_save_at, d = (size_t)desc->d;
  const size_t q = (size_t)desc->ode_order, P = (size_t)desc->num_params;
  struct Buf {
    void** dev;
    const void* host_in;
    void* host_out;
    size_t bytes;
  };
  void *d_u0 = 0, *d_par = 0, *d_tol = 0, *d_save = 0, *d_os = 0, *d_u = 0, *d_std = 0, *d_mm = 0, *d_mc = 0;
  void* d_sc = 0;
  void *d_nacc = 0, *d_nrej = 0, *d_stat = 0, *d_tt = 0, *d_tu = 0, *d_ts = 0, *d_tl = 0, *d_ws = 0;
  size_t ws_bytes = pn_b200_workspace_bytes(desc);
  Buf bufs[] = {
      {&d_u0, u0, nullptr, B * q * d * 8},
      {&d_par, P ? params : nullptr, nullptr, P ? B * P * 8 : 0},
      {&d_tol, tol, nullptr, tol ? B * 2 * 8 : 0},
      {&d_save, save_at, nullptr, rows * K * 8},
      {&d_os, output_scale0, nullptr, output_scale0 ? B * 8 : 0},
      {&d_u, nullptr, u, sz.u * 8},
      {&d_std, nullptr, u_std, sz.u_std * 8},
      {&d_mm, nullptr, marg_mean, marg_mean ? sz.marg_mean * 8 : 0},
      {&d_mc, nullptr, marg_chol, marg_chol ? sz.marg_chol * 8 : 0},
      {&d_sc, nullptr, output_scale, output_scale ? sz.output_scale * 8 : 0},
      {&d_nacc, nullptr, n_accepted, sz.n_accepted * 8},
      {&d_nrej, nullptr, n_rejected, sz.n_rejected * 8},
      {&d_stat, nullptr, status, sz.status * 4},
      {&d_tt, nullptr, traj_t, sz.traj_t * 8},
      {&d_tu, nullptr, traj_u, sz.traj_u * 8},
      {&d_ts, nullptr, traj_std, sz.traj_std * 8},
      {&d_tl, nullptr, traj_len, sz.traj_len * 8},
      {&d_ws, nullptr, nullptr, ws_bytes},
  };
  // The host entry allocates from a PRIVATE stream-ordered pool per device (never the process's default
  // pool, which other libraries share): freed blocks stay in it between calls, so the multi-GB workspace
  // is not re-mapped on every solve, and pn_b200_trim() hands the memory back to the driver.
  cudaMemPool_t pool = host_pool(device);
  if (!pool) return fail(PN_B200_ERR_CUDA, "cannot create the host entry point's memory pool");
  cudaStream_t stream;
  ce = cudaStreamCreate(&stream);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
  rc = PN_B200_SUCCESS;
  for (auto& bf : bufs) {
    if (!bf.bytes) continue;
    ce = cudaMallocFromPoolAsync(bf.dev, bf.bytes, pool, stream);
    if (ce != cudaSuccess) { rc = fail(PN_B200_ERR_CUDA, std::string("cudaMallocAsync: ") + cudaGetErrorString(ce)); break; }
    if (bf.host_in) {
      ce = cudaMemcpyAsync(*bf.dev, bf.host_in, bf.bytes, cudaMemcpyHostToDevice, stream);
      if (ce != cudaSuccess) { rc = fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce)); break; }
    }
  }
  if (rc == PN_B200_SUCCESS)
    rc = pn_b200_solve_save_at(desc, (const double*)d_u0, (const double*)d_par, (const double*)d_tol,
                               (const double*)d_save, (const double*)d_os, (double*)d_u, (double*)d_std,
                               (double*)d_mm, (double*)d_mc, (double*)d_sc, (int64_t*)d_nacc, (int64_t*)d_nrej,
                               (int32_t*)d_stat, (double*)d_tt, (double*)d_tu, (double*)d_ts, (int64_t*)d_tl,
                               d_ws, ws_bytes, stream);
  if (rc == PN_B200_SUCCESS) {
    for (auto& bf : bufs) {
      if (!bf.bytes || !bf.host_out) continue;
      ce = cudaMemcpyAsync(bf.host_out, *bf.dev, bf.bytes, cudaMemcpyDeviceToHost, stream);
      if (ce != cudaSuccess) { rc = fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce)); break; }
    }
  }
  ce = cudaStreamSynchronize(stream);
  if (ce != cudaSuccess && rc == PN_B200_SUCCESS) rc = fail(PN_B200_ERR_CUDA, std::string("stream sync: ") + cudaGetErrorString(ce));
  for (auto& bf : bufs)
    if (*bf.dev) cudaFreeAsync(*bf.dev, stream);
  cudaStreamSynchronize(stream);
  cudaStreamDestroy(stream);
  return rc;
}

int pn_b200_trim(int device) {
  std::lock_guard<std::mutex> lock(g_geom_mutex);
  for (auto& hp : g_host_pools)
    if (hp.dev == device) {
      cudaError_t ce = cudaMemPoolTrimTo(hp.pool, 0);
      return ce == cudaSuccess ? PN_B200_SUCCESS : fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
    }
  return PN_B200_SUCCESS;
}

// Test hook (not part of the public header): evaluates the kernels' branch-free rcp / sqrt / pow.
int pn_b200_selftest_math(const double* x, const double* y, double* r, double* sq, double* pw, long long n) {
  pn_selftest_math_kernel<<<(unsigned)((n + 255) / 256), 256>>>(x, y, r, sq, pw, n);
  return cudaGetLastError() == cudaSuccess ? 0 : PN_B200_ERR_CUDA;
}

// Test hook: the Householder reflector scalars of the kernels next to their plain composition (8 doubles per input).
int pn_b200_selftest_reflector(const double* alpha, const double* sigma2, double* out, long long n) {
  pn_selftest_reflector_kernel<<<(unsigned)((n + 255) / 256), 256>>>(alpha, sigma2, out, n);
  return cudaGetLastError() == cudaSuccess ? 0 : PN_B200_ERR_CUDA;
}

int pn_b200_measure_fp64_peak(double* tflops, void* cuda_stream) {
  cudaStream_t stream = (cudaStream_t)cuda_stream;
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceProp prop;
  cudaError_t ce = cudaGetDeviceProperties(&prop, dev);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
  const int threads = 256, ctas = prop.multiProcessorCount * 8, iters = 4096;
  double* out = nullptr;
  ce = cudaMalloc(&out, (size_t)threads * ctas * sizeof(double));
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0, stream);
    pn_dfma_peak_kernel<<<ctas, threads, 0, stream>>>(out, 0.999999, 1e-9, iters);
    cudaEventRecord(e1, stream);
    ce = cudaEventSynchronize(e1);
    if (ce != cudaSuccess) break;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    double flops = 2.0 * 16 * 8 * (double)iters * threads * (double)ctas;
    double tf = flops / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, cudaGetErrorString(ce));
  *tflops = best;
  return PN_B200_SUCCESS;
}

}  // extern "C"
