// pn_jit.cu -- user-defined vector fields: NVRTC compiles the kernel templates of the built-in problems for a user's
// functor at run time (pn_user_problem.cuh), one module per (problem, kernel family, nu, strategy), compiled on first
// use and cached for the life of the process.
//
// Modules are loaded as context-independent libraries (cudaLibraryLoadData); their kernel handles (cudaKernel_t)
// are accepted wherever the runtime takes a `const void*` kernel (cudaLaunchKernel, cudaFuncGetAttributes,
// cudaFuncSetAttribute, cudaOccupancy*), so the launch geometry code of pn_capi.cu serves them unchanged, on every
// device.  The headers the kernels need are embedded in the library at build time (pn_jit_sources.inc, generated
// by build.py): the library does not read the source tree at run time.
#include <nvrtc.h>
#include <string.h>

#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/pn_b200.h"
#include "pn_jit.h"

namespace pn {
namespace {

#include "pn_jit_sources.inc"  // kJitSources[]: {file name, text} of the headers below

// nvcc's flags for the built-in kernels (build.py), in NVRTC's spelling
const char* const kNvrtcOptions[] = {
    "-arch=sm_100a", "-std=c++17", "-lineinfo", "-fmad=false", "-prec-div=true", "-prec-sqrt=true",
    "-default-device", "-diag-suppress=177,128",
};

constexpr int MAX_DIM = 32;     // lane per dimension: one IVP per warp at most
constexpr int MAX_PARAMS = 64;  // parameters per member (the kernels keep them in registers)

struct ProblemRec {
  int id;
  std::string name, source;
  int form, d, q, P;
};

// the built-in problems that have a fixed size, for pn_b200_problem_evaluate
struct BuiltinRec {
  int id;
  const char* type;
  int d, q, P;
};
const BuiltinRec kBuiltins[] = {
    {PN_B200_LOGISTIC, "pn::Logistic", 1, 1, 2},   {PN_B200_RIGID_BODY, "pn::RigidBody", 3, 1, 3},
    {PN_B200_THREE_BODY, "pn::ThreeBody", 2, 2, 1}, {PN_B200_PLEIADES, "pn::Pleiades", 14, 2, 0},
    {PN_B200_VAN_DER_POL, "pn::VanDerPol", 1, 2, 1}, {PN_B200_LOTKA_VOLTERRA, "pn::LotkaVolterra", 2, 1, 4},
};

// a compiled module: its kernels' names, the cubin, and -- once loaded -- the library and kernel handles
struct Module {
  std::vector<std::string> lowered;
  std::vector<char> cubin;
  cudaLibrary_t lib = nullptr;
  std::vector<const void*> kernels;
};

enum : int { KIND_EVAL = 100 };  // module kinds beyond the kernel families

struct JitEntry {
  KernelEntry e;
  std::shared_ptr<Module> mod;
};

struct State {
  std::mutex mu;
  std::vector<ProblemRec> problems;
  std::deque<JitEntry> entries;  // stable addresses: pn_capi caches launch geometry per entry pointer
  std::vector<std::pair<std::string, std::shared_ptr<Module>>> modules;  // keyed by (problem, kind, nu, strategy)
};
State& st() {
  static State s;
  return s;
}

const ProblemRec* find_problem(int id) {
  for (const auto& r : st().problems)
    if (r.id == id) return &r;
  return nullptr;
}

// ---- layouts of the kernel templates for a runtime (n, d) ----------------------------------------------------------
struct Sizes {
  int bw, marg, pend, slot_fix, slot_filt;             // Layout<n, d>
  int dense_slot_fix, dense_slot_filt, dense_smooth;   // DenseLayout<n, d>
  int rows_smem_slot, rows_tables;                     // DenseRowsLayout<n, d>
  int mb_doubles, mb_ints;                             // pair::Mailbox<n, d>
};
template <int N, int D>
Sizes sizes_nd() {
  using L = Layout<N, D>;
  using DL = DenseLayout<N, D>;
  using RL = DenseRowsLayout<N, D>;
  using MB = pair::Mailbox<N, D>;
  return {L::BW, L::MARG, L::PEND, L::SLOT_FIX, L::SLOT_FILT, DL::SLOT_FIX, DL::SLOT_FILT, DL::SMEM_SMOOTH,
          RL::SMEM_SLOT, RL::TABLES, MB::DOUBLES, MB::INTS};
}
template <int N, size_t... I>
Sizes sizes_row(int d, std::index_sequence<I...>) {
  static const Sizes t[] = {sizes_nd<N, (int)I + 1>()...};
  return t[d - 1];
}
Sizes sizes(int n, int d) {
  const auto ds = std::make_index_sequence<MAX_DIM>{};
  switch (n) {
    case 2: return sizes_row<2>(d, ds);
    case 3: return sizes_row<3>(d, ds);
    case 4: return sizes_row<4>(d, ds);
    case 5: return sizes_row<5>(d, ds);
    case 6: return sizes_row<6>(d, ds);
    case 7: return sizes_row<7>(d, ds);
    case 8: return sizes_row<8>(d, ds);
    default: return sizes_row<9>(d, ds);
  }
}

constexpr size_t SMEM_LIMIT_BYTES = 227 * 1024;  // dynamic shared memory per CTA on sm_100
constexpr int DENSE_SAMPLE_WARPS = 4;            // launch_dense_sample

// ---- sources --------------------------------------------------------------------------------------------------
bool valid_name(const std::string& s) {
  if (s.empty() || s.size() > 128) return false;
  for (char c : s)
    if (!((c >= 'a' && c <= 'z') || (c >= 'A' && c <= 'Z') || (c >= '0' && c <= '9') || c == '_' || c == '-' || c == '.'))
      return false;
  return true;
}

// The user's text in its own namespace, then the Prob functor the kernels are instantiated with.  A time-dependent
// problem's functions take the time after the state (pn_user_problem.cuh).
std::string problem_text(const ProblemRec& r) {
  const std::string ns = "pn_user_" + std::to_string(r.id);
  const bool time = (r.form & PN_B200_FORM_TIME_DEPENDENT) != 0;
  const int form = r.form & ~PN_B200_FORM_TIME_DEPENDENT;
  std::string s = "namespace " + ns + " {\nusing namespace ::pn::jet;\n";
  if (form == PN_B200_FORM_SIMPLE) {
    // a Jacobian the user does not define resolves to this declaration (never defined: only its type is used)
    s += "struct pn_no_jac {};\ntemplate <class... A> pn_no_jac jac(A...);\n";
  }
  s += "#line 1 \"" + r.name + "\"\n" + r.source + "\n#line 1 \"" + r.name + " (adapter)\"\n}\nnamespace " + ns + " {\n";
  const std::string dims = std::to_string(r.d) + ", " + std::to_string(r.q) + ", " + std::to_string(r.P);
  if (form == PN_B200_FORM_SIMPLE && !time) {
    s += "struct PnSource {\n"
         "  template <class T> PN_DEV static void vf(const T* u, const double* p, T* f) { ::" + ns + "::vf<T>(u, p, f); }\n"
         "  template <int Z = 0> PN_DEV static void jac(const double* u, const double* p, double* J) { ::" + ns + "::jac(u, p, J); }\n"
         "};\n"
         "constexpr bool PN_HAS_JAC = !::pn::jet::IsSame<decltype(::" + ns + "::jac((const double*)0, (const double*)0, (double*)0)), pn_no_jac>::value;\n"
         "using Prob = ::pn::UserProblem<PnSource, " + dims + ", PN_HAS_JAC>;\n";
  } else if (form == PN_B200_FORM_SIMPLE) {
    s += "struct PnSource {\n"
         "  template <class T> PN_DEV static void vf(const T* u, const T& t, const double* p, T* f) { ::" + ns + "::vf<T>(u, t, p, f); }\n"
         "  template <int Z = 0> PN_DEV static void jac(const double* u, double t, const double* p, double* J) { ::" + ns + "::jac(u, t, p, J); }\n"
         "};\n"
         "constexpr bool PN_HAS_JAC = !::pn::jet::IsSame<decltype(::" + ns + "::jac((const double*)0, 0.0, (const double*)0, (double*)0)), pn_no_jac>::value;\n"
         "using Prob = ::pn::UserProblem<PnSource, " + dims + ", PN_HAS_JAC, true>;\n";
  } else {
    s += "static_assert(Problem::D == " + std::to_string(r.d) + ", \"Problem::D differs from the registered d\");\n"
         "static_assert(Problem::Q == " + std::to_string(r.q) + ", \"Problem::Q differs from the registered ode_order\");\n"
         "static_assert(Problem::P == " + std::to_string(r.P) + ", \"Problem::P differs from the registered num_params\");\n"
         "static_assert(::pn::TimeDependent<Problem>::value == " + (time ? "true" : "false") +
         ", \"Problem::TIME differs from the registered time dependence\");\n"
         "using Prob = ::pn::FullProblem<Problem>;\n";
  }
  s += "}\n";
  return s;
}

// NVRTC: compile `text` (after the headers it includes) and lower the name expressions
int compile(const std::string& what, const std::string& text, const std::vector<std::string>& names, Module* m) {
  std::vector<const char*> hdr_src, hdr_name;
  for (const auto& h : kJitSources) {
    hdr_name.push_back(h.name);
    hdr_src.push_back(h.text);
  }
  nvrtcProgram prog;
  nvrtcResult r = nvrtcCreateProgram(&prog, text.c_str(), "pn_jit_module.cu", (int)hdr_src.size(), hdr_src.data(), hdr_name.data());
  if (r != NVRTC_SUCCESS) return fail(PN_B200_ERR_CUDA, std::string("nvrtcCreateProgram: ") + nvrtcGetErrorString(r));
  for (const auto& n : names) nvrtcAddNameExpression(prog, n.c_str());
  r = nvrtcCompileProgram(prog, (int)(sizeof kNvrtcOptions / sizeof kNvrtcOptions[0]), kNvrtcOptions);
  if (r != NVRTC_SUCCESS) {
    size_t n = 0;
    nvrtcGetProgramLogSize(prog, &n);
    std::string log(n, '\0');
    if (n) nvrtcGetProgramLog(prog, &log[0]);
    while (!log.empty() && log.back() == '\0') log.pop_back();
    nvrtcDestroyProgram(&prog);
    return fail(PN_B200_ERR_ARGUMENT, "compiling " + what + " failed:\n" + log);
  }
  m->lowered.clear();
  for (const auto& n : names) {
    const char* low = nullptr;
    nvrtcGetLoweredName(prog, n.c_str(), &low);
    m->lowered.push_back(low ? low : "");
  }
  size_t cs = 0;
  nvrtcGetCUBINSize(prog, &cs);
  m->cubin.resize(cs);
  r = nvrtcGetCUBIN(prog, m->cubin.data());
  nvrtcDestroyProgram(&prog);
  if (r != NVRTC_SUCCESS) return fail(PN_B200_ERR_CUDA, std::string("nvrtcGetCUBIN: ") + nvrtcGetErrorString(r));
  return PN_B200_SUCCESS;
}

int load(Module* m) {
  if (m->lib) return PN_B200_SUCCESS;
  cudaLibrary_t lib = nullptr;
  cudaError_t ce = cudaLibraryLoadData(&lib, m->cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, std::string("cudaLibraryLoadData: ") + cudaGetErrorString(ce));
  std::vector<const void*> ks;
  for (const auto& n : m->lowered) {
    cudaKernel_t k = nullptr;
    ce = cudaLibraryGetKernel(&k, lib, n.c_str());
    if (ce != cudaSuccess) {
      cudaLibraryUnload(lib);
      return fail(PN_B200_ERR_CUDA, "cudaLibraryGetKernel(" + n + "): " + cudaGetErrorString(ce));
    }
    ks.push_back((const void*)k);
  }
  m->kernels = ks;
  m->lib = lib;
  return PN_B200_SUCCESS;
}

// the type name of a problem's functor inside a module, and the module's text up to the name expressions
std::string prob_type(int problem) {
  if (problem >= PN_B200_USER_PROBLEM_BASE) return "pn_user_" + std::to_string(problem) + "::Prob";
  for (const auto& b : kBuiltins)
    if (b.id == problem) return b.type;
  return "";
}
std::string module_text(int problem, bool solve_kernels) {
  std::string s = "#include \"pn_user_problem.cuh\"\n";
  if (solve_kernels) s += "#include \"pn_dense_rows_kernel.cuh\"\n#include \"pn_sample_kernel.cuh\"\n#include \"pn_lml_kernel.cuh\"\n";
  if (problem >= PN_B200_USER_PROBLEM_BASE) s += problem_text(*find_problem(problem));
  return s;
}
std::string problem_label(int problem) {
  const ProblemRec* r = find_problem(problem);
  return r ? "problem '" + r->name + "'" : "built-in problem " + std::to_string(problem);
}

// the module of (problem, kind, nu, strategy), compiled on first use; `names` are its name expressions
int get_module(int problem, int kind, int nu, int strategy, const std::vector<std::string>& names, std::shared_ptr<Module>* out) {
  const std::string key = std::to_string(problem) + "/" + std::to_string(kind) + "/" + std::to_string(nu) + "/" + std::to_string(strategy);
  for (auto& km : st().modules)
    if (km.first == key) {
      *out = km.second;
      return PN_B200_SUCCESS;
    }
  auto m = std::make_shared<Module>();
  int rc = compile(problem_label(problem), module_text(problem, kind != KIND_EVAL), names, m.get());
  if (rc) return rc;
  st().modules.push_back({key, m});
  *out = m;
  return PN_B200_SUCCESS;
}

// module kernels of a JIT entry, in this order: solve, sliced solve, smoothing, sampling, likelihood sweep
std::vector<std::string> entry_names(const KernelEntry& e) {
  const std::string P = prob_type(e.problem), nu = std::to_string(e.nu), S = std::to_string(e.strategy);
  const std::string n = std::to_string(e.N), T = std::to_string(e.threads);
  std::vector<std::string> v(5);
  if (e.family == FAMILY_DENSE_ROWS) {
    const std::string W = std::to_string(e.threads / 32);
    v[0] = "pn::pn_dense_rows_kernel<" + P + ", " + nu + ", " + S + ", " + std::to_string(e.group) + ", " + W + ">";
    v[2] = "pn::pn_dense_smooth_kernel<" + n + ", " + std::to_string(e.D) + ", " + S + ", " + W + ">";
    return v;
  }
  const std::string dl = std::to_string(e.group > 1 ? 1 : e.D);
  if (e.family == FAMILY_PAIR) {
    v[0] = "pn::pn_scalar_kernel<" + P + ", " + nu + ", 1, 1, 0, " + T + ", 0, 0, 0, 1>";
  } else {
    const std::string bd = (e.family == FAMILY_GROUP_BDIAG) ? "1" : "0";
    v[0] = "pn::pn_scalar_kernel<" + P + ", " + nu + ", " + S + ", " + std::to_string(e.group) + ", " + bd + ", " + T + ">";
    if (e.ctx_doubles > 0) v[1] = "pn::pn_scalar_kernel<" + P + ", " + nu + ", " + S + ", 1, 0, " + T + ", 0, 1>";
  }
  v[2] = "pn::pn_smooth_kernel<" + n + ", " + dl + ", " + S + ">";
  if (e.strategy == 1) {
    v[3] = "pn::pn_sample_kernel<" + n + ", " + dl + ">";
    v[4] = "pn::pn_lml_sweep_kernel<" + n + ", " + dl + ">";
  }
  return v;
}

// metadata of the build of `family` for a user problem, as the *Instance templates of pn_registry.h set it
bool make_entry(const ProblemRec& r, int family, int nu, int strategy, KernelEntry* out) {
  const int n = nu + 1, d = r.d;
  KernelEntry e;
  e.family = family;
  e.problem = r.id;
  e.nu = nu;
  e.strategy = strategy;
  e.N = n;
  e.D = d;
  e.Q = r.q;
  e.P = r.P;
  e.has_jac = true;
  e.jit = true;
  e.solve_func = nullptr;
  e.launch_solve = nullptr;
  e.launch_smooth = nullptr;
  const bool fix = strategy == PN_B200_FIXEDPOINT;
  if (family == FAMILY_DENSE_ROWS) {
    if (d < 2 || n * d > 32) return false;
    const Sizes z = sizes(n, d);
    const int lanes = (n * d <= 16) ? 16 : 32, warps = (lanes == 16) ? 2 : 1;
    e.group = lanes;
    e.dv = 1;
    e.threads = 32 * warps;
    e.slot_doubles = fix ? z.dense_slot_fix : z.dense_slot_filt;
    e.smem_doubles = (32 / lanes) * z.rows_smem_slot + (z.rows_tables + warps - 1) / warps;
    if ((size_t)e.smem_doubles * warps * sizeof(double) > SMEM_LIMIT_BYTES) return false;
    if (fix) e.sample_func = (const void*)&pn_dense_sample_kernel<DENSE_SAMPLE_WARPS>;
    *out = e;
    return true;
  }
  int group = 1;
  if (family == FAMILY_GROUP_ISO || family == FAMILY_GROUP_BDIAG) {
    if (d < 2) return false;
    while (group < d) group *= 2;
  } else if (family == FAMILY_SCALAR || family == FAMILY_PAIR) {
    if (d > 3) return false;  // the widest thread-per-IVP built-in; beyond it the lane-per-dimension kernels
    if (family == FAMILY_PAIR && (!fix || d > 2)) return false;  // a d = 3 mailbox does not fit beside 128 members
  } else {
    return false;
  }
  const int dl = (group > 1) ? 1 : d;
  const Sizes z = sizes(n, dl);
  e.group = group;
  e.dv = (group > 1) ? d : 1;
  e.slot_doubles = fix ? z.slot_fix : z.slot_filt;
  e.smem_doubles = (fix ? z.bw : 0) + z.pend + z.marg;
  // 128 threads per CTA while two CTAs' state fits an SM, else 64 (the built-ins' nu = 8 instances)
  e.threads = ((size_t)e.smem_doubles * 128 * sizeof(double) > SMEM_LIMIT_BYTES / 2) ? 64 : 128;
  if (family == FAMILY_PAIR) {
    e.threads = 128;
    e.extra_threads = 128;
    e.smem_doubles += z.mb_doubles + (z.mb_ints + 1) / 2;
    if ((size_t)e.smem_doubles * e.threads * sizeof(double) > SMEM_LIMIT_BYTES) return false;
  }
  if (family == FAMILY_SCALAR && fix) e.ctx_doubles = slice_ctx_doubles(z.bw, z.marg);
  *out = e;
  return true;
}

}  // namespace

bool jit_is_user_problem(int problem) { return problem >= PN_B200_USER_PROBLEM_BASE; }

const KernelEntry* jit_find(int family, int problem, int nu, int strategy, int d) {
  std::lock_guard<std::mutex> lock(st().mu);
  const ProblemRec* r = find_problem(problem);
  if (!r || r->d != d) return nullptr;
  for (const auto& je : st().entries)
    if (je.e.family == family && je.e.problem == problem && je.e.nu == nu && je.e.strategy == strategy) return &je.e;
  KernelEntry e;
  if (!make_entry(*r, family, nu, strategy, &e)) return nullptr;
  st().entries.push_back({e, nullptr});
  return &st().entries.back().e;
}

int jit_load(const KernelEntry* ke) {
  std::lock_guard<std::mutex> lock(st().mu);
  JitEntry* je = nullptr;
  for (auto& x : st().entries)
    if (&x.e == ke) je = &x;
  if (!je) return fail(PN_B200_ERR_ARGUMENT, "not a run-time compiled kernel");
  if (je->e.solve_func) return PN_B200_SUCCESS;
  std::vector<std::string> names = entry_names(je->e), used;
  for (const auto& n : names)
    if (!n.empty()) used.push_back(n);
  std::shared_ptr<Module> m;
  int rc = get_module(je->e.problem, je->e.family, je->e.nu, je->e.strategy, used, &m);
  if (rc == PN_B200_SUCCESS) rc = load(m.get());
  if (rc) return rc;
  const void* k[5] = {};
  for (size_t i = 0, j = 0; i < names.size(); ++i)
    if (!names[i].empty()) k[i] = m->kernels[j++];
  je->mod = m;
  je->e.solve_func_sliced = k[1];
  je->e.smooth_func = k[2];
  if (k[3]) je->e.sample_func = k[3];
  je->e.lml_func = k[4];
  je->e.solve_func = k[0];  // last: a set solve_func marks the entry as loaded
  return PN_B200_SUCCESS;
}

static cudaError_t launch(const void* f, unsigned grid, unsigned threads, size_t smem, cudaStream_t s, const void* args) {
  void* argv[] = {const_cast<void*>(args)};
  return cudaLaunchKernel(f, dim3(grid), dim3(threads), argv, smem, s);
}

cudaError_t jit_launch_solve(const KernelEntry* e, bool sliced, const SolveArgs& a, int grid, size_t smem, cudaStream_t s) {
  return launch(sliced ? e->solve_func_sliced : e->solve_func, (unsigned)grid, (unsigned)(e->threads + e->extra_threads), smem, s, &a);
}

cudaError_t jit_launch_smooth(const KernelEntry* e, const SmoothArgs& a, cudaStream_t s) {
  if (e->family == FAMILY_DENSE_ROWS) {
    const int warps = e->threads / 32;
    const size_t smem = (size_t)warps * sizes(e->N, e->D).dense_smooth * sizeof(double);
    cudaError_t ce = cudaFuncSetAttribute(e->smooth_func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return ce;
    return launch(e->smooth_func, (unsigned)((a.B + warps - 1) / warps), (unsigned)e->threads, smem, s, &a);
  }
  return launch(e->smooth_func, (unsigned)((a.B * a.dv + 127) / 128), 128, 0, s, &a);
}

cudaError_t jit_launch_sample(const KernelEntry* e, const SampleArgs& a, cudaStream_t s) {
  if (e->family == FAMILY_DENSE_ROWS) return launch_dense_sample(a, e->N * e->D, 0, s);
  const long long total = a.B * a.dv * a.S;
  return launch(e->sample_func, (unsigned)((total + 127) / 128), 128, 0, s, &a);
}

cudaError_t jit_launch_lml(const KernelEntry* e, const LmlArgs& a, cudaStream_t s) {
  cudaError_t ce = launch(e->lml_func, (unsigned)((a.B * a.dv + 127) / 128), 128, 0, s, &a);
  if (ce != cudaSuccess) return ce;
  pn_lml_reduce_kernel<0><<<(unsigned)((a.B + 127) / 128), 128, 0, s>>>(a);
  return cudaGetLastError();
}

}  // namespace pn

using namespace pn;

extern "C" {

int pn_b200_register_problem(const char* name, const char* source, int form, int32_t d, int32_t ode_order,
                             int32_t num_params, int32_t* problem_id) {
  if (!name || !source || !problem_id) return fail(PN_B200_ERR_ARGUMENT, "null name, source or problem_id");
  if (!valid_name(name)) return fail(PN_B200_ERR_ARGUMENT, "problem name: 1 to 128 characters of [A-Za-z0-9_.-]");
  const int base_form = form & ~PN_B200_FORM_TIME_DEPENDENT;
  if (base_form != PN_B200_FORM_SIMPLE && base_form != PN_B200_FORM_FULL) return fail(PN_B200_ERR_ARGUMENT, "unknown source form");
  if (d < 1 || d > MAX_DIM) return fail(PN_B200_ERR_ARGUMENT, "d must be in 1 .. 32");
  if (ode_order != 1 && ode_order != 2) return fail(PN_B200_ERR_ARGUMENT, "ode_order must be 1 or 2");
  if (num_params < 0 || num_params > MAX_PARAMS) return fail(PN_B200_ERR_ARGUMENT, "num_params must be in 0 .. 64");
  std::lock_guard<std::mutex> lock(st().mu);
  for (const auto& r : st().problems)
    if (r.name == name && r.source == source && r.form == form && r.d == d && r.q == ode_order && r.P == num_params) {
      *problem_id = r.id;
      return PN_B200_SUCCESS;
    }
  ProblemRec r{PN_B200_USER_PROBLEM_BASE + (int)st().problems.size(), name, source, form, d, ode_order, num_params};
  st().problems.push_back(r);
  // the evaluation kernel at nu = 1 is the check: it instantiates vf on doubles and on jets, and the Jacobian
  std::shared_ptr<Module> m;
  const std::string ev = "pn::pn_problem_eval_kernel<" + prob_type(r.id) + ", 1>";
  int rc = get_module(r.id, KIND_EVAL, 1, 0, {ev}, &m);
  if (rc) {
    st().problems.pop_back();
    return rc;
  }
  *problem_id = r.id;
  return PN_B200_SUCCESS;
}

int pn_b200_problem_evaluate(int32_t problem, int32_t nu, int64_t n, const double* u0, const double* params, double* f,
                             double* taylor, double* jac, void* cuda_stream) {
  return pn_b200_problem_evaluate_at(problem, nu, n, nullptr, u0, params, f, taylor, jac, cuda_stream);
}

int pn_b200_problem_evaluate_at(int32_t problem, int32_t nu, int64_t n, const double* t, const double* u0, const double* params,
                                double* f, double* taylor, double* jac, void* cuda_stream) {
  if (nu < 1 || nu > 8) return fail(PN_B200_ERR_ARGUMENT, "nu must be in 1 .. 8");
  if (n < 0) return fail(PN_B200_ERR_ARGUMENT, "n must be >= 0");
  int P = 0;
  bool has_jac = true;
  std::shared_ptr<Module> m;
  {
    std::lock_guard<std::mutex> lock(st().mu);
    if (const ProblemRec* r = find_problem(problem)) {
      P = r->P;
    } else {
      const BuiltinRec* b = nullptr;
      for (const auto& x : kBuiltins)
        if (x.id == problem) b = &x;
      if (!b) return fail(PN_B200_ERR_ARGUMENT, "unknown problem id (or a built-in problem without a fixed size)");
      P = b->P;
      has_jac = problem != PN_B200_PLEIADES;
    }
    if (jac && !has_jac) return fail(PN_B200_ERR_UNSUPPORTED, "problem has no Jacobian");
    const std::string ev = "pn::pn_problem_eval_kernel<" + prob_type(problem) + ", " + std::to_string(nu) + ">";
    int rc = get_module(problem, KIND_EVAL, nu, 0, {ev}, &m);
    if (rc == PN_B200_SUCCESS) rc = load(m.get());
    if (rc) return rc;
  }
  if (n == 0) return PN_B200_SUCCESS;
  if (!u0 || (P > 0 && !params)) return fail(PN_B200_ERR_ARGUMENT, "null u0 or params");
  long long nn = n;
  int np = P;
  void* args[] = {&nn, &np, &t, &u0, &params, &f, &taylor, &jac};
  cudaError_t ce = cudaLaunchKernel(m->kernels[0], dim3((unsigned)((n + 127) / 128)), dim3(128), args, 0, (cudaStream_t)cuda_stream);
  if (ce != cudaSuccess) return fail(PN_B200_ERR_CUDA, std::string("evaluation kernel launch: ") + cudaGetErrorString(ce));
  return PN_B200_SUCCESS;
}

// Test hook (not part of the public header): how many modules NVRTC has compiled in this process.
int pn_b200_jit_module_count(void) {
  std::lock_guard<std::mutex> lock(st().mu);
  return (int)st().modules.size();
}

// Test hook (not part of the public header): the embedded text of header `name`, NULL if it is not embedded.
const char* pn_b200_jit_source(const char* name) {
  for (const auto& h : kJitSources)
    if (name && strcmp(h.name, name) == 0) return h.text;
  return nullptr;
}

}  // extern "C"
