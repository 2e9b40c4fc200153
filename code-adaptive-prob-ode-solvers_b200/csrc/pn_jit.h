// pn_jit.h -- run-time compiled kernels of user-defined problems (pn_jit.cu), as seen by the C ABI (pn_capi.cu).
#pragma once
#include <string>

#include "pn_registry.h"

namespace pn {

int fail(int code, const std::string& msg);  // sets pn_b200_last_error, returns code

bool jit_is_user_problem(int problem);
// The entry of a user problem's build of `family` (metadata only: nothing is compiled), nullptr if the problem has no
// such build.  Entries live as long as the process.
const KernelEntry* jit_find(int family, int problem, int nu, int strategy, int d);
// Compiles (once per process) and loads the module behind a JIT entry: afterwards its *_func handles are set.
int jit_load(const KernelEntry* e);

cudaError_t jit_launch_solve(const KernelEntry* e, bool sliced, const SolveArgs& a, int grid, size_t smem, cudaStream_t s);
cudaError_t jit_launch_smooth(const KernelEntry* e, const SmoothArgs& a, cudaStream_t s);
cudaError_t jit_launch_sample(const KernelEntry* e, const SampleArgs& a, cudaStream_t s);
cudaError_t jit_launch_lml(const KernelEntry* e, const LmlArgs& a, cudaStream_t s);

}  // namespace pn
