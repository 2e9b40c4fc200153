// Dense-factorisation instance with d > 1 (warp per IVP, D x D factors in shared memory) for the one problem
// too wide for the register-column kernel (pn_inst_dense_rows.cu: D <= 32) and too narrow for the CTA-per-IVP
// kernel (pn_inst_dense_cta.cu: D > 40): the Brusselator with N = 4 (BASELINE config 5's dense sqrt-EKF1
// factorisation; D = 5 * 2N = 40).
#include "pn_registry.h"
namespace pn {
using Brusselator4d = Brusselator<4>;
}  // namespace pn
PN_REGISTER_DENSE(Brusselator4d, 4, 1, 1);
