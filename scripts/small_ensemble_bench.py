"""Small ensembles of the headline workload (VdP mu = 1e3, dense EKF1 + fixed-point, nu = 4, tol 1e-6, 50 checkpoints):
ms per pass with and without the PAIR build (PN_B200_PAIR=0).

    python scripts/small_ensemble_bench.py [members ...]      # on a B200
"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "code-adaptive-prob-ode-solvers_b200")); sys.path.insert(0, ROOT)
import numpy as np, torch
from odecheckpts_b200 import _cabi

K = 50
dev = torch.device("cuda:0")
sizes = [int(x) for x in sys.argv[1:]] or [1, 2048, 4736, 8192, 16384, 18944, 24576, 32768, 37888]
ref = {}
for B in sizes:
    rng = np.random.default_rng(0)
    u0 = np.stack([2.0 + 0.5 * rng.uniform(-1, 1, B), 0.5 * rng.uniform(-1, 1, B)], 1).reshape(B, 2, 1)
    desc = _cabi.Desc(5, 1, 4, 2, 2, 1, 1, 1, 1e-6, 1e-6, 0.01, 0.95, 0.2, 10.0, 0.3, 0.4, B, K, 0, 1, 0, 0)
    u0_d = torch.as_tensor(u0, device=dev); par = torch.full((B, 1), 1e3, dtype=torch.float64, device=dev)
    save = torch.linspace(0, 6.3, K, dtype=torch.float64, device=dev)
    for label, env in (("PAIR", {}), ("no PAIR", {"PN_B200_PAIR": "0"})):
        os.environ.pop("PN_B200_PAIR", None)
        os.environ.update(env)
        info = _cabi.kernel_info(desc)
        best, out = 1e30, None
        for it in range(3):
            torch.cuda.synchronize(); e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(); out = _cabi.solve_device(desc, u0_d, par, None, save, None, workspace=None if out is None else out["_workspace"]); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        sig = (out["u"].double().sum().item(), int(out["n_accepted"][:, -1].sum()), int(out["n_rejected"].sum()))
        same = ref.setdefault(B, sig) == sig
        print(f"members {B:6d}  {label:16s} {best:8.2f} ms   threads/CTA {info['threads_per_cta']}  grid {info.get('grid')}  identical {same}", flush=True)
