"""Cost of per-member time grids (PN_B200_FLAG_MEMBER_GRIDS) on the headline shape: 65,536 Van der Pol members
(bench.py's seeded ensemble, mu = 1e3), dense EKF1, nu = 4, fixed-point smoother, atol = rtol = 1e-6, 50 checkpoints.
Three variants, alternating, timed with CUDA events around the solve kernel (pn_b200_set_profiling):

  * shared   the shared grid [K] = linspace(0, 6.3, 50)
  * rows     a [B, K] grid whose rows all equal it (the flag's address arithmetic, the same arithmetic per member)
  * members  genuinely per-member grids: member b runs on [t0_b, t0_b + 6.3] with its own uneven checkpoints

"shared" and "rows" are checked to be bit-identical.  "members" solves different IVPs, so its time differs by what the
members' own horizons cost, not by the flag.

    python scripts/member_grids_cost.py [rounds = 7]        # on a B200
"""

import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "code-adaptive-prob-ode-solvers_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from odecheckpts_b200 import _cabi  # noqa: E402

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 7
dev = torch.device("cuda:0")
B, K, T1 = 65536, 50, 6.3

u0, params = bench.ensemble_inputs(0, B)
desc = _cabi.Desc(_cabi.PROBLEM_IDS["van_der_pol"], 1, 4, 2, _cabi.FACTORISATIONS["dense"], _cabi.CORRECTIONS["ts1"],
                  _cabi.STRATEGIES["fixedpoint"], _cabi.CALIBRATIONS["dynamic"], 1e-6, 1e-6, 0.01, 0.95, 0.2, 10.0, 0.3, 0.4,
                  B, K, 0, 1, 0, 0)  # fmt: skip
shared = np.linspace(0.0, T1, K)
rng = np.random.default_rng(1)
t0 = rng.uniform(0.0, 0.5, B)
inner = np.sort(rng.uniform(0.0, T1, (B, K - 2)), axis=1)
members = np.concatenate([t0[:, None], t0[:, None] + inner, (t0 + T1)[:, None]], axis=1)
assert np.all(np.diff(members, axis=1) > 0)
t = lambda x: torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device=dev)  # noqa: E731
grids = {"shared": t(shared), "rows": t(np.tile(shared, (B, 1))), "members": t(members)}
u0_d, par_d = t(u0), t(params)
ws = torch.empty((_cabi.workspace_bytes(desc) + 7) // 8, dtype=torch.int64, device=dev)

name = torch.cuda.get_device_name(dev)
query = ["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(dev.index or 0)]
power = subprocess.run(query, capture_output=True, text=True).stdout.strip() or "unknown"
print(f"# {name}, power limit {power}; {B} VdP members, dense EKF1 nu=4 fixed-point, K={K}, {rounds} alternating rounds",
      flush=True)  # fmt: skip
info = _cabi.kernel_info(desc)
print(f"# solve kernel: {info['registers_per_thread']} registers, {info['local_bytes_per_thread']} B local per thread, "
      f"grid {info['grid']} x {info['threads_per_cta']}", flush=True)  # fmt: skip

times, outs = {k: [] for k in grids}, {}
order = list(grids)
_cabi.set_profiling(True)
for r in range(rounds + 1):  # round 0 warms up
    for key in order if r % 2 == 0 else order[::-1]:
        out = _cabi.solve_device(desc, u0_d, par_d, None, grids[key], None, workspace=ws)
        solve_ms, _ = _cabi.last_timing()
        if r > 0:
            times[key].append(solve_ms)
        if r == rounds:
            outs[key] = {k: v.cpu().numpy() for k, v in out.items() if not k.startswith("_")}
_cabi.set_profiling(False)
for k in outs["shared"]:
    assert np.array_equal(outs["shared"][k], outs["rows"][k], equal_nan=True), f"rows equal to the shared grid: {k} differs"
for key in grids:
    x = np.asarray(times[key])
    steps = int(outs[key]["n_accepted"][:, -1].sum())
    assert (outs[key]["status"] == 0).all()
    print(f"{key:8s} solve kernel median {np.median(x):8.2f} ms  min {x.min():8.2f}  max {x.max():8.2f}  "
          f"({steps} accepted steps in all)", flush=True)  # fmt: skip
m = {k: np.median(v) for k, v in times.items()}
print(f"rows / shared: {100.0 * (m['rows'] / m['shared'] - 1.0):+.2f} % (outputs bit-identical)", flush=True)
