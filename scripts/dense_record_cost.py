"""Cost of trajectory recording (PN_B200_FLAG_RECORD) on the two dense filter kernels: the same filter solve with
and without recording, alternating, timed with CUDA events around the solve kernel (pn_b200_set_profiling).

  * rigid body, dense EKF1, nu = 4, 16,384 members (register-column kernel, two IVPs per warp)
  * Brusselator N = 16, dense EKF1, nu = 4, one IVP (CTA-per-IVP dense kernel, D = 160)

Both runs use save_at = [t0, t1], the shape solve_adaptive_save_every_step launches.  The outputs at the checkpoints
are checked to be bit-identical with and without recording.

    python scripts/dense_record_cost.py [repeats = 7]        # on a B200
"""

import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "code-adaptive-prob-ode-solvers_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from odecheckpts_b200 import _cabi  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 7
dev = torch.device("cuda:0")


def desc_for(problem, d, B, tol, record, cap):
    return _cabi.Desc(_cabi.PROBLEM_IDS[problem], d, 4, 1, _cabi.FACTORISATIONS["dense"], _cabi.CORRECTIONS["ts1"],
                      _cabi.STRATEGIES["filter"], _cabi.CALIBRATIONS["dynamic"], tol, tol, 0.01, 0.95, 0.2, 10.0, 0.3, 0.4,
                      B, 2, 0, 1 if problem == "brusselator" else 3, _cabi.FLAG_RECORD if record else 0, cap if record else 0)  # fmt: skip


def case_rigid_body():
    B = 16384
    rng = np.random.default_rng(0)
    u0 = (np.array([1.0, 0.0, 0.9]) + 0.1 * rng.uniform(-1, 1, (B, 3))).reshape(B, 1, 3)
    params = np.tile([-2.0, 1.25, -0.5], (B, 1))
    return "rigid body dense EKF1, 16384 members, t in [0, 20], tol 1e-8", "rigid_body", 3, B, 1e-8, u0, params, 20.0, 4096


def case_brusselator():
    N = 16
    x0 = np.linspace(0, 1, N)
    u0 = np.concatenate([np.sin(2 * np.pi * x0) + 1, 3.0 * np.ones(N)])[None, None]
    return "Brusselator N = 16 dense EKF1, one IVP, t in [0, 10], tol 1e-8", "brusselator", 2 * N, 1, 1e-8, u0, np.array([[0.02]]), 10.0, 1 << 16


def run(case):
    label, problem, d, B, tol, u0, params, t1, cap = case
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device=dev)  # noqa: E731
    u0, params, save_at = t(u0), t(params), t([0.0, t1])
    descs = {rec: desc_for(problem, d, B, tol, rec, cap) for rec in (False, True)}
    ws = torch.empty((max(_cabi.workspace_bytes(x) for x in descs.values()) + 7) // 8, dtype=torch.int64, device=dev)
    times, outs = {False: [], True: []}, {}
    _cabi.set_profiling(True)
    for i in range(reps + 1):  # the first pair warms up
        for rec in (False, True) if i % 2 == 0 else (True, False):
            out = _cabi.solve_device(descs[rec], u0, params, None, save_at, None, workspace=ws)
            solve_ms, _ = _cabi.last_timing()
            if i > 0:
                times[rec].append(solve_ms)
            outs[rec] = {k: v.cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    _cabi.set_profiling(False)
    for key in ("u", "u_std", "n_accepted", "n_rejected", "status"):
        assert np.array_equal(outs[False][key], outs[True][key]), f"{label}: {key} changes with recording"
    assert (outs[True]["traj_len"] < cap).all() and (outs[True]["status"] == 0).all()
    steps = int(outs[True]["n_accepted"][:, -1].sum())
    off, on = np.median(times[False]), np.median(times[True])
    print(f"{label}: {steps} accepted steps in all; solve kernel median of {reps}: without recording {off:9.3f} ms "
          f"(min {min(times[False]):.3f}), with recording {on:9.3f} ms (min {min(times[True]):.3f}), "
          f"{100.0 * (on / off - 1.0):+.1f} %", flush=True)  # fmt: skip


name = torch.cuda.get_device_name(dev)
query = ["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(dev.index or 0)]
power = subprocess.run(query, capture_output=True, text=True).stdout.strip() or "unknown"
print(f"# {name}, power limit {power}; filter strategy, save_at = [t0, t1], alternating runs", flush=True)
run(case_rigid_body())
run(case_brusselator())
