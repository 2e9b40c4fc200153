"""experiments/4_brusselator/run.py through the builder API on the GPU: for every grid size N the baseline step
count (solve_adaptive_terminal_values, run.py:82-90), the TEXTBOOK smoother (strategy_smoother +
solve_adaptive_save_every_step, run.py:98-117: one backward conditional per accepted step, while that fits the
reference's 4000 MB budget) and the CHECKPOINT solver (strategy_fixedpoint + solve_adaptive_save_at with 200
checkpoints, run.py:119-138) -- the paper's memory / run-time comparison (Fig. 4).

    python scripts/brusselator_run.py [max N = 128]        # on a B200
    python scripts/brusselator_run.py --dense [max N = 32]

--dense runs the same comparison with the dense EKF1 factorisation (BASELINE config 5's model; correction_ts1,
per-dimension std): the textbook route then records on the CTA-per-IVP dense kernel and keeps one dense D x D
conditional per accepted step, so it is skipped when those exceed the same 4000 MB.  The dense runs have no
golden step counts (the reference's run.py is isotropic); instead the textbook smoother's values at the 200
checkpoints are compared with the checkpoint solver's.
"""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "code-adaptive-prob-ode-solvers_b200"))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import ctypes  # noqa: E402

from odecheckpts_b200 import _cabi, ivps  # noqa: E402
from odecheckpts_b200.probdiffeq import impl, ivpsolve, stats, taylor  # noqa: E402
from odecheckpts_b200.probdiffeq import ivpsolvers as pdi  # noqa: E402

g = np.load(os.path.join(ROOT, "tests", "golden", "reference_goldens.npz"))
args = [a for a in sys.argv[1:] if not a.startswith("--")]
dense = "--dense" in sys.argv[1:]
max_n = int(args[0]) if args else (32 if dense else 128)
num, tol = 4, 1e-8
fact = "dense" if dense else "isotropic"


def workspace_mb(N, K, strategy):
    """Device workspace of one solve with K checkpoints (the backward conditionals dominate it)."""
    desc = _cabi.Desc(4, 2 * N, num, 1, _cabi.FACTORISATIONS[fact], 1 if dense else 0, strategy, 1, tol, tol, 0.01, 0.95, 0.2,
                      10.0, 0.3, 0.4, 1, K, 0, 1, 0, 0)  # fmt: skip
    fn = _cabi.lib().pn_b200_workspace_bytes
    fn.restype = ctypes.c_size_t
    return fn(ctypes.byref(desc)) / 1024**2


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t


if dense:
    dev = torch.cuda.current_device()
    power = os.popen("nvidia-smi --query-gpu=power.limit --format=csv,noheader -i %d" % dev).read().strip() or "unknown"
    print(f"# dense EKF1 (correction_ts1), nu = {num}, atol = rtol = {tol}; {torch.cuda.get_device_name(dev)}, power limit {power}",
          flush=True)  # fmt: skip
for idx, N in enumerate(g["brusselator_N"]):
    N = int(N)
    if N > max_n:
        break
    vf, u0, (t0, t1), params = ivps.brusselator(N=N)
    impl.impl.select(fact, ode_shape=(2 * N,))
    ctrl = ivpsolve.control_proportional_integral()
    ibm = pdi.prior_ibm(num_derivatives=num)
    ts0 = pdi.correction_ts1(ode_order=1) if dense else pdi.correction_ts0(ode_order=1)
    f = lambda *y, t=None: vf(*y, t=t, p=params)  # noqa: E731
    tcoeffs = taylor.odejet_unroll(lambda *y: vf(*y, t=t0, p=params), u0, num=num)
    solver = pdi.solver_dynamic(pdi.strategy_fixedpoint(ibm, ts0))
    init = solver.initial_condition(tcoeffs, 1.0)
    asolver = ivpsolve.adaptive(solver, atol=tol, rtol=tol, control=ctrl)
    # the reference's memory model: three copies of the state per accepted step (run.py:70-77)
    n = num + 1
    size_init = 3 * 8 * (n * 2 * N + 3 * n * n + n * 2 * N + 1)
    try:
        base, t_base = timed(lambda: ivpsolve.solve_adaptive_terminal_values(f, init, t0=t0, t1=t1, dt0=0.01, adaptive_solver=asolver))
    except NotImplementedError as e:
        print(f"N={N:4d}: no {fact} kernel ({e})", flush=True)
        continue
    steps = int(base.num_steps)
    if dense:  # the textbook route's dense conditionals on the device, one per accepted step
        mem_text = workspace_mb(N, steps + 1, 1)
        line = f"N={N:4d}: baseline {steps:8d} steps in {t_base:7.3f}s, textbook memory {mem_text:9.0f} MB; "
    else:
        mem_text = steps * size_init / 1024**2
        line = f"N={N:4d}: baseline {steps:8d} steps (golden {int(g['brusselator_num_steps_terminal'][idx]):8d}) in {t_base:7.3f}s, textbook memory {mem_text:9.0f} MB; "
    save_at = np.linspace(t0, t1, 200)
    text = None
    if mem_text < 4000:
        solver_s = pdi.solver_dynamic(pdi.strategy_smoother(ibm, ts0))
        asolver_s = ivpsolve.adaptive(solver_s, atol=tol, rtol=tol, control=ctrl)
        init_s = solver_s.initial_condition(tcoeffs, 1.0)
        text, t_text = timed(lambda: ivpsolve.solve_adaptive_save_every_step(f, init_s, t0=t0, t1=t1, dt0=0.01, adaptive_solver=asolver_s,
                                                                             max_steps=steps + 16))  # fmt: skip
        line += f"textbook smoother {t_text:7.3f}s, {workspace_mb(N, len(text.t), 1):8.1f} MB of conditionals on the device ({len(text.t)} grid points); "
        if dense:
            (u_off, _), t_off = timed(lambda: stats.offgrid_marginals_searchsorted(ts=save_at[1:-1], solution=text, solver=solver_s))
            line += f"off-grid values at the checkpoints {t_off:7.3f}s; "
    else:
        line += "textbook smoother skipped (over the reference's 4000 MB budget); "
    ck, t_ck = timed(lambda: ivpsolve.solve_adaptive_save_at(f, init, save_at=save_at, dt0=0.01, adaptive_solver=asolver, keep_conditionals=True))
    peak_ck = workspace_mb(N, 200, 1)
    line += f"checkpoint solver {t_ck:7.3f}s, {peak_ck:7.1f} MB of conditionals, "
    if dense:
        line += f"steps {'==' if int(np.max(ck.num_steps)) == steps else '!='} baseline"
        if text is not None:
            rel = np.max(np.abs(u_off - ck.u[1:-1]) / np.maximum(np.abs(ck.u[1:-1]), 1e-300))
            line += f", textbook vs checkpoint max rel diff {rel:.1e}"
    else:
        ok = int(np.max(ck.num_steps)) == int(g["brusselator_num_steps_checkpoint"][idx])
        line += f"steps {'==' if ok else '!='} golden"
    print(line, flush=True)
