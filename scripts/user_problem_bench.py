"""Run-time compiled vector fields against the built-in kernels on bench.py's headline workload.

    python scripts/user_problem_bench.py [--rounds 7] [--out FILE]

Headline workload (bench.py `vdp`): 65,536 stiff Van der Pol members (mu = 1e3), dense EKF1 + fixed-point smoother,
nu = 4, atol = rtol = 1e-6, 50 checkpoints on [0, 6.3].  Three builds of the same solve, timed in one process and
in alternating order with CUDA events around pn_b200_solve_save_at (solve + smoothing kernels, inputs and outputs
resident on the device):
  builtin  problem id 5, compiled by nvcc into the library
  full     a `struct Problem` delegating to pn::VanDerPol (form "full"), compiled by NVRTC
  simple   the formula templated on the number type (form "simple"), Taylor coefficients and Jacobian derived
Reports solves/s, registers and stack per thread of the solve kernel, whether the outputs are bit-identical to the
built-in's, and the NVRTC compile time of one module of each kernel family.

Time-dependent fields, on the same workload:
  simple-t  the simple-form formula registered time-dependent, vf(u, t, p, f) ignoring t, against `simple` (the same
            formula registered autonomous): the cost of passing the time, in registers, stack and time (alternating
            rounds)
  forced    forced Van der Pol, x'' = mu ((1 - x^2) x' - x) + A cos(w t), A = 1e3, with a forcing frequency w per
            member in [0.5, 2]: time per ensemble and attempted steps
"""

import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "code-adaptive-prob-ode-solvers_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from odecheckpts_b200 import _cabi as C  # noqa: E402

FULL = """struct Problem {
  static constexpr int D = 1, Q = 2, P = 1, ID = 0;
  static constexpr bool HAS_JAC = true;
  PN_DEV static void vf(const double* u, const double* p, double* f) { pn::VanDerPol::vf(u, p, f); }
  PN_DEV static void jac(const double* u, const double* p, double* J) { pn::VanDerPol::jac(u, p, J); }
  template <int N> PN_DEV static void vf_jet(const double* U, const double* p, double* F) { pn::VanDerPol::vf_jet<N>(U, p, F); }
};"""
SIMPLE = "template <class T> PN_DEV void vf(const T* u, const double* p, T* f) { f[0] = p[0] * fma(u[1], fma(-u[0], u[0], 1.0), -u[0]); }"
SIMPLE_T = "template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) { f[0] = p[0] * fma(u[1], fma(-u[0], u[0], 1.0), -u[0]); }"
FORCED = """template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) {
  f[0] = fma(p[0], fma(u[1], fma(-u[0], u[0], 1.0), -u[0]), p[1] * cos(p[2] * t));
}"""
LORENZ96 = """template <class T> PN_DEV void vf(const T* u, const double* p, T* f) {
  for (int i = 0; i < 8; ++i) f[i] = (u[(i + 1) % 8] - u[(i + 6) % 8]) * u[(i + 7) % 8] - u[i] + p[0];
}"""
LORENZ63 = """template <class T> PN_DEV void vf(const T* u, const double* p, T* f) {
  f[0] = p[0] * (u[1] - u[0]);
  f[1] = u[0] * (p[1] - u[2]) - u[1];
  f[2] = u[0] * u[1] - p[2] * u[2];
}"""


def headline_desc(problem, B, P=1):
    return C.Desc(problem, 1, bench.NU, 2, C.FACTORISATIONS["dense"], C.CORRECTIONS["ts1"], C.STRATEGIES["fixedpoint"],
                  C.CALIBRATIONS["dynamic"], bench.TOL, bench.TOL, 0.01, 0.95, 0.2, 10.0, 0.3, 0.4, B, bench.K_CHECKPOINTS,
                  0, P, 0, 0)  # fmt: skip


def desc_for(problem, d, nu, fact, corr, strat, B, P):
    return C.Desc(problem, d, nu, 1, C.FACTORISATIONS[fact], C.CORRECTIONS[corr], C.STRATEGIES[strat], C.CALIBRATIONS["dynamic"],
                  1e-6, 1e-6, 0.01, 0.95, 0.2, 10.0, 0.3, 0.4, B, 20, 0, P, 0, 0)  # fmt: skip


def alternate(descs, inputs, ws, outs, rounds):
    """ms per launch of each desc (CUDA events around solve + smoothing), rounds in rotating order"""
    times = {k: [] for k in descs}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    order = list(descs)
    for r in range(rounds):
        s = r % len(order)
        for k in order[s:] + order[:s]:  # rotate who goes first
            u0_d, par_d, save_d = inputs[k]
            ev0.record()
            C.solve_device(descs[k], u0_d, par_d, None, save_d, None, workspace=ws[k], out=outs[k])
            ev1.record()
            ev1.synchronize()
            times[k].append(ev0.elapsed_time(ev1))
    return {k: np.array(v) for k, v in times.items()}


def timed_compile(desc):
    t = time.perf_counter()
    C.compile_kernels(desc)
    return time.perf_counter() - t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--members", type=int, default=bench.MEMBERS)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda:0")
    props = torch.cuda.get_device_properties(dev)
    try:
        import subprocess

        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip()  # fmt: skip
    except OSError:
        power = "unknown"
    say(f"# {props.name}, power limit {power}; torch {torch.__version__}")
    B = args.members
    t = time.perf_counter()
    ids = {"builtin": C.PROBLEM_IDS["van_der_pol"]}
    ids["full"] = C.register_problem("vdp_full", FULL, d=1, ode_order=2, num_params=1, form="full")
    ids["simple"] = C.register_problem("vdp_simple", SIMPLE, d=1, ode_order=2, num_params=1)
    say(f"registration of both sources (two check kernels): {time.perf_counter() - t:.2f} s")

    # compile time of one module per kernel family (wall clock of pn_b200_compile: NVRTC + library load)
    say("\n## NVRTC compile time per kernel family (one module: solve kernel(s) + smoothing / sampling / likelihood)")
    l96 = C.register_problem("lorenz96", LORENZ96, d=8, num_params=1)
    l63 = C.register_problem("lorenz63", LORENZ63, d=3, num_params=3)
    families = [
        ("thread per IVP + time-sliced (vdp full, headline)", headline_desc(ids["full"], B)),
        ("thread per IVP + time-sliced (vdp simple, headline)", headline_desc(ids["simple"], B)),
        ("PAIR small ensemble (vdp full, nu=4)", headline_desc(ids["full"], 1000)),
        ("thread per IVP, d=3 (lorenz63 isotropic nu=4)", desc_for(l63, 3, 4, "isotropic", "ts0", "fixedpoint", 100000, 3)),
        ("lane per dimension isotropic (lorenz96 nu=4)", desc_for(l96, 8, 4, "isotropic", "ts0", "fixedpoint", 1000, 1)),
        ("lane per dimension blockdiag (lorenz96 nu=4)", desc_for(l96, 8, 4, "blockdiag", "ts0", "fixedpoint", 1000, 1)),
        ("dense register columns, D=32 (lorenz96 EKF1 nu=3)", desc_for(l96, 8, 3, "dense", "ts1", "fixedpoint", 1000, 1)),
    ]
    for name, desc in families:
        say(f"{name:55s} {timed_compile(desc):6.2f} s")

    u0, par = bench.ensemble_inputs(0, B)
    t64 = lambda x: torch.as_tensor(x, device=dev)  # noqa: E731
    u0_d, par_d = t64(u0), t64(par)
    save_d = t64(np.linspace(bench.T0, bench.T1, bench.K_CHECKPOINTS))
    descs = {k: headline_desc(v, B) for k, v in ids.items()}
    outs, ws = {}, {}
    for k, desc in descs.items():  # warm-up: module load, workspace, launch geometry
        o = C.solve_device(desc, u0_d, par_d, None, save_d, None)
        ws[k] = o["_workspace"]
        outs[k] = {key: o[key] for key in bench.DUMP_KEYS}
    torch.cuda.synchronize()

    say("\n## headline workload: " + f"{B} members, nu={bench.NU}, dense EKF1 + fixed-point, tol {bench.TOL:g}, {bench.K_CHECKPOINTS} checkpoints")
    say("kernel info of the solve kernel:")
    for k, desc in descs.items():
        info = C.kernel_info(desc)
        say(f"  {k:8s} registers {info['registers_per_thread']:3d}  stack {info['local_bytes_per_thread']:4d} B  "
            f"ctas/SM {info['ctas_per_sm']}  grid {info['grid']}")  # fmt: skip
    ref = {key: v.cpu().numpy() for key, v in outs["builtin"].items()}
    for k in ("full", "simple"):
        same = all(np.array_equal(outs[k][key].cpu().numpy(), ref[key]) for key in bench.DUMP_KEYS)
        say(f"  {k:8s} outputs (u, u_std, counters, status) bit-identical to the built-in's: {same}")

    times = alternate(descs, {k: (u0_d, par_d, save_d) for k in descs}, ws, outs, args.rounds)
    say(f"\nsolve + smoothing, CUDA events, {args.rounds} rounds in rotating order (ms per launch):")
    base = np.median(times["builtin"])
    for k, ts in times.items():
        say(f"  {k:8s} median {np.median(ts):8.2f}  min {ts.min():8.2f}  max {ts.max():8.2f}   "
            f"{B / np.median(ts) * 1e3:12.0f} solves/s   {np.median(ts) / base:6.3f}x built-in")  # fmt: skip

    # ---- time-dependent fields ----
    say("\n## time-dependent fields on the headline workload")
    t = time.perf_counter()
    ids_t = {"simple": ids["simple"], "simple-t": C.register_problem("vdp_simple", SIMPLE_T, d=1, ode_order=2, num_params=1, time_dependent=True),
             "forced": C.register_problem("vdp_forced", FORCED, d=1, ode_order=2, num_params=3, time_dependent=True)}  # fmt: skip
    descs_t = {k: headline_desc(v, B, P=3 if k == "forced" else 1) for k, v in ids_t.items()}
    for k in ("simple-t", "forced"):
        C.compile_kernels(descs_t[k])
    say(f"registration + compilation of the two time-dependent fields: {time.perf_counter() - t:.2f} s")
    rng = np.random.default_rng(1)
    par_f = np.stack([par[:, 0], np.full(B, 1e3), rng.uniform(0.5, 2.0, B)], 1)
    inputs = {"simple": (u0_d, par_d, save_d), "simple-t": (u0_d, par_d, save_d), "forced": (u0_d, t64(par_f), save_d)}
    outs_t, ws_t = {}, {}
    for k, desc in descs_t.items():
        o = C.solve_device(desc, *inputs[k][:2], None, save_d, None)
        ws_t[k] = o["_workspace"]
        outs_t[k] = {key: o[key] for key in bench.DUMP_KEYS}
    torch.cuda.synchronize()
    say("kernel info of the solve kernel:")
    for k, desc in descs_t.items():
        info = C.kernel_info(desc)
        say(f"  {k:8s} registers {info['registers_per_thread']:3d}  stack {info['local_bytes_per_thread']:4d} B  "
            f"ctas/SM {info['ctas_per_sm']}  grid {info['grid']}")  # fmt: skip
    same = all(np.array_equal(outs_t["simple-t"][key].cpu().numpy(), outs_t["simple"][key].cpu().numpy()) for key in bench.DUMP_KEYS)
    say(f"  simple-t outputs (u, u_std, counters, status) bit-identical to simple's: {same}")
    times = alternate(descs_t, inputs, ws_t, outs_t, args.rounds)
    say(f"\nsolve + smoothing, CUDA events, {args.rounds} rounds in rotating order (ms per launch):")
    base = np.median(times["simple"])
    for k, ts in times.items():
        o = {key: v.cpu().numpy() for key, v in outs_t[k].items()}
        att = (o["n_accepted"].reshape(B, -1)[:, -1] + o["n_rejected"].reshape(B, -1)[:, -1]).astype(np.int64)
        say(f"  {k:8s} median {np.median(ts):8.2f}  min {ts.min():8.2f}  max {ts.max():8.2f}   {np.median(ts) / base:6.3f}x simple   "
            f"attempted steps {att.sum():11d} (per member median {int(np.median(att))}, max {att.max()})  "
            f"status != 0: {int((o['status'] != 0).sum())}")  # fmt: skip
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
