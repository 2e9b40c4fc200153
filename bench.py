"""bench.py -- headline benchmark: Van der Pol ensemble of 65,536 randomised initial conditions.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--members B]
                    [--workload vdp|c4] [--scaling weak|strong] [--dump-outputs DIR]

Workload `vdp` (default; BASELINE.json configs[1], SURVEY 8d C2): stiff Van der Pol (mu=1e3), dense EKF1
(ode_order=2) + fixed-point smoother at 50 checkpoints on [0, 6.3], nu=4, dynamic calibration,
atol=rtol=1e-6, dt0=0.01; member b starts at u0 = 2 + 0.5 U(-1,1), u'0 = 0.5 U(-1,1) (seed 0).
Workload `c4` (BASELINE.json configs[3], SURVEY 8d C4): Pleiades (d=14, ode_order=2), blockdiag EKF0,
nu = 3, 4, 5, 16,384 members = 2,048 initial conditions x 8 tolerances 1e-3..1e-10 (per-member
tolerances: one launch per nu), 50 checkpoints on [0, 3].

A "step" is one pass of the hot path over the whole ensemble: the persistent solver kernel + the
smoothing sweep (c4: once per nu).  N>1: one ensemble shard per rank, then ONE NCCL all-gather of the
packed checkpoint results and step statistics.  `--scaling weak` (default): 65,536 members per rank;
with N>1 the same run also measures STRONG scaling (65,536 members in total, interleaved over the
ranks) and reports it under "strong_scaling" in the same JSON line.  `--scaling strong` makes the strong
run the headline `value`.

One JSON line on stdout (rank 0).  `value` = IVP solves/s with inputs resident in HBM; `e2e` = the
same through the public Python API with HOST buffers (H2D + solve + D2H inside the timed region);
`roofline` = the solver kernel's algorithmic fp64 flop rate against the DFMA peak measured on this
GPU by a register-resident FMA-chain kernel (MEASURED_PEAKS.json carries no fp64 entry; the path is
fp64-CUDA-core bound, not HBM or tensor bound -- `roofline.hbm` shows the HBM side for context);
`cpu_baseline` = the CPU oracle (C port of the reference algorithm; jax/probdiffeq cannot be
installed here) on the host cores on a bounded sample of the same members -- whose results are also
compared with the GPU's for those members, bit for bit (`parity_checked_members`): the bench fails if
they differ.

`--dump-outputs DIR` writes what the last timed step returned, so that two builds can be compared output
for output on identical seeded inputs: DIR/members.npy (global member indices) and DIR/nu<nu>_<key>.npy
for key in u, u_std, n_accepted, n_rejected, status (float64; the counters are exact), rows in member
order.  When all members would exceed DUMP_BYTES, a fixed seeded sample of members is written.
"""

import argparse
import glob
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "code-adaptive-prob-ode-solvers_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

MEMBERS = 65536
K_CHECKPOINTS = 50
T0, T1 = 0.0, 6.3
TOL = 1e-6
MU = 1e3
NU = 4
METRIC = "ivp_solves_per_s"
UNIT = "IVP-solves/s"
PARITY_TOL = 1e-9  # north_star: checkpoint means / standard deviations within 1e-9 relative
DUMP_BYTES = 32 << 20  # --dump-outputs writes at most this much
DUMP_KEYS = ("u", "u_std", "n_accepted", "n_rejected", "status")


def flops_dense_fixedpoint(n, d, f_vf, f_jac):
    """SURVEY 8d: dense EKF1 + fixed-point, D = n d: 20.33 D^3 + (2n + 8d) D^2 + 4 D d^2 + F_f + F_J."""
    D = n * d
    return 20.33 * D**3 + (2 * n + 8 * d) * D**2 + 4 * D * d**2 + f_vf + f_jac


def flops_blockdiag_fixedpoint(n, d, f_vf):
    """SURVEY 8d: blockdiag EKF0 + fixed-point: d (22.33 n^3 + 15 n^2 + 8 n + 10) + F_f."""
    return d * (22.33 * n**3 + 15 * n**2 + 8 * n + 10) + f_vf


def ensemble_inputs(first, count, stride=1):
    """Members first, first+stride, ... of the seeded global VdP ensemble (seed 0, SURVEY 8d C2)."""
    total = first + stride * count
    rng = np.random.default_rng(0)
    ab = rng.uniform(-1, 1, (total, 2))  # row b = member b, whatever the ensemble size
    idx = first + stride * np.arange(count)
    u0 = np.stack([2.0 + 0.5 * ab[idx, 0], 0.5 * ab[idx, 1]], 1).reshape(count, 2, 1)
    params = np.full((count, 1), MU)
    return np.ascontiguousarray(u0), params


PLEIADES_X = np.array([3.0, 3.0, -1.0, -3.0, 2.0, -2.0, 2.0, 3.0, -3.0, 2.0, 0.0, 0.0, -4.0, 4.0])
PLEIADES_DX = np.array([0, 0, 0, 0, 0, 1.75, -1.5, 0, 0, 0, -1.25, 1.0, 0, 0.0])
C4_TOLS = 10.0 ** -np.arange(3, 11)


def c4_inputs(first, count, stride=1):
    """Members of the seeded global Pleiades ensemble (seed 2, SURVEY 8d C4): member b has tolerance index
    (b // 8) % 8 and initial condition (b % 8) + 8 (b // 64) -- every run of 64 consecutive members is 8 initial
    conditions x 8 tolerances, and ranks that own members r, r + G, ... (G = 1, 2, 4, 8) all see the same mix of
    tolerances; positions perturbed by 0.01 N(0, I); rtol = 10 tol, atol = 1e-3 rtol
    (experiments/3_workprec_harder/run_harder.py:45-47)."""
    total = first + stride * count
    n_ic = 8 * ((total + 63) // 64)
    rng = np.random.default_rng(2)
    pos = PLEIADES_X + 0.01 * rng.standard_normal((n_ic, 14))
    idx = first + stride * np.arange(count)
    ic, it = (idx % 8) + 8 * (idx // 64), (idx // 8) % 8
    u0 = np.stack([pos[ic], np.tile(PLEIADES_DX, (count, 1))], 1)
    rtol = 10.0 * C4_TOLS[it]
    tol = np.stack([1e-3 * rtol, rtol], 1)
    return np.ascontiguousarray(u0), np.ascontiguousarray(tol)


class Workload:
    """What one bench step solves: a list of launches over the same seeded global ensemble."""

    def __init__(self, name):
        from odecheckpts_b200 import _cabi

        self.name = name
        self.cabi = _cabi
        if name == "vdp":
            self.default_members, self.K, self.d, self.q = MEMBERS, K_CHECKPOINTS, 1, 2
            self.save_at = np.linspace(T0, T1, self.K)
            self.nus = [NU]
            self.kernel_name = "pn_scalar_kernel<VanDerPol,4,fixedpoint>"
        elif name == "c4":
            self.default_members, self.K, self.d, self.q = 16384, 50, 14, 2
            self.save_at = np.linspace(0.0, 3.0, self.K)
            self.nus = [3, 4, 5]
            self.kernel_name = "pn_scalar_kernel<Pleiades,nu,fixedpoint,GROUP=16,blockdiag> (nu = 3, 4, 5)"
        else:
            raise SystemExit(f"unknown workload {name}")

    def inputs(self, first, count, stride):
        """(u0 [B,q,d], params [B,P] | None, tol [B,2] | None)"""
        if self.name == "vdp":
            u0, par = ensemble_inputs(first, count, stride)
            return u0, par, None
        u0, tol = c4_inputs(first, count, stride)
        return u0, None, tol

    def desc(self, nu, B):
        c = self.cabi
        if self.name == "vdp":
            return c.Desc(c.PROBLEM_IDS["van_der_pol"], 1, nu, 2, c.FACTORISATIONS["dense"], c.CORRECTIONS["ts1"],
                          c.STRATEGIES["fixedpoint"], c.CALIBRATIONS["dynamic"], TOL, TOL, 0.01,
                          0.95, 0.2, 10.0, 0.3, 0.4, B, self.K, 0, 1, 0, 0)  # fmt: skip
        return c.Desc(c.PROBLEM_IDS["pleiades"], 14, nu, 2, c.FACTORISATIONS["blockdiag"], c.CORRECTIONS["ts0"],
                      c.STRATEGIES["fixedpoint"], c.CALIBRATIONS["dynamic"], 1e-6, 1e-6, 0.1,
                      0.95, 0.2, 10.0, 0.3, 0.4, B, self.K, 0, 0, 0, 0)  # fmt: skip

    def oracle_config(self, nu):
        from oracle import pn_oracle

        if self.name == "vdp":
            return pn_oracle.make_config("van_der_pol", 1, nu, 2, factorisation="dense", correction="ts1",
                                         strategy="fixedpoint", calibration="dynamic", atol=TOL, rtol=TOL, dt0=0.01,
                                         num_params=1)  # fmt: skip
        # the lane-per-dimension kernel sums its norms with a 16-lane butterfly: same order in the oracle
        return pn_oracle.make_config("pleiades", 14, nu, 2, factorisation="blockdiag", correction="ts0",
                                     strategy="fixedpoint", calibration="dynamic", atol=1e-6, rtol=1e-6, dt0=0.1,
                                     num_params=0, reduction_group=16)  # fmt: skip

    def flops_per_attempt(self, nu):
        n = nu + 1
        if self.name == "vdp":
            return flops_dense_fixedpoint(n, 1, 8, 8)
        return flops_blockdiag_fixedpoint(n, 14, 42 * 13 + 42)

    def sweep_flops_per_checkpoint(self, nu):
        n = nu + 1
        return (5.33 * n**3 + 2 * n**2) * (1 if self.name == "vdp" else self.d)

    def algorithmic_bytes(self, B):
        # inputs (q d + P + 3 doubles) + outputs (K 2d doubles + (K + 2) counters) per member and launch (SURVEY 8d)
        P = 1 if self.name == "vdp" else 2
        return len(self.nus) * B * ((self.q * self.d + P + 3) * 8 + self.K * 2 * self.d * 8 + (self.K + 2) * 8)

    def describe(self, B, world, scaling):
        per = f"{B} members per GPU x {world} GPU(s)" if scaling == "weak" else f"{B * world} members in total over {world} GPU(s)"
        if self.name == "vdp":
            return (f"van_der_pol mu=1e3 ensemble, {per} (seed 0: u0=2+0.5U, u'0=0.5U), dense EKF1 (ode_order=2) + fixed-point "
                    f"smoother, nu={NU}, dynamic calibration, atol=rtol={TOL:g}, dt0=0.01, {self.K} checkpoints on [0, 6.3]")  # fmt: skip
        return (f"pleiades (d=14, ode_order=2) tolerance sweep, {per} = initial conditions (seed 2: positions + 0.01 N) x 8 "
                f"tolerances 1e-3..1e-10 (rtol = 10 tol, atol = 1e-3 rtol), blockdiag EKF0 + fixed-point smoother, "
                f"nu = 3, 4, 5 (one launch each), dynamic calibration, dt0=0.1, {self.K} checkpoints on [0, 3]")  # fmt: skip


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)  # fmt: skip
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for nm, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {
            "sm_mhz": float(np.median(sm)) if sm else None,
            "sm_max_mhz": float(max(smax)) if smax else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


def ncu_dram_bytes():
    """DRAM bytes of one solver-kernel launch on the headline workload, read from the newest committed
    `ncu --set full` summary of that kernel under profiles/ (dram__bytes_read.sum + dram__bytes_write.sum)."""
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_scalar_kernel*ncu.txt")))
    cands = [c for c in cands if "_v1_" not in c]
    if not cands:
        return None, None
    path = cands[-1]
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    total, seen = 0.0, 0
    for line in open(path):
        m = re.match(r"\s*dram__bytes_(read|write)\.sum\s+([0-9.eE+-]+)\s+(\w+)\s*$", line)
        if m and m.group(3) in scale:
            total += float(m.group(2)) * scale[m.group(3)]
            seen += 1
    return (total, os.path.relpath(path, ROOT)) if seen == 2 else (None, None)


def ncu_instruction_fetch():
    """The second bound of the headline kernel, from the same committed ncu summary: its straight-line step (40 KB of
    SASS) does not fit an SM's instruction cache, so every round of an SM's eight warps refetches it from the GPC-level
    instruction cache (ncu unit `gcc`), whose request rate is what the launch saturates (DESIGN.md 3.1)."""
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_scalar_kernel*ncu.txt")))
    cands = [c for c in cands if "_v1_" not in c]
    if not cands:
        return None
    vals = {}
    for line in open(cands[-1]):
        t = line.split()
        if len(t) >= 2 and t[0] in ("gcc__cache_requests_type_instruction.sum", "smsp__inst_executed.sum",
                                    "gcc__cache_requests_type_instruction.sum.pct_of_peak_sustained_elapsed"):
            vals[t[0]] = float(t[1])
    if len(vals) != 3:
        return None
    req, inst = vals["gcc__cache_requests_type_instruction.sum"], vals["smsp__inst_executed.sum"]
    return {
        "bound": "instruction fetch (GPC-level instruction cache requests)", "frac": vals["gcc__cache_requests_type_instruction.sum.pct_of_peak_sustained_elapsed"] / 100.0,
        "requests_per_launch": req, "warp_instructions_per_launch": inst, "lines_refetched_per_instruction_line": req * 8.0 / inst,
        "source": f"gcc__cache_requests_type_instruction.sum(.pct_of_peak_sustained_elapsed), ncu --set full, {os.path.relpath(cands[-1], ROOT)}",
    }  # fmt: skip


def cpu_sample_size(members, cores):
    return int(min(members, max(512, 640 * cores)))  # ~10-20 s of CPU work on the VdP workload


def cpu_oracle_run(wl, first, count, threads):
    """Runs the CPU oracle (C port of the reference algorithm, OpenMP over members) on members
    first .. first+count-1 of the seeded global ensemble, all launches of the workload.
    Returns (seconds, accepted steps, list of per-launch result dicts)."""
    from oracle import pn_oracle

    u0, par, tol = wl.inputs(first, count, 1)
    secs, acc, outs = 0.0, 0.0, []
    for nu in wl.nus:
        cfg = wl.oracle_config(nu)
        t0 = time.perf_counter()
        out = pn_oracle.solve_save_at_batch(cfg, u0, par if par is not None else np.zeros((count, 1)), wl.save_at,
                                            tol=tol, num_threads=threads)  # fmt: skip
        secs += time.perf_counter() - t0
        acc += float(out["n_accepted"][:, -1].sum())
        outs.append(out)
    return secs, acc, outs


def dump_outputs(path, nus, results, first=0):
    """--dump-outputs: results[i] = {key: [B, ...] numpy array or torch tensor} of the launch with nu = nus[i], row r
    being member first + r of the seeded ensemble.  All rows, or a fixed seeded sample of them that fits DUMP_BYTES."""
    B = len(results[0]["u"])
    per_member = 8 + sum(8 * int(np.prod(res[k].shape[1:])) for res in results for k in DUMP_KEYS)
    n = min(B, DUMP_BYTES // per_member)
    rows = np.arange(B) if n == B else np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "members.npy"), (first + rows).astype(np.float64))
    for nu, res in zip(nus, results):
        for k in DUMP_KEYS:
            x = res[k]
            if isinstance(x, np.ndarray):
                x = x[rows]
            else:
                import torch

                x = x[torch.from_numpy(rows).to(x.device)].cpu().numpy()
            np.save(os.path.join(path, f"nu{nu}_{k}.npy"), x.astype(np.float64))


def parity_against(outs_cpu, outs_gpu):
    """Compares oracle and GPU results member by member.  Returns (max relative difference of u / u_std,
    bit-exact?, counts identical?)."""
    worst, exact, counts = 0.0, True, True
    for c, g in zip(outs_cpu, outs_gpu):
        n = c["u"].shape[0]
        for key in ("u", "u_std"):
            a, b = c[key], g[key][:n]
            exact &= bool(np.array_equal(a, b, equal_nan=True))
            denom = np.maximum(np.abs(a), 1e-300)
            diff = np.where(np.isfinite(a) & np.isfinite(b), np.abs(a - b) / denom, np.where(np.isnan(a) & np.isnan(b), 0.0, np.inf))
            worst = max(worst, float(diff.max()) if diff.size else 0.0)
        for key in ("n_accepted", "n_rejected", "status"):
            counts &= bool(np.array_equal(c[key], g[key][:n]))
    return worst, exact, counts


def run_reference(args):
    """--impl reference: the reference algorithm's CPU implementation on the host cores.  The
    reference itself (JAX + probdiffeq, jit + vmap) cannot be installed in this image (no wheels,
    no network), so this is the validated C port under oracle/ with all host threads.  The timed steps
    together process exactly the sample `cpu_baseline` uses (the first 640 x cores members of the same
    seeded ensemble), one slice per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = Workload(args.workload)
    members = args.members or wl.default_members
    cores = os.cpu_count() or 1
    sample = cpu_sample_size(members, cores)
    chunk = max(cores, (sample + args.steps - 1) // args.steps)
    for _ in range(args.warmup):
        cpu_oracle_run(wl, 0, min(chunk, 4 * cores), cores)
    done, secs, acc = 0, 0.0, 0.0
    for i in range(args.steps):
        first = (i * chunk) % max(1, sample - chunk + 1) if sample > chunk else 0
        s, a, outs = cpu_oracle_run(wl, first, min(chunk, sample), cores)
        secs += s
        acc += a
        done += min(chunk, sample) * len(wl.nus)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, wl.nus, outs, first)
    value = done / secs
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "accepted_steps_per_s": acc / secs,
        "config": {"workload": wl.describe(members, args.gpus, "weak"),
                   "cpu_sample": f"{done // len(wl.nus)} members = the first {sample} of the seeded ensemble in slices of {chunk} per step"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"first {sample} members of the seeded ensemble, {chunk} per step, OpenMP over members"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference = C port of the reference's algorithm (oracle/); JAX/probdiffeq are not installable here",
    }  # fmt: skip
    print(json.dumps(line), flush=True)


_JSON_FD = None  # the original stdout when file descriptor 1 has been pointed at stderr (N > 1)


def _emit(line):
    text = json.dumps(line) + "\n"
    if _JSON_FD is None:
        sys.stdout.write(text)
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, text.encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="vdp", choices=["vdp", "c4"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--members", type=int, default=0, help="members per GPU (weak) / in total (strong); default: the workload's")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="N>1: skip the additional strong-scaling measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    from odecheckpts_b200 import _cabi, ensemble, ivps, ivpsolvers

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        # stdout carries ONE JSON line: libraries that write to file descriptor 1 themselves (NCCL prints its version
        # banner there at the first collective) are sent to stderr; the line goes to the original descriptor
        sys.stdout.flush()
        global _JSON_FD
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the solver has no CPU fallback")
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    _cabi.lib()
    wl = Workload(args.workload)
    members = args.members or wl.default_members
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(scaling, steps, warmup, sample_clocks, dump_dir=None):
        """Times `steps` passes over the ensemble.  weak: `members` per rank; strong: `members` in total.
        dump_dir: where rank 0 writes the results of the last timed step (--dump-outputs)."""
        B_total = members * world if scaling == "weak" else members
        sizes = ensemble.shard_sizes(B_total, world)
        B = sizes[rank]
        u0_h, par_h, tol_h = wl.inputs(rank, B, world)  # interleaved shard: members rank, rank + G, ...
        T = lambda x: None if x is None else torch.as_tensor(np.ascontiguousarray(x), device=dev)  # noqa: E731
        u0_d, par_d, tol_d, save_d = T(u0_h), T(par_h), T(tol_h), T(wl.save_at)
        launches = []
        for nu in wl.nus:
            desc = wl.desc(nu, B)
            packed = ensemble.PackedResults(B_total, wl.K, wl.d, world, dev)  # results live in ONE packed buffer
            out = packed.local(B)
            launches.append({"nu": nu, "desc": desc, "packed": packed, "out": out, "ws": None})

        def step():
            flush.zero_()  # evict L2 between timed iterations
            for L in launches:
                res = _cabi.solve_device(L["desc"], u0_d, par_d, tol_d, save_d, None, workspace=L["ws"], out=L["out"])
                L["ws"] = res["_workspace"]
                if world > 1:
                    L["gathered"] = L["packed"].all_gather()  # ONE collective per solve

        _cabi.set_profiling(True)
        for _ in range(max(warmup, 3)):
            step()
        barrier()
        sampler = ClockSampler(local_rank) if (sample_clocks and rank == 0) else None
        if sampler:
            sampler.start()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        barrier()
        elapsed_ms = e0.elapsed_time(e1)
        clocks = sampler.stop() if sampler else None
        if dump_dir and rank == 0:  # before the pass below overwrites the outputs
            res = [L["out"] if world == 1 else {k: L["packed"].member_order(v) for k, v in L["gathered"].items()}
                   for L in launches]  # fmt: skip
            dump_outputs(dump_dir, wl.nus, res)
        # kernel times of one more (untimed) pass, launch by launch, from events on the launching stream
        kernel_ms, smooth_ms = [], []
        flush.zero_()
        for L in launches:
            res = _cabi.solve_device(L["desc"], u0_d, par_d, tol_d, save_d, None, workspace=L["ws"], out=L["out"])
            a, b = _cabi.last_timing()
            kernel_ms.append(a)
            smooth_ms.append(b)
        _cabi.set_profiling(False)
        if world > 1:
            tt = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            elapsed_ms = float(tt.item())
        acc = sum(L["out"]["n_accepted"][:, -1].double().sum() for L in launches)
        rej = sum(L["out"]["n_rejected"].double().sum() for L in launches)
        bad = sum((L["out"]["status"] != 0).sum().double() for L in launches)
        stats = torch.stack([acc, rej, bad])
        local_attempts = [float((L["out"]["n_accepted"][:, -1].double().sum() + L["out"]["n_rejected"].double().sum()).item())
                          for L in launches]  # fmt: skip
        if world > 1:
            dist.all_reduce(stats)
        acc_t, rej_t, bad_t = (float(x) for x in stats.tolist())
        ms = elapsed_ms / steps
        return {
            "B": B, "B_total": B_total, "ms_per_step": ms, "value": B_total * len(wl.nus) / (ms * 1e-3),
            "acc": acc_t, "rej": rej_t, "bad": bad_t, "kernel_ms": kernel_ms, "smooth_ms": smooth_ms,
            "local_attempts": local_attempts, "clocks": clocks, "launches": launches,
            "inputs": (u0_h, par_h, tol_h), "info": _cabi.kernel_info(launches[0]["desc"]),
        }  # fmt: skip

    fp64_peak = _cabi.measure_fp64_peak()
    head = measure(args.scaling, args.steps, args.warmup, True, args.dump_outputs)
    other = None
    if world > 1 and not args.no_strong:
        other = measure("strong" if args.scaling == "weak" else "weak", args.steps, args.warmup, False)

    # ---- end-to-end through the public API with host buffers ------------------------------
    B, B_total = head["B"], head["B_total"]
    u0_h, par_h, tol_h = head["inputs"]
    e2e = None
    if wl.name == "vdp":
        vf, (y0, dy0), _ = ivps.van_der_pol(mu=MU)
        solve = ivpsolvers.solve(f"ts0-{NU}", vf, y0, save_at=wl.save_at, dt0=0.01, atol=TOL, rtol=TOL, ode_order=2,
                                 factorisation="dense", correction="ts1", return_marginals=False, device=local_rank)  # fmt: skip
        pin = [torch.empty((B, 1), dtype=torch.float64, pin_memory=True) for _ in range(2)]  # pinned host inputs
        pin[0].copy_(torch.from_numpy(u0_h[:, 0, :]))
        pin[1].copy_(torch.from_numpy(u0_h[:, 1, :]))
        u0_pin = (pin[0].numpy(), pin[1].numpy())
        e2e_steps = max(2, min(args.steps, 3))
        res, aux = solve(u0_pin, ())  # warm-up: two calls, so that both generations of recycled host result
        res, aux = solve(u0_pin, ())  # buffers exist (the previous results are still alive during a call)
        barrier()
        t_e2e = time.perf_counter()
        for _ in range(e2e_steps):
            res, aux = solve(u0_pin, ())
            sol = aux["solution"]
        barrier()
        e2e_s = (time.perf_counter() - t_e2e) / e2e_steps
        if world > 1:
            tt = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            e2e_s = float(tt.item())
        h2d = u0_h.nbytes + par_h.nbytes + wl.save_at.nbytes
        d2h = res.nbytes + sol.u_std.nbytes + sol.num_steps.nbytes + sol.num_rejected.nbytes + sol.status.nbytes
        e2e_ok = bool(np.array_equal(res, head["launches"][0]["out"]["u"].cpu().numpy()))
        e2e = {"value": B_total / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "api": "odecheckpts_b200.ivpsolvers.solve(...)(u0_host, p) -> pn_b200_solve_save_at_host",
               "matches_device_path": e2e_ok}  # fmt: skip
    else:
        # c4: the host-buffer C-ABI entry (per-member tolerances are not part of the reference's solve() signature)
        descs = [wl.desc(nu, B) for nu in wl.nus]
        for dsc in descs:
            _cabi.solve_host(dsc, u0_h, par_h, tol_h, wl.save_at, None, device=local_rank)
        barrier()
        t_e2e = time.perf_counter()
        d2h = 0
        for dsc in descs:
            r = _cabi.solve_host(dsc, u0_h, par_h, tol_h, wl.save_at, None, device=local_rank)
            d2h += sum(r[k].nbytes for k in ("u", "u_std", "n_accepted", "n_rejected", "status"))
        barrier()
        e2e_s = time.perf_counter() - t_e2e
        if world > 1:
            tt = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            e2e_s = float(tt.item())
        h2d = len(descs) * (u0_h.nbytes + tol_h.nbytes + wl.save_at.nbytes)
        e2e_ok = bool(np.array_equal(r["u"], head["launches"][-1]["out"]["u"].cpu().numpy()))
        e2e = {"value": B_total * len(wl.nus) / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "api": "pn_b200_solve_save_at_host (C ABI, host buffers), one call per nu", "matches_device_path": e2e_ok}  # fmt: skip

    if rank == 0:
        flops = 0.0
        for nu, att in zip(wl.nus, head["local_attempts"]):
            W = wl.flops_per_attempt(nu)
            flops += att * W + B * (wl.K - 1) * 1.3 * W  # + two extra predictions and a marginalisation per checkpoint
        k_ms = float(np.sum(head["kernel_ms"]))
        achieved = flops / (k_ms * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        hbm_ach = wl.algorithmic_bytes(B) / (k_ms * 1e-3) / 1e9
        traffic, traffic_src = ncu_dram_bytes() if (wl.name == "vdp" and B == MEMBERS) else (None, None)
        ms_per_step = head["ms_per_step"]
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "accepted_steps_per_s": head["acc"] / (ms_per_step * 1e-3),
            "attempted_steps_per_s": (head["acc"] + head["rej"]) / (ms_per_step * 1e-3),
            "accepted_per_member": head["acc"] / (B_total * len(wl.nus)), "rejected_per_member": head["rej"] / (B_total * len(wl.nus)),
            "failed_members": int(head["bad"]),
            "config": {
                "workload": wl.describe(members, world, args.scaling),
                "members_total": B_total,
                "parallelism": (f"ensemble sharded x{world} (member b on rank b mod {world}), ONE all-gather of the packed results per solve"
                                if world > 1 else "single GPU"),
                "l2": "256 MiB device memset between timed steps (L2 flush)",
                "kernel": head["info"],
                "scheduling": ("run to completion (PN_B200_NO_SLICE)" if os.environ.get("PN_B200_NO_SLICE")
                               else "time-sliced members: parked at quantum boundaries, most lagging ready member first"),
            },
            "gpu_launches": 2 * len(wl.nus) * args.steps,
            "e2e": e2e,
            "roofline": {
                "bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak,
                "traffic": traffic,
                "traffic_source": (f"dram__bytes_read.sum + dram__bytes_write.sum, ncu --set full, {traffic_src}" if traffic_src else None),
                "kernel": wl.kernel_name, "kernel_ms": k_ms,
                "smooth_kernel_ms": float(np.sum(head["smooth_ms"])),
                "flops_per_attempt": [wl.flops_per_attempt(nu) for nu in wl.nus] if len(wl.nus) > 1 else wl.flops_per_attempt(wl.nus[0]),
                "attempts_per_launch": head["local_attempts"] if len(wl.nus) > 1 else head["local_attempts"][0],
                "peak_source": "DFMA-chain microbenchmark in this run (pn_b200_measure_fp64_peak); MEASURED_PEAKS.json has no fp64 entry",
                "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650"},
                "instruction_fetch": ncu_instruction_fetch() if wl.name == "vdp" else None,
            },
            "clocks": head["clocks"],
        }  # fmt: skip
        if other is not None:
            key = "strong_scaling" if args.scaling == "weak" else "weak_scaling"
            line[key] = {
                "members_total": other["B_total"], "members_per_gpu": other["B"], "ms_per_step": other["ms_per_step"],
                "value": other["value"], "unit": UNIT, "kernel_ms": float(np.sum(other["kernel_ms"])),
                "note": "same seeded ensemble, interleaved over the ranks; measured in the same run with the same timing rules",
            }  # fmt: skip
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            sample = cpu_sample_size(B, cores)
            if wl.name != "vdp":
                sample = min(sample, 32 * cores)  # a Pleiades member costs ~40x a Van der Pol member on the CPU
            secs, acc_cpu, outs_cpu = cpu_oracle_run(wl, 0, sample, cores)
            outs_gpu = [{k: L["out"][k][:sample].cpu().numpy() for k in ("u", "u_std", "n_accepted", "n_rejected", "status")}
                        for L in head["launches"]]  # fmt: skip
            worst, exact, counts = parity_against(outs_cpu, outs_gpu)
            line["cpu_baseline"] = {
                "value": sample * len(wl.nus) / secs, "unit": UNIT, "cores": cores, "kind": "port",
                "accepted_steps_per_s": acc_cpu / secs, "seconds": secs,
                "sample": f"first {sample} members of the same seeded ensemble, C oracle with OpenMP over members "
                          "(JAX/probdiffeq not installable here)",
            }  # fmt: skip
            line["parity_checked_members"] = sample * len(wl.nus)
            line["parity_max_rel"] = worst
            line["parity_bit_exact"] = bool(exact and counts)
            if not (worst <= PARITY_TOL and counts):
                _emit(line)
                raise SystemExit(f"bench: GPU results differ from the oracle on the sampled members (max rel {worst:g}, counts equal: {counts})")
        _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
