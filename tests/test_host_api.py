"""CPU-only tests: host logic, argument errors, C-ABI symbols (no compute calls without a GPU)."""

import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_symbol_the_header_declares():
    from odecheckpts_b200 import _cabi

    lib = _cabi.lib()
    header = open(os.path.join(ROOT, "include", "pn_b200.h")).read()
    declared = set(re.findall(r"\b(pn_b200_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_cabi.EXPORTS)
    for name in declared:
        assert getattr(lib, name) is not None


def test_descriptor_struct_matches_header_layout():
    from odecheckpts_b200 import _cabi

    # 8 int32 + 8 doubles + 3 int64 + 2 int32 + 1 int64
    assert C.sizeof(_cabi.Desc) == 8 * 4 + 8 * 8 + 3 * 8 + 2 * 4 + 8
    assert C.sizeof(_cabi.KernelInfo) == 8 * 4


def _desc(_cabi, **over):
    base = dict(problem=5, d=1, nu=4, ode_order=2, factorisation=2, correction=1, strategy=1, calibration=1,
                atol=1e-6, rtol=1e-6, dt0=0.01, safety=0.95, factor_min=0.2, factor_max=10.0, power_integral=0.3,
                power_proportional=0.4, batch=8, num_save_at=5, max_attempts=0, num_params=1, flags=0, traj_capacity=0)  # fmt: skip
    base.update(over)
    return _cabi.Desc(*[base[name] for name, _ in _cabi.Desc._fields_])


def test_supported_and_workspace_queries_need_no_gpu(monkeypatch):
    from odecheckpts_b200 import _cabi

    # the opt-in cooperative kernel for scalar ODEs has no time-sliced scheduler: header + slots only
    n, D, K2, B2 = 5, 1, 50, 1000
    slot = (n * n + n * D + n * (n + 1) // 2) + (n * D + n * (n + 1) // 2)
    header2 = (256 + 2 * 128 * 4 + B2 * 8 + 255) // 256 * 256
    monkeypatch.setenv("PN_B200_COOP_MAX_BATCH", "20000")
    assert _cabi.workspace_bytes(_desc(_cabi, batch=B2, num_save_at=K2)) == header2 + K2 * slot * B2 * 8
    # the thread-per-IVP kernels (default)
    monkeypatch.delenv("PN_B200_COOP_MAX_BATCH")
    d = _desc(_cabi)
    assert _cabi.supported(d)
    n, D, K, B = 5, 1, 5, 8
    slot = (n * n + n * D + n * (n + 1) // 2) + (n * D + n * (n + 1) // 2)
    header = (256 + 2 * 128 * 4 + B * 8 + 255) // 256 * 256  # ticket + stats, ordering histogram / cursors, order[B]
    assert _cabi.workspace_bytes(d) == header + K * slot * B * 8  # [B][K][slot]
    # enough checkpoints for the time-sliced scheduler (fixed-point thread-per-IVP kernels): + ready queues
    # [K-1 groups][B] int32, a 1 KB control block, parked states [B][running conditional + state + 8 scalars]
    K2, B2 = 50, 1000
    header2 = (256 + 2 * 128 * 4 + B2 * 8 + 255) // 256 * 256
    queues = ((K2 - 1) * B2 * 4 + 255) // 256 * 256
    ctx = ((n * n + n * D + n * (n + 1) // 2) + (n * D + n * (n + 1) // 2) + 8 + 1) // 2 * 2
    # (ensembles of up to 148 x 128 members are served by the filter-lane + backward-lane build, which runs every
    # member to completion: no scheduler region)
    assert _cabi.workspace_bytes(_desc(_cabi, batch=B2, num_save_at=K2)) == header2 + K2 * slot * B2 * 8
    monkeypatch.setenv("PN_B200_PAIR", "0")
    assert _cabi.workspace_bytes(_desc(_cabi, batch=B2, num_save_at=K2)) == header2 + K2 * slot * B2 * 8 + queues + 1024 + B2 * ctx * 8
    monkeypatch.delenv("PN_B200_PAIR")
    # ... but not for the filter strategy, trajectory recording or fixed grids
    slot_f = n * D + n * (n + 1) // 2
    assert _cabi.workspace_bytes(_desc(_cabi, batch=B2, num_save_at=K2, strategy=0)) == header2 + K2 * slot_f * B2 * 8
    assert _cabi.workspace_bytes(_desc(_cabi, batch=B2, num_save_at=K2, flags=1)) == header2 + K2 * slot * B2 * 8
    assert not _cabi.supported(_desc(_cabi, problem=3, d=14))  # Pleiades has no thread-per-IVP kernel
    assert not _cabi.supported(_desc(_cabi, factorisation=0))  # isotropic + ts1 is not a valid model
    assert not _cabi.supported(_desc(_cabi, nu=9))
    with pytest.raises(NotImplementedError):
        _cabi.workspace_bytes(_desc(_cabi, nu=9))
    with pytest.raises(ValueError):
        _cabi.workspace_bytes(_desc(_cabi, num_save_at=1))


def test_vector_field_resolution_through_wrappers():
    from odecheckpts_b200 import ivps

    vf, u0, tspan = ivps.van_der_pol(mu=123.0)

    def wrapped(*y, t):
        return vf(*y, t=t, p=())

    field, params = ivps.resolve_vector_field(lambda *y, t: wrapped(*y, t=t), u0)
    assert field.name == "van_der_pol" and params == (123.0,)
    with pytest.raises(TypeError):
        ivps.resolve_vector_field(lambda y, t: -y, (np.zeros(1),))
    # called with real arrays the functor evaluates on the host
    np.testing.assert_allclose(vf(np.array([2.0]), np.array([0.0])), [-246.0])


def test_solve_factory_keeps_the_reference_error_conventions():
    from odecheckpts_b200 import ivps, ivpsolvers

    vf, u0, tspan, args = ivps.logistic()
    save_at = np.linspace(*tspan, num=5)
    with pytest.raises(ValueError):
        ivpsolvers.solve("ts1-4", vf, u0[0], save_at=save_at, dt0=0.1, atol=1e-3, rtol=1e-3)  # ivpsolvers.py:38-39
    with pytest.raises(ValueError):
        ivpsolvers.solve("ts0-4", vf, u0[0], save_at=save_at, dt0=0.1, atol=1e-3, rtol=1e-3, calibrate="mle")
    solve = ivpsolvers.solve("ts0-4", vf, u0[0], save_at=save_at, dt0=0.1, atol=1e-3, rtol=1e-3)
    with pytest.raises(ValueError, match="Tuple expected."):
        solve(u0[0], args)  # ivpsolvers.py:56-57


def test_builder_vocabulary_and_descriptor_assembly():
    from odecheckpts_b200 import _cabi, ivps
    from odecheckpts_b200.probdiffeq import impl, ivpsolve, ivpsolvers, taylor

    vf, (u0, du0), (t0, t1) = ivps.van_der_pol()
    impl.impl.select("dense", ode_shape=(1,))
    ibm = ivpsolvers.prior_ibm(num_derivatives=4)
    ts1 = ivpsolvers.correction_ts1(ode_order=2)
    strategy = ivpsolvers.strategy_filter(ibm, ts1)
    solver = ivpsolvers.solver_dynamic(strategy)
    tcoeffs = taylor.odejet_padded_scan(lambda *y: vf(*y, t=t0), [u0, du0], num=3)
    init = solver.initial_condition(tcoeffs, 1.0)
    field, params, inits, nu, fact = ivpsolve._prepare(vf, init, t0, None)
    assert (field.name, params, nu, fact) == ("van_der_pol", (1000.0,), 4, "dense")
    use_torch, B, batched, u0s, par, tol, scale = ivpsolve._stack_members(inits, params, None, 1.0, 1)
    assert (use_torch, B, batched) == (False, 1, False) and u0s.shape == (1, 2, 1) and par.shape == (1, 1) and scale is None
    ctrl = ivpsolve.control_proportional_integral()
    d = ivpsolve._make_desc(field, nu, fact, solver, 1e-3, 1e-3, ctrl, 0.01, 1, 2)
    assert (d.problem, d.nu, d.ode_order, d.factorisation, d.correction, d.strategy, d.calibration) == (5, 4, 2, 2, 1, 0, 1)
    assert _cabi.supported(d)
    # the textbook smoother is a strategy of the builder vocabulary; it has no descriptor of its own (it is served
    # by solve_adaptive_save_every_step + stats.offgrid_marginals_searchsorted over the fixed-point kernel)
    smoother = ivpsolvers.solver_dynamic(ivpsolvers.strategy_smoother(ibm, ts1))
    assert smoother.strategy.name == "smoother"
    with pytest.raises(ValueError):
        ivpsolve._make_desc(field, nu, fact, smoother, 1e-3, 1e-3, ctrl, 0.01, 1, 2)
    mle = ivpsolvers.solver_mle(ivpsolvers.strategy_fixedpoint(ibm, ts1))
    d_mle = ivpsolve._make_desc(field, nu, fact, mle, 1e-3, 1e-3, ctrl, 0.01, 1, 2)
    assert d_mle.calibration == 2 and _cabi.supported(d_mle)
    with pytest.raises(ValueError):
        ivpsolve._make_desc(field, 3, fact, solver, 1e-3, 1e-3, ctrl, 0.01, 1, 2)


def test_ensemble_batching_shapes():
    from odecheckpts_b200.probdiffeq import ivpsolve

    B = 7
    inits = (np.linspace(1, 2, B)[:, None], np.zeros(1))
    use_torch, Bn, batched, u0, par, tol, scale = ivpsolve._stack_members(
        inits, (np.linspace(10, 20, B),), np.array([1e-6, 1e-3]), np.full(B, 2.0), 1
    )
    assert Bn == B and batched and u0.shape == (B, 2, 1) and par.shape == (B, 1) and tol.shape == (B, 2) and scale.shape == (B,)
    np.testing.assert_array_equal(u0[:, 1, 0], 0.0)
    with pytest.raises(ValueError):
        ivpsolve._stack_members((np.zeros((3, 1)), np.zeros((4, 1))), (1.0,), None, 1.0, 1)


def test_no_gpu_means_loud_failure_not_a_fallback():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from odecheckpts_b200 import _cabi, ivps, ivpsolvers

    vf, u0, tspan, args = ivps.logistic()
    solve = ivpsolvers.solve("ts0-2", vf, u0[0], save_at=np.linspace(*tspan, num=5), dt0=0.1, atol=1e-3, rtol=1e-3)
    with pytest.raises(_cabi.SolverError):
        solve(u0, args)


def test_bench_reads_its_roofline_side_inputs_from_the_committed_ncu_summary():
    """bench.py takes the DRAM traffic and the instruction-fetch bound of the headline kernel from the newest
    committed `ncu --set full` summary under profiles/ (no hard-coded constants): both must parse."""
    import importlib.util
    import os

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("pn_bench_module", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    traffic, src = bench.ncu_dram_bytes()
    assert traffic is not None and 1e8 < traffic < 1e11 and src.startswith("profiles")
    fetch = bench.ncu_instruction_fetch()
    assert fetch is not None and 0.5 < fetch["frac"] <= 1.0
    assert 0.05 < fetch["lines_refetched_per_instruction_line"] < 0.5


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    """`bench.py --impl reference` (the C port of the reference algorithm on the host cores) needs no GPU: exactly one
    JSON line with the driver's keys, e2e equal to the line's own value and zero copy bytes."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--members", "64"], capture_output=True, text=True, env=env, timeout=600)  # fmt: skip
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.split("\n") if l.strip()]
    assert len(lines) == 1, lines
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "ivp_solves_per_s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # a rank other than 0 under torchrun exits without work and without output
    env.update(RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, timeout=600)  # fmt: skip
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_dumps_the_last_step_outputs(tmp_path, oracle):
    """`--dump-outputs DIR` writes the results of the last timed step as float64 .npy files: the oracle's results for
    the seeded members it names."""
    import subprocess
    import sys

    import bench

    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
                        "--members", "16", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, env=env,
                       timeout=600)  # fmt: skip
    assert r.returncode == 0, r.stderr[-2000:]
    keys = ("u", "u_std", "n_accepted", "n_rejected", "status")
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(["members.npy"] + [f"nu4_{k}.npy" for k in keys])
    got = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert all(x.dtype == np.float64 for x in got.values())
    members = got["members"].astype(np.int64)
    assert len(members) > 0 and np.array_equal(members, members[0] + np.arange(len(members)))
    u0, par = bench.ensemble_inputs(int(members[0]), len(members))
    cfg = oracle.make_config("van_der_pol", 1, 4, 2, factorisation="dense", correction="ts1", strategy="fixedpoint",
                             calibration="dynamic", atol=1e-6, rtol=1e-6, dt0=0.01, num_params=1)  # fmt: skip
    want = oracle.solve_save_at_batch(cfg, u0, par, np.linspace(0.0, 6.3, 50))
    for k in keys:
        assert np.array_equal(got[f"nu4_{k}"], want[k].astype(np.float64)), k


def test_bench_rejects_zero_steps():
    import subprocess
    import sys

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=600)  # fmt: skip
    assert r.returncode != 0 and "--steps" in r.stderr
