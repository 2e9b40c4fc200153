"""GPU parity tests (run on a B200 with -m gpu): CUDA path through the C ABI vs the CPU oracle.

Thread-per-IVP kernels follow the oracle's operation order with explicit FMAs, so means,
standard deviations and accepted/rejected counts are compared BIT FOR BIT (rtol = 0), far
inside the 1e-9 relative tolerance BASELINE.json's north_star states for fp64.
"""

import ctypes as C

import numpy as np
import pytest

import problems_util as pu

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cabi():
    import torch

    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from odecheckpts_b200 import _cabi

    _cabi.lib()
    return _cabi


def _desc(cabi, problem, d, nu, q, B, K, *, fact="isotropic", corr="ts0", strat="fixedpoint", calib="dynamic",
          atol=1e-6, rtol=1e-6, dt0=0.01, P=0, flags=0, cap=0, max_attempts=0):  # fmt: skip
    return cabi.Desc(cabi.PROBLEM_IDS[problem], d, nu, q, cabi.FACTORISATIONS[fact], cabi.CORRECTIONS[corr],
                     cabi.STRATEGIES[strat], cabi.CALIBRATIONS[calib], atol, rtol, dt0, 0.95, 0.2, 10.0, 0.3, 0.4,
                     B, K, max_attempts, P, flags, cap)  # fmt: skip


def _ocfg(oracle, problem, d, nu, q, **kw):
    m = dict(fact="factorisation", corr="correction", strat="strategy", calib="calibration", P="num_params")
    kw = {k: v for k, v in kw.items() if k not in ("flags", "cap")}
    kw2 = {m.get(k, k): v for k, v in kw.items()}
    return oracle.make_config(problem, d, nu, q, **kw2)


def _assert_bitwise(gpu, ora, keys=("u", "u_std", "n_accepted", "n_rejected", "status")):
    for k in keys:
        a, b = np.asarray(gpu[k]), np.asarray(ora[k])
        assert a.shape == b.shape, k
        same = (a == b) | (np.isnan(a.astype(float)) & np.isnan(b.astype(float)))
        if not same.all():
            bad = np.argwhere(~same)[0]
            raise AssertionError(f"{k}: first mismatch at {tuple(bad)}: gpu={a[tuple(bad)]!r} oracle={b[tuple(bad)]!r}; "
                                 f"{(~same).sum()} of {same.size} differ")  # fmt: skip


CASES = [
    # problem, d, nu, q, P, params, u0 fn, save_at, kwargs
    ("logistic", 1, 2, 1, 2, (1.0, 1.0), lambda: np.array([[0.1]]), np.linspace(0, 2.5, 5), dict(atol=1e-3, rtol=1e-3, dt0=0.1)),
    ("logistic", 1, 4, 1, 2, (1.0, 1.0), lambda: np.array([[0.1]]), np.linspace(0, 2.5, 5), dict(atol=1e-6, rtol=1e-6, dt0=0.1)),
    ("logistic", 1, 3, 1, 2, (1.0, 1.0), lambda: np.array([[0.1]]), np.linspace(0, 2.5, 7), dict(atol=1e-5, rtol=1e-5, dt0=0.1, fact="dense", corr="ts1")),
    ("van_der_pol", 1, 4, 2, 1, (1e3,), pu.van_der_pol_u0, np.linspace(0, 6.3, 50), dict(atol=1e-3, rtol=1e-3, fact="dense", corr="ts1")),
    ("van_der_pol", 1, 4, 2, 1, (1e3,), pu.van_der_pol_u0, np.linspace(0, 6.3, 50), dict(atol=1e-6, rtol=1e-6, fact="dense", corr="ts1")),
    ("van_der_pol", 1, 3, 2, 1, (1e1,), pu.van_der_pol_u0, np.linspace(0, 6.3, 20), dict(atol=1e-5, rtol=1e-5, fact="dense", corr="ts0")),
    ("van_der_pol", 1, 5, 2, 1, (1e2,), pu.van_der_pol_u0, np.linspace(0, 6.3, 20), dict(atol=1e-7, rtol=1e-7, fact="isotropic", corr="ts0")),
    ("van_der_pol", 1, 2, 2, 1, (1e1,), pu.van_der_pol_u0, np.linspace(0, 6.3, 20), dict(atol=1e-4, rtol=1e-4, fact="dense", corr="ts1", calib="none")),
    ("rigid_body", 3, 2, 1, 3, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0, np.linspace(0, 50, 5), dict(atol=1e-7, rtol=1e-4, dt0=50.0)),
    ("rigid_body", 3, 4, 1, 3, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0, np.linspace(0, 50, 5), dict(atol=1e-9, rtol=1e-6, dt0=50.0)),
    ("three_body", 2, 4, 2, 1, (pu.THREE_BODY_MU,), pu.three_body_u0, np.linspace(0, pu.THREE_BODY_T, 50), dict(atol=1e-7, rtol=1e-7, calib="none")),
    ("three_body", 2, 3, 2, 1, (pu.THREE_BODY_MU,), pu.three_body_u0, np.linspace(0, pu.THREE_BODY_T, 50), dict(atol=1e-5, rtol=1e-5)),
    ("lotka_volterra", 2, 4, 1, 4, (0.5, 0.05, 0.5, 0.05), lambda: np.array([[20.0, 20.0]]), np.linspace(0, 20, 30), dict(atol=1e-6, rtol=1e-6, dt0=0.1)),
]


@pytest.mark.parametrize("strat", ["fixedpoint", "filter"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}-nu{c[2]}-{c[8].get('fact', 'isotropic')}-{c[8].get('corr', 'ts0')}")
def test_single_ivp_bitwise_vs_oracle(cabi, oracle, case, strat):
    problem, d, nu, q, P, params, u0fn, save_at, kw = case
    kw = dict(kw, strat=strat, P=P)
    u0 = u0fn()
    K = len(save_at)
    desc = _desc(cabi, problem, d, nu, q, 1, K, **kw)
    gpu = cabi.solve_host(desc, u0[None], np.asarray([params]), None, save_at, None, full=True)
    ora = oracle.solve_save_at(_ocfg(oracle, problem, d, nu, q, **kw), u0, params, save_at, full=True)
    assert ora["status"] == 0 and int(ora["n_accepted"][-1]) > 10
    g1 = {k: v[0] for k, v in gpu.items()}
    _assert_bitwise(g1, ora)
    np.testing.assert_array_equal(g1["marg_mean"].reshape(K, -1), ora["marg_mean"].reshape(K, -1))
    np.testing.assert_array_equal(g1["marg_chol"].reshape(K, -1), ora["marg_chol"].reshape(K, -1))


def test_vdp_ensemble_bitwise_and_within_tolerance(cabi, oracle):
    # BASELINE config 2 in miniature: randomised initial conditions (SURVEY 8d, C2), seed 0
    rng = np.random.default_rng(0)
    B, K = 96, 50
    u0 = np.stack([2.0 + 0.5 * rng.uniform(-1, 1, B), 0.5 * rng.uniform(-1, 1, B)], 1).reshape(B, 2, 1)
    params = np.full((B, 1), 1e3)
    save_at = np.linspace(0, 6.3, K)
    kw = dict(atol=1e-6, rtol=1e-6, fact="dense", corr="ts1", P=1)
    gpu = cabi.solve_host(_desc(cabi, "van_der_pol", 1, 4, 2, B, K, **kw), u0, params, None, save_at, None)
    ora = oracle.solve_save_at_batch(_ocfg(oracle, "van_der_pol", 1, 4, 2, **kw), u0, params, save_at)
    assert (ora["status"] == 0).all()
    # north_star tolerance (1e-9 relative) first, then the stronger bit-for-bit statement
    np.testing.assert_allclose(gpu["u"], ora["u"], rtol=1e-9, atol=0)
    np.testing.assert_allclose(gpu["u_std"], ora["u_std"], rtol=1e-9, atol=0)
    _assert_bitwise(gpu, ora)
    assert gpu["n_accepted"][:, -1].min() > 10000


def test_tolerance_sweep_ensemble_per_member_tol(cabi, oracle):
    # BASELINE config 3 in miniature: rigid body, 8 tolerances x ICs in ONE launch (SURVEY 8d, C3)
    rng = np.random.default_rng(1)
    n_ic, tols = 6, 10.0 ** -np.arange(3, 9)
    u0 = (np.array([1.0, 0.0, 0.9]) + 0.05 * rng.standard_normal((n_ic, 3)))
    u0 = np.repeat(u0[:, None, :], len(tols), 0).reshape(-1, 1, 3)
    t = np.tile(tols * 100, n_ic)
    tol = np.stack([1e-3 * t, t], 1)  # run_simple.py:40-42
    B, K = len(u0), 5
    params = np.tile(np.asarray(pu.RIGID_BODY_PARAMS), (B, 1))
    save_at = np.linspace(0, 50, K)
    for nu in (2, 4):
        kw = dict(dt0=50.0, P=3)
        gpu = cabi.solve_host(_desc(cabi, "rigid_body", 3, nu, 1, B, K, **kw), u0, params, tol, save_at, None)
        ora = oracle.solve_save_at_batch(_ocfg(oracle, "rigid_body", 3, nu, 1, **kw), u0, params, save_at, tol=tol)
        _assert_bitwise(gpu, ora)


def test_three_body_golden_counts_on_gpu(cabi, goldens):
    # experiments/5_vs_interpolation/measure.py:44-68,191-192
    tols = goldens["threebody_tols"]
    B, K = len(tols), 50
    u0 = np.tile(pu.three_body_u0()[None], (B, 1, 1))
    tol = np.stack([tols, tols], 1)
    desc = _desc(cabi, "three_body", 2, 4, 2, B, K, calib="none", P=1)
    gpu = cabi.solve_host(desc, u0, np.full((B, 1), pu.THREE_BODY_MU), tol, np.linspace(0, pu.THREE_BODY_T, K), None)
    np.testing.assert_array_equal(gpu["n_accepted"][:, -1], goldens["threebody_num_steps"])


def test_vdp_save_every_step_matches_golden_prefix_and_oracle(cabi, oracle, goldens):
    # experiments/1_van_der_pol/vdp.py:61-80
    kw = dict(atol=1e-3, rtol=1e-3, fact="dense", corr="ts1", strat="filter", P=1)
    cap = 8192
    desc = _desc(cabi, "van_der_pol", 1, 4, 2, 1, 2, flags=cabi.FLAG_RECORD, cap=cap, **kw)
    gpu = cabi.solve_host(desc, pu.van_der_pol_u0()[None], np.array([[1e3]]), None, np.array([0.0, 6.3]), None)
    n = int(gpu["traj_len"][0])
    t, u = gpu["traj_t"][:n, 0], gpu["traj_u"][:n, 0, 0]
    ora = oracle.solve_save_every_step(_ocfg(oracle, "van_der_pol", 1, 4, 2, **kw), pu.van_der_pol_u0(), [1e3], 0.0, 6.3)
    np.testing.assert_array_equal(t, ora["t"])
    np.testing.assert_array_equal(u, ora["u"][:, 0])
    np.testing.assert_array_equal(gpu["traj_std"][:n, 0], ora["u_std"][:, 0])
    grid, sol = goldens["vdp_grid"], goldens["vdp_solution"][:, 0]
    np.testing.assert_allclose(t[:26], grid[:26], rtol=0, atol=2e-14)
    np.testing.assert_allclose(u[:26], sol[:26], rtol=0, atol=2e-14)
    assert abs((n - 1) - (len(grid) - 1)) <= 0.01 * (len(grid) - 1)


def test_vdp_fixed_grid_replay_of_the_golden_grid(cabi, oracle, goldens):
    # vdp.py:88-91: solve_fixed_grid on the adaptive grid
    grid, sol = goldens["vdp_grid"], goldens["vdp_solution"][:, 0]
    kw = dict(atol=1e-3, rtol=1e-3, fact="dense", corr="ts1", strat="filter", P=1)
    desc = _desc(cabi, "van_der_pol", 1, 4, 2, 1, len(grid), flags=cabi.FLAG_FIXED_GRID, **kw)
    gpu = cabi.solve_host(desc, pu.van_der_pol_u0()[None], np.array([[1e3]]), None, grid, None)
    ora = oracle.solve_fixed_grid(_ocfg(oracle, "van_der_pol", 1, 4, 2, **kw), pu.van_der_pol_u0(), [1e3], grid)
    np.testing.assert_array_equal(gpu["u"][0], ora["u"])
    rel = np.abs(gpu["u"][0, :, 0] - sol) / np.abs(sol)
    assert np.median(rel) < 1e-9


def test_status_words_and_batch_survival(cabi, oracle):
    # one member hits max_attempts, the rest finish: failure is per member (SURVEY 8b)
    B, K = 4, 10
    u0 = np.tile(pu.van_der_pol_u0()[None], (B, 1, 1))
    params = np.array([[1e1], [1e3], [1e1], [1e1]])
    kw = dict(atol=1e-6, rtol=1e-6, fact="dense", corr="ts1", P=1, max_attempts=3000)
    save_at = np.linspace(0, 6.3, K)
    gpu = cabi.solve_host(_desc(cabi, "van_der_pol", 1, 4, 2, B, K, **kw), u0, params, None, save_at, None)
    ora = oracle.solve_save_at_batch(_ocfg(oracle, "van_der_pol", 1, 4, 2, **kw), u0, params, save_at)
    assert list(gpu["status"]) == [0, 2, 0, 0] == list(ora["status"])
    assert np.isnan(gpu["u"][1]).all() and np.isfinite(gpu["u"][[0, 2, 3]]).all()
    _assert_bitwise(gpu, ora, keys=("u", "u_std", "n_rejected", "status"))


def test_many_checkpoints_inside_one_step(cabi, oracle):
    # several checkpoints fall inside a single accepted step (SURVEY A.5, unpinned by the reference)
    K = 400
    save_at = np.linspace(0, 2.5, K)
    kw = dict(atol=1e-3, rtol=1e-3, dt0=0.1, P=2)
    for strat in ("fixedpoint", "filter"):
        gpu = cabi.solve_host(_desc(cabi, "logistic", 1, 4, 1, 1, K, strat=strat, **kw), np.array([[[0.1]]]), np.array([[1.0, 1.0]]), None, save_at, None)
        ora = oracle.solve_save_at(_ocfg(oracle, "logistic", 1, 4, 1, strat=strat, **kw), np.array([[0.1]]), (1.0, 1.0), save_at)
        assert int(ora["n_accepted"][-1]) < K / 4
        _assert_bitwise({k: v[0] for k, v in gpu.items()}, ora)
        np.testing.assert_allclose(gpu["u"][0, :, 0], pu.logistic_exact(save_at), atol=3e-2)


def test_device_pointer_entry_and_public_api(cabi, oracle):
    import torch

    from odecheckpts_b200 import ivps, ivpsolvers

    vf, u0, tspan, args = ivps.logistic()
    save_at = np.linspace(*tspan, num=5)
    solve = ivpsolvers.solve("ts0-4", vf, u0[0], save_at=save_at, dt0=0.1, atol=1e-3, rtol=1e-3)
    # host path (numpy)
    sol_h, aux = solve(u0, args)
    assert "u0_solve" in aux and sol_h.shape == (5, 1)
    np.testing.assert_allclose(sol_h[:, 0], pu.logistic_exact(save_at), atol=np.sqrt(1e-3), rtol=np.sqrt(1e-3))
    # device path (torch CUDA tensors in -> torch CUDA tensors out), batched
    B = 33
    u0_b = torch.linspace(0.05, 0.5, B, dtype=torch.float64, device="cuda")[:, None]
    sol_d, _ = solve((u0_b,), args)
    assert sol_d.is_cuda and tuple(sol_d.shape) == (B, 5, 1)
    ora = oracle.solve_save_at_batch(
        oracle.make_config("logistic", 1, 4, 1, atol=1e-3, rtol=1e-3, dt0=0.1, num_params=2),
        u0_b.cpu().numpy().reshape(B, 1, 1), np.tile([1.0, 1.0], (B, 1)), save_at)  # fmt: skip
    np.testing.assert_array_equal(sol_d.cpu().numpy(), ora["u"])
    with pytest.raises(ValueError, match="Tuple expected."):
        solve(u0[0], args)


# ---- lane-per-dimension kernels (blockdiag, and isotropic for d = 14) ------------------------------
GROUP_CASES = [
    # problem, d, nu, q, P, params, u0 fn, save_at, group, kwargs
    ("pleiades", 14, 3, 2, 0, (), pu.pleiades_u0, np.linspace(0, 3, 50), 16, dict(atol=1e-7, rtol=1e-4, dt0=0.1, fact="isotropic")),
    ("pleiades", 14, 5, 2, 0, (), pu.pleiades_u0, np.linspace(0, 3, 50), 16, dict(atol=1e-9, rtol=1e-6, dt0=0.1, fact="isotropic")),
    ("pleiades", 14, 3, 2, 0, (), pu.pleiades_u0, np.linspace(0, 3, 50), 16, dict(atol=1e-7, rtol=1e-4, dt0=0.1, fact="blockdiag")),
    ("pleiades", 14, 4, 2, 0, (), pu.pleiades_u0, np.linspace(0, 3, 50), 16, dict(atol=1e-8, rtol=1e-5, dt0=0.1, fact="blockdiag")),
    ("pleiades", 14, 5, 2, 0, (), pu.pleiades_u0, np.linspace(0, 3, 50), 16, dict(atol=1e-9, rtol=1e-6, dt0=0.1, fact="blockdiag", calib="none")),
    ("pleiades", 14, 8, 2, 0, (), pu.pleiades_u0, np.linspace(0, 3, 20), 16, dict(atol=1e-10, rtol=1e-7, dt0=0.1, fact="blockdiag")),
    ("pleiades", 14, 3, 2, 0, (), pu.pleiades_u0, np.linspace(0, 3, 20), 16, dict(atol=1e-7, rtol=1e-4, dt0=0.1, fact="isotropic", strat="filter")),
    ("pleiades", 14, 5, 2, 0, (), pu.pleiades_u0, np.linspace(0, 3, 20), 16, dict(atol=1e-9, rtol=1e-6, dt0=0.1, fact="isotropic", strat="filter")),
    ("rigid_body", 3, 4, 1, 3, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0, np.linspace(0, 50, 5), 4, dict(atol=1e-9, rtol=1e-6, dt0=50.0, fact="blockdiag")),
    ("three_body", 2, 4, 2, 1, (pu.THREE_BODY_MU,), pu.three_body_u0, np.linspace(0, pu.THREE_BODY_T, 50), 2, dict(atol=1e-7, rtol=1e-7, fact="blockdiag")),
    ("lotka_volterra", 2, 4, 1, 4, (0.5, 0.05, 0.5, 0.05), lambda: np.array([[20.0, 20.0]]), np.linspace(0, 20, 30), 2, dict(atol=1e-6, rtol=1e-6, dt0=0.1, fact="blockdiag")),
]


@pytest.mark.parametrize("case", GROUP_CASES, ids=lambda c: f"{c[0]}-nu{c[2]}-{c[9]['fact']}-{c[9].get('strat', 'fixedpoint')}")
def test_lane_per_dimension_kernels_bitwise_vs_oracle(cabi, oracle, case):
    problem, d, nu, q, P, params, u0fn, save_at, group, kw = case
    kw = dict(kw, P=P)
    u0 = u0fn()
    K = len(save_at)
    B = 5  # members share a warp with others: perturb the initial values
    rng = np.random.default_rng(7)
    u0_b = u0[None] * (1.0 + 1e-3 * rng.standard_normal((B,) + u0.shape))
    u0_b[0] = u0
    par_b = np.tile(np.asarray(params, dtype=float), (B, 1)) if P else None
    desc = _desc(cabi, problem, d, nu, q, B, K, **kw)
    gpu = cabi.solve_host(desc, u0_b, par_b, None, save_at, None, full=True)
    ocfg = _ocfg(oracle, problem, d, nu, q, reduction_group=group, **kw)
    for b in range(B):
        ora = oracle.solve_save_at(ocfg, u0_b[b], params, save_at, full=True)
        assert ora["status"] == 0
        _assert_bitwise({k: v[b] for k, v in gpu.items()}, ora)
        np.testing.assert_array_equal(gpu["marg_mean"][b].reshape(K, -1), ora["marg_mean"].reshape(K, -1))
        np.testing.assert_array_equal(gpu["marg_chol"][b].reshape(K, -1), ora["marg_chol"].reshape(K, -1))


def test_pleiades_golden_checkpoint_rmse_on_gpu(cabi, oracle, goldens):
    # experiments/3_workprec_harder/run_harder.py:42-60 (isotropic EKF0, ode_order=2, 50 checkpoints)
    import scipy.integrate

    xs = goldens["pleiades_checkpoints"]
    y0 = pu.pleiades_u0()

    def f(t, y):
        return np.concatenate([y[14:], oracle.vf("pleiades", y.reshape(2, -1), [])])

    ref = scipy.integrate.solve_ivp(f, (xs[0], xs[-1]), y0.ravel(), t_eval=xs, method="DOP853", atol=1e-13, rtol=1e-13).y.T[:, :14]
    for nu, key in [(3, "pleiades_nu3"), (5, "pleiades_nu5")]:
        tols = goldens[key + "_list_of_args"][:5] * 10  # run_harder.py:45-47
        B = len(tols)
        tol = np.stack([1e-3 * tols, tols], 1)
        desc = _desc(cabi, "pleiades", 14, nu, 2, B, len(xs), dt0=0.1)
        gpu = cabi.solve_host(desc, np.tile(y0[None], (B, 1, 1)), None, tol, xs, None)
        assert (gpu["status"] == 0).all()
        rmse = np.linalg.norm((gpu["u"] - ref[None]).reshape(B, -1), axis=1) / np.sqrt(ref.size)
        np.testing.assert_allclose(rmse, goldens[key + "_precision"][:5], rtol=1e-3)


# experiments/4_brusselator/run.py:51-61,119-138 on the GPU: golden step counts + checkpoint means
@pytest.mark.parametrize("N,exact", [(2, False), (4, True), (8, True), (16, True)])
def test_brusselator_goldens_on_gpu(cabi, oracle, goldens, N, exact):
    d, K = 2 * N, 200
    save_at = np.linspace(0.0, 10.0, K)
    u0 = pu.brusselator_u0(N)
    kw = dict(atol=1e-8, rtol=1e-8, dt0=0.01, P=1)
    gpu = cabi.solve_host(_desc(cabi, "brusselator", d, 4, 1, 1, K, **kw), u0[None], np.array([[1.0 / 50.0]]), None, save_at, None)
    ora = oracle.solve_save_at(_ocfg(oracle, "brusselator", d, 4, 1, reduction_group=d, **kw), u0, [1.0 / 50.0], save_at)
    _assert_bitwise({k: v[0] for k, v in gpu.items()}, ora)
    idx = list(goldens["brusselator_N"]).index(N)
    want = int(goldens["brusselator_num_steps_checkpoint"][idx])
    got = int(gpu["n_accepted"][0, -1])
    if exact:
        assert got == want
        np.testing.assert_allclose(gpu["u"][0], goldens[f"brusselator_ys_N{N}"], rtol=0, atol=5e-9 if N == 8 else 1e-9)
    else:
        assert abs(got - want) <= max(3, 0.02 * want) or N == 2  # N=2 starts in steady state (degenerate)


def test_brusselator_ensemble_over_diffusion_parameter(cabi, oracle):
    # BASELINE config 5 in miniature: ensemble over alpha (seed 3, SURVEY 8d C5)
    rng = np.random.default_rng(3)
    N, B, K = 4, 12, 40
    alpha = (1.0 / 50.0) * 10.0 ** rng.uniform(-0.5, 0.5, B)
    u0 = np.tile(pu.brusselator_u0(N)[None], (B, 1, 1))
    save_at = np.linspace(0.0, 10.0, K)
    kw = dict(atol=1e-8, rtol=1e-8, dt0=0.01, P=1)
    gpu = cabi.solve_host(_desc(cabi, "brusselator", 2 * N, 4, 1, B, K, **kw), u0, alpha[:, None], None, save_at, None)
    ora = oracle.solve_save_at_batch(_ocfg(oracle, "brusselator", 2 * N, 4, 1, reduction_group=2 * N, **kw), u0, alpha[:, None], save_at)
    _assert_bitwise(gpu, ora)
    assert len(set(gpu["n_accepted"][:, -1].tolist())) > 4  # members really differ


# ---- dense factorisation with d > 1 (register columns; D = 40: D x D factors in shared memory) -----
DENSE_CASES = [
    ("rigid_body", 3, 2, 1, 3, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0, np.linspace(0, 50, 5), dict(atol=1e-7, rtol=1e-4, dt0=50.0, corr="ts1")),
    ("rigid_body", 3, 4, 1, 3, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0, np.linspace(0, 50, 5), dict(atol=1e-9, rtol=1e-6, dt0=50.0, corr="ts1")),
    ("rigid_body", 3, 4, 1, 3, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0, np.linspace(0, 50, 5), dict(atol=1e-9, rtol=1e-6, dt0=50.0, corr="ts0", calib="none")),
    ("lotka_volterra", 2, 4, 1, 4, (0.5, 0.05, 0.5, 0.05), lambda: np.array([[20.0, 20.0]]), np.linspace(0, 20, 30), dict(atol=1e-6, rtol=1e-6, dt0=0.1, corr="ts1")),
    ("three_body", 2, 4, 2, 1, (pu.THREE_BODY_MU,), pu.three_body_u0, np.linspace(0, pu.THREE_BODY_T, 20), dict(atol=1e-6, rtol=1e-6, corr="ts0")),
    ("brusselator", 4, 4, 1, 1, (0.02,), lambda: pu.brusselator_u0(2), np.linspace(0, 10, 40), dict(atol=1e-6, rtol=1e-6, corr="ts1")),
    ("brusselator", 8, 4, 1, 1, (0.02,), lambda: pu.brusselator_u0(4), np.linspace(0, 10, 20), dict(atol=1e-5, rtol=1e-5, corr="ts1")),
]


@pytest.mark.parametrize("case", DENSE_CASES, ids=lambda c: f"{c[0]}-d{c[1]}-nu{c[2]}-{c[8]['corr']}")
def test_dense_factorisation_bitwise_vs_oracle(cabi, oracle, case):
    problem, d, nu, q, P, params, u0fn, save_at, kw = case
    kw = dict(kw, P=P, fact="dense")
    u0 = u0fn()
    K = len(save_at)
    B = 3
    rng = np.random.default_rng(11)
    u0_b = u0[None] * (1.0 + 1e-3 * rng.standard_normal((B,) + u0.shape))
    u0_b[0] = u0
    par_b = np.tile(np.asarray(params, dtype=float), (B, 1))
    gpu = cabi.solve_host(_desc(cabi, problem, d, nu, q, B, K, **kw), u0_b, par_b, None, save_at, None, full=True)
    ocfg = _ocfg(oracle, problem, d, nu, q, **kw)
    for b in range(B):
        ora = oracle.solve_save_at(ocfg, u0_b[b], params, save_at, full=True)
        assert ora["status"] == 0 and int(ora["n_accepted"][-1]) >= 10
        _assert_bitwise({k: v[b] for k, v in gpu.items()}, ora)
        np.testing.assert_array_equal(gpu["marg_mean"][b].reshape(K, -1), ora["marg_mean"].reshape(K, -1))
        np.testing.assert_array_equal(gpu["marg_chol"][b].reshape(K, -1), ora["marg_chol"].reshape(K, -1))


def test_dense_filter_strategy_and_ekf0_vs_ekf1_accuracy(cabi, oracle):
    # BASELINE config 3's comparison in miniature: isotropic EKF0 vs dense EKF1 on the rigid body
    import scipy.integrate

    save_at = np.linspace(0, 50, 5)
    u0 = pu.rigid_body_u0()
    f = lambda t, y: oracle.vf("rigid_body", y.reshape(1, -1), pu.RIGID_BODY_PARAMS)  # noqa: E731
    ref = scipy.integrate.solve_ivp(f, (0, 50), u0[0], t_eval=save_at, method="DOP853", atol=1e-13, rtol=1e-13).y.T
    par = np.asarray([pu.RIGID_BODY_PARAMS])
    kw = dict(atol=1e-9, rtol=1e-6, dt0=50.0, P=3)
    filt = cabi.solve_host(_desc(cabi, "rigid_body", 3, 4, 1, 1, 5, fact="dense", corr="ts1", strat="filter", **kw), u0[None], par, None, save_at, None)
    ora = oracle.solve_save_at(_ocfg(oracle, "rigid_body", 3, 4, 1, fact="dense", corr="ts1", strat="filter", **kw), u0, pu.RIGID_BODY_PARAMS, save_at)
    _assert_bitwise({k: v[0] for k, v in filt.items()}, ora)
    ekf1 = cabi.solve_host(_desc(cabi, "rigid_body", 3, 4, 1, 1, 5, fact="dense", corr="ts1", **kw), u0[None], par, None, save_at, None)
    ekf0 = cabi.solve_host(_desc(cabi, "rigid_body", 3, 4, 1, 1, 5, fact="isotropic", corr="ts0", **kw), u0[None], par, None, save_at, None)
    for sol in (ekf0, ekf1):
        assert np.abs(sol["u"][0] - ref).max() < 1e-4


# ---- CTA-per-IVP wide kernel: Brusselator with a runtime grid size (d = 2N) -----------------------
@pytest.mark.parametrize("N,K,tol", [(20, 40, 1e-6), (32, 200, 1e-8), (100, 12, 1e-5)])
def test_wide_brusselator_bitwise_vs_oracle(cabi, oracle, goldens, N, K, tol):
    d = 2 * N
    save_at = np.linspace(0.0, 10.0, K)
    u0 = pu.brusselator_u0(N)
    B = 3
    alpha = np.array([1.0 / 50.0, 0.03, 0.012])
    kw = dict(atol=tol, rtol=tol, dt0=0.01, P=1)
    gpu = cabi.solve_host(_desc(cabi, "brusselator", d, 4, 1, B, K, **kw), np.tile(u0[None], (B, 1, 1)), alpha[:, None], None, save_at, None, full=True)
    ocfg = _ocfg(oracle, "brusselator", d, 4, 1, reduction_group=128, **kw)
    for b in range(B):
        ora = oracle.solve_save_at(ocfg, u0, [alpha[b]], save_at, full=True)
        assert ora["status"] == 0
        _assert_bitwise({k: v[b] for k, v in gpu.items()}, ora)
        np.testing.assert_array_equal(gpu["marg_mean"][b].reshape(K, -1), ora["marg_mean"].reshape(K, -1))
        np.testing.assert_array_equal(gpu["marg_chol"][b].reshape(K, -1), ora["marg_chol"].reshape(K, -1))
    if N == 32:
        # experiments/4_brusselator/run.py: N = 32 took 12,425 steps; ulp-chaotic at the 1 % level
        want = int(goldens["brusselator_num_steps_checkpoint"][list(goldens["brusselator_N"]).index(32)])
        assert abs(int(gpu["n_accepted"][0, -1]) - want) <= 0.02 * want
        np.testing.assert_allclose(gpu["u"][0], goldens["brusselator_ys_N32"], rtol=0, atol=5e-8)


def test_wide_brusselator_ensemble_beyond_one_member_per_sm(cabi, oracle):
    # up to 148 members the running member's mean arrays live in shared memory; beyond, in the per-member
    # global arrays (two CTAs per SM).  Same bits either way.
    N, B, K = 20, 200, 6
    rng = np.random.default_rng(5)
    alpha = (1.0 / 50.0) * 10.0 ** rng.uniform(-0.5, 0.5, B)
    u0 = np.tile(pu.brusselator_u0(N)[None], (B, 1, 1))
    save_at = np.linspace(0.0, 2.0, K)
    kw = dict(atol=1e-6, rtol=1e-6, dt0=0.01, P=1)
    many = cabi.solve_host(_desc(cabi, "brusselator", 2 * N, 4, 1, B, K, **kw), u0, alpha[:, None], None, save_at, None)
    few = cabi.solve_host(_desc(cabi, "brusselator", 2 * N, 4, 1, 100, K, **kw), u0[:100], alpha[:100, None], None, save_at, None)
    for key in ("u", "u_std", "n_accepted", "n_rejected", "status"):
        np.testing.assert_array_equal(many[key][:100], few[key])
    idx = [0, 99, 150, 199]
    ora = oracle.solve_save_at_batch(_ocfg(oracle, "brusselator", 2 * N, 4, 1, reduction_group=128, **kw), u0[idx], alpha[idx, None], save_at)
    _assert_bitwise({k: v[idx] for k, v in many.items()}, ora)


def test_wide_brusselator_one_warp_per_ivp_build_for_large_ensembles(cabi, oracle, monkeypatch):
    # from four members per SM on (592) the CTA-per-IVP family runs one WARP per IVP (the factor arithmetic every
    # thread replicates is then issued once, eight members fit an SM): same algorithm, norms summed by a 32-lane
    # butterfly (oracle reduction_group = 32)
    N, B, K = 24, 700, 5
    rng = np.random.default_rng(6)
    alpha = (1.0 / 50.0) * 10.0 ** rng.uniform(-0.5, 0.5, B)
    u0 = np.tile(pu.brusselator_u0(N)[None], (B, 1, 1))
    save_at = np.linspace(0.0, 1.0, K)
    kw = dict(atol=1e-6, rtol=1e-6, dt0=0.01, P=1)
    desc = _desc(cabi, "brusselator", 2 * N, 4, 1, B, K, **kw)
    assert cabi.kernel_info(desc)["threads_per_cta"] == 32
    got = cabi.solve_host(desc, u0, alpha[:, None], None, save_at, None)
    assert (got["status"] == 0).all()
    idx = [0, 1, 350, 699]
    ora = oracle.solve_save_at_batch(_ocfg(oracle, "brusselator", 2 * N, 4, 1, reduction_group=32, **kw), u0[idx], alpha[idx, None], save_at)
    _assert_bitwise({k: v[idx] for k, v in got.items()}, ora)
    # forcing it for a small ensemble gives the same numbers as the 128-thread build to rounding (different norm order)
    monkeypatch.setenv("PN_B200_WIDE_WARP", "1")
    small = cabi.solve_host(_desc(cabi, "brusselator", 2 * N, 4, 1, 4, K, **kw), u0[:4], alpha[:4, None], None, save_at, None)
    monkeypatch.setenv("PN_B200_WIDE_WARP", "0")
    ref = cabi.solve_host(_desc(cabi, "brusselator", 2 * N, 4, 1, 4, K, **kw), u0[:4], alpha[:4, None], None, save_at, None)
    np.testing.assert_allclose(small["u"], ref["u"], rtol=1e-9, atol=1e-12)


def test_wide_kernel_shared_memory_sizes_in_any_order(cabi):
    # one kernel, launched with different dynamic shared-memory sizes (2 d staging doubles + mean arrays):
    # large -> small -> large must work (the function attribute is only ever raised)
    save_at = np.linspace(0.0, 0.5, 4)
    kw = dict(atol=1e-5, rtol=1e-5, dt0=0.01, P=1)

    def run(N, B):
        u0 = np.tile(pu.brusselator_u0(N)[None], (B, 1, 1))
        return cabi.solve_host(_desc(cabi, "brusselator", 2 * N, 4, 1, B, 4, **kw), u0, np.full((B, 1), 0.02), None, save_at, None)

    first = run(100, 2)
    run(20, 2)
    run(20, 160)
    again = run(100, 2)
    assert (again["status"] == 0).all()
    np.testing.assert_array_equal(first["u"], again["u"])
    np.testing.assert_array_equal(first["n_accepted"], again["n_accepted"])


def test_wide_brusselator_terminal_values_and_filter(cabi, oracle):
    # solve_adaptive_terminal_values (run.py:82-90) = two checkpoints; also the filter strategy
    N = 24
    u0 = pu.brusselator_u0(N)
    for strat in ("fixedpoint", "filter"):
        kw = dict(atol=1e-6, rtol=1e-6, dt0=0.01, P=1, strat=strat)
        save_at = np.array([0.0, 2.0]) if strat == "fixedpoint" else np.linspace(0, 2.0, 9)
        K = len(save_at)
        gpu = cabi.solve_host(_desc(cabi, "brusselator", 2 * N, 4, 1, 1, K, **kw), u0[None], np.array([[0.02]]), None, save_at, None)
        ora = oracle.solve_save_at(_ocfg(oracle, "brusselator", 2 * N, 4, 1, reduction_group=128, **kw), u0, [0.02], save_at)
        _assert_bitwise({k: v[0] for k, v in gpu.items()}, ora)


@pytest.mark.parametrize("N", [64, 128, 256])
def test_wide_brusselator_reference_step_counts(cabi, goldens, N):
    # experiments/4_brusselator/run.py:119-138 (data_checkpoint.npy "num_steps"): 48,233 / 190,024 / 754,285
    K = 200
    desc = _desc(cabi, "brusselator", 2 * N, 4, 1, 1, K, atol=1e-8, rtol=1e-8, dt0=0.01, P=1)
    gpu = cabi.solve_host(desc, pu.brusselator_u0(N)[None], np.array([[1.0 / 50.0]]), None, np.linspace(0.0, 10.0, K), None)
    want = int(goldens["brusselator_num_steps_checkpoint"][list(goldens["brusselator_N"]).index(N)])
    assert int(gpu["status"][0]) == 0
    assert int(gpu["n_accepted"][0, -1]) == want


MORE_ORDER_CASES = [
    ("rigid_body", 3, 3, 1, 3, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0, np.linspace(0, 50, 5), 0, dict(atol=1e-8, rtol=1e-5, dt0=50.0)),
    ("rigid_body", 3, 5, 1, 3, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0, np.linspace(0, 50, 5), 0, dict(atol=1e-10, rtol=1e-7, dt0=50.0)),
    ("three_body", 2, 2, 2, 1, (pu.THREE_BODY_MU,), pu.three_body_u0, np.linspace(0, pu.THREE_BODY_T, 20), 0, dict(atol=1e-4, rtol=1e-4)),
    ("three_body", 2, 5, 2, 1, (pu.THREE_BODY_MU,), pu.three_body_u0, np.linspace(0, pu.THREE_BODY_T, 20), 0, dict(atol=1e-8, rtol=1e-8)),
    ("three_body", 2, 4, 2, 1, (pu.THREE_BODY_MU,), pu.three_body_u0, np.linspace(0, pu.THREE_BODY_T, 20), 0, dict(atol=1e-6, rtol=1e-6, fact="dense", corr="ts1")),
    ("lotka_volterra", 2, 3, 1, 4, (0.5, 0.05, 0.5, 0.05), lambda: np.array([[20.0, 20.0]]), np.linspace(0, 20, 30), 0, dict(atol=1e-5, rtol=1e-5, dt0=0.1)),
    ("logistic", 1, 5, 1, 2, (1.0, 1.0), lambda: np.array([[0.1]]), np.linspace(0, 2.5, 9), 0, dict(atol=1e-8, rtol=1e-8, dt0=0.1)),
    ("logistic", 1, 8, 1, 2, (1.0, 1.0), lambda: np.array([[0.1]]), np.linspace(0, 2.5, 9), 0, dict(atol=1e-9, rtol=1e-9, dt0=0.1)),
    ("pleiades", 14, 8, 2, 0, (), pu.pleiades_u0, np.linspace(0, 3, 50), 16, dict(atol=1e-6, rtol=1e-3, dt0=0.1)),
]


@pytest.mark.parametrize("case", MORE_ORDER_CASES, ids=lambda c: f"{c[0]}-nu{c[2]}-{c[9].get('fact', 'isotropic')}")
def test_more_prior_orders_bitwise_vs_oracle(cabi, oracle, case):
    problem, d, nu, q, P, params, u0fn, save_at, group, kw = case
    kw = dict(kw, P=P)
    u0 = u0fn()
    K = len(save_at)
    par = np.asarray([params], dtype=float) if P else None
    gpu = cabi.solve_host(_desc(cabi, problem, d, nu, q, 1, K, **kw), u0[None], par, None, save_at, None)
    ora = oracle.solve_save_at(_ocfg(oracle, problem, d, nu, q, reduction_group=group, **kw), u0, params, save_at)
    assert ora["status"] == 0
    _assert_bitwise({k: v[0] for k, v in gpu.items()}, ora)


def test_pleiades_prob8_golden_rmse_on_gpu(cabi, oracle, goldens):
    # Prob(8) of experiments/3_workprec_harder/run_harder.py:74-77, the three loosest tolerances
    import scipy.integrate

    xs = goldens["pleiades_checkpoints"]
    y0 = pu.pleiades_u0()
    f = lambda t, y: np.concatenate([y[14:], oracle.vf("pleiades", y.reshape(2, -1), [])])  # noqa: E731
    ref = scipy.integrate.solve_ivp(f, (xs[0], xs[-1]), y0.ravel(), t_eval=xs, method="DOP853", atol=1e-13, rtol=1e-13).y.T[:, :14]
    tols = goldens["pleiades_nu8_list_of_args"][:3] * 10
    B = len(tols)
    desc = _desc(cabi, "pleiades", 14, 8, 2, B, len(xs), dt0=0.1)
    gpu = cabi.solve_host(desc, np.tile(y0[None], (B, 1, 1)), None, np.stack([1e-3 * tols, tols], 1), xs, None)
    assert (gpu["status"] == 0).all()
    rmse = np.linalg.norm((gpu["u"] - ref[None]).reshape(B, -1), axis=1) / np.sqrt(ref.size)
    np.testing.assert_allclose(rmse, goldens["pleiades_nu8_precision"][:3], rtol=5e-3)


def test_single_attempted_step_parity(cabi, oracle):
    # SURVEY section 4, ladder item 1: one attempted step from the Taylor-initialised state, GPU vs
    # the oracle's single-step entry point: mean, factor (L L^T), via a 2-point fixed grid (always accepted)
    for problem, d, nu, q, params, u0, fact, corr, dt in [
        ("van_der_pol", 1, 4, 2, (1e3,), pu.van_der_pol_u0(), "dense", "ts1", 1e-4),
        ("rigid_body", 3, 4, 1, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0(), "isotropic", "ts0", 0.05),
        ("rigid_body", 3, 4, 1, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0(), "dense", "ts1", 0.05),
    ]:
        P = len(params)
        kw = dict(atol=1e-3, rtol=1e-3, dt0=dt, P=P, fact=fact, corr=corr, strat="filter")
        desc = _desc(cabi, problem, d, nu, q, 1, 2, flags=cabi.FLAG_FIXED_GRID, **kw)
        gpu = cabi.solve_host(desc, u0[None], np.asarray([params]), None, np.array([0.0, dt]), None, full=True)
        ocfg = _ocfg(oracle, problem, d, nu, q, **kw)
        m0 = oracle.taylor_init(problem, u0, nu, params)
        n = nu + 1
        dense = fact == "dense" and d > 1
        N = n * d if dense else n
        chol0 = np.zeros((1, N, N))
        step = oracle.attempt_step(ocfg, params, 0.0, dt, 1.0, 1.0, m0, chol0)
        np.testing.assert_array_equal(gpu["marg_mean"][0, 1].ravel(), step["mean"].ravel())
        np.testing.assert_array_equal(gpu["marg_chol"][0, 1].reshape(N, N), step["chol"][0])
        assert np.isfinite(step["error_norm"]) and step["dt_proposed"] > 0


SCALE_CASES = [
    # problem, d, nu, q, P, params, u0, save_at, oracle reduction_group, kwargs
    ("logistic", 1, 3, 1, 2, (1.0, 1.0), np.array([[0.1]]), np.linspace(0, 2.5, 7), 0, dict(atol=1e-5, rtol=1e-5, dt0=0.1)),
    ("van_der_pol", 1, 4, 2, 1, (1e3,), pu.van_der_pol_u0(), np.linspace(0, 6.3, 50), 0, dict(atol=1e-4, rtol=1e-4, fact="dense", corr="ts1")),
    ("van_der_pol", 1, 2, 2, 1, (1e1,), pu.van_der_pol_u0(), np.linspace(0, 6.3, 20), 0, dict(atol=1e-4, rtol=1e-4, fact="dense", corr="ts1", calib="none")),
    ("rigid_body", 3, 4, 1, 3, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0(), np.linspace(0, 50, 9), 4, dict(atol=1e-9, rtol=1e-6, dt0=50.0, fact="blockdiag")),
    ("pleiades", 14, 3, 2, 0, (), pu.pleiades_u0(), np.linspace(0, 3, 20), 16, dict(atol=1e-7, rtol=1e-4, dt0=0.1)),
    ("rigid_body", 3, 4, 1, 3, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0(), np.linspace(0, 50, 9), 0, dict(atol=1e-9, rtol=1e-6, dt0=50.0, fact="dense", corr="ts1")),
    ("rigid_body", 3, 4, 1, 3, pu.RIGID_BODY_PARAMS, pu.rigid_body_u0(), np.linspace(0, 50, 9), 0, dict(atol=1e-9, rtol=1e-6, dt0=50.0, fact="dense", corr="ts1", strat="filter")),
    ("brusselator", 64, 4, 1, 1, (0.02,), None, np.linspace(0, 2, 12), 128, dict(atol=1e-6, rtol=1e-6, dt0=0.01)),
]


@pytest.mark.parametrize("case", SCALE_CASES, ids=lambda c: f"{c[0]}-nu{c[2]}-{c[9].get('fact', 'isotropic')}-{c[9].get('strat', 'fixedpoint')}")
def test_output_scale_at_the_checkpoints_bitwise_vs_oracle(cabi, oracle, case):
    # solution.output_scale (SURVEY 8a, row a11): the calibrated scale of the accepted step that reached
    # or crossed each checkpoint; one per dimension for blockdiag
    problem, d, nu, q, P, params, u0, save_at, group, kw = case
    if u0 is None:
        N = d // 2
        u0 = np.concatenate([np.sin(2 * np.pi * np.linspace(0, 1, N)) + 1, 3 * np.ones(N)])[None]
    kw = dict(kw, P=P)
    K = len(save_at)
    par = np.asarray(params, dtype=float)[None] if P else None
    gpu = cabi.solve_host(_desc(cabi, problem, d, nu, q, 1, K, **kw), u0[None], par, None, save_at, None, full=True)
    ora = oracle.solve_save_at_lml(_ocfg(oracle, problem, d, nu, q, reduction_group=group, **kw), u0, params, save_at,
                                   np.zeros((K, d)), np.ones(K))  # fmt: skip
    assert ora["status"] == 0 and gpu["status"][0] == 0
    np.testing.assert_array_equal(gpu["u"][0], ora["u"])
    np.testing.assert_array_equal(gpu["output_scale"][0].reshape(K, -1), ora["output_scale"])
    assert gpu["output_scale"][0].reshape(K, -1)[0].tolist() == [1.0] * ora["output_scale"].shape[1]
    if kw.get("calib") == "none":
        assert (gpu["output_scale"] == 1.0).all()
    else:
        assert len(np.unique(gpu["output_scale"])) > K // 2


@pytest.mark.parametrize("N", [1024, 2048])
def test_wide_brusselator_largest_grids_bitwise_vs_oracle(cabi, oracle, N):
    # BASELINE config 5's largest grid (N = 1024, d = 2048) and the kernel's maximum (d = 4096), a short
    # interval so that the oracle finishes in seconds
    d, K = 2 * N, 3
    save_at = np.linspace(0.0, 0.002, K)
    u0 = pu.brusselator_u0(N)
    kw = dict(atol=1e-6, rtol=1e-6, dt0=1e-5, P=1)
    gpu = cabi.solve_host(_desc(cabi, "brusselator", d, 4, 1, 2, K, **kw), np.tile(u0[None], (2, 1, 1)), np.array([[0.02], [0.03]]), None, save_at, None)
    ocfg = _ocfg(oracle, "brusselator", d, 4, 1, reduction_group=128, **kw)
    for b, alpha in enumerate((0.02, 0.03)):
        ora = oracle.solve_save_at(ocfg, u0, [alpha], save_at)
        assert ora["status"] == 0 and ora["n_accepted"][-1] > 20
        _assert_bitwise({k: v[b] for k, v in gpu.items()}, ora)


def test_empty_ensemble_minimal_grid_and_unsupported_sizes(cabi, oracle):
    # B = 0: nothing to do, nothing written; K = 2 is the smallest grid; odd / oversized Brusselator
    # dimensions and K < 2 are refused with the reference-style exceptions
    save_at = np.array([0.0, 1.0])
    empty = cabi.solve_host(_desc(cabi, "logistic", 1, 2, 1, 0, 2, P=2), np.zeros((0, 1, 1)), np.zeros((0, 2)), None, save_at, None)
    assert empty["u"].shape == (0, 2, 1) and empty["status"].shape == (0,)
    one = cabi.solve_host(_desc(cabi, "logistic", 1, 2, 1, 1, 2, P=2, atol=1e-4, rtol=1e-4, dt0=0.1), np.array([[[0.1]]]), np.array([[1.0, 1.0]]), None, save_at, None)
    ora = oracle.solve_save_at(_ocfg(oracle, "logistic", 1, 2, 1, P=2, atol=1e-4, rtol=1e-4, dt0=0.1), np.array([[0.1]]), (1.0, 1.0), save_at)
    _assert_bitwise({k: v[0] for k, v in one.items()}, ora)
    with pytest.raises(NotImplementedError):
        cabi.solve_host(_desc(cabi, "brusselator", 4098, 4, 1, 1, 2, P=1), np.zeros((1, 1, 4098)), np.array([[0.02]]), None, save_at, None)
    with pytest.raises(NotImplementedError):
        cabi.solve_host(_desc(cabi, "brusselator", 101, 4, 1, 1, 2, P=1), np.zeros((1, 1, 101)), np.array([[0.02]]), None, save_at, None)
    with pytest.raises(ValueError):
        cabi.solve_host(_desc(cabi, "logistic", 1, 2, 1, 1, 1, P=2), np.array([[[0.1]]]), np.array([[1.0, 1.0]]), None, save_at[:1], None)
