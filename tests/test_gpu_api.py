"""GPU tests of the reference-facing Python API (the calls the reference's scripts and test make)."""

import numpy as np
import pytest

import problems_util as pu

pytestmark = pytest.mark.gpu


def test_reference_test_case_logistic_checkpoint_solver():
    # tests/test_ivpsolvers.py:31-52 of the reference, with the closed form in place of diffrax
    from odecheckpts_b200 import ivps, ivpsolvers

    vf, u0, time_span, args = ivps.logistic()
    dt0, atol, rtol = 0.1, 1e-3, 1e-3
    save_at = np.linspace(*time_span, num=5)
    for method in ("ts0-2", "ts0-4"):
        solve1 = ivpsolvers.solve(method, vf, u0[0], save_at, dt0=dt0, atol=atol, rtol=rtol)
        solution1, aux1 = solve1(u0, args)
        assert "u0_solve" in aux1.keys()
        assert np.allclose(solution1[:, 0], pu.logistic_exact(save_at), atol=np.sqrt(atol), rtol=np.sqrt(rtol))


def test_run_harder_style_pleiades_call():
    # experiments/3_workprec_harder/run_harder.py:42-60
    import scipy.integrate

    from odecheckpts_b200 import ivps, ivpsolvers

    vf_2nd, u0_2nd, (t0, t1) = ivps.pleiades_2nd()
    xs = np.linspace(t0, t1, num=50)
    tol = 1e-6 * 10
    fun = ivpsolvers.solve("ts0-5", vf_2nd, u0_2nd[0], save_at=xs, dt0=0.1, atol=1e-3 * tol, rtol=tol, ode_order=2)
    sol, aux = fun(u0_2nd, ())
    assert sol.shape == (50, 14)

    def f(t, y):
        return np.concatenate([y[14:], vf_2nd(y[:14], y[14:], t=t)])

    ref = scipy.integrate.solve_ivp(f, (t0, t1), np.concatenate(u0_2nd), t_eval=xs, method="DOP853", atol=1e-12, rtol=1e-12).y.T[:, :14]
    assert np.linalg.norm(sol - ref) / np.sqrt(ref.size) < 1e-6
    assert aux["solution"].num_steps[-1] > 500 and aux["solution"].status == 0


def test_brusselator_script_style_builder_calls():
    # experiments/4_brusselator/run.py:51-61,82-90,119-129 with the builder vocabulary
    from odecheckpts_b200 import ivps
    from odecheckpts_b200.probdiffeq import impl, ivpsolve, ivpsolvers, taylor

    N = 40
    vf, u0, (t0, t1), params = ivps.brusselator(N=N)
    impl.impl.select("isotropic", ode_shape=(2 * N,))
    num, tol = 4, 1e-6
    ctrl = ivpsolve.control_proportional_integral()
    ibm = ivpsolvers.prior_ibm(num_derivatives=num)
    ts0 = ivpsolvers.correction_ts0(ode_order=1)
    strategy = ivpsolvers.strategy_fixedpoint(ibm, ts0)
    solver = ivpsolvers.solver_dynamic(strategy)
    adaptive_solver = ivpsolve.adaptive(solver, atol=tol, rtol=tol, control=ctrl)
    tcoeffs = taylor.odejet_unroll(lambda *y: vf(*y, t=t0, p=params), u0, num=num)
    init = solver.initial_condition(tcoeffs, 1.0)
    terminal = ivpsolve.solve_adaptive_terminal_values(vf, init, t0=t0, t1=t1, dt0=0.01, adaptive_solver=adaptive_solver)
    save_at = np.linspace(t0, t1, num=200)
    solution = ivpsolve.solve_adaptive_save_at(vf, init, save_at=save_at, dt0=0.01, adaptive_solver=adaptive_solver)
    # no step clipping: both loops take the same number of steps (SURVEY 3.2)
    assert int(np.amax(solution.num_steps)) == int(terminal.num_steps)
    assert solution.u.shape == (200, 2 * N) and solution.u_std.shape == (200, 2 * N)
    np.testing.assert_allclose(solution.u[-1], terminal.u, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(solution.u[0], u0[0], atol=1e-13)
    # the stats calls of src/odecheckpts/ivpsolvers.py:80-89
    from odecheckpts_b200.probdiffeq import stats

    post = stats.markov_select_terminal(solution.posterior)
    margs = stats.markov_marginals(post, reverse=True)
    mean = np.concatenate([margs.mean, solution.posterior.init.mean[[-1], ...]])
    np.testing.assert_array_equal(mean[:, 0, :], solution.u)


def test_vdp_script_style_dense_ekf1_filter_and_fixed_grid(goldens):
    # experiments/1_van_der_pol/vdp.py:52-91
    from odecheckpts_b200 import ivps
    from odecheckpts_b200.probdiffeq import impl, ivpsolve, ivpsolvers, taylor

    vf, (u0, du0), (t0, t1) = ivps.van_der_pol(mu=1e3)
    impl.impl.select("dense", ode_shape=(1,))
    num = 4
    ibm = ivpsolvers.prior_ibm(num_derivatives=num)
    ts1 = ivpsolvers.correction_ts1(ode_order=2)
    strategy = ivpsolvers.strategy_filter(ibm, ts1)
    solver = ivpsolvers.solver_dynamic(strategy)
    tcoeffs = taylor.odejet_padded_scan(lambda *y: vf(*y, t=t0), [u0, du0], num=num - 1)
    init = solver.initial_condition(tcoeffs, 1.0)
    ctrl = ivpsolve.control_proportional_integral()
    adaptive_solver = ivpsolve.adaptive(solver, atol=1e-3, rtol=1e-3, control=ctrl)
    solution = ivpsolve.solve_adaptive_save_every_step(vf, init, t0=t0, t1=t1, dt0=0.01, adaptive_solver=adaptive_solver)
    grid = goldens["vdp_grid"]
    assert abs(len(solution.t) - len(grid)) <= 0.01 * len(grid) and solution.t[-1] == t1
    np.testing.assert_allclose(solution.t[:26], grid[:26], atol=2e-14)
    replay = ivpsolve.solve_fixed_grid(vf, init, grid=solution.t, solver=solver)
    # replaying t[k+1] - t[k] is not bit-identical to the adaptive dt (stiff: rounding is amplified)
    rel = np.abs(replay.u[:-1, 0] - solution.u[:-1, 0]) / np.abs(solution.u[:-1, 0])
    assert np.median(rel) < 1e-7 and rel.max() < 1e-2


def test_dense_ekf1_through_the_solve_factory_and_ensembles():
    import torch

    from odecheckpts_b200 import ivps, ivpsolvers

    vf, u0, tspan, args = ivps.rigid_body(time_span=(0.0, 10.0))
    save_at = np.linspace(*tspan, num=6)
    kw = dict(save_at=save_at, dt0=0.1, atol=1e-8, rtol=1e-6)
    s_iso, _ = ivpsolvers.solve("ts0-4", vf, u0[0], **kw)(u0, args)
    s_dense, _ = ivpsolvers.solve("ts1-4", vf, u0[0], factorisation="dense", **kw)(u0, args)
    s_bdiag, _ = ivpsolvers.solve("ts0-4", vf, u0[0], factorisation="blockdiag", **kw)(u0, args)
    assert np.abs(s_iso - s_dense).max() < 1e-4 and np.abs(s_iso - s_bdiag).max() < 1e-4
    B = 40
    u0_b = torch.as_tensor(u0[0], device="cuda")[None] + 0.01 * torch.randn(B, 3, dtype=torch.float64, device="cuda")
    s_b, aux = ivpsolvers.solve("ts1-4", vf, u0[0], factorisation="dense", **kw)((u0_b,), args)
    assert s_b.is_cuda and tuple(s_b.shape) == (B, 6, 3) and int((aux["solution"].status != 0).sum()) == 0


def test_posterior_sampling_matches_the_smoothed_marginals():
    # experiments/5_vs_interpolation/measure.py:44-77: three-body, isotropic EKF0 o2 nu=4 uncalibrated,
    # checkpoint solver + stats.markov_sample(reverse=True); parity here is distributional
    from odecheckpts_b200 import ivps
    from odecheckpts_b200.probdiffeq import impl, ivpsolve, ivpsolvers, stats, taylor

    vf, init, tspan = ivps.three_body_restricted()
    impl.impl.select("isotropic", ode_shape=(2,))
    ibm = ivpsolvers.prior_ibm(num_derivatives=4)
    ts0 = ivpsolvers.correction_ts0(ode_order=2)
    strategy = ivpsolvers.strategy_fixedpoint(ibm, ts0)
    solver = ivpsolvers.solver(strategy)
    ctrl = ivpsolve.control_proportional_integral()
    t0, t1 = tspan
    tcoeffs = taylor.odejet_padded_scan(lambda *y: vf(*y, t=t0), init, num=3)
    ic = solver.initial_condition(tcoeffs, np.ones(()))
    asolver = ivpsolve.adaptive(solver, atol=1e-4, rtol=1e-4, control=ctrl)
    save_at = np.linspace(t0, t1)
    solution = ivpsolve.solve_adaptive_save_at(vf, ic, save_at=save_at, dt0=0.01, adaptive_solver=asolver, keep_conditionals=True)
    assert int(solution.num_steps[-1]) == 448  # the reference's golden count at tol 1e-4
    posterior = stats.markov_select_terminal(solution.posterior)
    S = 20000
    (qoi, _), (init_s, _) = stats.markov_sample(1, posterior, shape=(S,), reverse=True)
    qoi = np.concatenate([qoi, init_s[..., None, :]], axis=-2)  # measure.py:76
    assert qoi.shape == (S, len(save_at), 2)
    mean, std = qoi.mean(axis=0), qoi.std(axis=0)
    # sample moments vs the smoothed marginals: 5 standard errors (+ a floor for the exactly-known t0)
    se = solution.u_std / np.sqrt(S)
    assert np.all(np.abs(mean - solution.u) <= 5 * se + 1e-12)
    big = solution.u_std > 1e-10
    np.testing.assert_allclose(std[big], solution.u_std[big], rtol=0.05)
    # joint structure: neighbouring checkpoints are strongly correlated draws of one trajectory
    k = len(save_at) // 2
    c = np.corrcoef(qoi[:, k, 0] - mean[k, 0], qoi[:, k + 1, 0] - mean[k + 1, 0])[0, 1]
    assert abs(c) > 0.2
    # a different key gives different draws, the same key the same draws
    (q2, _), _ = stats.markov_sample(2, posterior, shape=(8,), reverse=True)
    (q3, _), _ = stats.markov_sample(2, posterior, shape=(8,), reverse=True)
    np.testing.assert_array_equal(q2, q3)
    assert not np.array_equal(q2, qoi[:8, :-1])


def test_solve_via_interpolate_drop_in_matches_the_reference_goldens(goldens):
    # tests/test_ivpsolvers.py (reference) runs the same assertions for solve_via_interpolate;
    # experiments/2_workprec_simple/run_simple.py:58-80,200 committed its grid lengths and RMSEs
    import scipy.integrate

    from odecheckpts_b200 import ivps, ivpsolvers

    vf, u0, time_span, args = ivps.logistic()
    save_at = np.linspace(*time_span, num=5)
    sol, aux = ivpsolvers.solve_via_interpolate("ts0-4", vf, u0[0], save_at, dt0=0.1, atol=1e-3, rtol=1e-3)(u0, args)
    assert "u0_solve" in aux.keys() and sol.shape == (5, 1)
    assert np.allclose(sol[:, 0], pu.logistic_exact(save_at), atol=np.sqrt(1e-3), rtol=np.sqrt(1e-3))

    vf, u0, tspan, params = ivps.rigid_body(time_span=(0.0, 50.0))
    xs = goldens["rigid_checkpoints"]
    ref = scipy.integrate.solve_ivp(lambda t, y: vf(y, t=t, p=params), (0.0, 50.0), u0[0], t_eval=xs, method="DOP853", atol=1e-13, rtol=1e-13).y.T
    for nu, key in [(2, "rigid_interp_nu2"), (4, "rigid_interp_nu4")]:
        for tol, want_len, want_rmse in zip(goldens[key + "_list_of_args"], goldens[key + "_length_of_longest_vector"], goldens[key + "_precision"]):
            t = tol * 100  # run_simple.py:60-64
            fun = ivpsolvers.solve_via_interpolate(f"ts0-{nu}", vf, u0[0], save_at=xs, dt0=50.0, atol=1e-3 * t, rtol=t)
            sol, aux = fun(u0, params)
            assert abs(len(aux["u0_solve"]) - want_len) <= 0.04 * want_len
            rmse = np.linalg.norm(sol - ref) / np.sqrt(ref.size)
            assert abs(rmse / want_rmse - 1.0) < 0.15, (nu, tol, rmse, want_rmse)
    # the last (tightest) nu = 2 case is well conditioned: exact grid length, RMSE to 4 digits
    assert len(aux["u0_solve"]) > 0
    fun = ivpsolvers.solve_via_interpolate("ts0-2", vf, u0[0], save_at=xs, dt0=50.0, atol=1e-3 * 1e-5, rtol=1e-5)
    sol, aux = fun(u0, params)
    assert len(aux["u0_solve"]) == 4158
    assert abs(np.linalg.norm(sol - ref) / np.sqrt(ref.size) / goldens["rigid_interp_nu2_precision"][-1] - 1.0) < 1e-3


@pytest.mark.parametrize("m0", ["ts0-2", "ts0-4"])
@pytest.mark.parametrize("m1", ["bosh3", "tsit5"])
@pytest.mark.parametrize("which", ["checkpoint", "interpolate"])
def test_two_solvers_return_the_same_solution(oracle, m0, m1, which):
    # the reference's own test (tests/test_ivpsolvers.py:11-52), parametrisation for parametrisation; the
    # diffrax competitors (out of scope, SURVEY 2) are stood in for by scipy's Runge-Kutta pairs of the
    # same orders (Bogacki-Shampine 3(2) = RK23, a 5(4) pair = RK45) on the oracle's vector field
    import scipy.integrate

    from odecheckpts_b200 import ivps, ivpsolvers

    vf, u0, time_span, args = ivps.logistic()
    dt0 = 0.1
    atol, rtol = 1e-3, 1e-3
    save_at = np.linspace(*time_span, num=5)
    u0_like = u0[0]
    solver1 = ivpsolvers.solve if which == "checkpoint" else ivpsolvers.solve_via_interpolate
    solve1 = solver1(m0, vf, u0_like, save_at, dt0=dt0, atol=atol, rtol=rtol)
    solution1, aux1 = solve1(u0, args)

    def solve2(u0_, p):
        (init,) = u0_
        f = lambda t, y: oracle.vf("logistic", y.reshape(1, -1), list(p), t=t)  # noqa: E731
        sol = scipy.integrate.solve_ivp(f, (save_at[0], save_at[-1]), np.atleast_1d(init), t_eval=save_at, first_step=dt0,
                                        method={"bosh3": "RK23", "tsit5": "RK45"}[m1], atol=atol, rtol=rtol)  # fmt: skip
        return sol.y.T, {"solution": sol, "u0_solve": sol.y.T}

    solution2, aux2 = solve2(u0, args)
    assert "u0_solve" in aux1.keys()
    assert "u0_solve" in aux2.keys()
    assert np.allclose(solution1, solution2, atol=np.sqrt(atol), rtol=np.sqrt(rtol))


def test_textbook_smoother_route_and_checkpoint_solver_evaluate_the_same_posterior(oracle):
    """strategy_smoother + solve_adaptive_save_every_step + offgrid_marginals_searchsorted
    (src/odecheckpts/ivpsolvers.py:94-148, experiments/4_brusselator/run.py:102-117): one backward conditional
    per accepted step, O(#steps) memory.  (a) it is bit-identical to the oracle run with the accepted grid and
    save_at as checkpoints; (b) it agrees with the O(K) fixed-point checkpoint solver to rounding -- the
    equivalence the reference's paper is about; (c) its memory grows with the number of steps."""
    from odecheckpts_b200 import ivps, ivpsolvers
    from odecheckpts_b200.probdiffeq import ivpsolve, stats, taylor
    from odecheckpts_b200.probdiffeq import ivpsolvers as pdi

    vf, u0, tspan, params = ivps.rigid_body(time_span=(0.0, 10.0))
    save_at = np.linspace(0.0, 10.0, 6)
    tol = 1e-5
    dense, aux = ivpsolvers.solve_via_interpolate("ts0-4", vf, u0[0], save_at=save_at, dt0=0.1, atol=tol, rtol=tol)(u0, params)
    sol = aux["solution"]
    n_grid = len(sol.t)
    assert dense.shape == (6, 3) and n_grid > 50 and aux["u0_solve"].shape == (n_grid, 3)
    # (b) same posterior by two routes: the fixed-point solver on the same interval keeps K + 2 merged conditionals
    ext = np.concatenate([[sol.t[0]], save_at, [sol.t[-1]]])
    ckpt = ivpsolve._solve_on_checkpoints(sol.posterior.context, ext)
    assert int(ckpt.num_steps[-1]) == n_grid - 1
    np.testing.assert_allclose(dense, ckpt.u[1:-1], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(ivpsolvers.solve("ts0-4", vf, u0[0], save_at=save_at, dt0=0.1, atol=tol, rtol=tol)(u0, params)[0],
                               dense, atol=1e-4)  # the reference's own pair of routines (intervals differ by 1e-6)
    # (a) oracle: adaptive fixed-point solve on [t0 - 1e-6, t1 + 1e-6] with grid + save_at as checkpoints
    grid = np.asarray(sol.t)
    union = np.union1d(grid, save_at)
    cfg = oracle.make_config("rigid_body", 3, 4, 1, atol=tol, rtol=tol, dt0=0.1, num_params=3)
    ora = oracle.solve_save_at(cfg, u0[0][None], params, union)
    assert ora["status"] == 0 and ora["n_accepted"][-1] == n_grid - 1
    np.testing.assert_array_equal(dense, ora["u"][np.searchsorted(union, save_at)])
    ora_grid = oracle.solve_save_at(cfg, u0[0][None], params, grid)
    np.testing.assert_array_equal(np.asarray(sol.u), ora_grid["u"])
    # (c) the builder vocabulary the scripts use, and the memory the smoother holds on the device
    strategy = pdi.strategy_smoother(pdi.prior_ibm(num_derivatives=4), pdi.correction_ts0())
    solver = pdi.solver_dynamic(strategy)
    asolver = ivpsolve.adaptive(solver, atol=tol, rtol=tol, control=ivpsolve.control_proportional_integral())
    tcoeffs = taylor.odejet_padded_scan(lambda y, t: vf(y, t=t, p=params), u0, num=4)
    init = solver.initial_condition(tcoeffs, output_scale=1.0)
    s2 = ivpsolve.solve_adaptive_save_every_step(lambda y, t: vf(y, t=t, p=params), init, t0=0.0, t1=10.0, dt0=0.1,
                                                 adaptive_solver=asolver, factorisation="isotropic")  # fmt: skip
    u_off, marg = stats.offgrid_marginals_searchsorted(ts=np.array([2.5, 7.25]), solution=s2, solver=solver)
    assert u_off.shape == (2, 3) and marg.mean.shape == (2, 5, 3)
    truth = __import__("scipy.integrate").integrate.solve_ivp(lambda t, y: vf(y, t=t, p=params), (0.0, 10.0), u0[0], t_eval=[2.5, 7.25],
                                                              method="DOP853", atol=1e-12, rtol=1e-12).y.T  # fmt: skip
    np.testing.assert_allclose(u_off, truth, atol=1e-3)
