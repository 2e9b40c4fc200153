"""Trajectory recording (solve_adaptive_save_every_step) and the textbook smoother for the dense factorisation with
d > 1: the register-column kernel ((nu+1) d <= 32) and the CTA-per-IVP dense kernel (Brusselator, D >= 40).

traj_std is per dimension, [cap][d][B]: the std of component l is sqrt((L L^T)_ll) of the recorded factor.  The
kernels follow the oracle's operation order, so every recorded point is compared with
oracle.solve_save_every_step BIT FOR BIT.
"""

import numpy as np
import pytest

import problems_util as pu

RB_PARAMS = np.asarray(pu.RIGID_BODY_PARAMS)
RIGID_FULL = """
struct Problem {
  static constexpr int D = pn::RigidBody::D, Q = pn::RigidBody::Q, P = pn::RigidBody::P, ID = 0;
  static constexpr bool HAS_JAC = pn::RigidBody::HAS_JAC;
  PN_DEV static void vf(const double* u, const double* p, double* f) { pn::RigidBody::vf(u, p, f); }
  PN_DEV static void jac(const double* u, const double* p, double* J) { pn::RigidBody::jac(u, p, J); }
  template <int N> PN_DEV static void vf_jet(const double* U, const double* p, double* F) { pn::RigidBody::vf_jet<N>(U, p, F); }
};
"""
# u_i' = (i + 1) t^i: the solution t, t^2, t^3, t^4 is a polynomial of degree <= nu
POWERS4 = """template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) {
  f[0] = T(1.0);
  f[1] = 2.0 * t;
  f[2] = 3.0 * (t * t);
  f[3] = 4.0 * ((t * t) * t);
}"""


@pytest.fixture(scope="module")
def cabi():
    from odecheckpts_b200 import _cabi

    _cabi.lib()
    return _cabi


def _desc(cabi, problem, d, nu, B, K, *, fact="dense", corr="ts1", strat="filter", atol=1e-8, rtol=1e-6, P=0, record=True,
          cap=4096):  # fmt: skip
    pid = cabi.PROBLEM_IDS[problem] if isinstance(problem, str) else problem
    return cabi.Desc(pid, d, nu, 1, cabi.FACTORISATIONS[fact], cabi.CORRECTIONS[corr], cabi.STRATEGIES[strat],
                     cabi.CALIBRATIONS["dynamic"], atol, rtol, 0.01, 0.95, 0.2, 10.0, 0.3, 0.4, B, K, 0, P,
                     cabi.FLAG_RECORD if record else 0, cap if record else 0)  # fmt: skip


def _brusselator_u0(N):
    x0 = np.linspace(0, 1, N)
    return np.concatenate([np.sin(2 * np.pi * x0) + 1, 3.0 * np.ones(N)])


def _decay_problem(cabi, d):
    src = f"template <class T> PN_DEV void vf(const T* u, const double* p, T* f) {{ for (int i = 0; i < {d}; ++i) f[i] = -u[i]; }}"
    return cabi.register_problem(f"record_decay{d}", src, d=d)


# ---- CPU: selection, sizes, workspace -----------------------------------------------------------------------------
def _recording_configs(cabi):
    """(name, descriptor) of every recording configuration this file covers, with d > 1 and the dense factorisation"""
    user = _decay_problem(cabi, 3)
    return [
        ("rigid body dense ts0", _desc(cabi, "rigid_body", 3, 4, 100, 2, corr="ts0", P=3)),
        ("rigid body dense ts1", _desc(cabi, "rigid_body", 3, 4, 100, 2, P=3)),
        ("brusselator N=8 dense", _desc(cabi, "brusselator", 16, 4, 3, 2, P=1)),
        ("brusselator N=4 dense filter", _desc(cabi, "brusselator", 8, 4, 3, 2, P=1)),
        ("user d=3 dense ts1", _desc(cabi, user, 3, 4, 100, 2)),
    ]


def test_recording_is_supported_for_the_register_column_and_cta_dense_kernels(cabi):
    configs = _recording_configs(cabi)
    before = cabi.lib().pn_b200_jit_module_count()
    for name, desc in configs:
        assert cabi.supported(desc), name
        desc.strategy = cabi.STRATEGIES["fixedpoint"]  # recording needs the filter strategy
        assert not cabi.supported(desc), name
    assert cabi.lib().pn_b200_jit_module_count() == before  # selection never compiles
    # Brusselator N = 4 (D = 40): the fixed-point solve runs on the shared-memory dense kernel, which cannot record;
    # its filter solve runs on the CTA-per-IVP kernel, which can
    desc = _desc(cabi, "brusselator", 8, 4, 3, 2, strat="fixedpoint", P=1)
    assert not cabi.supported(desc)
    with pytest.raises(NotImplementedError, match="trajectory recording"):
        cabi.workspace_bytes(desc)
    desc.flags = 0
    assert cabi.supported(desc)
    assert cabi.supported(_desc(cabi, "brusselator", 8, 4, 3, 2, P=1))


def test_traj_std_is_per_dimension_for_dense_and_one_std_otherwise(cabi):
    from odecheckpts_b200 import _cabi

    for name, desc in _recording_configs(cabi):
        sz = cabi.output_sizes(desc)
        cap, d, B = desc.traj_capacity, desc.d, desc.batch
        assert (sz["traj_t"], sz["traj_u"], sz["traj_std"], sz["traj_len"]) == (cap * B, cap * d * B, cap * d * B, B), name
        assert _cabi._traj_std_shape(desc) == (cap, d, B)
    for fact, corr, d, problem in [("isotropic", "ts0", 3, "rigid_body"), ("dense", "ts1", 1, "van_der_pol")]:
        desc = _desc(cabi, problem, d, 4, 100, 2, fact=fact, corr=corr, P=3 if d == 3 else 1)
        desc.ode_order = 2 if problem == "van_der_pol" else 1
        sz = cabi.output_sizes(desc)
        assert sz["traj_std"] == desc.traj_capacity * 100 and sz["traj_u"] == desc.traj_capacity * d * 100, (fact, d)
        assert _cabi._traj_std_shape(desc) == (desc.traj_capacity, 100)


def test_workspace_does_not_depend_on_recording(cabi):
    for name, desc in _recording_configs(cabi):
        with_rec = cabi.workspace_bytes(desc)
        desc.flags, desc.traj_capacity = 0, 0
        assert cabi.workspace_bytes(desc) == with_rec, name


# ---- GPU helpers --------------------------------------------------------------------------------------------------
def _solve(cabi, desc, u0, params, save_at, tol=None):
    """Every output of a device solve, as numpy."""
    import torch

    dev = torch.device("cuda:0")
    t = lambda x: None if x is None else torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device=dev)  # noqa: E731
    out = cabi.solve_device(desc, t(u0), t(params), t(tol), t(save_at), None)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items() if not k.startswith("_")}


def _same(name, got, want):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{name}: shape {got.shape} vs {want.shape}"
    same = (got == want) | (np.isnan(got.astype(float)) & np.isnan(want.astype(float)))
    if not same.all():
        bad = tuple(np.argwhere(~same)[0])
        raise AssertionError(f"{name}: {(~same).sum()} of {same.size} differ, first at {bad}: {got[bad]!r} vs {want[bad]!r}")


def _check_member(name, out, b, ora):
    n = int(out["traj_len"][b])
    assert n == len(ora["t"]), f"{name}: member {b}: {n} recorded points, oracle {len(ora['t'])}"
    _same(f"{name} t[{b}]", out["traj_t"][:n, b], ora["t"])
    _same(f"{name} u[{b}]", out["traj_u"][:n, :, b], ora["u"])
    _same(f"{name} u_std[{b}]", out["traj_std"][:n, :, b], ora["u_std"])
    assert out["n_rejected"][b] == ora["n_rejected"] and out["status"][b] == 0, name


def _rigid_members(B, seed=0):
    rng = np.random.default_rng(seed)
    u0 = (np.array([1.0, 0.0, 0.9]) + 0.1 * rng.uniform(-1, 1, (B, 3))).reshape(B, 1, 3)
    params = RB_PARAMS[None] * (1.0 + 0.05 * rng.uniform(-1, 1, (B, 3)))
    tols = 10.0 ** rng.uniform(-8, -6, B)
    return u0, params, np.stack([tols, 100.0 * tols], 1)


T1_RB, T1_BR = 20.0, 2.0


# ---- GPU: bit for bit against the oracle --------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("corr", ["ts0", "ts1"])
def test_rigid_body_register_columns_record_bitwise(cabi, oracle, corr):
    """An odd ensemble with per-member parameters and tolerances: both 16-lane halves of a warp record their own
    member (and the last warp has one idle half)."""
    B = 37
    u0, params, tol = _rigid_members(B)
    desc = _desc(cabi, "rigid_body", 3, 4, B, 2, corr=corr, P=3)
    out = _solve(cabi, desc, u0, params, [0.0, T1_RB], tol)
    assert out["traj_std"].shape == (desc.traj_capacity, 3, B)
    spread = 0.0
    for b in range(B):
        cfg = oracle.make_config("rigid_body", 3, 4, 1, factorisation="dense", correction=corr, strategy="filter",
                                 atol=tol[b, 0], rtol=tol[b, 1], dt0=0.01, num_params=3)  # fmt: skip
        ora = oracle.solve_save_every_step(cfg, u0[b], params[b], 0.0, T1_RB)
        _check_member(f"rigid body {corr}", out, b, ora)
        s = ora["u_std"][1:]
        spread = max(spread, float(np.max((s.max(1) - s.min(1)) / s.max(1))))
    if corr == "ts1":
        assert spread > 0.5  # the components' stds really differ: a shared std would be wrong


@pytest.mark.gpu
@pytest.mark.parametrize("N", [4, 8])
def test_brusselator_cta_kernel_records_bitwise_against_the_blocked_oracle(cabi, oracle, N):
    B = 3
    u0 = np.tile(_brusselator_u0(N)[None, None], (B, 1, 1))
    alpha = np.array([[0.02], [0.01], [0.04]])
    desc = _desc(cabi, "brusselator", 2 * N, 4, B, 2, atol=1e-5, rtol=1e-5, P=1)
    out = _solve(cabi, desc, u0, alpha, [0.0, T1_BR])
    cfg = oracle.make_config("brusselator", 2 * N, 4, 1, factorisation="dense", correction="ts1", strategy="filter", atol=1e-5,
                             rtol=1e-5, dt0=0.01, num_params=1, reduction_group=256, dense_block=16)  # fmt: skip
    for b in range(B):
        ora = oracle.solve_save_every_step(cfg, u0[b], alpha[b], 0.0, T1_BR)
        assert len(ora["t"]) > 20
        _check_member(f"brusselator N={N}", out, b, ora)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["rows", "cta", "thread_per_ivp"])
def test_a_small_capacity_truncates_like_the_thread_per_ivp_kernel(cabi, kernel):
    """traj_len = min(accepted + 1, cap); the kept points are the first ones of an unbounded recording."""
    if kernel == "rows":
        u0, params, _ = _rigid_members(4, seed=2)
        desc, t1 = _desc(cabi, "rigid_body", 3, 4, 4, 2, P=3), T1_RB
    elif kernel == "cta":
        u0, params = np.tile(_brusselator_u0(8)[None, None], (2, 1, 1)), np.array([[0.02], [0.03]])
        desc, t1 = _desc(cabi, "brusselator", 16, 4, 2, 2, atol=1e-5, rtol=1e-5, P=1), T1_BR
    else:  # dense with d = 1 runs on the thread-per-IVP kernel
        u0, params = np.tile(pu.van_der_pol_u0()[None], (2, 1, 1)), np.array([[10.0], [20.0]])
        desc, t1 = _desc(cabi, "van_der_pol", 1, 4, 2, 2, atol=1e-5, rtol=1e-5, P=1), 3.0
        desc.ode_order = 2
    full = _solve(cabi, desc, u0, params, [0.0, t1])
    assert (full["traj_len"] > 12).all() and (full["traj_len"] < desc.traj_capacity).all()
    cap = 10
    desc.traj_capacity = cap
    small = _solve(cabi, desc, u0, params, [0.0, t1])
    assert (small["traj_len"] == cap).all()
    for key in ("traj_t", "traj_u", "traj_std"):
        _same(f"{kernel} {key}", small[key], full[key][:cap])
    for key in ("n_rejected", "status"):
        _same(f"{kernel} {key}", small[key], full[key])


@pytest.mark.gpu
def test_solve_adaptive_save_every_step_returns_per_dimension_std(oracle):
    from odecheckpts_b200 import ivps
    from odecheckpts_b200.probdiffeq import ivpsolve, taylor
    from odecheckpts_b200.probdiffeq import ivpsolvers as pdi

    vf, u0, _, params = ivps.rigid_body(time_span=(0.0, T1_RB))
    solver = pdi.solver_dynamic(pdi.strategy_filter(pdi.prior_ibm(num_derivatives=4), pdi.correction_ts1()))
    asolver = ivpsolve.adaptive(solver, atol=1e-8, rtol=1e-6, control=ivpsolve.control_proportional_integral())
    f = lambda y, t: vf(y, t=t, p=params)  # noqa: E731
    init = solver.initial_condition(taylor.odejet_padded_scan(f, u0, num=4), output_scale=1.0)
    sol = ivpsolve.solve_adaptive_save_every_step(f, init, t0=0.0, t1=T1_RB, dt0=0.01, adaptive_solver=asolver,
                                                  factorisation="dense")  # fmt: skip
    cfg = oracle.make_config("rigid_body", 3, 4, 1, factorisation="dense", correction="ts1", strategy="filter", atol=1e-8,
                             rtol=1e-6, dt0=0.01, num_params=3)  # fmt: skip
    ora = oracle.solve_save_every_step(cfg, u0[0][None], list(params), 0.0, T1_RB)
    assert np.shape(sol.u_std) == np.shape(sol.u) == (len(ora["t"]), 3)
    _same("t", sol.t, ora["t"])
    _same("u", sol.u, ora["u"])
    _same("u_std", sol.u_std, ora["u_std"])
    assert sol.num_steps == len(ora["t"]) - 1 and sol.num_rejected == ora["n_rejected"]
    # an ensemble of two: [cap, d, B]
    import torch

    u0b = torch.as_tensor(np.tile(u0[0], (2, 1)), device="cuda")
    initb = solver.initial_condition(taylor.odejet_padded_scan(f, (u0b,), num=4), output_scale=1.0)
    solb = ivpsolve.solve_adaptive_save_every_step(f, initb, t0=0.0, t1=T1_RB, dt0=0.01, adaptive_solver=asolver,
                                                   factorisation="dense", max_steps=2048)  # fmt: skip
    assert tuple(solb.u_std.shape) == (2048, 3, 2) and tuple(solb.u.shape) == (2048, 3, 2)
    n = len(ora["t"])
    for b in range(2):
        assert int(solb.num_steps[b]) == n - 1
        _same(f"ensemble u_std[{b}]", solb.u_std[:n, :, b].cpu().numpy(), ora["u_std"])


# ---- GPU: recording only observes ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["rows", "cta"])
def test_recording_does_not_change_the_checkpoint_outputs(cabi, kernel):
    if kernel == "rows":
        B = 37
        u0, params, tol = _rigid_members(B, seed=5)
        save_at = np.linspace(0.0, T1_RB, 23)
        mk = lambda rec: _desc(cabi, "rigid_body", 3, 4, B, len(save_at), P=3, record=rec)  # noqa: E731
    else:
        B, tol = 3, None
        u0, params = np.tile(_brusselator_u0(8)[None, None], (B, 1, 1)), np.array([[0.02], [0.01], [0.04]])
        save_at = np.linspace(0.0, T1_BR, 9)
        mk = lambda rec: _desc(cabi, "brusselator", 16, 4, B, len(save_at), atol=1e-5, rtol=1e-5, P=1, record=rec)  # noqa: E731
    import torch

    dev = torch.device("cuda:0")
    t = lambda x: None if x is None else torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device=dev)  # noqa: E731
    res = []
    for rec in (False, True):
        out = cabi.solve_device(mk(rec), t(u0), t(params), t(tol), t(save_at), None, full=True)
        torch.cuda.synchronize()
        res.append({k: v.cpu().numpy() for k, v in out.items() if not k.startswith("_")})
    plain, rec = res
    for key in ("u", "u_std", "marg_mean", "marg_chol", "output_scale", "n_accepted", "n_rejected", "status"):
        _same(f"{kernel} {key}", rec[key], plain[key])
    # the recording ends at the last checkpoint with the checkpoint's marginal
    for b in range(B):
        n = int(rec["traj_len"][b])
        # (a step that ends within 10 eps of t1 is a hit on it and records its own time)
        assert n == rec["n_accepted"][b, -1] + 1 and abs(rec["traj_t"][n - 1, b] - save_at[-1]) <= 1e-14 * abs(save_at[-1])
        _same(f"{kernel} last u[{b}]", rec["traj_u"][n - 1, :, b], rec["u"][b, -1])
        _same(f"{kernel} last u_std[{b}]", rec["traj_std"][n - 1, :, b], rec["u_std"][b, -1])


# ---- GPU: the textbook smoother -----------------------------------------------------------------------------------
def _smoother_case(problem):
    from odecheckpts_b200 import ivps
    from odecheckpts_b200.probdiffeq import taylor

    if problem == "rigid_body":
        vf, u0, _, params = ivps.rigid_body(time_span=(0.0, T1_RB))
        tol, t1, num = 1e-7, T1_RB, 4
        f = lambda y, t: vf(y, t=t, p=params)  # noqa: E731
        tcoeffs = taylor.odejet_padded_scan(f, u0, num=num)
    else:
        vf, u0, _, params = ivps.brusselator(N=8)
        tol, t1 = 1e-5, T1_BR
        f = lambda *y, t=None: vf(*y, t=t, p=params)  # noqa: E731
        tcoeffs = taylor.odejet_unroll(lambda *y: vf(*y, t=0.0, p=params), u0, num=4)
    return vf, u0, params, tol, t1, f, tcoeffs


@pytest.mark.gpu
@pytest.mark.parametrize("problem", ["rigid_body", "brusselator"])
def test_textbook_smoother_with_dense_ekf1(oracle, problem):
    """strategy_smoother + solve_adaptive_save_every_step + offgrid_marginals_searchsorted on a dense EKF1 solver:
    (a) the same posterior as the checkpoint solver at the same save_at, (b) bit-identical to the oracle run with
    grid + save_at as checkpoints."""
    from odecheckpts_b200.probdiffeq import ivpsolve, stats
    from odecheckpts_b200.probdiffeq import ivpsolvers as pdi

    vf, u0, params, tol, t1, f, tcoeffs = _smoother_case(problem)
    d = len(np.asarray(u0[0]))
    ctrl = ivpsolve.control_proportional_integral()
    ibm, ts1 = pdi.prior_ibm(num_derivatives=4), pdi.correction_ts1()

    def adaptive(strategy):
        solver = pdi.solver_dynamic(strategy)
        return solver, solver.initial_condition(tcoeffs, 1.0), ivpsolve.adaptive(solver, atol=tol, rtol=tol, control=ctrl)

    smoother, init_s, asolver_s = adaptive(pdi.strategy_smoother(ibm, ts1))
    _, init_c, asolver_c = adaptive(pdi.strategy_fixedpoint(ibm, ts1))
    text = ivpsolve.solve_adaptive_save_every_step(f, init_s, t0=0.0, t1=t1, dt0=0.01, adaptive_solver=asolver_s,
                                                   factorisation="dense")  # fmt: skip
    grid = np.asarray(text.t)
    assert grid[0] == 0.0 and grid[-1] == t1 and len(grid) > 20 and text.u.shape == (len(grid), d)
    save_at = np.linspace(0.0, t1, 7)
    inner = save_at[1:-1]
    u_off, marg = stats.offgrid_marginals_searchsorted(ts=inner, solution=text, solver=smoother)
    assert u_off.shape == (len(inner), d) and marg.mean.shape == (len(inner), 5, d)
    # (a) the checkpoint solver (fixed-point, O(K) memory) at the same save_at
    ckpt = ivpsolve.solve_adaptive_save_at(f, init_c, save_at=save_at, dt0=0.01, adaptive_solver=asolver_c, factorisation="dense")
    assert int(ckpt.num_steps[-1]) == len(grid) - 1
    np.testing.assert_allclose(u_off, ckpt.u[1:-1], rtol=1e-9, atol=1e-12)
    # (b) the oracle, fixed-point dense, with the accepted grid and save_at as checkpoints
    union = np.union1d(grid, inner)
    kw = dict(factorisation="dense", correction="ts1", atol=tol, rtol=tol, dt0=0.01, num_params=len(params))
    if problem == "brusselator":
        kw.update(reduction_group=256, dense_block=16)
    ora = oracle.solve_save_at(oracle.make_config(problem, d, 4, 1, **kw), np.asarray(u0[0])[None], list(params), union)
    assert ora["status"] == 0 and ora["n_accepted"][-1] == len(grid) - 1
    idx = np.searchsorted(union, inner)
    _same(f"{problem} smoother u", u_off, ora["u"][idx])
    # the smoothed grid values of the textbook route are the oracle's as well
    ora_grid = oracle.solve_save_at(oracle.make_config(problem, d, 4, 1, **kw), np.asarray(u0[0])[None], list(params), grid)
    _same(f"{problem} smoother grid u", text.u, ora_grid["u"])
    _same(f"{problem} smoother grid u_std", text.u_std, ora_grid["u_std"])


# ---- GPU: user problems -------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_user_rigid_body_records_like_the_builtin(cabi):
    B = 37
    u0, params, tol = _rigid_members(B, seed=7)
    pid = cabi.register_problem("rigid_body_record_full", RIGID_FULL, d=3, ode_order=1, num_params=3, form="full")
    desc = _desc(cabi, pid, 3, 4, B, 5, P=3)
    save_at = np.linspace(0.0, T1_RB, 5)
    user = _solve(cabi, desc, u0, params, save_at, tol)
    desc.problem = cabi.PROBLEM_IDS["rigid_body"]
    ref = _solve(cabi, desc, u0, params, save_at, tol)
    assert user.keys() == ref.keys() and "traj_std" in ref
    for key in ref:
        if key in ("traj_t", "traj_u", "traj_std"):  # entries past a member's traj_len are not written
            for b in range(B):
                n = int(ref["traj_len"][b])
                _same(f"user rigid body {key}[{b}]", user[key][:n, ..., b], ref[key][:n, ..., b])
        else:
            _same(f"user rigid body {key}", user[key], ref[key])
    assert (ref["status"] == 0).all() and ref["traj_len"].min() > 50


@pytest.mark.gpu
def test_time_dependent_user_problem_is_exact_at_every_recorded_point(cabi):
    """d = 4, nu = 4: D = 20, one IVP per warp (32 lanes).  The polynomial solution t .. t^4 is in the prior's span."""
    t0, t1 = 0.7, 3.2
    pid = cabi.register_problem("powers4_record", POWERS4, d=4, time_dependent=True)
    B = 4
    u0 = np.tile(np.array([t0, t0**2, t0**3, t0**4])[None, None], (B, 1, 1))
    desc = _desc(cabi, pid, 4, 4, B, 2, atol=1e-10, rtol=1e-10)
    desc.calibration = cabi.CALIBRATIONS["none"]
    out = _solve(cabi, desc, u0, None, [t0, t1])
    assert (out["status"] == 0).all() and out["traj_std"].shape == (desc.traj_capacity, 4, B)
    for b in range(B):
        n = int(out["traj_len"][b])
        t = out["traj_t"][:n, b]
        assert n >= 2 and t[0] == t0 and t[-1] == t1 and np.all(np.diff(t) > 0)
        want = t[:, None] ** np.arange(1, 5)[None]
        rel = np.abs(out["traj_u"][:n, :, b] - want) / np.maximum(1.0, np.abs(want))
        assert rel.max() <= 1e-10, f"member {b}: max relative error {rel.max():.3g}"
        assert (out["traj_std"][0, :, b] == 0).all() and np.isfinite(out["traj_std"][:n, :, b]).all()
