"""Time-dependent user vector fields (cuda_vector_field(..., time_dependent=True) / PN_B200_FORM_TIME_DEPENDENT):
registration and the flag, the host function, bit-identity of a field that ignores its time with its autonomous
registration in every kernel build, exact time handling on polynomial solutions, the Taylor coefficients and
Jacobians of non-autonomous fields, and forced ODEs solved end to end."""

import ctypes as C

import numpy as np
import pytest
import scipy.integrate

FORM_SIMPLE, FORM_FULL, FORM_TIME = 0, 1, 2

# ---- sources ------------------------------------------------------------------------------------------------------
VDP = "template <class T> PN_DEV void vf(const T* u, const double* p, T* f) { f[0] = p[0] * fma(u[1], fma(-u[0], u[0], 1.0), -u[0]); }"
VDP_T = "template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) { f[0] = p[0] * fma(u[1], fma(-u[0], u[0], 1.0), -u[0]); }"
RIGID = """template <class T> PN_DEV void vf(const T* u, const double* p, T* f) {
  f[0] = p[0] * (u[1] * u[2]);
  f[1] = p[1] * (u[0] * u[2]);
  f[2] = p[2] * (u[0] * u[1]);
}"""
RIGID_T = RIGID.replace("const T* u, const double* p", "const T* u, const T& t, const double* p")
VDP_FULL_T = """struct Problem {
  static constexpr int D = 1, Q = 2, P = 1, ID = 0;
  static constexpr bool HAS_JAC = true, TIME = true;
  PN_DEV static void vf(const double* u, double t, const double* p, double* f) { pn::VanDerPol::vf(u, p, f); }
  PN_DEV static void jac(const double* u, double t, const double* p, double* J) { pn::VanDerPol::jac(u, p, J); }
  template <int N> PN_DEV static void vf_jet(const double* U, const double* Tc, const double* p, double* F) { pn::VanDerPol::vf_jet<N>(U, p, F); }
};"""
# u' = 3 t^2 (u = t^3); u'' = 6 t (u = t^3); u_i' = (i + 1) t^i (u_i = t^(i + 1))
CUBIC = "template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) { f[0] = 3.0 * (t * t); }"
CUBIC2 = "template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) { f[0] = 6.0 * t; }"
POWERS4 = """template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) {
  f[0] = T(1.0);
  f[1] = 2.0 * t;
  f[2] = 3.0 * (t * t);
  f[3] = 4.0 * ((t * t) * t);
}"""
DUFFING = """template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) {
  f[0] = p[3] * cos(p[4] * t) - p[0] * u[1] - p[1] * u[0] - p[2] * ((u[0] * u[0]) * u[0]);
}"""
LORENZ96_T = """template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) {
  const T F = 8.0 + sin(p[0] * t);
  for (int i = 0; i < 8; ++i) f[i] = (u[(i + 1) % 8] - u[(i + 6) % 8]) * u[(i + 7) % 8] - u[i] + F;
}"""
FORCED_DECAY = "template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) { f[0] = sin(p[0] * t) - u[0]; }"


@pytest.fixture(scope="module")
def cabi():
    from odecheckpts_b200 import _cabi

    _cabi.lib()
    return _cabi


def _desc(cabi, problem, d, nu, q, B, K, *, fact="dense", corr="ts1", strat="fixedpoint", calib="dynamic", tol=1e-6, P=0,
          flags=0, cap=0, dt0=0.01):  # fmt: skip
    return cabi.Desc(problem, d, nu, q, cabi.FACTORISATIONS[fact], cabi.CORRECTIONS[corr], cabi.STRATEGIES[strat],
                     cabi.CALIBRATIONS[calib], tol, tol, dt0, 0.95, 0.2, 10.0, 0.3, 0.4, B, K, 0, P, flags, cap)  # fmt: skip


def _register_raw(cabi, name, src, form, d=1, q=1, P=0):
    pid = C.c_int32(-1)
    rc = cabi.lib().pn_b200_register_problem(name.encode(), src.encode(), form, d, q, P, C.byref(pid))
    return rc, pid.value


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_both_forms_register_with_the_flag(cabi):
    a = cabi.register_problem("vdp_t_simple", VDP_T, d=1, ode_order=2, num_params=1, time_dependent=True)
    b = cabi.register_problem("vdp_t_full", VDP_FULL_T, d=1, ode_order=2, num_params=1, form="full", time_dependent=True)
    assert a >= cabi.USER_PROBLEM_BASE and b >= cabi.USER_PROBLEM_BASE and a != b
    assert cabi.register_problem("vdp_t_simple", VDP_T, d=1, ode_order=2, num_params=1, time_dependent=True) == a
    assert _register_raw(cabi, "vdp_t_full", VDP_FULL_T, FORM_FULL | FORM_TIME, 1, 2, 1) == (0, b)


def test_the_flag_is_part_of_the_registration(cabi):
    both = VDP + "\n" + VDP_T  # a source with both signatures compiles either way
    a = cabi.register_problem("vdp_both", both, d=1, ode_order=2, num_params=1)
    b = cabi.register_problem("vdp_both", both, d=1, ode_order=2, num_params=1, time_dependent=True)
    assert a != b
    assert cabi.register_problem("vdp_both", both, d=1, ode_order=2, num_params=1) == a


def test_a_time_dependent_source_needs_the_flag(cabi):
    with pytest.raises(ValueError) as e:
        cabi.register_problem("cubic_without_flag", CUBIC, d=1)
    assert "cubic_without_flag (adapter)" in str(e.value) and "error" in str(e.value)
    with pytest.raises(ValueError, match="differs from the registered time dependence"):
        cabi.register_problem("vdp_t_full_without_flag", VDP_FULL_T, d=1, ode_order=2, num_params=1, form="full")
    # and an autonomous source does not compile as a time-dependent one
    with pytest.raises(ValueError):
        cabi.register_problem("vdp_autonomous_with_flag", VDP, d=1, ode_order=2, num_params=1, time_dependent=True)


@pytest.mark.parametrize("form", [4, FORM_SIMPLE | 4, FORM_TIME | 8, -1, 1 << 30])
def test_unknown_form_bits_are_rejected(cabi, form):
    assert _register_raw(cabi, "bad_form", CUBIC, form)[0] == -2
    assert "unknown source form" in cabi.lib().pn_b200_last_error().decode()


def test_the_host_function_receives_t(cabi):
    from odecheckpts_b200 import ivps

    vf = ivps.cuda_vector_field("forced_decay", FORCED_DECAY, d=1, num_params=1, time_dependent=True,
                                host=lambda u, w, t: np.sin(w * t) - u)  # fmt: skip
    assert vf.time_dependent
    np.testing.assert_allclose(vf(np.array([0.5]), t=0.3, p=(2.0,)), np.sin(0.6) - 0.5)
    # the solver finds the field behind a wrapper that passes t=
    found, _ = ivps.resolve_vector_field(lambda *y, t: vf(*y, t=t, p=(2.0,)), (np.ones(1),), t0=0.4)
    assert found is vf
    # autonomous fields keep host(*u, *params)
    auto = ivps.cuda_vector_field("decay_host", "template <class T> PN_DEV void vf(const T* u, const double* p, T* f) { f[0] = -p[0] * u[0]; }",
                                  d=1, num_params=1, host=lambda u, k: -k * u)  # fmt: skip
    assert not auto.time_dependent
    np.testing.assert_allclose(auto(np.array([2.0]), t=5.0, p=(3.0,)), [-6.0])


def test_supported_does_not_compile(cabi):
    l96 = cabi.register_problem("lorenz96_t", LORENZ96_T, d=8, num_params=1, time_dependent=True)
    duf = cabi.register_problem("duffing", DUFFING, d=1, ode_order=2, num_params=5, time_dependent=True)
    before = cabi.lib().pn_b200_jit_module_count()
    for pid, d, q, P, cases in [(l96, 8, 1, 1, [("isotropic", "ts0", 4), ("blockdiag", "ts0", 4), ("dense", "ts1", 3)]),
                                (duf, 1, 2, 5, [("dense", "ts1", 4), ("isotropic", "ts0", 4)])]:  # fmt: skip
        for fact, corr, nu in cases:
            for strat in ("fixedpoint", "filter"):
                desc = _desc(cabi, pid, d, nu, q, 1000, 10, fact=fact, corr=corr, strat=strat, P=P)
                assert cabi.supported(desc) and cabi.workspace_bytes(desc) > 0
    assert cabi.lib().pn_b200_jit_module_count() == before


# ---- GPU: a field that ignores t is bit-identical to its autonomous registration -----------------------------------
def _same(name, a, b):
    assert a.shape == b.shape, name
    assert np.array_equal(a, b, equal_nan=True), f"{name}: {np.sum(a != b)} of {a.size} entries differ"


def _solve_all(cabi, desc, u0, params, save_at, *, samples=True, lml=True):
    import torch

    dev = torch.device("cuda:0")
    t = lambda x: None if x is None else torch.as_tensor(np.ascontiguousarray(x), device=dev)  # noqa: E731
    out = cabi.solve_device(desc, t(u0), t(params), None, t(save_at), None, full=True)
    res = {k: v.cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    if desc.strategy == 1 and samples:
        res["samples"] = cabi.markov_sample_device(desc, out["_workspace"], out["status"], 7, 3).cpu().numpy()
    if desc.strategy == 1 and lml:
        data = out["u"] + 0.01
        res["lml"] = cabi.log_marginal_likelihood_device(desc, out["_workspace"], out["status"], data, 0.1).cpu().numpy()
    torch.cuda.synchronize()
    return res


def _compare_registrations(cabi, name, ids, desc, u0, params, save_at, **kw):
    desc.problem = ids[1]
    timed = _solve_all(cabi, desc, u0, params, save_at, **kw)
    info = cabi.kernel_info(desc)
    desc.problem = ids[0]
    ref = _solve_all(cabi, desc, u0, params, save_at, **kw)
    assert timed.keys() == ref.keys()
    for key in ref:
        _same(f"{name}: {key}", timed[key], ref[key])
    assert (ref["status"] == 0).all()
    return timed, info


def _vdp_members(B, mu=1e3, seed=0):
    rng = np.random.default_rng(seed)
    u0 = np.stack([2.0 + 0.5 * rng.uniform(-1, 1, B), 0.5 * rng.uniform(-1, 1, B)], 1).reshape(B, 2, 1)
    return u0, np.full((B, 1), mu)


@pytest.mark.gpu
@pytest.mark.parametrize("build", ["time-sliced", "pair", "mle", "filter-record", "fixed-grid"])
def test_thread_per_ivp_builds_ignore_an_unused_time_bitwise(cabi, build):
    ids = (cabi.register_problem("vdp_simple", VDP, d=1, ode_order=2, num_params=1),
           cabi.register_problem("vdp_t_simple", VDP_T, d=1, ode_order=2, num_params=1, time_dependent=True))  # fmt: skip
    if build == "time-sliced":
        B, K, kw = 65536, 20, dict(tol=1e-3)
        u0, params = _vdp_members(B)
        save_at = np.linspace(0.0, 6.3, K)
    elif build in ("pair", "mle"):
        B, K, kw = 300, 12, dict(tol=1e-5, calib="mle" if build == "mle" else "dynamic")
        u0, params = _vdp_members(B, seed=3)
        save_at = np.linspace(0.3, 2.3, K)
    elif build == "filter-record":
        B, K, kw = 64, 6, dict(tol=1e-5, strat="filter", flags=cabi.FLAG_RECORD, cap=3000)
        u0, params = _vdp_members(B, mu=10.0, seed=4)
        save_at = np.linspace(0.5, 3.5, K)
    else:
        B, K, kw = 64, 400, dict(tol=1e-5, flags=cabi.FLAG_FIXED_GRID)
        u0, params = _vdp_members(B, mu=10.0, seed=5)
        save_at = np.sort(np.random.default_rng(6).uniform(0.2, 3.0, K))
    nu = 3 if build == "filter-record" else 4
    desc = _desc(cabi, ids[0], 1, nu, 2, B, K, P=1, **kw)
    timed, info = _compare_registrations(cabi, f"vdp {build}", ids, desc, u0, params, save_at)
    if build == "time-sliced":
        assert info["grid"] * 128 < B
    if build == "pair":
        assert info["threads_per_cta"] == 256
    if build == "filter-record":
        assert timed["traj_len"].min() > 10


@pytest.mark.gpu
@pytest.mark.parametrize("fact, corr", [("isotropic", "ts0"), ("blockdiag", "ts0"), ("dense", "ts0"), ("dense", "ts1")])
def test_lane_per_dimension_and_register_columns_ignore_an_unused_time_bitwise(cabi, fact, corr):
    ids = (cabi.register_problem("rigid_simple", RIGID, d=3, num_params=3),
           cabi.register_problem("rigid_t_simple", RIGID_T, d=3, num_params=3, time_dependent=True))  # fmt: skip
    B, K = 500, 10
    rng = np.random.default_rng(1)
    u0 = (np.array([1.0, 0.0, 0.9]) + 0.1 * rng.uniform(-1, 1, (B, 3))).reshape(B, 1, 3)
    params = np.tile([-2.0, 1.25, -0.5], (B, 1))
    desc = _desc(cabi, ids[0], 3, 4, 1, B, K, fact=fact, corr=corr, tol=1e-7, P=3)
    _compare_registrations(cabi, f"rigid body {fact} {corr}", ids, desc, u0, params, np.linspace(0.5, 5.5, K), lml=fact != "dense")


# ---- GPU: exact time handling on polynomial solutions --------------------------------------------------------------
def _solve_exact(cabi, src, name, d, q, nu, save_at, u0, *, fact, corr, strat, fixed_grid=False):
    import torch

    pid = cabi.register_problem(name, src, d=d, ode_order=q, time_dependent=True)
    B, K = u0.shape[0], len(save_at)
    desc = _desc(cabi, pid, d, nu, q, B, K, fact=fact, corr=corr, strat=strat, calib="none", tol=1e-4,
                 flags=cabi.FLAG_FIXED_GRID if fixed_grid else 0)  # fmt: skip
    dev = torch.device("cuda:0")
    out = cabi.solve_device(desc, torch.as_tensor(u0, device=dev), None, None, torch.as_tensor(save_at, device=dev), None)
    torch.cuda.synchronize()
    return {k: out[k].cpu().numpy() for k in ("u", "n_accepted", "status")}


def _check_powers(name, u, save_at, powers):
    want = save_at[:, None] ** np.asarray(powers, dtype=np.float64)[None, :]
    err = np.abs(u.reshape(u.shape[0], len(save_at), -1) - want[None])
    rel = err / np.maximum(1.0, np.abs(want))[None]
    assert rel.max() <= 1e-10, f"{name}: max relative error {rel.max():.3g}"


ADAPTIVE_GRID = np.linspace(0.7, 3.2, 200)  # t0 != 0; several checkpoints fall inside one step
IRREGULAR_GRID = np.concatenate([[0.7], np.sort(np.random.default_rng(9).uniform(0.7, 3.2, 60)), [3.2]])


@pytest.mark.gpu
@pytest.mark.parametrize("strat, fact, corr, fixed_grid", [("fixedpoint", "dense", "ts1", False), ("filter", "dense", "ts1", False),
                                                           ("fixedpoint", "isotropic", "ts0", False), ("fixedpoint", "dense", "ts1", True),
                                                           ("filter", "isotropic", "ts0", True)])  # fmt: skip
def test_thread_per_ivp_is_exact_on_a_cubic(cabi, strat, fact, corr, fixed_grid):
    save_at = IRREGULAR_GRID if fixed_grid else ADAPTIVE_GRID
    t0 = save_at[0]
    for q, src, u0 in [(1, CUBIC, np.array([[t0**3]])), (2, CUBIC2, np.array([[t0**3], [3 * t0**2]]))]:
        u0 = np.tile(u0[None], (4, 1, 1))
        res = _solve_exact(cabi, src, f"cubic_q{q}", 1, q, 3, save_at, u0, fact=fact, corr=corr, strat=strat, fixed_grid=fixed_grid)
        assert (res["status"] == 0).all()
        _check_powers(f"t^3 (ode_order {q}, {strat} {fact})", res["u"], save_at, [3])
        if not fixed_grid:
            assert res["n_accepted"][:, -1].max() < len(save_at) // 4  # the checkpoint predictions did the work


@pytest.mark.gpu
@pytest.mark.parametrize("fact, corr", [("isotropic", "ts0"), ("blockdiag", "ts0"), ("dense", "ts0"), ("dense", "ts1")])
@pytest.mark.parametrize("fixed_grid", [False, True])
def test_lane_per_dimension_and_register_columns_are_exact_on_powers_of_t(cabi, fact, corr, fixed_grid):
    save_at = IRREGULAR_GRID if fixed_grid else ADAPTIVE_GRID
    t0 = save_at[0]
    u0 = np.tile(np.array([t0, t0**2, t0**3, t0**4])[None, None], (4, 1, 1))
    for strat in ("fixedpoint", "filter"):
        res = _solve_exact(cabi, POWERS4, "powers4", 4, 1, 4, save_at, u0, fact=fact, corr=corr, strat=strat, fixed_grid=fixed_grid)
        assert (res["status"] == 0).all()
        _check_powers(f"t^1..t^4 ({strat} {fact} {corr})", res["u"], save_at, [1, 2, 3, 4])


# ---- GPU: Taylor coefficients and Jacobians at several t0 -----------------------------------------------------------
def _evaluate_at(cabi, pid, nu, u0, t, d, q, params=None, jac=True):
    import torch

    dev = torch.device("cuda:0")
    p = None if params is None else torch.as_tensor(params, device=dev)
    out = cabi.problem_evaluate_device(pid, nu, torch.as_tensor(u0, device=dev), p, d=d, ode_order=q, jac=jac,
                                       t=torch.as_tensor(t, device=dev))  # fmt: skip
    return {k: v.cpu().numpy() for k, v in out.items()}


def _close(name, got, ref, rel=1e-13):
    scale = np.maximum(np.abs(ref).reshape(ref.shape[0], -1).max(axis=1), 1e-300).reshape((-1,) + (1,) * (ref.ndim - 1))
    err = np.abs(got - ref)
    assert (err <= rel * scale).all(), f"{name}: max relative error {(err / scale).max():.3g}"


T0S = np.array([-2.0, -0.3, 0.0, 0.4, 1.3, 2.9, 7.5])


@pytest.mark.gpu
def test_taylor_coefficients_of_non_autonomous_fields(cabi):
    nu = 8
    u0 = np.linspace(0.5, 1.5, len(T0S)).reshape(-1, 1, 1)
    # u' = sin t: u^(k)(t0) = sin^(k-1)(t0) = sin(t0 + (k - 1) pi / 2), k >= 1
    pid = cabi.register_problem("sin_t", "template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) { f[0] = sin(t); }",
                                d=1, time_dependent=True)  # fmt: skip
    got = _evaluate_at(cabi, pid, nu, u0, T0S, 1, 1)
    want = np.concatenate([u0[:, :, 0], np.sin(T0S[:, None] + np.arange(nu)[None] * np.pi / 2)], 1)
    _close("u' = sin t", got["taylor"][:, :, 0], want)
    np.testing.assert_allclose(got["f"][:, 0], np.sin(T0S), rtol=1e-15, atol=1e-16)
    assert (got["jac"] == 0).all()
    # u' = t u: u^(k+1) = t u^(k) + k u^(k-1)
    pid = cabi.register_problem("t_times_u", "template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) { f[0] = t * u[0]; }",
                                d=1, time_dependent=True)  # fmt: skip
    got = _evaluate_at(cabi, pid, nu, u0, T0S, 1, 1)
    want = np.zeros((len(T0S), nu + 1))
    want[:, 0] = u0[:, 0, 0]
    want[:, 1] = T0S * want[:, 0]
    for k in range(1, nu):
        want[:, k + 1] = T0S * want[:, k] + k * want[:, k - 1]
    _close("u' = t u", got["taylor"][:, :, 0], want)
    np.testing.assert_array_equal(got["jac"][:, 0, 0], T0S)
    # without t the evaluation is at t = 0
    import torch

    dev = torch.device("cuda:0")
    at0 = cabi.problem_evaluate_device(pid, 2, torch.as_tensor(u0, device=dev), None, d=1, ode_order=1)
    np.testing.assert_array_equal(at0["taylor"].cpu().numpy()[:, :, 0], np.stack([u0[:, 0, 0], 0 * T0S, u0[:, 0, 0]], 1))


@pytest.mark.gpu
def test_second_order_taylor_coefficients_with_time(cabi):
    # forced oscillator u'' = cos(w t) - u:  u^(k+2) = cos^(k)(w t) w^k - u^(k)
    nu = 7
    rng = np.random.default_rng(3)
    u0 = rng.uniform(-1, 1, (len(T0S), 2, 1))
    w = 1.7
    pid = cabi.register_problem("forced_osc", "template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) { f[0] = cos(p[0] * t) - u[0]; }",
                                d=1, ode_order=2, num_params=1, time_dependent=True)  # fmt: skip
    got = _evaluate_at(cabi, pid, nu, u0, T0S, 1, 2, params=np.full((len(T0S), 1), w))
    want = np.zeros((len(T0S), nu + 1))
    want[:, 0], want[:, 1] = u0[:, 0, 0], u0[:, 1, 0]
    for k in range(nu - 1):
        want[:, k + 2] = np.cos(w * T0S + k * np.pi / 2) * w**k - want[:, k]
    _close("u'' = cos(w t) - u", got["taylor"][:, :, 0], want)


@pytest.mark.gpu
def test_a_hand_written_time_dependent_jacobian_matches_the_derived_one(cabi):
    body = """template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) {
  f[0] = sin(t) * (u[0] * u[1]);
  f[1] = cos(p[0] * t) * u[0] + t * u[1];
}"""
    jac = """
PN_DEV void jac(const double* u, double t, const double* p, double* J) {
  J[0] = sin(t) * u[1];
  J[1] = sin(t) * u[0];
  J[2] = cos(p[0] * t);
  J[3] = t;
}"""
    derived = cabi.register_problem("tv_system", body, d=2, num_params=1, time_dependent=True)
    hand = cabi.register_problem("tv_system_jac", body + jac, d=2, num_params=1, time_dependent=True)
    rng = np.random.default_rng(4)
    u0 = rng.uniform(-2, 2, (len(T0S), 1, 2))
    params = rng.uniform(0.5, 2, (len(T0S), 1))
    a = _evaluate_at(cabi, derived, 4, u0, T0S, 2, 1, params=params)
    b = _evaluate_at(cabi, hand, 4, u0, T0S, 2, 1, params=params)
    _same("f", a["f"], b["f"])
    _same("taylor", a["taylor"], b["taylor"])
    _close("jac", a["jac"], b["jac"])
    u, v = u0[:, 0, 0], u0[:, 0, 1]
    want = np.stack([np.sin(T0S) * v, np.sin(T0S) * u, np.cos(params[:, 0] * T0S), T0S], 1).reshape(-1, 2, 2)
    _close("jac (closed form)", b["jac"], want)


# ---- GPU: forced ODEs end to end ------------------------------------------------------------------------------------
def _truth(f, y0, save_at, args=()):
    return scipy.integrate.solve_ivp(f, (save_at[0], save_at[-1]), y0, t_eval=save_at, method="DOP853", rtol=1e-12, atol=1e-13,
                                     args=args).y.T  # fmt: skip


def _check_against_truth(name, u, u_std, truth, tol, max_ratio=10.0):
    err = np.abs(u - truth)
    assert err.max() <= 50 * tol * max(1.0, np.abs(truth).max()), f"{name}: max error {err.max():.3g}"
    ratio = err[1:] / u_std[1:]
    assert np.isfinite(u_std).all() and (u_std[1:] > 0).all()
    assert 1e-4 < np.median(ratio) < max_ratio, f"{name}: median error / std {np.median(ratio):.3g}"


def _duffing_rhs(t, y, delta, alpha, beta, gamma, w):
    return [y[1], gamma * np.cos(w * t) - delta * y[1] - alpha * y[0] - beta * y[0] ** 3]


@pytest.mark.gpu
@pytest.mark.parametrize("B", [300, 65536])
def test_forced_duffing_ensemble_with_per_member_frequency(cabi, B):
    import torch

    pid = cabi.register_problem("duffing", DUFFING, d=1, ode_order=2, num_params=5, time_dependent=True)
    rng = np.random.default_rng(7)
    tol, K = 1e-8, 9
    save_at = np.linspace(0.5, 4.5, K)
    u0 = np.stack([rng.uniform(-1, 1, B), rng.uniform(-0.5, 0.5, B)], 1).reshape(B, 2, 1)
    params = np.stack([np.full(B, 0.3), np.full(B, -1.0), np.ones(B), np.full(B, 0.5), rng.uniform(1.0, 1.4, B)], 1)
    desc = _desc(cabi, pid, 1, 4, 2, B, K, tol=tol, P=5)
    dev = torch.device("cuda:0")
    t = lambda x: torch.as_tensor(x, device=dev)  # noqa: E731
    out = cabi.solve_device(desc, t(u0), t(params), None, t(save_at), None)
    torch.cuda.synchronize()
    info = cabi.kernel_info(desc)
    if B == 300:
        assert info["threads_per_cta"] == 256  # the PAIR build
    else:
        assert info["grid"] * 128 < B  # the time-sliced build
    u, u_std, status = (out[k].cpu().numpy() for k in ("u", "u_std", "status"))
    assert (status == 0).all()
    for b in rng.choice(B, 12, replace=False):
        truth = _truth(_duffing_rhs, u0[b, :, 0], save_at, tuple(params[b]))[:, :1]
        _check_against_truth(f"duffing[{b}]", u[b], u_std[b], truth, tol)


@pytest.mark.gpu
@pytest.mark.parametrize("fact, corr, nu", [("isotropic", "ts0", 4), ("blockdiag", "ts0", 4), ("dense", "ts1", 3)])
def test_periodically_forced_lorenz96_through_the_builder_api(cabi, fact, corr, nu):
    from odecheckpts_b200 import ivps
    from odecheckpts_b200.probdiffeq import impl, ivpsolve, ivpsolvers, taylor

    w = 2.0

    def host(u, w_, t):
        return (np.roll(u, -1) - np.roll(u, 2)) * np.roll(u, 1) - u + 8.0 + np.sin(w_ * t)

    vf = ivps.cuda_vector_field("lorenz96_t", LORENZ96_T, d=8, num_params=1, time_dependent=True, host=host)
    tol = 1e-8
    u0 = (8.0 + np.array([1.0, 0.5, -1.0, 2.0, 0.0, -0.5, 1.5, -2.0]),)
    save_at = np.linspace(0.3, 0.8, 6)  # the flow is chaotic: a short horizon keeps the global error near tol
    impl.impl.select(fact, ode_shape=(8,))
    ibm = ivpsolvers.prior_ibm(num_derivatives=nu)
    correction = ivpsolvers.correction_ts1() if corr == "ts1" else ivpsolvers.correction_ts0()
    solver = ivpsolvers.solver_dynamic(ivpsolvers.strategy_fixedpoint(ibm, correction))
    asolver = ivpsolve.adaptive(solver, atol=tol, rtol=tol, control=ivpsolve.control_proportional_integral())
    field = lambda *y, t: vf(*y, t=t, p=(w,))  # noqa: E731
    tcoeffs = taylor.odejet_padded_scan(lambda *y: field(*y, t=save_at[0]), u0, num=nu)
    init = solver.initial_condition(tcoeffs, 1.0)
    sol = ivpsolve.solve_adaptive_save_at(field, init, save_at=save_at, dt0=1e-2, adaptive_solver=asolver)
    assert sol.status == 0
    truth = _truth(lambda t, y: host(y, w, t), u0[0], save_at)
    # the isotropic model shares one output scale among the eight components of a chaotic flow (as for the
    # autonomous Lorenz-96 of test_user_problems.py)
    _check_against_truth(f"forced lorenz96 {fact}", sol.u, sol.u_std, truth, tol, max_ratio=30.0 if fact == "isotropic" else 10.0)
    np.testing.assert_allclose(vf(u0[0], t=0.7, p=(w,)), host(u0[0], w, 0.7))


@pytest.mark.gpu
def test_textbook_smoother_agrees_with_the_checkpoint_solver(cabi):
    from odecheckpts_b200 import ivps, ivpsolvers
    from odecheckpts_b200.probdiffeq import ivpsolve

    w = 3.0
    vf = ivps.cuda_vector_field("forced_decay", FORCED_DECAY, d=1, num_params=1, time_dependent=True,
                                host=lambda u, w_, t: np.sin(w_ * t) - u)  # fmt: skip
    save_at = np.linspace(0.4, 4.4, 9)
    u0 = (np.array([0.8]),)
    tol = 1e-7
    dense, aux = ivpsolvers.solve_via_interpolate("ts0-4", vf, u0[0], save_at=save_at, dt0=0.1, atol=tol, rtol=tol)(u0, (w,))
    sol = aux["solution"]
    assert (np.asarray(sol.status) == 0).all() and len(sol.t) > 20
    # the same posterior through the fixed-point solver on the accepted grid (the fixed-grid build)
    ext = np.concatenate([[sol.t[0]], save_at, [sol.t[-1]]])
    ckpt = ivpsolve._solve_on_checkpoints(sol.posterior.context, ext)
    np.testing.assert_allclose(dense, ckpt.u[1:-1], rtol=1e-9, atol=1e-12)
    # and the solution of the ODE started at save_at[0] - 1e-6
    truth = _truth(lambda t, y: vf(y, t=t, p=(w,)), u0[0], np.concatenate([[save_at[0] - 1e-6], save_at]))[1:]
    assert np.abs(dense - truth).max() < 50 * tol
    # and the checkpoint solver from save_at[0]
    u, aux2 = ivpsolvers.solve("ts0-4", vf, u0[0], save_at, dt0=0.1, atol=tol, rtol=tol)(u0, (w,))
    _check_against_truth("forced decay", u, aux2["solution"].u_std, _truth(lambda t, y: vf(y, t=t, p=(w,)), u0[0], save_at), tol)
