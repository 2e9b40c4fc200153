"""User-defined vector fields (ivps.cuda_vector_field / pn_b200_register_problem): registration and its errors,
family selection without compiling, the embedded headers, bit-identity of run-time compiled restatements of the
built-in problems with the built-in kernels, the Taylor arithmetic, and new ODEs solved end to end."""

import ctypes as C
import glob
import math
import os

import numpy as np
import pytest
import scipy.integrate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "code-adaptive-prob-ode-solvers_b200", "csrc")

# ---- sources ------------------------------------------------------------------------------------------------------
# form (b): the built-in functors restated, delegating to them
FULL_TEMPLATE = """
struct Problem {{
  static constexpr int D = pn::{t}::D, Q = pn::{t}::Q, P = pn::{t}::P, ID = 0;
  static constexpr bool HAS_JAC = pn::{t}::HAS_JAC;
  PN_DEV static void vf(const double* u, const double* p, double* f) {{ pn::{t}::vf(u, p, f); }}
  PN_DEV static void jac(const double* u, const double* p, double* J) {{ pn::{t}::jac(u, p, J); }}
  template <int N> PN_DEV static void vf_jet(const double* U, const double* p, double* F) {{ pn::{t}::vf_jet<N>(U, p, F); }}
}};
"""
# (type, d, q, P)
BUILTINS = {"van_der_pol": ("VanDerPol", 1, 2, 1), "rigid_body": ("RigidBody", 3, 1, 3), "pleiades": ("Pleiades", 14, 2, 0),
            "logistic": ("Logistic", 1, 1, 2), "three_body": ("ThreeBody", 2, 2, 1)}  # fmt: skip

# form (a): the same formulas on any number type, double arithmetic as in the built-ins
SIMPLE = {
    "logistic": "template <class T> PN_DEV void vf(const T* u, const double* p, T* f) { f[0] = (p[0] * u[0]) * fma(-p[1], u[0], 1.0); }",
    "van_der_pol": "template <class T> PN_DEV void vf(const T* u, const double* p, T* f) { f[0] = p[0] * fma(u[1], fma(-u[0], u[0], 1.0), -u[0]); }",
    "rigid_body": """template <class T> PN_DEV void vf(const T* u, const double* p, T* f) {
  f[0] = p[0] * (u[1] * u[2]);
  f[1] = p[1] * (u[0] * u[2]);
  f[2] = p[2] * (u[0] * u[1]);
}""",
    "three_body": """template <class T> PN_DEV T ipow32(const T& s) { return rcp(s * sqrt(s)); }
template <class T> PN_DEV void vf(const T* u, const double* p, T* f) {
  const double mu = p[0], mp = 1.0 - mu;
  const T x = u[0], y = u[1], xd = u[2], yd = u[3];
  const T a = x + mu, b = x - mp;
  const T p1 = ipow32(fma(y, y, a * a));
  const T p2 = ipow32(fma(y, y, b * b));
  f[0] = fma(-mu, b * p2, fma(-mp, a * p1, fma(2.0, yd, x)));
  f[1] = fma(-mu, y * p2, fma(-mp, y * p1, fma(-2.0, xd, y)));
}""",
}
LORENZ63 = """template <class T> PN_DEV void vf(const T* u, const double* p, T* f) {
  f[0] = p[0] * (u[1] - u[0]);
  f[1] = u[0] * (p[1] - u[2]) - u[1];
  f[2] = u[0] * u[1] - p[2] * u[2];
}"""
PENDULUM = "template <class T> PN_DEV void vf(const T* u, const double* p, T* f) { f[0] = -p[0] * sin(u[0]); }"
LORENZ96 = """template <class T> PN_DEV void vf(const T* u, const double* p, T* f) {
  for (int i = 0; i < 8; ++i) f[i] = (u[(i + 1) % 8] - u[(i + 6) % 8]) * u[(i + 7) % 8] - u[i] + p[0];
}"""


@pytest.fixture(scope="module")
def cabi():
    from odecheckpts_b200 import _cabi

    _cabi.lib()
    return _cabi


def _desc(cabi, problem, d, nu, q, B, K, *, fact="dense", corr="ts1", strat="fixedpoint", calib="dynamic", tol=1e-6, P=0,
          flags=0, cap=0):  # fmt: skip
    return cabi.Desc(problem, d, nu, q, cabi.FACTORISATIONS[fact], cabi.CORRECTIONS[corr], cabi.STRATEGIES[strat],
                     cabi.CALIBRATIONS[calib], tol, tol, 0.01, 0.95, 0.2, 10.0, 0.3, 0.4, B, K, 0, P, flags, cap)  # fmt: skip


def _full_id(cabi, name):
    t, d, q, P = BUILTINS[name]
    return cabi.register_problem(f"{name}_full", FULL_TEMPLATE.format(t=t), d=d, ode_order=q, num_params=P, form="full")


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_registration_compiles_both_forms(cabi):
    a = cabi.register_problem("vdp_simple", SIMPLE["van_der_pol"], d=1, ode_order=2, num_params=1)
    b = _full_id(cabi, "van_der_pol")
    assert a >= cabi.USER_PROBLEM_BASE and b >= cabi.USER_PROBLEM_BASE and a != b
    # the same registration again is the same problem
    assert cabi.register_problem("vdp_simple", SIMPLE["van_der_pol"], d=1, ode_order=2, num_params=1) == a


def test_a_compile_error_names_the_users_line(cabi):
    src = "template <class T> PN_DEV void vf(const T* u, const double* p, T* f) {\n  f[0] = u[0];\n  f[0] = u[0] +;\n}\n"
    with pytest.raises(ValueError) as e:
        cabi.register_problem("broken_field", src, d=1)
    assert "broken_field(3): error" in str(e.value)
    assert cabi.lib().pn_b200_register_problem(b"broken_field", src.encode(), 0, 1, 1, 0, C.byref(C.c_int32())) == -2
    # the whole log, not a truncated line
    assert "f[0] = u[0] +;" in cabi.lib().pn_b200_last_error().decode()


def test_a_form_b_problem_of_the_wrong_size_is_rejected(cabi):
    with pytest.raises(ValueError, match="differs from the registered d"):
        cabi.register_problem("vdp_wrong_d", FULL_TEMPLATE.format(t="VanDerPol"), d=2, ode_order=2, num_params=1, form="full")


@pytest.mark.parametrize("kw", [dict(d=0), dict(d=33), dict(ode_order=0), dict(ode_order=3), dict(num_params=-1),
                                dict(num_params=65), dict(form="other"), dict(name=""), dict(name='a"b'),
                                dict(name="x" * 129)])  # fmt: skip
def test_bad_sizes_and_names_are_rejected(cabi, kw):
    args = dict(name="ok_name", d=1, ode_order=1, num_params=0, form="simple") | kw
    name = args.pop("name")
    with pytest.raises(ValueError):
        cabi.register_problem(name, "template <class T> PN_DEV void vf(const T* u, const double* p, T* f) { f[0] = u[0]; }", **args)


@pytest.mark.parametrize(
    "d, fact, corr, nu, ok",
    [(1, "isotropic", "ts0", 4, True), (1, "dense", "ts1", 4, True), (3, "isotropic", "ts0", 4, True),
     (3, "blockdiag", "ts0", 4, True), (3, "dense", "ts1", 4, True), (3, "isotropic", "ts1", 4, False),
     (8, "isotropic", "ts0", 8, True), (8, "blockdiag", "ts0", 4, True), (8, "dense", "ts1", 3, True),
     (8, "dense", "ts1", 4, False), (32, "blockdiag", "ts0", 4, True), (32, "dense", "ts0", 1, False)],
)  # fmt: skip
def test_supported_follows_the_family_rules_and_does_not_compile(cabi, d, fact, corr, nu, ok):
    src = f"template <class T> PN_DEV void vf(const T* u, const double* p, T* f) {{ for (int i = 0; i < {d}; ++i) f[i] = -u[i]; }}"
    pid = cabi.register_problem(f"decay{d}", src, d=d)
    before = cabi.lib().pn_b200_jit_module_count()
    for strat in ("fixedpoint", "filter"):
        desc = _desc(cabi, pid, d, nu, 1, 1000, 10, fact=fact, corr=corr, strat=strat)
        assert cabi.supported(desc) == ok
        if ok:
            assert cabi.workspace_bytes(desc) > 0
        desc.d = d + 1  # the registered dimension only
        assert not cabi.supported(desc)
    assert cabi.lib().pn_b200_jit_module_count() == before


def test_embedded_sources_match_csrc(cabi):
    cabi.lib().pn_b200_jit_source.restype = C.c_char_p
    headers = sorted(glob.glob(os.path.join(CSRC, "*.cuh")))
    assert any(h.endswith("pn_user_problem.cuh") for h in headers)
    for h in headers:
        with open(h, encoding="utf-8") as f:
            text = f.read()
        assert cabi.lib().pn_b200_jit_source(os.path.basename(h).encode()).decode() == text, h


def test_python_callables_point_to_cuda_vector_field():
    from odecheckpts_b200 import ivps

    with pytest.raises(TypeError, match="cuda_vector_field"):
        ivps.resolve_vector_field(lambda u, t: -u, (np.ones(2),))


# ---- GPU: bit-identity with the built-in kernels ------------------------------------------------------------------
def _same(name, a, b):
    assert a.shape == b.shape, name
    assert np.array_equal(a, b, equal_nan=True), f"{name}: {np.sum(a != b)} of {a.size} entries differ"


def _solve_all(cabi, desc, u0, params, save_at, *, samples=True, lml=True):
    """Every output of a solve, plus samples and the likelihood where the strategy has them (numpy)."""
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


def _compare_with_builtin(cabi, name, builtin_id, desc, u0, params, save_at, **kw):
    user = _solve_all(cabi, desc, u0, params, save_at, **kw)
    info_user = cabi.kernel_info(desc)
    desc.problem = builtin_id
    ref = _solve_all(cabi, desc, u0, params, save_at, **kw)
    assert user.keys() == ref.keys()
    for key in ref:
        _same(f"{name}: {key}", user[key], ref[key])
    assert (ref["status"] == 0).all()
    return user, info_user


def _vdp_members(B, mu=1e3, seed=0):
    rng = np.random.default_rng(seed)
    u0 = np.stack([2.0 + 0.5 * rng.uniform(-1, 1, B), 0.5 * rng.uniform(-1, 1, B)], 1).reshape(B, 2, 1)
    return u0, np.full((B, 1), mu)


@pytest.mark.gpu
def test_van_der_pol_dense_ekf1_fixedpoint_headline_shape_bitwise(cabi):
    """More members than resident lanes: the time-sliced build of the thread-per-IVP kernel."""
    B, K = 65536, 20
    u0, params = _vdp_members(B)
    desc = _desc(cabi, _full_id(cabi, "van_der_pol"), 1, 4, 2, B, K, tol=1e-3, P=1)
    _, info = _compare_with_builtin(cabi, "vdp headline", 5, desc, u0, params, np.linspace(0.0, 6.3, K))
    assert info["grid"] * 128 < B and info["local_bytes_per_thread"] < 256


@pytest.mark.gpu
def test_van_der_pol_small_ensemble_pair_build_bitwise(cabi):
    B, K = 300, 12
    u0, params = _vdp_members(B, seed=3)
    desc = _desc(cabi, _full_id(cabi, "van_der_pol"), 1, 4, 2, B, K, tol=1e-5, P=1)
    _, info = _compare_with_builtin(cabi, "vdp pair", 5, desc, u0, params, np.linspace(0.0, 2.0, K))
    assert info["threads_per_cta"] == 256  # 128 filter lanes + 128 backward lanes


@pytest.mark.gpu
def test_van_der_pol_filter_with_trajectory_recording_bitwise(cabi):
    B, K, cap = 64, 6, 3000
    u0, params = _vdp_members(B, mu=10.0, seed=4)
    desc = _desc(cabi, _full_id(cabi, "van_der_pol"), 1, 3, 2, B, K, strat="filter", tol=1e-5, P=1, flags=cabi.FLAG_RECORD, cap=cap)
    user, _ = _compare_with_builtin(cabi, "vdp filter", 5, desc, u0, params, np.linspace(0.0, 3.0, K))
    assert user["traj_len"].min() > 10


@pytest.mark.gpu
@pytest.mark.parametrize("fact, corr", [("blockdiag", "ts0"), ("dense", "ts1")])
def test_rigid_body_lane_per_dimension_and_register_columns_bitwise(cabi, fact, corr):
    B, K = 500, 10
    rng = np.random.default_rng(1)
    u0 = (np.array([1.0, 0.0, 0.9]) + 0.1 * rng.uniform(-1, 1, (B, 3))).reshape(B, 1, 3)
    params = np.tile([-2.0, 1.25, -0.5], (B, 1))
    desc = _desc(cabi, _full_id(cabi, "rigid_body"), 3, 4, 1, B, K, fact=fact, corr=corr, tol=1e-7, P=3)
    _compare_with_builtin(cabi, f"rigid body {fact}", 1, desc, u0, params, np.linspace(0.0, 5.0, K), lml=fact != "dense")


@pytest.mark.gpu
def test_pleiades_isotropic_lane_per_dimension_bitwise(cabi):
    from problems_util import pleiades_u0

    B, K = 40, 8
    rng = np.random.default_rng(2)
    u0 = pleiades_u0()[None] + 0.01 * rng.uniform(-1, 1, (B, 2, 14))
    desc = _desc(cabi, _full_id(cabi, "pleiades"), 14, 4, 2, B, K, fact="isotropic", corr="ts0", tol=1e-6)
    _compare_with_builtin(cabi, "pleiades", 3, desc, u0, None, np.linspace(0.0, 3.0, K))


# ---- GPU: derivatives ---------------------------------------------------------------------------------------------
def _evaluate(cabi, pid, nu, u0, params, d, q, jac=True):
    import torch

    dev = torch.device("cuda:0")
    p = None if params is None else torch.as_tensor(params, device=dev)
    out = cabi.problem_evaluate_device(pid, nu, torch.as_tensor(u0, device=dev), p, d=d, ode_order=q, jac=jac)
    return {k: v.cpu().numpy() for k, v in out.items()}


def _close(name, got, ref, rel=1e-13, per_state=True):
    """|got - ref| <= rel * the largest |ref| of the state (per_state) or of the whole batch"""
    scale = np.abs(ref).reshape(ref.shape[0], -1).max(axis=1).reshape((-1,) + (1,) * (ref.ndim - 1))
    if not per_state:
        scale = np.abs(ref).max()
    err = np.abs(got - ref)
    assert (err <= rel * np.maximum(scale, 1e-300)).all(), f"{name}: max relative error {(err / scale).max():.3g}"


@pytest.mark.gpu
@pytest.mark.parametrize("name, builtin_id", [("logistic", 0), ("van_der_pol", 5), ("rigid_body", 1), ("three_body", 2)])
def test_derived_taylor_coefficients_and_jacobian_match_the_hand_written_ones(cabi, name, builtin_id):
    _, d, q, P = BUILTINS[name]
    pid = cabi.register_problem(f"{name}_simple", SIMPLE[name], d=d, ode_order=q, num_params=P)
    rng = np.random.default_rng(11)
    n = 256
    if name == "three_body":
        u0 = np.array([[0.994, 0.0], [0.0, -2.0015851063790825]]) + 0.05 * rng.uniform(-1, 1, (n, 2, 2))
        params = np.full((n, 1), 0.012277471)
    else:
        u0 = rng.uniform(0.2, 1.5, (n, q, d))
        params = rng.uniform(0.5, 2.0, (n, P))
    for nu in (1, 4, 8):
        got = _evaluate(cabi, pid, nu, u0, params, d, q)
        ref = _evaluate(cabi, builtin_id, nu, u0, params, d, q)
        _same(f"{name} vf", got["f"], ref["f"])
        _close(f"{name} taylor nu={nu}", got["taylor"], ref["taylor"])
        # a Jacobian entry can be a difference of nearly equal terms (logistic: a (1 - 2 b u)): batch scale
        _close(f"{name} jac", got["jac"], ref["jac"], per_state=False)


def _taylor_of(cabi, body, u0, nu, q=1):
    src = "template <class T> PN_DEV void vf(const T* u, const double* p, T* f) { " + body + " }"
    pid = cabi.register_problem("jet_" + str(abs(hash(body))), src, d=1, ode_order=q)
    return _evaluate(cabi, pid, nu, np.asarray(u0, dtype=np.float64).reshape(-1, q, 1), None, 1, q)["taylor"][:, :, 0]


@pytest.mark.gpu
def test_jet_primitives_against_closed_form_series(cabi):
    nu = 8
    k = np.arange(nu + 1)
    fact = np.array([math.factorial(i) for i in k], dtype=np.float64)
    u0 = np.array([0.3, 0.5, 1.7])
    # u' = u^2: u^(k) = k! u0^(k+1)   (product, integer power)
    want = fact[None] * u0[:, None] ** (k[None] + 1)
    for body in ("f[0] = u[0] * u[0];", "f[0] = pow(u[0], 2);"):
        _close(body, _taylor_of(cabi, body, u0, nu), want, 1e-14)
    # u' = u^1.5: u = (a - t/2)^-2, a = u0^-1/2:  u^(k) = (k+1)! 2^-k a^(-2-k)   (real power)
    a = u0 ** -0.5
    _close("u^1.5", _taylor_of(cabi, "f[0] = pow(u[0], 1.5);", u0, nu), fact[None] * (k[None] + 1) * 0.5 ** k[None] * a[:, None] ** (-2.0 - k[None]), 1e-13)
    # u' = exp(u): u = -log(e^-u0 - t):  u^(k) = (k-1)! e^(k u0), k >= 1
    want = np.concatenate([u0[:, None], fact[None, :-1] * np.exp(k[None, 1:] * u0[:, None])], 1)
    _close("exp", _taylor_of(cabi, "f[0] = exp(u[0]);", u0, nu), want, 1e-13)
    # u' = 1 / u: u = sqrt(u0^2 + 2 t):  u^(k) = prod_{j<k} (1/2 - j) 2^k u0^(1 - 2k)   (division and reciprocal)
    c = np.array([np.prod([0.5 - j for j in range(i)]) * 2.0**i for i in k])
    want = c[None] * u0[:, None] ** (1.0 - 2 * k[None])
    for body in ("f[0] = 1.0 / u[0];", "f[0] = rcp(u[0]);"):
        _close(body, _taylor_of(cabi, body, u0, nu), want, 1e-13)
    # u' = sqrt(u): u = (sqrt(u0) + t/2)^2
    want = np.zeros((3, nu + 1))
    want[:, 0], want[:, 1], want[:, 2] = u0, np.sqrt(u0), 0.5
    _close("sqrt", _taylor_of(cabi, "f[0] = sqrt(u[0]);", u0, nu), want, 1e-14)
    # u' = log(exp(u)) - u + 1 = 1
    want = np.zeros((3, nu + 1))
    want[:, 0], want[:, 1] = u0, 1.0
    _close("log(exp)", _taylor_of(cabi, "f[0] = log(exp(u[0])) - u[0] + 1.0;", u0, nu), want, 1e-13)
    # u' = cos(u): u'' = -sin u cos u, u''' = -cos(2u) cos(u)
    s, co = np.sin(u0), np.cos(u0)
    got = _taylor_of(cabi, "f[0] = cos(u[0]);", u0, 3)
    _close("cos", got, np.stack([u0, co, -s * co, -np.cos(2 * u0) * co], 1), 1e-14)
    # pendulum u'' = -sin(u): u''' = -cos(u) u', u'''' = sin(u) u'^2 - cos(u) u''
    y0 = np.stack([u0, 0.3 * np.ones(3)], 1)
    got = _taylor_of(cabi, "f[0] = -sin(u[0]);", y0, 4, q=2)
    y, yd = y0[:, 0], y0[:, 1]
    ydd = -np.sin(y)
    _close("sin", got, np.stack([y, yd, ydd, -np.cos(y) * yd, np.sin(y) * yd**2 - np.cos(y) * ydd], 1), 1e-14)


# ---- GPU: new ODEs end to end -------------------------------------------------------------------------------------
def _truth(f, y0, save_at, args):
    return scipy.integrate.solve_ivp(f, (save_at[0], save_at[-1]), y0, t_eval=save_at, method="DOP853", rtol=1e-13, atol=1e-13,
                                     args=args).y.T  # fmt: skip


def _check_against_truth(name, u, u_std, truth, tol, max_ratio=10.0):
    err = np.abs(u - truth)
    assert err.max() <= 50 * tol * max(1.0, np.abs(truth).max()), f"{name}: max error {err.max():.3g}"
    # calibration: the posterior standard deviations are neither vanishing nor orders of magnitude too large
    ratio = err[1:] / u_std[1:]
    assert np.isfinite(u_std).all() and (u_std[1:] > 0).all()
    assert 1e-4 < np.median(ratio) < max_ratio, f"{name}: median error / std {np.median(ratio):.3g}"


@pytest.mark.gpu
def test_lorenz63_ensemble_with_per_member_parameters(cabi):
    from odecheckpts_b200 import ivps, ivpsolvers

    def host(u, s, r, b):
        return np.stack([s * (u[..., 1] - u[..., 0]), u[..., 0] * (r - u[..., 2]) - u[..., 1], u[..., 0] * u[..., 1] - b * u[..., 2]], -1)

    vf = ivps.cuda_vector_field("lorenz63", LORENZ63, d=3, num_params=3, host=host)
    B, tol = 16, 1e-8
    rng = np.random.default_rng(5)
    u0 = np.array([1.0, 1.0, 1.0]) + 0.1 * rng.uniform(-1, 1, (B, 3))
    sigma, rho, beta = 10.0 + rng.uniform(-1, 1, B), 28.0 + rng.uniform(-2, 2, B), np.full(B, 8.0 / 3.0)
    save_at = np.linspace(0.0, 1.0, 11)
    solve = ivpsolvers.solve("ts0-5", vf, (u0[0],), save_at, dt0=1e-3, atol=tol, rtol=tol)
    u, aux = solve((u0,), (sigma, rho, beta))
    sol = aux["solution"]
    assert (np.asarray(sol.status) == 0).all()
    for b in range(B):
        truth = _truth(lambda t, y, *p: host(y, *p), u0[b], save_at, (sigma[b], rho[b], beta[b]))
        _check_against_truth(f"lorenz63[{b}]", u[b], sol.u_std[b], truth, tol)
    np.testing.assert_allclose(vf(u0[0], p=(sigma[0], rho[0], beta[0])), host(u0[0], sigma[0], rho[0], beta[0]))


@pytest.mark.gpu
def test_pendulum_second_order(cabi):
    from odecheckpts_b200 import ivps, ivpsolvers

    vf = ivps.cuda_vector_field("pendulum", PENDULUM, d=1, ode_order=2, num_params=1)
    tol = 1e-9
    save_at = np.linspace(0.0, 10.0, 21)
    u0, du0 = np.array([2.5]), np.array([0.0])
    u, aux = ivpsolvers.solve("ts0-6", vf, (u0, du0), save_at, dt0=1e-2, atol=tol, rtol=tol, ode_order=2)((u0, du0), (9.81,))
    truth = _truth(lambda t, y: [y[1], -9.81 * np.sin(y[0])], [2.5, 0.0], save_at, ())[:, :1]
    _check_against_truth("pendulum", u, aux["solution"].u_std, truth, tol)


@pytest.mark.gpu
@pytest.mark.parametrize("fact, corr, nu", [("isotropic", "ts0", 4), ("blockdiag", "ts0", 4), ("dense", "ts1", 3)])
def test_lorenz96_through_the_builder_api(cabi, fact, corr, nu):
    from odecheckpts_b200 import ivps
    from odecheckpts_b200.probdiffeq import impl, ivpsolve, ivpsolvers, stats, taylor

    vf = ivps.cuda_vector_field("lorenz96", LORENZ96, d=8, num_params=1)
    tol, F = 1e-8, 8.0
    u0 = (F + np.array([1.0, 0.5, -1.0, 2.0, 0.0, -0.5, 1.5, -2.0]),)
    save_at = np.linspace(0.0, 0.5, 6)  # the flow is chaotic: a short horizon keeps the global error near tol
    impl.impl.select(fact, ode_shape=(8,))
    ibm = ivpsolvers.prior_ibm(num_derivatives=nu)
    correction = ivpsolvers.correction_ts1() if corr == "ts1" else ivpsolvers.correction_ts0()
    solver = ivpsolvers.solver_dynamic(ivpsolvers.strategy_fixedpoint(ibm, correction))
    asolver = ivpsolve.adaptive(solver, atol=tol, rtol=tol, control=ivpsolve.control_proportional_integral())
    tcoeffs = taylor.odejet_padded_scan(lambda *y: vf(*y, t=0.0, p=(F,)), u0, num=nu)
    init = solver.initial_condition(tcoeffs, 1.0)
    sol = ivpsolve.solve_adaptive_save_at(lambda *y, t: vf(*y, t=t, p=(F,)), init, save_at=save_at, dt0=1e-2, adaptive_solver=asolver)
    assert sol.status == 0

    def f(t, y):
        return (np.roll(y, -1) - np.roll(y, 2)) * np.roll(y, 1) - y + F

    truth = _truth(f, u0[0], save_at, ())
    # the isotropic model shares one output scale among the eight components of a chaotic flow: its standard
    # deviations are the least faithful (median error / std 10.1 on a B200, against 1e-3 ... 10 elsewhere)
    _check_against_truth(f"lorenz96 {fact}", sol.u, sol.u_std, truth, tol, max_ratio=30.0 if fact == "isotropic" else 10.0)
    post = stats.markov_select_terminal(sol.posterior)
    margs = stats.markov_marginals(post, reverse=True)
    np.testing.assert_array_equal(np.concatenate([margs.mean, sol.posterior.init.mean[[-1], ...]])[:, 0, :], sol.u)
