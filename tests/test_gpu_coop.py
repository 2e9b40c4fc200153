"""Small ensembles of the d = 1 problems: the build the library picks (for the fixed-point strategy the PAIR build,
a backward lane per IVP) bit for bit against the CPU oracle AND against the plain thread-per-IVP kernel."""

import os

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


class _thread_per_ivp:
    """Forces the plain thread-per-IVP kernel for the calls inside (the library reads the variable per call)."""

    def __enter__(self):
        self.old = os.environ.get("PN_B200_PAIR")
        os.environ["PN_B200_PAIR"] = "0"

    def __exit__(self, *exc):
        if self.old is None:
            del os.environ["PN_B200_PAIR"]
        else:
            os.environ["PN_B200_PAIR"] = self.old


def _desc(cabi, problem, nu, q, B, K, *, fact="dense", corr="ts1", strat="fixedpoint", calib="dynamic", atol=1e-6, rtol=1e-6,
          dt0=0.01, P=1, flags=0, cap=0):  # fmt: skip
    return cabi.Desc(cabi.PROBLEM_IDS[problem], 1, nu, q, cabi.FACTORISATIONS[fact], cabi.CORRECTIONS[corr],
                     cabi.STRATEGIES[strat], cabi.CALIBRATIONS[calib], atol, rtol, dt0, 0.95, 0.2, 10.0, 0.3, 0.4,
                     B, K, 0, P, flags, cap)  # fmt: skip


def _same(name, a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, name
    ok = (a == b) | (np.isnan(a.astype(float)) & np.isnan(b.astype(float)))
    if not ok.all():
        bad = tuple(np.argwhere(~ok)[0])
        raise AssertionError(f"{name}: {(~ok).sum()} of {ok.size} differ, first at {bad}: {a[bad]!r} vs {b[bad]!r}")


def _vdp_members(B, seed=0):
    rng = np.random.default_rng(seed)
    ab = rng.uniform(-1, 1, (B, 2))
    u0 = np.stack([2.0 + 0.5 * ab[:, 0], 0.5 * ab[:, 1]], 1).reshape(B, 2, 1)
    u0[0] = [[2.0], [0.0]]
    return u0, np.full((B, 1), 1e3)


@pytest.mark.parametrize("B,tol,strat,corr,calib,nu", [
    (1, 1e-3, "fixedpoint", "ts1", "dynamic", 4), (7, 1e-3, "fixedpoint", "ts1", "dynamic", 4), (64, 1e-6, "fixedpoint", "ts1", "dynamic", 4),
    (13, 1e-4, "filter", "ts1", "dynamic", 4), (9, 1e-4, "fixedpoint", "ts0", "none", 4), (11, 1e-3, "fixedpoint", "ts1", "dynamic", 2),
])  # fmt: skip
def test_van_der_pol_bitwise_against_the_oracle_and_the_thread_per_ivp_kernel(cabi, oracle, B, tol, strat, corr, calib, nu):
    K = 20
    u0, params = _vdp_members(B)
    save_at = np.linspace(0.0, 6.3, K)
    kw = dict(corr=corr, strat=strat, calib=calib, atol=tol, rtol=tol)
    desc = _desc(cabi, "van_der_pol", nu, 2, B, K, **kw)
    got = cabi.solve_host(desc, u0, params, None, save_at, None, full=True)
    with _thread_per_ivp():
        ref = cabi.solve_host(desc, u0, params, None, save_at, None, full=True)
    cfg = oracle.make_config("van_der_pol", 1, nu, 2, factorisation="dense", correction=corr, strategy=strat, calibration=calib,
                             atol=tol, rtol=tol, dt0=0.01, num_params=1)  # fmt: skip
    ora = oracle.solve_save_at_batch(cfg, u0, params, save_at)
    assert (ora["status"] == 0).all() and ora["n_accepted"][:, -1].min() > 100
    for key in ("status", "n_accepted", "n_rejected", "u", "u_std"):
        _same(key + " (oracle)", got[key], ora[key])
    for key in ("status", "n_accepted", "n_rejected", "u", "u_std", "marg_mean", "marg_chol", "output_scale"):
        _same(key + " (thread-per-IVP kernel)", got[key], ref[key])


def test_per_member_tolerances_and_more_members_than_groups(cabi, oracle):
    B, K = 4000, 8
    u0, params = _vdp_members(B, seed=5)
    tol = np.stack([10.0 ** -np.random.default_rng(1).integers(2, 5, B).astype(float)] * 2, 1)
    save_at = np.linspace(0.0, 1.0, K)
    desc = _desc(cabi, "van_der_pol", 4, 2, B, K)
    got = cabi.solve_host(desc, u0, params, tol, save_at, None)
    with _thread_per_ivp():
        ref = cabi.solve_host(desc, u0, params, tol, save_at, None)
    cfg = oracle.make_config("van_der_pol", 1, 4, 2, factorisation="dense", correction="ts1", atol=1e-6, rtol=1e-6,
                             dt0=0.01, num_params=1)  # fmt: skip
    ora = oracle.solve_save_at_batch(cfg, u0, params, save_at, tol=tol)
    for key in ("status", "n_accepted", "n_rejected", "u", "u_std"):
        _same(key, got[key], ref[key])
        _same(key + " (oracle)", got[key], ora[key])
    assert (got["status"] == 0).all()


def test_logistic_and_fixed_grid(cabi, oracle):
    save_at = np.linspace(0.0, 2.5, 7)
    for nu in (2, 4):
        desc = _desc(cabi, "logistic", nu, 1, 3, len(save_at), fact="isotropic", corr="ts0", atol=1e-5, rtol=1e-5, dt0=0.1, P=2)
        u0 = np.array([0.1, 0.2, 0.05]).reshape(3, 1, 1)
        par = np.tile([1.0, 1.0], (3, 1))
        got = cabi.solve_host(desc, u0, par, None, save_at, None)
        cfg = oracle.make_config("logistic", 1, nu, 1, atol=1e-5, rtol=1e-5, dt0=0.1, num_params=2)
        ora = oracle.solve_save_at_batch(cfg, u0, par, save_at)
        for key in ("status", "n_accepted", "n_rejected", "u", "u_std"):
            _same(key, got[key], ora[key])
        np.testing.assert_allclose(got["u"][0, :, 0], pu.logistic_exact(save_at), rtol=1e-3)
    # solve_fixed_grid (vdp.py:88-91): the steps are given, no rejection
    grid = np.linspace(0.0, 0.02, 30)
    desc = _desc(cabi, "van_der_pol", 4, 2, 1, len(grid), strat="filter", flags=cabi.FLAG_FIXED_GRID)
    got = cabi.solve_host(desc, pu.van_der_pol_u0()[None], np.array([[1e3]]), None, grid, None)
    cfg = oracle.make_config("van_der_pol", 1, 4, 2, factorisation="dense", correction="ts1", strategy="filter", num_params=1)
    ora = oracle.solve_fixed_grid(cfg, pu.van_der_pol_u0(), [1e3], grid)
    _same("u", got["u"][0], ora["u"])
    _same("u_std", got["u_std"][0], ora["u_std"])


def test_save_every_step_recording(cabi, goldens):
    """solve_adaptive_save_every_step (vdp.py:77-79): the recorded grid is the same whichever thread-per-IVP build
    runs, and starts like the reference's golden grid."""
    cap = 4096
    desc = _desc(cabi, "van_der_pol", 4, 2, 1, 2, strat="filter", atol=1e-3, rtol=1e-3, flags=cabi.FLAG_RECORD, cap=cap)
    args = (pu.van_der_pol_u0()[None], np.array([[1e3]]), None, np.array([0.0, 6.3]), None)
    got = cabi.solve_host(desc, *args)
    with _thread_per_ivp():
        ref = cabi.solve_host(desc, *args)
    n = int(got["traj_len"][0])
    assert n == int(ref["traj_len"][0]) and 2800 < n < 3000
    for key in ("traj_t", "traj_u", "traj_std"):
        _same(key, got[key][:n], ref[key][:n])
    np.testing.assert_allclose(got["traj_t"][:20, 0], goldens["vdp_grid"][:20], rtol=1e-12)


def test_sampling_and_likelihood_kernels_read_the_pair_builds_workspace(cabi):
    import torch

    B, K = 5, 12
    u0, params = _vdp_members(B)
    save_at = np.linspace(0.0, 2.0, K)
    desc = _desc(cabi, "van_der_pol", 4, 2, B, K, atol=1e-4, rtol=1e-4)
    dev = torch.device("cuda")
    T = lambda x: torch.as_tensor(x, device=dev)  # noqa: E731
    outs = []
    for force in (False, True):
        ctx = _thread_per_ivp() if force else None
        if ctx:
            ctx.__enter__()
        try:
            out = cabi.solve_device(desc, T(u0), T(params), None, T(save_at), None)
            data = out["u"].clone()
            lml = cabi.log_marginal_likelihood_device(desc, out["_workspace"], out["status"], data, 0.1)
            smp = cabi.markov_sample_device(desc, out["_workspace"], out["status"], 7, 3)
            torch.cuda.synchronize()
            outs.append((lml.cpu().numpy(), smp.cpu().numpy()))
        finally:
            if ctx:
                ctx.__exit__()
    _same("lml", outs[0][0], outs[1][0])
    _same("samples", outs[0][1], outs[1][1])
