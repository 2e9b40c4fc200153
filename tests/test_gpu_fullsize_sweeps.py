"""Full-size tolerance sweeps (BASELINE configs 3 and 4 as SURVEY 8d sizes them: 2,048 initial
conditions x 8 tolerances = 16,384 members in ONE launch, every member with its own tolerance).
The oracle only re-solves a small subsample (bit for bit); the rest is checked through properties."""

import numpy as np
import pytest

import problems_util as pu
from test_gpu_parity import _assert_bitwise, _desc, _ocfg, cabi  # noqa: F401

pytestmark = pytest.mark.gpu


N_IC = 2048
TOLS = 10.0 ** -np.arange(3, 11)


def _sweep(u0_ic, scale):
    """members ordered [ic][tol] like scripts/config_throughput.py; tol = (atol, rtol) per member"""
    n_ic = len(u0_ic)
    u0 = np.repeat(u0_ic[:, None], len(TOLS), 1).reshape((-1,) + u0_ic.shape[1:])
    rtol = np.tile(TOLS * scale, n_ic)
    return u0, np.stack([1e-3 * rtol, rtol], 1)


def _check_sweep_properties(res, n_tols):
    assert (res["status"] == 0).all()
    assert np.isfinite(res["u"]).all() and np.isfinite(res["u_std"]).all()
    acc = res["n_accepted"][:, -1].reshape(-1, n_tols)
    # tighter tolerance -> more accepted steps, for (almost) every initial condition
    assert (np.diff(acc, axis=1) > 0).mean() > 0.97
    assert np.median(acc[:, -1] / acc[:, 0]) > 8
    # terminal values converge: error against the tightest member shrinks along the sweep
    uT = res["u"][:, -1].reshape(acc.shape[0], n_tols, -1)
    err = np.sqrt(np.mean((uT - uT[:, -1:]) ** 2, axis=-1))[:, :-1]
    med = np.median(err, axis=0)
    assert (np.diff(med) < 0).all() and med[-1] < 1e-3 * med[0]


@pytest.mark.parametrize("fact,corr,nu", [("isotropic", "ts0", 4), ("isotropic", "ts0", 2), ("dense", "ts1", 4)])
def test_rigid_body_sweep_16384_members(cabi, oracle, fact, corr, nu):
    rng = np.random.default_rng(1)
    ic = (np.array([1.0, 0.0, 0.9]) + 0.05 * rng.standard_normal((N_IC, 3)))[:, None, :]
    u0, tol = _sweep(ic, 100.0)  # experiments/2_rigid_body/run_simple.py:40-42
    B, K = len(u0), 5
    par = np.tile(np.asarray(pu.RIGID_BODY_PARAMS), (B, 1))
    save_at = np.linspace(0, 50, K)
    kw = dict(dt0=50.0, P=3, fact=fact, corr=corr)
    res = cabi.solve_host(_desc(cabi, "rigid_body", 3, nu, 1, B, K, **kw), u0, par, tol, save_at, None)
    _check_sweep_properties(res, len(TOLS))
    # three initial conditions (24 members) re-solved by the CPU oracle: identical bits
    idx = np.concatenate([np.arange(8) + 8 * i for i in (0, 777, N_IC - 1)])
    ora = oracle.solve_save_at_batch(_ocfg(oracle, "rigid_body", 3, nu, 1, **kw), u0[idx], par[idx], save_at, tol=tol[idx])
    _assert_bitwise({k: v[idx] for k, v in res.items()}, ora)


@pytest.mark.parametrize("fact", ["blockdiag", "isotropic"])
def test_pleiades_sweep_16384_members(cabi, oracle, fact):
    rng = np.random.default_rng(2)
    x, dx = pu.pleiades_u0()
    pos = x + 0.01 * rng.standard_normal((N_IC, 14))
    ic = np.stack([pos, np.tile(dx, (N_IC, 1))], 1)
    u0, tol = _sweep(ic, 10.0)  # experiments/3_pleiades/run_harder.py:45-47
    B, K = len(u0), 50
    save_at = np.linspace(0, 3, K)
    kw = dict(dt0=0.1, fact=fact)
    res = cabi.solve_host(_desc(cabi, "pleiades", 14, 5, 2, B, K, **kw), u0, None, tol, save_at, None)
    _check_sweep_properties(res, len(TOLS))
    idx = np.arange(8) + 8 * 1234  # one initial condition, all eight tolerances
    # reduction_group=16: the lane-per-dimension kernel sums norms over 16 lanes as a butterfly
    ora = oracle.solve_save_at_batch(_ocfg(oracle, "pleiades", 14, 5, 2, reduction_group=16, **kw), u0[idx], None, save_at, tol=tol[idx])
    _assert_bitwise({k: v[idx] for k, v in res.items()}, ora)
