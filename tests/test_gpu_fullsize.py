"""Full-size (BASELINE configs[1]: 65,536-member Van der Pol ensemble) checks through properties
that need no oracle run: the oracle would take minutes at this size, the properties take one launch."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def full_run():
    import torch

    import bench
    from odecheckpts_b200 import _cabi

    B, K = bench.MEMBERS, bench.K_CHECKPOINTS
    u0, par = bench.ensemble_inputs(0, B)
    save_at = np.linspace(bench.T0, bench.T1, K)
    desc = _cabi.Desc(5, 1, 4, 2, 2, 1, 1, 1, bench.TOL, bench.TOL, 0.01, 0.95, 0.2, 10.0, 0.3, 0.4, B, K, 0, 1, 0, 0)
    dev = torch.device("cuda:0")
    args = (torch.as_tensor(u0, device=dev), torch.as_tensor(par, device=dev), None, torch.as_tensor(save_at, device=dev), None)
    out = _cabi.solve_device(desc, *args)
    res = {k: v.cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    return _cabi, desc, u0, par, save_at, res


def test_full_ensemble_is_healthy(full_run):
    _, _, u0, _, _, res = full_run
    assert (res["status"] == 0).all()
    assert np.isfinite(res["u"]).all() and np.isfinite(res["u_std"]).all() and (res["u_std"] >= 0).all()
    # accepted counts are cumulative over the checkpoints
    assert (np.diff(res["n_accepted"], axis=1) >= 0).all() and (res["n_accepted"][:, 0] == 0).all()
    acc = res["n_accepted"][:, -1]
    assert 11000 < acc.min() and acc.max() < 20000 and 14500 < acc.mean() < 16000  # SURVEY 8d: ~15.3k accepted per member
    assert 500 < res["n_rejected"].mean() < 1500


def test_smoothing_back_to_t0_reproduces_the_initial_values(full_run):
    # SURVEY App. A.6: marginalising the checkpoint Markov chain back to t0 returns u0 (a free self-check
    # of every one of the 49 merged backward conditionals of every member)
    _, _, u0, _, _, res = full_run
    np.testing.assert_allclose(res["u"][:, 0, 0], u0[:, 0, 0], rtol=0, atol=1e-12)
    assert res["u_std"][:, 0, 0].max() < 1e-6


def test_members_do_not_depend_on_their_neighbours_or_the_schedule(full_run):
    # solving a member alone, in a different slot, or in a second launch gives the same bits:
    # the lane-level ticket queue makes the member->lane assignment timing dependent
    import torch

    _cabi, desc, u0, par, save_at, res = full_run
    idx = np.array([0, 1, 31, 32, 4095, 37888, 65535])
    d2 = _cabi.Desc(*[getattr(desc, n) for n, _ in _cabi.Desc._fields_])
    d2.batch = len(idx)
    sub = _cabi.solve_host(d2, u0[idx], par[idx], None, save_at, None)
    for key in ("u", "u_std", "n_accepted", "n_rejected", "status"):
        np.testing.assert_array_equal(sub[key], res[key][idx])
    perm = np.random.default_rng(5).permutation(desc.batch)[:8192]
    d3 = _cabi.Desc(*[getattr(desc, n) for n, _ in _cabi.Desc._fields_])
    d3.batch = len(perm)
    again = _cabi.solve_host(d3, u0[perm], par[perm], None, save_at, None)
    np.testing.assert_array_equal(again["u"], res["u"][perm])
    np.testing.assert_array_equal(again["n_rejected"], res["n_rejected"][perm])


def test_solution_stays_on_the_limit_cycle_and_agrees_with_a_tighter_solve(full_run):
    _cabi, desc, u0, par, save_at, res = full_run
    assert np.abs(res["u"]).max() < 2.6  # |u| <= ~2.0 on the Van der Pol limit cycle, ICs within 2 +- 0.5
    idx = np.arange(0, desc.batch, 4099)
    d2 = _cabi.Desc(*[getattr(desc, n) for n, _ in _cabi.Desc._fields_])
    d2.batch = len(idx)
    d2.atol = d2.rtol = 1e-9
    tight = _cabi.solve_host(d2, u0[idx], par[idx], None, save_at, None)
    # away from the relaxation jumps (|u'| ~ 1e3) the 1e-6 solve is within ~1e-4 of the 1e-9 one
    err = np.abs(tight["u"] - res["u"][idx])[:, :, 0]
    assert np.median(err) < 1e-5 and np.quantile(err, 0.9) < 1e-3


def test_time_sliced_scheduling_does_not_change_a_single_bit(full_run, monkeypatch):
    # 65,536 members on 37,888 resident lanes: the launch above ran time-sliced (members are parked
    # and taken over by other lanes).  Unsliced, and sliced with a tiny quantum (hundreds of hand-overs
    # per member), must give the same bits.
    import torch

    _cabi, desc, u0, par, save_at, res = full_run
    dev = torch.device("cuda:0")
    B = 40960  # just above the resident lanes: still sliced, cheaper to repeat
    d2 = _cabi.Desc(*[getattr(desc, n) for n, _ in _cabi.Desc._fields_])
    d2.batch = B
    args = (torch.as_tensor(u0[:B], device=dev), torch.as_tensor(par[:B], device=dev), None, torch.as_tensor(save_at, device=dev), None)
    runs = {}
    for name, env in (("unsliced", {"PN_B200_NO_SLICE": "1"}), ("quantum64", {"PN_B200_SLICE_QUANTUM": "64"}), ("default", {})):
        for k in ("PN_B200_NO_SLICE", "PN_B200_SLICE_QUANTUM"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        out = _cabi.solve_device(d2, *args, full=True)
        runs[name] = {k: v.cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    for name in ("unsliced", "quantum64", "default"):
        for key in ("u", "u_std", "n_accepted", "n_rejected", "status", "marg_mean", "marg_chol", "output_scale"):
            np.testing.assert_array_equal(runs[name][key], runs["unsliced"][key], err_msg=f"{name}:{key}")
        np.testing.assert_array_equal(runs[name]["u"], res["u"][:B])


@pytest.mark.parametrize("problem,d,nu,q,P", [("rigid_body", 3, 4, 1, 3), ("logistic", 1, 3, 1, 2), ("three_body", 2, 4, 2, 1)])
def test_time_sliced_scheduling_other_problems(monkeypatch, problem, d, nu, q, P):
    # the scheduler parks (running conditional + hidden state + 8 scalars) per member: sizes differ per
    # problem and order (odd totals are padded).  40,960 members, uniform tolerance, small quantum.
    import torch

    import problems_util as pu
    from odecheckpts_b200 import _cabi

    dev = torch.device("cuda:0")
    B, K = 40960, 9
    rng = np.random.default_rng(11)
    if problem == "rigid_body":
        u0 = (np.array([1.0, 0.0, 0.9]) + 0.05 * rng.standard_normal((B, 3)))[:, None, :]
        par, t1, tol, dt0 = np.tile(np.asarray(pu.RIGID_BODY_PARAMS), (B, 1)), 10.0, 1e-6, 0.1
    elif problem == "logistic":
        u0 = (0.05 + 0.1 * rng.random((B, 1)))[:, None, :]
        par, t1, tol, dt0 = np.tile([1.0, 1.0], (B, 1)), 2.5, 1e-9, 0.1
    else:
        u0 = pu.three_body_u0()[None] * (1.0 + 1e-7 * rng.standard_normal((B, 2, 2)))  # (the orbit starts 6e-3 from the second body)
        par, t1, tol, dt0 = np.full((B, 1), pu.THREE_BODY_MU), 3.0, 1e-7, 0.01
    desc = _cabi.Desc(_cabi.PROBLEM_IDS[problem], d, nu, q, 0, 0, 1, 1, tol, tol, dt0, 0.95, 0.2, 10.0, 0.3, 0.4, B, K, 20000, P, 0, 0)
    T = lambda x: torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device=dev)  # noqa: E731
    args = (T(u0), T(par), None, T(np.linspace(0.0, t1, K)), None)
    runs = {}
    for name, env in (("unsliced", {"PN_B200_NO_SLICE": "1"}), ("sliced", {"PN_B200_SLICE_QUANTUM": "16"})):
        for k in ("PN_B200_NO_SLICE", "PN_B200_SLICE_QUANTUM"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        out = _cabi.solve_device(desc, *args, full=True)
        runs[name] = {k: v.cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    assert (runs["unsliced"]["status"] == 0).all() and runs["unsliced"]["n_accepted"][:, -1].min() > 20
    for key in ("u", "u_std", "n_accepted", "n_rejected", "status", "marg_mean", "marg_chol", "output_scale"):
        np.testing.assert_array_equal(runs["sliced"][key], runs["unsliced"][key], err_msg=key)
