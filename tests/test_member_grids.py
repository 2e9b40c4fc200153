"""Per-member time grids (PN_B200_FLAG_MEMBER_GRIDS): save_at is [B][K] and row b is member b's grid -- its own t0, t1
and checkpoints, its own step grid with PN_B200_FLAG_FIXED_GRID, its own [t0_b, t1_b] with PN_B200_FLAG_RECORD.

The flag adds no algorithm, so a per-member-grid solve is compared with the oracle BIT FOR BIT, one member at a time
on that member's row; and a [B, K] grid whose rows all equal a shared grid gives the shared-grid call's bits.
"""

import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import problems_util as pu

RB_PARAMS = np.asarray(pu.RIGID_BODY_PARAMS)
CUBIC = "template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f) { f[0] = 3.0 * (t * t); }"
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


def _desc(cabi, problem, d, nu, q, B, K, *, fact="isotropic", corr="ts0", strat="fixedpoint", calib="dynamic", atol=1e-6,
          rtol=1e-6, dt0=0.01, P=0, flags=0, cap=0):  # fmt: skip
    pid = cabi.PROBLEM_IDS[problem] if isinstance(problem, str) else problem
    return cabi.Desc(pid, d, nu, q, cabi.FACTORISATIONS[fact], cabi.CORRECTIONS[corr], cabi.STRATEGIES[strat],
                     cabi.CALIBRATIONS[calib], atol, rtol, dt0, 0.95, 0.2, 10.0, 0.3, 0.4, B, K, 0, P, flags, cap)  # fmt: skip


def _rows(B, K, seed, t0=(0.0, 0.5), span=(2.0, 3.0), cluster=True):
    """[B, K] grids that really differ: t0_b and t1_b per member, uneven spacing, and (cluster) a run of checkpoints
    a few 1e-4 apart, so that several of them fall inside one step."""
    rng = np.random.default_rng(seed)
    rows = np.empty((B, K))
    for b in range(B):
        a = rng.uniform(*t0)
        e = a + rng.uniform(*span)
        inner = np.sort(rng.uniform(a, e, K - 2))
        if cluster and K >= 8:
            c = rng.uniform(a + 0.2 * (e - a), a + 0.8 * (e - a))
            inner[: 4] = c + 1e-4 * np.arange(4)
            inner = np.sort(inner)
        rows[b] = np.concatenate([[a], inner, [e]])
        assert np.all(np.diff(rows[b]) > 0)
    return rows


# ---- CPU ----------------------------------------------------------------------------------------------------------
def _configs(cabi):
    """(name, descriptor) covering every kernel family, a registered user problem and both other flags"""
    user = cabi.register_problem("member_grids_decay3",
                                 "template <class T> PN_DEV void vf(const T* u, const double* p, T* f) { for (int i = 0; i < 3; ++i) f[i] = -u[i]; }",
                                 d=3)  # fmt: skip
    R = cabi.FLAG_RECORD
    return [
        ("thread per IVP (headline)", _desc(cabi, "van_der_pol", 1, 4, 2, 65536, 50, fact="dense", corr="ts1", P=1)),
        ("thread per IVP (PAIR size)", _desc(cabi, "van_der_pol", 1, 4, 2, 300, 12, fact="dense", corr="ts1", P=1)),
        ("thread per IVP filter record", _desc(cabi, "logistic", 1, 3, 1, 64, 2, strat="filter", P=2, flags=R, cap=500)),
        ("thread per IVP fixed grid", _desc(cabi, "van_der_pol", 1, 4, 2, 64, 40, fact="dense", corr="ts1", P=1,
                                            flags=cabi.FLAG_FIXED_GRID)),  # fmt: skip
        ("lane per dimension isotropic", _desc(cabi, "pleiades", 14, 5, 2, 10, 20)),
        ("lane per dimension blockdiag", _desc(cabi, "rigid_body", 3, 4, 1, 10, 20, fact="blockdiag", P=3)),
        ("CTA per IVP isotropic", _desc(cabi, "brusselator", 64, 4, 1, 3, 6, P=1)),
        ("CTA per IVP isotropic, warp build", _desc(cabi, "brusselator", 48, 4, 1, 700, 6, P=1)),
        ("dense register columns", _desc(cabi, "rigid_body", 3, 4, 1, 37, 8, fact="dense", corr="ts1", P=3)),
        ("dense register columns record", _desc(cabi, "rigid_body", 3, 4, 1, 37, 2, fact="dense", corr="ts1", strat="filter",
                                                P=3, flags=R, cap=4096)),  # fmt: skip
        ("dense shared memory", _desc(cabi, "brusselator", 8, 4, 1, 3, 6, fact="dense", corr="ts1", P=1)),
        ("dense CTA", _desc(cabi, "brusselator", 16, 4, 1, 3, 6, fact="dense", corr="ts1", P=1)),
        ("user problem dense", _desc(cabi, user, 3, 4, 1, 100, 10, fact="dense", corr="ts1")),
        ("user problem blockdiag", _desc(cabi, user, 3, 4, 1, 100, 10, fact="blockdiag")),
    ]


def test_the_flag_changes_no_size_and_no_supported_configuration(cabi):
    configs = _configs(cabi)
    before = cabi.lib().pn_b200_jit_module_count()
    for name, desc in configs:
        shared = (cabi.supported(desc), cabi.workspace_bytes(desc), cabi.output_sizes(desc))
        desc.flags |= cabi.FLAG_MEMBER_GRIDS
        assert (cabi.supported(desc), cabi.workspace_bytes(desc), cabi.output_sizes(desc)) == shared, name
        assert shared[0], name
    assert cabi.lib().pn_b200_jit_module_count() == before  # none of these calls compiles


def test_the_binding_sets_the_flag_for_a_two_dimensional_grid(cabi):
    desc = _desc(cabi, "logistic", 1, 3, 1, 4, 5, P=2)
    assert cabi._grid_desc(desc, np.linspace(0, 1, 5)) is desc
    flagged = cabi._grid_desc(desc, np.tile(np.linspace(0, 1, 5), (4, 1)))
    assert flagged.flags == cabi.FLAG_MEMBER_GRIDS and desc.flags == 0  # the caller's descriptor is left alone
    with pytest.raises(ValueError, match="must have shape"):
        cabi._grid_desc(desc, np.zeros((3, 5)))
    with pytest.raises(ValueError, match="FLAG_MEMBER_GRIDS needs"):
        cabi._grid_desc(flagged, np.linspace(0, 1, 5))


def test_the_host_entry_point_rejects_a_row_that_is_not_strictly_increasing(cabi):
    B, K = 4, 5
    desc = _desc(cabi, "logistic", 1, 3, 1, B, K, P=2)
    rows = np.tile(np.linspace(0.0, 1.0, K), (B, 1))
    for bad in (0.1, 0.25, np.nan):  # out of order, repeated, NaN
        grid = rows.copy()
        grid[2, 2] = bad
        with pytest.raises(ValueError, match="row 2 is not strictly increasing"):
            cabi.solve_host(desc, np.full((B, 1, 1), 0.1), np.ones((B, 2)), None, grid, None)


def _logistic_init(B):
    from odecheckpts_b200 import ivps
    from odecheckpts_b200.probdiffeq import ivpsolve, ivpsolvers, taylor

    vf, _, _, args = ivps.logistic()
    solver = ivpsolvers.solver_dynamic(ivpsolvers.strategy_fixedpoint(ivpsolvers.prior_ibm(num_derivatives=3),
                                                                       ivpsolvers.correction_ts0(ode_order=1)))  # fmt: skip
    u0 = np.full((B, 1), 0.1) if B else np.array([0.1])
    init = solver.initial_condition(taylor.odejet_padded_scan(lambda *y: vf(*y, t=0.0, p=args), (u0,), num=3), 1.0)
    field = lambda *y, t: vf(*y, t=t, p=args)  # noqa: E731
    return field, init, ivpsolve.adaptive(solver, atol=1e-6, rtol=1e-6), solver


def test_python_validation_of_per_member_grids():
    from odecheckpts_b200.probdiffeq import ivpsolve

    B, K = 5, 6
    vf, init, asolver, solver = _logistic_init(B)
    rows = _rows(B, K, 0)
    kw = dict(dt0=0.01, factorisation="isotropic")
    with pytest.raises(ValueError, match="4 rows for an ensemble of 5"):
        ivpsolve.solve_adaptive_save_at(vf, init, rows[:4], asolver, **kw)
    bad = rows.copy()
    bad[3, [1, 2]] = bad[3, [2, 1]]
    with pytest.raises(ValueError, match="strictly increasing"):
        ivpsolve.solve_adaptive_save_at(vf, init, bad, asolver, **kw)
    with pytest.raises(ValueError, match="strictly increasing"):
        ivpsolve.solve_adaptive_save_at(vf, init, torch.as_tensor(bad), asolver, **kw)
    with pytest.raises(ValueError, match="4 rows"):
        ivpsolve.solve_fixed_grid(vf, init, rows[:4], solver, factorisation="isotropic")
    with pytest.raises(ValueError, match="rows for an ensemble"):
        ivpsolve.solve_adaptive_terminal_values(vf, init, rows[:4, 0], rows[:4, -1], asolver, **kw)
    with pytest.raises(ValueError, match="scalars or"):
        ivpsolve.solve_adaptive_terminal_values(vf, init, rows[:, :2], 3.0, asolver, **kw)
    vf1, init1, asolver1, _ = _logistic_init(0)
    with pytest.raises(ValueError, match="a single IVP takes save_at"):
        ivpsolve.solve_adaptive_save_at(vf1, init1, rows[:1], asolver1, **kw)
    with pytest.raises(ValueError, match="a single IVP"):
        ivpsolve.solve_adaptive_save_every_step(vf1, init1, np.array([0.0, 0.1]), np.array([1.0, 2.0]), asolver1, 0.01,
                                                factorisation="isotropic")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _shard_worker(rank, world, port, B, K):
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "code-adaptive-prob-ode-solvers_b200"))
    from odecheckpts_b200 import ensemble

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    grid = torch.as_tensor(_rows(B, K, 3))
    idx = ensemble.shard_indices(B, rank, world)
    mine = ensemble.shard_grid(grid, rank, world)
    ok = mine.shape == (len(idx), K) and bool(torch.equal(mine, grid[torch.as_tensor(idx)]))
    shared = torch.linspace(0.0, 1.0, K, dtype=torch.float64)
    ok &= ensemble.shard_grid(shared, rank, world) is shared
    ok &= np.array_equal(ensemble.shard_grid(grid.numpy(), rank, world), grid.numpy()[idx])
    # stand-in for the per-rank solve: every member reports the grid it was given; the gather restores member order
    out = ensemble.all_gather_results({"t": mine.contiguous()}, B)
    ok &= bool(torch.equal(out["t"], grid))
    t = torch.tensor([1.0 if ok else 0.0])
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if t.item() != 1.0:
        raise SystemExit(3)


@pytest.mark.parametrize("B", [10, 11])  # even and ragged shards
def test_grid_rows_shard_with_their_members(B):
    mp.spawn(_shard_worker, args=(2, _free_port(), B, 7), nprocs=2, join=True)


# ---- GPU helpers --------------------------------------------------------------------------------------------------
def _run(cabi, desc, u0, params, tol, save_at, *, full=True, samples=True, lml=True):
    """Every output of a device solve (+ samples and the likelihood of a fixed-point solve), as numpy."""
    dev = torch.device("cuda:0")
    t = lambda x: None if x is None else torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device=dev)  # noqa: E731
    out = cabi.solve_device(desc, t(u0), t(params), t(tol), t(save_at), None, full=full)
    res = {k: v.cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    if desc.strategy == cabi.STRATEGIES["fixedpoint"] and samples:
        res["samples"] = cabi.markov_sample_device(desc, out["_workspace"], out["status"], 7, 3).cpu().numpy()
    if desc.strategy == cabi.STRATEGIES["fixedpoint"] and lml:
        res["lml"] = cabi.log_marginal_likelihood_device(desc, out["_workspace"], out["status"], out["u"] + 0.01, 0.1).cpu().numpy()
    torch.cuda.synchronize()
    return res


def _same(name, got, want):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{name}: shape {got.shape} vs {want.shape}"
    same = (got == want) | (np.isnan(got.astype(float)) & np.isnan(want.astype(float)))
    if not same.all():
        bad = tuple(np.argwhere(~same)[0])
        raise AssertionError(f"{name}: {(~same).sum()} of {same.size} differ, first at {bad}: {got[bad]!r} vs {want[bad]!r}")


def _vdp(B, mu, seed):
    rng = np.random.default_rng(seed)
    u0 = np.stack([2.0 + 0.5 * rng.uniform(-1, 1, B), 0.5 * rng.uniform(-1, 1, B)], 1).reshape(B, 2, 1)
    return u0, np.full((B, 1), mu)


def _rigid(B, seed):
    rng = np.random.default_rng(seed)
    u0 = (np.array([1.0, 0.0, 0.9]) + 0.1 * rng.uniform(-1, 1, (B, 3))).reshape(B, 1, 3)
    return u0, RB_PARAMS[None] * (1.0 + 0.05 * rng.uniform(-1, 1, (B, 3)))


def _brusselator(N, B):
    return np.tile(pu.brusselator_u0(N)[None], (B, 1, 1)), np.array([[0.02], [0.01], [0.04]] * B)[:B]


# one configuration of every kernel family: (descriptor kwargs, members, whether the likelihood is implemented)
def _family(cabi, family):
    if family == "thread_per_ivp_pair":
        u0, par = _vdp(300, 100.0, 1)
        return _desc(cabi, "van_der_pol", 1, 4, 2, 300, 12, fact="dense", corr="ts1", atol=1e-5, rtol=1e-5, P=1), u0, par, True
    if family == "thread_per_ivp_sliced":
        u0, par = _vdp(65536, 1e3, 2)
        return _desc(cabi, "van_der_pol", 1, 4, 2, 65536, 20, fact="dense", corr="ts1", atol=1e-3, rtol=1e-3, P=1), u0, par, True
    if family == "lane_isotropic":
        u0 = np.tile(pu.pleiades_u0()[None], (5, 1, 1)) * (1.0 + 1e-3 * np.random.default_rng(3).standard_normal((5, 2, 14)))
        return _desc(cabi, "pleiades", 14, 5, 2, 5, 10, atol=1e-7, rtol=1e-5, dt0=0.1), u0, None, True
    if family == "lane_blockdiag":
        u0, par = _rigid(10, 4)
        return _desc(cabi, "rigid_body", 3, 4, 1, 10, 10, fact="blockdiag", atol=1e-8, rtol=1e-6, P=3), u0, par, True
    if family == "cta_isotropic":
        u0, par = _brusselator(32, 2)
        return _desc(cabi, "brusselator", 64, 4, 1, 2, 6, atol=1e-5, rtol=1e-5, P=1), u0, par, True
    if family == "dense_rows":
        u0, par = _rigid(37, 5)
        return _desc(cabi, "rigid_body", 3, 4, 1, 37, 8, fact="dense", corr="ts1", atol=1e-8, rtol=1e-6, P=3), u0, par, False
    if family == "dense_smem":
        u0, par = _brusselator(4, 3)
        return _desc(cabi, "brusselator", 8, 4, 1, 3, 6, fact="dense", corr="ts1", atol=1e-5, rtol=1e-5, P=1), u0, par, False
    assert family == "dense_cta"
    u0, par = _brusselator(8, 3)
    return _desc(cabi, "brusselator", 16, 4, 1, 3, 5, fact="dense", corr="ts1", atol=1e-4, rtol=1e-4, P=1), u0, par, False


FAMILIES = ["thread_per_ivp_pair", "thread_per_ivp_sliced", "lane_isotropic", "lane_blockdiag", "cta_isotropic", "dense_rows",
            "dense_smem", "dense_cta"]  # fmt: skip


# ---- GPU 1: rows equal to the shared grid give the shared grid's bits ----------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("family", FAMILIES)
def test_identical_rows_are_bit_identical_to_the_shared_grid(cabi, family):
    desc, u0, par, lml = _family(cabi, family)
    B, K = desc.batch, desc.num_save_at
    span = 0.5 if family in ("cta_isotropic", "dense_smem", "dense_cta") else (1.0 if family == "lane_isotropic" else 2.5)
    grid = np.linspace(0.3, 0.3 + span, K)
    shared = _run(cabi, desc, u0, par, None, grid, lml=lml)
    rows = _run(cabi, desc, u0, par, None, np.tile(grid, (B, 1)), lml=lml)
    assert shared.keys() == rows.keys() and "marg_chol" in shared and "samples" in shared
    for key in shared:
        _same(f"{family}: {key}", rows[key], shared[key])
    assert (shared["status"] == 0).all()
    if family == "thread_per_ivp_sliced":
        assert cabi.kernel_info(desc)["grid"] * 128 < B  # the time-sliced build runs


# ---- GPU 2: genuinely different rows against the oracle, member by member -------------------------------------------
def _oracle_member(oracle, problem, d, nu, q, b, u0, par, row, tol, **kw):
    cfg = oracle.make_config(problem, d, nu, q, atol=tol[0], rtol=tol[1], dt0=kw.pop("dt0", 0.01),
                             num_params=0 if par is None else par.shape[1], **kw)  # fmt: skip
    return oracle.solve_save_at(cfg, u0[b], [] if par is None else par[b], row, full=True)


def _check_against_oracle(name, got, b, ora, K):
    assert ora["status"] == 0, name
    for key in ("u", "u_std", "n_accepted"):
        _same(f"{name} {key}[{b}]", got[key][b], ora[key])
    assert got["n_rejected"][b] == ora["n_rejected"] and got["status"][b] == 0, name
    _same(f"{name} marg_mean[{b}]", got["marg_mean"][b].reshape(K, -1), ora["marg_mean"].reshape(K, -1))
    _same(f"{name} marg_chol[{b}]", got["marg_chol"][b].reshape(K, -1), ora["marg_chol"].reshape(K, -1))


ORACLE_CASES = {
    # name: (problem, d, nu, q, factorisation, correction, strategy, members, K, tol, oracle engine kwargs, env)
    "vdp_pair": ("van_der_pol", 1, 4, 2, "dense", "ts1", "fixedpoint", 200, 15, 1e-5, {}, {}),
    "logistic_filter": ("logistic", 1, 3, 1, "isotropic", "ts0", "filter", 50, 12, 1e-6, {}, {}),
    "pleiades_isotropic": ("pleiades", 14, 5, 2, "isotropic", "ts0", "fixedpoint", 5, 10, 1e-6, dict(reduction_group=16), {}),
    "rigid_blockdiag": ("rigid_body", 3, 4, 1, "blockdiag", "ts0", "fixedpoint", 10, 10, 1e-7, dict(reduction_group=4), {}),
    "brusselator32_pipe": ("brusselator", 64, 4, 1, "isotropic", "ts0", "fixedpoint", 1, 10, 1e-5, dict(reduction_group=128), {}),
    "brusselator32_ensemble": ("brusselator", 64, 4, 1, "isotropic", "ts0", "fixedpoint", 3, 10, 1e-5, dict(reduction_group=128),
                               {"PN_B200_WIDE_PIPE": "0"}),  # fmt: skip
    "rigid_dense_ts0": ("rigid_body", 3, 4, 1, "dense", "ts0", "fixedpoint", 37, 10, 1e-7, {}, {}),
    "rigid_dense_ts1_tolerances": ("rigid_body", 3, 4, 1, "dense", "ts1", "fixedpoint", 37, 10, None, {}, {}),
    "brusselator4_dense_smem": ("brusselator", 8, 4, 1, "dense", "ts1", "fixedpoint", 3, 8, 1e-5, {}, {}),
    "brusselator8_dense_cta": ("brusselator", 16, 4, 1, "dense", "ts1", "fixedpoint", 3, 6, 1e-4,
                               dict(reduction_group=256, dense_block=16), {}),  # fmt: skip
}


def _members(problem, d, B, seed):
    if problem == "van_der_pol":
        return _vdp(B, 100.0, seed)
    if problem == "logistic":
        rng = np.random.default_rng(seed)
        return rng.uniform(0.05, 0.2, (B, 1, 1)), np.tile([1.0, 1.0], (B, 1))
    if problem == "pleiades":
        return np.tile(pu.pleiades_u0()[None], (B, 1, 1)) * (1.0 + 1e-3 * np.random.default_rng(seed).standard_normal((B, 2, 14))), None
    if problem == "rigid_body":
        return _rigid(B, seed)
    return _brusselator(d // 2, B)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(ORACLE_CASES))
def test_per_member_grids_bitwise_against_the_oracle(cabi, oracle, monkeypatch, case):
    problem, d, nu, q, fact, corr, strat, B, K, tol, engine, env = ORACLE_CASES[case]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    u0, par = _members(problem, d, B, 11)
    short = problem == "brusselator" or problem == "pleiades"
    rows = _rows(B, K, 12, t0=(0.0, 0.3), span=(0.5, 1.0) if short else (2.0, 3.0), cluster=K >= 8)
    tols = None
    if tol is None:  # per-member tolerances: the longest-first order
        t = 10.0 ** np.random.default_rng(13).uniform(-8, -6, B)
        tols = np.stack([t, 100.0 * t], 1)
    desc = _desc(cabi, problem, d, nu, q, B, K, fact=fact, corr=corr, strat=strat, atol=tol or 1.0, rtol=tol or 1.0,
                 dt0=0.1 if problem == "pleiades" else 0.01, P=0 if par is None else par.shape[1])  # fmt: skip
    got = _run(cabi, desc, u0, par, tols, rows, samples=False, lml=False)
    for b in range(B):
        mtol = (tol, tol) if tols is None else tuple(tols[b])
        ora = _oracle_member(oracle, problem, d, nu, q, b, u0, par, rows[b], mtol, factorisation=fact, correction=corr,
                             strategy=strat, dt0=desc.dt0, **engine)  # fmt: skip
        _check_against_oracle(case, got, b, ora, K)
    assert len({int(n) for n in got["n_accepted"][:, -1]}) > 1 or B == 1


@pytest.mark.gpu
def test_warp_per_ivp_build_per_member_grids_bitwise_against_the_oracle(cabi, oracle):
    """From 592 members the CTA-per-IVP isotropic family runs its 32-thread build (one warp per IVP, norms summed by a
    32-lane butterfly: oracle reduction_group = 32)."""
    N, B, K = 24, 600, 8
    u0, _ = _brusselator(N, B)
    par = (1.0 / 50.0) * 10.0 ** np.random.default_rng(71).uniform(-0.5, 0.5, (B, 1))
    rows = _rows(B, K, 72, t0=(0.0, 0.3), span=(0.4, 0.8))
    desc = _desc(cabi, "brusselator", 2 * N, 4, 1, B, K, atol=1e-6, rtol=1e-6, P=1)
    assert cabi.kernel_info(desc)["threads_per_cta"] == 32
    got = _run(cabi, desc, u0, par, None, rows, samples=False, lml=False)
    assert (got["status"] == 0).all()
    for b in (0, 1, 299, 598, 599):
        ora = _oracle_member(oracle, "brusselator", 2 * N, 4, 1, b, u0, par, rows[b], (1e-6, 1e-6), reduction_group=32)
        _check_against_oracle("brusselator warp build", got, b, ora, K)


@pytest.mark.gpu
def test_time_sliced_per_member_grids_bitwise_against_the_oracle_and_the_unsliced_run(cabi, oracle, monkeypatch):
    B, K = 65536, 20
    u0, par = _vdp(B, 1e3, 21)
    rows = _rows(B, K, 22, t0=(0.0, 0.5), span=(4.0, 6.3), cluster=False)
    desc = _desc(cabi, "van_der_pol", 1, 4, 2, B, K, fact="dense", corr="ts1", atol=1e-3, rtol=1e-3, P=1)
    assert cabi.kernel_info(desc)["grid"] * 128 < B
    sliced = _run(cabi, desc, u0, par, None, rows, full=False, samples=False, lml=False)
    monkeypatch.setenv("PN_B200_NO_SLICE", "1")
    plain = _run(cabi, desc, u0, par, None, rows, full=False, samples=False, lml=False)
    for key in sliced:
        _same(f"sliced vs unsliced {key}", sliced[key], plain[key])
    cfg = oracle.make_config("van_der_pol", 1, 4, 2, factorisation="dense", correction="ts1", atol=1e-3, rtol=1e-3,
                             dt0=0.01, num_params=1)  # fmt: skip
    for b in (0, 1, 4097, 40000, B - 1):
        ora = oracle.solve_save_at_batch(cfg, u0[b:b + 1], par[b:b + 1], rows[b])
        for key in ("u", "u_std", "n_accepted", "n_rejected", "status"):
            _same(f"sliced {key}[{b}]", sliced[key][b], ora[key][0])


# ---- GPU 3: the other flags ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fixed_grid_rows_against_the_oracle(cabi, oracle):
    """The filter strategy against oracle.solve_fixed_grid (the oracle's fixed-grid replay is a filter); the
    fixed-point strategy: rows equal to a shared grid give its bits."""
    B, K = 40, 300
    u0, par = _vdp(B, 10.0, 31)
    rows = _rows(B, K, 32, t0=(0.0, 0.5), span=(1.5, 3.0), cluster=False)
    desc = _desc(cabi, "van_der_pol", 1, 4, 2, B, K, fact="dense", corr="ts1", strat="filter", P=1, flags=cabi.FLAG_FIXED_GRID)
    got = _run(cabi, desc, u0, par, None, rows, full=False)
    cfg = oracle.make_config("van_der_pol", 1, 4, 2, factorisation="dense", correction="ts1", strategy="filter", num_params=1)
    for b in range(B):
        ora = oracle.solve_fixed_grid(cfg, u0[b], par[b], rows[b])
        _same(f"fixed grid u[{b}]", got["u"][b], ora["u"])
        _same(f"fixed grid u_std[{b}]", got["u_std"][b], ora["u_std"])
    assert (got["status"] == 0).all()
    desc.strategy = cabi.STRATEGIES["fixedpoint"]
    shared = _run(cabi, desc, u0, par, None, rows[0])
    same_rows = _run(cabi, desc, u0, par, None, np.tile(rows[0], (B, 1)))
    for key in shared:
        _same(f"fixed grid, fixed point: {key}", same_rows[key], shared[key])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["logistic", "rigid_dense"])
def test_recording_rows_against_the_oracle(cabi, oracle, case):
    if case == "logistic":
        B, problem, d, fact, corr, P = 50, "logistic", 1, "isotropic", "ts0", 2
        u0, par = _members("logistic", 1, B, 41)
    else:
        B, problem, d, fact, corr, P = 37, "rigid_body", 3, "dense", "ts1", 3
        u0, par = _rigid(B, 42)
    rows = _rows(B, 2, 43, t0=(0.0, 1.0), span=(3.0, 8.0))
    desc = _desc(cabi, problem, d, 4, 1, B, 2, fact=fact, corr=corr, strat="filter", atol=1e-8, rtol=1e-6, P=P,
                 flags=cabi.FLAG_RECORD, cap=4096)  # fmt: skip
    out = _run(cabi, desc, u0, par, None, rows, full=False)
    cfg = oracle.make_config(problem, d, 4, 1, factorisation=fact, correction=corr, strategy="filter", atol=1e-8, rtol=1e-6,
                             dt0=0.01, num_params=P)  # fmt: skip
    for b in range(B):
        ora = oracle.solve_save_every_step(cfg, u0[b], par[b], rows[b, 0], rows[b, 1])
        n = int(out["traj_len"][b])
        assert n == len(ora["t"]) and n > 10, (b, n, len(ora["t"]))
        _same(f"{case} traj_t[{b}]", out["traj_t"][:n, b], ora["t"])
        assert ora["t"][0] == rows[b, 0] and ora["t"][-1] == rows[b, 1]
        _same(f"{case} traj_u[{b}]", out["traj_u"][:n, :, b], ora["u"])
        std = out["traj_std"][:n, :, b] if out["traj_std"].ndim == 3 else out["traj_std"][:n, b][:, None]
        _same(f"{case} traj_std[{b}]", std, ora["u_std"] if d > 1 and fact == "dense" else ora["u_std"][:, :1])
        assert out["n_rejected"][b] == ora["n_rejected"] and out["status"][b] == 0


@pytest.mark.gpu
def test_save_every_step_and_terminal_values_take_per_member_spans(cabi):
    from odecheckpts_b200 import ivps
    from odecheckpts_b200.probdiffeq import ivpsolve, ivpsolvers, taylor

    B = 6
    vf, _, _, args = ivps.logistic()
    u0 = np.full((B, 1), 0.1)
    t0 = np.linspace(0.0, 0.5, B)
    t1 = np.linspace(2.0, 3.0, B)
    field = lambda *y, t: vf(*y, t=t, p=args)  # noqa: E731
    for strat in (ivpsolvers.strategy_filter, ivpsolvers.strategy_fixedpoint):
        solver = ivpsolvers.solver_dynamic(strat(ivpsolvers.prior_ibm(num_derivatives=3), ivpsolvers.correction_ts0(ode_order=1)))
        init = solver.initial_condition(taylor.odejet_padded_scan(lambda *y: field(*y, t=0.0), (u0,), num=3), 1.0)
        asolver = ivpsolve.adaptive(solver, atol=1e-8, rtol=1e-8)
        term = ivpsolve.solve_adaptive_terminal_values(field, init, t0, t1, asolver, 0.01, factorisation="isotropic")
        # u(t) of the logistic equation from u(t0) = 0.1: the exact solution shifted by t0
        np.testing.assert_allclose(term.u[:, 0], pu.logistic_exact(t1 - t0), rtol=1e-6)
        if strat is ivpsolvers.strategy_filter:
            every = ivpsolve.solve_adaptive_save_every_step(field, init, t0, t1, asolver, 0.01, factorisation="isotropic")
            n = np.asarray(every.num_steps) + 1
            for b in range(B):
                assert every.t[0, b] == t0[b] and every.t[n[b] - 1, b] == t1[b]
                np.testing.assert_allclose(every.u[n[b] - 1, 0, b], term.u[b, 0], rtol=1e-6)


# ---- GPU 4: a time-dependent field starts at every member's own t0 --------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("strat, fact, corr, fixed_grid", [("fixedpoint", "dense", "ts1", False), ("filter", "dense", "ts1", False),
                                                           ("fixedpoint", "isotropic", "ts0", True)])  # fmt: skip
def test_time_dependent_field_is_exact_on_every_members_own_grid(cabi, strat, fact, corr, fixed_grid):
    B, K = 8, 60
    # own t0 and t1 per member, uneven but no near-coincident checkpoints: with gaps of 1e-4 the fixed-point solve of
    # t..t^4 loses digits to round-off (3e-8 relative measured), on a shared grid as on per-member ones
    rng = np.random.default_rng(51)
    t0, t1 = rng.uniform(0.3, 1.0, B), rng.uniform(2.3, 3.0, B)
    h = (t1 - t0) / (K - 1)
    jitter = np.concatenate([np.zeros((B, 1)), rng.uniform(-0.3, 0.3, (B, K - 2)), np.zeros((B, 1))], axis=1)
    rows = np.linspace(t0, t1, K).T + jitter * h[:, None]
    assert np.all(np.diff(rows, axis=1) > 0.3 * h[:, None])
    cases = [(CUBIC, "member_grids_cubic", 1, 3, [3], rows[:, 0:1] ** 3, fact, corr),
             (POWERS4, "member_grids_powers4", 4, 4, [1, 2, 3, 4], rows[:, 0:1] ** np.arange(1, 5)[None], fact, corr)]
    for src, name, d, nu, powers, u0, f, c in cases:
        pid = cabi.register_problem(name, src, d=d, time_dependent=True)
        desc = _desc(cabi, pid, d, nu, 1, B, K, fact=f, corr=c, strat=strat, calib="none", atol=1e-4, rtol=1e-4,
                     flags=cabi.FLAG_FIXED_GRID if fixed_grid else 0)  # fmt: skip
        got = _run(cabi, desc, u0.reshape(B, 1, d), None, None, rows, full=False, samples=False, lml=False)
        assert (got["status"] == 0).all()
        want = rows[:, :, None] ** np.asarray(powers, dtype=np.float64)[None, None]
        rel = np.abs(got["u"] - want) / np.maximum(1.0, np.abs(want))
        assert rel.max() <= 1e-10, f"{name} ({strat} {f}): max relative error {rel.max():.3g}"


# ---- GPU 5: likelihood and samples after a per-member-grid solve ----------------------------------------------------
@pytest.mark.gpu
def test_likelihood_and_samples_after_a_per_member_grid_solve(oracle):
    from odecheckpts_b200 import ivps
    from odecheckpts_b200.probdiffeq import ivpsolve, ivpsolvers, stats, taylor

    B, K = 6, 9
    vdp = ivps.van_der_pol()[0].inner  # the VectorField itself: mu is its parameter, one per subject here
    mu = 10.0 ** np.random.default_rng(60).uniform(0.5, 1.5, B)
    vf = lambda *y, t: vdp(*y, t=t, p=(mu,))  # noqa: E731
    u0, _ = _vdp(B, 10.0, 61)
    rows = _rows(B, K, 62, t0=(0.0, 0.5), span=(2.0, 3.0))
    solver = ivpsolvers.solver_dynamic(ivpsolvers.strategy_fixedpoint(ivpsolvers.prior_ibm(num_derivatives=4),
                                                                      ivpsolvers.correction_ts1(ode_order=2)))  # fmt: skip
    init = solver.initial_condition(taylor.odejet_padded_scan(lambda *y: vf(*y, t=0.0), (u0[:, 0], u0[:, 1]), num=3), 1.0)
    asolver = ivpsolve.adaptive(solver, atol=1e-5, rtol=1e-5)
    sol = ivpsolve.solve_adaptive_save_at(vf, init, torch.as_tensor(rows), asolver, 0.01, factorisation="dense",
                                          keep_conditionals=True)  # fmt: skip
    assert np.array_equal(sol.t, rows) and sol.u.shape == (B, K, 1)
    rng = np.random.default_rng(63)
    std = 0.05 + 0.1 * rng.random((B, K))
    data = sol.u + 0.1 * rng.standard_normal((B, K, 1))
    lml = stats.log_marginal_likelihood(data, standard_deviation=std, posterior=sol.posterior)
    cfg = oracle.make_config("van_der_pol", 1, 4, 2, factorisation="dense", correction="ts1", atol=1e-5, rtol=1e-5,
                             dt0=0.01, num_params=1)  # fmt: skip
    for b in range(B):
        ora = oracle.solve_save_at_lml(cfg, u0[b], [mu[b]], rows[b], data[b], std[b])
        assert ora["status"] == 0
        _same(f"u[{b}]", sol.u[b], ora["u"])
        assert lml[b] == ora["lml"], (b, lml[b], ora["lml"])
    S = 6000
    (qoi, _), (last, _) = stats.markov_sample(7, sol.posterior, shape=(S,), reverse=True)
    smp = np.concatenate([qoi, last[..., None, :]], axis=-2)  # [B, S, K, d]
    assert smp.shape == (B, S, K, 1) and np.isfinite(smp).all()
    for b in range(B):
        mean, sd = smp[b].mean(axis=0), smp[b].std(axis=0)
        assert np.all(np.abs(mean - sol.u[b]) <= 5 * sol.u_std[b] / np.sqrt(S) + 1e-12), b
        big = sol.u_std[b] > 1e-10
        np.testing.assert_allclose(sd[big], sol.u_std[b][big], rtol=0.07)
