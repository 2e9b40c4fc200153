"""The builds that move the backward conditional off the step's critical path -- PAIR (thread-per-IVP kernels,
a backward lane per IVP, small ensembles) and PIPE (CTA-per-IVP kernel, a backward warp, at most one member per
SM) -- against the plain kernels they replace: same operations in the same order, so every output must be
bit-identical, whichever build the library picks (PN_B200_PAIR=0 / PN_B200_WIDE_PIPE=0 switch them off)."""

import numpy as np
import pytest

import problems_util as pu
from test_gpu_parity import _assert_bitwise, _desc, _ocfg, cabi  # noqa: F401

pytestmark = pytest.mark.gpu
KEYS = ("u", "u_std", "marg_mean", "marg_chol", "n_accepted", "n_rejected", "status", "output_scale")


@pytest.mark.parametrize("B", [1, 33, 700])
def test_pair_build_equals_the_plain_thread_per_ivp_kernel(cabi, oracle, monkeypatch, B):
    rng = np.random.default_rng(B)
    K = 30
    u0 = np.stack([2.0 + 0.5 * rng.uniform(-1, 1, B), 0.5 * rng.uniform(-1, 1, B)], 1).reshape(B, 2, 1)
    params = np.full((B, 1), 1e3)
    # a tolerance sweep in one launch: members of one warp accept / reject / cross checkpoints at different times
    tol = np.stack([10.0 ** -rng.integers(3, 8, B).astype(float)] * 2, 1)
    save_at = np.linspace(0.0, 6.3, K)
    desc = _desc(cabi, "van_der_pol", 1, 4, 2, B, K, fact="dense", corr="ts1", P=1, atol=1e-5, rtol=1e-5)
    assert cabi.kernel_info(desc)["threads_per_cta"] == 256  # 128 filter lanes + 128 backward lanes
    pair = cabi.solve_host(desc, u0, params, tol, save_at, None, full=True)
    monkeypatch.setenv("PN_B200_PAIR", "0")
    assert cabi.kernel_info(desc)["threads_per_cta"] == 128
    plain = cabi.solve_host(desc, u0, params, tol, save_at, None, full=True)
    _assert_bitwise(pair, plain, KEYS)
    assert int((pair["status"] != 0).sum()) == 0 and len(set(pair["n_accepted"][:, -1].tolist())) > min(B, 3) - 1
    idx = np.arange(0, B, max(1, B // 8))
    ora = oracle.solve_save_at_batch(_ocfg(oracle, "van_der_pol", 1, 4, 2, fact="dense", corr="ts1", P=1, atol=1e-5, rtol=1e-5),
                                     u0[idx], params[idx], save_at, tol=tol[idx])  # fmt: skip
    _assert_bitwise({k: pair[k][idx] for k in ("u", "u_std", "n_accepted", "n_rejected", "status")}, ora)


def test_pair_build_other_problems_and_many_checkpoints_inside_one_step(cabi, oracle, monkeypatch):
    # three-body (d = 2, nu = 4) and the logistic ODE with checkpoints much denser than the steps (every mode of the
    # bookkeeping: overshoot, several checkpoints inside one step, exact hits on the terminal point)
    cases = [("three_body", 2, 4, 2, (pu.THREE_BODY_MU,), pu.three_body_u0(), np.linspace(0, 5.0, 40), dict(atol=1e-5, rtol=1e-5)),
             ("logistic", 1, 4, 1, (1.0, 1.0), np.array([[0.1]]), np.linspace(0, 2.5, 400), dict(atol=1e-3, rtol=1e-3, dt0=0.1)),
             ("logistic", 1, 2, 1, (1.0, 1.0), np.array([[0.1]]), np.linspace(0, 2.5, 7), dict(atol=1e-4, rtol=1e-4, dt0=0.1))]  # fmt: skip
    for problem, d, nu, q, par, u0, save_at, kw in cases:
        B, P = 5, len(par)
        u0_b = np.tile(u0[None], (B, 1, 1)) * (1.0 + 1e-3 * np.arange(B))[:, None, None]
        par_b = np.tile(np.asarray(par, dtype=float), (B, 1))
        desc = _desc(cabi, problem, d, nu, q, B, len(save_at), P=P, **kw)
        monkeypatch.delenv("PN_B200_PAIR", raising=False)
        assert cabi.kernel_info(desc)["threads_per_cta"] == 256
        pair = cabi.solve_host(desc, u0_b, par_b, None, save_at, None, full=True)
        monkeypatch.setenv("PN_B200_PAIR", "0")
        plain = cabi.solve_host(desc, u0_b, par_b, None, save_at, None, full=True)
        _assert_bitwise(pair, plain, KEYS)
        ora = oracle.solve_save_at(_ocfg(oracle, problem, d, nu, q, P=P, **kw), u0, par, save_at)
        _assert_bitwise({k: pair[k][0] for k in ("u", "u_std", "n_accepted")}, {k: ora[k] for k in ("u", "u_std", "n_accepted")},
                        ("u", "u_std", "n_accepted"))  # fmt: skip


@pytest.mark.parametrize("N,B", [(32, 1), (32, 5), (100, 2)])
def test_pipe_build_equals_the_plain_cta_per_ivp_kernel(cabi, monkeypatch, N, B):
    d, K = 2 * N, 25
    rng = np.random.default_rng(N)
    alpha = 0.02 * 10.0 ** rng.uniform(-0.3, 0.3, B)
    u0 = np.tile(pu.brusselator_u0(N)[None], (B, 1, 1))
    save_at = np.linspace(0.0, 2.0, K)
    desc = _desc(cabi, "brusselator", d, 4, 1, B, K, P=1, atol=1e-6, rtol=1e-6)
    assert cabi.kernel_info(desc)["threads_per_cta"] == 192  # 128 main threads, an idle warp, the backward warp
    pipe = cabi.solve_host(desc, u0, alpha[:, None], None, save_at, None, full=True)
    monkeypatch.setenv("PN_B200_WIDE_PIPE", "0")
    assert cabi.kernel_info(desc)["threads_per_cta"] == 128
    plain = cabi.solve_host(desc, u0, alpha[:, None], None, save_at, None, full=True)
    _assert_bitwise(pipe, plain, KEYS)
    assert int((pipe["status"] != 0).sum()) == 0
