"""ctypes loader for the CPU ORACLE (test infrastructure, NOT product code).

Only tests/, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs may
import this module.  See oracle/pn_oracle.h for what the oracle restates and how
it is pinned against the reference's golden artefacts.
"""

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libpn_oracle.so")

PROBLEMS = {
    "logistic": 0,
    "rigid_body": 1,
    "three_body": 2,
    "pleiades": 3,
    "brusselator": 4,
    "van_der_pol": 5,
    "lotka_volterra": 6,
}
FACTORISATIONS = {"isotropic": 0, "blockdiag": 1, "dense": 2}
CORRECTIONS = {"ts0": 0, "ts1": 1}
STRATEGIES = {"filter": 0, "fixedpoint": 1}
CALIBRATIONS = {"none": 0, "dynamic": 1, "mle": 2}


class Config(C.Structure):
    _fields_ = [
        ("problem", C.c_int32),
        ("d", C.c_int32),
        ("nu", C.c_int32),
        ("ode_order", C.c_int32),
        ("factorisation", C.c_int32),
        ("correction", C.c_int32),
        ("strategy", C.c_int32),
        ("calibration", C.c_int32),
        ("atol", C.c_double),
        ("rtol", C.c_double),
        ("dt0", C.c_double),
        ("safety", C.c_double),
        ("factor_min", C.c_double),
        ("factor_max", C.c_double),
        ("power_integral", C.c_double),
        ("power_proportional", C.c_double),
        ("max_attempts", C.c_int64),
        ("num_params", C.c_int32),
        ("reduction_group", C.c_int32),
        ("dense_block", C.c_int32),
    ]


class AttemptInfo(C.Structure):
    _fields_ = [
        ("error_norm", C.c_double),
        ("dt_proposed", C.c_double),
        ("sigma", C.c_double),
        ("sigma_hat", C.c_double),
    ]


def build(force=False):
    """Compile oracle/libpn_oracle.so with gcc (see oracle/Makefile) and return its path.  In a read-only
    tree whose library is missing or older than its sources, the library is built in a temporary directory
    (removed at exit) instead, so that running the tests or the benchmark never writes into the tree."""
    srcs = ["pn_linalg.c", "pn_blocked.c", "pn_problems.c", "pn_solver.c", "pn_oracle.h", "pn_internal.h", "Makefile"]
    if not force and os.path.exists(_LIB_PATH):
        newest = max(os.path.getmtime(os.path.join(_HERE, s)) for s in srcs)
        if os.path.getmtime(_LIB_PATH) >= newest:
            return _LIB_PATH
    out = _LIB_PATH
    if not os.access(_HERE, os.W_OK):
        tmp = tempfile.mkdtemp(prefix="pn_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libpn_oracle.so")
    subprocess.run(["make", "-C", _HERE, "-B", f"LIB={out}"], check=True, capture_output=True)
    return out


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        dp = C.POINTER(C.c_double)
        _lib.pn_det_pow.restype = C.c_double
        _lib.pn_det_pow.argtypes = [C.c_double, C.c_double]
        _lib.pn_det_log.restype = C.c_double
        _lib.pn_det_log.argtypes = [C.c_double]
        _lib.pn_det_exp.restype = C.c_double
        _lib.pn_det_exp.argtypes = [C.c_double]
        _lib.pn_oracle_solve_save_every_step.restype = C.c_int64
        del dp
    return _lib


def make_config(
    problem,
    d,
    nu,
    ode_order,
    *,
    factorisation="isotropic",
    correction="ts0",
    strategy="fixedpoint",
    calibration="dynamic",
    atol=1e-6,
    rtol=1e-6,
    dt0=0.01,
    max_attempts=0,
    num_params=0,
    safety=0.95,
    factor_min=0.2,
    factor_max=10.0,
    power_integral=0.3,
    power_proportional=0.4,
    reduction_group=0,
    dense_block=0,
):
    return Config(
        PROBLEMS[problem] if isinstance(problem, str) else int(problem),
        int(d),
        int(nu),
        int(ode_order),
        FACTORISATIONS[factorisation],
        CORRECTIONS[correction],
        STRATEGIES[strategy],
        CALIBRATIONS[calibration],
        float(atol),
        float(rtol),
        float(dt0),
        safety,
        factor_min,
        factor_max,
        power_integral,
        power_proportional,
        int(max_attempts),
        int(num_params),
        int(reduction_group),
        int(dense_block),
    )


def _dptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def _engine_dims(cfg):
    n = cfg.nu + 1
    if cfg.factorisation == 2:
        return 1, n * cfg.d, 1
    if cfg.factorisation == 1:
        return cfg.d, n, cfg.d
    return 1, n, cfg.d


def prior(nu):
    n = nu + 1
    a1 = np.zeros((n, n))
    lq = np.zeros((n, n))
    lib().pn_oracle_prior(C.c_int(nu), _dptr(a1), _dptr(lq))
    return a1, lq


def vf(problem, u, params=(), t=0.0):
    """u: (q, d) -> f: (d,)"""
    u = _f64(u)
    q, d = u.shape
    p = _f64(params if len(params) else [0.0])
    f = np.zeros(d)
    lib().pn_oracle_vf(C.c_int(PROBLEMS[problem]), C.c_int(d), _dptr(u), C.c_double(t), _dptr(p), _dptr(f))
    return f


def jac(problem, u, params=(), t=0.0):
    u = _f64(u)
    q, d = u.shape
    p = _f64(params if len(params) else [0.0])
    J = np.zeros((d, q * d))
    lib().pn_oracle_jac(C.c_int(PROBLEMS[problem]), C.c_int(d), _dptr(u), C.c_double(t), _dptr(p), _dptr(J))
    return J


def taylor_init(problem, u0, nu, params=(), t0=0.0):
    """u0: (q, d) -> (nu+1, d) derivatives u^{(k)}(t0)."""
    u0 = _f64(u0)
    q, d = u0.shape
    p = _f64(params if len(params) else [0.0])
    out = np.zeros((nu + 1, d))
    lib().pn_oracle_taylor_init(
        C.c_int(PROBLEMS[problem]), C.c_int(d), C.c_int(nu), C.c_int(q), _dptr(u0), C.c_double(t0), _dptr(p), _dptr(out)
    )
    return out


def attempt_step(cfg, params, t, dt, e_prev, output_scale, mean, chol, bw=None):
    F, N, Ct = _engine_dims(cfg)
    mean = _f64(mean).reshape(N * Ct)
    chol = _f64(chol).reshape(F * N * N)
    p = _f64(params if len(params) else [0.0])
    mo, co = np.zeros_like(mean), np.zeros_like(chol)
    Go, go, Lo = np.zeros(F * N * N), np.zeros(N * Ct), np.zeros(F * N * N)
    if bw is not None:
        G, g, Lam = (_f64(x).ravel() for x in bw)
    else:
        G = g = Lam = None
    info = AttemptInfo()
    rc = lib().pn_oracle_attempt_step(
        C.byref(cfg), _dptr(p), C.c_double(t), C.c_double(dt), C.c_double(e_prev), C.c_double(output_scale),
        _dptr(mean), _dptr(chol), _dptr(G), _dptr(g), _dptr(Lam),
        _dptr(mo), _dptr(co), _dptr(Go), _dptr(go), _dptr(Lo), C.byref(info),
    )  # fmt: skip
    if rc:
        raise ValueError(f"oracle rejected the configuration (rc={rc})")
    return {
        "mean": mo.reshape(N, Ct),
        "chol": co.reshape(F, N, N),
        "G": Go.reshape(F, N, N),
        "g": go.reshape(N, Ct),
        "Lam": Lo.reshape(F, N, N),
        "error_norm": info.error_norm,
        "dt_proposed": info.dt_proposed,
        "sigma": info.sigma,
        "sigma_hat": info.sigma_hat,
    }


def solve_save_at(cfg, u0, params, save_at, output_scale0=1.0, full=False):
    u0 = _f64(u0)
    save_at = _f64(save_at)
    K = len(save_at)
    d = cfg.d
    F, N, Ct = _engine_dims(cfg)
    p = _f64(params if len(params) else [0.0])
    u, u_std, filt = np.zeros((K, d)), np.zeros((K, d)), np.zeros((K, d))
    mm = np.zeros((K, N, Ct)) if full else None
    mc = np.zeros((K, F, N, N)) if full else None
    nacc = np.zeros(K, dtype=np.int64)
    nrej = C.c_int64(0)
    status = C.c_int32(0)
    rc = lib().pn_oracle_solve_save_at(
        C.byref(cfg), _dptr(u0), _dptr(p), _dptr(save_at), C.c_int64(K), C.c_double(output_scale0),
        _dptr(u), _dptr(u_std), _dptr(mm), _dptr(mc),
        nacc.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(nrej), C.byref(status), _dptr(filt),
    )  # fmt: skip
    if rc:
        raise ValueError(f"oracle rejected the configuration (rc={rc})")
    out = {
        "u": u,
        "u_std": u_std,
        "filt_u": filt,
        "n_accepted": nacc,
        "n_rejected": int(nrej.value),
        "status": int(status.value),
    }
    if full:
        out["marg_mean"], out["marg_chol"] = mm, mc
    return out


def solve_save_at_lml(cfg, u0, params, save_at, data, obs_std, output_scale0=1.0):
    """Checkpoint solve + stats.log_marginal_likelihood(data, standard_deviation=obs_std, posterior=...)
    (train_util.py:22-24).  Also returns the backward conditionals and per-checkpoint output scales."""
    u0 = _f64(u0)
    save_at = _f64(save_at)
    K = len(save_at)
    d = cfg.d
    F, N, Ct = _engine_dims(cfg)
    p = _f64(params if len(params) else [0.0])
    data = _f64(np.asarray(data, dtype=float).reshape(K, d))
    obs_std = _f64(np.broadcast_to(np.asarray(obs_std, dtype=float), (K,)))
    u, u_std = np.zeros((K, d)), np.zeros((K, d))
    mm, mc = np.zeros((K, N, Ct)), np.zeros((K, F, N, N))
    cond = np.zeros((K, 2 * F * N * N + N * Ct))
    scale = np.zeros((K, F))
    lml = C.c_double(0.0)
    status = C.c_int32(0)
    rc = lib().pn_oracle_solve_save_at_lml(
        C.byref(cfg), _dptr(u0), _dptr(p), _dptr(save_at), C.c_int64(K), C.c_double(output_scale0),
        _dptr(data), _dptr(obs_std), _dptr(u), _dptr(u_std), _dptr(mm), _dptr(mc), _dptr(cond), _dptr(scale),
        C.byref(lml), C.byref(status),
    )  # fmt: skip
    if rc:
        raise ValueError(f"oracle rejected the configuration (rc={rc})")
    FNN = F * N * N
    return {
        "u": u, "u_std": u_std, "marg_mean": mm, "marg_chol": mc, "status": int(status.value), "lml": float(lml.value),
        "output_scale": scale,
        "cond_G": cond[:, :FNN].reshape(K, F, N, N), "cond_g": cond[:, FNN:FNN + N * Ct].reshape(K, N, Ct),
        "cond_Lam": cond[:, FNN + N * Ct:].reshape(K, F, N, N),
    }  # fmt: skip


def solve_save_at_batch(cfg, u0, params, save_at, tol=None, output_scale0=None, num_threads=0):
    """u0: (B, q, d); params: (B, P)."""
    u0 = _f64(u0)
    B = u0.shape[0]
    save_at = _f64(save_at)
    K = len(save_at)
    d = cfg.d
    params = _f64(params).reshape(B, -1) if cfg.num_params > 0 else np.zeros((B, 1))
    tol_a = _f64(tol) if tol is not None else None
    os0 = _f64(output_scale0) if output_scale0 is not None else None
    u, u_std = np.zeros((B, K, d)), np.zeros((B, K, d))
    nacc = np.zeros((B, K), dtype=np.int64)
    nrej = np.zeros(B, dtype=np.int64)
    status = np.zeros(B, dtype=np.int32)
    rc = lib().pn_oracle_solve_save_at_batch(
        C.byref(cfg), C.c_int64(B), _dptr(u0), _dptr(params), _dptr(tol_a), _dptr(save_at), C.c_int64(K),
        _dptr(os0), _dptr(u), _dptr(u_std),
        nacc.ctypes.data_as(C.POINTER(C.c_int64)), nrej.ctypes.data_as(C.POINTER(C.c_int64)),
        status.ctypes.data_as(C.POINTER(C.c_int32)), C.c_int(num_threads),
    )  # fmt: skip
    if rc:
        raise ValueError(f"oracle rejected the configuration (rc={rc})")
    return {"u": u, "u_std": u_std, "n_accepted": nacc, "n_rejected": nrej, "status": status}


def solve_save_every_step(cfg, u0, params, t0, t1, output_scale0=1.0, max_grid=1 << 20):
    u0 = _f64(u0)
    d = cfg.d
    p = _f64(params if len(params) else [0.0])
    grid = np.zeros(max_grid)
    u = np.zeros((max_grid, d))
    u_std = np.zeros((max_grid, d))
    nrej = C.c_int64(0)
    cnt = lib().pn_oracle_solve_save_every_step(
        C.byref(cfg), _dptr(u0), _dptr(p), C.c_double(t0), C.c_double(t1), C.c_double(output_scale0),
        C.c_int64(max_grid), _dptr(grid), _dptr(u), _dptr(u_std), C.byref(nrej),
    )  # fmt: skip
    if cnt < 0:
        raise RuntimeError(f"save_every_step failed (rc={cnt})")
    return {"t": grid[:cnt].copy(), "u": u[:cnt].copy(), "u_std": u_std[:cnt].copy(), "n_rejected": int(nrej.value)}


def solve_fixed_grid(cfg, u0, params, grid, output_scale0=1.0):
    u0 = _f64(u0)
    grid = _f64(grid)
    G = len(grid)
    d = cfg.d
    p = _f64(params if len(params) else [0.0])
    u, u_std, en = np.zeros((G, d)), np.zeros((G, d)), np.zeros(G)
    rc = lib().pn_oracle_solve_fixed_grid(
        C.byref(cfg), _dptr(u0), _dptr(p), _dptr(grid), C.c_int64(G), C.c_double(output_scale0),
        _dptr(u), _dptr(u_std), _dptr(en),
    )  # fmt: skip
    if rc:
        raise ValueError(f"oracle rejected the configuration (rc={rc})")
    return {"u": u, "u_std": u_std, "error_norms": en}


QR_SHAPES = {"full": 0, "toptri_botfull": 1, "topfull_bottri": 2}


def qr_blocked(M, ncols=None, shape="full", ntop=0, nb=16):
    """Blocked Householder QR (R only) of a copy of M in the CUDA kernel's operation order (pn_blocked.c)."""
    M = np.array(M, dtype=np.float64, order="C")
    rows, cols = M.shape
    lib().pn_qr_blocked(_dptr(M), C.c_int(cols), C.c_int(rows), C.c_int(cols), C.c_int(cols if ncols is None else ncols),
                        C.c_int(QR_SHAPES[shape]), C.c_int(ntop), C.c_int(nb))  # fmt: skip
    return M


def solve_upper_blocked(R, B, nb=64):
    """X = R^{-1} B by blocked back substitution in the CUDA kernel's operation order (pn_blocked.c)."""
    R, B = _f64(R), _f64(B)
    n, c = B.shape
    X = np.zeros((n, c))
    lib().pn_solve_upper_blocked(_dptr(R), C.c_int(R.shape[1]), _dptr(B), C.c_int(c), _dptr(X), C.c_int(c), C.c_int(n),
                                 C.c_int(c), C.c_int(nb))  # fmt: skip
    return X


def gemm_chain(A, B, C0=None, neg=False):
    """C = (C0 or 0) -/+ A B with the ascending-k fma chain per element (the tensor-core product contract)."""
    A, B = _f64(A), _f64(B)
    M, K = A.shape
    N = B.shape[1]
    C0 = _f64(C0) if C0 is not None else None
    out = np.zeros((M, N))
    lib().pn_gemm_chain(_dptr(out), _dptr(A), _dptr(B), C.c_int(M), C.c_int(N), C.c_int(K), _dptr(C0), C.c_int(1 if neg else 0))
    return out
