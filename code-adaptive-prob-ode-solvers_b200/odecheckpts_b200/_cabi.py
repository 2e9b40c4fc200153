"""ctypes binding of the C ABI in include/pn_b200.h (libpn_b200.so).

There is deliberately no CPU fallback: if the CUDA library is missing or the descriptor has
no compiled kernel, the call raises.
"""

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG, "libpn_b200.so")

PROBLEM_IDS = {
    "logistic": 0,
    "rigid_body": 1,
    "three_body": 2,
    "pleiades": 3,
    "brusselator": 4,
    "van_der_pol": 5,
    "lotka_volterra": 6,
}
USER_PROBLEM_BASE = 1024  # ids of problems registered at run time (register_problem) start here
SOURCE_FORMS = {"simple": 0, "full": 1}
FORM_TIME_DEPENDENT = 2  # OR-ed into the form: the field takes the time (include/pn_b200.h)
FACTORISATIONS = {"isotropic": 0, "blockdiag": 1, "dense": 2}
CORRECTIONS = {"ts0": 0, "ts1": 1}
STRATEGIES = {"filter": 0, "fixedpoint": 1}
CALIBRATIONS = {"none": 0, "dynamic": 1, "mle": 2}
FLAG_FIXED_GRID = 1
FLAG_RECORD = 2
FLAG_MEMBER_GRIDS = 4  # save_at is [B, K]: one grid per ensemble member
STATUS_OK, STATUS_NAN, STATUS_MAX_ATTEMPTS = 0, 1, 2


class Desc(C.Structure):
    """pn_b200_desc"""

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
        ("batch", C.c_int64),
        ("num_save_at", C.c_int64),
        ("max_attempts", C.c_int64),
        ("num_params", C.c_int32),
        ("flags", C.c_int32),
        ("traj_capacity", C.c_int64),
    ]


class KernelInfo(C.Structure):
    """pn_b200_kernel_info"""

    _fields_ = [
        ("threads_per_cta", C.c_int32),
        ("ctas_per_sm", C.c_int32),
        ("num_sms", C.c_int32),
        ("grid", C.c_int32),
        ("registers_per_thread", C.c_int32),
        ("static_smem_bytes", C.c_int32),
        ("dynamic_smem_bytes", C.c_int32),
        ("local_bytes_per_thread", C.c_int32),
    ]


class Sizes(C.Structure):
    """pn_b200_sizes"""

    _fields_ = [(name, C.c_size_t) for name in (
        "u", "u_std", "marg_mean", "marg_chol", "output_scale", "n_accepted", "n_rejected", "status",
        "traj_t", "traj_u", "traj_std", "traj_len")]  # fmt: skip


EXPORTS = (
    "pn_b200_supported",
    "pn_b200_workspace_bytes",
    "pn_b200_output_sizes",
    "pn_b200_trim",
    "pn_b200_solve_save_at",
    "pn_b200_solve_save_at_host",
    "pn_b200_get_kernel_info",
    "pn_b200_measure_fp64_peak",
    "pn_b200_markov_sample",
    "pn_b200_log_marginal_likelihood",
    "pn_b200_set_profiling",
    "pn_b200_get_last_timing",
    "pn_b200_last_error",
    "pn_b200_register_problem",
    "pn_b200_problem_evaluate",
    "pn_b200_problem_evaluate_at",
    "pn_b200_compile",
)

_lib = None


class LibraryMissing(RuntimeError):
    pass


def lib():
    """Load libpn_b200.so; fail loudly if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LibraryMissing(
                f"{LIB_PATH} not found: build it with `python code-adaptive-prob-ode-solvers_b200/build.py` "
                "(there is no CPU fallback)"
            )
        L = C.CDLL(LIB_PATH)
        vp, dp = C.c_void_p, C.c_void_p
        L.pn_b200_supported.restype = C.c_int
        L.pn_b200_supported.argtypes = [C.POINTER(Desc)]
        L.pn_b200_workspace_bytes.restype = C.c_size_t
        L.pn_b200_workspace_bytes.argtypes = [C.POINTER(Desc)]
        L.pn_b200_output_sizes.restype = C.c_int
        L.pn_b200_output_sizes.argtypes = [C.POINTER(Desc), C.POINTER(Sizes)]
        L.pn_b200_trim.restype = C.c_int
        L.pn_b200_trim.argtypes = [C.c_int]
        L.pn_b200_solve_save_at.restype = C.c_int
        L.pn_b200_solve_save_at.argtypes = [C.POINTER(Desc)] + [dp] * 17 + [vp, C.c_size_t, vp]
        L.pn_b200_solve_save_at_host.restype = C.c_int
        L.pn_b200_solve_save_at_host.argtypes = [C.POINTER(Desc)] + [dp] * 17 + [C.c_int]
        L.pn_b200_get_kernel_info.restype = C.c_int
        L.pn_b200_get_kernel_info.argtypes = [C.POINTER(Desc), C.POINTER(KernelInfo)]
        L.pn_b200_measure_fp64_peak.restype = C.c_int
        L.pn_b200_measure_fp64_peak.argtypes = [C.POINTER(C.c_double), vp]
        L.pn_b200_markov_sample.restype = C.c_int
        L.pn_b200_markov_sample.argtypes = [C.POINTER(Desc), vp, C.c_size_t, vp, C.c_uint64, C.c_int64, vp, vp]
        L.pn_b200_log_marginal_likelihood.restype = C.c_int
        L.pn_b200_log_marginal_likelihood.argtypes = [C.POINTER(Desc), vp, C.c_size_t, vp, vp, vp, vp, vp]
        L.pn_b200_set_profiling.restype = C.c_int
        L.pn_b200_set_profiling.argtypes = [C.c_int]
        L.pn_b200_get_last_timing.restype = C.c_int
        L.pn_b200_get_last_timing.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.pn_b200_last_error.restype = C.c_char_p
        L.pn_b200_last_error.argtypes = []
        L.pn_b200_register_problem.restype = C.c_int
        L.pn_b200_register_problem.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int32, C.c_int32, C.c_int32,
                                               C.POINTER(C.c_int32)]  # fmt: skip
        L.pn_b200_problem_evaluate.restype = C.c_int
        L.pn_b200_problem_evaluate.argtypes = [C.c_int32, C.c_int32, C.c_int64] + [vp] * 6
        L.pn_b200_problem_evaluate_at.restype = C.c_int
        L.pn_b200_problem_evaluate_at.argtypes = [C.c_int32, C.c_int32, C.c_int64] + [vp] * 7
        L.pn_b200_compile.restype = C.c_int
        L.pn_b200_compile.argtypes = [C.POINTER(Desc)]
        _lib = L
    return _lib


class SolverError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        msg = lib().pn_b200_last_error().decode()
        if rc == -1:
            raise NotImplementedError(f"pn_b200: unsupported configuration: {msg}")
        if rc == -2:
            raise ValueError(f"pn_b200: bad argument: {msg}")
        raise SolverError(f"pn_b200 error {rc}: {msg}")


def supported(desc):
    return lib().pn_b200_supported(C.byref(desc)) == 0


def workspace_bytes(desc):
    check(lib().pn_b200_supported(C.byref(desc)))
    return int(lib().pn_b200_workspace_bytes(C.byref(desc)))


def output_sizes(desc):
    """Element counts of every output buffer (pn_b200_output_sizes)."""
    sz = Sizes()
    check(lib().pn_b200_output_sizes(C.byref(desc), C.byref(sz)))
    return {name: int(getattr(sz, name)) for name, _ in Sizes._fields_}


def register_problem(name, source, *, d, ode_order=1, num_params=0, form="simple", time_dependent=False):
    """Compile a user-defined vector field (CUDA C++ source, see include/pn_b200.h) and return its problem id.
    ``time_dependent``: the field's functions take the time after the state.  A compile error raises ValueError
    with the compiler log."""
    if form not in SOURCE_FORMS:
        raise ValueError(f"form must be one of {sorted(SOURCE_FORMS)}")
    code = SOURCE_FORMS[form] | (FORM_TIME_DEPENDENT if time_dependent else 0)
    pid = C.c_int32(-1)
    check(lib().pn_b200_register_problem(name.encode(), source.encode(), code, int(d), int(ode_order), int(num_params),
                                         C.byref(pid)))  # fmt: skip
    return pid.value


def compile_kernels(desc):
    """Compile and load the kernels that serve `desc` now (user problems; a no-op for built-in ones)."""
    check(lib().pn_b200_compile(C.byref(desc)))


def problem_evaluate_device(problem, nu, u0, params, *, d, ode_order, f=True, taylor=True, jac=True, stream=None, t=None):
    """The functor of `problem` at n states u0 [n, ode_order, d] (torch CUDA float64) and times t [n] (None: 0):
    dict with f [n, d], taylor [n, nu + 1, d] (the Taylor-mode initialisation) and jac [n, d, ode_order * d], as
    requested."""
    import torch

    dev = u0.device
    n = u0.shape[0]
    u0 = u0.to(torch.float64).contiguous()
    params = None if params is None else params.to(device=dev, dtype=torch.float64).contiguous()
    if t is not None:
        t = torch.as_tensor(t, dtype=torch.float64, device=dev).contiguous()
        if t.shape != (n,):
            raise ValueError(f"t must have shape ({n},), got {tuple(t.shape)}")
    f64 = dict(dtype=torch.float64, device=dev)
    out = {}
    if f:
        out["f"] = torch.empty((n, d), **f64)
    if taylor:
        out["taylor"] = torch.empty((n, nu + 1, d), **f64)
    if jac:
        out["jac"] = torch.empty((n, d, ode_order * d), **f64)

    def ptr(x):
        return None if x is None else C.c_void_p(x.data_ptr())

    s = torch.cuda.current_stream(dev) if stream is None else stream
    with torch.cuda.device(dev):
        rc = lib().pn_b200_problem_evaluate_at(int(problem), int(nu), int(n), ptr(t), ptr(u0), ptr(params), ptr(out.get("f")),
                                               ptr(out.get("taylor")), ptr(out.get("jac")), C.c_void_p(s.cuda_stream))  # fmt: skip
    check(rc)
    return out


def kernel_info(desc):
    info = KernelInfo()
    check(lib().pn_b200_get_kernel_info(C.byref(desc), C.byref(info)))
    return {name: getattr(info, name) for name, _ in KernelInfo._fields_}


def measure_fp64_peak(stream=0):
    out = C.c_double(0.0)
    check(lib().pn_b200_measure_fp64_peak(C.byref(out), C.c_void_p(stream)))
    return out.value


def set_profiling(enable):
    check(lib().pn_b200_set_profiling(C.c_int(1 if enable else 0)))


def last_timing():
    """(solver-kernel ms, smoothing-kernel ms) of the last profiled solve; waits for it."""
    a, b = C.c_float(0), C.c_float(0)
    check(lib().pn_b200_get_last_timing(C.byref(a), C.byref(b)))
    return a.value, b.value


def markov_sample_device(desc, workspace, status, seed, num_samples, stream=None):
    """[B, S, K, d] joint samples (torch CUDA tensor) from the conditionals a finished solve left in `workspace`."""
    import torch

    dev = workspace.device
    out = torch.empty((desc.batch, int(num_samples), desc.num_save_at, desc.d), dtype=torch.float64, device=dev)
    s = torch.cuda.current_stream(dev) if stream is None else stream
    with torch.cuda.device(dev):
        rc = lib().pn_b200_markov_sample(
            C.byref(desc), C.c_void_p(workspace.data_ptr()), C.c_size_t(workspace.numel() * workspace.element_size()),
            C.c_void_p(status.data_ptr()), C.c_uint64(int(seed) & (2**64 - 1)), C.c_int64(int(num_samples)),
            C.c_void_p(out.data_ptr()), C.c_void_p(s.cuda_stream),
        )  # fmt: skip
    check(rc)
    return out


def log_marginal_likelihood_device(desc, workspace, status, data, obs_std, stream=None):
    """[B] log marginal likelihoods (torch CUDA tensor) of `data` [B, K, d] observed with noise `obs_std`
    [B, K] at the checkpoints, from the conditionals a finished fixed-point solve left in `workspace`."""
    import torch

    dev = workspace.device
    B, K, d = desc.batch, desc.num_save_at, desc.d
    data = torch.as_tensor(data, dtype=torch.float64, device=dev).expand(B, K, d).contiguous()
    obs_std = torch.as_tensor(obs_std, dtype=torch.float64, device=dev).expand(B, K).contiguous()
    out = torch.empty((B,), dtype=torch.float64, device=dev)
    s = torch.cuda.current_stream(dev) if stream is None else stream
    with torch.cuda.device(dev):
        rc = lib().pn_b200_log_marginal_likelihood(
            C.byref(desc), C.c_void_p(workspace.data_ptr()), C.c_size_t(workspace.numel() * workspace.element_size()),
            C.c_void_p(status.data_ptr()), C.c_void_p(data.data_ptr()), C.c_void_p(obs_std.data_ptr()),
            C.c_void_p(out.data_ptr()), C.c_void_p(s.cuda_stream),
        )  # fmt: skip
    check(rc)
    return out


def _np_ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _chol_shape(desc):
    """marg_chol: [B, K, n, n] (isotropic, dense d == 1), [B, K, d, n, n] (blockdiag) or
    [B, K, D, D] (dense, D = n d, derivative-major)."""
    B, K, d, n = desc.batch, desc.num_save_at, desc.d, desc.nu + 1
    if desc.factorisation == FACTORISATIONS["blockdiag"]:
        return (B, K, d, n, n)
    if desc.factorisation == FACTORISATIONS["dense"] and d > 1:
        return (B, K, n * d, n * d)
    return (B, K, n, n)


def _traj_std_shape(desc):
    """traj_std: [cap, B], or [cap, d, B] for the dense factorisation with d > 1 (one std per dimension; the
    size pn_b200_output_sizes reports)."""
    cap, B, d = desc.traj_capacity, desc.batch, desc.d
    if desc.factorisation == FACTORISATIONS["dense"] and d > 1:
        return (cap, d, B)
    return (cap, B)


class _HostPool:
    """Recycled page-locked result buffers for the host entry point.

    Fresh pageable arrays cost a page fault per 4 KB while the device-to-host copy fills them, and
    page-locking a fresh buffer on every call costs more than it saves.  So large result buffers are
    page-locked ONCE (torch's pinned allocator) and come back here when the numpy array handed to the
    caller -- and every view of it -- has been garbage collected; the next solve of the same size takes
    them again.  Capped; anything beyond the cap is simply freed."""

    MIN_BYTES = 1 << 20
    MAX_POOLED_BYTES = 2 << 30

    def __init__(self):
        self.free = {}
        self.pooled = 0

    def take(self, shape, dtype):
        import weakref

        import torch

        nbytes = int(np.prod(shape, dtype=np.int64)) * np.dtype(dtype).itemsize
        blocks = self.free.get(nbytes)
        if blocks:
            block = blocks.pop()
            self.pooled -= nbytes
        else:
            block = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        base = block.numpy()
        weakref.finalize(base, self._give_back, block, nbytes)
        return base.view(dtype).reshape(shape)

    def _give_back(self, block, nbytes):
        if self.pooled + nbytes <= self.MAX_POOLED_BYTES:
            self.free.setdefault(nbytes, []).append(block)
            self.pooled += nbytes


_host_pool = _HostPool()


def _scale_shape(desc):
    """output_scale: [B, K], or [B, K, d] for blockdiag (one scale per dimension)."""
    if desc.factorisation == FACTORISATIONS["blockdiag"] and desc.d > 1:
        return (desc.batch, desc.num_save_at, desc.d)
    return (desc.batch, desc.num_save_at)


def _host_empty(shape, dtype=np.float64):
    """Result buffer on the host: recycled page-locked memory for large results, plain numpy otherwise."""
    nbytes = int(np.prod(shape, dtype=np.int64)) * np.dtype(dtype).itemsize
    if nbytes >= _HostPool.MIN_BYTES:
        try:
            import torch

            if torch.cuda.is_available():
                return _host_pool.take(shape, dtype)
        except (ImportError, RuntimeError):
            pass
    return np.empty(shape, dtype=dtype)


def _grid_desc(desc, save_at):
    """`desc` for a grid of shape [K] (shared by all members), or a copy with FLAG_MEMBER_GRIDS set for a grid
    of shape [B, K] (row b: member b's grid)."""
    if save_at is None or save_at.ndim == 1:
        if desc.flags & FLAG_MEMBER_GRIDS:
            raise ValueError(f"FLAG_MEMBER_GRIDS needs save_at of shape ({desc.batch}, {desc.num_save_at})")
        return desc
    if tuple(save_at.shape) != (desc.batch, desc.num_save_at):
        raise ValueError(f"save_at must have shape ({desc.num_save_at},) or ({desc.batch}, {desc.num_save_at}), "
                         f"got {tuple(save_at.shape)}")  # fmt: skip
    desc = Desc.from_buffer_copy(desc)
    desc.flags |= FLAG_MEMBER_GRIDS
    return desc


def solve_host(desc, u0, params, tol, save_at, output_scale0, *, full=False, device=0):
    """Host-buffer entry point (numpy in, numpy out).  save_at: [K], or [B, K] for one grid per member."""
    B, K, d, n = desc.batch, desc.num_save_at, desc.d, desc.nu + 1
    f64 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)  # noqa: E731
    u0, params, tol, save_at, output_scale0 = map(f64, (u0, params, tol, save_at, output_scale0))
    desc = _grid_desc(desc, save_at)
    out = {
        "u": _host_empty((B, K, d)),
        "u_std": _host_empty((B, K, d)),
        "n_accepted": _host_empty((B, K), np.int64),
        "n_rejected": _host_empty((B,), np.int64),
        "status": _host_empty((B,), np.int32),
    }
    mm = _host_empty((B, K, n, d)) if full else None
    mc = _host_empty(_chol_shape(desc)) if full else None
    sc = _host_empty(_scale_shape(desc)) if full else None
    rec = bool(desc.flags & FLAG_RECORD)
    cap = desc.traj_capacity
    tt = _host_empty((cap, B)) if rec else None
    tu = _host_empty((cap, d, B)) if rec else None
    ts = _host_empty(_traj_std_shape(desc)) if rec else None
    tl = _host_empty((B,), np.int64) if rec else None
    rc = lib().pn_b200_solve_save_at_host(
        C.byref(desc), _np_ptr(u0), _np_ptr(params), _np_ptr(tol), _np_ptr(save_at), _np_ptr(output_scale0),
        _np_ptr(out["u"]), _np_ptr(out["u_std"]), _np_ptr(mm), _np_ptr(mc), _np_ptr(sc),
        _np_ptr(out["n_accepted"]), _np_ptr(out["n_rejected"]), _np_ptr(out["status"]),
        _np_ptr(tt), _np_ptr(tu), _np_ptr(ts), _np_ptr(tl), C.c_int(device),
    )  # fmt: skip
    check(rc)
    if full:
        out["marg_mean"], out["marg_chol"], out["output_scale"] = mm, mc, sc
    if rec:
        out.update(traj_t=tt, traj_u=tu, traj_std=ts, traj_len=tl)
    return out


def solve_device(desc, u0, params, tol, save_at, output_scale0, *, full=False, workspace=None, out=None, stream=None):
    """Device-pointer entry point: torch CUDA tensors in, torch CUDA tensors out (asynchronous).  save_at: [K], or
    [B, K] for one grid per member (each row strictly increasing: not checked here)."""
    import torch

    dev = u0.device
    B, K, d, n = desc.batch, desc.num_save_at, desc.d, desc.nu + 1
    f64 = dict(dtype=torch.float64, device=dev)

    def ptr(x):
        return None if x is None else C.c_void_p(x.data_ptr())

    def chk(x, name):
        if x is None:
            return None
        if x.device != dev or x.dtype != torch.float64 or not x.is_contiguous():
            raise ValueError(f"{name}: need a contiguous float64 tensor on {dev}")
        return x

    u0, params, tol, save_at, output_scale0 = (
        chk(x, nm) for x, nm in zip((u0, params, tol, save_at, output_scale0), ("u0", "params", "tol", "save_at", "output_scale0"))
    )
    desc = _grid_desc(desc, save_at)
    if out is None:
        out = {
            "u": torch.empty((B, K, d), **f64),
            "u_std": torch.empty((B, K, d), **f64),
            "n_accepted": torch.empty((B, K), dtype=torch.int64, device=dev),
            "n_rejected": torch.empty(B, dtype=torch.int64, device=dev),
            "status": torch.empty(B, dtype=torch.int32, device=dev),
        }
        if full:
            out["marg_mean"] = torch.empty((B, K, n, d), **f64)
            out["marg_chol"] = torch.empty(_chol_shape(desc), **f64)
            out["output_scale"] = torch.empty(_scale_shape(desc), **f64)
        if desc.flags & FLAG_RECORD:
            cap = desc.traj_capacity
            out["traj_t"] = torch.empty((cap, B), **f64)
            out["traj_u"] = torch.empty((cap, d, B), **f64)
            out["traj_std"] = torch.empty(_traj_std_shape(desc), **f64)
            out["traj_len"] = torch.empty(B, dtype=torch.int64, device=dev)
    need = workspace_bytes(desc)
    if workspace is None or workspace.numel() * workspace.element_size() < need:
        workspace = torch.empty((need + 7) // 8, dtype=torch.int64, device=dev)
    s = torch.cuda.current_stream(dev) if stream is None else stream
    with torch.cuda.device(dev):
        rc = lib().pn_b200_solve_save_at(
            C.byref(desc), ptr(u0), ptr(params), ptr(tol), ptr(save_at), ptr(output_scale0),
            ptr(out["u"]), ptr(out["u_std"]), ptr(out.get("marg_mean")), ptr(out.get("marg_chol")),
            ptr(out.get("output_scale")),
            ptr(out["n_accepted"]), ptr(out["n_rejected"]), ptr(out["status"]),
            ptr(out.get("traj_t")), ptr(out.get("traj_u")), ptr(out.get("traj_std")), ptr(out.get("traj_len")),
            C.c_void_p(workspace.data_ptr()), C.c_size_t(workspace.numel() * workspace.element_size()),
            C.c_void_p(s.cuda_stream),
        )  # fmt: skip
    check(rc)
    out["_workspace"] = workspace
    return out
