"""Initial value problems (mirror of src/odecheckpts/ivps.py).

Each constructor returns what the reference's returns -- ``(vf, u0, time_span[, params])`` --
but ``vf`` is a :class:`VectorField`: a tag for a vector field that is COMPILED INTO the CUDA
kernels as a device functor (csrc/pn_problems.cuh).  It keeps the reference's calling
convention ``vf(*u, t=..., p=...)`` (src/odecheckpts/ivpsolvers.py:59-60) so user code that wraps
it in lambdas keeps working: the solver discovers the functor behind any wrapper by calling
it once with tracer arguments (the moral equivalent of jax tracing).  Called with real
arrays it evaluates the same formula with numpy on the host (handy for truth solutions).

Other ODEs: :func:`cuda_vector_field` compiles a user's CUDA C++ vector field at run time into
the same kernels.
"""

import threading

import numpy as np

from . import _cabi
from ._cabi import PROBLEM_IDS

_trace = threading.local()


class _Tracer:
    """Stands in for an ODE state while the solver looks for the VectorField behind a wrapper."""

    def __init__(self, shape):
        self.shape = tuple(shape)


class VectorField:
    def __init__(self, name, d, ode_order, num_params, fun, problem_id=None, time_dependent=False):
        self.name = name
        self.problem_id = PROBLEM_IDS[name] if problem_id is None else problem_id
        self.d = d
        self.ode_order = ode_order
        self.num_params = num_params
        self.time_dependent = time_dependent
        self._fun = fun

    def __call__(self, *u, t=None, p=()):
        if any(isinstance(x, _Tracer) for x in u):
            rec = getattr(_trace, "records", None)
            if rec is not None:
                rec.append((self, p))
            return _Tracer(u[0].shape)
        if self._fun is None:
            raise TypeError(f"{self.name}: no host function was given (cuda_vector_field(..., host=...))")
        args = [np.asarray(x, dtype=np.float64) for x in u] + _flat_params(p)
        if self.time_dependent:
            return self._fun(*args, t=t)
        return self._fun(*args)

    def __repr__(self):
        return f"VectorField({self.name!r}, d={self.d}, ode_order={self.ode_order})"


def _flat_params(p):
    if p is None:
        return []
    if np.ndim(p) == 0 and not isinstance(p, (tuple, list)):
        return [p]
    return list(p)


def resolve_vector_field(vf, u0, t0=0.0):
    """Find the VectorField (and the parameters bound to it) behind an arbitrary Python wrapper."""
    if isinstance(vf, VectorField):
        return vf, None
    _trace.records = []
    try:
        tracers = [_Tracer(np.shape(x)) for x in u0]
        try:
            vf(*tracers, t=t0)
        except TypeError:
            vf(*tracers)
        records = _trace.records
    finally:
        _trace.records = None
    if len(records) != 1:
        raise TypeError(
            "the vector field must be (a wrapper around) one odecheckpts_b200.ivps VectorField: vector "
            "fields are compiled into the CUDA kernels as device functors, arbitrary Python callables "
            "cannot run on the GPU; write the vector field in CUDA C++ with ivps.cuda_vector_field"
        )
    return records[0]


def cuda_vector_field(name, source, *, d, ode_order=1, num_params=0, form="simple", host=None, time_dependent=False):
    """A user-defined vector field, compiled at run time into the solver kernels.

    ``source`` is CUDA C++.  ``form="simple"``: one function templated on the number type,

        template <class T> PN_DEV void vf(const T* u, const double* p, T* f)

    with u = (u, u', ...) of length ode_order * d, p the num_params parameters and f of length d;
    T is double or a truncated Taylor series (pn::Jet), so use arithmetic, fma, sqrt, rcp, exp, log,
    sin, cos and pow.  An optional ``PN_DEV void jac(const double* u, const double* p, double* J)``
    (J[d][ode_order * d]) replaces the derived Jacobian.  ``form="full"``: a ``struct Problem`` with the
    interface of the built-in functors (csrc/pn_problems.cuh).  Compile errors raise ValueError with
    the compiler log; its line numbers are the lines of ``source``.

    ``time_dependent=True`` registers a non-autonomous field: the functions take the time after the
    state, ``vf(const T* u, const T& t, const double* p, T* f)`` and ``jac(u, double t, p, J)``
    (``form="full"``: ``TIME = true``, ``vf(u, t, p, f)``, ``jac(u, t, p, J)``, ``vf_jet<N>(U, Tc, p, F)``).
    The solver evaluates the field at the time the step or checkpoint it attempts commits.

    ``host`` is an optional numpy function ``host(*u, *params)`` (``host(*u, *params, t=t)`` for a
    time-dependent field) kept for truth solutions; it is what the returned VectorField evaluates
    when called with arrays."""
    pid = _cabi.register_problem(name, source, d=d, ode_order=ode_order, num_params=num_params, form=form,
                                 time_dependent=time_dependent)  # fmt: skip
    return VectorField(name, d, ode_order, num_params, host, problem_id=pid, time_dependent=time_dependent)


# ---- the zoo ---------------------------------------------------------------------------------


def logistic():
    """ivps.py:8-17 (diffeqzoo logistic: u' = a u (1 - b u), u0 = 0.1, t in [0, 2.5])."""
    vf = VectorField("logistic", 1, 1, 2, lambda u, a, b: a * u * (1.0 - b * u))
    return vf, (np.array([0.1]),), (0.0, 2.5), (1.0, 1.0)


def rigid_body(*, time_span=(0.0, 10.0)):
    """ivps.py:20-29 (diffeqzoo rigid_body)."""

    def f(u, a, b, c):
        return np.stack([a * u[..., 1] * u[..., 2], b * u[..., 0] * u[..., 2], c * u[..., 0] * u[..., 1]], axis=-1)

    vf = VectorField("rigid_body", 3, 1, 3, f)
    return vf, (np.array([1.0, 0.0, 0.9]),), tuple(time_span), (-2.0, 1.25, -0.5)


THREE_BODY_MU = 0.012277471


def three_body_restricted():
    """ivps.py:32-41 (diffeqzoo three_body_restricted; parameters are baked in like the reference does)."""
    mu = THREE_BODY_MU

    def f(u, du, mu_):
        mp = 1.0 - mu_
        x, y = u[..., 0], u[..., 1]
        d1 = ((x + mu_) ** 2 + y**2) ** 1.5
        d2 = ((x - mp) ** 2 + y**2) ** 1.5
        ddx = x + 2 * du[..., 1] - mp * (x + mu_) / d1 - mu_ * (x - mp) / d2
        ddy = y - 2 * du[..., 0] - mp * y / d1 - mu_ * y / d2
        return np.stack([ddx, ddy], axis=-1)

    inner = VectorField("three_body", 2, 2, 1, f)

    def vf(*u, t=None, p=()):  # noqa: ARG001  (ivps.py:38-39 ignores p)
        return inner(*u, t=t, p=(mu,))

    u0 = np.array([0.994, 0.0])
    du0 = np.array([0.0, -2.00158510637908252240537862224])
    return vf, (u0, du0), (0.0, 17.0652165601579625588917206249)


def pleiades_2nd():
    """ivps.py:59-99."""
    # fmt: off
    u0 = np.array([3.0, 3.0, -1.0, -3.00, 2.0, -2.00, 2.0, 3.0, -3.0, 2.0, 0.00, 0.0, -4.00, 4.0])
    du0 = np.array([0.0, 0.0, 0.0, 0.00, 0.0, 1.75, -1.5, 0.0, 0.0, 0.0, -1.25, 1.0, 0.00, 0.0])
    # fmt: on

    def f(u, du):  # noqa: ARG001
        x, y = u[0:7], u[7:14]
        dx, dy = x[None, :] - x[:, None], y[None, :] - y[:, None]
        r3 = (dx**2 + dy**2) ** 1.5
        np.fill_diagonal(r3, np.inf)
        mj = np.arange(1, 8)[None, :]
        return np.concatenate([np.sum(mj * dx / r3, axis=1), np.sum(mj * dy / r3, axis=1)])

    vf = VectorField("pleiades", 14, 2, 0, f)
    return vf, (u0, du0), (0.0, 3.0)


def brusselator(N, t0=0.0, tmax=10.0, alpha=1.0 / 50.0):
    """ivps.py:124-156.  The reference hard-codes alpha = 1/50 (ivps.py:128); here it is the
    problem's parameter so ensembles can vary it (BASELINE config 5)."""

    def f(y, alpha_):
        c = alpha_ * (N + 1) ** 2
        u, v = y[:N], y[N:]
        u_ = np.concatenate([[1.0], u, [1.0]])
        v_ = np.concatenate([[3.0], v, [3.0]])
        lap_u = u_[:-2] - 2 * u + u_[2:]
        lap_v = v_[:-2] - 2 * v + v_[2:]
        return np.concatenate([1.0 + u**2 * v - 4 * u + c * lap_u, 3 * u - u**2 * v + c * lap_v])

    vf = VectorField("brusselator", 2 * N, 1, 1, f)
    x0 = np.linspace(0, 1, num=N)
    y0 = np.concatenate([np.sin(2 * np.pi * x0) + 1, 3.0 * np.ones(N)])
    return vf, (y0,), (t0, tmax), (alpha,)


def van_der_pol(mu=10.0**3):
    """ivps.py:159-167; mu is the problem's parameter (bound here like the reference's closure)."""
    inner = VectorField("van_der_pol", 1, 2, 1, lambda y, yd, mu_: mu_ * (yd * (1 - y**2) - y))

    def vf(y, ydot, *, t=None, p=()):  # noqa: ARG001
        return inner(y, ydot, t=t, p=(mu,))

    vf.inner = inner
    return vf, (np.array([2.0]), np.array([0.0])), (0.0, 6.3)


def lotka_volterra():
    """diffeqzoo lotka_volterra defaults."""

    def f(u, a, b, c, d):
        return np.stack([a * u[..., 0] - b * u[..., 0] * u[..., 1], -c * u[..., 1] + d * u[..., 0] * u[..., 1]], axis=-1)

    vf = VectorField("lotka_volterra", 2, 1, 4, f)
    return vf, (np.array([20.0, 20.0]),), (0.0, 20.0), (0.5, 0.05, 0.5, 0.05)
