"""``probdiffeq.ivpsolve``: step-size control and the solve routines, backed by libpn_b200.so.

Reference call sites: control_proportional_integral / adaptive (src/odecheckpts/ivpsolvers.py:52-53),
solve_adaptive_save_at (ivpsolvers.py:71-77, experiments/4_brusselator/run.py:122-129),
solve_adaptive_terminal_values (run.py:82-90), solve_adaptive_save_every_step
(experiments/1_van_der_pol/vdp.py:77-79), solve_fixed_grid (vdp.py:88-91).

Beyond the reference: every routine accepts BATCHED initial values (leading ensemble axis on the
Taylor-coefficient inits and/or on the vector-field parameters) and solves the whole ensemble in
one persistent-kernel launch; `tol=` gives per-member (atol, rtol).
"""

from typing import NamedTuple

import numpy as np

from .. import _cabi
from ..ivps import resolve_vector_field
from . import impl as _impl
from .ivpsolvers import InitialCondition, Solver, Strategy
from .stats import MarkovSeq, Normal


class Control(NamedTuple):
    safety: float
    factor_min: float
    factor_max: float
    power_integral_unscaled: float
    power_proportional_unscaled: float


def control_proportional_integral(
    *, safety=0.95, factor_min=0.2, factor_max=10.0, power_integral_unscaled=0.3, power_proportional_unscaled=0.4, clip=False
):
    """PI controller (SURVEY A.3).  The reference never clips steps to checkpoints (ivpsolvers.py:52)."""
    if clip:
        raise NotImplementedError("clip=True is not used by the reference and not implemented")
    return Control(safety, factor_min, factor_max, power_integral_unscaled, power_proportional_unscaled)


class AdaptiveSolver(NamedTuple):
    solver: Solver
    atol: float
    rtol: float
    control: Control


def adaptive(solver, atol=1e-4, rtol=1e-2, control=None):
    if control is None:
        control = control_proportional_integral()
    return AdaptiveSolver(solver, atol, rtol, control)


class Solution(NamedTuple):
    t: object            # [K]
    u: object            # [K, d]  (ensembles: [B, K, d])
    u_std: object        # like u
    output_scale: object
    marginals: object    # Normal(mean [K, n, d], cholesky [K, n, n]) or None
    posterior: object    # MarkovSeq or None
    num_steps: object    # [K] cumulative accepted steps (ensembles: [B, K])
    num_rejected: object  # scalar (ensembles: [B])
    status: object        # 0 ok, 1 NaN, 2 max_attempts


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _prepare(vf, init, t0, factorisation):
    """Resolve (problem functor, params, u0 batch) from the reference-style arguments."""
    if not isinstance(init, InitialCondition):
        raise TypeError("initial condition must come from solver.initial_condition(tcoeffs, output_scale)")
    tc = init.tcoeffs
    inits = tc.inits
    probe = [x[0] if np.ndim(x) == 2 else x for x in inits]
    field, p_solve = resolve_vector_field(vf, probe, t0)
    field_t, p_taylor = resolve_vector_field(tc.vf, probe, t0)
    if field_t is not field:
        raise ValueError("the Taylor initialisation and the solve must use the same vector field")
    params = p_solve if p_solve is not None else p_taylor
    if len(inits) != field.ode_order:
        raise ValueError(f"{field.name}: expected {field.ode_order} initial arrays (u, u', ...), got {len(inits)}")
    nu = tc.num + field.ode_order - 1
    fact = factorisation if factorisation is not None else _impl.impl.selected()
    return field, params, inits, nu, fact


def _stack_members(inits, params, tol, output_scale, num_params):
    """-> use_torch, B, batched, u0 [B, q, d], params [B, P] | None, tol [B, 2] | None, scale [B] | None"""
    use_torch = any(_is_torch(x) and x.is_cuda for x in inits)
    if use_torch:
        import torch

        dev = next(x.device for x in inits if _is_torch(x) and x.is_cuda)
        asarr = lambda x: torch.as_tensor(x, dtype=torch.float64, device=dev)  # noqa: E731
        stack, ndim = torch.stack, lambda x: x.dim()
        bcast = lambda x, B: x.expand(B, *x.shape).contiguous()  # noqa: E731
    else:
        asarr = lambda x: np.asarray(x.detach().cpu() if _is_torch(x) else x, dtype=np.float64)  # noqa: E731
        stack, ndim = np.stack, np.ndim
        bcast = lambda x, B: np.ascontiguousarray(np.broadcast_to(x, (B,) + x.shape))  # noqa: E731
    inits = [asarr(x) for x in inits]
    plist = [] if params is None else [asarr(x) for x in (params if isinstance(params, (tuple, list)) else (params,))]
    if len(plist) != num_params:
        raise ValueError(f"expected {num_params} vector-field parameters, got {len(plist)}")
    sizes = [x.shape[0] for x in inits if ndim(x) == 2] + [x.shape[0] for x in plist if ndim(x) == 1]
    if tol is not None:
        tol = asarr(tol)
        if ndim(tol) == 2:
            sizes.append(tol.shape[0])
    batched = len(sizes) > 0
    B = sizes[0] if batched else 1
    if any(s != B for s in sizes):
        raise ValueError(f"inconsistent ensemble sizes {sizes}")
    inits = [x if ndim(x) == 2 else bcast(x, B) for x in inits]
    u0 = stack(inits, 1)
    u0 = u0.contiguous() if use_torch else np.ascontiguousarray(u0)
    par = None
    if plist:
        par = stack([x if ndim(x) == 1 else bcast(x, B) for x in plist], 1)
        par = par.contiguous() if use_torch else np.ascontiguousarray(par)
    if tol is not None:
        tol = tol if ndim(tol) == 2 else bcast(tol, B)
        tol = tol.contiguous() if use_torch else np.ascontiguousarray(tol)
    scale = None
    if output_scale is not None and not (np.ndim(output_scale) == 0 and float(output_scale) == 1.0):
        scale = asarr(output_scale)
        scale = scale if ndim(scale) == 1 else bcast(scale, B)
        scale = scale.contiguous() if use_torch else np.ascontiguousarray(scale)
    return use_torch, B, batched, u0, par, tol, scale


def _make_desc(field, nu, fact, solver, atol, rtol, control, dt0, B, K, flags=0, traj_capacity=0, max_attempts=0):
    strat = solver.strategy
    if strat.name == "smoother":
        raise ValueError("strategy_smoother is served by solve_adaptive_save_every_step + stats.offgrid_marginals_searchsorted")
    if strat.prior.num_derivatives != nu:
        raise ValueError(
            f"prior has num_derivatives={strat.prior.num_derivatives} but the Taylor coefficients carry nu={nu}"
        )
    if strat.correction.ode_order != field.ode_order:
        raise ValueError(f"correction has ode_order={strat.correction.ode_order}, the problem has {field.ode_order}")
    return _cabi.Desc(
        field.problem_id, field.d, nu, field.ode_order,
        _cabi.FACTORISATIONS[fact], _cabi.CORRECTIONS[strat.correction.name],
        _cabi.STRATEGIES[strat.name], _cabi.CALIBRATIONS[solver.calibration],
        float(atol), float(rtol), float(dt0),
        control.safety, control.factor_min, control.factor_max,
        control.power_integral_unscaled, control.power_proportional_unscaled,
        int(B), int(K), int(max_attempts), field.num_params, int(flags), int(traj_capacity),
    )  # fmt: skip


def _solve(vf, init, save_at, adaptive_solver, dt0, *, factorisation, return_marginals, tol, max_attempts, device,
           flags=0, traj_capacity=0, keep_conditionals=False):  # fmt: skip
    save_np = np.asarray(save_at.detach().cpu() if _is_torch(save_at) else save_at, dtype=np.float64)
    if save_np.ndim not in (1, 2) or save_np.shape[-1] < 2 or not np.all(np.diff(save_np, axis=-1) > 0):
        raise ValueError("save_at must be a strictly increasing grid with at least two points: [K], or [B, K] with one "
                         "row per ensemble member")  # fmt: skip
    field, params, inits, nu, fact = _prepare(vf, init, float(save_np.flat[0]), factorisation)
    use_torch, B, batched, u0, par, tol, scale = _stack_members(inits, params, tol, init.output_scale, field.num_params)
    if save_np.ndim == 2:
        if not batched:
            raise ValueError("a [B, K] grid gives every ensemble member its own grid; a single IVP takes save_at [K]")
        if save_np.shape[0] != B:
            raise ValueError(f"save_at has {save_np.shape[0]} rows for an ensemble of {B} members")
    desc = _make_desc(field, nu, fact, adaptive_solver.solver, adaptive_solver.atol, adaptive_solver.rtol,
                      adaptive_solver.control, dt0, B, save_np.shape[-1], flags, traj_capacity, max_attempts)  # fmt: skip
    if use_torch or keep_conditionals:
        import torch

        as_numpy = not use_torch
        if as_numpy:  # keep the workspace on the device: run the device path, hand numpy back
            dev = torch.device(f"cuda:{device or 0}")
            u0, par, tol, scale = (None if x is None else torch.as_tensor(x, device=dev) for x in (u0, par, tol, scale))
        save_dev = torch.as_tensor(save_np, dtype=torch.float64, device=u0.device)
        out = _cabi.solve_device(desc, u0, par, tol, save_dev, scale, full=return_marginals)
        t_out = save_dev
        if keep_conditionals:
            out["_handle"] = (desc, out["_workspace"], out["status"], as_numpy, batched)
        if as_numpy:
            t_out = save_np
            out = {k: (v.cpu().numpy() if hasattr(v, "cpu") and not k.startswith("_") else v) for k, v in out.items()}
    else:
        out = _cabi.solve_host(desc, u0, par, tol, save_np, scale, full=return_marginals, device=device or 0)
        t_out = save_np
    return desc, out, t_out, batched


def _solution(out, t_out, batched, return_marginals):
    sel = (lambda x: x) if batched else (lambda x: x[0])
    marg = post = scale = None
    if return_marginals:
        scale = sel(out["output_scale"])
        marg = Normal(sel(out["marg_mean"]), sel(out["marg_chol"]))
        mm, mc = out["marg_mean"], out["marg_chol"]
        init = Normal(sel(mm[:, 1:]), sel(mc[:, 1:])) if batched else Normal(mm[0, 1:], mc[0, 1:])
        post = MarkovSeq(init, marg, out.get("_handle"))
    return Solution(
        t=t_out, u=sel(out["u"]), u_std=sel(out["u_std"]), output_scale=scale, marginals=marg, posterior=post,
        num_steps=sel(out["n_accepted"]), num_rejected=sel(out["n_rejected"]), status=sel(out["status"]),
    )  # fmt: skip


def _span(t0, t1):
    """The grid [t0, t1]: [2], or [B, 2] when t0 or t1 is given per ensemble member ([B])."""
    t0, t1 = (np.asarray(x.detach().cpu() if _is_torch(x) else x, dtype=np.float64) for x in (t0, t1))
    if t0.ndim == 0 and t1.ndim == 0:
        return np.asarray([t0, t1])
    if t0.ndim > 1 or t1.ndim > 1:
        raise ValueError("t0 and t1 must be scalars or [B] arrays (one per ensemble member)")
    return np.stack(np.broadcast_arrays(t0, t1), axis=1)


def solve_adaptive_save_at(vf, initial_condition, save_at, adaptive_solver, dt0, *, factorisation=None,
                           return_marginals=True, tol=None, max_attempts=0, device=None, keep_conditionals=False):  # fmt: skip
    """Adaptive solve that returns the posterior at the checkpoints `save_at` with O(K) memory
    (fixed-point smoother) -- the reference's hot path (ivpsolvers.py:71-77; SURVEY 3.2).  For an ensemble,
    save_at may be [B, K]: row b is member b's grid (its own t0, t1 and checkpoints; `Solution.t` is then
    [B, K], and stats.log_marginal_likelihood observes data[b, k] at save_at[b, k])."""
    if keep_conditionals and not return_marginals:
        raise ValueError("keep_conditionals=True needs return_marginals=True (the posterior object carries the handle)")
    _, out, t_out, batched = _solve(vf, initial_condition, save_at, adaptive_solver, dt0, factorisation=factorisation,
                                    return_marginals=return_marginals, tol=tol, max_attempts=max_attempts, device=device,
                                    keep_conditionals=keep_conditionals)  # fmt: skip
    return _solution(out, t_out, batched, return_marginals)


def solve_adaptive_terminal_values(vf, initial_condition, t0, t1, adaptive_solver, dt0, *, factorisation=None,
                                   tol=None, max_attempts=0, device=None):  # fmt: skip
    """run.py:82-90: the same loop with a single checkpoint at t1.  For an ensemble, t0 and t1 may be [B]."""
    sol = solve_adaptive_save_at(vf, initial_condition, _span(t0, t1), adaptive_solver, dt0,
                                 factorisation=factorisation, return_marginals=True, tol=tol,
                                 max_attempts=max_attempts, device=device)  # fmt: skip
    last = lambda x: x[..., -1, :] if x is not None else None  # noqa: E731
    marg = Normal(sol.marginals.mean[..., -1, :, :], sol.marginals.cholesky[..., -1, :, :])
    return Solution(t=t1, u=last(sol.u), u_std=last(sol.u_std), output_scale=None, marginals=marg, posterior=None,
                    num_steps=sol.num_steps[..., -1], num_rejected=sol.num_rejected, status=sol.status)  # fmt: skip


def _with_strategy(adaptive_solver, name):
    st = adaptive_solver.solver.strategy
    solver = Solver(Strategy(name, st.prior, st.correction), adaptive_solver.solver.calibration)
    return AdaptiveSolver(solver, adaptive_solver.atol, adaptive_solver.rtol, adaptive_solver.control)


def _solve_on_checkpoints(ctx, checkpoints):
    """Smoother context -> fixed-point solve with `checkpoints` (a superset of the accepted grid) as save_at."""
    return solve_adaptive_save_at(ctx["vf"], ctx["init"], checkpoints, _with_strategy(ctx["adaptive_solver"], "fixedpoint"),
                                  ctx["dt0"], factorisation=ctx["factorisation"], return_marginals=True, device=ctx["device"])  # fmt: skip


def _solve_smoother_every_step(vf, initial_condition, t0, t1, adaptive_solver, dt0, factorisation, max_steps, device):
    """strategy_smoother + solve_adaptive_save_every_step (src/odecheckpts/ivpsolvers.py:133-142): the textbook
    O(#steps) smoother.  Pass 1 (filter kernel, trajectory recording) finds the accepted grid; pass 2 runs
    the fixed-point kernel with EVERY accepted grid point as a checkpoint: each is hit exactly, so the running
    backward conditional is emitted and reset at every step -- the workspace then holds one un-merged
    conditional per accepted step (the smoother's posterior, #steps x slot bytes of device memory) and the
    backward sweep marginalises through all of them.  Single IVP (the members of an ensemble have different
    grids; loop over them)."""
    every = solve_adaptive_save_every_step(vf, initial_condition, t0, t1, _with_strategy(adaptive_solver, "filter"), dt0,
                                           factorisation=factorisation, max_steps=max_steps, device=device)  # fmt: skip
    if np.ndim(every.t) != 1:
        raise NotImplementedError("strategy_smoother solves one IVP per call (every member has its own grid)")
    grid = np.asarray(every.t.detach().cpu() if _is_torch(every.t) else every.t, dtype=np.float64)
    ctx = dict(vf=vf, init=initial_condition, adaptive_solver=adaptive_solver, solver=adaptive_solver.solver, dt0=dt0,
               factorisation=factorisation, device=device, grid=grid)  # fmt: skip
    sol = _solve_on_checkpoints(ctx, grid)
    if int(np.asarray(sol.num_steps if not _is_torch(sol.num_steps) else sol.num_steps.cpu())[-1]) != len(grid) - 1:
        raise RuntimeError("smoother pass did not reproduce the accepted grid of the filter pass")
    post = MarkovSeq(sol.posterior.init, sol.posterior.marginals_all, None, ctx)
    return Solution(t=sol.t, u=sol.u, u_std=sol.u_std, output_scale=sol.output_scale, marginals=sol.marginals,
                    posterior=post, num_steps=len(grid) - 1, num_rejected=every.num_rejected, status=sol.status)  # fmt: skip


def solve_adaptive_save_every_step(vf, initial_condition, t0, t1, adaptive_solver, dt0, *, factorisation=None,
                                   max_steps=1 << 16, device=None):  # fmt: skip
    """vdp.py:77-79: every accepted state is recorded; the last grid point is t1 (interpolated).
    Filter strategy: the recorded filter solution (what vdp.py uses).  Smoother strategy
    (src/odecheckpts/ivpsolvers.py:133-142): the smoothed solution at every accepted grid point plus the
    per-step backward conditionals (see _solve_smoother_every_step).  Unbatched results are trimmed to the
    accepted grid; ensembles (filter only) return padded arrays plus `num_steps`.  With the dense factorisation and d > 1,
    `u_std` is per dimension: [n, d] unbatched, [cap, d, B] for ensembles; the other factorisations record one std
    for all dimensions.  For an ensemble (filter strategy), t0 and t1 may be [B]: member b's last point is at t1[b]."""
    if adaptive_solver.solver.strategy.name == "smoother":
        return _solve_smoother_every_step(vf, initial_condition, t0, t1, adaptive_solver, dt0, factorisation, max_steps, device)
    desc, out, _, batched = _solve(vf, initial_condition, _span(t0, t1), adaptive_solver, dt0,
                                   factorisation=factorisation, return_marginals=False, tol=None, max_attempts=0,
                                   device=device, flags=_cabi.FLAG_RECORD, traj_capacity=int(max_steps))  # fmt: skip
    tt, tu, ts, tl = out["traj_t"], out["traj_u"], out["traj_std"], out["traj_len"]
    per_dim = ts.ndim == 3  # dense with d > 1: one std per dimension, [cap, d, B]
    if not batched:
        n = int(tl[0])
        if n >= max_steps:
            raise RuntimeError(f"more than max_steps={max_steps} accepted steps; raise max_steps")
        u = tu[:n, :, 0]
        if per_dim:
            std = ts[:n, :, 0]
        else:
            std = ts[:n, 0][:, None] * (np.ones((1, desc.d)) if not _is_torch(ts) else 1.0)
        return Solution(t=tt[:n, 0], u=u, u_std=std, output_scale=None, marginals=None, posterior=None,
                        num_steps=n - 1, num_rejected=out["n_rejected"][0], status=out["status"][0])  # fmt: skip
    return Solution(t=tt, u=tu, u_std=ts, output_scale=None, marginals=None, posterior=None,
                    num_steps=tl - 1, num_rejected=out["n_rejected"], status=out["status"])  # fmt: skip


def solve_fixed_grid(vf, initial_condition, grid, solver, *, factorisation=None, atol=1.0, rtol=1.0, device=None):
    """vdp.py:88-91: the same step on a given grid, no error control.  For an ensemble, grid may be [B, K]: row b
    is member b's grid."""
    asolver = AdaptiveSolver(solver, atol, rtol, control_proportional_integral())
    _, out, t_out, batched = _solve(vf, initial_condition, grid, asolver, 1.0, factorisation=factorisation,
                                    return_marginals=False, tol=None, max_attempts=0, device=device,
                                    flags=_cabi.FLAG_FIXED_GRID)  # fmt: skip
    return _solution(out, t_out, batched, False)
