"""The differentiable solve: ``plan_batch_differentiable``, the dynamics-consistent ``plan_batch`` as a
``torch.autograd.Function``.

The forward is ``plan_batch(..., dynamics_consistent=True)`` (gradient mode 3, 6 with spheres, 7 with a
reference, 8 with both).  The backward is ``dart_se3mpc_solve_vjp_batch``: the implicit-function
derivative of the returned plan with its active set held (contract in include/dart_se3mpc.h), on the
GPU.  Gradients flow to the start state, the goals or the reference, and the four cost weights.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import replace
from typing import Optional

import numpy as np

from . import _cabi
from .config import SE3MPCConfig, make_params
from .planner import _torch, plan_batch, reference_rows, sphere_rows

WEIGHT_FIELDS = ("position_weight", "velocity_weight", "acceleration_weight", "thrust_weight")


class _Spec:
    """What the backward needs besides the tensors: the solve's parameters and its fixed inputs."""

    def __init__(self, cfg, params, kw, spheres, margin, has_goal, track, wdev):
        self.cfg, self.params, self.kw = cfg, params, kw
        self.spheres, self.margin, self.has_goal, self.track, self.wdev = spheres, margin, has_goal, track, wdev


def _make_fn():
    torch = _torch()

    class PlanFn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, spec, p0, v0, goal, rP, rV, w):
            ref = (rP, rV) if spec.track else None
            sol = plan_batch(p0, v0, goal, spec.cfg, dynamics_consistent=True, reference=ref, spheres=spec.spheres,
                             sphere_margin=spec.margin, has_goal=spec.has_goal, **spec.kw)
            x, cost = sol.x.contiguous(), sol.cost.clone()
            ctx.spec = spec
            ctx.save_for_backward(p0, v0, goal, rP, rV, x)
            return x, cost

        @staticmethod
        def backward(ctx, gx, gcost):
            spec = ctx.spec
            p0, v0, goal, rP, rV, x = ctx.saved_tensors
            B, dev = x.shape[0], x.device
            N = int(spec.params.horizon)
            f8 = dict(dtype=torch.float64, device=dev)
            soa = lambda t: t.detach().to(**f8).reshape(B, -1).t().contiguous()  # noqa: E731
            ins = [soa(p0), soa(v0), soa(goal) if goal is not None else None, soa(x),
                   soa(gx) if gx is not None else None, gcost.detach().to(**f8).contiguous() if gcost is not None else None]
            hg = None
            if spec.has_goal is not None:
                hg = torch.as_tensor(np.asarray(spec.has_goal, np.uint8) if not torch.is_tensor(spec.has_goal)
                                     else spec.has_goal).to(dev, torch.uint8).reshape(B).contiguous()
            ref = rows = None
            if spec.track:
                rows = reference_rows(rP.detach(), None if rV is None else rV.detach(), B, B, dev)
                ref = _cabi.TrackRef(N, 0, rows.data_ptr())
            sph = lst = None
            if spec.spheres is not None:
                s = sphere_rows(spec.spheres)
                lst = torch.as_tensor(s).to(dev) if len(s) else None
                sph = _cabi.Spheres(len(s), 0, None if lst is None else lst.data_ptr(), float(spec.margin))
            gp0, gv0 = (torch.empty((3, B), **f8) for _ in range(2))
            ggoal = None if spec.track else torch.empty((3, B), **f8)
            gref = torch.empty((6 * N, B), **f8) if spec.track else None
            gw = torch.empty((4, B), **f8)
            status = torch.empty(B, dtype=torch.int32, device=dev)
            ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
            with torch.cuda.device(dev):
                rc = _cabi.lib().dart_se3mpc_solve_vjp_batch(
                    C.byref(spec.params), B, B, *(ptr(t) for t in ins[:3]), ptr(hg), ptr(ins[3]),
                    None if ref is None else C.byref(ref), None if sph is None else C.byref(sph), ptr(ins[4]),
                    ptr(ins[5]), ptr(gp0), ptr(gv0), ptr(ggoal), ptr(gref), ptr(gw), ptr(status),
                    torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(rc, "dart_se3mpc_solve_vjp_batch")
            out = [None, gp0.t().reshape(p0.shape).to(p0.dtype), gv0.t().reshape(v0.shape).to(v0.dtype),
                   None, None, None, None]
            if goal is not None:
                # with a reference the goals are not read: their gradient is zero
                out[3] = torch.zeros_like(goal) if spec.track else ggoal.t().reshape(goal.shape).to(goal.dtype)
            if spec.track:
                out[4] = gref[:3 * N].t().reshape(rP.shape).to(rP.dtype)
                if rV is not None:
                    out[5] = gref[3 * N:].t().reshape(rV.shape).to(rV.dtype)
            if ctx.needs_input_grad[6]:
                out[6] = gw.sum(1).to(spec.wdev)
            return tuple(out)

    return PlanFn


_FN = None


def plan_batch_differentiable(positions, velocities, goals, config: Optional[SE3MPCConfig] = None, *, weights=None,
                              reference=None, spheres=None, sphere_margin: Optional[float] = None, has_goal=None,
                              x_warm=None, warm_mask=None, mass: float = 1.5, gravity: float = 9.81,
                              dt: Optional[float] = None):
    """The dynamics-consistent batched solve with gradients: returns ``(x (B, 9N), cost (B,))``, CUDA float64
    tensors, through a ``torch.autograd.Function``.

    The forward is ``plan_batch(positions, velocities, goals, config, dynamics_consistent=True, ...)`` with the
    same arguments (gradient mode 3; 6 with ``spheres``; 7 with ``reference``; 8 with both; horizons 1..16);
    its x and cost are bit-identical to that call's.  The backward holds the returned plan's active set (thrust
    entries exactly on their bounds) and differentiates the solution map through the implicit function theorem
    on the GPU (``dart_se3mpc_solve_vjp_batch``; the contract is in include/dart_se3mpc.h).  It is defined at
    whatever plan the solve returned, converged or not; where the reduced Hessian is not positive definite
    (possible with spheres) or the linear solve fails, that problem's gradients are NaN.

    positions, velocities (B, 3); goals (B, 3), or None with ``reference``; reference = (P (B, N, 3), V (B, N, 3)
    or None); ``weights``: an optional (4,) tensor (w_pos, w_vel, w_acc, w_thrust) that overrides the config's
    four cost weights.  Gradients flow to whichever of these tensors require them; the weights' gradient is
    summed over the batch.  No gradient flows to warm starts, sphere centres or radii, ``obstacle_weight`` or the
    derived arrays (attitudes, rates)."""
    global _FN
    torch = _torch()
    cfg = config or SE3MPCConfig()
    dev = torch.device("cuda", torch.cuda.current_device())

    def as_t(a):
        return (a if torch.is_tensor(a) else torch.as_tensor(np.asarray(a, np.float64))).to(dev, torch.float64)

    w = None
    if weights is not None:
        w = weights if torch.is_tensor(weights) else torch.as_tensor(np.asarray(weights, np.float64))
        if tuple(w.shape) != (4,):
            raise ValueError("weights must be a (4,) tensor: w_pos, w_vel, w_acc, w_thrust")
        cfg = replace(cfg, **{f: float(v) for f, v in zip(WEIGHT_FIELDS, w.detach().cpu().tolist())})
    track = reference is not None
    if goals is None and not track:
        raise ValueError("goals may be None only with reference=")
    mode = 6 if spheres is not None else 3
    if track:
        mode = 7 if mode == 3 else 8
    params = make_params(cfg, mass=mass, gravity=gravity, dt=dt, gradient_mode=mode)
    if not 1 <= int(params.horizon) <= 16:
        raise ValueError("plan_batch_differentiable serves horizons 1..16")
    margin = cfg.safety_margin if sphere_margin is None else float(sphere_margin)
    kw = dict(x_warm=x_warm, warm_mask=warm_mask, mass=mass, gravity=gravity, dt=dt)
    spec = _Spec(cfg, params, kw, spheres, margin, has_goal, track, None if w is None else w.device)
    p0, v0 = as_t(positions), as_t(velocities)
    goal = None if goals is None else as_t(goals)
    rP = rV = None
    if track:
        rP = as_t(reference[0])
        rV = None if reference[1] is None else as_t(reference[1])
    if _FN is None:
        _FN = _make_fn()
    wt = None if w is None else w.to(torch.float64)
    return _FN.apply(spec, p0, v0, goal, rP, rV, wt)
