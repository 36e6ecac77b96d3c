"""PyTorch autograd for the RK4 step and the single-shooting rollout.

The forward pass calls the value entries (`BatchEvaluator.step_rk4`, `BatchEvaluator.rollout_rk4`); the backward pass calls the
reverse-mode entries (`step_rk4_vjp`, `rollout_rk4_vjp`), which contract the adjoint with the per-stage derivative matrices on the
GPU and never form the dense step Jacobian.  Both functions are first-order only (`once_differentiable`).  `step_rk4_2` is the step
differentiable twice: its backward is itself a differentiable Function of the step VJP, whose backward is one Hessian-vector product
(`step_rk4_hvp`), so double backward, `torch.autograd.functional.hessian` and `gradgradcheck` work without any dense matrix.

    from mpc_fatigue_b200 import autograd as mad
    qt, qdt, ft = mad.rollout_rk4(ev, q0, qd0, f0, tau, N, dt)   # tau.requires_grad_()
    loss = (ft[:, -B:] ** 2).sum(); loss.backward()              # tau.grad = d loss / d tau
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

from .evaluator import BatchEvaluator


def _grad(g: torch.Tensor | None) -> torch.Tensor | None:
    return None if g is None else g.contiguous()


class _StepRK4(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ev: BatchEvaluator, q, qd, tau, f, dt):
        ctx.ev = ev
        ctx.dt_tensor = isinstance(dt, torch.Tensor)
        ctx.save_for_backward(q, qd, tau, f, *((dt,) if ctx.dt_tensor else ()))
        if not ctx.dt_tensor:
            ctx.dt = float(dt)
        return ev.step_rk4(q, qd, tau, f, dt)

    @staticmethod
    @once_differentiable
    def backward(ctx, gqn, gqdn, gfn):
        q, qd, tau, f, *rest = ctx.saved_tensors
        dt = rest[0] if ctx.dt_tensor else ctx.dt
        want_dt = ctx.dt_tensor and ctx.needs_input_grad[5]
        out = ctx.ev.step_rk4_vjp(q, qd, tau, f, dt, _grad(gqn), _grad(gqdn), _grad(gfn), want_dt=want_dt)
        gq, gqd, gtau, gf = out[:4]
        return None, gq, gqd, gtau, gf, (out[4] if want_dt else None)


class _StepRK4Vjp(torch.autograd.Function):
    """(gq, gqd, gtau, gf[, gdt]) = lambda^T J of the step as a function of (q, qd, tau, f, dt) and lambda = (lq, lqd, lf).  Its
    backward with the cotangent v of these outputs is (H v for z, J v for lambda): one `step_rk4_hvp` call."""

    @staticmethod
    def forward(ctx, ev: BatchEvaluator, q, qd, tau, f, dt, lq, lqd, lf):
        ctx.ev = ev
        ctx.dt_tensor = isinstance(dt, torch.Tensor)
        ctx.save_for_backward(q, qd, tau, f, dt if ctx.dt_tensor else None, lq, lqd, lf)
        if not ctx.dt_tensor:
            ctx.dt = float(dt)
        return ev.step_rk4_vjp(q, qd, tau, f, dt, lq, lqd, lf, want_dt=ctx.dt_tensor)

    @staticmethod
    @once_differentiable
    def backward(ctx, vq, vqd, vtau, vf, vdt=None):
        q, qd, tau, f, dt, lq, lqd, lf = ctx.saved_tensors
        if not ctx.dt_tensor:
            dt = ctx.dt
        want_dt = ctx.dt_tensor and ctx.needs_input_grad[5]
        want_jv = any(ctx.needs_input_grad[6:9])
        out = ctx.ev.step_rk4_hvp(q, qd, tau, f, dt, (lq, lqd, lf), tuple(_grad(g) for g in (vq, vqd, vtau, vf, vdt)),
                                  want_dt=want_dt, want_jv=want_jv)
        hdt = out[4] if want_dt else None
        jq, jqd, jf = out[-1] if want_jv else (None, None, None)
        return None, *out[:4], hdt, jq, jqd, jf


class _StepRK4Twice(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ev: BatchEvaluator, q, qd, tau, f, dt):
        ctx.ev = ev
        ctx.dt_tensor = isinstance(dt, torch.Tensor)
        ctx.save_for_backward(q, qd, tau, f, *((dt,) if ctx.dt_tensor else ()))
        if not ctx.dt_tensor:
            ctx.dt = float(dt)
        return ev.step_rk4(q, qd, tau, f, dt)

    @staticmethod
    def backward(ctx, gqn, gqdn, gfn):
        q, qd, tau, f, *rest = ctx.saved_tensors
        dt = rest[0] if ctx.dt_tensor else ctx.dt
        out = _StepRK4Vjp.apply(ctx.ev, q, qd, tau, f, dt, _grad(gqn), _grad(gqdn), _grad(gfn))
        return None, *out[:4], (out[4] if ctx.dt_tensor else None)


class _RolloutRK4(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ev: BatchEvaluator, q0, qd0, f0, tau, N: int, dt: float):
        qt, qdt, ft = ev.rollout_rk4(q0, qd0, f0, tau, N, dt)
        ctx.ev, ctx.N, ctx.dt = ev, int(N), float(dt)
        ctx.save_for_backward(q0, qd0, f0, tau, qt, qdt, ft)
        return qt, qdt, ft

    @staticmethod
    @once_differentiable
    def backward(ctx, gqt, gqdt, gft):
        q0, qd0, f0, tau, qt, qdt, ft = ctx.saved_tensors
        gtau, gq0, gqd0, gf0 = ctx.ev.rollout_rk4_vjp(q0, qd0, f0, tau, ctx.N, ctx.dt, (qt, qdt, ft), _grad(gqt), _grad(gqdt), _grad(gft))
        return None, gq0, gqd0, gf0, gtau, None, None


def step_rk4(ev: BatchEvaluator, q, qd, tau, f, dt):
    """(q+, qd+, f+) = one RK4 step (`BatchEvaluator.step_rk4`), differentiable in q, qd, tau, f, and in dt when dt is a
    per-unit tensor [U]."""
    return _StepRK4.apply(ev, q, qd, tau, f, dt)


def step_rk4_2(ev: BatchEvaluator, q, qd, tau, f, dt):
    """`step_rk4`, differentiable twice: the same values and first derivatives, and a backward that is itself differentiable (in
    q, qd, tau, f, dt as a [U] tensor, and in the incoming cotangents)."""
    return _StepRK4Twice.apply(ev, q, qd, tau, f, dt)


def rollout_rk4(ev: BatchEvaluator, q0, qd0, f0, tau, N: int, dt: float):
    """(qt, qdt, ft) = single-shooting rollout (`BatchEvaluator.rollout_rk4`), differentiable in x0 = (q0, qd0, f0) and tau
    (not in the scalar dt)."""
    return _RolloutRK4.apply(ev, q0, qd0, f0, tau, int(N), float(dt))
