"""torch.autograd functions of the dynamics: gradients of a loss of tau or ydd with respect to q, yd and ydd / tau.

    tau = grbda.autograd.inverse_dynamics(m, q, yd, ydd)
    ydd = grbda.autograd.forward_dynamics(m, q, yd, tau)

The forward pass runs the model's inverse / forward dynamics kernels, the backward pass one launch of the
vector-Jacobian product kernel (grbda_cuda_{inverse,forward}_dynamics_vjp_f64): the gradient of a scalar costs a
small multiple of one evaluation, without building the nv x nv Jacobians. FP64 only, first derivatives only
(a backward with create_graph=True raises). The gradient of q is taken with respect to the stored position
entries; for the forward dynamics its component off the unit quaternion / the loop-constraint manifold is
defined in include/grbda_cuda.h.
"""
import functools

import torch
from torch.autograd.function import once_differentiable


def _first_order(backward):
    """once_differentiable, and a backward with create_graph=True fails at once instead of when its result is used."""
    inner = once_differentiable(backward)

    @functools.wraps(backward)
    def wrapper(ctx, grad):
        if torch.is_grad_enabled():
            raise RuntimeError("grbda.autograd: the dynamics are differentiable once; backward with create_graph=True "
                               "(second derivatives) is not supported")
        return inner(ctx, grad)
    return wrapper


def _check_inputs(*tensors):
    for t in tensors:
        if t.dtype != torch.float64:
            raise TypeError("grbda.autograd: float64 tensors are required, got %s" % t.dtype)


def _backward(ctx, grad, vjp):
    need = ctx.needs_input_grad[1:]
    if not any(need):
        return None, None, None, None
    q, yd, aux = ctx.saved_tensors
    bars = vjp(q, yd, aux, grad.contiguous())
    return (None,) + tuple(b if n else None for b, n in zip(bars, need))


class _InverseDynamics(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, q, yd, ydd):
        _check_inputs(q, yd, ydd)
        ctx.model = model
        ctx.save_for_backward(q, yd, ydd)
        return model.inverseDynamics(q, yd, ydd)

    @staticmethod
    @_first_order
    def backward(ctx, grad_tau):
        return _backward(ctx, grad_tau, ctx.model.inverseDynamicsVJP)


class _ForwardDynamics(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, q, yd, tau):
        _check_inputs(q, yd, tau)
        ctx.model = model
        ctx.save_for_backward(q, yd, tau)
        return model.forwardDynamics(q, yd, tau)

    @staticmethod
    @_first_order
    def backward(ctx, grad_ydd):
        return _backward(ctx, grad_ydd, ctx.model.forwardDynamicsVJP)


def inverse_dynamics(model, q, yd, ydd):
    """tau[batch, nv] = ID(q, yd, ydd) with a grad_fn: q [batch, nq], yd / ydd [batch, nv], contiguous FP64 CUDA tensors."""
    return _InverseDynamics.apply(model, q, yd, ydd)


def forward_dynamics(model, q, yd, tau):
    """ydd[batch, nv] = FD(q, yd, tau) with a grad_fn: q [batch, nq], yd / tau [batch, nv], contiguous FP64 CUDA tensors."""
    return _ForwardDynamics.apply(model, q, yd, tau)
