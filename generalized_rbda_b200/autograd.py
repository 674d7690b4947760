"""torch.autograd functions of the dynamics, of the contact-point kinematics and of the integration / simulation
steps: gradients of a loss of tau, ydd, the contact positions / velocities or a whole rollout with respect to q, yd,
ydd / tau and the external forces.

    tau = grbda.autograd.inverse_dynamics(m, q, yd, ydd, f_ext=None)
    ydd = grbda.autograd.forward_dynamics(m, q, yd, tau, f_ext=None)
    p, v = grbda.autograd.contact_kinematics(m, q, yd)
    q1, yd1, flags = grbda.autograd.integrate(m, q, yd, ydd, dt)
    q1, yd1, flags = grbda.autograd.step(m, q, yd, tau, dt, f_ext=None)

The forward pass runs the model's kernels, the backward pass one call of the vector-Jacobian product entry point
(grbda_cuda_{inverse,forward}_dynamics_vjp_f64, their _ext_vjp_f64 variants with external forces,
grbda_cuda_contact_kinematics_vjp_f64, grbda_cuda_integrate_vjp_f64, grbda_cuda_step_vjp_f64): the gradient of a
scalar costs a small multiple of one evaluation, without building the nv x nv or contact Jacobians. FP64 only, first derivatives only (a backward with create_graph=True
raises). The gradient of q is taken with respect to the stored position entries; for the forward dynamics its
component off the unit quaternion / the loop-constraint manifold is defined in include/grbda_cuda.h.
"""
import functools

import torch
from torch.autograd.function import once_differentiable


def _first_order(backward):
    """once_differentiable, and a backward with create_graph=True fails at once instead of when its result is used."""
    inner = once_differentiable(backward)

    @functools.wraps(backward)
    def wrapper(ctx, *grads):
        if torch.is_grad_enabled():
            raise RuntimeError("grbda.autograd: the dynamics are differentiable once; backward with create_graph=True "
                               "(second derivatives) is not supported")
        return inner(ctx, *grads)
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


# ---- with external forces: the inputs are (model, q, yd, ydd / tau, f_ext) ----------------------------------------
def _backward_ext(ctx, grad, vjp):
    need = ctx.needs_input_grad[1:]
    if not any(need):
        return (None,) * 5
    q, yd, aux, f_ext = ctx.saved_tensors
    bars = vjp(q, yd, aux, grad.contiguous(), f_ext=f_ext)
    return (None,) + tuple(b if n else None for b, n in zip(bars, need))


class _InverseDynamicsExt(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, q, yd, ydd, f_ext):
        _check_inputs(q, yd, ydd, f_ext)
        ctx.model = model
        ctx.save_for_backward(q, yd, ydd, f_ext)
        return model.inverseDynamics(q, yd, ydd, f_ext=f_ext)

    @staticmethod
    @_first_order
    def backward(ctx, grad_tau):
        return _backward_ext(ctx, grad_tau, ctx.model.inverseDynamicsVJP)


class _ForwardDynamicsExt(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, q, yd, tau, f_ext):
        _check_inputs(q, yd, tau, f_ext)
        ctx.model = model
        ctx.save_for_backward(q, yd, tau, f_ext)
        return model.forwardDynamics(q, yd, tau, f_ext=f_ext)

    @staticmethod
    @_first_order
    def backward(ctx, grad_ydd):
        return _backward_ext(ctx, grad_ydd, ctx.model.forwardDynamicsVJP)


# ---- contact kinematics: the inputs are (model, q, yd), the outputs (p, v) ------------------------------------------
def _backward_contacts(ctx, grad_p, grad_v, vjp):
    # an output without a gradient arrives as zeros (autograd materialises it, ctx.set_materialize_grads)
    need = ctx.needs_input_grad[1:]
    if not any(need):
        return None, None, None
    q, yd = ctx.saved_tensors
    bars = vjp(q, yd, grad_p.contiguous(), grad_v.contiguous())
    return (None,) + tuple(b if n else None for b, n in zip(bars, need))


class _ContactKinematics(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, q, yd):
        _check_inputs(q, yd)
        ctx.model = model
        ctx.save_for_backward(q, yd)
        return model.contactKinematics(q, yd)

    @staticmethod
    @_first_order
    def backward(ctx, grad_p, grad_v):
        return _backward_contacts(ctx, grad_p, grad_v, ctx.model.contactKinematicsVJP)


# ---- integration / simulation step: the inputs are (model, dt, q, yd, ydd / tau[, f_ext]), the outputs (q', yd', flags)
class _Integrate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, dt, q, yd, ydd):
        _check_inputs(q, yd, ydd)
        ctx.model, ctx.dt = model, dt
        ctx.save_for_backward(q, yd, ydd)
        if q.shape[0] == 0:  # nothing to integrate (grbda_cuda_integrate_f64 refuses the NULL data of empty tensors)
            q_out, yd_out = torch.empty_like(q), torch.empty_like(yd)
            flags = torch.empty((0,), dtype=torch.int32, device=q.device)
        else:
            q_out, yd_out, flags = model.integrate(q, yd, ydd, dt)
        ctx.mark_non_differentiable(flags)
        return q_out, yd_out, flags

    @staticmethod
    @_first_order
    def backward(ctx, grad_q, grad_yd, _):
        need = ctx.needs_input_grad[2:]
        if not any(need):
            return (None,) * 5
        q, yd, ydd = ctx.saved_tensors
        bars = ctx.model.integrateVJP(q, yd, ydd, ctx.dt, grad_q.contiguous(), grad_yd.contiguous())[:3]
        return (None, None) + tuple(b if n else None for b, n in zip(bars, need))


class _Step(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, dt, q, yd, tau, f_ext):
        _check_inputs(q, yd, tau, *(() if f_ext is None else (f_ext,)))
        ctx.model, ctx.dt = model, dt
        ctx.save_for_backward(q, yd, tau, f_ext)
        q_out, yd_out, flags = model.step(q, yd, tau, dt, f_ext=f_ext)
        ctx.mark_non_differentiable(flags)
        return q_out, yd_out, flags

    @staticmethod
    @_first_order
    def backward(ctx, grad_q, grad_yd, _):
        need = ctx.needs_input_grad[2:]
        if not any(need):
            return (None,) * 6
        q, yd, tau, f_ext = ctx.saved_tensors
        bars = ctx.model.stepVJP(q, yd, tau, ctx.dt, grad_q.contiguous(), grad_yd.contiguous(), f_ext=f_ext)[:-1]
        return (None, None) + tuple(b if n else None for b, n in zip(bars, need)) + (None,) * (4 - len(bars))


def inverse_dynamics(model, q, yd, ydd, f_ext=None):
    """tau[batch, nv] = ID(q, yd, ydd) with a grad_fn: q [batch, nq], yd / ydd [batch, nv], contiguous FP64 CUDA tensors.
    f_ext: world-frame spatial forces on model.externalForceBodies(), [batch, nf, 6] or [batch, 6 nf] (tau = ID - J^T f,
    as model.inverseDynamics takes them); its gradient has its shape."""
    if f_ext is None:
        return _InverseDynamics.apply(model, q, yd, ydd)
    return _InverseDynamicsExt.apply(model, q, yd, ydd, f_ext)


def forward_dynamics(model, q, yd, tau, f_ext=None):
    """ydd[batch, nv] = FD(q, yd, tau) with a grad_fn: q [batch, nq], yd / tau [batch, nv], contiguous FP64 CUDA tensors.
    f_ext as in inverse_dynamics (ydd = FD(q, yd, tau + J^T f))."""
    if f_ext is None:
        return _ForwardDynamics.apply(model, q, yd, tau)
    return _ForwardDynamicsExt.apply(model, q, yd, tau, f_ext)


def contact_kinematics(model, q, yd):
    """(p, v), each [batch, n_cp, 3]: world position / linear velocity of the model's contact points with a grad_fn;
    q [batch, nq], yd [batch, nv], contiguous FP64 CUDA tensors."""
    return _ContactKinematics.apply(model, q, yd)


def integrate(model, q, yd, ydd, dt):
    """(q', yd', flags) = model.integrate(q, yd, ydd, dt) with a grad_fn (flags has none): q [batch, nq], yd / ydd
    [batch, nv], contiguous FP64 CUDA tensors. The gradient of q is the exact derivative of the step for every stored
    position entry; gradients of flagged states are meaningless (include/grbda_cuda.h)."""
    return _Integrate.apply(model, dt, q, yd, ydd)


def step(model, q, yd, tau, dt, f_ext=None):
    """(q', yd', flags) = model.step(q, yd, tau, dt, f_ext) with a grad_fn: one differentiable simulation step, for
    rollouts. f_ext as in forward_dynamics; the gradient of q keeps the convention of forward_dynamics."""
    return _Step.apply(model, dt, q, yd, tau, f_ext)
