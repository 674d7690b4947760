"""Reverse mode: vector-Jacobian products of the inverse and forward dynamics and the torch.autograd functions
built on them.

  * CPU: the emitted VJP programs, replayed in numpy, against the oracle's Jacobians contracted with a random
    cotangent; the inverse-dynamics q_bar also against a complex-step replay of the inverse-dynamics program on every
    stored position entry (the exact derivative, also off the unit quaternion / the loop-constraint manifold);
    operation counts against the primal programs and the Jacobian programs.
  * GPU: the C ABI against the replayed programs and the Jacobian entry points, gradcheck and the autograd plumbing.
"""
import ctypes as C
import types

import numpy as np
import pytest

from tape import load_tape, run_tape

ROBOTS = ["revolute_chain_with_rotor_4", "revolute_pair_chain_with_rotor_4", "mini_cheetah", "mit_humanoid",
          "tello_with_arms"]
GPU_ROBOTS = ["revolute_chain_with_rotor_4", "mini_cheetah", "mit_humanoid", "tello_with_arms"]
TOL_ID, TOL_FD = 1e-10, 1e-9  # relative to the largest entry of each row


def rel(a, b):
    a, b = a.reshape(b.shape[0], -1), b.reshape(b.shape[0], -1)
    return float((np.abs(a - b).max(1) / np.maximum(1e-300, np.abs(b).max(1))).max())


def quat_to_R(q):  # ori::quaternionToRotationMatrix, q = (w, x, y, z)
    e0, e1, e2, e3 = q
    R = np.array([[1 - 2 * (e2 * e2 + e3 * e3), 2 * (e1 * e2 - e0 * e3), 2 * (e1 * e3 + e0 * e2)],
                  [2 * (e1 * e2 + e0 * e3), 1 - 2 * (e1 * e1 + e3 * e3), 2 * (e2 * e3 - e0 * e1)],
                  [2 * (e1 * e3 - e0 * e2), 2 * (e2 * e3 + e0 * e1), 1 - 2 * (e1 * e1 + e2 * e2)]])
    return R.T


def quat_product(a, b):  # ori::quatProduct
    r = a[0] * b[0] - a[1:] @ b[1:]
    v = a[0] * b[1:] + b[0] * a[1:] + np.cross(a[1:], b[1:])
    return np.concatenate([[r], v])


def tangent_map(o, q):
    """T[b] (nq x nv): d q / d dq of the tangent-space perturbation the Jacobians are taken along - the linearisation
    of the reference test's `plus` for the floating base and one-dof joints, dq_span = G dy for implicit clusters."""
    B = q.shape[0]
    T = np.zeros((B, o.nq, o.nv))
    for ci, c in enumerate(o.clusters()):
        pi, vi, N, n = c["position_index"], c["velocity_index"], c["num_positions"], c["num_velocities"]
        for b in range(B):
            if c["implicit"]:
                T[b, pi:pi + N, vi:vi + n] = o.cluster_constraint(ci, q[b], np.zeros(o.nv))[0]
            elif N == 7 and n == 6:  # [p; quat] (+) [dw; dp] = [p + R^T dp; quat + 1/2 quat (x) (0, dw)]
                quat = q[b, pi + 3:pi + 7]
                T[b, pi:pi + 3, vi + 3:vi + 6] = quat_to_R(quat).T
                for k in range(3):
                    T[b, pi + 3:pi + 7, vi + k] = 0.5 * quat_product(quat, np.eye(4)[1 + k])
            else:
                T[b, pi + np.arange(n), vi + np.arange(n)] = 1.0
    return T


def run_tape_complex(t, inputs):
    """run_tape in complex arithmetic (complex step); OP_SELECT_GT compares the real parts."""
    B = inputs[0].shape[0]
    v = [None] * len(t["op"])
    unary = {6: np.negative, 7: np.sin, 8: np.cos, 9: np.sqrt}
    binary = {2: np.add, 3: np.subtract, 4: np.multiply, 5: np.divide}
    for i, (op, a, b, c, e) in enumerate(zip(t["op"], t["a"], t["b"], t["c"], t["e"])):
        if op == 0:
            v[i] = np.full(B, t["val"][i], dtype=complex)
        elif op == 1:
            v[i] = inputs[a][:, b].astype(complex)
        elif op in binary:
            v[i] = binary[op](v[a], v[b])
        elif op in unary:
            v[i] = unary[op](v[a])
        elif op == 10:
            v[i] = np.where(v[a].real > v[b].real, v[c], v[e])
        else:
            raise ValueError("unknown op %d" % op)
    return [np.stack([v[j] for j in o], axis=1) for o in t["outs"]]


def replay(m, algo, q, yd, aux, w, path):
    counts = m.dump_program(algo, str(path))
    return run_tape(load_tape(str(path)), [q, yd, np.concatenate([aux, w], axis=1)]), counts


@pytest.mark.parametrize("robot", ROBOTS)
def test_vjp_programs_match_oracle(grbda, oracle, robot, tmp_path):
    """Replayed VJP tapes: yd_bar = w^T dout/dyd, ydd_bar = H w / tau_bar = H^-1 w, q_bar T = w^T dout/ddq; and the
    reverse sweep stays a small multiple of the primal program, below the dense Jacobian programs."""
    m = grbda.ClusterTreeModel.from_robot(robot, device=None)
    o = oracle.OracleModel(robot)
    q, yd, aux = o.generate_states(6, seed=7)
    w = np.random.default_rng(1).uniform(-1.0, 1.0, (q.shape[0], o.nv))
    H = o.mass_matrix(q)
    T = tangent_map(o, q)
    for algo, forward, tol in ((grbda.ALGO_ID_VJP, False, TOL_ID), (grbda.ALGO_FD_VJP, True, TOL_FD)):
        (q_bar, yd_bar, aux_bar), counts = replay(m, algo, q, yd, aux, w, tmp_path / ("v%d.tape" % algo))
        assert q_bar.shape == q.shape and yd_bar.shape == aux_bar.shape == w.shape
        d = o.dynamics_derivatives(q, yd, aux, forward)
        assert rel(yd_bar, np.einsum("bi,bij->bj", w, d[1])) < tol
        assert rel(np.einsum("bk,bkj->bj", q_bar, T), np.einsum("bi,bij->bj", w, d[0])) < tol
        want_aux = np.linalg.solve(H, w[:, :, None])[:, :, 0] if forward else np.einsum("bij,bj->bi", H, w)
        assert rel(aux_bar, want_aux) < tol
        # cost: at most 5x the primal program (FD: the factorisation program the VJP is built on), and below the
        # Jacobian programs wherever those are large
        primal = m.dump_program(grbda.PROGRAM_FD_LTL if forward else grbda.ALGO_ID)["flops"]
        assert counts["flops"] <= 5 * primal
        if o.nv >= 18:
            assert counts["flops"] < m.dump_program(grbda.ALGO_FD_DERIV if forward else grbda.ALGO_ID_DERIV)["flops"]


@pytest.mark.parametrize("robot", ROBOTS)
def test_id_vjp_positions_are_exact_program_derivatives(grbda, oracle, robot, tmp_path):
    """Inverse dynamics q_bar against a complex-step replay of the inverse-dynamics program on every stored position
    entry, at the oracle states and at positions pushed off the unit quaternion / off phi = 0."""
    m = grbda.ClusterTreeModel.from_robot(robot, device=None)
    o = oracle.OracleModel(robot)
    q, yd, aux = o.generate_states(4, seed=9)
    rng = np.random.default_rng(2)
    q = np.concatenate([q, q + rng.uniform(-0.05, 0.05, q.shape)])
    yd, aux = np.concatenate([yd, yd]), np.concatenate([aux, aux])
    B, nq, nv = q.shape[0], o.nq, o.nv
    w = rng.uniform(-1.0, 1.0, (B, nv))
    (q_bar, _, _), _ = replay(m, grbda.ALGO_ID_VJP, q, yd, aux, w, tmp_path / "id_vjp.tape")
    m.dump_program(grbda.ALGO_ID, str(tmp_path / "id.tape"))
    h = 1e-30
    Q = np.repeat(q[:, None, :], nq, axis=1).astype(complex)
    Q[:, np.arange(nq), np.arange(nq)] += 1j * h
    tau = run_tape_complex(load_tape(str(tmp_path / "id.tape")),
                           [Q.reshape(B * nq, nq), np.repeat(yd, nq, axis=0), np.repeat(aux, nq, axis=0)])[0]
    dtau_dq = tau.imag.reshape(B, nq, nv) / h  # [b, k, i] = d tau_i / d q_k
    assert rel(q_bar, np.einsum("bi,bki->bk", w, dtau_dq)) < TOL_ID


def test_vjp_programs_compile_for_sm100a_without_a_device(grbda, tmp_path):
    m = grbda.ClusterTreeModel.from_robot("revolute_chain_with_rotor_4", device=None)
    for algo in (grbda.ALGO_ID_VJP, grbda.ALGO_FD_VJP):
        src, cubin = str(tmp_path / ("v%d.cu" % algo)), str(tmp_path / ("v%d.cubin" % algo))
        m.jit_compile(algo, False, src, cubin)
        blob = open(cubin, "rb").read()
        assert blob[:4] == b"\x7fELF" and len(blob) > 10000
        assert "N_IN2 = %d" % (2 * m.nv) in open(src).read()


def test_vjp_refuses_host_only_handles(grbda):
    m = grbda.ClusterTreeModel.from_robot("revolute_chain_with_rotor_4", device=None)
    for fn in (grbda.lib().grbda_cuda_inverse_dynamics_vjp_f64, grbda.lib().grbda_cuda_forward_dynamics_vjp_f64):
        assert fn(m._h, None, None, None, None, None, None, None, 1, None) == 4  # GRBDA_ERR_NO_DEVICE
        assert fn(None, None, None, None, None, None, None, None, 1, None) == 1  # GRBDA_ERR_INVALID_ARGUMENT


# ---- GPU ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


@pytest.mark.gpu
@pytest.mark.parametrize("robot", GPU_ROBOTS)
def test_vjp_on_gpu(grbda, oracle, torch, robot, tmp_path):
    """C ABI against the replayed programs and the oracle, and against the Jacobian entry points on the same states."""
    m = grbda.ClusterTreeModel.from_robot(robot, device=0)
    o = oracle.OracleModel(robot)
    B = 300  # ragged: two full tiles and a tail
    q, yd, aux, flags = m.generateStates(B)
    assert int(flags.sum()) == 0
    w = torch.rand(B, m.nv, dtype=torch.float64, device=q.device) * 2 - 1
    qn, ydn, auxn, wn = (t.cpu().numpy() for t in (q, yd, aux, w))
    T = tangent_map(o, qn)
    H = m.getMassMatrix(q)
    for algo, tol in ((grbda.ALGO_ID_VJP, TOL_ID), (grbda.ALGO_FD_VJP, TOL_FD)):
        forward = algo == grbda.ALGO_FD_VJP
        got = (m.forwardDynamicsVJP if forward else m.inverseDynamicsVJP)(q, yd, aux, w)
        torch.cuda.synchronize()
        want, _ = replay(m, algo, qn, ydn, auxn, wn, tmp_path / ("v%d.tape" % algo))
        for g, r in zip(got, want):
            assert rel(g.cpu().numpy(), r) < tol
        d = o.dynamics_derivatives(qn, ydn, auxn, forward)
        assert rel(got[1].cpu().numpy(), np.einsum("bi,bij->bj", wn, d[1])) < tol
        assert rel(np.einsum("bk,bkj->bj", got[0].cpu().numpy(), T), np.einsum("bi,bij->bj", wn, d[0])) < tol
        # the Jacobian entry points on the same states
        jac = (m.forwardDynamicsDerivatives if forward else m.inverseDynamicsDerivatives)(q, yd, aux)
        assert _rel_t(got[1], torch.einsum("bi,bij->bj", w, jac[1])) < tol
        Tq = torch.from_numpy(T).to(q.device)
        assert _rel_t(torch.einsum("bk,bkj->bj", got[0], Tq), torch.einsum("bi,bij->bj", w, jac[0])) < tol
        third = torch.einsum("bi,bij->bj", w, jac[2]) if forward else torch.einsum("bij,bj->bi", H, w)
        assert _rel_t(got[2], third) < tol


def _rel_t(a, b):
    return rel(a.detach().cpu().numpy(), b.detach().cpu().numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["revolute_chain_with_rotor_4", "mini_cheetah", "tello_with_arms"])
def test_gradcheck(grbda, torch, robot):
    """All inputs where positions are tangent coordinates; yd and ydd / tau on the floating-base models."""
    gad = grbda.autograd
    m = grbda.ClusterTreeModel.from_robot(robot, device=0)
    q, yd, aux, _ = m.generateStates(4)
    all_inputs = robot == "revolute_chain_with_rotor_4"
    for fn in (gad.inverse_dynamics, gad.forward_dynamics):
        if all_inputs:
            args = tuple(t.clone().requires_grad_(True) for t in (q, yd, aux))
            assert torch.autograd.gradcheck(lambda a, b, c: fn(m, a, b, c), args)
        else:
            args = tuple(t.clone().requires_grad_(True) for t in (yd, aux))
            assert torch.autograd.gradcheck(lambda b, c: fn(m, q, b, c), args)


@pytest.mark.gpu
def test_autograd_plumbing(grbda, torch):
    gad = grbda.autograd
    m = grbda.ClusterTreeModel.from_robot("mini_cheetah", device=0)
    q, yd, aux, _ = m.generateStates(64)
    B, nv = q.shape[0], m.nv
    for fn, vjp, plain in ((gad.inverse_dynamics, m.inverseDynamicsVJP, m.inverseDynamics),
                           (gad.forward_dynamics, m.forwardDynamicsVJP, m.forwardDynamics)):
        qa, ya, xa = (t.clone().requires_grad_(True) for t in (q, yd, aux))
        out = fn(m, qa, ya, xa)
        assert torch.equal(out.detach(), plain(q, yd, aux))
        w = torch.rand(B, nv, dtype=torch.float64, device=q.device)
        (out * w).sum().backward()
        want = vjp(q, yd, aux, w)
        for g, r in zip((qa.grad, ya.grad, xa.grad), want):
            assert torch.equal(g, r)  # loss.backward() is one VJP launch
        # partial requires_grad: the backward returns None for the inputs that need no gradient ...
        ctx = types.SimpleNamespace(needs_input_grad=(False, False, True, False), saved_tensors=(q, yd, aux))
        grads = gad._backward(ctx, w, vjp)
        assert grads[0] is None and grads[1] is None and grads[3] is None and torch.equal(grads[2], want[1])
        # ... and launches nothing when no input needs one
        ctx.needs_input_grad = (False,) * 4
        launches = grbda.launch_count()
        assert gad._backward(ctx, w, vjp) == (None,) * 4 and grbda.launch_count() == launches
        ya = yd.clone().requires_grad_(True)
        fn(m, q, ya, aux).sum().backward()
        assert torch.equal(ya.grad, vjp(q, yd, aux, torch.ones_like(w))[1])
        # a non-contiguous grad_output
        xa = aux.clone().requires_grad_(True)
        out = fn(m, q, yd, xa)
        g2 = torch.rand(nv, B, dtype=torch.float64, device=q.device).t()
        assert not g2.is_contiguous()
        out.backward(g2)
        assert _rel_t(xa.grad, vjp(q, yd, aux, g2.contiguous())[2]) == 0.0
        # second derivatives are refused
        xa = aux.clone().requires_grad_(True)
        with pytest.raises(RuntimeError, match="create_graph"):
            torch.autograd.grad(fn(m, q, yd, xa).sum(), xa, create_graph=True)
        # no states
        e = [t[:0].clone().requires_grad_(True) for t in (q, yd, aux)]
        fn(m, *e).sum().backward()
        assert all(t.grad is not None and t.grad.shape == t.shape for t in e)
    # the plain methods stay without a grad_fn
    assert m.inverseDynamics(q, yd, aux.clone().requires_grad_(True)).grad_fn is None
    with pytest.raises(TypeError):
        gad.inverse_dynamics(m, q.float(), yd.float(), aux.float())


@pytest.mark.gpu
def test_vjp_c_abi_arguments(grbda, torch):
    m = grbda.ClusterTreeModel.from_robot("mini_cheetah", device=0)
    q, yd, aux, _ = m.generateStates(8)
    out = [torch.empty_like(q), torch.empty_like(yd), torch.empty_like(yd)]
    p = [C.c_void_p(t.data_ptr()) for t in (q, yd, aux, aux)]
    o = [C.c_void_p(t.data_ptr()) for t in out]
    for fn in (grbda.lib().grbda_cuda_inverse_dynamics_vjp_f64, grbda.lib().grbda_cuda_forward_dynamics_vjp_f64):
        assert fn(m._h, *p, *o, 0, None) == 0  # batch 0: nothing to do
        assert fn(m._h, *p, *o, -1, None) == 1
        for k in range(4):  # null inputs
            args = list(p)
            args[k] = None
            assert fn(m._h, *args, *o, 8, None) == 1
        for k in range(3):  # null outputs
            args = list(o)
            args[k] = None
            assert fn(m._h, *p, *args, 8, None) == 1
        assert fn(m._h, *p, *o, 8, None) == 0
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_tello_forward_dynamics_gradient_of_tau_is_inverse_mass_matrix(grbda, torch):
    """d (sum ydd) / d tau = H^-1 1."""
    m = grbda.ClusterTreeModel.from_robot("tello_with_arms", device=0)
    q, yd, tau, _ = m.generateStates(256)
    tau = tau.clone().requires_grad_(True)
    grbda.autograd.forward_dynamics(m, q, yd, tau).sum().backward()
    H = m.getMassMatrix(q)
    want = torch.linalg.solve(H, torch.ones(q.shape[0], m.nv, 1, dtype=torch.float64, device=q.device))[:, :, 0]
    assert _rel_t(tau.grad, want) < 1e-9
