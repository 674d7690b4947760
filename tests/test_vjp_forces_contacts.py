"""Reverse mode with external forces and of the contact-point kinematics: the vector-Jacobian product programs of
tau_in +/- J^T f (ALGO_GFA_VJP / ALGO_GFS_VJP) and of contactKinematics (ALGO_CONTACT_KIN_VJP), the C entry points
that compose them with the dynamics VJPs, and the torch.autograd functions built on them.

  * CPU: the emitted programs, replayed in numpy, against the oracle (f_bar exactly, by linearity in f; yd_bar =
    J_lin^T v_bar; the tangent part of the contact q_bar) and against a complex-step replay of the primal programs on
    every stored position entry (q_bar, also off the unit quaternion / off phi = 0); operation counts; sm_100a cubins.
  * GPU: the C ABI against the replayed programs composed as the entry points compose them, gradcheck, the autograd
    plumbing, contact-set and force-set changes, argument checks.
"""
import ctypes as C
import types

import numpy as np
import pytest

from tape import load_tape, run_tape
from test_compiler_cpu import contact_set
from test_vjp import rel, replay, run_tape_complex, tangent_map

TOL = 1e-10      # programs linear in the cotangent: relative to the largest entry of each row
TOL_FD = 1e-9    # through H^-1
# (robot, forces on every body instead of the terminal links)
GF_CASES = [("tello_with_arms", False), ("mini_cheetah", False), ("revolute_chain_with_rotor_4", False),
            ("four_bar", False), ("mit_humanoid", True)]
CONTACT_ROBOTS = ["tello_with_arms", "mini_cheetah", "revolute_pair_chain_with_rotor_4"]


def oracle_model(oracle, m, robot):
    from mirror import mirror_to_oracle
    return mirror_to_oracle(m, oracle) if robot == "four_bar" else oracle.OracleModel(robot)


def force_model(grbda, oracle, robot, all_bodies):
    m = grbda.ClusterTreeModel.from_robot(robot, device=None)
    if all_bodies:
        m.setExternalForceBodies(list(range(m.nb)))
    return m, oracle_model(oracle, m, robot)


def f_bar_oracle(o, bodies, q, yd, aux, w, forward):
    """f_bar[b, k] = w . (ext(f = e_k) - ext(f = 0)): the oracle's dynamics with external forces are affine in f."""
    B, nf = q.shape[0], len(bodies)
    f = np.zeros((B, o.nb, 6))
    base = o.dynamics_with_external_forces(q, yd, aux, f, forward=forward)
    out = np.zeros((B, 6 * nf))
    for k in range(6 * nf):
        f[:] = 0.0
        f[:, bodies[k // 6], k % 6] = 1.0
        d = o.dynamics_with_external_forces(q, yd, aux, f, forward=forward) - base
        out[:, k] = np.einsum("bi,bi->b", w, d)
    return out


def complex_step_q_bar(t, q, others, w):
    """sum_i w_i d out_i / d q_k for every stored entry k of the program on tape t (outputs concatenated)."""
    B, nq = q.shape
    h = 1e-30
    Q = np.repeat(q[:, None, :], nq, axis=1).astype(complex)
    Q[:, np.arange(nq), np.arange(nq)] += 1j * h
    outs = run_tape_complex(t, [Q.reshape(B * nq, nq)] + [np.repeat(x, nq, axis=0) for x in others])
    d = np.concatenate(outs, axis=1).imag.reshape(B, nq, -1) / h  # [b, k, i] = d out_i / d q_k
    return np.einsum("bi,bki->bk", w, d)


def states_on_and_off(o, count, seed):
    """Oracle states, and the same states with positions pushed off the unit quaternion / off phi = 0."""
    q, yd, aux = o.generate_states(count, seed=seed)
    rng = np.random.default_rng(seed)
    q = np.concatenate([q, q + rng.uniform(-0.05, 0.05, q.shape)])
    return q, np.concatenate([yd, yd]), np.concatenate([aux, aux])


def dump(m, algo, path):
    m.dump_program(algo, str(path))
    return load_tape(str(path))


# ---- CPU: external-force programs ------------------------------------------------------------------------------
@pytest.mark.parametrize("robot,all_bodies", GF_CASES)
def test_gf_vjp_programs_match_oracle(grbda, oracle, robot, all_bodies, tmp_path):
    """gfs tape with cotangent w: f_bar = -J w against ID_ext; gfa tape with mu = H^-1 w: f_bar = J mu against FD_ext
    with w (FD_ext is affine in f); q_bar against a complex-step replay of the gfa / gfs programs on every stored
    position entry, on and off the manifold; at most 5x the primal program."""
    m, o = force_model(grbda, oracle, robot, all_bodies)
    bodies = m.externalForceBodies()
    assert bodies and (not all_bodies or bodies == list(range(m.nb)))
    q, yd, aux = states_on_and_off(o, 4, seed=23)
    B, nf6 = q.shape[0], 6 * len(bodies)
    rng = np.random.default_rng(3)
    w = rng.uniform(-1.0, 1.0, (B, o.nv))
    f = rng.uniform(-20.0, 20.0, (B, nf6))
    H = o.mass_matrix(q[:B // 2])
    mu = np.concatenate([np.linalg.solve(H, w[:B // 2, :, None])[:, :, 0], w[B // 2:]])
    for algo, primal, cot, forward in ((grbda.ALGO_GFS_VJP, grbda.ALGO_GFS, w, False),
                                       (grbda.ALGO_GFA_VJP, grbda.ALGO_GFA, mu, True)):
        t = dump(m, algo, tmp_path / ("v%d.tape" % algo))
        assert list(t["n_in"]) == [o.nq, nf6, o.nv]
        q_bar, f_bar = run_tape(t, [q, f, cot])
        assert q_bar.shape == q.shape and f_bar.shape == f.shape
        # f_bar on the manifold states (the oracle's own states), where the oracle's dynamics are defined
        n = B // 2
        want = f_bar_oracle(o, bodies, q[:n], yd[:n], aux[:n], w[:n], forward)
        assert rel(f_bar[:n], want) < (TOL_FD if forward else TOL)
        tp = dump(m, primal, tmp_path / ("p%d.tape" % primal))
        assert rel(q_bar, complex_step_q_bar(tp, q, [f, aux], cot)) < TOL
        flops = m.dump_program(algo)["flops"]
        assert flops <= 5 * m.dump_program(primal)["flops"]


# ---- CPU: contact kinematics -------------------------------------------------------------------------------------
@pytest.mark.parametrize("robot", CONTACT_ROBOTS)
def test_contact_vjp_program_matches_oracle(grbda, oracle, robot, tmp_path):
    """yd_bar = v_bar^T J_lin; with v_bar = 0, q_bar T = p_bar^T J_lin; the full q_bar against a complex-step replay of
    the contact-kinematics program on every stored entry; at most 5x the contact-kinematics program. (The contact
    Jacobian program is about as cheap as the kinematics - rotated motion subspaces, no sweep - so the reverse sweep
    has more operations than it; what it saves is the 6 nv n_cp outputs per state and their contraction.)"""
    m = grbda.ClusterTreeModel.from_robot(robot, device=None)
    o = oracle.OracleModel(robot)
    bodies, offsets, ee = contact_set(m)
    m.setContactPoints(bodies, offsets, ee)
    o.set_contact_points(bodies, offsets, ee)
    q, yd, _ = states_on_and_off(o, 4, seed=29)
    B, ncp = q.shape[0], m.ncp
    rng = np.random.default_rng(4)
    p_bar, v_bar = rng.uniform(-1.0, 1.0, (B, ncp, 3)), rng.uniform(-1.0, 1.0, (B, ncp, 3))
    t = dump(m, grbda.ALGO_CONTACT_KIN_VJP, tmp_path / "ckv.tape")
    assert list(t["n_in"]) == [o.nq, o.nv, 6 * ncp]
    packed = np.concatenate([p_bar.reshape(B, -1), v_bar.reshape(B, -1)], axis=1)
    q_bar, yd_bar = run_tape(t, [q, yd, packed])
    assert q_bar.shape == q.shape and yd_bar.shape == yd.shape
    n = B // 2  # the oracle's Jacobians on its own (manifold) states
    J_lin = o.contact_jacobians(q[:n], world=True)[:, :, 3:, :]
    assert rel(yd_bar[:n], np.einsum("bci,bcik->bk", v_bar[:n], J_lin)) < TOL
    q_bar_p, _ = run_tape(t, [q[:n], yd[:n], np.concatenate([p_bar[:n].reshape(n, -1), np.zeros((n, 3 * ncp))], 1)])
    T = tangent_map(o, q[:n])
    assert rel(np.einsum("bk,bkj->bj", q_bar_p, T), np.einsum("bci,bcik->bk", p_bar[:n], J_lin)) < TOL
    tp = dump(m, grbda.ALGO_CONTACT_KIN, tmp_path / "ck.tape")
    assert rel(q_bar, complex_step_q_bar(tp, q, [yd], packed)) < TOL
    assert m.dump_program(grbda.ALGO_CONTACT_KIN_VJP)["flops"] <= 5 * m.dump_program(grbda.ALGO_CONTACT_KIN)["flops"]


def test_new_vjp_programs_compile_for_sm100a_without_a_device(grbda, tmp_path):
    m = grbda.ClusterTreeModel.from_robot("revolute_pair_chain_with_rotor_4", device=None)
    bodies, offsets, ee = contact_set(m)
    m.setContactPoints(bodies, offsets, ee)
    nf6 = 6 * len(m.externalForceBodies())
    for algo, n_in2 in ((grbda.ALGO_GFA_VJP, m.nv), (grbda.ALGO_GFS_VJP, m.nv), (grbda.ALGO_CONTACT_KIN_VJP, 6 * m.ncp)):
        src, cubin = str(tmp_path / ("v%d.cu" % algo)), str(tmp_path / ("v%d.cubin" % algo))
        m.jit_compile(algo, False, src, cubin)
        blob = open(cubin, "rb").read()
        assert blob[:4] == b"\x7fELF" and len(blob) > 10000
        text = open(src).read()
        assert "N_IN2 = %d" % n_in2 in text
        if algo != grbda.ALGO_CONTACT_KIN_VJP:
            assert "N_IN1 = %d" % nf6 in text and "N_OUT1 = %d" % nf6 in text


def test_new_vjps_refuse_host_only_handles_and_missing_contact_points(grbda):
    L = grbda.lib()
    m = grbda.ClusterTreeModel.from_robot("revolute_chain_with_rotor_4", device=None)
    for fn in (L.grbda_cuda_inverse_dynamics_ext_vjp_f64, L.grbda_cuda_forward_dynamics_ext_vjp_f64):
        assert fn(m._h, *([None] * 9), 1, None) == 4  # GRBDA_ERR_NO_DEVICE
        assert fn(None, *([None] * 9), 1, None) == 1  # GRBDA_ERR_INVALID_ARGUMENT
    ck, ckv = L.grbda_cuda_contact_kinematics_f64, L.grbda_cuda_contact_kinematics_vjp_f64
    # no contact points: the error of contact_kinematics
    assert ckv(m._h, *([None] * 6), 1, None) == ck(m._h, *([None] * 4), 1, None) == 1
    assert "no contact points" in L.grbda_cuda_last_error_string().decode()
    bodies, offsets, ee = contact_set(m)
    m.setContactPoints(bodies, offsets, ee)
    assert ckv(m._h, *([None] * 6), 1, None) == 4
    assert ckv(None, *([None] * 6), 1, None) == 1


# ---- GPU ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def _np(t):
    return t.detach().cpu().numpy()


def _rand(torch, shape, like, lo=-1.0, hi=1.0, seed=0):
    g = torch.Generator(device=like.device).manual_seed(seed)
    return torch.rand(shape, dtype=torch.float64, device=like.device, generator=g) * (hi - lo) + lo


def _contact_model(grbda, robot):
    m = grbda.ClusterTreeModel.from_robot(robot, device=0)
    bodies, offsets, ee = contact_set(m)
    m.setContactPoints(bodies, offsets, ee)
    return m, (bodies, offsets, ee)


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["revolute_chain_with_rotor_4", "mini_cheetah", "tello_with_arms"])
def test_ext_vjp_on_gpu(grbda, oracle, torch, robot, tmp_path):
    """The C entry points with forces against the replayed tapes composed as they compose them, and against the
    oracle (f_bar by linearity, yd_bar through the Jacobians, tau_bar = H^-1 w)."""
    m = grbda.ClusterTreeModel.from_robot(robot, device=0)
    o = oracle.OracleModel(robot)
    bodies = m.externalForceBodies()
    B = 300  # ragged: two full tiles and a tail
    q, yd, aux, flags = m.generateStates(B)
    assert int(flags.sum()) == 0
    w = _rand(torch, (B, m.nv), q, seed=1)
    f = _rand(torch, (B, len(bodies), 6), q, -20.0, 20.0, seed=2)
    qn, ydn, auxn, wn, fn = (_np(t) for t in (q, yd, aux, w, f))
    ff = fn.reshape(B, -1)
    n = 32  # oracle checks on the first states
    # inverse dynamics: ID VJP + GFS VJP
    got = m.inverseDynamicsVJP(q, yd, aux, w, f_ext=f)
    assert len(got) == 4 and got[3].shape == f.shape
    idv, _ = replay(m, grbda.ALGO_ID_VJP, qn, ydn, auxn, wn, tmp_path / "id.tape")
    gq, gf = run_tape(dump(m, grbda.ALGO_GFS_VJP, tmp_path / "gfs.tape"), [qn, ff, wn])
    for g, r in zip(got, (idv[0] + gq, idv[1], idv[2], gf.reshape(fn.shape))):
        assert rel(_np(g), r) < TOL
    assert rel(_np(got[3]).reshape(B, -1)[:n], f_bar_oracle(o, bodies, qn[:n], ydn[:n], auxn[:n], wn[:n], False)) < TOL
    # forward dynamics: GFA, FD VJP at tau' = tau + J^T f, GFA VJP with tau_bar
    got = m.forwardDynamicsVJP(q, yd, aux, w, f_ext=f)
    tau_eff = run_tape(dump(m, grbda.ALGO_GFA, tmp_path / "gfa.tape"), [qn, ff, auxn])[0]
    fdv, _ = replay(m, grbda.ALGO_FD_VJP, qn, ydn, tau_eff, wn, tmp_path / "fd.tape")
    gq, gf = run_tape(dump(m, grbda.ALGO_GFA_VJP, tmp_path / "gfav.tape"), [qn, ff, fdv[2]])
    for g, r in zip(got, (fdv[0] + gq, fdv[1], fdv[2], gf.reshape(fn.shape))):
        assert rel(_np(g), r) < TOL_FD
    H = o.mass_matrix(qn[:n])
    assert rel(_np(got[2])[:n], np.linalg.solve(H, wn[:n, :, None])[:, :, 0]) < TOL_FD
    assert rel(_np(got[3]).reshape(B, -1)[:n], f_bar_oracle(o, bodies, qn[:n], ydn[:n], auxn[:n], wn[:n], True)) < TOL_FD
    d = o.dynamics_derivatives(qn[:n], ydn[:n], tau_eff[:n], True)
    assert rel(_np(got[1])[:n], np.einsum("bi,bij->bj", wn[:n], d[1])) < TOL_FD


@pytest.mark.gpu
def test_fd_ext_vjp_is_fd_vjp_at_the_effective_torque_plus_the_force_part(grbda, torch, tmp_path):
    """q_bar, yd_bar, tau_bar of the FD-with-forces VJP = forwardDynamicsVJP at tau' = GFA(q, f, tau), plus the
    external-force part of q_bar (the GFA VJP with tau_bar)."""
    m = grbda.ClusterTreeModel.from_robot("tello_with_arms", device=0)
    B = 1000
    q, yd, tau, _ = m.generateStates(B, seed=5)
    w = _rand(torch, (B, m.nv), q, seed=6)
    f = _rand(torch, (B, len(m.externalForceBodies()), 6), q, -20.0, 20.0, seed=7)
    qn, fn = _np(q), _np(f).reshape(B, -1)
    tau_eff = torch.from_numpy(run_tape(dump(m, grbda.ALGO_GFA, tmp_path / "gfa.tape"), [qn, fn, _np(tau)])[0]).to(q.device)
    # the effective torque the entry point uses is the one forwardDynamics with forces integrates
    assert rel(_np(m.forwardDynamics(q, yd, tau_eff)), _np(m.forwardDynamics(q, yd, tau, f_ext=f))) < TOL_FD
    got = m.forwardDynamicsVJP(q, yd, tau, w, f_ext=f)
    plain = m.forwardDynamicsVJP(q, yd, tau_eff, w)
    gq, gf = run_tape(dump(m, grbda.ALGO_GFA_VJP, tmp_path / "gfav.tape"), [qn, fn, _np(plain[2])])
    assert rel(_np(got[0]), _np(plain[0]) + gq) < TOL_FD
    assert rel(_np(got[1]), _np(plain[1])) < TOL_FD
    assert rel(_np(got[2]), _np(plain[2])) < TOL_FD
    assert rel(_np(got[3]).reshape(B, -1), gf) < TOL_FD


@pytest.mark.gpu
def test_ext_vjp_without_forces_is_the_plain_vjp(grbda, torch):
    """f_ext = NULL: bit for bit the VJP without forces, and f_bar is not written."""
    L = grbda.lib()
    m = grbda.ClusterTreeModel.from_robot("mini_cheetah", device=0)
    B = 300
    q, yd, aux, _ = m.generateStates(B)
    w = _rand(torch, (B, m.nv), q, seed=8)
    nf6 = 6 * len(m.externalForceBodies())
    P = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
    for ext, plain in ((L.grbda_cuda_inverse_dynamics_ext_vjp_f64, m.inverseDynamicsVJP),
                       (L.grbda_cuda_forward_dynamics_ext_vjp_f64, m.forwardDynamicsVJP)):
        outs = [torch.full_like(q, 7.0), torch.full_like(yd, 7.0), torch.full_like(yd, 7.0)]
        f_bar = torch.full((B, nf6), 7.0, dtype=torch.float64, device=q.device)
        assert ext(m._h, P(q), P(yd), P(aux), None, P(w), *[P(t) for t in outs], P(f_bar), B, None) == 0
        assert ext(m._h, P(q), P(yd), P(aux), None, P(w), *[P(t) for t in outs], None, B, None) == 0
        torch.cuda.synchronize()
        for g, r in zip(outs, plain(q, yd, aux, w)):
            assert torch.equal(g, r)
        assert bool((f_bar == 7.0).all())
        assert len(plain(q, yd, aux, w, f_ext=None)) == 3


@pytest.mark.gpu
def test_contact_vjp_on_gpu(grbda, oracle, torch, tmp_path):
    """The C entry point against the replayed tape and the oracle's J_lin^T v_bar on a ragged batch."""
    for robot in CONTACT_ROBOTS:
        m, (bodies, offsets, ee) = _contact_model(grbda, robot)
        o = oracle.OracleModel(robot)
        o.set_contact_points(bodies, offsets, ee)
        B = 300
        q, yd, _, _ = m.generateStates(B)
        p_bar, v_bar = _rand(torch, (B, m.ncp, 3), q, seed=9), _rand(torch, (B, m.ncp, 3), q, seed=10)
        got = m.contactKinematicsVJP(q, yd, p_bar, v_bar)
        qn, ydn = _np(q), _np(yd)
        packed = np.concatenate([_np(p_bar).reshape(B, -1), _np(v_bar).reshape(B, -1)], axis=1)
        want = run_tape(dump(m, grbda.ALGO_CONTACT_KIN_VJP, tmp_path / ("%s.tape" % robot)), [qn, ydn, packed])
        for g, r in zip(got, want):
            assert rel(_np(g), r) < TOL
        J = o.contact_jacobians(qn[:32], world=True)
        assert rel(_np(got[1])[:32], np.einsum("bci,bcik->bk", _np(v_bar)[:32], J[:, :, 3:, :])) < TOL


@pytest.mark.gpu
def test_gradcheck_with_forces_and_contacts(grbda, torch):
    gad = grbda.autograd
    for robot in ("mini_cheetah", "tello_with_arms", "revolute_chain_with_rotor_4"):
        m = grbda.ClusterTreeModel.from_robot(robot, device=0)
        q, yd, aux, _ = m.generateStates(3)
        f = _rand(torch, (3, len(m.externalForceBodies()), 6), q, seed=11)
        for fn in (gad.inverse_dynamics, gad.forward_dynamics):
            if robot == "revolute_chain_with_rotor_4":  # positions are tangent coordinates: every input
                args = tuple(t.clone().requires_grad_(True) for t in (q, yd, aux, f))
                assert torch.autograd.gradcheck(lambda a, b, c, d: fn(m, a, b, c, f_ext=d), args)
            else:
                args = tuple(t.clone().requires_grad_(True) for t in (yd, aux, f))
                assert torch.autograd.gradcheck(lambda b, c, d: fn(m, q, b, c, f_ext=d), args)
    for robot, with_q in (("revolute_pair_chain_with_rotor_4", True), ("mini_cheetah", False)):
        m, _ = _contact_model(grbda, robot)
        q, yd, _, _ = m.generateStates(3)
        if with_q:
            args = (q.clone().requires_grad_(True), yd.clone().requires_grad_(True))
            assert torch.autograd.gradcheck(lambda a, b: gad.contact_kinematics(m, a, b), args)
        else:
            args = (yd.clone().requires_grad_(True),)
            assert torch.autograd.gradcheck(lambda b: gad.contact_kinematics(m, q, b), args)


@pytest.mark.gpu
def test_autograd_plumbing_with_forces(grbda, torch):
    gad = grbda.autograd
    m = grbda.ClusterTreeModel.from_robot("mini_cheetah", device=0)
    q, yd, aux, _ = m.generateStates(64)
    B, nv = q.shape[0], m.nv
    f = _rand(torch, (B, len(m.externalForceBodies()), 6), q, -20.0, 20.0, seed=12)
    for fn, vjp, plain in ((gad.inverse_dynamics, m.inverseDynamicsVJP, m.inverseDynamics),
                           (gad.forward_dynamics, m.forwardDynamicsVJP, m.forwardDynamics)):
        qa, ya, xa, fa = (t.clone().requires_grad_(True) for t in (q, yd, aux, f))
        out = fn(m, qa, ya, xa, f_ext=fa)
        assert torch.equal(out.detach(), plain(q, yd, aux, f_ext=f))
        w = _rand(torch, (B, nv), q, seed=13)
        (out * w).sum().backward()
        want = vjp(q, yd, aux, w, f_ext=f)
        for g, r in zip((qa.grad, ya.grad, xa.grad, fa.grad), want):
            assert torch.equal(g, r)  # loss.backward() is one call of the entry point
        # partial requires_grad: only the forces
        fa = f.clone().requires_grad_(True)
        fn(m, q, yd, aux, f_ext=fa).backward(w)
        assert torch.equal(fa.grad, want[3])
        # the backward returns None for inputs that need no gradient and launches nothing when none needs one
        ctx = types.SimpleNamespace(needs_input_grad=(False, False, True, False, False), saved_tensors=(q, yd, aux, f))
        grads = gad._backward_ext(ctx, w, vjp)
        assert len(grads) == 5 and all(grads[k] is None for k in (0, 1, 3, 4)) and torch.equal(grads[2], want[1])
        ctx.needs_input_grad = (False,) * 5
        launches = grbda.launch_count()
        assert gad._backward_ext(ctx, w, vjp) == (None,) * 5 and grbda.launch_count() == launches
        # flat forces [B, 6 nf]: the gradient has their shape
        ff = f.reshape(B, -1).clone().requires_grad_(True)
        fn(m, q, yd, aux, f_ext=ff).backward(w)
        assert ff.grad.shape == ff.shape and torch.equal(ff.grad, want[3].reshape(B, -1))
        # second derivatives are refused
        fa = f.clone().requires_grad_(True)
        with pytest.raises(RuntimeError, match="create_graph"):
            torch.autograd.grad(fn(m, q, yd, aux, f_ext=fa).sum(), fa, create_graph=True)
        # no states
        e = [t[:0].clone().requires_grad_(True) for t in (q, yd, aux, f)]
        fn(m, *e[:3], f_ext=e[3]).sum().backward()
        assert all(t.grad is not None and t.grad.shape == t.shape for t in e)
    # without forces: the classes and the backward of the plain dynamics
    assert type(gad.inverse_dynamics(m, q, yd, aux.clone().requires_grad_(True)).grad_fn).__name__.startswith(
        "_InverseDynamicsBackward")
    with pytest.raises(TypeError):
        gad.forward_dynamics(m, q, yd, aux, f_ext=f.float())


@pytest.mark.gpu
def test_autograd_plumbing_contacts(grbda, torch):
    gad = grbda.autograd
    m, _ = _contact_model(grbda, "tello_with_arms")
    q, yd, _, _ = m.generateStates(64)
    B = q.shape[0]
    qa, ya = q.clone().requires_grad_(True), yd.clone().requires_grad_(True)
    p, v = gad.contact_kinematics(m, qa, ya)
    pp, vv = m.contactKinematics(q, yd)
    assert torch.equal(p.detach(), pp) and torch.equal(v.detach(), vv)
    wp, wv = _rand(torch, p.shape, q, seed=14), _rand(torch, v.shape, q, seed=15)
    ((p * wp).sum() + (v * wv).sum()).backward()
    want = m.contactKinematicsVJP(q, yd, wp, wv)
    assert torch.equal(qa.grad, want[0]) and torch.equal(ya.grad, want[1])
    # one output without a gradient: zeros in its place
    qa = q.clone().requires_grad_(True)
    _, v = gad.contact_kinematics(m, qa, yd)
    (v * wv).sum().backward()
    assert torch.equal(qa.grad, m.contactKinematicsVJP(q, yd, torch.zeros_like(wv), wv)[0])
    # partial requires_grad returns None for the other input; nothing to differentiate: no launch
    ctx = types.SimpleNamespace(needs_input_grad=(False, False, True), saved_tensors=(q, yd))
    grads = gad._backward_contacts(ctx, wp, wv, m.contactKinematicsVJP)
    assert grads[0] is None and grads[1] is None and torch.equal(grads[2], want[1])
    ctx.needs_input_grad = (False,) * 3
    launches = grbda.launch_count()
    assert gad._backward_contacts(ctx, wp, wv, m.contactKinematicsVJP) == (None,) * 3
    assert grbda.launch_count() == launches
    with pytest.raises(RuntimeError, match="create_graph"):
        ya = yd.clone().requires_grad_(True)
        torch.autograd.grad(gad.contact_kinematics(m, q, ya)[1].sum(), ya, create_graph=True)
    e = [t[:0].clone().requires_grad_(True) for t in (q, yd)]
    p, v = gad.contact_kinematics(m, *e)
    (p.sum() + v.sum()).backward()
    assert all(t.grad is not None and t.grad.shape == t.shape for t in e)
    assert B == 64


@pytest.mark.gpu
def test_contact_vjp_follows_a_changed_contact_set(grbda, torch, tmp_path):
    """setContactPoints to another set drops the compiled contact VJP: the next call matches a replay for the new set."""
    m, (bodies, offsets, ee) = _contact_model(grbda, "mini_cheetah")
    B = 300
    q, yd, _, _ = m.generateStates(B)
    m.contactKinematicsVJP(q, yd, torch.ones(B, m.ncp, 3, dtype=torch.float64, device=q.device),
                           torch.ones(B, m.ncp, 3, dtype=torch.float64, device=q.device))
    new_bodies = list(bodies[:2])
    new_offsets = np.asarray(offsets[:2]) + 0.1
    m.setContactPoints(new_bodies, new_offsets, [1, 0])
    assert m.ncp == 2
    p_bar, v_bar = _rand(torch, (B, 2, 3), q, seed=16), _rand(torch, (B, 2, 3), q, seed=17)
    got = m.contactKinematicsVJP(q, yd, p_bar, v_bar)
    packed = np.concatenate([_np(p_bar).reshape(B, -1), _np(v_bar).reshape(B, -1)], axis=1)
    want = run_tape(dump(m, grbda.ALGO_CONTACT_KIN_VJP, tmp_path / "new.tape"), [_np(q), _np(yd), packed])
    for g, r in zip(got, want):
        assert rel(_np(g), r) < TOL


@pytest.mark.gpu
def test_ext_vjp_follows_a_changed_force_set(grbda, oracle, torch, tmp_path):
    """setExternalForceBodies(subset): f_bar takes the subset's shape and its values."""
    m = grbda.ClusterTreeModel.from_robot("tello_with_arms", device=0)
    o = oracle.OracleModel("tello_with_arms")
    B = 300
    q, yd, aux, _ = m.generateStates(B)
    w = _rand(torch, (B, m.nv), q, seed=18)
    f = _rand(torch, (B, len(m.externalForceBodies()), 6), q, seed=19)
    m.inverseDynamicsVJP(q, yd, aux, w, f_ext=f)  # the default set's programs are loaded
    subset = [m.nb - 1, 0, 5]
    m.setExternalForceBodies(subset)
    try:
        fs = _rand(torch, (B, 3, 6), q, seed=20)
        qn, ydn, auxn, wn = (_np(t) for t in (q, yd, aux, w))
        for vjp, forward in ((m.inverseDynamicsVJP, False), (m.forwardDynamicsVJP, True)):
            got = vjp(q, yd, aux, w, f_ext=fs)
            assert got[3].shape == (B, 3, 6)
            want = f_bar_oracle(o, subset, qn[:32], ydn[:32], auxn[:32], wn[:32], forward)
            assert rel(_np(got[3]).reshape(B, -1)[:32], want) < (TOL_FD if forward else TOL)
        algo = grbda.ALGO_GFS_VJP
        gq, gf = run_tape(dump(m, algo, tmp_path / "gfs.tape"), [qn, _np(fs).reshape(B, -1), wn])
        got = m.inverseDynamicsVJP(q, yd, aux, w, f_ext=fs)
        idv, _ = replay(m, grbda.ALGO_ID_VJP, qn, ydn, auxn, wn, tmp_path / "id.tape")
        assert rel(_np(got[0]), idv[0] + gq) < TOL and rel(_np(got[3]).reshape(B, -1), gf) < TOL
    finally:
        m.setExternalForceBodies([])


@pytest.mark.gpu
def test_new_vjp_c_abi_arguments(grbda, torch):
    L = grbda.lib()
    m, _ = _contact_model(grbda, "mini_cheetah")
    B = 8
    q, yd, aux, _ = m.generateStates(B)
    f = torch.zeros(B, 6 * len(m.externalForceBodies()), dtype=torch.float64, device=q.device)
    P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    for fn in (L.grbda_cuda_inverse_dynamics_ext_vjp_f64, L.grbda_cuda_forward_dynamics_ext_vjp_f64):
        ins = [P(t) for t in (q, yd, aux, f, aux)]
        outs = [P(t) for t in (torch.empty_like(q), torch.empty_like(yd), torch.empty_like(yd), torch.empty_like(f))]
        assert fn(m._h, *ins, *outs, 0, None) == 0  # batch 0: nothing to do
        assert fn(m._h, *ins, *outs, -1, None) == 1
        for k in (0, 1, 2, 4):  # null inputs (f_ext = NULL means no forces)
            args = list(ins)
            args[k] = None
            assert fn(m._h, *args, *outs, B, None) == 1
        for k in range(4):  # null outputs
            args = list(outs)
            args[k] = None
            assert fn(m._h, *ins, *args, B, None) == 1
        assert fn(m._h, *ins, *outs, B, None) == 0
    fn = L.grbda_cuda_contact_kinematics_vjp_f64
    bars = torch.zeros(B, 3 * m.ncp, dtype=torch.float64, device=q.device)
    ins = [P(t) for t in (q, yd, bars, bars)]
    outs = [P(t) for t in (torch.empty_like(q), torch.empty_like(yd))]
    assert fn(m._h, *ins, *outs, 0, None) == 0
    assert fn(m._h, *ins, *outs, -1, None) == 1
    for k in range(4):
        args = list(ins)
        args[k] = None
        assert fn(m._h, *args, *outs, B, None) == 1
    for k in range(2):
        args = list(outs)
        args[k] = None
        assert fn(m._h, *ins, *args, B, None) == 1
    assert fn(m._h, *ins, *outs, B, None) == 0
    torch.cuda.synchronize()
