"""Models with a roll-pitch-yaw floating base (GRBDA_CLUSTER_FREE_RPY, ClusterJoints::Free with
ori_representation::RollPitchYaw) on every entry point, against the oracle.

The rpy base has its own branch in the model compiler: forward kinematics builds E = Rx(r) Ry(p) Rz(y) from three
sin/cos pairs, the derivative programs use the identity tangent map (nq == nv for that cluster, so `plus` is q + dq),
the state generator stores the raw draws, and the integration step refuses the state. The models are built from a
quaternion model's schedule with cluster_type[0] switched to 1: MiniCheetah and MIT Humanoid (the oracle has the
reference's own builders for them, buildMiniCheetah(false) / buildMitHumanoid(false)) and one floating-base model of
the URDF corpus (the oracle is mirrored from the product's topology). None of them is compiled ahead of time, so every
kernel comes from the run-time compiler.

  * CPU: the emitted programs replayed in numpy against the oracle (dynamics, kinematics, forces, operational space,
    Jacobians, vector-Jacobian products), the Jacobians and the oracle's own derivatives against central differences,
    the emitted CUDA text compiled for the host (including the range check on the rpy angles), sm_100a cubins.
  * GPU: every entry point on a ragged batch against the oracle, FP32 against the FP64 oracle, gradients, gimbal lock,
    angles beyond the fast sin/cos range, NaN angles, and the refusal of the integration step.
"""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from mirror import mirror_to_oracle
from tape import load_tape, run_tape
from test_compiler_cpu import LTL, TOL, contact_set, run_emitted_source
from test_gpu_parity import TOL32, relrows
from test_vjp import rel
from test_vjp_forces_contacts import complex_step_q_bar, f_bar_oracle

HERE = os.path.dirname(os.path.abspath(__file__))
URDF = os.path.join(HERE, "urdf_corpus", "revolute_rotor_branch_2_3.urdf")  # floating base, not ahead of time
# product model (quaternion base) -> oracle model with the rpy base (None: mirrored from the product's topology)
MODELS = {"mini_cheetah": "mini_cheetah_rpy", "mit_humanoid": "mit_humanoid_rpy", "urdf": None}
TOL_FD, TOL_OSIM = 1e-9, 1e-8
FD_H, FD_BOUND = 1e-6, 2e-6  # central differences: step and bound of test_oracle_derivatives_against_finite_differences
N = 3 * 128 + 5              # ragged GPU batch
TURNS = 4.0e11               # whole turns: 2.5e12 rad, beyond the 1e12 of the fast FP64 reduction
ROLL, PITCH, YAW = 3, 4, 5   # position entries of the rpy angles (the base is cluster 0)


def quaternion_model(grbda, name, device=None):
    if name == "urdf":
        return grbda.ClusterTreeModel.from_urdf(URDF, device=device)
    return grbda.ClusterTreeModel.from_robot(name, device=device)


def rpy_model(grbda, name, device=None):
    """The model `name` with its quaternion base switched to roll-pitch-yaw through the schedule."""
    s = quaternion_model(grbda, name, device=None).to_schedule()
    assert s.cluster_type[0] == 0  # GRBDA_CLUSTER_FREE_QUATERNION
    s.cluster_type = s.cluster_type.copy()
    s.cluster_type[0] = 1          # GRBDA_CLUSTER_FREE_RPY
    return grbda.ClusterTreeModel.from_schedule(s, device=device)


def rpy_oracle(oracle, m, name):
    return oracle.OracleModel(MODELS[name]) if MODELS[name] else mirror_to_oracle(m, oracle)


def gimbal_states(o, count, seed):
    """Oracle states, the last four at gimbal lock: pitch = +-pi/2 exactly and +-pi/2 +- 1e-9."""
    q, yd, aux = o.generate_states(count, seed=seed)
    q[-4:, PITCH] = [np.pi / 2, -np.pi / 2, np.pi / 2 + 1e-9, -np.pi / 2 - 1e-9]
    return q, yd, aux


def central_differences(f, q, h=FD_H):
    """d f / d q[k] for every stored position entry (the rpy base has no manifold: `plus` is q + dq).
    f: q -> list of [B, ...] arrays. Returns one [B, n_out, nq] array per output."""
    outs = None
    for k in range(q.shape[1]):
        qp, qm = q.copy(), q.copy()
        qp[:, k] += h
        qm[:, k] -= h
        d = [(a - b).reshape(q.shape[0], -1) / (2 * h) for a, b in zip(f(qp), f(qm))]
        if outs is None:
            outs = [np.zeros(x.shape + (q.shape[1],)) for x in d]
        for o_, x in zip(outs, d):
            o_[:, :, k] = x
    return outs


def dump(m, algo, path):
    m.dump_program(algo, str(path))
    return load_tape(str(path))


def positions_read(m, algo, path):
    """The position entries the program of `algo` reads."""
    t = dump(m, algo, path)
    return {int(b) for op, a, b in zip(t["op"], t["a"], t["b"]) if op == 1 and a == 0}


# ---- CPU: the models -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(MODELS))
def test_rpy_models_match_oracle(grbda, oracle, name):
    """nq drops by one, nv stays; topology, inertias and tree transforms as the oracle's rpy builders give them; the
    kernels are run-time compiled."""
    quat = quaternion_model(grbda, name, device=None)
    m = rpy_model(grbda, name)
    o = rpy_oracle(oracle, m, name)
    assert (m.nq, m.nv, m.nb, m.nc) == (quat.nq - 1, quat.nv, quat.nb, quat.nc)
    assert (m.nq, m.nv, m.nb, m.nc) == (o.nq, o.nv, o.nb, o.nc) and m.nq == m.nv
    assert m.clusters()[0]["type"] == 1 and m.clusters()[0]["num_positions"] == 6
    assert o.clusters()[0]["joint_type"] == "Free" and o.clusters()[0]["num_positions"] == 6
    assert m.hash != quat.hash
    for a, b in zip(m.clusters(), o.clusters()):
        for k in ("parent", "num_bodies", "num_positions", "num_velocities", "position_index", "velocity_index"):
            assert a[k] == b[k], (k, a, b)
        assert (a["type"] == 3) == bool(b["implicit"])
    for a, b in zip(m.bodies(), o.bodies()):
        assert a["parent"] == b["parent"] and a["cluster"] == b["cluster"] and a["sub_index"] == b["sub_index"]
        assert np.abs(a["E"] - b["E"]).max() < 1e-15 and np.abs(a["r"] - b["r"]).max() < 1e-15
        assert np.abs(a["inertia"] - b["inertia"]).max() < 1e-12
    for algo in (grbda.ALGO_ID, grbda.ALGO_FD, grbda.ALGO_FK, grbda.ALGO_H):
        assert m.kernel_info(algo)["source"] == "jit"


@pytest.mark.parametrize("name", sorted(MODELS))
def test_oracle_rpy_states_are_the_raw_draws(oracle, grbda, name):
    """The oracle's rpy states hold the draws the quaternion model turns into a quaternion: the same positions, the
    angles in [-1, 1) with rpyToQuat(angles) = the quaternion, the same joint coordinates, velocities and aux."""
    m = rpy_model(grbda, name)
    o = rpy_oracle(oracle, m, name)
    oq = oracle.OracleModel(name) if MODELS[name] else mirror_to_oracle(quaternion_model(grbda, name), oracle)
    q, yd, aux = o.generate_states(64, seed=5, first_index=100)
    qq, ydq, auxq = oq.generate_states(64, seed=5, first_index=100)
    assert np.array_equal(q[:, :3], qq[:, :3]) and np.array_equal(q[:, 6:], qq[:, 7:])
    assert np.array_equal(yd, ydq) and np.array_equal(aux, auxq)
    assert (q[:, 3:6] >= -1.0).all() and (q[:, 3:6] < 1.0).all()
    # the rotation of the rpy base is the one of the quaternion base (forward kinematics of the base body)
    _, R, _ = o.forward_kinematics(q, yd)
    _, Rq, _ = oq.forward_kinematics(qq, ydq)
    assert np.abs(R - Rq).max() < 1e-14


# ---- CPU: the emitted programs -------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(MODELS))
def test_emitted_programs_match_oracle(grbda, oracle, name, tmp_path):
    """ID, FD (both programs), FK, H, the external-force programs (default set and every body), contact kinematics,
    contact Jacobians, applyTestForce and OSIM, replayed in numpy against the oracle, at generated states and at
    gimbal lock."""
    m = rpy_model(grbda, name)
    o = rpy_oracle(oracle, m, name)
    q, yd, aux = gimbal_states(o, 28, seed=7)
    B = q.shape[0]
    ins = [q, yd, aux]
    # what the base coordinates may enter: the dynamics see the base orientation only through gravity, which is along
    # the world z axis (invariant under the yaw, the first rotation of E = Rx Ry Rz); the mass matrix in body
    # coordinates does not depend on the base at all; forward kinematics reads every base coordinate
    base = set(range(6))
    for algo, want in ((grbda.ALGO_ID, {ROLL, PITCH}), (grbda.ALGO_FD, {ROLL, PITCH}), (LTL, {ROLL, PITCH}),
                       (grbda.ALGO_H, set()), (grbda.ALGO_FK, base)):
        assert positions_read(m, algo, tmp_path / "reads") & base == want, algo
    assert rel(run_tape(dump(m, grbda.ALGO_ID, tmp_path / "id"), ins)[0], o.inverse_dynamics(q, yd, aux)) < TOL
    ydd = o.forward_dynamics(q, yd, aux)
    assert rel(run_tape(dump(m, grbda.ALGO_FD, tmp_path / "fd"), ins)[0], ydd) < TOL
    assert rel(run_tape(dump(m, LTL, tmp_path / "ltl"), ins)[0], ydd) < TOL
    assert rel(run_tape(dump(m, grbda.ALGO_H, tmp_path / "h"), ins)[0].reshape(-1, o.nv, o.nv), o.mass_matrix(q)) < TOL
    p, R, v = o.forward_kinematics(q, yd)
    fk = run_tape(dump(m, grbda.ALGO_FK, tmp_path / "fk"), ins)
    for got, want in zip(fk, (p, R, v)):
        assert rel(got.reshape(want.shape), want) < TOL
    # contact points (placed on the default force bodies, so before those become every body)
    bodies, offsets, ee = contact_set(m)
    m.setContactPoints(bodies, offsets, ee)
    o.set_contact_points(bodies, offsets, ee)
    pc, vc = run_tape(dump(m, grbda.ALGO_CONTACT_KIN, tmp_path / "ck"), ins)
    po, vo = o.contact_kinematics(q, yd)
    assert rel(pc.reshape(po.shape), po) < TOL and rel(vc.reshape(vo.shape), vo) < TOL
    J = run_tape(dump(m, grbda.ALGO_CONTACT_JAC, tmp_path / "cj"), ins)[0].reshape(B, m.ncp, 6, m.nv)
    assert rel(J, o.contact_jacobians(q, world=True)) < TOL
    assert rel(np.einsum("bcik,bk->bci", J[:, :, 3:, :], yd), vo) < 1e-12
    ft = np.random.default_rng(2).uniform(-1, 1, size=(B, m.ncp, 3))
    d, lam = run_tape(dump(m, grbda.ALGO_TEST_FORCE, tmp_path / "tf"), [q, ft.reshape(B, -1), aux])
    do, lamo = o.apply_test_force(q, ft)
    assert rel(d.reshape(do.shape), do) < TOL_OSIM and rel(lam.reshape(lamo.shape), lamo) < TOL_OSIM
    L = run_tape(dump(m, grbda.ALGO_OSIM, tmp_path / "os"), ins)[0].reshape(B, 6 * m.nee, 6 * m.nee)
    assert rel(L, o.inverse_osim(q)) < TOL_OSIM
    # external forces: the default set (terminal links), then every body
    rng = np.random.default_rng(5)
    tau_plain = o.inverse_dynamics(q, yd, aux)
    for bodies_f in (m.externalForceBodies(), list(range(m.nb))):
        m.setExternalForceBodies(bodies_f)
        f = rng.uniform(-20, 20, size=(B, len(bodies_f), 6))
        f_full = np.zeros((B, o.nb, 6))
        f_full[:, bodies_f, :] = f
        ff = f.reshape(B, -1)
        tau_ext = o.dynamics_with_external_forces(q, yd, aux, f_full, forward=False)
        assert rel(run_tape(dump(m, grbda.ALGO_GFS, tmp_path / "gfs"), [q, ff, tau_plain])[0], tau_ext) < TOL
        assert rel(tau_ext, tau_plain) > 1e-3
        tau_eff = run_tape(dump(m, grbda.ALGO_GFA, tmp_path / "gfa"), [q, ff, aux])[0]
        ydd_ext = o.dynamics_with_external_forces(q, yd, aux, f_full, forward=True)
        assert rel(o.forward_dynamics(q, yd, tau_eff), ydd_ext) < TOL_FD
    m.setExternalForceBodies([])


# ---- CPU: derivatives ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(MODELS))
def test_jacobian_programs_match_oracle_and_finite_differences(grbda, oracle, name, tmp_path):
    """Programs 12 / 13 against the oracle's dual-number Jacobians, and both against central differences of the oracle's
    primal functions (the identity tangent map of the rpy base: d / d q of every stored entry), so that a convention
    the two share cannot hide."""
    m = rpy_model(grbda, name)
    o = rpy_oracle(oracle, m, name)
    q, yd, aux = gimbal_states(o, 8, seed=3)
    for algo, forward, tol in ((grbda.ALGO_ID_DERIV, False, TOL), (grbda.ALGO_FD_DERIV, True, TOL_FD)):
        outs = run_tape(dump(m, algo, tmp_path / ("d%d" % algo)), [q, yd, aux])
        want = o.dynamics_derivatives(q, yd, aux, forward)
        assert len(outs) == len(want)
        for got, w in zip(outs, want):
            assert rel(got.reshape(w.shape).transpose(0, 2, 1), w) < tol  # the programs write column-major matrices
        f = o.forward_dynamics if forward else o.inverse_dynamics
        num = central_differences(lambda x: [f(x, yd, aux)], q)[0]
        assert rel(want[0], num) < FD_BOUND
        num_v = np.stack([(f(q, yd + FD_H * e, aux) - f(q, yd - FD_H * e, aux)) / (2 * FD_H) for e in np.eye(o.nv)], 2)
        assert rel(want[1], num_v) < FD_BOUND


@pytest.mark.parametrize("name", sorted(MODELS))
def test_vjp_programs_match_oracle(grbda, oracle, name, tmp_path):
    """Programs 14-18 against the oracle's Jacobians contracted with random cotangents. The rpy base has no manifold, so
    q_bar = w^T d out / d q on EVERY stored position entry, for the forward dynamics as well. The external-force and
    contact q_bar against central differences of the oracle (it has no Jacobians of those) and against a complex-step
    replay of the primal programs."""
    m = rpy_model(grbda, name)
    o = rpy_oracle(oracle, m, name)
    q, yd, aux = gimbal_states(o, 8, seed=11)
    B = q.shape[0]
    rng = np.random.default_rng(1)
    w = rng.uniform(-1.0, 1.0, (B, o.nv))
    H = o.mass_matrix(q)
    vjp = {}
    for algo, forward, tol in ((grbda.ALGO_ID_VJP, False, TOL), (grbda.ALGO_FD_VJP, True, TOL_FD)):
        q_bar, yd_bar, aux_bar = run_tape(dump(m, algo, tmp_path / ("v%d" % algo)), [q, yd, np.concatenate([aux, w], 1)])
        d = o.dynamics_derivatives(q, yd, aux, forward)
        assert q_bar.shape == q.shape
        assert rel(q_bar, np.einsum("bi,bij->bj", w, d[0])) < tol
        assert rel(yd_bar, np.einsum("bi,bij->bj", w, d[1])) < tol
        want_aux = np.linalg.solve(H, w[:, :, None])[:, :, 0] if forward else np.einsum("bij,bj->bi", H, w)
        assert rel(aux_bar, want_aux) < tol
        vjp[forward] = (q_bar, aux_bar)
    # external forces on every body: tau = ID - J^T f and ydd = FD(tau + J^T f)
    m.setExternalForceBodies(list(range(m.nb)))
    f = rng.uniform(-20.0, 20.0, (B, 6 * m.nb))
    f_full = f.reshape(B, m.nb, 6)
    bodies = list(range(m.nb))
    tau_eff = run_tape(dump(m, grbda.ALGO_GFA, tmp_path / "gfa"), [q, f, aux])[0]
    fdv = run_tape(dump(m, grbda.ALGO_FD_VJP, tmp_path / "fdv"), [q, yd, np.concatenate([tau_eff, w], 1)])
    for algo, primal, cot, base, forward in ((grbda.ALGO_GFS_VJP, grbda.ALGO_GFS, w, vjp[False][0], False),
                                             (grbda.ALGO_GFA_VJP, grbda.ALGO_GFA, fdv[2], fdv[0], True)):
        gq, gf = run_tape(dump(m, algo, tmp_path / ("v%d" % algo)), [q, f, cot])
        assert rel(gf, f_bar_oracle(o, bodies, q, yd, aux, w, forward)) < (TOL_FD if forward else TOL)
        assert rel(gq, complex_step_q_bar(dump(m, primal, tmp_path / ("p%d" % primal)), q, [f, aux], cot)) < TOL
        ext = lambda x: [o.dynamics_with_external_forces(x, yd, aux, f_full, forward=forward)]  # noqa: E731
        num = central_differences(ext, q)[0]
        assert rel(base + gq, np.einsum("bi,bik->bk", w, num)) < FD_BOUND
    m.setExternalForceBodies([])
    # contact kinematics
    bodies, offsets, ee = contact_set(m)
    m.setContactPoints(bodies, offsets, ee)
    o.set_contact_points(bodies, offsets, ee)
    p_bar, v_bar = rng.uniform(-1.0, 1.0, (B, m.ncp, 3)), rng.uniform(-1.0, 1.0, (B, m.ncp, 3))
    packed = np.concatenate([p_bar.reshape(B, -1), v_bar.reshape(B, -1)], axis=1)
    q_bar, yd_bar = run_tape(dump(m, grbda.ALGO_CONTACT_KIN_VJP, tmp_path / "ckv"), [q, yd, packed])
    J_lin = o.contact_jacobians(q, world=True)[:, :, 3:, :]
    assert rel(yd_bar, np.einsum("bci,bcik->bk", v_bar, J_lin)) < TOL
    dp, dv = central_differences(lambda x: list(o.contact_kinematics(x, yd)), q)
    want = np.einsum("bi,bik->bk", p_bar.reshape(B, -1), dp) + np.einsum("bi,bik->bk", v_bar.reshape(B, -1), dv)
    assert rel(q_bar, want) < FD_BOUND
    assert rel(q_bar, complex_step_q_bar(dump(m, grbda.ALGO_CONTACT_KIN, tmp_path / "ck"), q, [yd], packed)) < TOL


# ---- CPU: the emitted CUDA text and the run-time compiler ----------------------------------------------------
def test_emitted_cuda_text_on_the_host(grbda, oracle, tmp_path):
    """The CUDA text of ID, FD (both programs, plain and parked), H and FK compiled for the host against the oracle;
    the generated range check rejects a state whose roll, pitch or yaw is beyond the fast sin/cos range."""
    m = rpy_model(grbda, "mini_cheetah")
    o = rpy_oracle(oracle, m, "mini_cheetah")
    q, yd, aux = gimbal_states(o, 24, seed=29)
    want = {0: o.inverse_dynamics(q, yd, aux), 1: o.forward_dynamics(q, yd, aux), LTL: o.forward_dynamics(q, yd, aux),
            3: o.mass_matrix(q).reshape(q.shape[0], -1)}
    for program, park in [(0, False), (0, True), (1, False), (LTL, False), (LTL, True), (3, False)]:
        outs, in_range, _ = run_emitted_source(m, program, park, [q] if program == 3 else [q, yd, aux], tmp_path,
                                               "p%d_%d" % (program, park))
        assert rel(outs[0], want[program]) < TOL, (program, park)
        assert in_range == q.shape[0]
    p, R, v = o.forward_kinematics(q, yd)
    outs, in_range, _ = run_emitted_source(m, 2, False, [q, yd], tmp_path, "fk")
    for got, w in zip(outs, (p, R, v)):
        assert rel(got.reshape(w.shape), w) < TOL
    assert in_range == q.shape[0]
    # a state is out of range when an angle the program reads is: roll and pitch for the dynamics, all three for FK
    far = ((1, ROLL), (5, PITCH), (9, YAW))
    q_far = q.copy()
    for row, k in far:
        q_far[row, k] += 2.0 * np.pi * TURNS
    for program, ins, n_far in ((0, [q_far, yd, aux], 2), (LTL, [q_far, yd, aux], 2), (2, [q_far, yd], 3)):
        _, in_range, _ = run_emitted_source(m, program, False, ins, tmp_path, "far%d" % program)
        assert in_range == q.shape[0] - n_far, program


def test_run_time_compiler_builds_rpy_cubins(grbda, tmp_path):
    """NVRTC, without a device: FP64 ID / FD / FK / H, the state generator and FP32 ID / FK / H of an rpy model."""
    jobs = [(a, False) for a in (grbda.ALGO_ID, grbda.ALGO_FD, grbda.ALGO_FK, grbda.ALGO_H, -1)] + \
           [(a, True) for a in (grbda.ALGO_ID, grbda.ALGO_FK, grbda.ALGO_H)]

    def compile_one(job):
        algo, f32 = job
        m = rpy_model(grbda, "mini_cheetah")  # one handle per thread
        src, cubin = str(tmp_path / ("%d_%d.cu" % job)), str(tmp_path / ("%d_%d.cubin" % job))
        m.jit_compile(algo, f32, src, cubin)
        return open(src).read(), open(cubin, "rb").read()

    with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as pool:
        results = list(pool.map(compile_one, jobs))
    for (algo, f32), (text, blob) in zip(jobs, results):
        assert blob[:4] == b"\x7fELF" and len(blob) > 10000, (algo, f32)
        if algo == -1:
            # the generator stores the rpy draws as they are; the integration step refuses the state
            assert "rpyToQuat" not in text and "q[3 + i] = rpy[i]" in text and "ok = false;" in text
        else:
            assert "// kernel: grbda_kernels::" in text


# ---- GPU ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


_GPU = {}


def gpu_case(grbda, oracle, torch, name):
    """Device model, oracle and a ragged batch of generated states, shared by the GPU tests of one model."""
    if name not in _GPU:
        m = rpy_model(grbda, name, device=0)
        o = rpy_oracle(oracle, m, name)
        q, yd, aux, flags = m.generateStates(N, seed=42)
        assert int(flags.sum()) == 0
        _GPU[name] = dict(m=m, o=o, q=q, yd=yd, aux=aux, np=[t.cpu().numpy() for t in (q, yd, aux)])
    return _GPU[name]


def _np(t):
    return t.detach().cpu().numpy()


def _rand(torch, shape, like, lo=-1.0, hi=1.0, seed=0):
    g = torch.Generator(device=like.device).manual_seed(seed)
    return torch.rand(shape, dtype=torch.float64, device=like.device, generator=g) * (hi - lo) + lo


def _check_dynamics(m, o, q, yd, aux, tol=TOL):
    """ID, FD, H, FK and the bias force against the oracle (the criteria of test_dynamics_parity_f64)."""
    qn, ydn, auxn = _np(q), _np(yd), _np(aux)
    tau_o = o.inverse_dynamics(qn, ydn, auxn)
    outs = dict(tau=m.inverseDynamics(q, yd, aux), ydd=m.forwardDynamics(q, yd, aux), H=m.getMassMatrix(q))
    p, R, v = m.forwardKinematics(q, yd)
    C = m.getBiasForceVector(q, yd)
    for t in list(outs.values()) + [p, R, v, C]:
        assert bool(t.isfinite().all())
    assert relrows(_np(outs["tau"]), tau_o) < tol
    assert relrows(_np(outs["ydd"]), o.forward_dynamics(qn, ydn, auxn)) < tol
    assert relrows(_np(outs["H"]), o.mass_matrix(qn)) < tol
    for g, w in zip((p, R, v), o.forward_kinematics(qn, ydn)):
        assert relrows(_np(g), w) < tol
    C_o = o.inverse_dynamics(qn, ydn, np.zeros_like(ydn))
    scale = np.maximum(np.abs(tau_o).max(1), np.abs(C_o).max(1))
    assert (np.abs(_np(C) - C_o).max(1) / np.maximum(1e-3, scale)).max() < tol


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MODELS))
def test_state_generator_matches_oracle(grbda, oracle, torch, name):
    """generateStates bit for bit equal to the oracle's states; the rpy angles are the raw draws in [-1, 1), which the
    quaternion model turns into its quaternion."""
    c = gpu_case(grbda, oracle, torch, name)
    m, o = c["m"], c["o"]
    q, yd, aux, flags = m.generateStates(N, seed=123, first_index=1000)
    assert int(flags.sum()) == 0
    for got, want in zip((q, yd, aux), o.generate_states(N, seed=123, first_index=1000)):
        assert np.array_equal(_np(got), want)
    angles = _np(q)[:, ROLL:YAW + 1]
    assert (angles >= -1.0).all() and (angles < 1.0).all() and np.unique(angles).size == angles.size
    quat = quaternion_model(grbda, name, device=0)
    qq, ydq, auxq, _ = quat.generateStates(N, seed=123, first_index=1000)
    assert torch.equal(q[:, :3], qq[:, :3]) and torch.equal(q[:, 6:], qq[:, 7:])
    assert torch.equal(yd, ydq) and torch.equal(aux, auxq)
    _, R, _ = m.forwardKinematics(q, yd)
    _, Rq, _ = quat.forwardKinematics(qq, ydq)
    assert float((R[:, 0] - Rq[:, 0]).abs().max()) < 1e-14


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MODELS))
def test_dynamics_parity_f64(grbda, oracle, torch, name):
    c = gpu_case(grbda, oracle, torch, name)
    _check_dynamics(c["m"], c["o"], c["q"], c["yd"], c["aux"])
    for algo in (grbda.ALGO_ID, grbda.ALGO_FD, grbda.ALGO_FK, grbda.ALGO_H):
        assert c["m"].kernel_info(algo)["source"] == "jit"


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MODELS))
def test_dynamics_parity_f32(grbda, oracle, torch, name):
    """FP32 ID, H and FK against the FP64 oracle on float-rounded states."""
    c = gpu_case(grbda, oracle, torch, name)
    m, o = c["m"], c["o"]
    q32, yd32, aux32 = c["q"].float(), c["yd"].float(), c["aux"].float()
    qn, ydn, auxn = (x.double().cpu().numpy() for x in (q32, yd32, aux32))
    assert relrows(_np(m.inverseDynamics(q32, yd32, aux32).double()), o.inverse_dynamics(qn, ydn, auxn)) < TOL32
    assert relrows(_np(m.getMassMatrix(q32).double()), o.mass_matrix(qn)) < TOL32
    for g, w in zip(m.forwardKinematics(q32, yd32), o.forward_kinematics(qn, ydn)):
        g = _np(g.double())
        assert np.isfinite(g).all() and np.abs(g - w).max() / np.abs(w).max() < TOL32
    assert m.kernel_info(grbda.ALGO_FK, True)["source"] == "jit"


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MODELS))
def test_external_forces(grbda, oracle, torch, name):
    """inverseDynamics / forwardDynamics with f_ext on the default bodies and on every body."""
    c = gpu_case(grbda, oracle, torch, name)
    m, o, (q, yd, aux), (qn, ydn, auxn) = c["m"], c["o"], (c["q"], c["yd"], c["aux"]), c["np"]
    try:
        for seed, bodies in ((3, m.externalForceBodies()), (4, list(range(m.nb)))):
            m.setExternalForceBodies(bodies)
            f = _rand(torch, (N, len(bodies), 6), q, -20.0, 20.0, seed=seed)
            f_full = np.zeros((N, o.nb, 6))
            f_full[:, bodies, :] = _np(f)
            tau = m.inverseDynamics(q, yd, aux, f_ext=f)
            assert relrows(_np(tau), o.dynamics_with_external_forces(qn, ydn, auxn, f_full, forward=False)) < TOL
            ydd = m.forwardDynamics(q, yd, aux, f_ext=f)
            assert relrows(_np(ydd), o.dynamics_with_external_forces(qn, ydn, auxn, f_full, forward=True)) < TOL
    finally:
        m.setExternalForceBodies([])


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MODELS))
def test_operational_space(grbda, oracle, torch, name):
    c = gpu_case(grbda, oracle, torch, name)
    m, o, q, yd, (qn, ydn, _) = c["m"], c["o"], c["q"], c["yd"], c["np"]
    bodies, offsets, ee = contact_set(m)
    m.setContactPoints(bodies, offsets, ee)
    o.set_contact_points(bodies, offsets, ee)
    p, v = m.contactKinematics(q, yd)
    po, vo = o.contact_kinematics(qn, ydn)
    assert relrows(_np(p), po) < TOL and relrows(_np(v), vo) < TOL
    J = m.contactJacobians(q)
    assert relrows(_np(J), o.contact_jacobians(qn, world=True)) < TOL
    f = _rand(torch, (N, m.ncp, 3), q, -0.5, 0.5, seed=5)
    d, lam = m.applyTestForce(q, f)
    do, lamo = o.apply_test_force(qn, _np(f))
    assert relrows(_np(d), do) < TOL_OSIM and relrows(_np(lam), lamo, floor=1e-12) < TOL_OSIM
    assert relrows(_np(m.inverseOperationalSpaceInertiaMatrix(q)), o.inverse_osim(qn)) < TOL_OSIM


@pytest.mark.gpu
def test_derivatives_and_gradients(grbda, oracle, torch, tmp_path):
    """MiniCheetah with an rpy base: the Jacobian entry points, every VJP entry point (plain, with forces, contact) and
    gradcheck through the autograd functions with q requiring grad (no manifold to project onto)."""
    c = gpu_case(grbda, oracle, torch, "mini_cheetah")
    m, o, (q, yd, aux), (qn, ydn, auxn) = c["m"], c["o"], (c["q"], c["yd"], c["aux"]), c["np"]
    for fn, forward, tol in ((m.inverseDynamicsDerivatives, False, TOL), (m.forwardDynamicsDerivatives, True, TOL_FD)):
        for g, w in zip(fn(q, yd, aux), o.dynamics_derivatives(qn, ydn, auxn, forward)):
            assert rel(_np(g), w) < tol
    w = _rand(torch, (N, m.nv), q, seed=1)
    wn = _np(w)
    H = o.mass_matrix(qn)
    jac = {}
    for vjp, forward, tol in ((m.inverseDynamicsVJP, False, TOL), (m.forwardDynamicsVJP, True, TOL_FD)):
        q_bar, yd_bar, aux_bar = (_np(t) for t in vjp(q, yd, aux, w))
        jac[forward] = d = o.dynamics_derivatives(qn, ydn, auxn, forward)
        assert rel(q_bar, np.einsum("bi,bij->bj", wn, d[0])) < tol  # every stored entry
        assert rel(yd_bar, np.einsum("bi,bij->bj", wn, d[1])) < tol
        want_aux = np.linalg.solve(H, wn[:, :, None])[:, :, 0] if forward else np.einsum("bij,bj->bi", H, wn)
        assert rel(aux_bar, want_aux) < tol
    # with forces: f_bar by linearity against the oracle; q_bar against central differences of the oracle's dynamics
    # with forces on the first states; yd_bar / tau_bar against the oracle's Jacobians
    bodies = m.externalForceBodies()
    f = _rand(torch, (N, len(bodies), 6), q, -20.0, 20.0, seed=2)
    f_full = np.zeros((N, o.nb, 6))
    f_full[:, bodies, :] = _np(f)
    n = 8
    for vjp, forward, tol in ((m.inverseDynamicsVJP, False, TOL), (m.forwardDynamicsVJP, True, TOL_FD)):
        q_bar, yd_bar, aux_bar, f_bar = (_np(t) for t in vjp(q, yd, aux, w, f_ext=f))
        assert rel(f_bar.reshape(N, -1)[:n], f_bar_oracle(o, bodies, qn[:n], ydn[:n], auxn[:n], wn[:n], forward)) < tol
        ext = lambda x: [o.dynamics_with_external_forces(x, ydn[:n], auxn[:n], f_full[:n], forward=forward)]  # noqa
        assert rel(q_bar[:n], np.einsum("bi,bik->bk", wn[:n], central_differences(ext, qn[:n])[0])) < FD_BOUND
        if forward:
            tau_eff = _np(m.inverseDynamics(q, yd, m.forwardDynamics(q, yd, aux, f_ext=f)))
            d = o.dynamics_derivatives(qn[:n], ydn[:n], tau_eff[:n], True)
            assert rel(aux_bar[:n], np.linalg.solve(H[:n], wn[:n, :, None])[:, :, 0]) < tol
        else:
            d = jac[False]
            assert rel(aux_bar, np.einsum("bij,bj->bi", H, wn)) < tol
        assert rel(yd_bar[:n], np.einsum("bi,bij->bj", wn[:n], d[1][:n])) < tol
    # contact kinematics
    cb, offsets, ee = contact_set(m)
    m.setContactPoints(cb, offsets, ee)
    o.set_contact_points(cb, offsets, ee)
    p_bar, v_bar = _rand(torch, (N, m.ncp, 3), q, seed=9), _rand(torch, (N, m.ncp, 3), q, seed=10)
    q_bar, yd_bar = (_np(t) for t in m.contactKinematicsVJP(q, yd, p_bar, v_bar))
    pb, vb = _np(p_bar).reshape(N, -1), _np(v_bar).reshape(N, -1)
    assert rel(yd_bar, np.einsum("bi,bik->bk", vb, o.contact_jacobians(qn, world=True)[:, :, 3:, :].reshape(N, -1, m.nv))) < TOL
    dp, dv = central_differences(lambda x: list(o.contact_kinematics(x, ydn[:n])), qn[:n])
    assert rel(q_bar[:n], np.einsum("bi,bik->bk", pb[:n], dp) + np.einsum("bi,bik->bk", vb[:n], dv)) < FD_BOUND
    want = run_tape(dump(m, grbda.ALGO_CONTACT_KIN_VJP, tmp_path / "ckv"), [qn, ydn, np.concatenate([pb, vb], 1)])
    assert rel(q_bar, want[0]) < TOL and rel(yd_bar, want[1]) < TOL
    # gradcheck: every input, q included
    gad = grbda.autograd
    qs, yds, auxs = (t[:3].clone() for t in (q, yd, aux))
    fs = f[:3].clone()
    for fn in (gad.inverse_dynamics, gad.forward_dynamics):
        args = tuple(t.clone().requires_grad_(True) for t in (qs, yds, auxs))
        assert torch.autograd.gradcheck(lambda a, b, c_: fn(m, a, b, c_), args)
        args = tuple(t.clone().requires_grad_(True) for t in (qs, yds, auxs, fs))
        assert torch.autograd.gradcheck(lambda a, b, c_, d_: fn(m, a, b, c_, f_ext=d_), args)
    args = (qs.clone().requires_grad_(True), yds.clone().requires_grad_(True))
    assert torch.autograd.gradcheck(lambda a, b: gad.contact_kinematics(m, a, b), args)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MODELS))
def test_gimbal_lock(grbda, oracle, torch, name):
    """pitch = +-pi/2 exactly and +-pi/2 +- 1e-9 on every state: R is well defined and the velocities are a body
    twist, so ID, FD, FK and H hold the normal tolerance, without NaN."""
    c = gpu_case(grbda, oracle, torch, name)
    q = c["q"].clone()
    q[:, PITCH] = torch.tensor([np.pi / 2, -np.pi / 2, np.pi / 2 + 1e-9, -np.pi / 2 - 1e-9],
                               dtype=torch.float64, device=q.device).repeat(N // 4 + 1)[:N]
    _check_dynamics(c["m"], c["o"], q, c["yd"], c["aux"])


def _entry_points(grbda, c):
    """(program, call, oracle reference) of ID, FD, H and FK on the states of a GPU case."""
    m, o, yd, aux = c["m"], c["o"], c["yd"], c["aux"]
    ydn, auxn = c["np"][1:]
    return [(grbda.ALGO_ID, lambda x: (m.inverseDynamics(x, yd, aux),), lambda x: [o.inverse_dynamics(x, ydn, auxn)]),
            (grbda.ALGO_FD, lambda x: (m.forwardDynamics(x, yd, aux),), lambda x: [o.forward_dynamics(x, ydn, auxn)]),
            (grbda.ALGO_H, lambda x: (m.getMassMatrix(x),), lambda x: [o.mass_matrix(x)]),
            (grbda.ALGO_FK, lambda x: m.forwardKinematics(x, yd), lambda x: o.forward_kinematics(x, ydn))]


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MODELS))
def test_rpy_angles_beyond_the_fast_sincos_range(grbda, oracle, torch, name, tmp_path):
    """The generated range check must bound the rpy angles. Whole turns (2.5e12 rad) on the roll of a state in tile 0
    and on the yaw of a state in tile 2, and a pitch of 1e16 rad in tile 1 (where the fast reduction itself breaks
    down: |x| 2 / pi > 2^51). A tile is flagged when it holds such an angle that the program reads (the dynamics read
    roll and pitch, FK all three, H none). The flagged tiles match the oracle, and their other states were recomputed
    by the flagged-tile pass with the library sin/cos (not all bit for bit the fast kernel's); every other tile is bit
    for bit the unperturbed call; each call is the fast kernel plus the flagged-tile pass."""
    c = gpu_case(grbda, oracle, torch, name)
    m, q = c["m"], c["q"]
    for algo, call, ref in _entry_points(grbda, c):
        base = [_np(t).reshape(N, -1) for t in call(q)]
        b = m.kernel_info(algo)["block"]
        far = ((5, ROLL), (b + 5, PITCH), (2 * b + 5, YAW))
        qf = q.clone()
        qf[far[0]] += 2.0 * np.pi * TURNS
        qf[far[1]] = 1.0e16
        qf[far[2]] -= 2.0 * np.pi * TURNS
        torch.cuda.synchronize()
        before = grbda.launch_count()
        outs = [_np(t).reshape(N, -1) for t in call(qf)]
        torch.cuda.synchronize()
        assert grbda.launch_count() - before == 2, algo
        reads = positions_read(m, algo if algo != grbda.ALGO_FD else m.kernel_info(algo)["program"], tmp_path / "t")
        flagged = np.zeros(N, dtype=bool)
        tiles = [range(r // b * b, min(N, (r // b + 1) * b)) for r, k in far if k in reads]
        for t in tiles:
            flagged[list(t)] = True
        assert len(tiles) == {grbda.ALGO_H: 0, grbda.ALGO_FK: 3}.get(algo, 2), algo
        for g, g0, w in zip(outs, base, ref(_np(qf))):
            w = w.reshape(N, -1)
            assert np.isfinite(g).all()
            if flagged.any():
                assert relrows(g[flagged], w[flagged]) < TOL, (algo, "flagged tiles")
            assert np.array_equal(g[~flagged], g0[~flagged]), (algo, "unflagged tiles changed")
        for t in tiles:
            rows = [r for r in t if r not in (r_ for r_, _ in far)]
            assert any(not np.array_equal(g[rows], g0[rows]) for g, g0 in zip(outs, base)), (algo, "tile not recomputed")


@pytest.mark.gpu
def test_nan_rpy_angle_stays_in_its_state(grbda, oracle, torch, tmp_path):
    """A NaN roll, pitch or yaw gives NaN in that state's outputs that read the angle, and nowhere else."""
    c = gpu_case(grbda, oracle, torch, "mini_cheetah")
    m, q = c["m"], c["q"]
    rows = {130: ROLL, 200: PITCH, 300: YAW}
    qn = q.clone()
    for r, k in rows.items():
        qn[r, k] = float("nan")
    for algo, call, _ in _entry_points(grbda, c):
        reads = positions_read(m, algo if algo != grbda.ALGO_FD else m.kernel_info(algo)["program"], tmp_path / "t")
        for out in call(qn):
            flat = _np(out).reshape(N, -1)
            for r in range(N):
                assert np.isnan(flat[r]).any() == (rows.get(r) in reads), (algo, r)
                assert np.isnan(flat[r]).any() or np.isfinite(flat[r]).all(), (algo, r)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MODELS))
def test_integration_step_refuses_rpy_states(grbda, oracle, torch, name):
    """integrate / step have no rpy rule: every state is flagged, the base positions are copied, the velocities are
    still advanced (yd_out = yd + dt ydd) and the other clusters move with them."""
    c = gpu_case(grbda, oracle, torch, name)
    m, q, yd, aux = c["m"], c["q"], c["yd"], c["aux"]
    dt = 1e-3
    ydd = m.forwardDynamics(q, yd, aux)
    for q1, yd1, flags in (m.integrate(q, yd, ydd, dt), m.step(q, yd, aux, dt)):
        assert bool((flags == 1).all())
        assert torch.equal(q1[:, :6], q[:, :6])
        assert float((yd1 - (yd + dt * ydd)).abs().max()) < 1e-15
        assert float((q1[:, 6:] - (q[:, 6:] + dt * yd1[:, 6:])).abs().max()) < 1e-15
