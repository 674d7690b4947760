"""Reverse mode of the integration step and of the simulation step: grbda_cuda_integrate_vjp_f64,
grbda_cuda_step_vjp_f64 and the torch.autograd functions built on them (differentiable rollouts).

  * CPU: a reference built from the oracle (explicit clusters analytically, the quaternion base by complex step of a
    numpy restatement of the step, implicit clusters by G^T at the projected point), itself checked against central
    differences of the oracle's step on every stored entry, on and off the unit quaternion / phi = 0; the emitted
    `struct StepVjp` compiled with g++ and run against it, at rest, at tiny and at large base angular velocities and
    on both sides of the series switch; the sm_100a cubin; refusals.
  * GPU: the C ABI against the reference, the step VJP against the composition of the forward-dynamics VJP and the
    integration VJP, gradcheck, 10-step rollouts against central differences, the autograd plumbing.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_compiler_cpu import contact_set
from test_rpy_base import rpy_model
from test_vjp import quat_product, quat_to_R, rel

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "generalized_rbda_b200", "csrc")
ROBOTS = ["revolute_chain_with_rotor_4", "mini_cheetah", "mit_humanoid", "tello_with_arms", "four_bar", "six_bar",
          "planar_leg_linkage"]
ORACLE_ROBOTS = ("revolute_chain_with_rotor_4", "mini_cheetah", "mit_humanoid", "tello_with_arms")
INTEGRATE_VJP = -2  # program id of the reverse integration step (grbda_cuda_jit_compile / grbda_cuda_model_prepare)
DT = 0.05           # a t = |omega| / 40: base angular velocities of order one use the closed form, 1e-5 the series
SWITCH = 1e-2 / (0.5 * DT)  # |omega| where integrateFreeQuaternionVjp switches (a t = 1e-2)
TOL = 1e-11
# The kernel and the oracle project with the same Newton iteration but round phi differently, so they can stop at
# points ~1e-13 apart on phi = 0; G at those points differs by the conditioning of K_dep, which for the planar leg
# linkage reaches ~5e-11 of G (measured over 300 states).
TOL_PROJECTION = {"planar_leg_linkage": 1e-10}


def oracle_model(oracle, m, robot):
    from mirror import mirror_to_oracle
    return oracle.OracleModel(robot) if robot in ORACLE_ROBOTS else mirror_to_oracle(m, oracle)


# ---- CPU reference ------------------------------------------------------------------------------------------------
def quat_increment(om, dt):
    """d(omega) = (cos(a t), sin(a t) / t omega), a = dt / 2, t = |omega|, written analytically in omega (even in t) so
    that the complex step sees its derivative also at omega = 0."""
    a = 0.5 * dt
    u = a * a * (om @ om)
    if abs(u) < 1e-6:
        c = 1 - u / 2 + u * u / 24 - u ** 3 / 720
        S = a * (1 - u / 6 + u * u / 120 - u ** 3 / 5040)
    else:
        at = np.sqrt(u)
        c, S = np.cos(at), a * np.sin(at) / at
    return np.concatenate([[c], S * om])


def free_step(x, dt):
    """The quaternion base of the step, x = [p (3), quat (4), omega_b (3), v_b (3)] -> [p', quat'] (stategen.cuh)."""
    R = quat_to_R(x[3:7]).T  # body -> world, the polynomial of the raw entries
    om, v = R @ x[7:10], R @ x[10:13]
    r = quat_product(quat_increment(om, dt), x[3:7])
    return np.concatenate([x[:3] + dt * v, r / np.sqrt(r @ r)])


def free_step_jacobian(q7, v6, dt):
    """[7, 13] = d [p', quat'] / d [p, quat, omega_b, v_b] by complex step."""
    x = np.concatenate([q7, v6]).astype(complex)
    J = np.zeros((7, 13))
    h = 1e-30
    for k in range(13):
        xk = x.copy()
        xk[k] += 1j * h
        J[:, k] = free_step(xk, dt).imag / h
    return J


def reference_vjp(m, o, q, yd, ydd, dt, q_out_bar, yd_out_bar, q_next=None):
    """(q_bar, yd_bar, ydd_bar) of the integration step, state by state. The implicit clusters are differentiated at
    q_next, the projected positions (default: those of the oracle's step)."""
    if q_next is None:
        q_next = o.integrate(q, yd, ydd, dt)[0]
    ydn = yd + dt * ydd
    q_bar = np.zeros_like(q)
    v_bar = yd_out_bar.copy()
    for ci, c in enumerate(m.clusters()):
        pi, vi, N, n = c["position_index"], c["velocity_index"], c["num_positions"], c["num_velocities"]
        for b in range(q.shape[0]):
            qob = q_out_bar[b, pi:pi + N]
            if c["type"] == 0:  # quaternion base
                J = free_step_jacobian(q[b, pi:pi + 7], ydn[b, vi:vi + 6], dt)
                q_bar[b, pi:pi + 7] = J[:, :7].T @ qob
                v_bar[b, vi:vi + 6] += J[:, 7:].T @ qob
            elif c["type"] == 1:  # roll-pitch-yaw base: copied
                q_bar[b, pi:pi + 6] = qob
            elif c["type"] == 3:  # implicit: G^T q_out_bar at the projected point
                G = o.cluster_constraint(ci, q_next[b], np.zeros(o.nv))[0]
                ind_bar = G.T @ qob
                q_bar[b, pi + np.flatnonzero(c["independent"])] = ind_bar
                v_bar[b, vi:vi + n] += dt * ind_bar
            else:
                q_bar[b, pi:pi + N] = qob
                v_bar[b, vi:vi + n] += dt * qob
    return q_bar, v_bar, dt * v_bar


def random_cotangents(B, nq, nv, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(-1.0, 1.0, (B, nq)), rng.uniform(-1.0, 1.0, (B, nv))


def states(o, count, seed):
    """Oracle states (ydd = aux), and the same with positions pushed off the unit quaternion / off phi = 0."""
    q, yd, ydd = o.generate_states(count, seed=seed)
    rng = np.random.default_rng(seed)
    q = np.concatenate([q, q + rng.uniform(-0.05, 0.05, q.shape)])
    return q, np.concatenate([yd, yd]), np.concatenate([ydd, ydd])


def base_angular_velocities(q, yd, ydd, speeds, seed):
    """Copies of the first state whose NEW base angular velocity yd + dt ydd (the base is cluster 0) has the given
    norms, along one direction."""
    e = np.random.default_rng(seed).normal(size=3)
    q, yd, ydd = (np.repeat(x[:1], len(speeds), axis=0) for x in (q, yd, ydd))
    ydd[:, :3] = 0.0
    yd[:, :3] = np.outer(speeds, e / np.linalg.norm(e))
    return q, yd, ydd


@pytest.mark.parametrize("robot", ROBOTS)
def test_reference_matches_central_differences(grbda, oracle, robot):
    """The reference against central differences of the oracle's step on every stored entry of q, yd and ydd."""
    m = grbda.ClusterTreeModel.from_robot(robot, device=None)
    o = oracle_model(oracle, m, robot)
    q, yd, ydd = states(o, 3, seed=41)
    B, nq, nv = q.shape[0], o.nq, o.nv
    qob, ydob = random_cotangents(B, nq, nv, 5)
    want = reference_vjp(m, o, q, yd, ydd, DT, qob, ydob)
    x = np.concatenate([q, yd, ydd], axis=1)
    n = x.shape[1]
    h = 1e-6

    def loss(X):
        qn, ydn, _ = o.integrate(np.ascontiguousarray(X[:, :nq]), np.ascontiguousarray(X[:, nq:nq + nv]),
                                 np.ascontiguousarray(X[:, nq + nv:]), DT)
        return np.einsum("bi,bi->b", np.repeat(qob, n, axis=0), qn) + np.einsum("bi,bi->b", np.repeat(ydob, n, axis=0), ydn)

    Xp = np.repeat(x[:, None, :], n, axis=1)
    Xm = Xp.copy()
    Xp[:, np.arange(n), np.arange(n)] += h
    Xm[:, np.arange(n), np.arange(n)] -= h
    cd = ((loss(Xp.reshape(B * n, n)) - loss(Xm.reshape(B * n, n))) / (2 * h)).reshape(B, n)
    assert rel(np.concatenate(want, axis=1), cd) < 1e-6


# ---- the emitted struct StepVjp on the host -------------------------------------------------------------------------
HOST_MAIN = r'''
#include "host_body_prelude.h"
// one state on the host: the device shell and the thread indices are not needed
#define GRBDA_KERNELS_BATCHED_KERNEL_CUH
#define __global__
#define __launch_bounds__(n)
static inline unsigned __umulhi(unsigned a, unsigned b) { return (unsigned)(((unsigned long long)a * b) >> 32); }
static struct { unsigned x; } blockIdx, blockDim, threadIdx;
namespace grbda_kernels { using namespace host_body; } // grbda_sincos of the emitted evaluators
#include "step_vjp.cu"
#include <cstdio>
#include <vector>
int main(int argc, char **argv)
{
    using S = grbda_jit::StepVjp;
    FILE *f = std::fopen(argv[1], "rb");
    int64_t B = 0;
    double dt = 0;
    if (!f || std::fread(&B, 8, 1, f) != 1 || std::fread(&dt, 8, 1, f) != 1) return 2;
    std::vector<double> q(B * S::NQ), yd(B * S::NV), ydd(B * S::NV), qob(B * S::NQ), ydob(B * S::NV);
    for (auto *v : {&q, &yd, &ydd, &qob, &ydob})
        if (std::fread(v->data(), 8, v->size(), f) != v->size()) return 3;
    std::fclose(f);
    std::vector<double> qb(B * S::NQ), ydb(B * S::NV), yddb(B * S::NV), flags(B);
    for (int64_t b = 0; b < B; b++)
        flags[b] = grbda_kernels::integrateVjpState<S>(&q[b * S::NQ], &yd[b * S::NV], &ydd[b * S::NV], dt,
                                                       &qob[b * S::NQ], &ydob[b * S::NV], &qb[b * S::NQ],
                                                       &ydb[b * S::NV], &yddb[b * S::NV]) ? 0.0 : 1.0;
    f = std::fopen(argv[2], "wb");
    for (auto *v : {&qb, &ydb, &yddb, &flags})
        std::fwrite(v->data(), 8, v->size(), f);
    std::fclose(f);
    return 0;
}
'''


def host_step_vjp(m, tag, tmp_path):
    """Compile the run-time source of the reverse integration step (emitted StepVjp + kernels/stategen.cuh) with g++;
    returns run(q, yd, ydd, dt, q_out_bar, yd_out_bar) -> (q_bar, yd_bar, ydd_bar, flags)."""
    d = tmp_path / tag
    d.mkdir()
    m.jit_compile(INTEGRATE_VJP, False, str(d / "step_vjp.cu"), None)
    (d / "main.cpp").write_text(HOST_MAIN)
    exe = str(d / "run")
    subprocess.run(["/usr/bin/g++", "-O1", "-std=c++17", "-I", HERE, "-I", CSRC, "-I", str(d), "-o", exe,
                    str(d / "main.cpp")], check=True)

    def run(q, yd, ydd, dt, qob, ydob):
        B = q.shape[0]
        with open(d / "in.bin", "wb") as f:
            f.write(np.int64(B).tobytes() + np.float64(dt).tobytes())
            for a in (q, yd, ydd, qob, ydob):
                f.write(np.ascontiguousarray(a, dtype=np.float64).tobytes())
        subprocess.run([exe, str(d / "in.bin"), str(d / "out.bin")], check=True)
        raw = np.fromfile(d / "out.bin", dtype=np.float64)
        nq, nv = m.nq, m.nv
        sizes = np.cumsum([B * nq, B * nv, B * nv])
        qb, ydb, yddb, flags = np.split(raw, sizes)
        return qb.reshape(B, nq), ydb.reshape(B, nv), yddb.reshape(B, nv), flags.astype(np.int32)
    return run, (d / "step_vjp.cu").read_text()


@pytest.mark.parametrize("robot", ROBOTS)
def test_emitted_step_vjp_on_the_host(grbda, oracle, robot, tmp_path):
    m = grbda.ClusterTreeModel.from_robot(robot, device=None)
    o = oracle_model(oracle, m, robot)
    run, text = host_step_vjp(m, "s", tmp_path)
    assert "struct StepVjp" in text and "grbda_integrate_vjp_kernel<grbda_jit::StepVjp>" in text
    q, yd, ydd = states(o, 6, seed=17)
    if m.clusters()[0]["type"] == 0:
        # base angular velocities: at rest, tiny, on both sides of the series switch, of order one and large
        speeds = [0.0, 1e-9, 1e-5, SWITCH * (1 - 1e-12), SWITCH * (1 + 1e-12), 1.0, 30.0]
        qs, yds, ydds = base_angular_velocities(*o.generate_states(1, seed=19), speeds, seed=3)
        q, yd, ydd = np.concatenate([q, qs]), np.concatenate([yd, yds]), np.concatenate([ydd, ydds])
    qob, ydob = random_cotangents(q.shape[0], o.nq, o.nv, 7)
    qob[-7:], ydob[-7:] = qob[-7], ydob[-7]  # one cotangent for the copies
    got = run(q, yd, ydd, DT, qob, ydob)
    flags = o.integrate(q, yd, ydd, DT)[2]
    assert np.array_equal(got[3], flags)
    ok = flags == 0
    assert ok.sum() >= q.shape[0] - 1
    want = reference_vjp(m, o, q, yd, ydd, DT, qob, ydob)
    for g, w in zip(got[:3], want):
        assert np.all(np.isfinite(g[ok])) and rel(g[ok], w[ok]) < TOL_PROJECTION.get(robot, TOL)
    if m.clusters()[0]["type"] == 0:
        for g in got[:3]:  # continuous across the switch
            assert rel(g[-4:-3], g[-3:-2]) < 1e-11


def test_emitted_step_vjp_of_an_rpy_base(grbda, oracle, tmp_path):
    """Roll-pitch-yaw base: every state flagged, its positions' q_bar is q_out_bar (the derivative of the copy)."""
    from mirror import mirror_to_oracle
    m = rpy_model(grbda, "mini_cheetah")
    o = mirror_to_oracle(m, oracle)
    run, text = host_step_vjp(m, "rpy", tmp_path)
    assert "ok = false;" in text
    q, yd, ydd = o.generate_states(8, seed=13)
    qob, ydob = random_cotangents(8, o.nq, o.nv, 9)
    q_bar, yd_bar, ydd_bar, flags = run(q, yd, ydd, DT, qob, ydob)
    assert np.all(flags == 1)
    assert np.array_equal(q_bar[:, :6], qob[:, :6])
    want = reference_vjp(m, o, q, yd, ydd, DT, qob, ydob)
    for g, w in zip((q_bar, yd_bar, ydd_bar), want):
        assert rel(g, w) < TOL


def test_generator_and_reverse_step_share_the_cluster_evaluators(grbda, tmp_path):
    """One evaluator per implicit cluster in both sources; only the reverse step's has the K_ind function."""
    m = grbda.ClusterTreeModel.from_robot("tello_with_arms", device=None)
    m.jit_compile(-1, False, str(tmp_path / "gen.cu"), None)
    m.jit_compile(INTEGRATE_VJP, False, str(tmp_path / "vjp.cu"), None)
    gen, vjp = (tmp_path / "gen.cu").read_text(), (tmp_path / "vjp.cu").read_text()
    implicit = sum(c["type"] == 3 for c in m.clusters())
    assert implicit > 0 and gen.count(" eval(const double *q") == implicit == vjp.count(" eval(const double *q")
    assert "jacobian(" not in gen and vjp.count(" jacobian(const double *q") == implicit
    assert "struct StepVjp" not in gen and "struct Gen" not in vjp


def test_integrate_vjp_compiles_for_sm100a_without_a_device(grbda, tmp_path):
    for robot in ("tello_with_arms", "mini_cheetah"):
        m = grbda.ClusterTreeModel.from_robot(robot, device=None)
        cubin = str(tmp_path / (robot + ".cubin"))
        m.jit_compile(INTEGRATE_VJP, False, None, cubin)
        blob = open(cubin, "rb").read()
        assert blob[:4] == b"\x7fELF" and len(blob) > 5000


def test_integrate_vjp_refuses_host_only_handles(grbda):
    m = grbda.ClusterTreeModel.from_robot("mini_cheetah", device=None)
    L = grbda.lib()
    assert L.grbda_cuda_integrate_vjp_f64(m._h, None, None, None, 0.1, None, None, None, None, None, None, 1, None) == 4
    assert L.grbda_cuda_step_vjp_f64(m._h, None, None, None, None, 0.1, None, None, None, None, None, None, None, 1,
                                     None) == 4  # GRBDA_ERR_NO_DEVICE
    assert L.grbda_cuda_integrate_vjp_f64(None, None, None, None, 0.1, None, None, None, None, None, None, 1, None) == 1
    assert L.grbda_cuda_step_vjp_f64(None, None, None, None, None, 0.1, None, None, None, None, None, None, None, 1,
                                     None) == 1
    with pytest.raises(grbda.GrbdaError):
        m.prepare(INTEGRATE_VJP)


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def _np(t):
    return t.detach().cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ROBOTS)
def test_integrate_vjp_on_gpu(grbda, oracle, torch, robot):
    m = grbda.ClusterTreeModel.from_robot(robot, device=0)
    o = oracle_model(oracle, m, robot)
    B = 300  # ragged: two full CTAs and a tail
    q, yd, ydd, flags = m.generateStates(B)
    assert int(flags.sum()) == 0
    g = torch.Generator(device=q.device).manual_seed(11)
    qob = torch.rand(B, m.nq, dtype=torch.float64, device=q.device, generator=g) * 2 - 1
    ydob = torch.rand(B, m.nv, dtype=torch.float64, device=q.device, generator=g) * 2 - 1
    launches = grbda.launch_count()
    q_bar, yd_bar, ydd_bar, fl = m.integrateVJP(q, yd, ydd, DT, qob, ydob)
    assert grbda.launch_count() == launches + 1  # one kernel (include/grbda_cuda.h)
    q_next, _, flags = m.integrate(q, yd, ydd, DT)
    assert torch.equal(fl, flags)
    ok = _np(fl) == 0
    assert ok.sum() >= 0.8 * B  # steps of 0.05 s at unit velocities: Newton fails on a few TelloWithArms states
    # at the kernel's own projected positions, where the VJP is defined: the device's Newton iteration (fused
    # multiply-adds) need not stop where the oracle's does
    want = reference_vjp(m, o, *(_np(t) for t in (q, yd, ydd)), DT, _np(qob), _np(ydob), q_next=_np(q_next))
    for got, w in zip((q_bar, yd_bar, ydd_bar), want):
        assert rel(_np(got)[ok], w[ok]) < TOL


def _with_forces(m, torch, B, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.rand(B, len(m.externalForceBodies()), 6, dtype=torch.float64, device="cuda", generator=g) * 40 - 20


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["mini_cheetah", "tello_with_arms", "revolute_chain_with_rotor_4", "four_bar"])
def test_step_vjp_is_the_composition(grbda, torch, robot):
    """stepVJP = forwardDynamicsVJP after integrateVJP at ydd = FD(q, yd, tau [+ J^T f]); the launch count the header
    states; f_bar untouched without forces."""
    m = grbda.ClusterTreeModel.from_robot(robot, device=0)
    B = 300
    q, yd, tau, _ = m.generateStates(B)
    qob, ydob = torch.rand_like(q) * 2 - 1, torch.rand_like(yd) * 2 - 1
    for f in (None, _with_forces(m, torch, B, 3)):
        ydd = m.forwardDynamics(q, yd, tau, f_ext=f)
        qi, ydi, yddb, fli = m.integrateVJP(q, yd, ydd, DT, qob, ydob)
        dyn = m.forwardDynamicsVJP(q, yd, tau, yddb, f_ext=f)
        c0 = grbda.launch_count()
        m.forwardDynamics(q, yd, tau, f_ext=f)
        c1 = grbda.launch_count()
        m.forwardDynamicsVJP(q, yd, tau, yddb, f_ext=f)
        c2 = grbda.launch_count()
        got = m.stepVJP(q, yd, tau, DT, qob, ydob, f_ext=f)
        assert grbda.launch_count() - c2 == (c1 - c0) + 1 + (c2 - c1) + 1
        assert torch.equal(got[-1], fli)
        assert rel(_np(got[0]), _np(dyn[0] + qi)) < 1e-12 and rel(_np(got[1]), _np(dyn[1] + ydi)) < 1e-12
        assert rel(_np(got[2]), _np(dyn[2])) < 1e-12
        if f is not None:
            assert got[3].shape == f.shape and rel(_np(got[3]), _np(dyn[3])) < 1e-12
    # f_ext = NULL: f_bar is not written
    sentinel = torch.full((B, 6), 7.0, dtype=torch.float64, device=q.device)
    out = [torch.empty_like(q), torch.empty_like(yd), torch.empty_like(yd)]
    p = [C.c_void_p(t.data_ptr()) for t in (q, yd, tau)]
    st = grbda.lib().grbda_cuda_step_vjp_f64(m._h, *p, None, C.c_double(DT), C.c_void_p(qob.data_ptr()),
                                             C.c_void_p(ydob.data_ptr()), *[C.c_void_p(t.data_ptr()) for t in out],
                                             C.c_void_p(sentinel.data_ptr()), None, B, None)
    torch.cuda.synchronize()
    assert st == 0 and torch.all(sentinel == 7.0)


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["revolute_chain_with_rotor_4", "mini_cheetah"])
def test_gradcheck(grbda, torch, robot):
    """integrate over (q, yd, ydd): its q_bar is the exact derivative of the step; step over (yd, tau, f_ext)."""
    gad = grbda.autograd
    m = grbda.ClusterTreeModel.from_robot(robot, device=0)
    q, yd, aux, _ = m.generateStates(3)
    f = _with_forces(m, torch, 3, 5)
    args = tuple(t.clone().requires_grad_(True) for t in (q, yd, aux))
    assert torch.autograd.gradcheck(lambda a, b, c: gad.integrate(m, a, b, c, DT)[:2], args)
    args = tuple(t.clone().requires_grad_(True) for t in (yd, aux, f))
    assert torch.autograd.gradcheck(lambda b, c, d: gad.step(m, q, b, c, DT, f_ext=d)[:2], args)


@pytest.mark.gpu
@pytest.mark.parametrize("robot,tol", [("mini_cheetah", 1e-6), ("tello_with_arms", 1e-5)])
def test_rollout_gradients(grbda, torch, robot, tol):
    """10 steps of autograd.step at dt = 1e-3; the loss weights the final q, yd and the contact positions / velocities.
    Directional derivatives of the tau and f_ext sequences, of yd0 and of q0 along the retraction
    h -> integrate(q0, u, 0, h) against central differences of the same rollout with m.step."""
    gad = grbda.autograd
    m = grbda.ClusterTreeModel.from_robot(robot, device=0)
    bodies, offsets, ee = contact_set(m)
    m.setContactPoints(bodies, offsets, ee)
    B, T, dt, h = 8, 10, 1e-3, 1e-6
    q0, yd0, _, _ = m.generateStates(B)
    gen = torch.Generator(device="cuda").manual_seed(2)

    def rand(*shape):
        return torch.rand(*shape, dtype=torch.float64, device="cuda", generator=gen) * 2 - 1

    nf = len(m.externalForceBodies())
    taus, fs = rand(T, B, m.nv) * 5, rand(T, B, nf, 6) * 10
    wq, wyd, wp, wv = rand(B, m.nq), rand(B, m.nv), rand(B, m.ncp, 3), rand(B, m.ncp, 3)

    def loss_of(q, yd):
        p, v = gad.contact_kinematics(m, q, yd)
        return (wq * q).sum() + (wyd * yd).sum() + (wp * p).sum() + (wv * v).sum()

    def rollout(q, yd, taus, fs, differentiable):
        for t in range(T):
            if differentiable:
                q, yd, flags = gad.step(m, q, yd, taus[t], dt, f_ext=fs[t])
            else:
                q, yd, flags = m.step(q, yd, taus[t], dt, f_ext=fs[t])
            assert int(flags.sum()) == 0
        return loss_of(q, yd)

    leaves = [t.clone().requires_grad_(True) for t in (q0, yd0, taus, fs)]
    rollout(*leaves, True).backward()
    q_grad, yd_grad, tau_grad, f_grad = (t.grad for t in leaves)

    def check(analytic, plus, minus):
        with torch.no_grad():
            cd = (rollout(*plus, False) - rollout(*minus, False)).item() / (2 * h)
        assert abs(analytic - cd) <= tol * max(abs(cd), abs(analytic)), (analytic, cd)

    d = rand(T, B, m.nv)
    check((tau_grad * d).sum().item(), (q0, yd0, taus + h * d, fs), (q0, yd0, taus - h * d, fs))
    d = rand(T, B, nf, 6)
    check((f_grad * d).sum().item(), (q0, yd0, taus, fs + h * d), (q0, yd0, taus, fs - h * d))
    d = rand(B, m.nv)
    check((yd_grad * d).sum().item(), (q0, yd0 + h * d, taus, fs), (q0, yd0 - h * d, taus, fs))
    u = rand(B, m.nv)
    zero = torch.zeros_like(u)
    qp, qm = m.integrate(q0, u, zero, h)[0], m.integrate(q0, u, zero, -h)[0]
    check((q_grad * (qp - qm)).sum().item() / (2 * h), (qp, yd0, taus, fs), (qm, yd0, taus, fs))


@pytest.mark.gpu
def test_autograd_plumbing(grbda, torch):
    gad = grbda.autograd
    m = grbda.ClusterTreeModel.from_robot("mini_cheetah", device=0)
    B = 64
    q, yd, tau, _ = m.generateStates(B)
    f = _with_forces(m, torch, B, 7)
    wq, wyd = torch.rand_like(q), torch.rand_like(yd)
    # forward results bit for bit those of m.integrate / m.step, flags without a gradient
    for fn, plain in ((lambda *a: gad.integrate(m, *a, DT), lambda *a: m.integrate(*a, DT)),
                      (lambda *a: gad.step(m, *a, DT, f_ext=f), lambda *a: m.step(*a, DT, f_ext=f))):
        args = [t.clone().requires_grad_(True) for t in (q, yd, tau)]
        out = fn(*args)
        for a, b in zip(out, plain(q, yd, tau)):
            assert torch.equal(a.detach(), b)
        assert out[0].grad_fn is not None and out[2].grad_fn is None and not out[2].requires_grad
        # one VJP call: the gradients are what the entry point returns
        c0 = grbda.launch_count()
        ((out[0] * wq).sum() + (out[1] * wyd).sum()).backward()
        assert grbda.launch_count() > c0
    want = m.stepVJP(q, yd, tau, DT, wq, wyd, f_ext=f)
    # subsets of the inputs: only tau, only yd, only f_ext
    for k in range(3):
        xs = [q, yd, tau]
        x = xs[k].clone().requires_grad_(True)
        xs[k] = x
        qo, ydo, _ = gad.step(m, *xs, DT, f_ext=f)
        ((qo * wq).sum() + (ydo * wyd).sum()).backward()
        assert torch.equal(x.grad, want[k])
    fa = f.clone().requires_grad_(True)
    qo, ydo, _ = gad.step(m, q, yd, tau, DT, f_ext=fa)
    ((qo * wq).sum() + (ydo * wyd).sum()).backward()
    assert torch.equal(fa.grad, want[3])
    # only yd_out used: the q_out cotangent is zero
    ya = yd.clone().requires_grad_(True)
    gad.integrate(m, q, ya, tau, DT)[1].sum().backward()
    assert torch.equal(ya.grad, m.integrateVJP(q, yd, tau, DT, torch.zeros_like(q), torch.ones_like(yd))[1])
    # second derivatives, float32
    xa = tau.clone().requires_grad_(True)
    with pytest.raises(RuntimeError, match="create_graph"):
        torch.autograd.grad(gad.step(m, q, yd, xa, DT)[1].sum(), xa, create_graph=True)
    with pytest.raises(TypeError):
        gad.step(m, q.float(), yd.float(), tau.float(), DT)
    with pytest.raises(TypeError):
        gad.integrate(m, q.float(), yd.float(), tau.float(), DT)
    # no states
    e = [t[:0].clone().requires_grad_(True) for t in (q, yd, tau)]
    qo, ydo, flags = gad.step(m, *e, DT)
    (qo.sum() + ydo.sum()).backward()
    assert flags.shape == (0,) and all(t.grad is not None and t.grad.shape == t.shape for t in e)
    e = [t[:0].clone().requires_grad_(True) for t in (q, yd, tau)]
    qo, ydo, _ = gad.integrate(m, *e, DT)
    (qo.sum() + ydo.sum()).backward()
    assert all(t.grad is not None and t.grad.shape == t.shape for t in e)


@pytest.mark.gpu
def test_vjp_c_abi_arguments(grbda, torch):
    m = grbda.ClusterTreeModel.from_robot("mini_cheetah", device=0)
    B = 8
    q, yd, tau, _ = m.generateStates(B)
    f = _with_forces(m, torch, B, 1)
    vp = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    dt = C.c_double(DT)
    L = grbda.lib()
    m.prepare(INTEGRATE_VJP)  # before graph capture, say
    # integrate VJP: q, yd, ydd, q_out_bar, yd_out_bar -> q_bar, yd_bar, ydd_bar (flags optional)
    ins = [vp(t) for t in (q, yd, tau)]
    bars = [vp(t) for t in (q, yd)]
    outs = [vp(torch.empty_like(t)) for t in (q, yd, yd)]
    flags = vp(torch.empty(B, dtype=torch.int32, device=q.device))
    fn = L.grbda_cuda_integrate_vjp_f64
    assert fn(m._h, *ins, dt, *bars, *outs, flags, B, None) == 0
    assert fn(m._h, *ins, dt, *bars, *outs, None, B, None) == 0
    c = grbda.launch_count()
    assert fn(m._h, *ins, dt, *bars, *outs, flags, 0, None) == 0 and grbda.launch_count() == c
    assert fn(m._h, *ins, dt, *bars, *outs, flags, -1, None) == 1
    for k in range(8):
        args = ins + bars + outs
        args[k] = None
        assert fn(m._h, *args[:3], dt, *args[3:], flags, B, None) == 1
    # step VJP: q, yd, tau, f_ext, q_out_bar, yd_out_bar -> q_bar, yd_bar, tau_bar, f_bar (f_bar needed with f_ext)
    fn = L.grbda_cuda_step_vjp_f64
    f_bar = vp(torch.empty_like(f))
    assert fn(m._h, *ins, vp(f), dt, *bars, *outs, f_bar, flags, B, None) == 0
    assert fn(m._h, *ins, vp(f), dt, *bars, *outs, None, flags, B, None) == 1
    c = grbda.launch_count()
    assert fn(m._h, *ins, vp(f), dt, *bars, *outs, f_bar, flags, 0, None) == 0 and grbda.launch_count() == c
    assert fn(m._h, *ins, None, dt, *bars, *outs, None, flags, -1, None) == 1
    for k in range(8):
        args = ins + bars + outs
        args[k] = None
        assert fn(m._h, *args[:3], None, dt, *args[3:], None, flags, B, None) == 1
    torch.cuda.synchronize()
