"""Rigid point contacts: contact-constrained forward dynamics (ALGO_CONTACT_FD) and contact impulses
(ALGO_CONTACT_IMPULSE), the C entry points grbda_cuda_contact_forward_dynamics_f64 / grbda_cuda_contact_impulse_f64 and
ClusterTreeModel.contactForwardDynamics / contactImpulse.

The reference solution is a dense numpy solve of the same damped, masked system built from the oracle's mass matrix,
bias forces (inverse dynamics at ydd = 0), world contact Jacobians and contact-point accelerations at ydd = 0; it
shares no code with the model compiler. The contact-point accelerations come from the oracle's own
forwardAccelerationKinematics (tests/oracle_contact_accelerations.cpp) and are pinned by central differences of the
oracle's contact velocities along its own integration step.

  * CPU: the emitted programs replayed in numpy against that solution (random masks, all active, all inactive; eps = 0
    on full-rank contact sets, eps > 0 on redundant ones), one emitted body compiled for the host, sm_100a cubins,
    the refusals a host-only handle can show.
  * GPU: parity with the oracle on 2^12 states per model, the physical residuals, the cross-check with external
    forces, batch / alignment / flagged-tile edges, a changed contact set, every refusal.
"""
import ctypes as C
import os

import numpy as np
import pytest

from tape import load_tape, run_tape

HERE = os.path.dirname(os.path.abspath(__file__))
# Per-state relative error of the replayed programs and of the kernels against the dense reference (Ref.check): below
# TOL, or below 2e-14 cond(A) where that is larger, on states with cond(A) <= COND_MAX. Measured: at most 4e-12 on the
# full-rank sets (cond(A) <= 6e3); on the toe-and-heel set (eps = 1e-6, cond(A) up to ~5e7) at most 4.5e-15 cond(A)
# over 2^12 states on a B200.
TOL = 1e-9
COND_MAX = 1e8
ORACLE_ROBOTS = ("mini_cheetah", "tello_with_arms", "mit_humanoid", "revolute_pair_chain_with_rotor_4")


def rel(a, b):
    return np.abs(a - b).max() / max(1e-300, np.abs(b).max())


_ACCEL = {}


def contact_accelerations(o, q, yd, ydd):
    """[B, n_cp, 3]: the oracle's classical world acceleration of every contact point at (q, yd, ydd), gravity excluded
    (tests/oracle_contact_accelerations.cpp, compiled once per process with the oracle's C API into a library of its
    own that reads the oracle's handles)."""
    if "lib" not in _ACCEL:
        import subprocess
        import tempfile
        _ACCEL["dir"] = tempfile.TemporaryDirectory(prefix="grbda_contact_oracle_")
        path = os.path.join(_ACCEL["dir"].name, "liboracle_contact_accelerations.so")
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.run([cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-w", "-I", os.path.join(os.path.dirname(HERE), "oracle"),
                        "-o", path, os.path.join(HERE, "oracle_contact_accelerations.cpp"), "-lpthread"], check=True)
        _ACCEL["lib"] = C.CDLL(path)
    q, yd, ydd = (np.ascontiguousarray(x, dtype=np.float64) for x in (q, yd, ydd))
    a = np.zeros((q.shape[0], o.ncp, 3))
    P = lambda x: x.ctypes.data_as(C.POINTER(C.c_double))  # noqa: E731
    rc = _ACCEL["lib"].oracle_contact_accelerations(o._h, P(q), P(yd), P(ydd), P(a), C.c_int64(q.shape[0]), 0)
    assert rc == 0
    return a


def load_model(grbda, name, device=None):
    if name.endswith(".urdf"):
        return grbda.ClusterTreeModel.from_urdf(os.path.join(HERE, "urdf_corpus", name), device=device)
    return grbda.ClusterTreeModel.from_robot(name, device=device)


def oracle_model(oracle, m, name):
    if name in ORACLE_ROBOTS:
        return oracle.OracleModel(name)
    from mirror import mirror_to_oracle
    return mirror_to_oracle(m, oracle)


# (model, contact set, damping). "feet": one point with an offset on each of the first `n` terminal links (distinct
# bodies); "toe_heel": two points on each of the first two terminal links (6 rows of rank 5 per foot).
CASES = {
    "mini_cheetah": ("mini_cheetah", "feet", 4, 0.0),
    "tello_with_arms": ("tello_with_arms", "feet", 4, 0.0),
    "mit_humanoid": ("mit_humanoid", "feet", 4, 0.0),
    "four_bar": ("four_bar", "feet", 1, 1e-3),                                     # nv = 1: 3 rows of rank 1
    "revolute_pair_chain_with_rotor_4": ("revolute_pair_chain_with_rotor_4", "feet", 1, 1e-4),  # planar: rank 2
    "four_bar_branch_2_3": ("four_bar_branch_2_3.urdf", "feet", 2, 0.0),          # floating base, four-bar loops
    "tello_toe_heel": ("tello_with_arms", "toe_heel", 2, 1e-6),
}


def contact_points(m, kind, n):
    feet = m.externalForceBodies()[:n]
    rng = np.random.default_rng(7)
    if kind == "feet":
        return list(feet), rng.uniform(-0.05, 0.05, (len(feet), 3))
    bodies = [b for b in feet for _ in range(2)]
    offsets = np.array([[0.08, 0.0, -0.04], [-0.05, 0.0, -0.04]] * len(feet))
    return bodies, offsets


def setup(grbda, oracle, case, device=None):
    name, kind, n, eps = CASES[case]
    m = load_model(grbda, name, device)
    o = oracle_model(oracle, m, name)
    bodies, offsets = contact_points(m, kind, n)
    m.setContactPoints(bodies, offsets)
    o.set_contact_points(bodies, offsets)
    return m, o, eps


def kkt_reference(o, q, yd, tau, s, eps, impulse=False, restitution=0.0):
    """Dense solve of the masked, damped system of include/grbda_cuda.h from the oracle's quantities: a Ref with out =
    ydd (dynamics) or yd_plus (impulse), lam [B, n_cp, 3] and cond(A) per state."""
    q, yd, tau = (np.ascontiguousarray(x) for x in (q, yd, tau))
    B, nv = q.shape[0], o.nv
    H = o.mass_matrix(q)
    J = o.contact_jacobians(q, world=True)[:, :, 3:, :].reshape(B, -1, nv)
    m = J.shape[1]
    Y = np.linalg.solve(H, np.swapaxes(J, 1, 2))                               # [B, nv, m]
    S = np.repeat(s.astype(np.float64), 3, axis=1)                              # [B, m]
    A = S[:, :, None] * np.einsum("bik,bkj->bij", J, Y) * S[:, None, :]
    A += (1.0 - S)[:, :, None] * np.eye(m) + eps * np.eye(m)
    if impulse:
        base = yd
        b = -(1.0 + restitution) * S * np.einsum("bik,bk->bi", J, yd)
    else:
        Cb = o.inverse_dynamics(q, yd, np.zeros_like(yd))
        base = np.linalg.solve(H, (tau - Cb)[:, :, None])[:, :, 0]
        c = contact_accelerations(o, q, yd, np.zeros_like(yd)).reshape(B, m)
        b = -S * (np.einsum("bik,bk->bi", J, base) + c)
    lam = np.linalg.solve(A, b[:, :, None])[:, :, 0]
    corr = np.einsum("bkm,bm->bk", Y, lam)
    out = base + corr
    # scale of out: the larger of its two terms (the constrained ydd can be a small difference of large ones)
    out_scale = np.maximum(np.abs(base).max(1), np.abs(corr).max(1))
    return Ref(out, lam.reshape(B, -1, 3), np.linalg.cond(A), out_scale)


class Ref:
    def __init__(self, out, lam, cond, out_scale):
        self.out, self.lam, self.cond, self.out_scale = out, lam, cond, out_scale

    def errors(self, out, lam, active, against=None):
        """Per-state relative errors of (out, lam) against (self.out, self.lam) or `against`: out against out_scale,
        lam against its largest entry (states with an active contact)."""
        out_ref, lam_ref = against if against is not None else (self.out, self.lam)
        e_out = np.abs(out.reshape(out.shape[0], -1) - out_ref.reshape(out.shape[0], -1)).max(1)
        e_out = e_out / np.maximum(1e-300, self.out_scale)
        e_lam = np.where(active.any(1), rows_rel(lam, lam_ref), 0.0)
        return np.maximum(e_out, e_lam)

    def check(self, out, lam, active, against=None):
        """Relative error below cond_bound on the states with cond(A) <= COND_MAX, at least half the states checked."""
        e = self.errors(out, lam, active, against)
        ok = self.cond <= COND_MAX
        assert ok.sum() >= len(ok) // 2, self.cond
        bound = cond_bound(self.cond)
        assert (e[ok] < bound[ok]).all(), (e[ok].max(), (e / bound)[ok].max())


def cond_bound(cond):
    """TOL, or 2e-14 cond(A) where that is larger (nearly redundant contacts with a small damping): the forward error
    of a backward-stable m x m solve grows as cond(A) times a small multiple of m u."""
    return np.maximum(TOL, 2e-14 * cond)


def packed_fd(tau, s, eps):
    return np.concatenate([tau, s.astype(np.float64), np.full((tau.shape[0], 1), eps)], axis=1)


def packed_impulse(s, restitution, eps):
    B = s.shape[0]
    return np.concatenate([s.astype(np.float64), np.full((B, 1), restitution), np.full((B, 1), eps)], axis=1)


def masks(B, ncp, seed):
    """Random masks on the first half, then all active, then all inactive."""
    rng = np.random.default_rng(seed)
    s = rng.integers(0, 2, (B, ncp)).astype(np.uint8)
    s[B // 2:B // 2 + B // 4] = 1
    s[B // 2 + B // 4:] = 0
    return s


def rows_rel(a, b):
    """Per-state relative error against the largest entry of the reference row."""
    a, b = a.reshape(a.shape[0], -1), b.reshape(b.shape[0], -1)
    return np.abs(a - b).max(1) / np.maximum(1e-300, np.abs(b).max(1))


def dump(m, algo, path):
    m.dump_program(algo, str(path))
    return load_tape(str(path))


# ---- CPU: the oracle's contact accelerations ------------------------------------------------------------------
@pytest.mark.parametrize("case", ["mini_cheetah", "tello_with_arms", "four_bar", "four_bar_branch_2_3"])
def test_oracle_contact_accelerations_by_central_differences(grbda, oracle, case):
    """d/dt of the contact velocity along the oracle's integration step (+/- dt from the same state) is the contact
    acceleration at (q, yd, ydd), gravity excluded (quaternion base, implicit loops included)."""
    m, o, _ = setup(grbda, oracle, case)
    q, yd, ydd = o.generate_states(8, seed=3)
    dt = 1e-5
    qp, ydp, fp = o.integrate(q, yd, ydd, dt)
    qm, ydm, fm = o.integrate(q, yd, ydd, -dt)
    assert not fp.any() and not fm.any()
    fd = (o.contact_kinematics(qp, ydp)[1] - o.contact_kinematics(qm, ydm)[1]) / (2 * dt)
    a = contact_accelerations(o, q, yd, ydd)
    assert rel(a, fd) < 1e-6
    # the ydd-dependent part is J ydd, and gravity does not enter
    J = o.contact_jacobians(q, world=True)[:, :, 3:, :]
    a0 = contact_accelerations(o, q, yd, np.zeros_like(ydd))
    assert rel(a - a0, np.einsum("bcik,bk->bci", J, ydd)) < 1e-11
    assert np.abs(contact_accelerations(o, q, np.zeros_like(yd), np.zeros_like(ydd))).max() == 0.0


# ---- CPU: the programs -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", sorted(CASES))
def test_contact_programs_match_the_dense_solution(grbda, oracle, case, tmp_path):
    m, o, eps = setup(grbda, oracle, case)
    q, yd, tau = o.generate_states(24, seed=11)
    B, ncp = q.shape[0], m.ncp
    s = masks(B, ncp, seed=5)
    t_fd = dump(m, grbda.ALGO_CONTACT_FD, tmp_path / "fd.tape")
    t_im = dump(m, grbda.ALGO_CONTACT_IMPULSE, tmp_path / "im.tape")
    assert list(t_fd["n_in"]) == [m.nq, m.nv, m.nv + ncp + 1] and list(t_im["n_in"]) == [m.nq, m.nv, ncp + 2]
    ydd, lam = run_tape(t_fd, [q, yd, packed_fd(tau, s, eps)])
    assert ydd.shape == (B, m.nv) and lam.shape == (B, 3 * ncp)
    kkt_reference(o, q, yd, tau, s, eps).check(ydd, lam, s)
    # inactive contacts: exact zeros; all inactive: the forward dynamics itself
    assert (lam.reshape(B, ncp, 3)[s == 0] == 0.0).all()
    none = ~s.any(1)
    ltl = run_tape(dump(m, grbda.PROGRAM_FD_LTL, tmp_path / "ltl.tape"), [q, yd, tau])[0]
    assert rel(ydd[none], ltl[none]) < 1e-12
    assert rel(ltl, o.forward_dynamics(q, yd, tau)) < 1e-9
    for e in (0.0, 0.5, 1.0):
        yp, imp = run_tape(t_im, [q, yd, packed_impulse(s, e, eps)])
        kkt_reference(o, q, yd, tau, s, eps, impulse=True, restitution=e).check(yp, imp, s)
        assert (imp.reshape(B, ncp, 3)[s == 0] == 0.0).all()
        assert (yp[none] == yd[none]).all()


def test_contact_residuals_on_the_tapes(grbda, oracle, tmp_path):
    """H ydd + C = tau + J^T lambda; J_a ydd + c_a = -eps lambda_a; J_a yd_plus = -e J_a yd - eps impulse_a - on a
    redundant set (toe and heel of each foot) with eps > 0 and on a full-rank one with eps = 0. The redundant set's A
    has cond up to ~5e7, which its residuals inherit (~1e-15 cond)."""
    for case, tol in (("tello_toe_heel", 1e-7), ("mini_cheetah", 1e-9)):
        m, o, eps = setup(grbda, oracle, case)
        q, yd, tau = o.generate_states(16, seed=13)
        B, ncp = q.shape[0], m.ncp
        s = np.ones((B, ncp), dtype=np.uint8)
        s[::3, 0] = 0
        ydd, lam = run_tape(dump(m, grbda.ALGO_CONTACT_FD, tmp_path / "fd.tape"), [q, yd, packed_fd(tau, s, eps)])
        J = o.contact_jacobians(q, world=True)[:, :, 3:, :].reshape(B, -1, m.nv)
        tau_back = o.inverse_dynamics(q, yd, ydd) - np.einsum("bik,bi->bk", J, lam)
        assert rel(tau_back, tau) < tol
        S = np.repeat(s, 3, axis=1).astype(bool)
        acc = contact_accelerations(o, q, yd, ydd).reshape(B, -1)
        scale = np.abs(np.einsum("bik,bk->bi", J, ydd)).max()
        assert np.abs(acc + eps * lam)[S].max() < tol * scale
        yp, imp = run_tape(dump(m, grbda.ALGO_CONTACT_IMPULSE, tmp_path / "im.tape"), [q, yd, packed_impulse(s, 0.3, eps)])
        v0, v1 = np.einsum("bik,bk->bi", J, yd), np.einsum("bik,bk->bi", J, yp)
        assert np.abs(v1 + 0.3 * v0 + eps * imp)[S].max() < tol * np.abs(v0).max()


def test_emitted_contact_body_on_the_host(grbda, oracle, tmp_path):
    """The emitted CUDA text of the contact dynamics (plain and parked), compiled for the host (tests/
    host_body_prelude.h), against the dense solution."""
    from test_compiler_cpu import run_emitted_source
    m, o, eps = setup(grbda, oracle, "mini_cheetah")
    q, yd, tau = o.generate_states(12, seed=17)
    s = masks(q.shape[0], m.ncp, seed=2)
    ref = kkt_reference(o, q, yd, tau, s, eps)
    assert (ref.cond <= COND_MAX).all()
    for park in (False, True):
        outs, in_range, text = run_emitted_source(m, grbda.ALGO_CONTACT_FD, park, [q, yd, packed_fd(tau, s, eps)],
                                                  tmp_path, "p%d" % park)
        assert in_range == q.shape[0] and ("PARKED = true" in text) == park
        ref.check(outs[0], outs[1], s)


def test_contact_programs_compile_for_sm100a_without_a_device(grbda, tmp_path):
    for case in sorted(CASES):
        name, kind, n, _ = CASES[case]
        m = load_model(grbda, name)
        bodies, offsets = contact_points(m, kind, n)
        m.setContactPoints(bodies, offsets)
        for algo, n_in2 in ((grbda.ALGO_CONTACT_FD, m.nv + m.ncp + 1), (grbda.ALGO_CONTACT_IMPULSE, m.ncp + 2)):
            src, cubin = str(tmp_path / ("%s_%d.cu" % (case, algo))), str(tmp_path / ("%s_%d.cubin" % (case, algo)))
            m.jit_compile(algo, False, src, cubin)
            blob = open(cubin, "rb").read()
            assert blob[:4] == b"\x7fELF" and len(blob) > 10000
            text = open(src).read()
            assert "N_IN2 = %d" % n_in2 in text and "N_OUT0 = %d, N_OUT1 = %d" % (m.nv, 3 * m.ncp) in text


def test_contact_entry_points_refuse_on_the_host(grbda):
    """What a host-only handle can show: no contact points, bad damping / restitution (GRBDA_ERR_INVALID_ARGUMENT)
    before GRBDA_ERR_NO_DEVICE; prepare / kernel_info / programs without contact points."""
    L = grbda.lib()
    fd, im = L.grbda_cuda_contact_forward_dynamics_f64, L.grbda_cuda_contact_impulse_f64
    m = grbda.ClusterTreeModel.from_robot("mini_cheetah", device=None)
    assert fd(m._h, None, None, None, None, 0.0, None, None, 1, None) == 1
    assert "no contact points" in L.grbda_cuda_last_error_string().decode()
    assert im(m._h, None, None, None, 0.0, 0.0, None, None, 1, None) == 1
    assert fd(None, None, None, None, None, 0.0, None, None, 1, None) == 1
    with pytest.raises(grbda.GrbdaError):
        m.dump_program(grbda.ALGO_CONTACT_FD)
    with pytest.raises(grbda.GrbdaError):
        m.kernel_info(grbda.ALGO_CONTACT_IMPULSE)
    bodies, offsets = contact_points(m, "feet", 4)
    m.setContactPoints(bodies, offsets)
    for eps in (-1e-9, float("nan"), float("inf")):
        assert fd(m._h, None, None, None, None, eps, None, None, 1, None) == 1
        assert im(m._h, None, None, None, 0.0, eps, None, None, 1, None) == 1
    for e in (-0.1, 1.5, float("nan")):
        assert im(m._h, None, None, None, e, 0.0, None, None, 1, None) == 1
    assert fd(m._h, None, None, None, None, 0.0, None, None, 1, None) == 4
    assert im(m._h, None, None, None, 1.0, 0.0, None, None, 1, None) == 4
    info = m.kernel_info(grbda.ALGO_CONTACT_FD)
    assert info["source"] == "jit" and not info["ready"]
    with pytest.raises(grbda.GrbdaError):
        m.prepare(grbda.ALGO_CONTACT_FD)  # host-only handle
    assert m.dump_program(grbda.ALGO_CONTACT_FD)["flops"] > m.dump_program(grbda.ALGO_TEST_FORCE)["flops"] > 0


# ---- GPU -----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def _np(t):
    return t.detach().cpu().numpy()


def _gpu_case(grbda, oracle, torch, case, B, seed):
    m, o, eps = setup(grbda, oracle, case, device=0)
    q, yd, tau, flags = m.generateStates(B, seed=seed)
    assert int(flags.sum()) == 0
    s = torch.from_numpy(masks(B, m.ncp, seed)).to(q.device)
    return m, o, eps, q, yd, tau, s


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_contact_entry_points_match_the_oracle(grbda, oracle, torch, case, tmp_path):
    """2^12 states per model: both entry points against the dense solution and against the replayed programs (the
    same per-state scale and cond(A) bound, Ref.check)."""
    B = 1 << 12
    m, o, eps, q, yd, tau, s = _gpu_case(grbda, oracle, torch, case, B, seed=21)
    ydd, lam = m.contactForwardDynamics(q, yd, tau, active=s, damping=eps)
    yp, imp = m.contactImpulse(q, yd, active=s.bool(), restitution=0.4, damping=eps)
    qn, ydn, taun, sn = _np(q), _np(yd), _np(tau), _np(s)
    assert lam.shape == (B, m.ncp, 3) and imp.shape == (B, m.ncp, 3)
    r_fd = run_tape(dump(m, grbda.ALGO_CONTACT_FD, tmp_path / "fd.tape"), [qn, ydn, packed_fd(taun, sn, eps)])
    r_im = run_tape(dump(m, grbda.ALGO_CONTACT_IMPULSE, tmp_path / "im.tape"), [qn, ydn, packed_impulse(sn, 0.4, eps)])
    ref = kkt_reference(o, qn, ydn, taun, sn, eps)
    ref.check(_np(ydd), _np(lam), sn)
    ref.check(_np(ydd), _np(lam), sn, against=r_fd)
    ref = kkt_reference(o, qn, ydn, taun, sn, eps, impulse=True, restitution=0.4)
    ref.check(_np(yp), _np(imp), sn)
    ref.check(_np(yp), _np(imp), sn, against=r_im)
    assert bool((lam[s == 0] == 0).all()) and bool((imp[s == 0] == 0).all())
    none = ~s.bool().any(1)
    assert torch.equal(yp[none], yd[none])
    # forwardDynamics may run the articulated-body program (four_bar), not the factorisation the contact program uses
    assert rows_rel(_np(ydd[none]), _np(m.forwardDynamics(q, yd, tau)[none])).max() < 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["mini_cheetah", "tello_toe_heel", "four_bar_branch_2_3"])
def test_contact_physical_residuals(grbda, oracle, torch, case):
    """On the device, per state with cond(A) <= COND_MAX and bound cond_bound: ID(q, yd, ydd) - J^T lambda = tau
    (relative to the larger of tau and J^T lambda); the oracle's contact accelerations at ydd are -eps lambda on the
    active contacts (relative to J ydd and c); J_a yd_plus = -e J_a yd - eps impulse_a (relative to J yd)."""
    B = 2048
    m, o, eps, q, yd, tau, s = _gpu_case(grbda, oracle, torch, case, B, seed=23)
    qn, ydn, taun, sn = _np(q), _np(yd), _np(tau), _np(s)
    ydd, lam = m.contactForwardDynamics(q, yd, tau, active=s, damping=eps)
    J = m.contactJacobians(q)[:, :, 3:, :].reshape(B, -1, m.nv)
    JTl = torch.einsum("bik,bi->bk", J, lam.reshape(B, -1))
    r = _np(m.inverseDynamics(q, yd, ydd) - JTl - tau)
    scale = np.maximum(np.abs(taun).max(1), np.abs(_np(JTl)).max(1))
    cond = kkt_reference(o, qn, ydn, taun, sn, eps).cond
    ok = cond <= COND_MAX
    bound = cond_bound(cond)
    assert ok.sum() >= B // 2
    assert ((np.abs(r).max(1) / scale < bound)[ok]).all()
    S = sn.repeat(3, axis=1).astype(bool)
    Jn, yddn, lamn = _np(J), _np(ydd), _np(lam).reshape(B, -1)
    acc = contact_accelerations(o, qn, ydn, yddn).reshape(B, -1)
    c = contact_accelerations(o, qn, ydn, np.zeros_like(ydn)).reshape(B, -1)
    scale = np.maximum(np.abs(np.einsum("bik,bk->bi", Jn, yddn)).max(1), np.abs(c).max(1))
    res = np.where(S, np.abs(acc + eps * lamn), 0.0).max(1)
    assert ((res / scale < bound)[ok]).all()
    for e in (0.0, 0.7):
        yp, imp = m.contactImpulse(q, yd, active=s, restitution=e, damping=eps)
        v0, v1 = np.einsum("bik,bk->bi", Jn, ydn), np.einsum("bik,bk->bi", Jn, _np(yp))
        res = np.where(S, np.abs(v1 + e * v0 + eps * _np(imp).reshape(B, -1)), 0.0).max(1)
        assert ((res / np.abs(v0).max(1) < bound)[ok]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["mini_cheetah", "tello_with_arms", "mit_humanoid"])
def test_contact_forces_are_external_forces(grbda, oracle, torch, case):
    """With the force bodies set to the contact bodies (distinct, one contact each), forwardDynamics with the world
    spatial forces [p x lambda; lambda] (moments about the world origin) reproduces the constrained ydd."""
    B = 1024
    m, o, eps, q, yd, tau, s = _gpu_case(grbda, oracle, torch, case, B, seed=25)
    bodies, _ = contact_points(m, *CASES[case][1:3])
    ydd, lam = m.contactForwardDynamics(q, yd, tau, active=s, damping=eps)
    p, _ = m.contactKinematics(q, yd)
    f = torch.cat([torch.linalg.cross(p, lam, dim=2), lam], dim=2)
    m.setExternalForceBodies(bodies)
    try:
        assert m.externalForceBodies() == list(bodies)
        ydd_ext = m.forwardDynamics(q, yd, tau, f_ext=f.contiguous())
    finally:
        m.setExternalForceBodies([])
    assert rows_rel(_np(ydd_ext), _np(ydd)).max() < 1e-9


@pytest.mark.gpu
def test_contact_edges(grbda, oracle, torch, tmp_path):
    """Batches 0, 1, 127, 129, 2^17 + 1; inputs and outputs at an 8-byte (not 16-byte) offset; flagged tiles (joint
    angles of ~2.5e12 rad); a NULL mask equals an all-ones mask; launches: one pack kernel per call besides the
    program's own."""
    m, o, eps = setup(grbda, oracle, "tello_with_arms", device=0)
    N = (1 << 17) + 1
    q, yd, tau, _ = m.generateStates(N, seed=27)
    s = torch.from_numpy(masks(N, m.ncp, 3)).to(q.device)
    t_fd = dump(m, grbda.ALGO_CONTACT_FD, tmp_path / "fd.tape")
    t_im = dump(m, grbda.ALGO_CONTACT_IMPULSE, tmp_path / "im.tape")

    def check(n, qq, yy, tt, ss, got_fd, got_im, rows=None):
        rows = slice(0, n) if rows is None else rows
        qn, yn, tn, sn = _np(qq)[rows], _np(yy)[rows], _np(tt)[rows], _np(ss)[rows]
        want_fd = run_tape(t_fd, [qn, yn, packed_fd(tn, sn, eps)])
        want_im = run_tape(t_im, [qn, yn, packed_impulse(sn, 0.5, eps)])
        for g, r in zip(got_fd + got_im, want_fd + want_im):
            assert rows_rel(_np(g)[rows].reshape(r.shape[0], -1), r).max() < TOL, n

    for n in (0, 1, 127, 129, N):
        got_fd = m.contactForwardDynamics(q[:n], yd[:n], tau[:n], active=s[:n], damping=eps)
        got_im = m.contactImpulse(q[:n], yd[:n], active=s[:n], restitution=0.5, damping=eps)
        assert got_fd[0].shape == (n, m.nv) and got_im[1].shape == (n, m.ncp, 3)
        if n:
            check(n, q[:n], yd[:n], tau[:n], s[:n], got_fd, got_im, rows=None if n < N else slice(0, N, 97))
    # batch 0 launches nothing
    launches = grbda.launch_count()
    m.contactForwardDynamics(q[:0], yd[:0], tau[:0])
    assert grbda.launch_count() == launches
    m.contactForwardDynamics(q[:300], yd[:300], tau[:300])
    assert grbda.launch_count() > launches + 1
    # NULL mask == all-ones mask, bit for bit
    ones = torch.ones_like(s[:300])
    for a, b in zip(m.contactForwardDynamics(q[:300], yd[:300], tau[:300], damping=eps),
                    m.contactForwardDynamics(q[:300], yd[:300], tau[:300], active=ones, damping=eps)):
        assert torch.equal(a, b)
    for a, b in zip(m.contactImpulse(q[:300], yd[:300], restitution=0.2), m.contactImpulse(q[:300], yd[:300], active=ones,
                                                                                            restitution=0.2)):
        assert torch.equal(a, b)
    # 8-byte offsets of every input and output (the flagged-tile pass serves unaligned pointers)
    n = 300
    L = grbda.lib()
    P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    off = [torch.empty(n * k + 1, dtype=torch.float64, device=q.device)[1:].view(n, k) for k in (m.nq, m.nv, m.nv)]
    for dst, src in zip(off, (q, yd, tau)):
        dst.copy_(src[:n])
    sm = torch.empty(n * m.ncp + 1, dtype=torch.uint8, device=q.device)[1:].view(n, m.ncp)
    sm.copy_(s[:n])
    outs = [torch.empty(n * k + 1, dtype=torch.float64, device=q.device)[1:].view(n, k) for k in (m.nv, 3 * m.ncp)]
    assert L.grbda_cuda_contact_forward_dynamics_f64(m._h, *[P(t) for t in off], P(sm), eps, *[P(t) for t in outs], n,
                                                     None) == 0
    outs2 = [torch.empty(n * k + 1, dtype=torch.float64, device=q.device)[1:].view(n, k) for k in (m.nv, 3 * m.ncp)]
    assert L.grbda_cuda_contact_impulse_f64(m._h, P(off[0]), P(off[1]), P(sm), 0.5, eps, *[P(t) for t in outs2], n,
                                            None) == 0
    torch.cuda.synchronize()
    check(n, q[:n], yd[:n], tau[:n], s[:n], outs, outs2)
    # flagged tiles: whole turns beyond the fast sin/cos range on a state in tile 0 and one in tile 2
    qf = q[:n].clone()
    joint = m.clusters()[-1]["position_index"]
    for r in (5, 260):
        qf[r, joint] += 2 * np.pi * 4.0e11
    got_fd = m.contactForwardDynamics(qf, yd[:n], tau[:n], active=s[:n], damping=eps)
    got_im = m.contactImpulse(qf, yd[:n], active=s[:n], restitution=0.5, damping=eps)
    check(n, qf, yd[:n], tau[:n], s[:n], got_fd, got_im)


@pytest.mark.gpu
def test_contact_set_change_follows(grbda, oracle, torch, tmp_path):
    """setContactPoints drops the compiled contact programs: sizes and results follow the new set."""
    m, o, eps = setup(grbda, oracle, "mini_cheetah", device=0)
    B = 300
    q, yd, tau, _ = m.generateStates(B, seed=29)
    ydd4, lam4 = m.contactForwardDynamics(q, yd, tau)
    m.contactImpulse(q, yd)
    assert lam4.shape == (B, 4, 3)
    bodies, offsets = contact_points(m, "feet", 4)
    m.setContactPoints(bodies[:2], np.asarray(offsets[:2]) + 0.02)
    o.set_contact_points(bodies[:2], np.asarray(offsets[:2]) + 0.02)
    ydd, lam = m.contactForwardDynamics(q, yd, tau)
    yp, imp = m.contactImpulse(q, yd, restitution=0.1)
    assert lam.shape == (B, 2, 3) and imp.shape == (B, 2, 3)
    qn, ydn, taun = _np(q), _np(yd), _np(tau)
    s = np.ones((B, 2), dtype=np.uint8)
    kkt_reference(o, qn[:32], ydn[:32], taun[:32], s[:32], 0.0).check(_np(ydd)[:32], _np(lam)[:32], s[:32])
    kkt_reference(o, qn[:32], ydn[:32], taun[:32], s[:32], 0.0, impulse=True, restitution=0.1).check(
        _np(yp)[:32], _np(imp)[:32], s[:32])
    assert rel(_np(ydd), _np(ydd4)) > 1e-3


@pytest.mark.gpu
def test_contact_refusals(grbda, torch, monkeypatch):
    L = grbda.lib()
    fd, im = L.grbda_cuda_contact_forward_dynamics_f64, L.grbda_cuda_contact_impulse_f64
    m = grbda.ClusterTreeModel.from_robot("mini_cheetah", device=0)
    B = 8
    q, yd, tau, _ = m.generateStates(B)
    P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    out = [torch.empty_like(yd), torch.empty(B, 12, dtype=torch.float64, device=q.device)]
    assert fd(m._h, P(q), P(yd), P(tau), None, 0.0, *[P(t) for t in out], B, None) == 1  # no contact points
    with pytest.raises(grbda.GrbdaError):
        m.prepare(grbda.ALGO_CONTACT_FD)
    bodies, offsets = contact_points(m, "feet", 4)
    m.setContactPoints(bodies, offsets)
    ins = [P(t) for t in (q, yd, tau)]
    outs = [P(t) for t in out]
    assert fd(m._h, *ins, None, 0.0, *outs, B, None) == 0
    assert im(m._h, *ins[:2], None, 1.0, 0.0, *outs, B, None) == 0
    assert fd(m._h, *ins, None, 0.0, *outs, -1, None) == 1
    assert im(m._h, *ins[:2], None, 0.0, 0.0, *outs, -1, None) == 1
    assert fd(m._h, *ins, None, -1.0, *outs, B, None) == 1
    assert fd(m._h, *ins, None, float("inf"), *outs, B, None) == 1
    assert im(m._h, *ins[:2], None, 1.01, 0.0, *outs, B, None) == 1
    assert im(m._h, *ins[:2], None, 0.5, float("nan"), *outs, B, None) == 1
    for k in range(3):
        args = list(ins)
        args[k] = None
        assert fd(m._h, *args, None, 0.0, *outs, B, None) == 1
        if k < 2:
            assert im(m._h, *args[:2], None, 0.0, 0.0, *outs, B, None) == 1
    for k in range(2):
        args = list(outs)
        args[k] = None
        assert fd(m._h, *ins, None, 0.0, *args, B, None) == 1
        assert im(m._h, *ins[:2], None, 0.0, 0.0, *args, B, None) == 1
    assert fd(m._h, None, None, None, None, 0.0, None, None, 0, None) == 0  # batch 0: nothing to do
    m.prepare(grbda.ALGO_CONTACT_FD)
    m.prepare(grbda.ALGO_CONTACT_IMPULSE)
    assert m.kernel_info(grbda.ALGO_CONTACT_FD)["ready"] and m.kernel_info(grbda.ALGO_CONTACT_IMPULSE)["ready"]
    with pytest.raises(grbda.GrbdaError):
        m.prepare(grbda.ALGO_CONTACT_FD, f32=True)
    with pytest.raises(ValueError):
        m.contactForwardDynamics(q, yd, tau, active=torch.ones(B, 3, dtype=torch.bool, device=q.device))
    with pytest.raises(ValueError):
        m.contactImpulse(q, yd, active=torch.ones(B, 4, dtype=torch.float64, device=q.device))
    monkeypatch.setenv("GRBDA_JIT", "0")
    assert fd(m._h, *ins, None, 0.0, *outs, B, None) == 3  # GRBDA_ERR_NOT_COMPILED
    assert im(m._h, *ins[:2], None, 0.0, 0.0, *outs, B, None) == 3
    with pytest.raises(grbda.GrbdaError):
        m.prepare(grbda.ALGO_CONTACT_IMPULSE)
    torch.cuda.synchronize()
