"""CPU tests of the oracle itself (no GPU): pin it against the reference's known answers and
restate the reference's cross-implementation property tests."""
import json
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
KAT = json.load(open(os.path.join(HERE, "golden", "codegen_kat.json")))
ROBOTS = ["mini_cheetah", "mit_humanoid", "tello", "tello_with_arms",
          "revolute_chain_with_rotor_4", "revolute_pair_chain_with_rotor_4"]


def rel(a, b):
    return np.abs(a - b).max() / max(1e-300, np.abs(b).max())


@pytest.mark.parametrize("case", KAT["cases"], ids=lambda c: c["robot"])
@pytest.mark.parametrize("suffix", ["", ":generic"])
def test_oracle_matches_reference_generated_dynamics(oracle, case, suffix):
    """Golden vectors produced by the reference's own CasADi-generated Lagrangian dynamics
    (reference test: UnitTests/testReflectedInertiaAlgos.cpp:144-222, tol 1e-5; here 1e-11)."""
    m = oracle.OracleModel(case["robot"] + suffix)
    for s in case["states"]:
        y, yd, tau = (np.array(s[k])[None, :] for k in ("y", "yd", "tau"))
        ydd_ref = np.array(s["ydd_fwd"])[None, :]
        ydd = m.forward_dynamics(y, yd, tau, threads=1)
        assert rel(ydd, ydd_ref) < 1e-11
        tau_ref = np.array(s["tau_inv_of_ydd"])[None, :]
        assert rel(m.inverse_dynamics(y, yd, ydd_ref, threads=1), tau_ref) < 1e-11


def test_appendix_d_vectors(oracle):
    """SURVEY Appendix D: values obtained by running the reference's generated C."""
    m = oracle.OracleModel("revolute_chain_with_rotor_2")
    ydd = m.forward_dynamics(np.array([[0.3, -0.2]]), np.array([[0.1, 0.4]]), np.array([[1.0, -0.5]]))
    assert np.allclose(ydd[0], [-1.20437344732216, 0.883601589583859], rtol=0, atol=1e-12)
    m = oracle.OracleModel("revolute_pair_chain_with_rotor_4")
    ydd = m.forward_dynamics(np.array([[0.3, -0.2, 0.5, -0.7]]), np.array([[0.1, 0.4, -0.3, 0.2]]),
                             np.array([[1.0, -0.5, 0.25, 0.75]]))
    assert np.allclose(ydd[0], [-1.95721149070437, 3.81858808738384, -6.10723858523103, 6.55749123258841],
                       rtol=0, atol=1e-11)


@pytest.mark.parametrize("robot", ROBOTS)
def test_reference_property_tests(oracle, robot):
    """UnitTests/testRigidBodyDynamicsAlgos.cpp:113-239 restated: cluster model = Generic re-build,
    ID(FD(tau)) = tau, H symmetric positive definite, H ydd + C = tau."""
    m, g = oracle.OracleModel(robot), oracle.OracleModel(robot + ":generic")
    B = 20
    q, yd, tau = m.generate_states(B, seed=11)
    assert m.validate_states(q).all()
    ydd = m.forward_dynamics(q, yd, tau)
    assert rel(g.forward_dynamics(q, yd, tau), ydd) < 5e-8
    assert rel(m.inverse_dynamics(q, yd, ydd), tau) < 5e-8
    H = m.mass_matrix(q)
    assert rel(g.mass_matrix(q), H) < 5e-8
    assert np.abs(H - H.transpose(0, 2, 1)).max() < 1e-12
    assert np.linalg.eigvalsh(H).min() > 0
    C = m.inverse_dynamics(q, yd, np.zeros_like(yd))
    assert rel(g.inverse_dynamics(q, yd, np.zeros_like(yd)), C) < 5e-8
    assert rel(np.einsum("bij,bj->bi", H, ydd) + C, tau) < 5e-8


@pytest.mark.parametrize("robot", ["tello", "mit_humanoid"])
def test_external_forces_round_trip(oracle, robot):
    """ForwardAndInverseDynamics with random spatial forces on every body (:201-236)."""
    m = oracle.OracleModel(robot)
    q, yd, tau = m.generate_states(8, seed=3)
    f = np.random.default_rng(0).uniform(-1, 1, (8, m.nb, 6))
    ydd = m.dynamics_with_external_forces(q, yd, tau, f, forward=True)
    assert rel(m.dynamics_with_external_forces(q, yd, ydd, f, forward=False), tau) < 5e-8
    assert rel(ydd, m.forward_dynamics(q, yd, tau)) > 1e-3  # the forces do act


@pytest.mark.parametrize("robot", ["tello", "tello_with_arms"])
def test_implicit_constraint_identities(oracle, robot):
    """UnitTests/testLoopConstraints.cpp:286-341: K G = 0 and K g = k for GenericImplicit."""
    m = oracle.OracleModel(robot)
    q, yd, _ = m.generate_states(10, seed=5)
    for c, info in enumerate(m.clusters()):
        if not info["implicit"]:
            continue
        for b in range(q.shape[0]):
            G, K, g, k = m.cluster_constraint(c, q[b], yd[b])
            assert np.abs(K @ G).max() < 1e-10
            assert np.abs(K @ g - k).max() < 1e-10


def test_state_generator_is_index_keyed(oracle):
    """Shards are reproducible regardless of how the index range is split."""
    m = oracle.OracleModel("tello")
    q, yd, aux = m.generate_states(16, seed=9)
    q2, yd2, aux2 = m.generate_states(8, seed=9, first_index=8)
    assert np.array_equal(q[8:], q2) and np.array_equal(yd[8:], yd2) and np.array_equal(aux[8:], aux2)
    assert np.abs(np.linalg.norm(q[:, 3:7], axis=1) - 1).max() < 1e-12  # rpyToQuat gives unit quaternions
    assert np.abs(yd).max() <= 1.0 and np.abs(aux).max() <= 1.0
