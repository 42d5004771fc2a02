"""Row f-2 (SURVEY.md §8f): leg Jacobian + joint-torque epilogue.

CPU: the oracle's factored restatement of J_force_moment against a literal transcription of the
reference's expanded formulas (LegController.cpp:130-166), kept here as test data.
GPU: tau = J^T (-rBody [F;M]) fused into the solve kernel vs the oracle (double, un-narrowed inputs)."""
import numpy as np
import pytest
from numpy import cos, sin

from conftest import rel_err
from hector_simulation_b200 import scenarios


def J_literal(q, leg):
    q0, q1, q2, q3, q4 = q
    side = 1.0 if leg == 0 else -1.0
    J = np.zeros((6, 5))
    J[0, 0] = sin(q0)*(0.04*sin(q2 + q3 + q4) + 0.22*sin(q2 + q3) + 0.22*sin(q2) + 0.0135) + cos(q0)*(0.015*side + cos(q1)*(0.018*side + 0.0025) - 1.0*sin(q1)*(0.04*cos(q2 + q3 + q4) + 0.22*cos(q2 + q3) + 0.22*cos(q2)))
    J[1, 0] = sin(q0)*(0.015*side + cos(q1)*(0.018*side + 0.0025) - 1.0*sin(q1)*(0.04*cos(q2 + q3 + q4) + 0.22*cos(q2 + q3) + 0.22*cos(q2))) - 1.0*cos(q0)*(0.04*sin(q2 + q3 + q4) + 0.22*sin(q2 + q3) + 0.22*sin(q2) + 0.0135)
    J[5, 0] = 1.0
    J[0, 1] = -1.0*sin(q0)*(sin(q1)*(0.018*side + 0.0025) + cos(q1)*(0.04*cos(q2 + q3 + q4) + 0.22*cos(q2 + q3) + 0.22*cos(q2)))
    J[1, 1] = cos(q0)*(sin(q1)*(0.018*side + 0.0025) + cos(q1)*(0.04*cos(q2 + q3 + q4) + 0.22*cos(q2 + q3) + 0.22*cos(q2)))
    J[2, 1] = sin(q1)*(0.04*cos(q2 + q3 + q4) + 0.22*cos(q2 + q3) + 0.22*cos(q2)) - 1.0*cos(q1)*(0.018*side + 0.0025)
    J[3, 1], J[4, 1] = cos(q0), sin(q0)
    for k, (a, b) in enumerate([(0.22, 0.22), (0.22, 0.0), (0.0, 0.0)]):
        S = 0.04*sin(q2 + q3 + q4) + a*sin(q2 + q3) + b*sin(q2)
        C = 0.04*cos(q2 + q3 + q4) + a*cos(q2 + q3) + b*cos(q2)
        J[0, 2 + k] = sin(q0)*sin(q1)*S - 1.0*cos(q0)*C
        J[1, 2 + k] = -1.0*sin(q0)*C - 1.0*cos(q0)*sin(q1)*S
        J[2, 2 + k] = cos(q1)*S
        J[3, 2 + k], J[4, 2 + k], J[5, 2 + k] = -cos(q1)*sin(q0), cos(q0)*cos(q1), sin(q1)
    return J


def test_jacobian_restatement_matches_reference_formulas(oracle):
    rng = np.random.default_rng(1)
    for _ in range(50):
        q = rng.normal(0, 1, 5)
        for leg in (0, 1):
            assert np.abs(J_literal(q, leg) - oracle.leg_jacobian_fm(q, leg)).max() < 1e-15


def test_torque_oracle_stand_is_symmetric(oracle):
    from conftest import load_golden

    g = load_golden("cfg1_h10")
    b = scenarios.stand_inputs(10)
    tau = oracle.joint_torques(g["q_soln"][0, :12], b["rBody"], b["q_leg"], [1, 1])[0]
    # mirror-symmetric stance: sagittal joints (2,3,4) carry equal torques; the frontal joints have opposite
    # signs (not equal magnitudes: the reference's Jacobian has the side-asymmetric lever 0.018*side + 0.0025)
    assert np.allclose(tau[2:5], tau[7:10], atol=1e-4)
    assert tau[1] > 0 > tau[6]
    assert 9.0 < tau[3] < 10.0   # knee holds most of the 47.8 N per foot


@pytest.mark.gpu
def test_fused_torque_epilogue_vs_oracle(oracle):
    from conftest import qpoases_sample
    from hector_simulation_b200 import interface

    recs, inputs = scenarios.make_batch(3, 256, horizon=10, seed=31)
    mpc = interface.BatchedMPC(256, 10)
    w, tau, st = mpc.solve_batch_torques(recs)
    assert (interface.status_code(st) == 0).all()
    ref_w, rc = qpoases_sample("torques256", recs)             # qpOASES' first-step wrenches of the same records
    assert (rc == 0).all()
    rB = np.array([b["rBody"] for b in inputs])
    ql = np.array([b["q_leg"] for b in inputs])
    contact = np.array([b["gait"][:2] for b in inputs])
    ref_tau = oracle.joint_torques(ref_w[:, :12], rB, ql, contact)
    assert rel_err(tau, ref_tau).max() < 1e-4      # float-narrowed angles + wrench parity
    assert np.median(rel_err(tau, ref_tau)) < 2e-6
    assert (tau.reshape(-1, 2, 5)[contact == 0] == 0).all()   # swing legs: no feed-forward torque
    # the plain call returns the same wrench (the epilogue does not disturb the solve)
    w2, st2 = mpc.solve_batch(recs)
    assert np.array_equal(w, w2) and np.array_equal(st, st2)
    mpc.close()
