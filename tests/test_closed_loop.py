"""BASELINE config 5 (scaled for test time): consecutive MPC ticks in closed loop.

Each robot's single rigid body is integrated with the same forward-Euler model the MPC predicts with
(SolverMPC.cpp:145-146, 312-331: x+ = x + dt (A x + B u), feet pinned in the world), the first-step wrench of
every tick is fed back, the gait table advances one segment per tick, and every tick's GPU result is checked
against the oracle on a strided sample.  Like the reference, every tick is a cold start (there is no warm start
in SolverMPC.cpp); the fp64-assembly oracle quantifies what fp32 assembly costs along the trajectory."""
import numpy as np
import pytest

from conftest import reference_solve, rel_err
from hector_simulation_b200 import interface, scenarios

pytestmark = pytest.mark.gpu

I_BODY = np.diag([0.5413, 0.5200, 0.0691])  # RobotState.cpp:45
MASS = 9.0                                   # SolverMPC.cpp:423


def _step(state, u0, feet, dt):
    """One Euler step of the SRBD the MPC uses: state = (rpy, p, w, v)."""
    rpy, p, w, v = state
    R = scenarios.quat_to_R(scenarios.rpy_to_quat(rpy))
    cy, sy, cp, sp = np.cos(rpy[2]), np.sin(rpy[2]), np.cos(rpy[1]), np.sin(rpy[1])
    E = np.array([[cy * cp, -sy, 0], [sy * cp, cy, 0], [-sp, 0, 1]])
    Iw_inv = np.linalg.inv(R @ I_BODY @ R.T)
    F = [u0[0:3], u0[3:6]]
    M = [u0[6:9], u0[9:12]]
    torque = sum(np.cross(feet[i] - p, F[i]) + M[i] for i in range(2))
    force = F[0] + F[1]
    return (rpy + dt * np.linalg.solve(E, w), p + dt * v, w + dt * Iw_inv @ torque,
            v + dt * (force / MASS + np.array([0, 0, -9.81])))


def test_closed_loop_ticks_match_oracle(oracle):
    from oracle import qp_dual_active_set as G

    # The harness has no swing-leg foot placement (out of scope), so single-support robots tip over after
    # ~0.6 s; the loop is run for the 12 ticks (0.48 s) in which every robot is still upright.
    N, B, T = 10, 192, 12
    rng = np.random.default_rng(505)
    setup = oracle.make_setup(N)
    mpc = interface.BatchedMPC(B, N)
    states, feet, joints, phase = [], [], [], []
    for i in range(B):
        b = scenarios._random_state(rng, N, scenarios.walking_table(N, i % N), moving=True)
        rpy = scenarios.quat_to_rpy(b["q"])
        states.append((rpy, b["p"].copy(), b["w"].copy() * 0.2, b["v"].copy() * 0.2))
        feet.append(b["p_foot"].copy())
        joints.append(rng.normal(0, 0.05, 10))
        phase.append(i % N)
    worst, worst64, refereed = 0.0, 0.0, 0
    recs = np.zeros(B, dtype=scenarios.UPDATE_DTYPE)
    for t in range(T):
        for i in range(B):
            rpy, p, w, v = states[i]
            table = scenarios.standing_table(N) if i % 4 == 0 else scenarios.walking_table(N, (phase[i] + t) % N)
            b = scenarios.boundary_inputs(p, rpy, v, w, joints[i], table, N, feet_world=feet[i])
            scenarios.to_record(b, N, recs[i])
        wrench, status = mpc.solve_batch(recs)
        assert (interface.status_code(status) == 0).all(), (t, np.bincount(interface.status_code(status)))
        idx = np.arange(t % 4, B, 4)
        ref, info = reference_solve(oracle, recs[idx], setup)
        assert (info[:, 0] == 0).all()
        e = rel_err(wrench[idx], ref, 12)
        worst = max(worst, float(e.max()))
        # where the two solvers differ by more than 2e-5, a tight-tolerance fp64 referee decides who is off:
        # qpOASES stops at a homotopy tolerance of 2.2e-7 (Options.cpp:206) and loses digits near degenerate
        # optima (a foot unloading); the GPU result must sit on the referee's optimum
        for k in np.nonzero(e > 2e-5)[0][:2]:
            Q = oracle.reduced_qp(recs[idx[k]], setup)
            x, inf = G.solve(Q["H"], Q["g"], Q["A"], Q["lb"], Q["ub"], tol=1e-12)
            full = np.zeros(12 * N)
            full[Q["var_ind"]] = x
            assert inf["status"] == 0
            assert rel_err(wrench[idx[k]][None], full[None], 12)[0] < 2e-6
            refereed += 1
        if t % 6 == 0:
            ref64, _ = reference_solve(oracle, recs[idx], setup, assembly_fp64=True)
            worst64 = max(worst64, float(rel_err(wrench[idx], ref64, 12).max()))
        for i in range(B):
            states[i] = _step(states[i], wrench[i, :12], feet[i], scenarios.DT_MPC)
    heights = np.array([s[1][2] for s in states])
    print("closed loop: worst rel err vs qpOASES %.3e (refereed cases: %d), vs fp64-assembly oracle %.3e, heights %.3f..%.3f"
          % (worst, refereed, worst64, heights.min(), heights.max()))
    assert worst < 1e-4, worst                  # the contract, every tick; median is ~1e-7
    assert worst64 < 2e-3, worst64              # fp32-vs-fp64 assembly: the reference's own rounding noise, reported
    assert np.isfinite(heights).all() and heights.min() > 0.45 and heights.max() < 0.65  # bodies still up
    mpc.close()
