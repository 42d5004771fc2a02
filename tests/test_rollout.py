"""Row f-3 (SURVEY §8f), BASELINE config 5: the closed loop on the device (hmpc_rollout_device = prepare -> solve ->
advance per tick, no host in the loop) against (1) the numpy mirror of the advance step driven from the host and
(2) the oracle on the records the device loop logged."""
import numpy as np
import pytest

from conftest import reference_solve, rel_err
from hector_simulation_b200 import interface, scenarios
from test_state_prepare import _host_prepared

N = 10


def _walkers(n, seed=None):
    _, inputs = scenarios.make_batch(5, n, horizon=N, seed=seed)
    return scenarios.make_rollout(inputs, N)


def test_rollout_record_layout():
    d = scenarios.ROLLOUT_DTYPE
    assert d.itemsize == 80 and d.fields["gait_offset"][1] == 48 and d.fields["iteration"][1] == 64 and d.fields["ticks"][1] == 76


def test_gait_advance_matches_gait_class():
    """advance_numpy's next-tick table == Gait::mpc_gait of the advanced counter (GaitGenerator.cpp:85-103)."""
    states, loop = _walkers(6)
    zero_w, zero_s = np.zeros((6, 12 * N)), np.zeros(6, np.int32)
    zero_w[:, 2] = zero_w[:, 5] = 44.0  # hold the body up
    for t in range(1, 14):
        scenarios.advance_numpy(states, loop, zero_w, zero_s, N)
        for i in range(6):
            assert np.array_equal(states["gait"][i, : 2 * N], scenarios.walking_table(N, (i + t) % N))
    assert (loop["ticks"] == 13).all() and (loop["iteration"] == np.arange(6) + 13).all()


def test_numpy_loop_with_oracle_keeps_walkers_upright(oracle):
    """The loop semantics (plant, touch-down placement, set-point integration) with qpOASES (or, where it is not built,
    the exact fp64 referee of the same QPs) as the solver."""
    states, loop = _walkers(4)
    cmd = states["state_des"][:, 2].copy()
    x0 = states["position"][:, 0].copy()
    setup = oracle.make_setup(N)
    T = 40
    for t in range(T):
        q, info = reference_solve(oracle, _host_prepared(states, N), setup)
        assert (info[:, 0] == 0).all()
        scenarios.advance_numpy(states, loop, q, (info[:, 1].astype(np.int32) << 8), N)
    assert (np.abs(states["position"][:, 2] - 0.56) < 0.03).all() and (np.abs(states["rpy"][:, :2]) < 0.05).all()
    # the commanded forward velocity is tracked (within 30 % + 2 cm/s) over the last second
    assert (np.abs(states["vWorld"][:, 0] - cmd) < 0.3 * np.abs(cmd) + 0.02).all(), (states["vWorld"][:, 0], cmd)
    assert (np.sign(states["position"][:, 0] - x0) == np.sign(cmd)).all()


def _to_dev(a):
    import torch

    return torch.from_numpy(a.view(np.uint8).reshape(a.shape[0], -1).copy()).cuda()


@pytest.mark.gpu
def test_device_rollout_matches_host_driven_loop(oracle):
    import torch

    B, T = 96, 25
    states, loop = _walkers(B, seed=9)
    mpc = interface.BatchedMPC(B, N)
    d_states, d_loop = _to_dev(states), _to_dev(loop)
    d_wlog = torch.zeros((T, B, 12), dtype=torch.float32, device="cuda")
    d_rlog = torch.zeros((T, B, interface.record_bytes(N)), dtype=torch.uint8, device="cuda")
    mpc.rollout_device(d_states, d_loop, B, T, d_wlog, d_rlog)
    torch.cuda.synchronize()
    dev_states = d_states.cpu().numpy().view(scenarios.STATE_DTYPE).reshape(B)
    dev_loop = d_loop.cpu().numpy().view(scenarios.ROLLOUT_DTYPE).reshape(B)
    wlog, rlog = d_wlog.cpu().numpy(), d_rlog.cpu().numpy()
    assert (dev_loop["failures"] == 0).all() and (dev_loop["ticks"] == T).all()

    # (1) the same loop driven from the host: GPU solve per tick + numpy advance
    worst_w = 0.0
    for t in range(T):
        w, s = mpc.solve_batch_states(states)
        worst_w = max(worst_w, float(rel_err(wlog[t].astype(np.float64), w[:, :12], 12).max()))
        scenarios.advance_numpy(states, loop, w, s, N)
    for k in ("position", "vWorld", "omegaWorld", "rpy", "orientation", "leg_p", "world_position_desired"):
        assert np.abs(dev_states[k] - states[k]).max() < 1e-6, (k, np.abs(dev_states[k] - states[k]).max())
    assert np.array_equal(dev_states["gait"], states["gait"]) and np.array_equal(dev_loop["iteration"], loop["iteration"])
    assert np.abs(dev_loop["feet_world"] - loop["feet_world"]).max() < 1e-6
    assert worst_w < 1e-5, worst_w
    assert (np.abs(dev_states["position"][:, 2] - 0.56) < 0.03).all()

    # (2) the records the device loop logged, solved by the oracle (strided sample), against the logged wrenches
    setup = oracle.make_setup(N)
    worst = 0.0
    for t in range(0, T, 4):
        idx = np.arange(t % 8, B, 8)
        recs = interface.unpack_records(rlog[t][idx], N)
        ref, info = reference_solve(oracle, recs, setup)
        assert (info[:, 0] == 0).all()
        worst = max(worst, float(rel_err(wlog[t][idx].astype(np.float64), ref[:, :12], 12).max()))
    print("device rollout vs oracle on logged records: worst rel err %.3e; vs host-driven loop %.3e" % (worst, worst_w))
    assert worst < 1e-4, worst
    mpc.close()


@pytest.mark.gpu
def test_config5_200_ticks_on_device(oracle):
    """BASELINE configs[4]: batch 4096, 200 consecutive ticks with warm start (every tick proposes the previous tick's
    working set), and the fp32 kernel against the fp64-assembly oracle along the way (strided sample of the logged
    records of all 200 ticks)."""
    import torch

    B, T = 4096, 200
    states, loop = _walkers(B, seed=4242)
    cmd = states["state_des"][:, 2].copy()
    x0 = states["position"][:, 0].copy()
    yaw0 = states["rpy"][:, 2].copy()
    mpc = interface.BatchedMPC(B, N)
    d_states, d_loop = _to_dev(states), _to_dev(loop)
    d_wlog = torch.zeros((T, B, 12), dtype=torch.float32, device="cuda")
    d_rlog = torch.zeros((T, B, interface.record_bytes(N)), dtype=torch.uint8, device="cuda")
    mpc.rollout_device(d_states, d_loop, B, T, d_wlog, d_rlog)
    torch.cuda.synchronize()
    st = d_states.cpu().numpy().view(scenarios.STATE_DTYPE).reshape(B)
    lo = d_loop.cpu().numpy().view(scenarios.ROLLOUT_DTYPE).reshape(B)
    changes = lo["iters_total"].sum() / lo["ticks"].sum()
    print("config 5: mean working-set changes per tick (relative to the warm proposal) %.2f" % changes)
    assert changes < 6.0, changes   # cold start: ~12 rows installed per tick
    # strided sample over ALL ticks: (i) the warm-started result equals a cold solve of the same record (same optimum),
    # (ii) the contract vs qpOASES, (iii) fp32 assembly vs the fp64-assembly oracle (the reference's own rounding noise)
    tick_idx = np.arange(0, T, 8)
    rob_idx = np.arange(5, B, 257)
    sel_r = d_rlog[torch.from_numpy(tick_idx).cuda()][:, torch.from_numpy(rob_idx).cuda()].cpu().numpy()
    sel_w = d_wlog[torch.from_numpy(tick_idx).cuda()][:, torch.from_numpy(rob_idx).cuda()].cpu().numpy().astype(np.float64)
    recs = interface.unpack_records(sel_r.reshape(-1, sel_r.shape[-1]), N)
    cold = interface.BatchedMPC(len(recs), N)
    w_cold, s_cold = cold.solve_batch(recs)
    cold.close()
    wc = rel_err(sel_w.reshape(-1, 12), w_cold[:, :12], 12)
    print("config 5: warm-started loop vs cold solve of the same records: worst rel err %.3e" % wc.max())
    assert wc.max() < 1e-6   # float32 output resolution; the optimum is the same point
    setup = oracle.make_setup(N)
    ref, info = reference_solve(oracle, recs, setup)
    ok = info[:, 0] == 0
    e32 = rel_err(sel_w.reshape(-1, 12)[ok], ref[ok][:, :12], 12)
    ref64, info64 = reference_solve(oracle, recs, setup, assembly_fp64=True)
    ok64 = ok & (info64[:, 0] == 0)
    e64 = rel_err(sel_w.reshape(-1, 12)[ok64], ref64[ok64][:, :12], 12)
    print("config 5 (%d records over %d ticks): vs qpOASES worst %.3e median %.3e; fp32 kernel vs fp64-assembly oracle worst %.3e median %.3e"
          % (len(recs), len(tick_idx), e32.max(), np.median(e32), e64.max(), np.median(e64)))
    assert e32.max() < 1e-4 and np.median(e32) < 1e-5
    assert e64.max() < 2e-3 and np.median(e64) < 1e-4
    assert (lo["ticks"] == T).all() and lo["failures"].sum() == 0, lo["failures"].sum()
    assert np.isfinite(st["position"]).all()
    assert (np.abs(st["position"][:, 2] - 0.56) < 0.04).all() and (np.abs(st["rpy"][:, :2]) < 0.08).all()
    # 8 s of walking: displacement follows the velocity command
    straight = st["state_des"][:, 4] == 0
    disp = (st["position"][:, 0] - x0)[straight]
    want = cmd[straight] * T * scenarios.DT_MPC
    # the reference's weights/clamped position set-point track ~76 % of the commanded speed in steady state (the same
    # ratio with qpOASES in the loop, tests/tools/rollout_cpu_sim.py); initial-velocity transients move it by a few cm
    fast = np.abs(want) > 1.0
    ratio = disp[fast] / want[fast]
    dev = np.abs(disp - 0.76 * want)
    print("config 5: displacement/command ratio median %.3f, 1%%..99%% %.3f..%.3f, min %.3f max %.3f; |disp - 0.76 cmd T| max %.3f m"
          % (np.median(ratio), np.percentile(ratio, 1), np.percentile(ratio, 99), ratio.min(), ratio.max(), dev.max()))
    assert 0.70 < np.median(ratio) < 0.82
    assert np.percentile(ratio, 1) > 0.6 and np.percentile(ratio, 99) < 0.95
    assert ratio.min() > 0.4 and ratio.max() < 1.2 and dev.max() < 0.6   # nobody runs away or stalls
    # commanded yaw rate: followed at ~68 % (same with qpOASES in the loop)
    yr = st["state_des"][~straight, 4]
    sel = np.abs(yr) > 0.1
    yaw_ratio = ((st["rpy"][:, 2] - yaw0)[~straight] / (T * scenarios.DT_MPC))[sel] / yr[sel]
    print("config 5: yaw-rate tracking ratio %.3f..%.3f" % (yaw_ratio.min(), yaw_ratio.max()))
    assert yaw_ratio.min() > 0.5 and yaw_ratio.max() < 0.9
    mpc.close()
