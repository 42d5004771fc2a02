"""GPU (-m gpu): parity of the CUDA path, called through the C-ABI, with the oracle.

Bars:  formulation stage (H, g, constraint rows, bounds) — BIT-EXACT against the oracle's fp32 restatement;
       optimal wrenches — within 1e-4 relative of the reference's qpOASES output (BASELINE.json north_star),
       asserted at 5e-5 to keep a margin; eliminated (swing) entries exactly 0.
Nothing here reads /root/reference: the oracle is the prebuilt oracle/_ref/*.so or the committed fixtures.
"""
import os

import numpy as np
import pytest

from conftest import load_golden, qpoases_sample, reference_solve, rel_err
from hector_simulation_b200 import interface, scenarios

pytestmark = pytest.mark.gpu

TOL = 5e-5  # asserted; the contract is 1e-4


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a B200"
    return torch


def _solve(records, N, strict=True):
    mpc = interface.BatchedMPC(max(len(records), 1), N)
    try:
        return mpc.solve_batch(records, strict=strict)
    finally:
        mpc.close()


@pytest.mark.parametrize("name", ["cfg1_h10", "cfg2_h10", "cfg3_h10", "cfg4_h5", "cfg4_h16"])
def test_wrench_matches_golden_qpoases(torch_cuda, name):
    g = load_golden(name)
    N = g["horizon"]
    w, st = _solve(g["records"], N)
    assert (interface.status_code(st) == 0).all()
    assert rel_err(w, g["q_soln"], 12).max() < TOL          # first-step wrench: what the caller uses
    # whole horizon; the N=16 extension config (cond(H) ~ 1.5e7, outside the reference's N=10 regime) is
    # held to the 1e-4 contract itself rather than to the tighter internal margin
    assert rel_err(w, g["q_soln"]).max() < (TOL if N <= 10 else 1e-4)
    assert (w[g["q_soln"] == 0.0] == 0.0).all()             # eliminated variables are exactly 0
    # the plain dual iteration (block start off) and qpOASES both start from an empty working set and add one row per
    # change: on non-degenerate problems the counts coincide (the symmetric stand sits exactly on the Mx >= 0 rows, where
    # the two feasibility tolerances differ, so it is excluded) — and the block start lands on the same point
    if len(st) > 1:
        os.environ["HMPC_BLOCK_ROUNDS"] = "0"
        try:
            w1, st1 = _solve(g["records"], N)
        finally:
            del os.environ["HMPC_BLOCK_ROUNDS"]
        assert np.median(np.abs(interface.status_iters(st1).astype(int) - g["info"][:, 1])) == 0
        assert rel_err(w1, w).max() < 1e-6


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3"])
def test_wrench_vs_compiled_reference_vectors(torch_cuda, name):
    """Against outputs of the reference's OWN formulation sources (SolverMPC.cpp & co. compiled unchanged against
    oracle/eigen_shim + its qpOASES; tests/golden/make_ref_compiled.py).  The reference's TU evaluates its trig with
    libm's float functions, the kernel reproduces the canonical double-trig restatement, so this comparison carries
    last-bit trig effects on top of the solver tolerances: held to the 1e-4 contract itself (CPU-side prediction with an
    fp64 referee on the canonical QP: 2.3e-5 worst on these records)."""
    import os

    from conftest import GOLDEN

    z = np.load(os.path.join(GOLDEN, "ref_compiled_h10.npz"))
    g = load_golden(name + "_h10")
    q_ref = z[name + "_q"]
    w, st = _solve(g["records"], 10)
    assert (interface.status_code(st) == 0).all()
    assert rel_err(w, q_ref, 12).max() < 1e-4
    assert rel_err(w, q_ref).max() < 1e-4
    assert (w[q_ref == 0.0] == 0.0).all()


@pytest.mark.parametrize("name", ["cfg2_h10", "cfg3_h10", "cfg4_h5", "cfg4_h16"])
def test_formulation_is_bit_exact(torch_cuda, name):
    torch = torch_cuda
    g = load_golden(name)
    N = g["horizon"]
    nf = g["H"].shape[0]
    mpc = interface.BatchedMPC(nf, N)
    packed = torch.from_numpy(interface.pack_records(g["records"][:nf], N)).cuda()
    out = mpc.assemble_device(packed, nf)
    torch.cuda.synchronize()
    iu = np.triu_indices(12 * N)
    for i in range(nf):
        H = out["H"][i].cpu().numpy()
        assert np.array_equal(H[iu].view(np.uint32), g["H"][i][iu].view(np.uint32))  # the triangle the solver uses
        assert np.array_equal(H, H.T)
        for k in ("g", "lb", "ub"):
            assert np.array_equal(out[k][i].cpu().numpy().view(np.uint32), g[k][i].view(np.uint32)), k
        assert np.array_equal(out["Fblk"][i].cpu().numpy().view(np.uint32), g["Fblk"][i].view(np.uint32))
    mpc.close()


def test_formulation_bit_exact_vs_live_oracle_many(torch_cuda, oracle):
    """256 fresh random states (not in the fixtures): H upper triangle, g, rows all bit-identical."""
    torch = torch_cuda
    N = 10
    recs, _ = scenarios.make_batch(3, 256, horizon=N, seed=777)
    mpc = interface.BatchedMPC(256, N)
    packed = torch.from_numpy(interface.pack_records(recs, N)).cuda()
    out = mpc.assemble_device(packed, 256)
    H, gg, F = out["H"].cpu().numpy(), out["g"].cpu().numpy(), out["Fblk"].cpu().numpy()
    setup = oracle.make_setup(N)
    iu = np.triu_indices(12 * N)
    ndiff = 0
    for i in range(256):
        f = oracle.formulate_f32(recs[i], setup)
        ndiff += int((H[i][iu].view(np.uint32) != f["H"][iu].view(np.uint32)).sum())
        ndiff += int((gg[i].view(np.uint32) != f["g"].view(np.uint32)).sum())
        ndiff += int((F[i].view(np.uint32) != f["Fblk"].view(np.uint32)).sum())
    assert ndiff == 0
    mpc.close()


def test_reference_boundary_single_robot(torch_cuda):
    """setup_problem / update_problem_data / get_solution exactly as ConvexMPCLocomotion.cpp:410-430 calls them."""
    g = load_golden("cfg1_h10")
    b = scenarios.stand_inputs(10)
    interface.setup_problem(scenarios.DT_MPC, 10, scenarios.MU_PASSED, scenarios.F_MAX)
    interface.update_solver_settings(500, 1e-7, 1e-8, 1.5, 1e-7, 0.0)
    interface.update_problem_data(b["p"], b["v"], b["q"], b["w"], b["r"], b["joint_angles"], b["yaw"], b["weights"],
                                  b["state_trajectory"], b["Alpha_K"], b["gait"])
    sol = np.array([interface.get_solution(i) for i in range(120)])
    assert rel_err(sol[None], g["q_soln"][:1], 12)[0] < TOL
    assert interface.status_code(interface.reference_last_status()) == 0
    # a second tick with a walking table re-solves in place (setup_problem is called every tick, :410)
    g2 = load_golden("cfg2_h10")
    recs2, inputs2 = scenarios.make_batch(2, 3, horizon=10)
    b2 = inputs2[2]
    interface.setup_problem(scenarios.DT_MPC, 10, scenarios.MU_PASSED, scenarios.F_MAX)
    interface.update_problem_data(b2["p"], b2["v"], b2["q"], b2["w"], b2["r"], b2["joint_angles"], b2["yaw"], b2["weights"],
                                  b2["state_trajectory"], b2["Alpha_K"], b2["gait"])
    sol2 = np.array([interface.get_solution(i) for i in range(120)])
    assert rel_err(sol2[None], g2["q_soln"][2:3])[0] < TOL
    leg_swing = 1 if b2["gait"][0] == 1 else 0
    assert all(sol2[3 * leg_swing + c] == 0.0 and sol2[6 + 3 * leg_swing + c] == 0.0 for c in range(3))


def test_full_size_configs_vs_live_oracle(torch_cuda):
    """BASELINE configs[1] (B=1024 walking) in full; configs[2] (B=8192 mixed) on a strided sample, against qpOASES'
    recorded optimum of the same seeded inputs."""
    recs, _ = scenarios.make_batch(2, 1024, horizon=10)
    w, st = _solve(recs, 10)
    ref, _ = qpoases_sample("full_cfg2", recs)
    assert (interface.status_code(st) == 0).all()
    e = rel_err(w, ref, 12)
    assert e.max() < TOL and np.median(e) < 1e-6
    recs3, _ = scenarios.make_batch(3, 8192, horizon=10)
    w3, st3 = _solve(recs3, 10)
    assert (interface.status_code(st3) == 0).all()
    idx = np.arange(0, 8192, 16)
    ref3, _ = qpoases_sample("full_cfg3", recs3[idx])
    assert rel_err(w3[idx], ref3, 12).max() < TOL
    assert rel_err(w3[idx], ref3).max() < TOL


def test_kkt_residuals_at_full_size(torch_cuda, oracle):
    """Size-independent property: every returned point is a KKT point of its own QP (fp64 check on the
    oracle's restated QP data): primal feasible, and the gradient lies in the cone of active rows."""
    recs, _ = scenarios.make_batch(3, 2048, horizon=10, seed=4242)
    w, st = _solve(recs, 10)
    assert (interface.status_code(st) == 0).all()
    setup = oracle.make_setup(10)
    for i in range(0, 2048, 64):
        Q = oracle.reduced_qp(recs[i], setup)
        x = w[i][Q["var_ind"]]
        Ax = Q["A"] @ x
        scale = max(1.0, np.abs(x).max())
        tol = 2e-5 * scale  # fp32 output rounding of ~100 N forces
        assert (Ax >= Q["lb"] - tol).all() and (Ax <= Q["ub"] + tol).all()
        Hs = np.triu(Q["H"]) + np.triu(Q["H"], 1).T
        grad = Hs @ x + Q["g"]
        lo = np.abs(Ax - Q["lb"]) < tol
        hi = np.abs(Ax - Q["ub"]) < tol
        rows = np.concatenate([Q["A"][lo], -Q["A"][hi]])
        if len(rows):
            from scipy.optimize import nnls

            lam, rn = nnls(rows.T, grad)
        else:
            rn = np.linalg.norm(grad)
        assert rn <= 2e-3 * max(1.0, np.linalg.norm(Q["g"]))


def test_determinism_and_batch_permutation(torch_cuda):
    recs, _ = scenarios.make_batch(3, 300, horizon=10, seed=99)
    w1, s1 = _solve(recs, 10)
    w2, s2 = _solve(recs, 10)
    assert np.array_equal(w1, w2) and np.array_equal(s1, s2)
    perm = np.random.default_rng(0).permutation(300)
    w3, s3 = _solve(recs[perm], 10)
    assert np.array_equal(w3, w1[perm]) and np.array_equal(s3, s1[perm])


def test_edge_cases(torch_cuda):
    N = 10
    mpc = interface.BatchedMPC(64, N)
    # empty batch
    w, s = mpc.solve_batch(np.zeros(0, dtype=scenarios.UPDATE_DTYPE))
    assert w.shape == (0, 120)
    # a robot with no foot in contact over the whole horizon: everything eliminated -> all zeros
    b = scenarios.stand_inputs(N)
    b["gait"][:] = 0
    rec = scenarios.to_record(b, N)
    w, s = mpc.solve_batch(np.array([rec]))
    assert (w == 0).all() and interface.status_code(s)[0] == 0
    # flight for the first steps, then double support (ragged contact schedule)
    b = scenarios.stand_inputs(N)
    b["gait"][:8] = 0
    rec = scenarios.to_record(b, N)
    w, s = mpc.solve_batch(np.array([rec]))
    assert interface.status_code(s)[0] == 0 and (w[0, :48] == 0).all() and np.abs(w[0, 48:]).max() > 1
    # batch larger than the context's capacity is refused, not truncated
    recs, _ = scenarios.make_batch(2, 65, horizon=N)
    with pytest.raises(interface.HmpcError):
        mpc.solve_batch(recs)
    mpc.close()


def test_edge_cases_vs_oracle(torch_cuda):
    N = 10
    rng = np.random.default_rng(5)
    recs = []
    for k in range(48):
        table = (rng.random(2 * N) < 0.6).astype(np.int32)  # arbitrary ragged contact schedules
        b = scenarios._random_state(rng, N, table, moving=True)
        recs.append(scenarios.to_record(b, N))
    recs = np.array(recs)
    w, s = _solve(recs, N)
    ref, rc = qpoases_sample("ragged48", recs)
    assert (interface.status_code(s) == 0).all() and (rc == 0).all()
    assert rel_err(w, ref).max() < TOL
    assert (w[ref == 0.0] == 0.0).all()


def test_device_resident_path_and_status_words(torch_cuda):
    torch = torch_cuda
    g = load_golden("cfg3_h10")
    N = 10
    B = len(g["records"])
    mpc = interface.BatchedMPC(B, N)
    assert mpc.launches_per_solve >= 1
    packed = torch.from_numpy(interface.pack_records(g["records"], N)).cuda()
    d_w = torch.full((B, 12 * N), float("nan"), dtype=torch.float32, device="cuda")
    d_s = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    mpc.solve_device(packed, B, d_w, d_s)
    torch.cuda.synchronize()
    w, s = d_w.cpu().numpy().astype(np.float64), d_s.cpu().numpy()
    assert np.isfinite(w).all() and (s >= 0).all()      # every slot written: never silently stale
    assert rel_err(w, g["q_soln"]).max() < TOL
    assert (interface.status_nactive(s) <= interface.status_iters(s)).all()
    mpc.close()


def test_massively_degenerate_optimum_escalates_and_converges(torch_cuda):
    """A falling robot whose optimal contact forces are all zero: ~100 active rows on 120 variables.  The working
    set outgrows class 1's capacity; the kernel hands the robot to the full-capacity class and still returns
    a KKT point (status 0), matching qpOASES (which needs 163 working-set changes) in absolute terms."""
    g = load_golden("degenerate_zero_force_h10")
    w, st = _solve(g["records"], 10)
    assert (interface.status_code(st) == 0).all(), st
    assert interface.status_nactive(st).max() > 64          # really beyond the regular working-set capacity
    # moments ~0.6 N m, forces ~0: absolute comparison.  qpOASES' own point is 2e-3 off in one moment component
    # (a tight fp64 referee, stored in the fixture, reaches a lower objective); the GPU sits on the referee's optimum
    assert np.abs(w - g["q_soln"]).max() < 5e-3
    assert np.abs(w - g["q_referee"]).max() < 2e-5
    assert np.abs(w[:, :6]).max() < 1e-3                    # first-step forces are (numerically) zero


def test_stress_large_perturbations_all_converge(torch_cuda, oracle):
    """8192 robots with 3x the nominal state scatter (rpy 0.15 rad, v 0.3 m/s, w 0.6 rad/s, joints 0.15 rad) and random
    ragged contact schedules: every instance must end in a KKT point (status 0, never an iteration cap or an
    'infeasible' verdict — the QP always has the feasible point u = 0), and a sample must match qpOASES."""
    N, B = 10, 8192
    rng = np.random.default_rng(9001)
    recs = np.zeros(B, dtype=scenarios.UPDATE_DTYPE)
    for i in range(B):
        kind = i % 3
        if kind == 0:
            table = scenarios.walking_table(N, int(rng.integers(0, N)))
        elif kind == 1:
            table = scenarios.standing_table(N)
        else:
            table = (rng.random(2 * N) < 0.7).astype(np.int32)
        rpy = rng.normal(0.0, 0.15, 3)
        pos = np.array([0.0, 0.0, scenarios.BODY_HEIGHT]) + rng.normal(0.0, 0.06, 3)
        vx = rng.uniform(-1.0, 1.0)
        b = scenarios.boundary_inputs(pos, rpy, rng.normal(0, 0.3, 3) + [vx, 0, 0], rng.normal(0, 0.6, 3), rng.normal(0, 0.15, 10),
                                      table, N, v_des_body=(vx, 0.0), yaw_rate=rng.uniform(-0.5, 0.5), pos_des_err=rng.normal(0, 0.05, 2))
        scenarios.to_record(b, N, recs[i])
    w, st = _solve(recs, N, strict=False)
    codes = np.bincount(interface.status_code(st), minlength=5)
    assert codes[1:].sum() == 0, codes
    assert np.isfinite(w).all()
    from oracle import qp_dual_active_set as G

    idx = np.arange(0, B, 32)
    setup = oracle.make_setup(N)
    ref, info = reference_solve(oracle, recs[idx], setup)
    good = info[:, 0] == 0
    e0, ef = rel_err(w[idx], ref, 12), rel_err(w[idx], ref)
    assert e0[good].max() < 1e-4 and np.median(e0[good]) < 1e-5   # first-step wrench: the contract
    # whole horizon: far from the nominal regime qpOASES itself is up to ~1e-4 away from the exact optimum
    # (termination tolerance 2.2e-7 in homotopy length); the three largest gaps are refereed in fp64
    for k in np.argsort(-np.where(good, ef, 0))[:3]:
        Q = oracle.reduced_qp(recs[idx[k]], setup)
        x, inf = G.solve(Q["H"], Q["g"], Q["A"], Q["lb"], Q["ub"], tol=1e-12, max_iter=3000)
        full = np.zeros(12 * N)
        full[Q["var_ind"]] = x
        assert inf["status"] == 0 and rel_err(w[idx[k]][None], full[None])[0] < 1e-6
    assert ef[good].max() < 3e-4


def test_in_place_mode_equals_staged_path():
    """hmpc_pin_host_buffer: records read in place from the caller's update_data_t array, double results written in
    place — the same solve as the staged (pack + copy + widen) path at every horizon, mixed size classes: status words
    identical, and the in-place doubles (the fp64 solve's own bits) round to exactly the staged path's floats."""
    for horizon, cfg, B in ((10, 3, 700), (5, 4, 64), (16, 4, 48), (10, 1, 1)):
        recs, _ = scenarios.make_batch(cfg, B, horizon=horizon, seed=31 + horizon)
        mpc = interface.BatchedMPC(B, horizon)
        w_ref, s_ref = mpc.solve_batch(recs)                      # staged: nothing pinned yet
        staged, recs = recs, interface.page_aligned(recs.shape, recs.dtype)   # registered arrays own their pages
        recs[...] = staged
        w = interface.page_aligned((B, 12 * horizon), np.float64)
        s = interface.page_aligned(B, np.int32)
        w[...] = np.nan
        s[...] = -1
        mpc.pin(recs, w, s)
        mpc.solve_batch(recs, out=(w, s))
        assert np.array_equal(s, s_ref) and np.array_equal(w.astype(np.float32), w_ref.astype(np.float32)), (horizon, np.abs(w - w_ref).max())
        # a second tick with changed records in the same buffers (what a control loop does)
        recs2, _ = scenarios.make_batch(cfg, B, horizon=horizon, seed=77)
        recs[:] = recs2
        mpc.solve_batch(recs, out=(w, s))
        mpc.unpin(recs, w, s)
        w2, s2 = mpc.solve_batch(recs2)
        assert np.array_equal(s, s2) and np.array_equal(w.astype(np.float32), w2.astype(np.float32))
        mpc.close()


def test_in_place_mode_escalates_on_the_device():
    """A working-set overflow in the in-place mode: the chain (class 0 classifies -> class 1 -> class 2) escalates on the
    device, and the doubles written in place round to the staged path's floats."""
    g = load_golden("degenerate_zero_force_h10")
    recs = np.ascontiguousarray(np.repeat(g["records"].view(scenarios.UPDATE_DTYPE).reshape(-1)[:1], 3))
    mpc = interface.BatchedMPC(3, 10)
    w_ref, s_ref = mpc.solve_batch(recs)
    staged, recs = recs, interface.page_aligned(recs.shape, recs.dtype)
    recs[...] = staged
    w = interface.page_aligned(w_ref.shape, w_ref.dtype)
    s = interface.page_aligned(s_ref.shape, s_ref.dtype)
    mpc.pin(recs, w, s)
    mpc.solve_batch(recs, out=(w, s))
    assert (interface.status_code(s) == 0).all() and np.array_equal(w.astype(np.float32), w_ref.astype(np.float32))
    assert interface.status_nactive(s).max() > 64
    mpc.close()


def test_contexts_of_different_horizons_coexist(torch_cuda):
    """The runtime-horizon kernel instantiations are shared by every context of the process, and their dynamic
    shared-memory attribute is process-wide: a horizon-8 context created after a horizon-10 one (and the reference-style
    global context) must not lower it under the others' launches.  Also: a misaligned device record pointer is an
    argument error, not a device fault."""
    torch = torch_cuda
    ctx = {}
    for N in (10, 8, 16, 5):  # created in this order, all alive together
        recs, _ = scenarios.make_batch(3, 96, horizon=N, seed=700 + N)
        ctx[N] = (interface.BatchedMPC(96, N), recs)
    b = scenarios.stand_inputs(10)
    interface.setup_problem(scenarios.DT_MPC, 10, scenarios.MU_PASSED, scenarios.F_MAX)   # the global one-robot context too
    for _ in range(2):
        for N, (mpc, recs) in ctx.items():
            packed = torch.from_numpy(interface.pack_records(recs, N)).cuda()
            d_w = torch.zeros((96, 12 * N), dtype=torch.float32, device="cuda")
            d_s = torch.full((96,), -1, dtype=torch.int32, device="cuda")
            mpc.solve_device(packed, 96, d_w, d_s)
            torch.cuda.synchronize()
            assert (interface.status_code(d_s.cpu().numpy()) == 0).all(), N
            w, s = mpc.solve_batch(recs)
            assert rel_err(d_w.cpu().numpy().astype(np.float64), w).max() < 1e-6
        interface.update_problem_data(b["p"], b["v"], b["q"], b["w"], b["r"], b["joint_angles"], b["yaw"], b["weights"],
                                      b["state_trajectory"], b["Alpha_K"], b["gait"])
        assert abs(interface.get_solution(2) - 47.84) < 0.05
    mpc, recs = ctx[10]
    raw = torch.zeros(96 * interface.record_bytes(10) + 64, dtype=torch.uint8, device="cuda")
    view = raw[8: 8 + 96 * interface.record_bytes(10)].view(96, -1)     # 8 bytes off: not 16-byte aligned
    d_w = torch.zeros((96, 120), dtype=torch.float32, device="cuda")
    d_s = torch.zeros((96,), dtype=torch.int32, device="cuda")
    with pytest.raises(interface.HmpcError, match="16-byte aligned"):
        mpc.solve_device(view, 96, d_w, d_s)
    for mpc, _ in ctx.values():
        mpc.close()


def test_sharded_entry_points_single_rank(torch_cuda):
    """hmpc_shard_* with a one-rank group: the slice comes back on the caller's arrays like hmpc_solve_batch, and the
    (here trivial) ncclAllGather delivers the float wrenches to the device buffer, tick after tick (double-buffered)."""
    torch = torch_cuda
    from hector_simulation_b200 import sharding

    N, B = 10, 200
    recs, _ = scenarios.make_batch(3, B, horizon=N, seed=77)
    ref = interface.BatchedMPC(B, N)
    w_ref, s_ref = ref.solve_batch(recs)
    ref.close()
    sh = sharding.ShardedMPC(B, N, 0, 1, lambda bl: sharding.GpuBackend(bl, N, 0, 1, 0, lambda b: b), scenarios.UPDATE_DTYPE)
    for tick in range(3):
        w, s = sh.tick(recs, gather=False)
        sh.backend.solve(sh.recs, sh.out_w, sh.out_s, True)     # the gather path itself (world == 1 skips it in tick())
        torch.cuda.synchronize()
        assert np.array_equal(s, s_ref) and np.array_equal(w.astype(np.float32), w_ref.astype(np.float32))
        g = sh.backend.gathered()
        assert np.array_equal(g, w_ref.astype(np.float32))
    sh.close()


@pytest.mark.parametrize("N", [5, 10, 16])
def test_horizon_sweep_batch_4096(torch_cuda, oracle, N):
    """BASELINE configs[3] (N = 20 is refused, like horizons above 19 by the reference): 4096 mixed robots per horizon, every
    instance converges, and on a strided sample
      * the first-step wrench (what the caller uses) is inside the 1e-4 contract against qpOASES;
      * the whole horizon is held to 1e-4 too, EXCEPT where a tight-tolerance fp64 referee shows that qpOASES itself is the
        party that is off (its termination tolerance is 2.2e-7 in homotopy length, Options.cpp:206, and the N = 16 Hessians
        have cond ~1.5e7): every such case is adjudicated here — the GPU result must sit on the referee's optimum (1e-6) —
        and even then the gap to qpOASES stays below 3e-4."""
    B = 4096
    recs, _ = scenarios.make_batch(4, B, horizon=N, seed=1000 + N)
    mpc = interface.BatchedMPC(B, N)
    w, st = mpc.solve_batch(recs, strict=False)
    mpc.close()
    assert (interface.status_code(st) == 0).all(), np.bincount(interface.status_code(st))
    from oracle import qp_dual_active_set as G

    idx = np.arange(3, B, 64 if N <= 10 else 128)
    setup = oracle.make_setup(N)
    ref, rc = qpoases_sample("sweep_h%d" % N, recs[idx])
    good = rc == 0
    e0, ef = rel_err(w[idx], ref, 12), rel_err(w[idx], ref)
    assert e0[good].max() < 1e-4 and np.median(e0[good]) < 1e-5
    refereed = 0
    for k in np.nonzero(good & (ef > 5e-5))[0]:
        Q = oracle.reduced_qp(recs[idx[k]], setup)
        x, inf = G.solve(Q["H"], Q["g"], Q["A"], Q["lb"], Q["ub"], tol=1e-12, max_iter=3000)
        full = np.zeros(12 * N)
        full[Q["var_ind"]] = x
        assert inf["status"] == 0
        assert rel_err(w[idx[k]][None], full[None])[0] < 1e-6, (N, int(idx[k]))          # the GPU sits on the exact optimum
        assert rel_err(ref[k][None], full[None])[0] > 0.5 * ef[k]                          # ... and qpOASES is what is off
        refereed += 1
    print("horizon %d, %d robots: first step worst %.2e, whole horizon worst %.2e vs qpOASES (%d cases above 5e-5 refereed in fp64)"
          % (N, len(idx), e0[good].max(), ef[good].max(), refereed))
    assert ef[good].max() < 3e-4
