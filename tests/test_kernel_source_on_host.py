"""CPU: the SOURCE of the product's device code, compiled for the host through a fake CUDA prelude and held to the oracle
and to the reference's compiled controller — without a GPU.

tests/host_emul/ builds hector_simulation_b200/csrc/hmpc_device.cuh (inline PTX blanked, nothing else changed) into a
throw-away host library and runs the one-thread-per-robot kernels (data preparation f-1, closed-loop advance f-3,
swing-leg controller f-4) plus the stage-1 device functions of the solve kernel (SRBD linearisation, foot rotations,
constraint rows, a5-a11) and the torque epilogue function (f-2).  This is test infrastructure: the product has no CPU path
(test_capi_cpu.py asserts that), and the cooperative stages of the solve kernel are covered by the -m gpu tests only.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from hector_simulation_b200 import interface, scenarios

HERE = os.path.join(ROOT, "tests", "host_emul")
BUILD = os.path.join(HERE, "_build")
DEVICE_HEADER = os.path.join(ROOT, "hector_simulation_b200", "csrc", "hmpc_device.cuh")


def _blank_inline_ptx(text: str):
    """Replace every `asm volatile( ... );` statement by a comment, matching parentheses outside string literals."""
    out, i, n = [], 0, 0
    key = "asm volatile("
    while True:
        j = text.find(key, i)
        if j < 0:
            out.append(text[i:])
            return "".join(out), n
        out.append(text[i:j])
        k, depth, in_str = j + len(key), 1, False
        while depth:
            c = text[k]
            if in_str:
                if c == "\\":
                    k += 1
                elif c == '"':
                    in_str = False
            elif c == '"':
                in_str = True
            elif c == "(":
                depth += 1
            elif c == ")":
                depth -= 1
            k += 1
        assert text[k] == ";", text[j:k + 20]
        out.append("/* inline PTX blanked for the host build */")
        i, n = k, n + 1


def _replace_body(text: str, signature: str, body: str) -> str:
    """Swap the body of the (unique) function whose definition starts with `signature`."""
    assert text.count(signature) == 1, signature
    j = text.index(signature) + len(signature)
    k = text.index("{", j)
    depth, e = 1, k + 1
    while depth:
        depth += {"{": 1, "}": -1}.get(text[e], 0)
        e += 1
    return text[:k] + "{ " + body + " }" + text[e:]


def _host_buildable(src: str) -> str:
    """The substitutions a host compiler needs (documented in tests/host_emul/kernel_source_on_host.cpp)."""
    src = _replace_body(src, "void mbar_init(uint64_t* bar, int count)", "(void)count; hmpc_emul_mbar_init(bar);")
    src = _replace_body(src, "void mbar_expect_tx(uint64_t* bar, uint32_t bytes)", "(void)bar; (void)bytes;")
    src = _replace_body(src, "void mbar_wait(uint64_t* bar, uint32_t phase)", "hmpc_emul_mbar_wait(bar, phase);")
    src = _replace_body(src, "void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar)",
                        "hmpc_emul_bulk_g2s(dst, src, bytes, bar);")
    src = _replace_body(src, "void dmma884(double& c0, double& c1, double a, double b)", "hmpc_emul_dmma884(c0, c1, a, b);")
    rcp = 'asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));'
    assert src.count(rcp) == 1
    src = src.replace(rcp, "r = 1.0 / x;  /* host build: exact seed instead of MUFU.RCP64H */")
    smem = "extern __shared__ __align__(16) unsigned char smem[];"
    assert src.count(smem) == 1
    src = src.replace(smem, "unsigned char* const smem = hmpc_emul::cta_smem();")
    src, n = _blank_inline_ptx(src)
    assert n == 4, n   # pdl_trigger, pdl_wait, fence.mbarrier_init, fence.proxy.async
    assert "asm" not in src.replace("/* inline PTX blanked", "")
    return src


@pytest.fixture(scope="module")
def emul():
    os.makedirs(BUILD, exist_ok=True)
    hdr = os.path.join(BUILD, "hmpc_device_host.cuh")
    with open(hdr, "w") as f:
        f.write(_host_buildable(open(DEVICE_HEADER).read()))
    lib = os.path.join(BUILD, "libkernel_source_on_host.so")
    cmd = ["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-w", "-pthread",
           "-I" + os.path.join(HERE, "fake_cuda"), "-I" + os.path.join(ROOT, "include"),
           '-DHMPC_DEVICE_HEADER="%s"' % hdr, os.path.join(HERE, "kernel_source_on_host.cpp"), "-o", lib,
           "-l:libstdc++.so.6"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    L = ctypes.CDLL(lib)
    L.emul_leg_torque.restype = ctypes.c_double
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _prepare(L, states, N, dt_mpc=0.04):
    B = len(states)
    stride = L.emul_record_stride(N)
    assert stride == interface.record_bytes(N)
    out = np.full((B, stride), 0xAB, np.uint8)
    st = np.ascontiguousarray(states)
    L.emul_prepare(_p(st), B, N, ctypes.c_double(dt_mpc), _p(out))
    return out


# ---- f-1 ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("horizon,cfg,batch", [(10, 3, 96), (5, 4, 32), (16, 4, 32), (10, 1, 4)])
def test_prepare_kernel_source_equals_host_mirror(emul, horizon, cfg, batch):
    from test_state_prepare import _host_prepared

    _, inputs = scenarios.make_batch(cfg, batch, horizon=horizon)
    states = scenarios.make_states(inputs, horizon)
    want = interface.pack_records(_host_prepared(states, horizon), horizon)
    got = _prepare(emul, states, horizon)
    assert np.array_equal(got, want)


def _case_ticks(oracle, case):
    from test_reference_tick import CASES, committed_ticks

    C = CASES[case]
    c = C["command"]
    cmd5 = np.array([c["roll"], c["pitch"], c["v_des"][0], c["v_des"][1], c["yaw_rate"]])
    return C, cmd5, list(committed_ticks(oracle, case))


@pytest.mark.parametrize("case", ["walk", "walk_zero_command", "walk_saturated", "stand"])
def test_prepare_kernel_source_reproduces_the_reference_controllers_records(emul, oracle, case):
    """Including the zero-command branches of the reference trajectory, the engaged set-point clamp and the standing gait."""
    from test_reference_tick import DT_MPC, N, _pose, _state_record

    C, cmd5, ticks = _case_ticks(oracle, case)
    which = [k for k, o in enumerate(ticks) if o["mpc_ran"]]
    states = np.zeros(len(which), dtype=scenarios.STATE_DTYPE)
    for n, k in enumerate(which):
        pos, rpy, vel, omega, _ = _pose(int(k), C["pose"])
        states[n] = _state_record(ticks[k], pos, vel, scenarios.rpy_to_quat(rpy), omega, cmd5)
    ref = np.array([np.frombuffer(ticks[k]["update_record"].tobytes(), dtype=scenarios.UPDATE_DTYPE)[0] for k in which])
    assert np.array_equal(_prepare(emul, states, N, DT_MPC), interface.pack_records(ref, N))


# ---- f-4 ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["walk", "walk_saturated", "stand"])
def test_swing_kernel_source_follows_the_reference_controller(emul, oracle, case):
    from test_reference_tick import DT, DT_MPC, N, _pose, _state_record

    C, cmd5, ticks = _case_ticks(oracle, case)
    loop = np.zeros(1, dtype=scenarios.ROLLOUT_DTYPE)
    loop["gait_offset"], loop["gait_duration"] = C["offsets"], C["durations"]
    sw = scenarios.make_swing(1)
    cmd = np.zeros(1, dtype=scenarios.SWING_CMD_DTYPE)
    checked, worst_q = 0, 0.0
    for k, o in enumerate(ticks):
        pos, rpy, vel, omega, _ = _pose(k, C["pose"])
        st = np.array([_state_record(o, pos, vel, scenarios.rpy_to_quat(rpy), omega, cmd5)])
        ph = np.array([o["phase"]])
        for _ in range(2):
            emul.emul_swing(_p(st), _p(loop), _p(ph), _p(sw), 1, N, ctypes.c_double(DT), ctypes.c_double(DT_MPC), _p(cmd))
        assert np.array_equal(sw["swing_time"][0], o["swing_times"]) and np.array_equal(sw["first_swing"][0], o["first_swing"]), k
        assert np.array_equal(cmd["pf"][0], o["pf"]), k
        for leg in range(2):
            s3, s5 = slice(3 * leg, 3 * leg + 3), slice(5 * leg, 5 * leg + 5)
            if o["swing_states"][leg] > 0:
                checked += 1
                assert cmd["swing"][0][leg] == 1
                assert np.array_equal(sw["p0"][0][s3], o["p0"][s3]), k
                assert np.array_equal(cmd["p_des"][0][s3], o["p_des"][s3]) and np.array_equal(cmd["v_des"][0][s3], o["v_des"][s3]), k
                worst_q = max(worst_q, float(np.abs(cmd["q_des"][0][s5] - o["q_des"][s5]).max()))
            else:
                assert cmd["swing"][0][leg] == 0 and not cmd["q_des"][0][s5].any()
    assert checked > (300 if case == "walk" else (100 if case == "walk_saturated" else -1)) and worst_q < 1e-12


# ---- f-3 ------------------------------------------------------------------------------------------------------------
def test_advance_kernel_source_equals_numpy_mirror(emul):
    N, B = 10, 48
    _, inputs = scenarios.make_batch(2, B, horizon=N, seed=11)
    states, loop = scenarios.make_rollout(inputs, N)
    s_k, l_k = states.copy(), loop.copy()
    rng = np.random.default_rng(3)
    for tick in range(12):
        wrench = np.zeros((B, 12 * N), np.float32)
        wrench[:, 2] = wrench[:, 5] = 45.0
        wrench[:, :12] += rng.normal(0, 2.0, (B, 12)).astype(np.float32)
        status = (rng.integers(0, 15, B) << 8).astype(np.int32)
        scenarios.advance_numpy(states, loop, wrench, status, N)
        emul.emul_advance(_p(s_k), _p(l_k), B, N, ctypes.c_double(0.04), _p(wrench), _p(status))
        for f in ("position", "vWorld", "orientation", "omegaWorld", "rpy", "leg_p", "world_position_desired"):
            assert np.abs(s_k[f] - states[f]).max() < 1e-12, (tick, f)
        assert np.array_equal(s_k["gait"], states["gait"])
        assert np.abs(l_k["feet_world"] - loop["feet_world"]).max() < 1e-12
        for f in ("iteration", "failures", "iters_total", "ticks"):
            assert np.array_equal(l_k[f], loop[f]), f


# ---- a5-a11: stage 1 of the solve kernel ------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", [2, 3])
def test_stage1_source_is_bit_exact_against_the_oracle(emul, oracle, cfg):
    N, B = 10, 64
    recs, _ = scenarios.make_batch(cfg, B, horizon=N, seed=5 + cfg)
    setup = oracle.make_setup(N)
    packed = interface.pack_records(recs, N)
    for i in range(B):
        rf = np.ascontiguousarray(packed[i, : 54 * 4].view(np.float32))
        Fblk, x0 = np.zeros(192, np.float32), np.zeros(13, np.float32)
        Acd, Bcd = np.zeros(169, np.float32), np.zeros(156, np.float32)
        emul.emul_stage1(_p(rf), ctypes.c_float(0.04), _p(Fblk), _p(x0), _p(Acd), _p(Bcd))
        F = oracle.formulate_f32(recs[i], setup)
        assert np.array_equal(Fblk.reshape(16, 12), F["Fblk"]), i
        assert np.array_equal(x0, F["x0"]), i
        assert np.array_equal(Acd.reshape(13, 13), F["Acd"]), i
        assert np.array_equal(Bcd.reshape(13, 12), F["Bcd"]), i


# ---- f-2: torque epilogue function -------------------------------------------------------------------------------------
def test_leg_torque_source_equals_jacobian_transpose(emul, oracle):
    rng = np.random.default_rng(2)
    for _ in range(40):
        q5, f6 = rng.normal(0, 0.8, 5), rng.normal(0, 30, 6)
        for leg in (0, 1):
            J = oracle.leg_jacobian_fm(q5, leg)
            want = J.T @ f6
            got = np.array([emul.emul_leg_torque(_p(q5), leg, j, _p(f6)) for j in range(5)])
            assert np.abs(got - want).max() < 1e-12 * max(1.0, np.abs(want).max())


# ---- the solve kernel itself, all stages, one OS thread per CUDA thread ------------------------------------------------
def _solve(L, records, N, dump=False, tau=True):
    """The device-resident path of hmpc_capi.cu (classification + class launches + escalation) on the host."""
    B = len(records)
    packed = np.ascontiguousarray(interface.pack_records(records, N))
    n = 12 * N
    w = np.zeros((B, n), np.float32)
    st = np.full(B, -1, np.int32)
    t = np.zeros((B, 10), np.float32)
    launched = np.zeros(3, np.int32)
    d = None
    if dump:
        d = dict(H=np.zeros((B, n, n), np.float32), g=np.zeros((B, n), np.float32), Fblk=np.zeros((B, 16, 12), np.float32),
                 lb=np.zeros((B, 16 * N), np.float32), ub=np.zeros((B, 16 * N), np.float32))
    ptrs = [_p(d[k]) for k in ("H", "g", "Fblk", "lb", "ub")] if dump else [None] * 5
    rc = L.emul_solve(_p(packed), B, N, ctypes.c_float(0.04), ctypes.c_float(500.0), 500, _p(w), _p(st), _p(t) if tau else None,
                      _p(launched), *ptrs)
    assert rc == 0
    return w.astype(np.float64), st, t.astype(np.float64), launched, d


def _solve_plain(L, records, N):
    """The same launch with the block start of the active-set stage switched off (HMPC_BLOCK_ROUNDS=0, read per call by
    the emulation driver like hmpc_create reads it): the plain dual iteration from the unconstrained minimiser."""
    old = os.environ.get("HMPC_BLOCK_ROUNDS")
    os.environ["HMPC_BLOCK_ROUNDS"] = "0"
    try:
        w, st, _, _, _ = _solve(L, records, N, tau=False)
    finally:
        if old is None:
            del os.environ["HMPC_BLOCK_ROUNDS"]
        else:
            os.environ["HMPC_BLOCK_ROUNDS"] = old
    return w, st


def test_solve_kernel_source_assembly_is_bit_exact(emul):
    """Stages 0-3 of the kernel source (TMA staging, SRBD linearisation, powers/Toeplitz blocks, prefix-chain Hessian, swing
    elimination), through the kernel's own assembly-dump mode, against the golden fp32 QP data — the bar the -m gpu suite
    holds the GPU to, here for the source executed on the host."""
    from conftest import load_golden

    for name in ("cfg2_h10", "cfg3_h10", "cfg4_h5", "cfg4_h16"):
        g = load_golden(name)
        N, nf = g["horizon"], min(g["H"].shape[0], 2 if name == "cfg4_h16" else 4)
        _, _, _, _, d = _solve(emul, g["records"][:nf], N, dump=True)
        iu = np.triu_indices(12 * N)
        for i in range(nf):
            assert np.array_equal(d["H"][i][iu].view(np.uint32), g["H"][i][iu].view(np.uint32)), (name, i)
            assert np.array_equal(d["H"][i], d["H"][i].T)
            for k in ("g", "lb", "ub", "Fblk"):
                assert np.array_equal(d[k][i].view(np.uint32), g[k][i].view(np.uint32)), (name, i, k)


def test_solve_kernel_source_single_support_class(emul, oracle):
    """Class 0 (64 threads per CTA, compile-time horizon-10 layout): walking-gait robots of configs[1]."""
    from conftest import load_golden, rel_err

    g = load_golden("cfg2_h10")
    B = 6
    w, st, tau, launched, _ = _solve(emul, g["records"][:B], 10)
    assert launched.tolist() == [B, 0, 0]
    assert (interface.status_code(st) == 0).all()
    assert rel_err(w, g["q_soln"][:B], 12).max() < 5e-6 and rel_err(w, g["q_soln"][:B]).max() < 5e-5
    assert (w[g["q_soln"][:B] == 0.0] == 0.0).all()
    # the plain dual iteration (block start off) makes the same number of working-set changes as qpOASES and lands on
    # the same point as the block start
    w1, st1 = _solve_plain(emul, g["records"][:B], 10)
    assert np.array_equal(interface.status_iters(st1), g["info"][:B, 1]) and np.abs(w1 - w).max() < 1e-9 * np.abs(w).max()
    assert np.array_equal(interface.status_nactive(st1), interface.status_nactive(st))
    # torque epilogue (row f-2) of the same launch
    _, inputs = scenarios.make_batch(2, 64, horizon=10)
    rB = np.array([b["rBody"] for b in inputs[:B]]); ql = np.array([b["q_leg"] for b in inputs[:B]])
    contact = np.array([b["gait"][:2] for b in inputs[:B]])
    ref_tau = oracle.joint_torques(g["q_soln"][:B, :12], rB, ql, contact)
    assert rel_err(tau, ref_tau).max() < 1e-4


def test_solve_kernel_source_double_support_class(emul):
    """Class 1 (224 threads per CTA, 120 variables): the stand of configs[0] and the standing robots of configs[2]."""
    from conftest import load_golden, rel_err

    g1, g3 = load_golden("cfg1_h10"), load_golden("cfg3_h10")
    stand = np.nonzero(g3["info"][:, 2] == 120)[0][:2]
    recs = np.concatenate([g1["records"][:1], g3["records"][stand]])
    want = np.concatenate([g1["q_soln"][:1], g3["q_soln"][stand]])
    w, st, _, launched, _ = _solve(emul, recs, 10, tau=False)
    assert launched.tolist() == [0, len(recs), 0]
    assert (interface.status_code(st) == 0).all()
    assert rel_err(w, want, 12).max() < 5e-5 and rel_err(w, want).max() < 5e-5
    assert abs(w[0, 2] - 47.84) < 0.05 and abs(w[0, 5] - 47.84) < 0.05


@pytest.mark.parametrize("name,B", [("cfg4_h5", 8), ("cfg4_h16", 3)])
def test_solve_kernel_source_runtime_horizon(emul, name, B):
    """The runtime-layout instantiations: horizon 5 (64 / 224 threads) and the horizon-16 extension (224 / 544 threads),
    mixed contact schedules, both classes."""
    from conftest import load_golden, rel_err

    g = load_golden(name)
    N = g["horizon"]
    w, st, _, launched, _ = _solve(emul, g["records"][:B], N, tau=False)
    assert launched[:2].sum() == B and launched[2] == 0 and (launched[:2] > 0).all()
    assert (interface.status_code(st) == 0).all()
    assert rel_err(w, g["q_soln"][:B], 12).max() < 5e-6 and rel_err(w, g["q_soln"][:B]).max() < 5e-5
    assert (w[g["q_soln"][:B] == 0.0] == 0.0).all()
    w1, st1 = _solve_plain(emul, g["records"][:B], N)
    assert np.array_equal(interface.status_iters(st1), g["info"][:B, 1]) and np.abs(w1 - w).max() < 1e-9 * np.abs(w).max()


def test_solve_kernel_source_escalates_a_degenerate_optimum(emul):
    """Working-set overflow: class 1 hands the falling robot to class 2 through the escalation list (the kernel appends to
    the next class's list itself), which still returns a KKT point on the fp64 referee's optimum."""
    from conftest import load_golden

    g = load_golden("degenerate_zero_force_h10")
    w, st, _, launched, _ = _solve(emul, g["records"], 10, tau=False)
    assert launched.tolist() == [0, 1, 1]
    assert (interface.status_code(st) == 0).all(), st
    assert interface.status_nactive(st).max() > 64
    assert np.abs(w - g["q_soln"]).max() < 5e-3
    assert np.abs(w - g["q_referee"]).max() < 2e-5
    assert np.abs(w[:, :6]).max() < 1e-3


def test_solve_kernel_source_against_the_compiled_reference(emul):
    """The kernel source against outputs of the reference's own solve_mpc (tests/golden/ref_compiled_h10.npz): the 1e-4
    contract, no restatement in between."""
    from conftest import GOLDEN, load_golden, rel_err

    z = np.load(os.path.join(GOLDEN, "ref_compiled_h10.npz"))
    g = load_golden("cfg3_h10")
    B = 8
    w, st, _, _, _ = _solve(emul, g["records"][:B], 10, tau=False)
    assert (interface.status_code(st) == 0).all()
    assert rel_err(w, z["cfg3_q"][:B], 12).max() < 1e-4 and rel_err(w, z["cfg3_q"][:B]).max() < 1e-4


# ---- race check of the kernel source (ThreadSanitizer on the emulated CTA) ----------------------------------------------
def test_solve_kernel_source_has_no_data_races(emul, tmp_path):
    """Every CUDA thread is an OS thread and every barrier / warp primitive real synchronisation, so ThreadSanitizer sees
    any two conflicting accesses the kernel does not order (removing a single __syncwarp from the active-set loop makes it
    report within one QP).  Paths: class 0, class 1, class 1 -> class 2 escalation, runtime-horizon variants (up to 544
    threads), the in-place gather mode with double stores, the warm start."""
    from conftest import load_golden

    exe = os.path.join(BUILD, "race_driver_tsan")
    cmd = ["g++", "-std=c++17", "-O1", "-g", "-ffp-contract=off", "-fsanitize=thread", "-w", "-pthread",
           "-I" + os.path.join(HERE, "fake_cuda"), "-I" + os.path.join(ROOT, "include"),
           '-DHMPC_DEVICE_HEADER="%s"' % os.path.join(BUILD, "hmpc_device_host.cuh"),
           os.path.join(HERE, "kernel_source_on_host.cpp"), os.path.join(HERE, "race_driver.cpp"), "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("no ThreadSanitizer runtime with this toolchain: " + r.stderr[-300:])
    cases = [("cfg2_h10", [0, 1, 2], ()), ("cfg1_h10", [0], ()), ("degenerate_zero_force_h10", [0], ()),
             ("cfg4_h5", [0, 1, 2, 3], ()), ("cfg4_h16", [0, 1, 2], ()),       # runtime horizons: 64/224 and 224/544 threads
             ("cfg3_h10", [0, 1], ("raw",)),          # in-place gather of update_data_t records, double results
             ("cfg2_h10", [3, 4], ("warm",))]         # S-pair warm start
    env = dict(os.environ, TSAN_OPTIONS="halt_on_error=0 exitcode=66")
    for name, idx, flags in cases:
        g = load_golden(name)
        f = tmp_path / (name + "".join(flags) + ".bin")
        if "raw" in flags:
            np.ascontiguousarray(g["records"][idx]).tofile(f)
        else:
            np.ascontiguousarray(interface.pack_records(g["records"][idx], g["horizon"])).tofile(f)
        r = subprocess.run([exe, str(f), str(g["horizon"]), *flags], capture_output=True, text=True, env=env, timeout=900)
        assert "ThreadSanitizer" not in r.stderr, (name, flags, r.stderr[:3000])
        assert r.returncode == 0, (name, flags, r.returncode, r.stdout, r.stderr[-500:])
    # working sets beyond the column cache (the full-product primal steps share gq's memory with zb)
    big = scenarios.make_batch(2, 1024, horizon=10, seed=scenarios.config_seed(2) + 4000)[0][[217]]
    f = tmp_path / "beyond_cache.bin"
    np.ascontiguousarray(interface.pack_records(big, 10)).tofile(f)
    r = subprocess.run([exe, str(f), "10"], capture_output=True, text=True, env=env, timeout=900)
    assert "ThreadSanitizer" not in r.stderr and r.returncode == 0, r.stderr[:3000]
    # the stress workload: the no-cache class with ~80 rows, the noise-level stop (record 9) and the conditioning check
    gs = np.load(os.path.join(ROOT, "tests", "golden", "stress_referee.npz"))
    for key, idx in (("h10_x8_records", [9, 21]), ("h10_lying_records", [0])):
        recs = np.ascontiguousarray(gs[key]).view(scenarios.UPDATE_DTYPE).reshape(-1)[idx]
        f = tmp_path / (key + ".bin")
        np.ascontiguousarray(interface.pack_records(recs, 10)).tofile(f)
        r = subprocess.run([exe, str(f), "10"], capture_output=True, text=True, env=env, timeout=1800)
        assert "ThreadSanitizer" not in r.stderr, (key, r.stderr[:3000])
        assert r.returncode == (0 if key.startswith("h10_x8") else 1), (key, r.returncode, r.stdout)   # lying: reported, not solved


def test_solve_kernel_source_edge_cases(emul):
    """The contact-schedule edge cases of the -m gpu suite on the kernel source: no foot in contact over the whole horizon
    (everything eliminated), flight then double support, and arbitrary ragged schedules against qpOASES' recorded optimum."""
    from conftest import qpoases_sample, rel_err

    N = 10
    b = scenarios.stand_inputs(N)
    b["gait"][:] = 0
    b2 = scenarios.stand_inputs(N)
    b2["gait"][:8] = 0
    rng = np.random.default_rng(5)
    recs = [scenarios.to_record(b, N), scenarios.to_record(b2, N)]
    for _ in range(6):
        table = (rng.random(2 * N) < 0.6).astype(np.int32)
        recs.append(scenarios.to_record(scenarios._random_state(rng, N, table, moving=True), N))
    recs = np.array(recs)
    w, st, _, _, _ = _solve(emul, recs, N, tau=False)
    assert (interface.status_code(st) == 0).all()
    assert (w[0] == 0).all()
    assert (w[1, :48] == 0).all() and np.abs(w[1, 48:]).max() > 1
    ref, rc = qpoases_sample("edges8", recs)
    assert (rc == 0).all()
    assert rel_err(w[1:], ref[1:]).max() < 5e-5
    assert (w[ref == 0.0] == 0.0).all()


def test_solve_kernel_source_working_sets_beyond_the_column_cache(emul):
    """Class 0 caches H^-1 a_j for its first N + 4 working-set slots and holds up to 2N + 4 rows: walking robots whose optimum
    has more active rows than the cache (15, 16 and 19 here; ~1 % of the configs[1] batches) stay in class 0 — their primal
    steps go through a full H^-1 product for the slots beyond the cache — instead of being handed to the slower class 1."""
    from conftest import qpoases_sample, rel_err

    N = 10
    picks = ((1000, [780, 20]), (4000, [217]))
    recs = np.concatenate([scenarios.make_batch(2, 1024, horizon=N, seed=scenarios.config_seed(2) + off)[0][idx] for off, idx in picks])
    w, st, _, launched, _ = _solve(emul, recs, N, tau=False)
    assert launched.tolist() == [3, 0, 0]                              # nobody escalates
    assert (interface.status_code(st) == 0).all()
    assert sorted(interface.status_nactive(st).tolist()) == [15, 16, 19]
    ref, rc = qpoases_sample("column_cache", recs)
    assert (rc == 0).all() and rel_err(w, ref, 12).max() < 5e-6 and rel_err(w, ref).max() < 5e-5


def test_solve_kernel_source_is_insensitive_to_its_two_tolerances(emul):
    """The active-set stage has two literals: the KKT tolerance (a row counts as violated below -1e-9 max(1, |x0|)) and the
    dependence threshold (curvature below 1e-11 a'H^-1a).  Neither is tuned to the fixtures: swept over four decades each,
    every instance still converges and the optimum moves far less than the 1e-4 contract."""
    from conftest import load_golden

    g = load_golden("cfg3_h10")
    recs = g["records"][:10]      # walking and standing robots, both size classes
    w0, st0, _, _, _ = _solve(emul, recs, 10, tau=False)
    assert (interface.status_code(st0) == 0).all()
    for var, vals in (("HMPC_TOL_KKT", ("1e-11", "1e-7")), ("HMPC_TOL_DEP", ("1e-13", "1e-9"))):
        for v in vals:
            os.environ[var] = v
            try:
                w, st, _, _, _ = _solve(emul, recs, 10, tau=False)
            finally:
                del os.environ[var]
            assert (interface.status_code(st) == 0).all(), (var, v)
            assert np.abs(w - w0).max() < 1e-5 * np.abs(w0).max(), (var, v, np.abs(w - w0).max())
            assert np.array_equal(interface.status_nactive(st), interface.status_nactive(st0)), (var, v)


def test_solve_kernel_source_in_place_and_warm_start_modes(emul):
    """The other modes of the same kernel: gathering the live bytes of the caller's update_data_t records in place (the
    host-buffer path's in-place mode), double-precision result stores, and the optional S-pair warm start."""
    from conftest import load_golden, rel_err

    g = load_golden("cfg3_h10")
    N, B = 10, 6
    recs = np.ascontiguousarray(g["records"][:B])
    w0, st0, tau0, _, _ = _solve(emul, recs, N)
    w = np.zeros((B, 12 * N), np.float32)
    w64 = np.zeros((B, 12 * N), np.float64)
    st = np.full(B, -1, np.int32)
    tau = np.zeros((B, 10), np.float32)
    rc = emul.emul_solve_ex(None, _p(recs), B, N, ctypes.c_float(0.04), ctypes.c_float(500.0), 500, 0, _p(w), _p(w64), _p(st), _p(tau),
                            None, None, None, None, None, None)
    assert rc == 0
    assert np.array_equal(w.astype(np.float64), w0) and np.array_equal(st, st0) and np.array_equal(tau.astype(np.float64), tau0)
    assert np.array_equal(w64.astype(np.float32), w)   # the double store keeps the fp64 solve's bits; rounded it is the float result
    assert np.abs(w64 - w0).max() > 0                  # ... and it is not just the float result widened
    packed = np.ascontiguousarray(interface.pack_records(recs, N))
    ww = np.zeros((B, 12 * N), np.float32)
    sw = np.full(B, -1, np.int32)
    rc = emul.emul_solve_ex(_p(packed), None, B, N, ctypes.c_float(0.04), ctypes.c_float(500.0), 500, 1, _p(ww), None, _p(sw), None,
                            None, None, None, None, None, None)
    assert rc == 0 and (interface.status_code(sw) == 0).all()
    assert rel_err(ww.astype(np.float64), g["q_soln"][:B]).max() < 5e-5


def test_closed_loop_of_kernel_sources(emul, oracle):
    """hmpc_rollout_device's tick — data-preparation kernel -> classification + solve kernels -> advance kernel — with all
    three kernels' sources chained on the host, against the same loop driven from the host (host mirror of the preparation,
    the same solve, numpy mirror of the advance step: the comparison tests/test_rollout.py makes on the GPU), with qpOASES
    (or, where it is not built, the exact fp64 referee of the same QPs) checking every tick's wrench."""
    from conftest import reference_solve, rel_err
    from test_rollout import _host_prepared, _walkers

    N, B, T = 10, 3, 8
    states, loop = _walkers(B)
    s_k, l_k = states.copy(), loop.copy()
    setup = oracle.make_setup(N)
    stride = interface.record_bytes(N)

    def solve(packed):
        w = np.zeros((B, 12 * N), np.float32)
        st = np.full(B, -1, np.int32)
        assert emul.emul_solve(_p(packed), B, N, ctypes.c_float(0.04), ctypes.c_float(500.0), 500, _p(w), _p(st), None, None,
                               None, None, None, None, None) == 0
        assert (interface.status_code(st) == 0).all()
        return w, st

    # third loop: the kernels' loop again, but every tick proposes the previous tick's working set (hmpc_rollout_device's
    # warm start) — must stay on the cold loops' trajectory and need far fewer working-set changes
    s_w, l_w = states.copy(), loop.copy()
    ws = np.zeros((B, emul.emul_ws_ints()), np.int32)
    warm_changes, cold_changes = 0, 0
    for t in range(T):
        # host-driven loop
        recs = _host_prepared(states, N)
        w_h, st_h = solve(np.ascontiguousarray(interface.pack_records(recs, N)))
        q, info = reference_solve(oracle, recs, setup)
        assert (info[:, 0] == 0).all() and rel_err(w_h.astype(np.float64), q, 12).max() < 5e-5
        scenarios.advance_numpy(states, loop, w_h, st_h, N)
        # the kernels' loop
        packed = np.zeros((B, stride), np.uint8)
        emul.emul_prepare(_p(s_k), B, N, ctypes.c_double(0.04), _p(packed))
        w_k, st_k = solve(packed)
        emul.emul_advance(_p(s_k), _p(l_k), B, N, ctypes.c_double(0.04), _p(w_k), _p(st_k))
        # warm loop
        packed = np.zeros((B, stride), np.uint8)
        emul.emul_prepare(_p(s_w), B, N, ctypes.c_double(0.04), _p(packed))
        emul.emul_set_ws(_p(ws), 1)
        w_w = np.zeros((B, 12 * N), np.float32)
        st_w = np.full(B, -1, np.int32)
        assert emul.emul_solve_ex(_p(packed), None, B, N, ctypes.c_float(0.04), ctypes.c_float(500.0), 500, 1, _p(w_w), None, _p(st_w),
                                  None, None, None, None, None, None, None) == 0
        emul.emul_set_ws(None, 0)
        assert (interface.status_code(st_w) == 0).all()
        assert np.abs(w_w.astype(np.float64) - w_k).max() < 1e-5 * np.abs(w_k).max()   # same optimum (float output)
        if t > 0:
            warm_changes += int(interface.status_iters(st_w).sum())
            cold_changes += int(interface.status_iters(st_k).sum())
        emul.emul_advance(_p(s_w), _p(l_w), B, N, ctypes.c_double(0.04), _p(w_w), _p(st_w))
        for f in ("position", "vWorld", "orientation", "omegaWorld", "rpy", "leg_p", "world_position_desired"):
            assert np.abs(s_w[f] - states[f]).max() < 1e-6, (t, f, np.abs(s_w[f] - states[f]).max())
        for f in ("position", "vWorld", "orientation", "omegaWorld", "rpy", "leg_p", "world_position_desired"):
            assert np.abs(s_k[f] - states[f]).max() < 1e-9, (t, f, np.abs(s_k[f] - states[f]).max())
        assert np.array_equal(s_k["gait"], states["gait"])
        assert np.abs(l_k["feet_world"] - loop["feet_world"]).max() < 1e-9
    assert (l_k["failures"] == 0).all() and np.array_equal(l_k["ticks"], np.full(B, T))
    assert np.array_equal(l_k["iters_total"], loop["iters_total"])
    print("closed loop of kernel sources: working-set changes per tick: cold %.2f, warm %.2f" % (cold_changes / (B * (T - 1)), warm_changes / (B * (T - 1))))
    assert warm_changes < 0.5 * cold_changes


def test_solve_kernel_source_warm_start_survives_any_proposal(emul):
    """The warm start only PROPOSES rows to the block start; what it proposes must not be able to change the optimum.  Hostile
    states — random rows, all ten rows of a block (linearly dependent: 10 rows on 6 variables), rows of the wrong side of
    every friction pair, swing-phase blocks, counts out of range, the true working set shifted by the wrong number of steps —
    all end at the cold solve's optimum with status 0 (dependent proposals are dropped and the plain dual iteration runs)."""
    from conftest import load_golden

    g = load_golden("cfg3_h10")
    N, B = 10, 8
    recs = np.ascontiguousarray(g["records"][:B])   # walking and standing robots
    packed = np.ascontiguousarray(interface.pack_records(recs, N))
    W = emul.emul_ws_ints()

    def run(ws, shift):
        w = np.zeros((B, 12 * N), np.float32)
        st = np.full(B, -1, np.int32)
        emul.emul_set_ws(_p(ws) if ws is not None else None, shift)
        try:
            rc = emul.emul_solve_ex(_p(packed), None, B, N, ctypes.c_float(0.04), ctypes.c_float(500.0), 500, 1 if ws is not None else 0,
                                    _p(w), None, _p(st), None, None, None, None, None, None, None)
        finally:
            emul.emul_set_ws(None, 0)
        assert rc == 0
        return w.astype(np.float64), st

    w0, st0 = run(None, 0)
    assert (interface.status_code(st0) == 0).all()
    # the true working sets, written back by a recording pass (warm flag on, empty proposals)
    true_ws = np.zeros((B, W), np.int32)
    w1, st1 = run(true_ws, 0)
    assert np.array_equal(w1, w0) and (true_ws[:, 0] > 0).all()
    rng = np.random.default_rng(7)
    cases = {}
    rnd = np.zeros((B, W), np.int32)
    for b in range(B):
        c = int(rng.integers(1, W))
        rnd[b, 0] = c
        rnd[b, 1:1 + c] = (rng.integers(0, 2 * N, c) << 8) | rng.integers(0, 20, c)
    cases["random rows"] = (rnd, 0)
    dep = np.zeros((B, W), np.int32)
    dep[:, 0] = 20
    for b in range(B):
        blk = int(true_ws[b, 1]) >> 8            # a block that is in stance (it holds an active row)
        leg = blk & 1
        dep[b, 1:11] = (blk << 8) | (leg * 10 + np.arange(10))
        dep[b, 11:21] = (((blk + 2) % (2 * N)) << 8) | (leg * 10 + np.arange(10))
    cases["all ten rows of two blocks"] = (dep, 0)
    opp = true_ws.copy()
    for b in range(B):
        c = opp[b, 0]
        t = (opp[b, 1:1 + c] & 0xff) % 10
        flip = np.where(t < 4, t ^ 1, t)          # the other side of the friction pair (rows 0/1 and 2/3)
        opp[b, 1:1 + c] = (opp[b, 1:1 + c] & ~0xff) | ((opp[b, 1:1 + c] & 0xff) - t + flip)
    cases["opposite friction sides"] = (opp, 0)
    cases["true set, shifted by three steps"] = (true_ws.copy(), 3)
    cases["true set, shifted backwards"] = (true_ws.copy(), -2)
    bad = true_ws.copy()
    bad[::2, 0] = W + 5
    bad[1::2, 0] = -3
    cases["counts out of range"] = (bad, 0)
    for name, (ws, shift) in cases.items():
        w, st = run(ws.copy(), shift)
        assert (interface.status_code(st) == 0).all(), (name, st)
        assert np.abs(w - w0).max() < 1e-5 * np.abs(w0).max(), (name, np.abs(w - w0).max())
        assert np.array_equal(interface.status_nactive(st), interface.status_nactive(st0)), name


def test_solve_kernel_source_far_outside_the_operating_envelope(emul):
    """Robustness workload (tests/golden/stress_referee.npz, scenarios.make_stress_batch): states 4-8 x the walking batches'
    perturbations under walking / standing / random contact tables, up to ~100 active rows at massively degenerate optima;
    all three size classes (the last one without column cache).  qpOASES itself is off the exact optimum by up to 4e-4 of
    the first-step wrench on these problems, so the kernel is held to the tight-tolerance fp64 REFEREE stored in the
    fixture: every instance converges, sits on the referee's optimum, and where the two CPU answers differ it is the kernel
    that agrees with the exact one.  Record 9 of the x8 set is the regression case of the noise-level stop: its last
    "violated" row is a dependent one, violated by round-off only — reported as infeasible before."""
    from conftest import GOLDEN, rel_err

    g = np.load(os.path.join(GOLDEN, "stress_referee.npz"))
    n_far = 0
    for name, N, idx in (("h10_x8", 10, [9, 21, 22]), ("h10_x4", 10, [12, 24]), ("h14_x4", 14, [14])):
        recs = np.ascontiguousarray(g[name + "_records"]).view(scenarios.UPDATE_DTYPE).reshape(-1)[idx]
        ref, q = g[name + "_referee"][idx], g[name + "_qpoases"][idx]
        w, st, _, launched, _ = _solve(emul, recs, N, tau=False)
        assert (interface.status_code(st) == 0).all(), (name, st)
        assert interface.status_nactive(st).max() > 30
        assert rel_err(w, ref, 12).max() < 5e-5 and rel_err(w, ref).max() < 1e-5, (name, rel_err(w, ref, 12), rel_err(w, ref))
        far = rel_err(q, ref, 12) > 5e-5                 # qpOASES off the exact optimum
        assert (rel_err(w, ref, 12)[far] < 0.5 * rel_err(q, ref, 12)[far]).all()
        n_far += int(far.sum())
    assert n_far >= 3


def test_solve_kernel_source_reports_a_hessian_beyond_its_conditioning_limit(emul):
    """The in-place sweep inversion loses accuracy like the square of the scaled condition number (DESIGN.md §2).  A robot
    lying on its side (fixture record h10_lying: max_i H_ii (H^-1)_ii = 2.9e5 against 2e2 ... 1e4 on BASELINE's workloads)
    would come back 8e-3 off the exact optimum with a clean status; the conditioning check of stage 5 reports it as not
    solved instead (status code 4, 'failed to solve!' at the reference boundary).  With the check lifted (HMPC_KAPPA_MAX)
    the same record shows what it guards against."""
    from conftest import GOLDEN, rel_err

    g = np.load(os.path.join(GOLDEN, "stress_referee.npz"))
    recs = np.ascontiguousarray(g["h10_lying_records"]).view(scenarios.UPDATE_DTYPE).reshape(-1)
    ref = g["h10_lying_referee"]
    assert rel_err(g["h10_lying_qpoases"], ref, 12).max() < 2e-5       # the reference's solver handles it
    w, st, _, launched, _ = _solve(emul, recs, 10, tau=False)
    assert interface.status_code(st).tolist() == [4]
    os.environ["HMPC_KAPPA_MAX"] = "1e12"
    try:
        w, st, _, _, _ = _solve(emul, recs, 10, tau=False)
    finally:
        del os.environ["HMPC_KAPPA_MAX"]
    assert interface.status_code(st).tolist() == [0] and 1e-3 < rel_err(w, ref, 12)[0] < 5e-2
