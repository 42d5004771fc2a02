#!/usr/bin/env python
"""bench.py — QP solves/sec of the batched force-and-moment MPC hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle/_ref)

A "step" is one pass of the hot path over one batch: BASELINE.json configs[1] — batch = 1024 Hector
walking-gait states per GPU, horizon 10 — i.e. 1024 complete `solve_mpc` equivalents per step per GPU.

  value : whole-job QP solves/s with the packed records already resident in HBM (device-timed with CUDA
          events on the launch stream, max over ranks).  Every step reads a different input buffer
          out of a ring larger than L2, so no step finds its inputs cached.
  e2e   : the same metric through the reference-facing C-ABI call hmpc_solve_batch with HOST buffers
          (pack + H2D + kernels + D2H inside the timed region).
Multi-GPU: robots are independent, the batch is sharded (weak scaling: 1024 per GPU), no data-path
collective; one all_gather of the results per step is included in the e2e leg only when N > 1.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HORIZON = 10
BATCH_PER_GPU = 1024
METRIC = "QP solves/sec (batched MPC ticks), horizon N=10"
UNIT = "QP/s"


def algorithmic_bytes_per_qp(N: int) -> int:
    return 216 + 98 * N  # SURVEY.md §8d: inputs that change per tick + the 12N-float result


def algorithmic_flops_per_qp(N: int, nv: float, k_iter: float) -> float:
    """SURVEY.md §8d formulas, with nv = reduced variable count (12N double support, 6N walking)."""
    f_asm = 2 * nv * nv * 13 * N + 2 * nv * 13 * N + 2 * 13 * 13 * N + N * (2 * 13 ** 3 + 2 * 13 * 13 * 12)
    f_it = nv ** 3 / 3 + 2 * 16 * 12 * 12 * N * (nv / (12.0 * N)) + 4 * nv * nv + 2 * nv * nv + 4 * 16 * 12 * N * (nv / (12.0 * N))
    return f_asm + k_iter * f_it


_SAMPLER_SRC = r"""
import subprocess, sys, time
gpu = int(sys.argv[1])
names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
try:
    import pynvml as nv
    nv.nvmlInit()
    h = nv.nvmlDeviceGetHandleByIndex(gpu)
    mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
    bits = [nv.nvmlClocksThrottleReasonHwSlowdown, nv.nvmlClocksThrottleReasonHwThermalSlowdown,
            nv.nvmlClocksThrottleReasonSwThermalSlowdown, nv.nvmlClocksThrottleReasonSwPowerCap]
    def sample():
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        return float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), mx, [n for b, n in zip(bits, names) if r & b]
    period = 0.004
except Exception:
    q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    def sample():
        out = subprocess.run(["nvidia-smi", "-i", str(gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        r = [c.strip() for c in out.split(",")]
        return float(r[0]), float(r[1]), [names[i] for i in range(4) if r[2 + i].lower().startswith("active")]
    period = 0.05
print("ready", flush=True)
while True:
    try:
        sm, mx_, rs = sample()
        print("%.6f %.1f %.1f %s" % (time.monotonic(), sm, mx_, ",".join(rs)), flush=True)
    except Exception:
        pass
    time.sleep(period)
"""


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (NVML every ~4 ms; nvidia-smi as fallback).
    Runs as a separate process so that sampling never contends with the timed host code for the interpreter
    lock; samples carry CLOCK_MONOTONIC stamps and only those inside [start(), stop()] are kept."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = subprocess.Popen([sys.executable, "-c", _SAMPLER_SRC, str(gpu_index)], stdout=subprocess.PIPE,
                                     stderr=subprocess.DEVNULL, text=True)
        self.proc.stdout.readline()  # "ready": interpreter and NVML are up
        self.t0 = None

    def start(self):
        self.t0 = time.monotonic()

    def stop(self) -> dict:
        t1 = time.monotonic()
        time.sleep(0.01)
        self.proc.terminate()
        out, _ = self.proc.communicate(timeout=10)
        sm, reasons, mx = [], set(), None
        for ln in out.splitlines():
            f = ln.split(" ")
            if len(f) < 3:
                continue
            try:
                t, v, m = float(f[0]), float(f[1]), float(f[2])
            except ValueError:
                continue
            mx = m
            if self.t0 <= t <= t1:
                sm.append(v)
                if len(f) > 3 and f[3]:
                    reasons.update(f[3].split(","))
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, per launch, from the committed
    `ncu --set full` summary of this round (profiles/ncu_r1_final_summary.txt); None if absent."""
    p = os.path.join(ROOT, "profiles", "ncu_r2_final_summary.txt")
    if not os.path.exists(p):
        p = os.path.join(ROOT, "profiles", "ncu_r1_final_summary.txt")
    if not os.path.exists(p):
        return None
    tot, unit_mul = 0.0, {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    found = 0
    for ln in open(p):
        if ln.startswith("dram__bytes_read.sum:") or ln.startswith("dram__bytes_write.sum:"):
            _, v, u = ln.split()
            tot += float(v) * unit_mul.get(u, 1.0)
            found += 1
    return tot if found == 2 else None


def measured_peaks() -> dict:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        d["_source"] = "measured (MEASURED_PEAKS.json)"
        return d
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback (B200_PROFILING.md)"}


def _physical_cpus() -> list[int]:
    """One logical CPU per physical core among the CPUs this process may use (first sibling of every core)."""
    allowed = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    seen, out = set(), []
    for c in allowed:
        try:
            sib = open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read().strip()
        except OSError:
            sib = str(c)
        if sib not in seen:
            seen.add(sib)
            out.append(c)
    return out


def _cpu_worker(args):
    """One solver pinned to one core, running for a fixed wall time: returns (end time, seconds) of every solve."""
    cpu, recs, t_end = args
    try:
        os.sched_setaffinity(0, {cpu})
    except (AttributeError, OSError):
        pass
    from oracle import oracle_py as O

    setup = O.make_setup(HORIZON)
    O.time_solves(recs[:4], setup, 4)  # page in the library and the solver's buffers
    stamps, lats = [], []
    i = 0
    while time.monotonic() < t_end:
        lo = (i * 16) % len(recs)
        chunk = recs[lo:lo + 16] if lo + 16 <= len(recs) else recs[:16]
        lat = O.time_solves(chunk, setup, len(chunk))
        now = time.monotonic()
        stamps.append(now)
        lats.append(np.asarray(lat))
        i += 1
    return np.array(stamps), lats


def cpu_reference_leg(records, steps: int, warmup: int, window_s: float | None = None, budget_s: float = 150.0):
    """Times the reference's CPU implementation of the path — oracle/_ref/liboracle_mpc.so: solve_mpc restated
    (bit-identical to the reference's own sources compiled against a stand-in, tests/test_reference_compiled.py) + the
    reference's qpOASES 3.2 compiled unchanged — with one independent solver per PHYSICAL core (the reference is
    single-threaded and non-reentrant), each pinned to its core and running for a fixed wall time with no barrier between
    steps.  A "step" is a window of `window_s` seconds; the first `warmup` windows are not counted.
    Returns (QP/s, cores, per-solve seconds, window_s, per-core QP/s)."""
    import multiprocessing as mp

    cpus = _physical_cpus()
    # a container's CPU-time quota (cgroup cpu.max) can be far below the visible core count: more workers than that only
    # get throttled in 100 ms periods (seen as a 50-90 ms p99 on a 1 ms solve)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            cpus = cpus[: max(1, int(float(quota) / float(period)))]
    except (OSError, ValueError):
        pass
    cores = len(cpus)
    if window_s is None:
        window_s = min(1.0, budget_s / (warmup + steps))
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        t0 = time.monotonic() + 1.0  # workers start up, then everybody runs until the common deadline
        t_end = t0 + (warmup + steps) * window_s
        outs = pool.map(_cpu_worker, [(c, records, t_end) for c in cpus], chunksize=1)
    lo, hi = t0 + warmup * window_s, t_end
    solves, lat = 0, []
    for stamps, lats in outs:
        for ts, l in zip(stamps, lats):
            if lo < ts <= hi:
                solves += len(l)
                lat.append(l)
    lat = np.concatenate(lat) if lat else np.zeros(1)
    qps = solves / (hi - lo)
    return qps, cores, lat, window_s, qps / cores


def run_reference(args):
    from hector_simulation_b200 import scenarios

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    recs, _ = scenarios.make_batch(2, BATCH_PER_GPU, horizon=HORIZON)
    from oracle import oracle_py as O

    if not O.has_qpoases():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref built without qpOASES (no /root/reference, no prebuilt .so)"}))
        return
    qps, cores, lat, win, per_core = cpu_reference_leg(recs, args.steps, max(args.warmup, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": win * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 assembly / f64 solve",
        "data": "synthetic", "config": {"workload": "configs[1]: batch=1024 Hector walking-gait states, horizon=10 — same records as the GPU arm; a step is a fixed wall-time window over them",
                                       "horizon": HORIZON, "window_s": win},
        "cpu_baseline": cpu_baseline_entry(qps, cores, lat, win, per_core, args.steps),
        "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def cpu_baseline_entry(qps, cores, lat, win, per_core, steps):
    return {"value": qps, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{steps} windows of {win:.2f} s, one solver process pinned to each of the {cores} physical cores, cycling through the 1024 records, no barrier between windows",
            "what": "oracle/_ref/liboracle_mpc.so: solve_mpc restated without Eigen (bit-identical to the reference's own sources compiled against an Eigen stand-in, oracle/_ref/libref_mpc.so, tests/test_reference_compiled.py) + the reference's qpOASES 3.2 compiled unchanged",
            "per_core_qps": per_core, "latency_ms_p50": float(np.percentile(lat, 50) * 1e3), "latency_ms_p99": float(np.percentile(lat, 99) * 1e3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="robots per GPU (default: BASELINE configs[1])")
    ap.add_argument("--workload", default="walk", choices=["walk", "mixed"],
                    help="walk: BASELINE configs[1] (walking-gait states); mixed: configs[2] (25 %% stand / 75 %% walk, randomized)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step of the device and end-to-end legs as DIR/<name>.npy "
                         "(with several GPUs: rank 0's robots)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    from hector_simulation_b200 import interface, scenarios

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this path has no CPU fallback (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own banner ("NCCL version ...", printed when NCCL_DEBUG is set)
        # goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    B, N = args.batch, HORIZON
    K, W = args.steps, args.warmup

    # synthetic states (configs[1] walking gait / configs[2] mixed); each rank gets its own shard (different seed)
    cfg = 2 if args.workload == "walk" else 3
    seed_rank = int(os.environ.get("HMPC_BENCH_SEED_RANK", rank))  # (developer knob: another rank's shard on this GPU)
    recs, inputs = scenarios.make_batch(cfg, B, horizon=N, seed=scenarios.config_seed(cfg) + 1000 * seed_rank)
    mpc = interface.BatchedMPC(B, N, device=local_rank)
    stride = interface.record_bytes(N)
    packed = torch.from_numpy(interface.pack_records(recs, N)).cuda()
    # ring of input/output buffers larger than L2 (126 MB): no step re-reads cached inputs
    ring = max(8, int(np.ceil(192e6 / (B * (stride + 48 * N + 4)))))
    d_in = packed.unsqueeze(0).repeat(ring, 1, 1).contiguous()
    d_out = torch.zeros((ring, B, 12 * N), dtype=torch.float32, device="cuda")
    d_st = torch.zeros((ring, B), dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident leg ----------------
    for i in range(W):
        mpc.solve_device(d_in[i % ring], B, d_out[i % ring], d_st[i % ring])
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    e_all0, e_all1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_all0.record(stream)
    for i in range(K):
        j = (W + i) % ring
        ev[i][0].record(stream)
        mpc.solve_device(d_in[j], B, d_out[j], d_st[j])
        ev[i][1].record(stream)
    e_all1.record(stream)
    barrier()
    total_ms = e_all0.elapsed_time(e_all1)
    step_ms = np.array([a.elapsed_time(b) for a, b in ev])
    print("[bench] rank %d device leg: %.4f ms per step (p50 of steps %.4f)" % (rank, total_ms / K, float(np.percentile(step_ms, 50))), file=sys.stderr)
    # ---------------- end-to-end leg (host buffers through the C-ABI) ----------------
    # Every rank ticks its own slice through sharding.ShardedMPC -> hmpc_solve_batch_sharded: the reference-facing call on
    # the caller's registered update_data_t / result arrays (records read and double wrenches written in place over PCIe),
    # this rank's slice back on ITS host arrays.  N > 1: the library also enqueues the path's ONE collective, an
    # ncclAllGather of the float wrenches into a device buffer on every rank, on a side stream beside the next tick; the
    # last gather is waited for inside the timed region.  Same code path at N = 1 (no gather).
    from hector_simulation_b200 import sharding

    def bcast(b):
        box = [b]
        if world > 1:
            dist.broadcast_object_list(box, src=0)
        return box[0]

    if world > 1:
        factory = lambda bl: sharding.GpuBackend(bl, N, rank, world, local_rank, bcast)
    else:
        factory = None
    recs_c = interface.page_aligned(recs.shape, recs.dtype)   # a control loop's registered arrays own their pages
    recs_c[...] = recs
    if world > 1:
        sh = sharding.ShardedMPC(world * B, N, rank, world, factory, scenarios.UPDATE_DTYPE)
        out_w, out_s = sh.out_w, sh.out_s
        sh.records[:B] = recs_c.view(scenarios.UPDATE_DTYPE).reshape(-1)  # the loop's registered array, filled in place

        def e2e_step():
            sh.tick()
    else:
        out_w = interface.page_aligned((B, 12 * N), np.float64)  # caller-owned result buffers, reused every tick
        out_s = interface.page_aligned(B, np.int32)
        mpc.pin(recs_c, out_w, out_s)

        def e2e_step():
            mpc.solve_batch(recs_c, out=(out_w, out_s))
    for _ in range(W):
        e2e_step()
    if world > 1:
        sh.backend.wait()  # no gather in flight while torch's own communicator runs the barrier below (two NCCL
                           # communicators must not have collectives in flight on one device in different orders)
    barrier()
    t0 = time.perf_counter()
    e2e_lat = []
    for _ in range(K):
        t1 = time.perf_counter()
        e2e_step()
        e2e_lat.append(time.perf_counter() - t1)
    if world > 1:
        sh.backend.wait()  # the last tick's gather
    barrier()
    e2e_s = time.perf_counter() - t0
    assert (interface.status_code(out_s[:B]) == 0).all(), "non-converged instances in the end-to-end leg"
    # the end-to-end leg's result arrays are reused below: keep what its last timed step returned
    e2e_w_last, e2e_s_last = np.array(out_w[:B]), np.array(out_s[:B])
    # after the timed region: what the gather delivered (every rank's slice, on this device) against the oracle
    parity = None
    if world > 1:
        whole = sh.whole_batch()
        if rank == 0:
            try:
                from oracle import oracle_py as O

                if O.has_qpoases():
                    worst, checked = 0.0, 0
                    for r in range(world):
                        rr, _ = scenarios.make_batch(cfg, B, horizon=N, seed=scenarios.config_seed(cfg) + 1000 * r)
                        idx = np.arange(r % 7, B, max(1, B // 6))[:6]
                        ref, info = O.solve_batch(rr[idx], O.make_setup(N))
                        got = whole[r * B + idx].astype(np.float64)
                        ok = info[:, 0] == 0
                        e = np.linalg.norm(got[ok, :12] - ref[ok, :12], axis=1) / np.maximum(np.linalg.norm(ref[ok, :12], axis=1), 1e-9)
                        worst = max(worst, float(e.max()))
                        checked += int(ok.sum())
                    parity = {"gathered_vs_oracle_worst_rel_err": worst, "robots_checked": checked, "ranks": world, "contract": 1e-4}
            except Exception as e:  # reported, never required
                parity = {"unavailable": str(e)}
        sh.close()
    clocks = sampler.stop()

    t = torch.tensor([total_ms, e2e_s * 1e3, float(np.percentile(step_ms, 99))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, p99_step_ms = (float(x) for x in t.cpu())
    st = d_st[(W + K - 1) % ring].cpu().numpy()
    assert (interface.status_code(st) == 0).all(), "non-converged instances in the timed region"
    iters = interface.status_iters(st)
    if args.dump_outputs and rank == 0:
        # inputs are seeded (scenarios.make_batch), so two builds run with the same arguments can be compared array for array
        os.makedirs(args.dump_outputs, exist_ok=True)
        dump = {"device_wrench": d_out[(W + K - 1) % ring].cpu().numpy(),
                "device_status_code": interface.status_code(st), "device_status_iters": iters,
                "e2e_wrench": e2e_w_last, "e2e_status_code": interface.status_code(e2e_s_last),
                "e2e_status_iters": interface.status_iters(e2e_s_last)}
        rows = np.arange(B)
        row_bytes = sum(int(np.prod(np.shape(a)[1:])) * (8 if np.asarray(a).dtype == np.float64 else 4) for a in dump.values()) + 8
        if B * row_bytes > 64 << 20:  # at most 64 MB: a fixed, seeded sample of the robots
            rows = np.sort(np.random.default_rng(0).choice(B, (64 << 20) // row_bytes, replace=False))
        for name, a in dump.items():
            a = np.asarray(a)[rows]
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))
        np.save(os.path.join(args.dump_outputs, "robot_index.npy"), rows.astype(np.float64))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    qps = world * B * K / (total_ms * 1e-3)
    e2e_qps = world * B * K / (e2e_ms * 1e-3)
    peaks = measured_peaks()
    k_mean = float(iters.mean())
    nv = 6.0 * N if args.workload == "walk" else 6.0 * N * 1.25  # walking gait: one stance leg per step; mix: a quarter stands
    flops = algorithmic_flops_per_qp(N, nv, k_mean) * B
    byts = algorithmic_bytes_per_qp(N) * B
    kern_ms = float(np.mean(step_ms))  # all launches of one step (classification + one per size class)
    ach_tf = flops / (kern_ms * 1e-3) / 1e12
    ach_gbs = byts / (kern_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 assembly (bit-exact to reference arithmetic) / f64 solve", "data": "synthetic",
        "config": {"workload": ("configs[1]: batch=%d Hector walking-gait states per GPU, horizon=10, cold start every tick" % B) if args.workload == "walk" else
                               ("configs[2]: %d randomized CoM/velocity/contact-schedule states per GPU (25 %% stand / 75 %% walk), horizon=10, cold start every tick" % B),
                   "horizon": N, "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"batch-sharded x{world}",
                   "l2": f"ring of {ring} input/output buffers ({ring * B * (stride + 48 * N + 4) / 1e6:.0f} MB > L2)"},
        "latency_ms": {"batch_p50": float(np.percentile(step_ms, 50)), "batch_p99": p99_step_ms,
                       "note": "device time for the whole 1024-robot batch; every robot's result is ready within it"},
        "solver": {"mean_working_set_changes": k_mean, "max": int(iters.max())},
        "e2e": {"value": e2e_qps, "unit": UNIT, "h2d_bytes_per_step": int(B * stride), "d2h_bytes_per_step": int(B * (96 * N + 4)),
                "transfer": "in place, per rank: kernels gather the live 720 B of every host update_data_t over PCIe and store double wrenches + status into the caller's registered arrays"
                            + ("; plus ONE ncclAllGather of the float wrenches (device to device, %d B per rank) on a side stream beside the next tick, last one waited for inside the timed region" % (B * 48 * N) if world > 1 else ""),
                "ms_per_step": e2e_ms / K, "latency_ms_p99": float(np.percentile(e2e_lat, 99) * 1e3)},
        "gpu_launches": int(K * mpc.launches_per_solve),  # per step: one solve-kernel launch per size class (class 0 classifies on the way)
        "launch_config": {"class0": mpc.class_config(0), "class1": mpc.class_config(1)},
        "clocks": clocks,
        "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": ach_tf / peaks["bf16_tflops"],
                     "traffic": ncu_traffic_bytes(), "traffic_unit": "bytes per launch (dominant kernel, 1024 QPs; algorithmic = %d)" % byts,
                     "peak_source": peaks["_source"],
                     "note": "algorithmic flops (SURVEY.md §8d: F_asm + k*F_it, nv=6N) / mean step time against the measured bf16 tensor peak (the schema's denominator); the kernel's tensor-pipe work is the fp64 sweep (mma.m8n8k4.f64), whose own pipe peak is ~37 TFLOP/s (tests/tools/ubench.cu), the assembly is bit-exact fp32 on CUDA cores — DESIGN.md §6",
                     "hbm": {"achieved": ach_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach_gbs / peaks["hbm_gbs"],
                             "bytes_per_qp": algorithmic_bytes_per_qp(N)}},
    }
    if parity is not None:
        line["parity"] = parity
    if world == 1:
        # one robot through the reference's own boundary (setup_problem / update_problem_data / get_solution),
        # the call sequence of ConvexMPCLocomotion.cpp:410-430 — per-tick latency against the 500 Hz (2 ms) deadline
        try:
            tick = []
            for name, b in (("stand", scenarios.stand_inputs(N)), ("walk", scenarios.make_batch(2, 1, horizon=N)[1][0])):
                lat = []
                for it in range(220):
                    t1 = time.perf_counter()
                    interface.setup_problem(scenarios.DT_MPC, N, scenarios.MU_PASSED, scenarios.F_MAX)
                    interface.update_problem_data(b["p"], b["v"], b["q"], b["w"], b["r"], b["joint_angles"], b["yaw"], b["weights"],
                                                  b["state_trajectory"], b["Alpha_K"], b["gait"])
                    u0 = [interface.get_solution(i) for i in range(12)]
                    lat.append(time.perf_counter() - t1)
                lat = np.array(lat[20:]) * 1e3
                tick.append((name, float(np.percentile(lat, 50)), float(np.percentile(lat, 99))))
            line["single_robot_tick_ms"] = {n: {"p50": a, "p99": b_} for n, a, b_ in tick}
            line["single_robot_tick_ms"]["note"] = "reference C boundary incl. Python/ctypes call overhead; deadline 2 ms (500 Hz)"
        except Exception as e:
            line["single_robot_tick_ms"] = {"unavailable": str(e)}
        # row f-1 variant of the end-to-end call: the caller hands over 352-byte robot states and the data
        # preparation (trajectory, foot positions, joint offsets) runs on the device (hmpc_solve_batch_states)
        states = scenarios.make_states(inputs, N)
        for _ in range(W):
            mpc.solve_batch_states(states, out=(out_w, out_s))
        t1 = time.perf_counter()
        for _ in range(K):
            mpc.solve_batch_states(states, out=(out_w, out_s))
        dt_states = time.perf_counter() - t1
        assert (interface.status_code(out_s) == 0).all()
        line["e2e_states"] = {"value": B * K / dt_states, "unit": UNIT, "ms_per_step": dt_states / K * 1e3,
                              "h2d_bytes_per_step": int(B * scenarios.STATE_DTYPE.itemsize), "d2h_bytes_per_step": int(B * (48 * N + 4)),
                              "note": "hmpc_solve_batch_states: updateMPCIfNeeded's data preparation on the device (SURVEY 8f row f-1)"}
        # BASELINE configs[4]: 4096 robots, 200 consecutive ticks, closed loop resident on the device (row f-3):
        # per tick prepare -> classify -> solve -> advance, nothing crosses PCIe inside the timed region
        try:
            Bc, Tc = 4096, 200
            _, cin = scenarios.make_batch(5, Bc, horizon=N, seed=4242)
            cst, clo = scenarios.make_rollout(cin, N)
            mpc5 = interface.BatchedMPC(Bc, N, device=local_rank)
            h_st = torch.from_numpy(cst.view(np.uint8).reshape(Bc, -1).copy())
            h_lo = torch.from_numpy(clo.view(np.uint8).reshape(Bc, -1).copy())
            d_cst, d_clo = h_st.cuda(), h_lo.cuda()
            mpc5.rollout_device(d_cst, d_clo, Bc, 10)  # warm-up ticks
            d_cst.copy_(h_st); d_clo.copy_(h_lo)
            torch.cuda.synchronize()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(stream)
            mpc5.rollout_device(d_cst, d_clo, Bc, Tc)
            c1.record(stream)
            torch.cuda.synchronize()
            ms5 = c0.elapsed_time(c1)
            lo5 = d_clo.cpu().numpy().view(scenarios.ROLLOUT_DTYPE).reshape(Bc)
            z5 = d_cst.cpu().numpy().view(scenarios.STATE_DTYPE).reshape(Bc)["position"][:, 2]
            line["closed_loop"] = {"workload": "configs[4]: batch=4096 walking robots, 200 consecutive ticks with warm start (previous tick's working set proposed), loop resident on the device",
                                   "value": Bc * Tc / (ms5 * 1e-3), "unit": UNIT, "ms_per_tick": ms5 / Tc, "failures": int(lo5["failures"].sum()),
                                   "mean_working_set_changes": float(lo5["iters_total"].sum() / lo5["ticks"].sum()),
                                   "mean_working_set_changes_note": "changes relative to the warm-start proposal (a cold start installs ~12 rows per tick)",
                                   "body_height_min_max": [float(z5.min()), float(z5.max())]}
            mpc5.close()
        except Exception as e:
            line["closed_loop"] = {"unavailable": str(e)}
        # other BASELINE configs on this GPU, device-resident, short runs (extra keys): configs[2]'s mix at 8192 robots and
        # the horizon-16 extension at 4096
        extra = {}
        for name, cfg_x, Bx, Nx in (("configs2_mix_8192_robots", 3, 8192, 10), ("configs3_horizon16_4096_robots", 4, 4096, 16),
                                    ("configs3_horizon5_4096_robots", 4, 4096, 5)):
            try:
                rx, _ = scenarios.make_batch(cfg_x, Bx, horizon=Nx)
                mx = interface.BatchedMPC(Bx, Nx, device=local_rank)
                px = torch.from_numpy(interface.pack_records(rx, Nx)).cuda()
                wx = torch.zeros((Bx, 12 * Nx), dtype=torch.float32, device="cuda")
                sx = torch.zeros((Bx,), dtype=torch.int32, device="cuda")
                for _ in range(2):
                    mx.solve_device(px, Bx, wx, sx)
                torch.cuda.synchronize()
                x0e, x1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                x0e.record(stream)
                for _ in range(5):
                    mx.solve_device(px, Bx, wx, sx)
                x1e.record(stream)
                torch.cuda.synchronize()
                msx = x0e.elapsed_time(x1e) / 5
                codes = np.bincount(interface.status_code(sx.cpu().numpy()), minlength=5)
                extra[name] = {"value": Bx / (msx * 1e-3), "unit": UNIT, "ms_per_step": msx, "not_converged": int(codes[1:].sum())}
                mx.close()
            except Exception as e:
                extra[name] = {"unavailable": str(e)}
        line["other_configs"] = extra
    if not args.no_cpu_baseline and world == 1:
        try:
            from oracle import oracle_py as O

            if O.has_qpoases():
                cq, cores, lat, win, per_core = cpu_reference_leg(recs, 10, 2, window_s=1.0)
                line["cpu_baseline"] = cpu_baseline_entry(cq, cores, lat, win, per_core, 10)
        except Exception as e:  # the baseline is reported, never required for the GPU number
            line["cpu_baseline"] = {"unavailable": str(e)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
