"""Regenerates tests/golden/qpoases_samples.npz (needs the oracle built with qpOASES, i.e. where oracle/Makefile
finds the original project's sources).

    python tests/golden/make_qpoases_samples.py

qpOASES' optimum (the reference's own solver, through the oracle) for exactly the inputs the solver-parity tests draw:
the full-size configs, the ragged contact schedules and the horizon sweep of tests/test_gpu_parity.py, the edge cases and
column-cache overflows of tests/test_kernel_source_on_host.py, and the fused torque epilogue of tests/test_leg_torques.py.
The inputs are seeded (scenarios.make_batch) and are not stored; a fingerprint of them is (<case>_inputs,
conftest.records_fingerprint), and the tests check it before they compare.  Solutions are stored as float32 (relative
rounding 6e-8, far below the 5e-6 .. 1e-4 bars they are held to; exact zeros of eliminated variables stay exact), with
qpOASES' return code per robot."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from hector_simulation_b200 import scenarios  # noqa: E402
from conftest import records_fingerprint  # noqa: E402
from oracle import oracle_py as O  # noqa: E402


def ragged_records(n, seed=5, N=10, fixed_edges=False):
    """Arbitrary ragged contact schedules (test_edge_cases_vs_oracle, test_solve_kernel_source_edge_cases)."""
    rng = np.random.default_rng(seed)
    recs = []
    if fixed_edges:
        b = scenarios.stand_inputs(N)
        b["gait"][:] = 0
        b2 = scenarios.stand_inputs(N)
        b2["gait"][:8] = 0
        recs = [scenarios.to_record(b, N), scenarios.to_record(b2, N)]
    for _ in range(n):
        table = (rng.random(2 * N) < 0.6).astype(np.int32)
        recs.append(scenarios.to_record(scenarios._random_state(rng, N, table, moving=True), N))
    return np.array(recs)


def sweep_records(N):
    """test_horizon_sweep_batch_4096: the strided sample of 4096 mixed robots."""
    recs, _ = scenarios.make_batch(4, 4096, horizon=N, seed=1000 + N)
    return recs[np.arange(3, 4096, 64 if N <= 10 else 128)]


def column_cache_records():
    """test_solve_kernel_source_working_sets_beyond_the_column_cache: walkers with 15, 16 and 19 active rows."""
    picks = ((1000, [780, 20]), (4000, [217]))
    return np.concatenate([scenarios.make_batch(2, 1024, horizon=10, seed=scenarios.config_seed(2) + off)[0][idx] for off, idx in picks])


def cases():
    """(name, records, horizon, stored columns): of the 1024 configs[1] robots only the first-step wrench is compared."""
    yield "full_cfg2", scenarios.make_batch(2, 1024, horizon=10)[0], 10, 12
    yield "full_cfg3", scenarios.make_batch(3, 8192, horizon=10)[0][np.arange(0, 8192, 16)], 10, None
    yield "ragged48", ragged_records(48), 10, None
    yield "edges8", ragged_records(6, fixed_edges=True), 10, None
    yield "column_cache", column_cache_records(), 10, None
    yield "torques256", scenarios.make_batch(3, 256, horizon=10, seed=31)[0], 10, 12
    for N in (5, 10, 16):
        yield "sweep_h%d" % N, sweep_records(N), N, None


def main():
    assert O.has_qpoases()
    out = {}
    for name, recs, N, cols in cases():
        q, info = O.solve_batch(recs, O.make_setup(N))
        out[name + "_q"] = q[:, :cols].astype(np.float32)
        out[name + "_rc"] = info[:, 0].astype(np.int8)
        out[name + "_inputs"] = records_fingerprint(recs)
        print(name, q.shape, "rc != 0:", int((info[:, 0] != 0).sum()))
    np.savez_compressed(os.path.join(HERE, "qpoases_samples.npz"), **out)


if __name__ == "__main__":
    main()
