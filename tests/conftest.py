import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def pytest_sessionstart(session):
    """A fresh checkout has no built libraries (they are git-ignored): build them once, the way the driver's build() does.
    On the GPU box the libraries travel with the snapshot, so nothing happens there."""
    lib = os.path.join(ROOT, "hector_simulation_b200", "libhector_mpc_b200.so")
    if os.path.exists(lib):
        return
    try:
        import __graft_entry__

        __graft_entry__.build()
    except Exception as e:  # the tests that need the library then fail with their own, more specific message
        print("conftest: __graft_entry__.build() failed: %r" % (e,))


def load_golden(name):
    from hector_simulation_b200.scenarios import UPDATE_DTYPE

    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    d = {k: z[k] for k in z.files}
    d["records"] = np.ascontiguousarray(d["records"]).view(UPDATE_DTYPE).reshape(-1)
    d["horizon"] = int(d["horizon"])
    return d


@pytest.fixture(scope="session")
def oracle():
    """The CPU oracle (test infrastructure).  Skips solver-dependent checks if qpOASES is not linked."""
    from oracle import oracle_py

    oracle_py.lib()
    return oracle_py


def records_fingerprint(records):
    """A few position-weighted sums over the records' inputs: tells whether two record arrays hold the same robots in the
    same order, robust to last-bit differences of the host's libm."""
    w = np.arange(1, len(records) + 1, dtype=np.float64)
    f = [np.tensordot(w, np.asarray(records[k], np.float64).reshape(len(records), -1), 1).sum()
         for k in ("p", "v", "q", "w", "r", "joint_angles", "yaw", "traj", "gait")]
    return np.array(f + [len(records)])


def qpoases_sample(name, records):
    """qpOASES' optimum (float32) and return code for the seeded inputs of case `name`, recorded through the oracle by
    tests/golden/make_qpoases_samples.py, so that solver-parity tests run where the reference's solver is not built.
    `records` are the inputs the test solves: they must be the ones the answers were recorded for."""
    z = np.load(os.path.join(GOLDEN, "qpoases_samples.npz"))
    want = z[name + "_inputs"]
    assert np.allclose(records_fingerprint(records), want, rtol=1e-6, atol=1e-6), ("inputs differ from the recorded case", name)
    return z[name + "_q"].astype(np.float64), z[name + "_rc"].astype(np.int32)


def reference_solve(oracle, records, setup, assembly_fp64=False):
    """For records a test cannot know in advance (they come out of the loop under test): qpOASES' optimum through the
    oracle where it is built with the original project's solver, elsewhere the exact optimum (tolerance 1e-12) of the same
    reduced QP from the fp64 referee oracle/qp_dual_active_set.py, which qpOASES matches to its termination tolerance.
    -> (q [n, 12N], info [n, 2] = {return code (0 = solved), working-set changes})."""
    if oracle.has_qpoases():
        q, info = oracle.solve_batch(records, setup, assembly_fp64)
        return q, info[:, :2]
    from oracle import qp_dual_active_set as G

    N = int(setup["horizon"][0])
    q = np.zeros((len(records), 12 * N))
    info = np.zeros((len(records), 2), np.int32)
    for i in range(len(records)):
        Q = oracle.reduced_qp(records[i], setup, assembly_fp64)
        if len(Q["var_ind"]):
            x, inf = G.solve(Q["H"], Q["g"], Q["A"], Q["lb"], Q["ub"], tol=1e-12, max_iter=3000)
            q[i, Q["var_ind"]] = x
            info[i] = inf["status"], inf["iters"]
    return q, info


def rel_err(a, b, width=None):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    if width is not None:
        a, b = a[:, :width], b[:, :width]
    return np.linalg.norm(a - b, axis=1) / np.maximum(np.linalg.norm(b, axis=1), 1e-9)
