"""CPU, world_size 2 over gloo: the multi-GPU path's host logic — sharding.ShardedMPC.tick / whole_batch, the very
functions bench.py drives on GPUs (contiguous equal slices, padded tail, this rank's slice back on its own arrays, ONE
all-gather of the float wrenches).  The backend differs: here the per-slice solve is stood in for by a lookup of the
committed qpOASES solutions of the same records (tests/golden/cfg3_h10.npz) and the gather goes through
torch.distributed/gloo instead of the library's ncclAllGather — what is under test is the partition / padding / ordering
logic, not a CPU product path."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import load_golden
from hector_simulation_b200 import sharding


def test_shard_bounds():
    assert sharding.shard_bounds(8192, 8) == [(i * 1024, (i + 1) * 1024) for i in range(8)]
    b = sharding.shard_bounds(10, 4)
    assert b == [(0, 3), (3, 6), (6, 9), (9, 10)]          # equal slices of ceil(B / world), the tail holds the rest
    assert sharding.shard_bounds(1, 2) == [(0, 1), (1, 1)]
    assert sharding.shard_bounds(0, 2) == [(0, 0), (0, 0)]


def _worker(rank, world, port, n, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = load_golden("cfg3_h10")
    recs = g["records"][:n]
    row = {recs[i].tobytes(): i for i in range(n)}

    def solve_local(r):
        # records that are not among the batch's (a padded tail) get a zero answer, which must never reach the results
        w = np.zeros((len(r), 120))
        s = np.zeros(len(r), np.int32)
        for k, x in enumerate(r):
            if x.tobytes() in row:
                w[k], s[k] = g["q_soln"][row[x.tobytes()]], g["info"][row[x.tobytes()], 1]
        return w, s

    from hector_simulation_b200 import scenarios

    sh = sharding.ShardedMPC(n, 10, rank, world, lambda b: sharding.TorchBackend(b, 10, world, solve_local), scenarios.UPDATE_DTYPE)
    mine = sh.local_slice(recs.view(scenarios.UPDATE_DTYPE).reshape(-1))
    ok = True
    for tick in range(2):                                     # two ticks through the same registered arrays:
        w_loc, s_loc = sh.tick(mine) if tick == 0 else sh.tick()  # records handed over, then left in place
        lo, hi = sh.bounds[rank]
        ok &= np.array_equal(w_loc, g["q_soln"][lo:hi]) and np.array_equal(s_loc, g["info"][lo:hi, 1])
        whole = sh.whole_batch()                              # every rank ends up with the whole batch, global order
        ok &= whole.shape == (n, 120) and np.array_equal(whole, g["q_soln"][:n].astype(np.float32))
    sh.close()
    q.put((rank, bool(ok)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("n", [7, 16])
def test_two_rank_shard_and_gather(n):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, n, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]
