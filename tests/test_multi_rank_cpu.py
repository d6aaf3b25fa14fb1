"""world_size-2 (and 3) gloo tests of the multi-GPU host logic: shard bounds and the all_gather + point-sum of the
per-rank partials.  The per-rank MSMs are produced by the CPU oracle here (no GPU in this container); the exchange and
the summation are the product's (proof_systems_b200.parallel, zk_jacobian_sum)."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, n, q):
    import sys
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import srs_fixture
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import proof_systems_b200 as zk
    from oracle import oracle as orc
    from proof_systems_b200.parallel import all_gather_point_sum, shard_bounds
    z = srs_fixture.load("vesta", n)
    g = orc.decompress(orc.VESTA, z["g_cmp"][:n].tobytes())
    sc = orc.random_scalars(orc.FP, n, seed=3)
    lo, hi = shard_bounds(n, world, rank)
    _, jac = orc.msm(orc.VESTA, g[lo:hi], sc[lo:hi], want_jac=True)       # stand-in for this rank's GPU partial
    total = all_gather_point_sum(zk.VESTA, jac)
    aff = zk.jacobian_to_affine(zk.VESTA, total)
    want = orc.msm(orc.VESTA, g, sc)
    q.put((rank, bool(np.array_equal(aff, want)), aff.tobytes()))
    dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 1000), (3, 257)])
def test_all_gather_point_sum_identical_on_every_rank(world, n):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    assert all(ok for _, ok, _ in res)
    assert len({b for _, _, b in res}) == 1      # identical bits on every rank


def test_shard_bounds_partition():
    from proof_systems_b200.parallel import shard_bounds
    for n in (0, 1, 7, 64, 1000, 1 << 20):
        for world in (1, 2, 3, 4, 8):
            b = [shard_bounds(n, world, r) for r in range(world)]
            assert b[0][0] == 0 and b[-1][1] == n
            assert all(b[i][1] == b[i + 1][0] for i in range(world - 1))
            sizes = [hi - lo for lo, hi in b]
            assert max(sizes) - min(sizes) <= 1
