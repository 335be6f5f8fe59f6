"""world_size-2 gloo test (CPU) of the multi-GPU host logic: contiguous game sharding, the counter
all-reduce and max-over-ranks timing.  The data path itself has no collective (SURVEY 8e)."""
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import nfsp_b200
    from nfsp_b200 import sharding

    game0, n = sharding.shard_games(1_000_003, rank, world)
    stats = torch.zeros(16, dtype=torch.int64)
    stats[11] = n          # transitions
    stats[8] = -(rank + 1)  # a negative reward sum survives the reduction
    tot = sharding.allreduce_stats(stats)
    t = sharding.max_over_ranks(1.0 + rank)
    q.put((rank, game0, n, int(tot[11]), int(tot[8]), t))
    dist.destroy_process_group()


def test_sharding_two_ranks():
    with socket.socket() as s:  # a port nobody holds now: suites running side by side on one host must not collide
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in ps:
        p.start()
    res = sorted(q.get(timeout=120) for _ in ps)
    for p in ps:
        p.join(60)
        assert p.exitcode == 0
    (r0, g0, n0, tot0, rew0, t0), (r1, g1, n1, tot1, rew1, t1) = res
    assert g0 == 0 and g1 == n0 and n0 + n1 == 1_000_003 and abs(n0 - n1) <= 1
    assert tot0 == tot1 == 1_000_003 and rew0 == rew1 == -3 and t0 == t1 == 2.0


def test_shard_ranges_cover_exactly():
    sys.path.insert(0, ROOT)
    from nfsp_b200 import sharding

    for total in (1, 7, 8, 1 << 20, 8_388_608, 1_000_003):
        for world in (1, 2, 4, 8):
            ranges = [sharding.shard_games(total, r, world) for r in range(world)]
            assert ranges[0][0] == 0 and sum(n for _, n in ranges) == total
            for (a, n), (b, _) in zip(ranges[:-1], ranges[1:]):
                assert a + n == b
    with pytest.raises(ValueError):
        sharding.shard_games(10, 2, 2)
