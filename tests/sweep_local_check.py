"""Learners that train alone under a process group (not collected by pytest; tests/test_gpu_sweep.py runs it under torchrun
with two ranks, which may share one GPU):

    python -m torch.distributed.run --standalone --nnodes=1 --nproc-per-node 2 tests/sweep_local_check.py

Every rank builds runs whose learners are Learner(data_parallel=False) in a gloo process group of two ranks: no peer
exchange, the one-launch fit, a RunBatch accepted.  Between two barriers the ranks train different numbers of updates
-- a data-parallel learner would wait in a collective for the rank that stopped -- and both reach the second barrier.
A RunBatch of a data-parallel learner is still refused."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import nfsp_b200  # noqa: E402
from nfsp_b200.learner import Learner  # noqa: E402
from nfsp_b200.runs import RunBatch  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
dev = torch.device("cuda", local % torch.cuda.device_count())
torch.cuda.set_device(dev)
dist.init_process_group("gloo")
assert world == 2


def run(seed, **kw):
    sp = nfsp_b200.SelfPlay(2048, seed=seed, device=dev, eta=0.3, epsilon=0.2, rl_capacity=1 << 14, sl_capacity=1 << 12,
                            max_steps_per_call=8, deterministic=True)
    return sp, Learner(sp, target_update_rate=2, **kw)


sp, ln = run(10 + rank, data_parallel=False)
assert ln._peers is None and ln.one_launch and not ln.data_parallel
rb = RunBatch(*zip(*[run(20 + 2 * rank + k, data_parallel=False) for k in range(2)]))
dist.barrier()
trained, n_trained = 0, 0
for it in range(3 + 5 * rank):   # rank 0: 3 iterations, rank 1: 8
    sp.rollout(8)
    mask = ln.update(sync=it % 2 == 0)["trained"]
    trained, n_trained = trained | mask, n_trained + (mask != 0)
    rb.step(8, sync=it % 3 == 0)
torch.cuda.synchronize()
assert trained == 0xF and ln.updates == n_trained >= 2 + 5 * rank, (trained, ln.updates)
assert all(m.updates >= 2 + 5 * rank for m in rb.learners)
dist.barrier()

# a data-parallel learner (the default) in a batch under a process group of two ranks: refused
sp2 = nfsp_b200.SelfPlay(256, seed=1, device=dev, rl_capacity=1 << 12, sl_capacity=1 << 12, max_steps_per_call=8)
try:
    RunBatch([sp2], [Learner(sp2, fused=False)])
    raise AssertionError("a RunBatch accepted a data-parallel learner with world 2")
except ValueError as e:
    assert "data_parallel" in str(e), e
dist.barrier()
if rank == 0:
    print("sweep local check ok: world", world)
dist.destroy_process_group()
