"""Two GPUs of one box (not collected by pytest; run it under torchrun with a scratch directory):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/mgpu_checkpoint_check.py DIR

A deterministic 2-rank run with the peer exchange inside the fit, saved after k iterations and loaded into fresh objects
(fresh exchange buffers, epoch 0), equals the run that never stopped on every rank.  A checkpoint whose rank-1 file is
rank 0's is refused on both ranks, and neither rank's objects change."""
import os
import shutil
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import nfsp_b200  # noqa: E402
from nfsp_b200 import checkpoint  # noqa: E402
from nfsp_b200.learner import Learner  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
root = sys.argv[1]
n, k, K = 4096, 3, 7


def make():
    sp = nfsp_b200.SelfPlay(n, seed=5, game0=rank * n, device=dev, eta=0.3, epsilon=0.2, rl_capacity=1 << 15,
                            sl_capacity=1 << 13, max_steps_per_call=8, deterministic=True)
    ln = Learner(sp, target_update_rate=3)
    assert ln._peers is not None, getattr(ln, "_peer_note", "no peers")
    return sp, ln


def iterate(sp, ln, it):
    sp.rollout(8)
    return ln.update(sync=it % 2 == 0)


def same(a, b, la, lb, tag):
    torch.cuda.synchronize()
    assert torch.equal(a.env.state_words(), b.env.state_words()), tag
    assert a.env.step_counter == b.env.step_counter and torch.equal(a.stats, b.stats), tag
    for ma, mb in zip(a.rl + a.sl, b.rl + b.sl):
        assert torch.equal(ma.total, mb.total) and torch.equal(ma.store, mb.store), tag
        assert ma.sample_calls == mb.sample_calls, tag
    assert torch.equal(a.weights, b.weights) and a.epsilons == b.epsilons, tag
    assert torch.equal(la.target, lb.target), tag
    for f in ("iteration", "target_update_count", "temp", "lr_br", "exploitability", "updates"):
        assert getattr(la, f) == getattr(lb, f), (tag, f)


a, la = make()
b, lb = make()
for it in range(k):
    assert iterate(a, la, it) == iterate(b, lb, it)
d = os.path.join(root, "ck")
checkpoint.save(d, k, selfplay=b, learner=lb)
dist.barrier()
c, lc = make()
assert checkpoint.load(d, selfplay=c, learner=lc) == {"calls": k}
for it in range(k, K):
    assert iterate(a, la, it) == iterate(c, lc, it), it
    same(a, c, la, lc, "rank %d iteration %d" % (rank, it))
ref = a.weights.clone()
dist.broadcast(ref, 0)
assert torch.equal(ref, a.weights), "weights differ between ranks"

# rank 1's file replaced by rank 0's: both ranks refuse
bad = os.path.join(root, "bad")
if rank == 0:
    os.makedirs(bad)
    for r in range(world):
        shutil.copy(os.path.join(d, checkpoint.file_name(0, world)), os.path.join(bad, checkpoint.file_name(r, world)))
dist.barrier()
e, le = make()
before = (e.state_dict(), le.state_dict())
try:
    checkpoint.load(bad, selfplay=e, learner=le)
    raise AssertionError("rank %d loaded another rank's file" % rank)
except ValueError as err:
    print("rank %d refused: %s" % (rank, err))
after = (e.state_dict(), le.state_dict())
for x, y in zip(before, after):
    for key in x:
        if isinstance(x[key], torch.Tensor):
            assert torch.equal(x[key], y[key]), key
        elif key not in ("rl", "sl"):
            assert x[key] == y[key], key
for p in range(2):
    for m in ("rl", "sl"):
        assert torch.equal(before[0][m][p]["slots"], after[0][m][p]["slots"])
for L in (la, lb, lc, le):
    L.close_peers()
if rank == 0:
    print("mgpu checkpoint check ok: world", world)
dist.destroy_process_group()
