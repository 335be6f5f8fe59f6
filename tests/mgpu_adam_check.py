"""Two or more GPUs of one box (not collected by pytest; run it under torchrun):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/mgpu_adam_check.py

Adam through the peer exchange (nfsp_learner_fit_peers_adam) against Adam through one NCCL all-reduce per step
(nfsp_learner_grads + all-reduce + nfsp_adam_apply) on identical memories: the weights and moments of the peer path
are bit-identical on every rank, and both paths agree to fp32 rounding of the order the ranks' gradients are summed in."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import nfsp_b200  # noqa: E402
from nfsp_b200.learner import Learner  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
n, steps = 4096, 8


def filled():
    sp = nfsp_b200.SelfPlay(n, seed=5, game0=rank * n, device=dev, eta=0.3, epsilon=0.2, rl_capacity=1 << 16,
                            sl_capacity=1 << 16, max_steps_per_call=steps, deterministic=True)
    for _ in range(4):
        sp.rollout(steps)
    return sp


a, b = filled(), filled()
La = Learner(a, fused=True, optimizer="adam", lr_br=0.002, lr_ar=0.001)
Lb = Learner(b, fused=False, optimizer="adam", lr_br=0.002, lr_ar=0.001)
assert La._peers is not None, getattr(La, "_peer_note", "no peers")


def same_on_every_rank(x, what):
    ref = x.clone()
    dist.broadcast(ref, 0)
    assert torch.equal(x, ref), "peer path: %s differs between ranks" % what


for k in range(4):
    ra, rb = La.update(), Lb.update()
    assert ra["trained"] == rb["trained"] == 0xF and La.adam_t == Lb.adam_t == [8 * (k + 1)] * 4
    for x, what in ((a.weights, "weights"), (La.adam_m, "m"), (La.adam_v, "v"), (b.weights, "NCCL-path weights")):
        same_on_every_rank(x, what)
    d = (a.weights - b.weights).abs().max().item()
    assert d <= 1e-3 * 0.002 * La.adam_t[0], (k, d)
assert int(La._peer_err.item()) == 0
if rank == 0:
    print("mgpu adam check ok: world", world)
dist.destroy_process_group()
