"""Where Learner.update() goes on one GPU: device time of its pieces (CUDA events) and host time of the whole call.

    python profiles/time_learner.py
"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import nfsp_b200  # noqa: E402
from nfsp_b200.learner import Learner  # noqa: E402

n, T = 1 << 20, 8
sp = nfsp_b200.SelfPlay(n, seed=1234, rl_capacity=1 << 25, sl_capacity=1 << 23, max_steps_per_call=T)
for _ in range(3):
    sp.rollout(T)
L = Learner(sp, cfg=nfsp_b200.load_config(None))
for _ in range(3):
    L.update()
ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
acc = {}
for it in range(10):
    torch.cuda.synchronize()
    marks, names = [ev()], []
    marks[0].record()
    idx_rl, idx_sl = L._sample_positions()
    marks.append(ev()); marks[-1].record(); names.append("positions of the 4 minibatches")
    L._fit_one_launch(idx_rl, idx_sl, 15)
    marks.append(ev()); marks[-1].record(); names.append("fit kernel (8 SGD steps)")
    for row0 in range(0, 32, 32):
        L._step(idx_rl, idx_sl, row0, 32, 15)
    marks.append(ev()); marks[-1].record(); names.append("one grads + apply step")
    sp.set_weights(sp.weights)
    marks.append(ev()); marks[-1].record(); names.append("set_weights (3 pack kernels)")
    torch.cuda.synchronize()
    for k, name in enumerate(names):
        acc.setdefault(name, []).append(marks[k].elapsed_time(marks[k + 1]) * 1e3)
    t0 = time.perf_counter()
    L.update(sync=False)
    acc.setdefault("host time of update(sync=False)", []).append((time.perf_counter() - t0) * 1e6)
    torch.cuda.synchronize()
for k, v in acc.items():
    print("%-34s %8.1f us" % (k, sum(v[2:]) / len(v[2:])))
