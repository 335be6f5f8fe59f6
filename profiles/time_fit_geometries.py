"""Device time of the one-launch fit (nfsp_learner_fit, nfsp_learner_fit_runs) per batch geometry, and of
nfsp_sample_indices, through the C ABI only -- so the same script times any build of the library.

    python profiles/time_fit_geometries.py [--root TREE] [--iters 200]

TREE (default: this repository) is the tree whose package and libnfsp_b200.so are loaded.  Geometries: the learner's
default (minibatch 128, fit batch 32: row-parallel kernel) and two that run the register kernel (minibatch 512 with fit
batch 32; minibatch 128 with fit batch 128), two epochs each; one run and 8 runs per launch.  65 536 games, two rollouts
of 8 steps fill the memories.  Each figure is CUDA events around `--iters` back-to-back launches, after 20 warm-up
launches.  Prints one JSON line."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--iters", type=int, default=200)
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))

import torch  # noqa: E402

import nfsp_b200  # noqa: E402
from nfsp_b200.batched import _ptr, _stream  # noqa: E402
from nfsp_b200.learner import Learner  # noqa: E402

if not torch.cuda.is_available():
    raise SystemExit("time_fit_geometries.py measures on the GPU: no CUDA device")
lib = nfsp_b200.lib()
dev = torch.device("cuda", 0)
sp = nfsp_b200.SelfPlay(65536, seed=1234, rl_capacity=200000, sl_capacity=2000000, max_steps_per_call=8)
for _ in range(2):
    sp.rollout(8)


def timed(fn, iters):
    for _ in range(20):
        nfsp_b200._lib.check(fn())
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


out = {"card": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip(), "root": os.path.abspath(args.root)}
st = _stream(dev)
for mb, fb in ((128, 32), (512, 32), (128, 128)):
    ln = Learner(sp, minibatch=mb, fit_batch=fb, epochs=2)
    idx_rl, idx_sl = ln._sample_positions()
    io = ln._io(idx_rl, idx_sl, 0, mb, 15)
    lr = (C.c_float * 4)(0.1, 0.05, 0.1, 0.05)
    w_out = torch.empty_like(sp.weights)  # the acting nets stay as they are: every launch fits the same inputs
    out["fit_%d_%d_ms" % (mb, fb)] = timed(lambda: lib.nfsp_learner_fit(C.byref(io), mb, fb, 2, lr, _ptr(w_out), st),
                                           args.iters)
    R = 8
    ios = (nfsp_b200._lib.LearnerIO * R)(*([io] * R))
    lrs = (C.c_float * (4 * R))(*(list(lr) * R))
    outs = [torch.empty_like(sp.weights) for _ in range(R)]
    ptrs = (C.c_void_p * R)(*[o.data_ptr() for o in outs])
    out["fit_runs8_%d_%d_ms" % (mb, fb)] = timed(lambda: lib.nfsp_learner_fit_runs(ios, R, mb, fb, 2, lrs, ptrs, st),
                                                 args.iters)
mem = sp.rl[0]
for b in (256, 1024):
    idx = torch.empty(b, dtype=torch.int64, device=dev)
    n = torch.empty(1, dtype=torch.int32, device=dev)
    out["sample_indices_%d_ms" % b] = timed(lambda: lib.nfsp_sample_indices(mem.seed, 0, _ptr(mem.total), mem.capacity, 1, b,
                                                                           _ptr(idx), _ptr(n), st), args.iters)
torch.cuda.synchronize()
print(json.dumps(out))
