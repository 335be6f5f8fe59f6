"""Save and load times and file sizes of checkpoints (nfsp_b200.checkpoint) at main.py's default shape.

    python profiles/time_checkpoint.py --out DIR [--reps 3] [--batch-runs 32] [--train-calls 10000]

One run = SelfPlay(65 536 games, MRLSize 200 000, MSLSize 2 000 000) + its Learner, every memory full (slots filled with
random words, `total` past the capacity): the file then holds 2 x 64 MB of reservoir slots, 2 x 3.2 MB of ring slots and
0.5 MB of game words.  Measured with a host clock around each call (state_dict() and load_state_dict() synchronise the
device): checkpoint.save into a temporary directory (state dicts, torch.save, fsync, rename) and checkpoint.load into a
fresh pair, `--reps` times; the same once for a RunBatch of `--batch-runs` runs when the temporary file system has room.
The checkpoint files are deleted; only the timings are written.

The cost of --checkpoint-every at its default: main.train's sequential loop (rollout(8), update, a report with the exact
exploitability every 100 calls) is timed over `--train-calls` calls at the same shape, and one save is charged to every
main.CHECKPOINT_EVERY calls of it.  The card's name and power limit are read in the same call.  Writes
DIR/time_checkpoint.json and DIR/time_checkpoint.txt."""
from __future__ import annotations

import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import nfsp_b200  # noqa: E402
from nfsp_b200 import checkpoint, main as drv  # noqa: E402
from nfsp_b200.learner import Learner  # noqa: E402
from nfsp_b200.runs import RunBatch  # noqa: E402

GAMES, RL, SL, STEPS = 65536, 200000, 2000000, 8


def make(seed=1234, fill=False):
    sp = nfsp_b200.SelfPlay(GAMES, seed=seed, rl_capacity=RL, sl_capacity=SL, max_steps_per_call=STEPS)
    if fill:
        g = torch.Generator(device=sp.device).manual_seed(seed)
        for m in sp.rl + sp.sl:
            m.store.copy_(torch.randint(-2 ** 31, 2 ** 31 - 1, m.store.shape, generator=g, device=sp.device,
                                        dtype=torch.int64).to(torch.int32))
            m.total.fill_(3 * m.capacity)
    return sp, Learner(sp, cfg=nfsp_b200.load_config(None))


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t


def dir_bytes(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--batch-runs", type=int, default=32)
    ap.add_argument("--train-calls", type=int, default=10000)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                          capture_output=True, text=True).stdout.strip()
    res = {"card": card, "games": GAMES, "MRLSize": RL, "MSLSize": SL, "checkpoint_every": drv.CHECKPOINT_EVERY}
    tmp_root = tempfile.mkdtemp(prefix="nfsp-ckpt-")
    try:
        # ---- one run ----
        sp, ln = make(fill=True)
        fresh = make(seed=1234)
        saves, loads, size = [], [], None
        for r in range(args.reps):
            d = os.path.join(tmp_root, "one-%d" % r)
            saves.append(timed(lambda: checkpoint.save(d, 1, selfplay=sp, learner=ln)))
            size = dir_bytes(d)
            loads.append(timed(lambda: checkpoint.load(d, selfplay=fresh[0], learner=fresh[1])))
            shutil.rmtree(d)
        res["one_run"] = {"save_s": saves, "load_s": loads, "bytes": size}
        del sp, ln, fresh
        torch.cuda.empty_cache()

        # ---- main.train's loop at the same shape: seconds per call ----
        sp, ln = make(seed=7)
        # a first short train() measures the hands per call, so that the timed one stops after about --train-calls calls
        r0 = drv.train(sp, ln, episodes=1, report_every=100, log=lambda *a, **k: None)
        hands_per_call = r0[-1]["hands"] / r0[-1]["calls"]
        sp, ln = make(seed=7)
        t = time.perf_counter()
        rows = drv.train(sp, ln, episodes=int(hands_per_call * args.train_calls), report_every=100,
                         log=lambda *a, **k: None)
        torch.cuda.synchronize()
        elapsed = time.perf_counter() - t
        calls = rows[-1]["calls"]
        per_call = elapsed / calls
        save = statistics.median(res["one_run"]["save_s"])
        res["train"] = {"calls": calls, "seconds": elapsed, "seconds_per_call": per_call, "hands_per_call": hands_per_call}
        res["share_at_default"] = save / (drv.CHECKPOINT_EVERY * per_call + save)
        res["calls_for_1_percent"] = 99.0 * save / per_call
        del sp, ln
        torch.cuda.empty_cache()

        # ---- a RunBatch ----
        R = args.batch_runs
        need = R * size * 1.1
        free = shutil.disk_usage(tmp_root).free
        if free < need:
            res["batch"] = {"runs": R, "not_measured": "%.1f GB free in %s, %.1f GB needed" % (free / 1e9, tmp_root, need / 1e9)}
        else:
            runs = [make(seed=100 + r, fill=True) for r in range(R)]
            rb = RunBatch([s for s, _ in runs], [l_ for _, l_ in runs])
            d = os.path.join(tmp_root, "batch")
            save_b = timed(lambda: checkpoint.save(d, 1, runs=rb))
            size_b = dir_bytes(d)
            del rb, runs
            torch.cuda.empty_cache()
            runs = [make(seed=100 + r) for r in range(R)]
            rb = RunBatch([s for s, _ in runs], [l_ for _, l_ in runs])
            load_b = timed(lambda: checkpoint.load(d, runs=rb))
            shutil.rmtree(d)
            # the batch's iteration time, for its share
            for _ in range(5):
                rb.step(STEPS)
            it_s = timed(lambda: [rb.step(STEPS) for _ in range(50)]) / 50
            res["batch"] = {"runs": R, "save_s": save_b, "load_s": load_b, "bytes": size_b, "seconds_per_call": it_s,
                            "share_at_default": save_b / (drv.CHECKPOINT_EVERY * it_s + save_b)}
    finally:
        shutil.rmtree(tmp_root, ignore_errors=True)
    with open(os.path.join(args.out, "time_checkpoint.json"), "w") as f:
        json.dump(res, f, indent=1)
    one = res["one_run"]
    lines = [card, "",
             "one run (65 536 games, memories full): file %.1f MB, save %s s, load %s s" %
             (one["bytes"] / 1e6, " ".join("%.3f" % x for x in one["save_s"]), " ".join("%.3f" % x for x in one["load_s"])),
             "main.train loop: %.3f ms per call over %d calls (report + exact exploitability every 100)" %
             (1e3 * res["train"]["seconds_per_call"], res["train"]["calls"]),
             "saving every %d calls: %.2f %% of training time; 1 %% needs >= %.0f calls between saves" %
             (drv.CHECKPOINT_EVERY, 100 * res["share_at_default"], res["calls_for_1_percent"])]
    b = res["batch"]
    if "not_measured" in b:
        lines.append("RunBatch of %d: not measured (%s)" % (b["runs"], b["not_measured"]))
    else:
        lines.append("RunBatch of %d: file %.2f GB, save %.2f s, load %.2f s; %.3f ms per iteration, saving every %d "
                     "calls: %.2f %%" % (b["runs"], b["bytes"] / 1e9, b["save_s"], b["load_s"], 1e3 * b["seconds_per_call"],
                                         drv.CHECKPOINT_EVERY, 100 * b["share_at_default"]))
    with open(os.path.join(args.out, "time_checkpoint.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
