"""Independent runs side by side (nfsp_b200.runs.RunBatch) against the same runs stepped one after another.

    python profiles/time_runs.py --out DIR [--runs 1,2,4,8,16,32] [--games 65536] [--iters 20] [--reps 5]

One self-play iteration of a run = rollout(8) + the insert of its records + Learner.update(), at `--games` games per run
with main.py's configuration (config.ini capacities, staged records).  For every R both forms train R fresh runs to the
steady state (every memory past a minibatch), then alternate: `--iters` iterations of the batched form, `--iters` of the
sequential one, `--reps` times, timed with CUDA events around the whole host loop (what a user waits for).  A second,
separate pass per form runs torch.profiler over a few iterations and lists the device time per kernel, the inserts'
share among them.  The card's name and power limit are read in the same call.  Writes DIR/time_runs.json and
DIR/time_runs.txt."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import nfsp_b200  # noqa: E402
from nfsp_b200.learner import Learner  # noqa: E402
from nfsp_b200.runs import RunBatch  # noqa: E402

STEPS = 8


def make_runs(R, games, seed0):
    out = []
    for r in range(R):
        sp = nfsp_b200.SelfPlay(games, seed=seed0 + r, eta=0.1, epsilon=0.06, rl_capacity=200000, sl_capacity=2000000,
                                max_steps_per_call=STEPS)
        out.append((sp, Learner(sp)))
    return out


def step_sequential(runs):
    for sp, ln in runs:
        sp.rollout(STEPS)
        ln.update(sync=False)


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def kernel_table(fn, iters):
    """{kernel name: (device ms per iteration, launches per iteration)} from torch.profiler over `iters` calls of fn."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0 and e.count > 0:
            out[e.key] = (t / 1000.0 / iters, e.count / iters)
    return out


def short(name):
    for k in ("rollout_states_kernel", "learner_fit_rows_runs_kernel", "learner_fit_rows_kernel", "insert_kernel",
              "sample_gather_wide_kernel", "sample_gather_kernel", "pack_images_kernel", "states_pack_kernel"):
        if k in name:
            return k + ("<runs>" if k == "rollout_states_kernel" and "RolloutRuns" in name else "")
    return name[:60]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", default="1,2,4,8,16,32")
    ap.add_argument("--games", type=int, default=65536)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile-runs", default="1,8,32")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_runs.py measures on the GPU: no CUDA device")
    os.makedirs(args.out, exist_ok=True)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                          capture_output=True, text=True).stdout.strip()
    res = {"card": card, "games_per_run": args.games, "steps_per_rollout": STEPS, "iters": args.iters, "reps": args.reps,
           "rows": []}
    lines = [card, "", "ms per iteration of ALL R runs (rollout(8) + inserts + update), median over %d reps of %d iterations"
             % (args.reps, args.iters), "%4s %12s %12s %8s   %s" % ("R", "batched", "sequential", "speedup", "spread (min-max) b / s")]
    prof_runs = {int(x) for x in args.profile_runs.split(",") if x}
    for R in (int(x) for x in args.runs.split(",")):
        batch = make_runs(R, args.games, 1000)
        seq = make_runs(R, args.games, 1000)
        rb = RunBatch([sp for sp, _ in batch], [ln for _, ln in batch])
        for _ in range(3):  # warm-up: every memory past a minibatch, every launch shape seen
            rb.step(STEPS)
            step_sequential(seq)
        tb, ts = [], []
        for _ in range(args.reps):
            tb.append(timed(lambda: rb.step(STEPS), args.iters))
            ts.append(timed(lambda: step_sequential(seq), args.iters))
        row = {"R": R, "batched_ms": statistics.median(tb), "sequential_ms": statistics.median(ts), "batched_all": tb,
               "sequential_all": ts}
        row["speedup"] = row["sequential_ms"] / row["batched_ms"]
        if R in prof_runs:
            kb = kernel_table(lambda: rb.step(STEPS), 5)
            ks = kernel_table(lambda: step_sequential(seq), 5)
            row["kernels_batched"] = {short(k): v for k, v in kb.items()}
            row["kernels_sequential"] = {short(k): v for k, v in ks.items()}
        res["rows"].append(row)
        lines.append("%4d %12.3f %12.3f %8.2f   %.3f-%.3f / %.3f-%.3f" % (R, row["batched_ms"], row["sequential_ms"], row["speedup"],
                                                                         min(tb), max(tb), min(ts), max(ts)))
        print(lines[-1], flush=True)
        del rb, batch, seq
        torch.cuda.empty_cache()
    lines.append("")
    for row in res["rows"]:
        for form in ("batched", "sequential"):
            kt = row.get("kernels_" + form)
            if not kt:
                continue
            tot = sum(v[0] for v in kt.values())
            ins = sum(v[0] for k, v in kt.items() if "insert_kernel" in k)
            lines.append("R = %d, %s: device time per iteration %.3f ms in kernels; inserts %.3f ms (%.1f %%)"
                         % (row["R"], form, tot, ins, 100.0 * ins / max(tot, 1e-12)))
            for k, (t, c) in sorted(kt.items(), key=lambda kv: -kv[1][0]):
                lines.append("    %-40s %9.4f ms  %6.1f launches  %.4f ms each" % (k, t, c, t / max(c, 1e-12)))
    with open(os.path.join(args.out, "time_runs.json"), "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(args.out, "time_runs.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
