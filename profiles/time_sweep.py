"""A sweep's runs spread over ranks (main.py --sweep): iterations per second for one rank and for W ranks.

    python profiles/time_sweep.py --out DIR [--runs 32] [--worlds 1,8] [--games 65536] [--iters 200] [--warmup 20]

For every world size W the script starts W ranks under torch.distributed.run (gloo, as main.py --sweep does; rank r on
cuda:(r % the visible GPUs)).  Each rank builds its contiguous block of the `--runs` runs (sweep.rank_runs) as one
RunBatch as main.py --sweep builds it without --deterministic (config.ini capacities, Learner(data_parallel=False)), trains
`--warmup` iterations, then times `--iters` iterations with a host clock around work that ends in a device synchronise,
and then one report's host work: read_stats and the exact exploitability of each of its runs.  The slowest rank's times
count.  The card's name and power limit are read in the same call.  Writes DIR/time_sweep.json and DIR/time_sweep.txt."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def rank_main(a):
    import torch
    import torch.distributed as dist

    import nfsp_b200
    from nfsp_b200 import sweep
    from nfsp_b200.learner import Learner
    from nfsp_b200.runs import RunBatch

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")) % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("gloo")
    sweep.check_layout(a.runs, world)
    pairs = []
    for i in sweep.rank_runs(a.runs, rank, world):
        sp = nfsp_b200.SelfPlay(a.games, seed=1234 + i, device=dev, eta=0.1, epsilon=0.06, rl_capacity=200000,
                                sl_capacity=2000000, max_steps_per_call=8, direct_rings="auto")
        pairs.append((sp, Learner(sp, data_parallel=False)))
    rb = RunBatch(*zip(*pairs))
    for _ in range(a.warmup):
        rb.step(8)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(a.iters):
        rb.step(8)
    torch.cuda.synchronize(dev)
    step_s = (time.perf_counter() - t0) / a.iters
    t0 = time.perf_counter()
    rb.update(sync=True)
    for sp in rb.sps:
        sp.read_stats()
    rb.exploitability()
    report_s = time.perf_counter() - t0
    mine = dict(rank=rank, runs=rb.n_runs, step_ms=1e3 * step_s, report_s=report_s)
    rows = [mine]
    if world > 1:
        rows = [None] * world
        dist.all_gather_object(rows, mine)
        dist.destroy_process_group()
    if rank == 0:
        print("RESULT " + json.dumps(rows))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--runs", type=int, default=32)
    ap.add_argument("--worlds", default="1,8")
    ap.add_argument("--games", type=int, default=1 << 16)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rank-main", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.rank_main:
        return rank_main(a)
    import torch

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()
    out = dict(card=card, gpus=torch.cuda.device_count(), runs=a.runs, games=a.games, iters=a.iters, results=[])
    lines = ["%d runs of %d games; card %s; %d GPU(s) visible" % (a.runs, a.games, card[:1], out["gpus"])]
    for w in [int(x) for x in a.worlds.split(",")]:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nnodes=1", "--nproc-per-node", str(w),
               os.path.abspath(__file__), "--rank-main", "--runs", str(a.runs), "--games", str(a.games),
               "--iters", str(a.iters), "--warmup", str(a.warmup)]
        p = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=3600)
        res = [ln for ln in p.stdout.splitlines() if ln.startswith("RESULT ")]
        if p.returncode != 0 or not res:
            raise SystemExit("world %d failed:\n%s\n%s" % (w, p.stdout[-3000:], p.stderr[-3000:]))
        ranks = json.loads(res[-1][len("RESULT "):])
        step_ms = max(r["step_ms"] for r in ranks)
        report_s = max(r["report_s"] for r in ranks)
        row = dict(world=w, ranks=ranks, step_ms=step_ms, iters_per_s=1e3 / step_ms,
                   run_iters_per_s=a.runs * 1e3 / step_ms, report_s=report_s)
        out["results"].append(row)
        lines.append("W = %d: %.3f ms per iteration of every run (slowest rank), %.1f iterations/s, %.0f run-iterations/s;"
                     " one report's host work %.2f s" % (w, step_ms, row["iters_per_s"], row["run_iters_per_s"], report_s))
    print("\n".join(lines))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "time_sweep.json"), "w") as f:
            json.dump(out, f, indent=1)
        with open(os.path.join(a.out, "time_sweep.txt"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
