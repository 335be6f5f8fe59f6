"""SGD against Adam on the B200: the fit's time, an iteration's time, and what each learns in a sweep.

    python profiles/time_adam.py --out DIR [--games 65536] [--reps 200] [--episodes 3000000000] [--report-every 1000]

1. Fit time at the default geometry (minibatch 128, fit batch 32, 2 epochs: 8 steps, the row-parallel kernel) on memories
   filled by a rollout of `--games` games: one run's one-launch fit (Learner._fit_one_launch on fixed sampled rows), and
   RunBatch.update() of 32 runs (one sampling launch, one fit launch of 128 CTAs, the host schedules).  CUDA events around
   `--reps` calls, SGD and Adam alternating five times; the median of the five is reported.
2. One iteration of the sequential training loop (rollout(8) + Learner.update()) of one run with each optimizer, timed the
   same way.
3. Learning: main.py --sweep at `--games` games, the same --episodes for every sweep, 3 seeds per point: SGD at
   config.ini's rates (LearningRateBR 0.05, LearningRateAR 0.1), Adam at those rates, and Adam at
   LearningRateBR x LearningRateAR in {1e-3, 1e-4}^2.  Every report row's exact exploitability is kept with its hand
   count and the wall time since the sweep started (transitions / transitions_per_sec of the row).
The card's name and power limit are read in the same call.  Writes DIR/time_adam.json and DIR/time_adam.txt."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _events(fn, reps):
    import torch

    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) * 1000.0 / reps   # us per call


def _alternate(fns, reps, rounds=5):
    """{name: median us per call} over `rounds` rounds that run every fn once each, in turn."""
    times = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            times[k].append(_events(fn, reps))
    return {k: statistics.median(v) for k, v in times.items()}


def timings(a):
    import torch

    import nfsp_b200
    from nfsp_b200.learner import Learner
    from nfsp_b200.runs import RunBatch

    dev = torch.device("cuda", 0)

    def selfplay(seed):
        sp = nfsp_b200.SelfPlay(a.games, seed=seed, device=dev, rl_capacity=200000, sl_capacity=2000000,
                                max_steps_per_call=8, direct_rings="auto")
        for _ in range(4):
            sp.rollout(8)
        return sp

    out = {}
    # 1a. one run's fit
    fits = {}
    for opt in ("sgd", "adam"):
        sp = selfplay(1234)
        ln = Learner(sp, optimizer=opt)
        mask = ln._ready_mask()
        assert mask == 15, mask
        idx_rl, idx_sl = ln._sample_positions()
        w_out = sp.weights.clone()
        fits[opt] = (lambda ln=ln, i=(idx_rl, idx_sl), w=w_out: ln._fit_one_launch(i[0], i[1], 15, w_out=w))
        for _ in range(20):
            fits[opt]()
    torch.cuda.synchronize()
    out["fit_us"] = _alternate(fits, a.reps)
    # 1b. RunBatch.update() of 32 runs
    batches = {}
    for opt in ("sgd", "adam"):
        pairs = []
        for r in range(32):
            sp = nfsp_b200.SelfPlay(a.games, seed=1234 + r, device=dev, rl_capacity=200000, sl_capacity=2000000,
                                    max_steps_per_call=8, direct_rings="auto")
            pairs.append((sp, Learner(sp, optimizer=opt)))
        rb = RunBatch(*zip(*pairs))
        for _ in range(4):
            rb.rollout(8)
        batches[opt] = rb
        for _ in range(10):
            rb.update()
    torch.cuda.synchronize()
    out["runs32_update_us"] = _alternate({k: rb.update for k, rb in batches.items()}, max(a.reps // 4, 10))
    del batches
    # 2. one iteration of the sequential loop
    loops = {}
    for opt in ("sgd", "adam"):
        sp = selfplay(4321)
        ln = Learner(sp, optimizer=opt)

        def it(sp=sp, ln=ln):
            sp.rollout(8)
            ln.update(sync=False)
        for _ in range(20):
            it()
        loops[opt] = it
    torch.cuda.synchronize()
    out["iteration_us"] = _alternate(loops, a.reps)
    return out


SWEEPS = {
    "sgd-config-rates": ["--optimizer", "sgd", "--sweep", "Seed=1234"],
    "adam-config-rates": ["--optimizer", "adam", "--sweep", "Seed=1234"],
    "adam-small-rates": ["--optimizer", "adam", "--sweep", "LearningRateBR=0.001,0.0001",
                         "--sweep", "LearningRateAR=0.001,0.0001"],
}


def learning(a):
    from nfsp_b200 import main as drv

    res = {}
    for name, args in SWEEPS.items():
        rows = drv.main(["--games", str(a.games), "--episodes", str(a.episodes), "--report-every", str(a.report_every),
                         "--runs", "3", "--results", os.path.join(a.out, "sweep_%s.jsonl" % name)] + args)
        runs = [r for r in rows if r["kind"] == "run"]
        points = {}
        for r in runs:
            p = points.setdefault(r["point"], dict(hparams=r["hparams"], seeds=[], curve={}))
            if r["seed"] not in p["seeds"]:
                p["seeds"].append(r["seed"])
            p["curve"].setdefault(r["calls"], []).append(
                dict(seed=r["seed"], hands=r["hands"], seconds=r["transitions"] / r["transitions_per_sec"],
                     exploitability=r["exploitability"]["value"]))
        res[name] = list(points.values())
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--games", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--episodes", type=int, default=3_000_000_000)
    ap.add_argument("--report-every", type=int, default=1000)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()
    out = dict(card=card, games=a.games, reps=a.reps, episodes=a.episodes)
    out.update(timings(a))
    out["learning"] = learning(a)
    lines = ["card %s; %d games per run" % (card[:1], a.games),
             "one run's fit (8 steps): SGD %.1f us, Adam %.1f us" % (out["fit_us"]["sgd"], out["fit_us"]["adam"]),
             "RunBatch.update() of 32 runs: SGD %.1f us, Adam %.1f us" % (out["runs32_update_us"]["sgd"],
                                                                          out["runs32_update_us"]["adam"]),
             "one iteration (rollout(8) + update): SGD %.1f us, Adam %.1f us" % (out["iteration_us"]["sgd"],
                                                                                 out["iteration_us"]["adam"]),
             "exact exploitability (chips/hand), mean over seeds [min, max], at each report:"]
    for name, points in out["learning"].items():
        for p in points:
            lines.append("%s %s (seeds %s):" % (name, json.dumps(p["hparams"], sort_keys=True), p["seeds"]))
            for calls in sorted(p["curve"]):
                e = [x["exploitability"] for x in p["curve"][calls]]
                lines.append("  calls %6d  hands %.3e  %7.1f s  %.4f [%.4f, %.4f]" % (
                    calls, min(x["hands"] for x in p["curve"][calls]), max(x["seconds"] for x in p["curve"][calls]),
                    statistics.fmean(e), min(e), max(e)))
    with open(os.path.join(a.out, "time_adam.json"), "w") as f:
        json.dump(out, f, indent=1)
    with open(os.path.join(a.out, "time_adam.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines[:5]))


if __name__ == "__main__":
    main()
