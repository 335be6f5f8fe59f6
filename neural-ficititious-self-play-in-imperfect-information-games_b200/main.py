"""Drop-in for the reference's training driver (main.py:21-158), batched.

    python -m nfsp_b200.main [--games N] [--episodes E] [--steps-per-call T] [--config ./config.ini]
    python -m torch.distributed.run --nproc-per-node G -m nfsp_b200.main ...     # games sharded over G GPUs
    python -m nfsp_b200.main --runs R ...     # R independent runs (seeds Seed, Seed + 1, ...) side by side on one GPU
    python -m nfsp_b200.main --checkpoint DIR ...   # save the training state; --resume DIR continues it (DESIGN.md 7c)
    python -m torch.distributed.run --nproc-per-node G -m nfsp_b200.main --sweep Eta=0.05,0.1 --sweep LearningRateBR=0.01,0.05 \
        --runs R --results FILE ...   # a grid of settings x R seeds, independent runs spread over G ranks (DESIGN.md 7d)

A sweep (`--sweep KEY=V1,V2,...`, repeatable; the keys of sweep.RUN_KEYS, with or without their section) trains the
Cartesian product of the values given, each grid point with R seeds, as independent runs of `--games` games each.  The
ranks take contiguous blocks of runs, one RunBatch each, and never shard a run; rank r uses cuda:(LOCAL_RANK % the
number of visible GPUs), so several ranks may share a GPU.  Every report gathers every run's row on every rank, adds the
mean and standard deviation of the exact exploitability over each grid point's seeds, and rank 0 prints them and
appends them to `--results FILE` (JSON Lines).

The reference plays one hand at a time: `train(env, player1, player2)` alternates the dealer, draws each
player's per-hand policy with probability eta, lets the agents `play` until both have seen the terminal
state, calls `update_strategy()` every 128 decisions of an agent and prints the action histogram and the
exploitability proxy every 100 episodes (main.py:27-75, agent.py:153-154).  All of the per-hand control flow
lives inside the fused rollout kernel here (DESIGN.md section 1); this driver is the outer loop only:

    repeat:  rollout(T) for every game  ->  records into M_RL / M_SL  ->  Learner.update()  ->  stats

Same config.ini keys (config.ini:1-40, incl. MRLSize / MSLSize, which the reference defines but never
reads), same seeds, same printed quantities.  `--human` is accepted and ignored, as in the reference
(main.py:152-158).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import time

import torch
import torch.distributed as dist

from . import checkpoint as ckpt
from . import sharding, sweep
from .batched import SelfPlay
from .config import load_config
from .exploitability import exploitability
from .learner import OPTIMIZERS, Learner, PipelinedTrainer
from .runs import RunBatch


# rollout calls between two checkpoints: a save at the default shape (65 536 games, config.ini's memories, full: 135 MB,
# 0.17 s) then costs under 1 % of the training time (0.110 ms per call; B200 at 1000 W, DESIGN.md 7c)
CHECKPOINT_EVERY = 200000


def _is_report(calls, report_every):
    return calls % report_every == 0 or calls == 1


def _stopped(calls, report_every, hands, episodes):
    """Whether a run resumed at `calls` with `hands` played had stopped there: the loop ends at a report call."""
    return calls > 0 and _is_report(calls, report_every) and hands >= episodes


def _mark_optimizer(row, learner):
    """A reported row names the optimizer when it is not the reference's SGD (SGD rows stay as they always were)."""
    if learner.optimizer != "sgd":
        row["optimizer"] = learner.optimizer


def sampled_actions(stats, player):
    """agent.Agent.sampled_actions (agent.py:196-204): share of fold / call / raise among `player`'s actions."""
    a = [stats["a%d_%s" % (player, k)] for k in ("fold", "call", "raise")]
    tot = max(sum(a), 1)
    return [x / tot for x in a]


def train(sp: SelfPlay, learner: Learner, episodes: int, steps_per_call: int = 8, report_every: int = 100,
          world: int = 1, log=print, true_exploitability: bool = True, pipelined: bool = False, updates_per_call: int = 1,
          checkpoint=None, checkpoint_every: int = CHECKPOINT_EVERY, resume=None):
    """main.train (main.py:21-124).  Plays until `episodes` hands have finished over all games and ranks.
    Returns the list of reported rows (the reference's `plotter`, main.py:75, plus what it prints).
    pipelined: the learner's update runs beside the next rollout (learner.PipelinedTrainer: acting nets one update
    behind, the learner's time hidden).
    updates_per_call: update_strategy() calls per rollout call.  The reference updates an agent every 128 of ITS decisions
    (agent.py:153-154); a rollout call is n_games * steps_per_call / 2 decisions per agent, so the reference's cadence is
    updates_per_call = n_games * steps_per_call / 256 (sequential loop only).
    checkpoint: a directory; the training state is saved there every `checkpoint_every` calls and when training ends.
    resume: a checkpoint directory to load before the loop; training continues from its calls counter and hand count."""
    if pipelined and updates_per_call != 1:
        raise ValueError("the pipelined trainer runs one update beside each rollout")
    rows, calls, tr0 = [], 0, 0
    trainer = PipelinedTrainer(sp, learner) if pipelined else None
    objs = dict(selfplay=sp, learner=learner, trainer=trainer)
    if resume is not None:
        calls = ckpt.load(resume, **objs)["calls"]
        tot = dict(zip(sp.STAT_NAMES, sharding.allreduce_stats(sp.stats).tolist()))
        if _stopped(calls, report_every, tot["hands"], episodes):
            return rows
        tr0 = tot["transitions"]                  # the rate counts this process's transitions

    def save():
        if trainer is not None:
            trainer.finish()                      # waits for the update in flight; the next step acts as before
        ckpt.save(checkpoint, calls, **objs)

    t0 = time.time()
    while True:
        calls += 1
        report = _is_report(calls, report_every)
        if trainer is None:
            sp.rollout(steps_per_call)            # main.py:27-67 for every game, T decisions each
            for _ in range(updates_per_call - 1):
                learner.update(sync=False, pack=False)
            st = learner.update(sync=report)      # agent.py:153-154 -> 192-194 -> 209-264; host reads only when reporting
        else:
            st = trainer.step(steps_per_call, sync=report)
            if report:                            # the exact exploitability below is that of the newest nets
                trainer.finish()
        if not report:
            if checkpoint is not None and calls % checkpoint_every == 0:
                save()
            continue
        tot = sharding.allreduce_stats(sp.stats).tolist()
        stats = dict(zip(sp.STAT_NAMES, (int(v) for v in tot)))
        row = {"calls": calls, "hands": stats["hands"], "transitions": stats["transitions"],
               "exploitability_proxy": st.get("exploitability"),   # agent.py:234-238 summed over players, main.py:73
               "actions": [sampled_actions(stats, p) for p in range(2)],
               "transitions_per_sec": (stats["transitions"] - tr0) / max(time.time() - t0, 1e-9)}
        if true_exploitability:
            row["exploitability"] = exploitability(sp)  # exact best response to the average policies (SURVEY 8 f-2)
        _mark_optimizer(row, learner)
        rows.append(row)
        log("================ Stats ==================")
        for p in range(2):
            f, c, r = row["actions"][p]
            log("Player%d: fold %.3f call %.3f raise %.3f" % (p, f, c, r))
        log("Exploitability: {}".format(row["exploitability_proxy"]))
        if true_exploitability:
            log("Exact exploitability of the average policies: %.4f chips/hand" % row["exploitability"]["value"])
        log("hands %d  transitions %d  (%.3e transitions/s)" % (row["hands"], row["transitions"], row["transitions_per_sec"]))
        done = stats["hands"] >= episodes
        if checkpoint is not None and (done or calls % checkpoint_every == 0):
            save()
        if done:
            return rows


def train_runs(rb: RunBatch, episodes: int, steps_per_call: int = 8, report_every: int = 100, log=print,
               true_exploitability: bool = True, checkpoint=None, checkpoint_every: int = CHECKPOINT_EVERY, resume=None):
    """train() for the independent runs of a RunBatch: one batched iteration per call, until every run has played
    `episodes` hands.  A reported row carries each run's values under "runs" and, with true_exploitability, the mean
    and standard deviation of the runs' exact exploitability.  checkpoint / checkpoint_every / resume: as in train()."""
    rows, calls, tr0 = [], 0, 0
    if resume is not None:
        calls = ckpt.load(resume, runs=rb)["calls"]
        saved = [sp.read_stats() for sp in rb.sps]
        if _stopped(calls, report_every, min(s["hands"] for s in saved), episodes):
            return rows
        tr0 = sum(s["transitions"] for s in saved)
    t0 = time.time()
    while True:
        calls += 1
        report = _is_report(calls, report_every)
        sts = rb.step(steps_per_call, sync=report)
        if not report:
            if checkpoint is not None and calls % checkpoint_every == 0:
                ckpt.save(checkpoint, calls, runs=rb)
            continue
        runs = []
        for sp, st in zip(rb.sps, sts):
            stats = sp.read_stats()
            runs.append({"seed": sp.env.seed, "hands": stats["hands"], "transitions": stats["transitions"],
                         "exploitability_proxy": st.get("exploitability"),
                         "actions": [sampled_actions(stats, p) for p in range(2)]})
        row = {"calls": calls, "runs": runs, "hands": sum(r["hands"] for r in runs),
               "transitions": sum(r["transitions"] for r in runs)}
        row["transitions_per_sec"] = (row["transitions"] - tr0) / max(time.time() - t0, 1e-9)
        if true_exploitability:
            for run, e in zip(runs, rb.exploitability()):
                run["exploitability"] = e
            values = [r["exploitability"]["value"] for r in runs]
            row["exploitability_mean"] = statistics.fmean(values)
            row["exploitability_std"] = statistics.stdev(values) if len(values) > 1 else 0.0
        _mark_optimizer(row, rb.learners[0])
        rows.append(row)
        log("================ Stats ==================")
        for k, run in enumerate(runs):
            line = "run %d (seed %d): hands %d  exploitability proxy %s" % (k, run["seed"], run["hands"], run["exploitability_proxy"])
            if true_exploitability:
                line += "  exact exploitability %.4f chips/hand" % run["exploitability"]["value"]
            log(line)
        if true_exploitability:
            log("Exact exploitability over %d runs: mean %.4f  std %.4f chips/hand" %
                (len(runs), row["exploitability_mean"], row["exploitability_std"]))
        log("hands %d  transitions %d  (%.3e transitions/s)" % (row["hands"], row["transitions"], row["transitions_per_sec"]))
        done = min(r["hands"] for r in runs) >= episodes
        if checkpoint is not None and (done or calls % checkpoint_every == 0):
            ckpt.save(checkpoint, calls, runs=rb)
        if done:
            return rows


def _gather(obj):
    """[rank 0's obj, rank 1's obj, ...] over the process group (one all_gather_object), or [obj] without one."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return [obj]
    out = [None] * dist.get_world_size()
    dist.all_gather_object(out, obj)
    return out


def _keep_results(path, calls):
    """The results file as a run resumed at `calls` continues it: the lines of later reports dropped."""
    lines = []
    if os.path.exists(path):
        with open(path) as f:
            lines = [ln for ln in f if ln.strip() and json.loads(ln)["calls"] <= calls]
    with open(path, "w") as f:
        f.writelines(lines)


def _point_rows(run_rows, calls, true_exploitability):
    """One row per grid point: its runs and seeds and, with the exact exploitability, its mean and standard deviation
    over the seeds."""
    out = []
    for p in sorted({r["point"] for r in run_rows}):
        rs = [r for r in run_rows if r["point"] == p]
        row = {"kind": "point", "calls": calls, "point": p, "hparams": rs[0]["hparams"], "runs": [r["run"] for r in rs],
               "seeds": [r["seed"] for r in rs], "hands": min(r["hands"] for r in rs)}
        if true_exploitability:
            values = [r["exploitability"]["value"] for r in rs]
            row["exploitability_mean"] = statistics.fmean(values)
            row["exploitability_std"] = statistics.stdev(values) if len(values) > 1 else 0.0
        if "optimizer" in rs[0]:
            row["optimizer"] = rs[0]["optimizer"]
        out.append(row)
    return out


def train_sweep(rb: RunBatch, runs, record, episodes: int, steps_per_call: int = 8, report_every: int = 100, log=print,
                true_exploitability: bool = True, results=None, checkpoint=None, checkpoint_every: int = CHECKPOINT_EVERY,
                resume=None):
    """train_runs() for one rank's block of a sweep.  `runs` are the definitions (sweep.expand) of rb's runs in order,
    `record` the whole sweep's checkpoint record (sweep.record).  At a report call every rank evaluates its own runs
    (counters, the proxy, the exact exploitability) and one all_gather_object gives every rank every run's row, in run
    order, followed by one row per grid point (_point_rows); every rank returns the same rows and stops at the same call,
    once every run of the sweep has played `episodes` hands.  results: a file rank 0 writes those rows to as JSON Lines
    (on resume, first without the lines of reports after the checkpoint).  checkpoint / checkpoint_every / resume: as in
    train(); the file also holds `record`, and a resume of another sweep or world size is refused on every rank."""
    rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
    rows, calls, tr0 = [], 0, [0] * rb.n_runs
    if resume is not None:
        calls = ckpt.load(resume, runs=rb, sweep=record)["calls"]
        saved = [sp.read_stats() for sp in rb.sps]
        tr0 = [s["transitions"] for s in saved]
        if results is not None and rank == 0:
            _keep_results(results, calls)
        if _stopped(calls, report_every, min(h for hs in _gather([s["hands"] for s in saved]) for h in hs), episodes):
            return rows
    elif results is not None and rank == 0:
        open(results, "w").close()
    t0 = time.time()
    while True:
        calls += 1
        report = _is_report(calls, report_every)
        sts = rb.step(steps_per_call, sync=report)
        if not report:
            if checkpoint is not None and calls % checkpoint_every == 0:
                ckpt.save(checkpoint, calls, runs=rb, sweep=record)
            continue
        dt = max(time.time() - t0, 1e-9)
        ex = rb.exploitability() if true_exploitability else None
        mine = []
        for k, (run, sp, st) in enumerate(zip(runs, rb.sps, sts)):
            stats = sp.read_stats()
            row = {"kind": "run", "calls": calls, "run": run["run"], "rank": rank, "point": run["point"], "seed": run["seed"],
                   "hparams": dict(run["hparams"]), "hands": stats["hands"], "transitions": stats["transitions"],
                   "exploitability_proxy": st.get("exploitability"),
                   "actions": [sampled_actions(stats, p) for p in range(2)],
                   "transitions_per_sec": (stats["transitions"] - tr0[k]) / dt}
            if true_exploitability:
                row["exploitability"] = ex[k]
            _mark_optimizer(row, rb.learners[k])
            mine.append(row)
        run_rows = [r for part in _gather(mine) for r in part]
        new = run_rows + _point_rows(run_rows, calls, true_exploitability)
        rows.extend(new)
        log("================ Stats ==================")
        for r in new:
            hp = " ".join("%s=%s" % kv for kv in r["hparams"].items())
            if r["kind"] == "run":
                line = "run %d (rank %d, seed %d, %s): hands %d  exploitability proxy %s" % (
                    r["run"], r["rank"], r["seed"], hp, r["hands"], r["exploitability_proxy"])
                if true_exploitability:
                    line += "  exact exploitability %.4f chips/hand" % r["exploitability"]["value"]
            else:
                line = "point %d (%s): %d seeds" % (r["point"], hp, len(r["seeds"]))
                if true_exploitability:
                    line += "  exact exploitability mean %.4f  std %.4f chips/hand" % (r["exploitability_mean"],
                                                                                      r["exploitability_std"])
            log(line)
        if results is not None and rank == 0:
            with open(results, "a") as f:
                f.writelines(json.dumps(r) + "\n" for r in new)
        done = min(r["hands"] for r in run_rows) >= episodes
        if checkpoint is not None and (done or calls % checkpoint_every == 0):
            ckpt.save(checkpoint, calls, runs=rb, sweep=record)
        if done:
            return rows


def main(argv=None):
    ap = argparse.ArgumentParser(description="NFSP self-play on Leduc Hold'em, B200-native")
    ap.add_argument("--human", action="store_true", help="accepted and ignored, as in the reference (main.py:152-158)")
    ap.add_argument("--config", default="./config.ini")
    ap.add_argument("--games", type=int, default=1 << 16, help="parallel games over all GPUs")
    ap.add_argument("--episodes", type=int, default=None, help="hands to play (default: Common.Episodes)")
    ap.add_argument("--steps-per-call", type=int, default=8)
    ap.add_argument("--report-every", type=int, default=100)
    ap.add_argument("--no-true-exploitability", action="store_true")
    ap.add_argument("--pipelined", action="store_true", help="run the learner's update beside the next rollout")
    ap.add_argument("--others-to-target", action="store_true",
                    help="untaken Q outputs regress to the target net's predictions, as the reference's fit does (agent.py:220)")
    ap.add_argument("--terminal-bootstraps", action="store_true",
                    help="terminal transitions bootstrap too (the reference's `t is True` never holds, agent.py:227)")
    ap.add_argument("--deterministic", action="store_true",
                    help="fix the order of the records in the memories (one staging segment per block of 32 games)")
    ap.add_argument("--variant", default="default", choices=["default", "states", "cuda", "pairs", "tcgen05", "tcgen05_ws"],
                    help="rollout kernel: the nets tabulated over the game's decision states (default) or evaluated per decision")
    ap.add_argument("--updates-per-call", type=int, default=1,
                    help="update_strategy() calls per rollout call (the reference's cadence: games * steps / 256)")
    ap.add_argument("--runs", type=int, default=1,
                    help="independent runs with seeds Seed, Seed + 1, ... trained side by side on one GPU, their launches shared; "
                         "with --sweep, the seeds of every grid point")
    ap.add_argument("--sweep", action="append", default=None, metavar="KEY=V1,V2,...",
                    help="train every combination of the values given (repeatable; keys: %s, with or without their "
                         "section), --runs seeds each, as independent runs spread over all ranks" % ", ".join(sweep.RUN_KEYS))
    ap.add_argument("--results", metavar="FILE", default=None,
                    help="with --sweep: write every reported row of every run and grid point to FILE as JSON Lines")
    ap.add_argument("--optimizer", default="sgd", choices=list(OPTIMIZERS),
                    help="the learner's optimizer: the reference's plain SGD (default) or Keras 2's Adam, with the "
                         "configured learning rates; every run of a sweep uses the same one")
    ap.add_argument("--checkpoint", metavar="DIR", default=None,
                    help="save the training state to DIR every --checkpoint-every rollout calls and when training ends")
    ap.add_argument("--checkpoint-every", type=int, default=CHECKPOINT_EVERY, metavar="CALLS",
                    help="rollout calls between two checkpoints (default %(default)s: under 1%% of the training time)")
    ap.add_argument("--resume", metavar="DIR", default=None,
                    help="continue the run saved in DIR; the command line must give the shape it was trained with")
    args = ap.parse_args(argv)
    cfg = load_config(args.config)
    rank, world, local = sharding.env_rank_world()
    if args.runs < 1:
        ap.error("--runs must be at least 1")
    runs = None
    if args.sweep is not None:
        if args.pipelined:
            ap.error("--sweep trains with the sequential loop: not with --pipelined")
        if args.updates_per_call != 1:
            ap.error("--sweep runs one update per rollout call: not --updates-per-call %d" % args.updates_per_call)
        if args.variant not in ("default", "states"):
            ap.error("--sweep plays the state-table rollout (--variant default / states): not --variant %s" % args.variant)
        try:
            runs = sweep.expand(sweep.parse_axes(args.sweep), args.runs, cfg)
            sweep.check_layout(len(runs), world)
        except ValueError as e:
            ap.error(str(e))
    elif args.runs > 1 and (args.pipelined or world > 1):
        ap.error("--runs > 1 trains on one GPU with the sequential loop: not with --pipelined or more than one rank")
    if args.results is not None and runs is None:
        ap.error("--results needs --sweep")
    if args.checkpoint_every < 1:
        ap.error("--checkpoint-every must be at least 1")
    saving = dict(checkpoint=args.checkpoint, checkpoint_every=args.checkpoint_every, resume=args.resume)
    if runs is not None:   # several ranks may share a GPU: a sweep's ranks exchange nothing on the device
        local %= max(torch.cuda.device_count(), 1)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and runs is not None:   # host-side collectives only: the report gather, the stop, the checkpoint agreement
        dist.init_process_group("gloo")
    elif world > 1:
        dist.init_process_group("nccl", device_id=dev)
    seed = cfg.getint("Utils", "Seed")              # main.py:132-133
    game0, n = sharding.shard_games(args.games, rank, world)
    episodes = args.episodes if args.episodes is not None else cfg.getint("Common", "Episodes")

    def make_run(run_seed, hp, n=n, game0=game0, data_parallel=True):
        sp_ = SelfPlay(n, seed=run_seed, game0=game0, device=dev, eta=hp["Eta"], epsilon=hp["Epsilon"],
                       rl_capacity=cfg.getint("Agent", "MRLSize"),
                       sl_capacity=cfg.getint("Agent", "MSLSize"), max_steps_per_call=args.steps_per_call,
                       deterministic=args.deterministic, direct_rings=False if args.deterministic else "auto",
                       variant=args.variant)
        return sp_, Learner(sp_, minibatch=cfg.getint("Agent", "MiniBatchSize"), lr_br=hp["LearningRateBR"],
                            lr_ar=hp["LearningRateAR"], gamma=hp["Gamma"], target_update_rate=hp["TargetModelUpdateRate"],
                            terminal_bootstraps=args.terminal_bootstraps, others_to_target=args.others_to_target,
                            data_parallel=data_parallel, optimizer=args.optimizer)

    if runs is not None:   # no run is sharded: run i plays games 0 .. --games - 1 whatever the world size
        mine = [runs[i] for i in sweep.rank_runs(len(runs), rank, world)]
        rb = RunBatch(*zip(*[make_run(r["seed"], r["hparams"], args.games, 0, False) for r in mine]))
        rows = train_sweep(rb, mine, sweep.record(runs, world), episodes, args.steps_per_call, args.report_every,
                           log=print if rank == 0 else (lambda *a, **k: None),
                           true_exploitability=not args.no_true_exploitability, results=args.results, **saving)
        if world > 1:
            dist.destroy_process_group()
        return rows
    hp = sweep.config_hparams(cfg)
    if args.runs > 1:
        rb = RunBatch(*zip(*[make_run(seed + r, hp) for r in range(args.runs)]))
        return train_runs(rb, episodes, args.steps_per_call, args.report_every,
                          true_exploitability=not args.no_true_exploitability, **saving)
    sp, learner = make_run(seed, hp)
    rows = train(sp, learner, episodes, args.steps_per_call, args.report_every, world,
                 log=print if rank == 0 else (lambda *a, **k: None),
                 true_exploitability=not args.no_true_exploitability, pipelined=args.pipelined,
                 updates_per_call=args.updates_per_call, **saving)
    if world > 1:
        dist.destroy_process_group()
    return rows


if __name__ == "__main__":
    main()
