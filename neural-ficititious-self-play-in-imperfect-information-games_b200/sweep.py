"""Hyperparameter sweeps: a grid of settings, each with several seeds, trained as independent runs over all ranks.

`main.py --sweep KEY=V1,V2,... [--sweep ...] --runs R` names the values of the config keys a run owns (DESIGN.md 7d).  The
runs are the Cartesian product of the values, in the order given, times R seeds per grid point (base ... base + R - 1,
the innermost dimension).  Run i has one definition -- its grid point, seed and hyperparameters -- whatever the number
of ranks; the ranks take contiguous, balanced blocks of runs and train each block as one `runs.RunBatch`.  Everything
here is host-side and touches no device, so the command line is refused before a GPU is used.
"""
from __future__ import annotations

import itertools
import math

from . import _lib
from .sharding import shard_games

# the config keys a run may own, with their type: what SelfPlay / Learner take per run
RUN_KEYS = {"Agent.Eta": float, "Agent.Epsilon": float, "Agent.LearningRateBR": float, "Agent.LearningRateAR": float,
            "Agent.Gamma": float, "Agent.TargetModelUpdateRate": int, "Utils.Seed": int}
# keys every run of a batch must share: they set the shape of the launches and memories
SHARED_KEYS = ("Agent.MiniBatchSize", "Agent.MRLSize", "Agent.MSLSize", "Agent.HiddenLayer")
HPARAMS = ("Eta", "Epsilon", "LearningRateBR", "LearningRateAR", "Gamma", "TargetModelUpdateRate")


def _canonical(key):
    """'Eta' or 'Agent.Eta' -> 'Agent.Eta'; raises ValueError for a key runs must share or do not know."""
    for full in RUN_KEYS:
        if key in (full, full.split(".")[1]):
            return full
    shared = key.startswith("Environment.") or any(key in (full, full.split(".")[1]) for full in SHARED_KEYS)
    if shared:
        raise ValueError("--sweep %s: this key is shared by every run of a batch and cannot be swept" % key)
    raise ValueError("--sweep %s: unknown key (a sweep varies %s)" % (key, ", ".join(RUN_KEYS)))


def _number(key, text, kind):
    try:
        v = float(text)
    except ValueError:
        raise ValueError("--sweep %s: %r is not a number" % (key, text)) from None
    if not math.isfinite(v):
        raise ValueError("--sweep %s: %r is not a finite number" % (key, text))
    if kind is int:
        if v != int(v):
            raise ValueError("--sweep %s: %r is not an integer" % (key, text))
        v = int(text) if text.strip().lstrip("+-").isdigit() else int(v)
    if key == "Agent.TargetModelUpdateRate" and v < 1:
        raise ValueError("--sweep %s: %r is below 1" % (key, text))
    return v


def parse_axes(specs):
    """The --sweep options ["KEY=V1,V2", ...] -> [(full key, [values]), ...] in the order given; raises ValueError."""
    axes = []
    for spec in specs:
        key, eq, values = spec.partition("=")
        key = key.strip()
        if not eq:
            raise ValueError("--sweep %s: expected KEY=V1,V2,..." % spec)
        full = _canonical(key)
        if any(full == k for k, _ in axes):
            raise ValueError("--sweep %s: the key is given twice" % full)
        texts = values.split(",")
        if any(not t.strip() for t in texts):
            raise ValueError("--sweep %s: empty value in %r" % (full, values))
        axes.append((full, [_number(full, t.strip(), RUN_KEYS[full]) for t in texts]))
    return axes


def config_hparams(cfg):
    """The hyperparameters a run owns, as config.ini gives them (read as Learner(cfg=...) and main.py read them)."""
    return {k: (cfg.getint if RUN_KEYS["Agent." + k] is int else cfg.getfloat)("Agent", k) for k in HPARAMS}


def expand(axes, seeds_per_point, cfg):
    """Every run of the sweep: [{"run": i, "point": p, "seed": s, "hparams": {Eta: ..., ...}}, ...].  Grid points are
    the product of the axes' values in the order given (the last axis fastest); each has `seeds_per_point` runs, seeds
    base ... base + R - 1 (base: the point's Utils.Seed, config.ini's when not swept)."""
    runs = []
    for p, values in enumerate(itertools.product(*[v for _, v in axes])):
        hp, base = config_hparams(cfg), cfg.getint("Utils", "Seed")
        for (key, _), v in zip(axes, values):
            if key == "Utils.Seed":
                base = v
            else:
                hp[key.split(".")[1]] = v
        for s in range(seeds_per_point):
            runs.append(dict(run=len(runs), point=p, seed=base + s, hparams=dict(hp)))
    return runs


def rank_runs(n_runs, rank, world):
    """The runs rank `rank` trains: a contiguous block, the blocks' sizes differing by at most one."""
    first, n = shard_games(n_runs, rank, world)
    return range(first, first + n)


def check_layout(n_runs, world):
    """Raises ValueError unless every rank has at least one run and at most NFSP_MAX_RUNS."""
    if n_runs < world:
        raise ValueError("the sweep has %d runs but %d ranks: every rank needs a run" % (n_runs, world))
    if -(-n_runs // world) > _lib.MAX_RUNS:
        raise ValueError("the sweep puts %d runs on one rank (%d runs over %d ranks); a rank trains at most %d" %
                         (-(-n_runs // world), n_runs, world, _lib.MAX_RUNS))


def record(runs, world):
    """The sweep's part of a checkpoint's driver record: the whole run list and the world size."""
    return dict(runs=[dict(r, hparams=dict(r["hparams"])) for r in runs], world=world)


def record_difference(saved, here):
    """None when the sweep record `saved` (from a checkpoint) equals `here`, else what differs, in words."""
    if not isinstance(saved, dict) or not isinstance(saved.get("runs"), list):
        return "the checkpoint holds no sweep"
    if saved.get("world") != here["world"]:
        return "the sweep was saved by %r ranks but %d run it here" % (saved.get("world"), here["world"])
    if len(saved["runs"]) != len(here["runs"]):
        return "the checkpoint's sweep has %d runs but this one %d" % (len(saved["runs"]), len(here["runs"]))
    for a, b in zip(saved["runs"], here["runs"]):
        if not isinstance(a, dict):
            return "run %d of the checkpoint's sweep is malformed" % b["run"]
        for k in ("point", "seed"):
            if a.get(k) != b[k]:
                return "run %d: %s is %r in the checkpoint but %r here" % (b["run"], k, a.get(k), b[k])
        ha = a.get("hparams") if isinstance(a.get("hparams"), dict) else {}
        for k in HPARAMS:
            if ha.get(k) != b["hparams"][k]:
                return "run %d: %s is %r in the checkpoint but %r here" % (b["run"], k, ha.get(k), b["hparams"][k])
    return None
