"""Checkpoints of training runs: save a run's whole state to a directory and resume it bit for bit.

A checkpoint is a directory with one `torch.save` file per rank, `rank{r}-of-{world}.pt`.  Each file holds the format
version, the world size and rank, a small driver record (the training loop's `calls` counter; a sweep's also holds its
run list and world size, main.py --sweep) and the `state_dict()` of
every object it was given: a SelfPlay and its Learner (plus a PipelinedTrainer), or a RunBatch.  Every random draw of a
run is Philox keyed by counters those state dicts carry (the env step counter, each memory's `total` and
`sample_calls`), so a run loaded from a checkpoint continues exactly as the saved one would have, wherever that run is
itself deterministic (`SelfPlay(deterministic=True)`).

A file is written to a temporary name in the same directory, flushed to disk and renamed over the old one: a crash
during a save leaves the previous checkpoint loadable.  Each rank's memories hold the records of its own games, so a
checkpoint loads only into the same number of ranks with the same games per rank.
"""
from __future__ import annotations

import os
import tempfile

import torch
import torch.distributed as dist

from .sweep import record_difference

FORMAT = 1
PARTS = ("selfplay", "learner", "trainer", "runs")


def _rank_world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def file_name(rank: int, world: int) -> str:
    return "rank%d-of-%d.pt" % (rank, world)


def _given(selfplay, learner, trainer, runs):
    objs = dict(selfplay=selfplay, learner=learner, trainer=trainer, runs=runs)
    return {k: v for k, v in objs.items() if v is not None}


def save(path, calls, selfplay=None, learner=None, trainer=None, runs=None, sweep=None):
    """Writes this rank's file of the checkpoint directory `path` (created if missing): the driver record {"calls":
    calls} (plus {"sweep": sweep}, a sweep.record(), when given) and the state dicts of the objects given.  Every state
    dict is taken before anything is written, so a refusal (records staged but not flushed) leaves the directory as it
    was."""
    rank, world = _rank_world()
    state = dict(format=FORMAT, world=world, rank=rank, driver=dict(calls=int(calls)))
    if sweep is not None:
        state["driver"]["sweep"] = sweep
    for name, obj in _given(selfplay, learner, trainer, runs).items():
        state[name] = obj.state_dict()
    os.makedirs(path, exist_ok=True)
    name = file_name(rank, world)
    fd, tmp = tempfile.mkstemp(prefix="." + name + ".", suffix=".tmp", dir=path)
    try:
        with os.fdopen(fd, "wb") as f:
            torch.save(state, f)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, os.path.join(path, name))
    except BaseException:
        try:
            os.unlink(tmp)
        except OSError:
            pass
        raise
    dfd = os.open(path, os.O_RDONLY)  # the rename itself is durable once the directory is
    try:
        os.fsync(dfd)
    finally:
        os.close(dfd)


def _read(path, rank, world, objs, sweep=None):
    """This rank's file, checked against the objects without changing them; raises ValueError."""
    fname = os.path.join(path, file_name(rank, world))
    others = sorted(f for f in os.listdir(path) if f.startswith("rank%d-of-" % rank)) if os.path.isdir(path) else []
    if not os.path.exists(fname) and others:
        raise ValueError("%s is missing: the checkpoint was saved by another number of ranks (%s) than the %d here" %
                         (fname, ", ".join(others), world))
    try:
        state = torch.load(fname, map_location="cpu", weights_only=True)
    except Exception as e:  # noqa: BLE001  a missing or unreadable file is a refusal like any other
        raise ValueError("cannot read checkpoint file %s: %s" % (fname, e)) from None
    if not isinstance(state, dict) or state.get("format") != FORMAT:
        raise ValueError("%s: format %r, this version reads format %d" %
                         (fname, state.get("format") if isinstance(state, dict) else None, FORMAT))
    for k, v in (("world", world), ("rank", rank)):
        if state.get(k) != v:
            raise ValueError("%s: %s is %r in the checkpoint but %d here" % (fname, k, state.get(k), v))
    driver = state.get("driver")
    if not (isinstance(driver, dict) and type(driver.get("calls")) is int and driver["calls"] >= 0):
        raise ValueError("%s: no driver record with a calls counter" % fname)
    if sweep is not None:
        why = record_difference(driver.get("sweep"), sweep)
        if why is not None:
            raise ValueError("%s: %s" % (fname, why))
    elif "sweep" in driver:
        raise ValueError("%s: the checkpoint is of a sweep (--sweep)" % fname)
    held = sorted(k for k in PARTS if k in state)
    if held != sorted(objs):
        raise ValueError("%s: the checkpoint holds %s but %s were given" % (fname, held, sorted(objs)))
    for name, obj in objs.items():
        obj.check_state_dict(state[name])
    return state


def load(path, selfplay=None, learner=None, trainer=None, runs=None, sweep=None) -> dict:
    """Loads this rank's file of the checkpoint directory `path` into the objects given and returns the driver record.
    Everything is validated first -- format, world size, rank, the objects' shapes (n_games, game0, capacities, ...),
    the sweep's run list when `sweep` (a sweep.record()) is given, and, with several ranks, that every rank's file holds
    the same `calls` -- and all ranks agree on the outcome with one collective, so they refuse together (ValueError) and
    every object is then left as it was."""
    rank, world = _rank_world()
    objs = _given(selfplay, learner, trainer, runs)
    state, why = None, None
    try:
        state = _read(path, rank, world, objs, sweep)
    except ValueError as e:
        why = str(e)
    if world > 1:
        calls = state["driver"]["calls"] if state is not None else 0
        dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
        flags = torch.tensor([int(state is not None), calls, -calls], dtype=torch.int64, device=dev)
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        ok, lo, hi = int(flags[0]), int(flags[1]), -int(flags[2])
        if why is None and not ok:
            why = "another rank refused its checkpoint file"
        elif why is None and lo != hi:
            why = "the ranks' files are of different generations (calls %d .. %d)" % (lo, hi)
    if why is not None:
        raise ValueError("rank %d: %s" % (rank, why))
    for name, obj in objs.items():
        obj.load_state_dict(state[name])
    return dict(state["driver"])
