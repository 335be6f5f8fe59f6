"""Independent NFSP runs side by side on one GPU, their hot launches shared.

An exploitability curve means little without several seeds, and the thesis the reference comes from compares settings of
eta and of the learning rates, so users train many runs.  Each run alone leaves most of the B200 idle: the fit is four
CTAs, and a rollout of 65 536 games is latency, not throughput.  A `RunBatch` takes R ordinary runs -- a `SelfPlay` (its
own env handle, memories, counters) plus the `Learner` that trains it -- and issues their hot steps together:

    rollout(T)   one nfsp_rollout_runs launch for all runs (plus one image and one state-table launch when learners have
                 updated), then the inserts in groups of up to four memories (nfsp_insert_multi)
    update()     one sampling launch for the 4R memories, one nfsp_learner_fit_runs launch (4R CTAs; with Adam learners
                 nfsp_learner_fit_runs_adam, each run's moments and steps its own), then each learner's own host
                 schedules (Learner._finish_update)

Run r does exactly what it would do alone, bit for bit: games, records, memories, weights, schedules.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import check, lib
from .batched import SelfPlay, _ptr, _stream
from .learner import GRAD, _world


def _selfplay_shape(sp):
    return (sp.device, sp.n, sp.max_steps, sp.direct_rings, sp.deterministic, sp.rl[0].capacity, sp.rl[1].capacity,
            sp.sl[0].capacity, sp.sl[1].capacity, sp.n_seg, sp.cap_rl, sp.cap_sl)


def _learner_shape(ln):
    return (ln.minibatch, ln.fit_batch, ln.epochs, ln.terminal_bootstraps, ln.others_to_target, ln.fused, ln.optimizer)


class RunBatch:
    """R independent runs of one shape trained side by side; see the module docstring.

    selfplays[r] is trained by learners[r].  The runs must share device, n_games, max_steps_per_call, the default
    ("states") rollout variant, direct_rings, deterministic, the memories' capacities and the learner's minibatch, fit
    batch, epochs, flags and optimizer; seeds, eta, epsilons and learning rates are each run's own.  One GPU only; with a process
    group of several ranks (a sweep, sweep.py) every learner must train alone (Learner(data_parallel=False))."""

    def __init__(self, selfplays, learners):
        sps, lns = list(selfplays), list(learners)
        if not sps or len(sps) != len(lns):
            raise ValueError("one learner per self-play, at least one run")
        if len(sps) > _lib.MAX_RUNS:
            raise ValueError("at most %d runs per batch" % _lib.MAX_RUNS)
        if _world() > 1 and any(ln.data_parallel for ln in lns):
            raise ValueError("a RunBatch trains its runs on one GPU: world > 1 needs learners that train alone "
                             "(Learner(data_parallel=False))")
        if len({id(sp) for sp in sps}) != len(sps):
            raise ValueError("a self-play appears twice")
        for r, (sp, ln) in enumerate(zip(sps, lns)):
            if ln.sp is not sp:
                raise ValueError("learner %d does not train self-play %d" % (r, r))
            if SelfPlay.VARIANTS[sp.variant] not in (0, 6):
                raise ValueError("run %d: runs play the default rollout variant ('states'), not %r" % (r, sp.variant))
            if _selfplay_shape(sp) != _selfplay_shape(sps[0]):
                raise ValueError("run %d differs from run 0 in shape (device, games, steps per call, record mode, "
                                 "capacities)" % r)
            if _learner_shape(ln) != _learner_shape(lns[0]):
                raise ValueError("run %d's learner differs from run 0's (minibatch, fit batch, epochs, flags, optimizer)" % r)
            if not ln.fused:
                raise ValueError("run %d: the batched update is the one-launch fit (fused=True)" % r)
        self.sps, self.learners = sps, lns
        self.device = sps[0].device
        R = self.n_runs = len(sps)
        self._h = (C.c_void_p * R)(*[sp.env._h.value for sp in sps])
        self._eta = (C.c_double * R)()
        self._eps = (C.c_double * R)()
        self._io = (_lib.RolloutIO * R)()
        self._io_src = [None] * R
        self._w = (C.c_void_p * R)()
        self._refresh = False  # a learner has written its run's acting nets: the next rollout rebuilds the images
        # the inserts: every run's memories in groups of up to NFSP_MAX_INSERT_REQS (direct rings: both runs' reservoirs of
        # a pair of runs per launch; staged: one run's four memories per launch)
        mems = [(sp, m) for sp in sps for m in sp._insert_mems()]
        self._inserts = []
        for k in range(0, len(mems), 4):
            group = mems[k:k + 4]
            arr = (_lib.InsertReq * len(group))()
            for req, (sp, m) in zip(arr, group):
                sp._insert_req(req, *m)
            self._inserts.append((arr, len(group)))
        b = lns[0].minibatch
        self._pos = torch.empty((R, 4, b), dtype=torch.int64, device=self.device)  # per run: rl0, rl1, sl0, sl1
        self._sample_reqs = (_lib.SampleReq * (4 * R))()
        self._learner_io = (_lib.LearnerIO * R)()
        self._lr = (C.c_float * (4 * R))()
        self._w_out = (C.c_void_p * R)()
        self._adam = (_lib.AdamState * R)() if lns[0].optimizer == "adam" else None

    def rollout(self, n_steps=8):
        """SelfPlay.rollout(n_steps) of every run: one nfsp_rollout_runs call (rebuilding the weight images of the runs
        when their learners have updated since the last rollout), then the grouped inserts."""
        if n_steps > self.sps[0].max_steps:
            raise ValueError("n_steps %d exceeds max_steps_per_call %d" % (n_steps, self.sps[0].max_steps))
        for r, sp in enumerate(self.sps):
            io = sp._rollout_io()
            if io is not self._io_src[r]:  # first call, or the counters moved (sample_minibatches(with_stats=True))
                self._io[r] = io
                self._io_src[r] = io
            dst = self._io[r]
            dst.variant = SelfPlay.VARIANTS[sp.variant]
            dst.epsilon_per_player, dst.epsilon_p1 = int(sp.epsilons[0] != sp.epsilons[1]), sp.epsilons[1]
            dst.reserve_sms = 0
            self._eta[r], self._eps[r] = sp.eta, sp.epsilons[0]
        w = None
        if self._refresh:
            for r, sp in enumerate(self.sps):
                self._w[r] = sp.weights.data_ptr()
            w = self._w
        check(lib().nfsp_rollout_runs(self._h, self.n_runs, n_steps, self._eta, self._eps, self._io, w,
                                      _stream(self.device)))
        self._refresh = False
        self.flush()

    def flush(self):
        """SelfPlay.flush() of every run, up to four memories per nfsp_insert_multi launch."""
        st = _stream(self.device)
        for arr, n in self._inserts:
            check(lib().nfsp_insert_multi(arr, n, st))

    def update(self, sync=False):
        """Learner.update(sync) of every run: the ready masks, ONE sampling launch for the memories of every run that
        trains, ONE fit launch, then each learner's schedules.  The acting images are rebuilt by the next rollout().
        Returns the per-run dicts Learner.update returns."""
        lns, sps = self.learners, self.sps
        masks = [ln._ready_mask() for ln in lns]
        active = [r for r in range(self.n_runs) if masks[r]]
        out = [{"trained": 0}] * self.n_runs
        if not active:
            return out
        b, st = lns[0].minibatch, _stream(self.device)
        for k, r in enumerate(active):
            ln = lns[r]
            ln._begin_update(masks[r])
            ln._sample_requests(snapshot=False, which="both")
            ln._mems = None  # the fit reads the memories themselves
            for j in range(4):
                self._sample_reqs[4 * k + j] = ln._pos_reqs[j]
        check(lib().nfsp_sample_minibatches(self._sample_reqs, 4 * len(active), b, _ptr(self._pos), None, st))
        for k, r in enumerate(active):
            ln, pos = lns[r], self._pos[k]
            self._learner_io[k], self._lr[4 * k:4 * k + 4] = ln._fit_args([pos[0], pos[1]], [pos[2], pos[3]], masks[r])
            self._w_out[k] = sps[r].weights.data_ptr()
        fit = (self._learner_io, len(active), b, lns[0].fit_batch, lns[0].epochs, self._lr, self._w_out)
        if self._adam is None:
            check(lib().nfsp_learner_fit_runs(*fit, st))
        else:
            for k, r in enumerate(active):
                lns[r].adam_state(self._adam[k])
            check(lib().nfsp_learner_fit_runs_adam(*fit, self._adam, st))
            for r in active:
                lns[r]._adam_advance(masks[r], lns[r].fit_steps)
        out = list(out)
        for r in active:
            ln = lns[r]
            out[r] = ln._finish_update(masks[r], ln.flat[GRAD:], sync, sps[r].weights, pack=False)
        self._refresh = True
        return out

    def step(self, n_steps=8, sync=False):
        """rollout(n_steps) then update(sync): one iteration of every run."""
        self.rollout(n_steps)
        return self.update(sync)

    def state_dict(self) -> dict:
        """The runs' states in order, each {"selfplay": SelfPlay.state_dict(), "learner": Learner.state_dict()}: the
        format of a run trained alone, so a run can move between a batch and a standalone SelfPlay / Learner."""
        return dict(runs=[dict(selfplay=sp.state_dict(), learner=ln.state_dict()) for sp, ln in zip(self.sps, self.learners)])

    def check_state_dict(self, d):
        """Raises ValueError, naming the run and field, if load_state_dict(d) would refuse d."""
        runs = d.get("runs") if isinstance(d, dict) else None
        if not isinstance(runs, list) or len(runs) != self.n_runs:
            raise ValueError("RunBatch: the state holds %s runs but this batch %d" %
                             (len(runs) if isinstance(runs, list) else "no", self.n_runs))
        for r, (run, sp, ln) in enumerate(zip(runs, self.sps, self.learners)):
            if not (isinstance(run, dict) and {"selfplay", "learner"} <= run.keys()):
                raise ValueError("RunBatch: run %d must hold a selfplay and a learner state" % r)
            try:
                sp.check_state_dict(run["selfplay"])
                ln.check_state_dict(run["learner"])
            except ValueError as e:
                raise ValueError("run %d: %s" % (r, e)) from None

    def load_state_dict(self, d):
        """Validates every run's state, then loads them all."""
        self.check_state_dict(d)
        for run, sp, ln in zip(d["runs"], self.sps, self.learners):
            sp.load_state_dict(run["selfplay"])
            ln.load_state_dict(run["learner"])

    def exploitability(self):
        """exploitability.exploitability(sp) of every run (exact, of the average policies)."""
        from .exploitability import exploitability

        if self._refresh:  # the images the exact computation reads must be those of the newest nets
            for sp in self.sps:
                sp.set_weights(sp.weights)
            self._refresh = False
        return [exploitability(sp) for sp in self.sps]
