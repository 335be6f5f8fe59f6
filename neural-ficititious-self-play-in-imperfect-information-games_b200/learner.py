"""Learner half of agent.Agent (agent.py:209-273), SURVEY.md section 8 f-1.

`Learner.update()` is `update_strategy()` (agent.py:192-194) of BOTH agents at once: it samples a
minibatch from each of the four memories, then runs Keras' `fit(..., epochs=2)` (default batch 32,
so 8 SGD steps) for the four nets.  On one GPU the eight steps are ONE launch (`nfsp_learner_fit`: the
weights stay in registers between the steps).  With several GPUs every SGD step is: one `nfsp_learner_grads` launch (all four
nets, gradients into one flat fp32 buffer with the exploitability statistics behind them), ONE
all-reduce of that buffer over the GPUs (NCCL; C1 + C2 of SURVEY 2a), one `nfsp_sgd_apply` launch.
Weights therefore stay bit-identical on every rank.

`optimizer="adam"` trains with Keras 2's Adam (beta1 0.9, beta2 0.999, epsilon 1e-7) instead of the reference's plain SGD,
through the same paths: the `_adam` entries of the fit kernels and `nfsp_adam_apply` in place of `nfsp_sgd_apply`.

What follows the reference literally (host arithmetic): the schedules of agent.py:245-253 per player
(`iteration` advanced twice per update, temperature, BR learning-rate decay, each agent's own
`epsilon ** 1/iteration` == epsilon/iteration by operator precedence) and the target-net copy every
TargetModelUpdateRate updates (agent.py:266-273).  What does NOT (documented in DESIGN.md): the reference
overwrites only row 0 of the target batch (agent.py:241) and never treats a transition as terminal
(agent.py:227, kept behind `terminal_bootstraps=True`); here every row gets its own TD target, and the two
outputs a row did not take have zero error unless `others_to_target=True` (agent.py:220: they regress to the
target net's predictions).  Keras shuffles the rows
each epoch with an unseeded RNG; the minibatches here are the sampled rows in order.  The NN
arithmetic itself is unpinned (no Keras/TensorFlow to compare with).
"""
from __future__ import annotations

import ctypes as C
import math

import torch
import torch.distributed as dist

from . import _lib
from ._lib import check, lib
from .batched import _ptr, _stream, check_fields, check_numbers, check_tensor

GRAD = 4 * _lib.NET_PARAMS
N_STATS = 8
OPTIMIZERS = ("sgd", "adam")


def _world():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


class Learner:
    def __init__(self, selfplay, cfg=None, minibatch=128, fit_batch=32, epochs=2, lr_br=0.05, lr_ar=0.1, gamma=0.95,
                 target_update_rate=150, terminal_bootstraps=False, fused=True, use_multicast=True, others_to_target=False,
                 peer_transport="auto", data_parallel=True, optimizer="sgd"):
        if cfg is not None:
            minibatch = cfg.getint("Agent", "MiniBatchSize")
            lr_br, lr_ar = cfg.getfloat("Agent", "LearningRateBR"), cfg.getfloat("Agent", "LearningRateAR")
            gamma = cfg.getfloat("Agent", "Gamma")
            target_update_rate = cfg.getint("Agent", "TargetModelUpdateRate")
        self.sp = selfplay
        self.device = selfplay.device
        # data_parallel=False: this learner trains its own run alone and ignores an initialised process group (no peer
        # exchange, no gradient all-reduce, no agreement on the ready mask) -- a run of a sweep spread over ranks
        self.data_parallel = bool(data_parallel)
        self.minibatch, self.fit_batch, self.epochs = int(minibatch), int(fit_batch), int(epochs)
        self.lr_br0, self.lr_ar, self.gamma = float(lr_br), float(lr_ar), float(gamma)
        self.lr_br = [self.lr_br0, self.lr_br0]
        self.target_update_rate = int(target_update_rate)
        self.terminal_bootstraps = bool(terminal_bootstraps)
        # the two Q outputs a row did not take: zero error (default), or regressed to the target net's predictions as the
        # reference's `target = target_br_model.predict(s_batch)` does (agent.py:220,243)
        self.others_to_target = bool(others_to_target)
        self.fused = bool(fused)  # single GPU: the whole fit() as one kernel; False = one launch pair per SGD step
        if optimizer not in OPTIMIZERS:
            raise ValueError("optimizer must be one of %s, not %r" % (", ".join(OPTIMIZERS), optimizer))
        self.optimizer = optimizer
        if optimizer == "adam":
            # Adam's state, per net as each Keras model has its own optimizer: the moments on the device (the kernels
            # update them in place) and the steps taken (on the host, which knows every fit's mask and step count)
            self.adam_m = torch.zeros((4, _lib.NET_PARAMS), dtype=torch.float32, device=self.device)
            self.adam_v = torch.zeros((4, _lib.NET_PARAMS), dtype=torch.float32, device=self.device)
            self.adam_t = [0, 0, 0, 0]
        self.target = selfplay.weights[[1, 3]].clone().contiguous()   # agent.py:70-72
        self.flat = torch.zeros(GRAD + N_STATS, dtype=torch.float32, device=self.device)
        self._peers = None
        self.peer_check_every = 64  # updates between two reads of the peer-exchange error word when nothing else syncs
        self.use_multicast = use_multicast
        if peer_transport not in ("auto", "symm", "ipc"):
            raise ValueError("peer_transport must be 'auto', 'symm' or 'ipc'")
        self.peer_transport = peer_transport
        if self.fused and self._world() > 1 and self.minibatch <= _lib.FIT_ROWS_MAX_MINIBATCH and self.fit_batch <= _lib.FIT_ROWS_MAX_STEP:
            # every rank must take the same path (a rank in the peer exchange and one in an NCCL all-reduce would wait
            # for each other forever): _setup_peers agrees on every phase collectively
            self._setup_peers()
        self.iteration = [0, 0]
        self.target_update_count = [0, 0]
        self.temp = [1.0, 1.0]
        self.exploitability = [0.0, 0.0]
        self.updates = 0

    def _world(self):
        """The ranks this learner trains over: every rank of the process group, or 1 without data_parallel."""
        return _world() if self.data_parallel else 1

    @property
    def one_launch(self) -> bool:
        """The whole fit runs as one kernel (one GPU, or several with the peer exchange): what weights_in / weights_out
        and PipelinedTrainer need.  The same on every rank (the peer set-up is collective)."""
        return self.fused and (self._world() == 1 or self._peers is not None)

    def _snapshot_buffers(self):
        """Where the sampling launch leaves packed copies of the sampled records (4 x minibatch rows, 24 KB): once they
        exist the update no longer reads the memories, so a rollout that writes the rings in place, or the next insert,
        may run beside the fit."""
        b = self.minibatch
        if not hasattr(self, "_gath"):
            self._gath = ([torch.zeros((b, 4), dtype=torch.int32, device=self.device) for _ in range(2)],
                          [torch.zeros((b, 8), dtype=torch.int32, device=self.device) for _ in range(2)],
                          torch.arange(b, dtype=torch.int64, device=self.device))
        return self._gath

    def _io(self, idx_rl, idx_sl, row0, rows, mask, w_in=None):
        sp = self.sp
        io = _lib.LearnerIO()
        io.d_weights, io.d_target_weights = (sp.weights if w_in is None else w_in).data_ptr(), self.target.data_ptr()
        mem_rl, mem_sl = getattr(self, "_mems", None) or ([m.store for m in sp.rl], [m.store for m in sp.sl])
        for p in range(2):
            io.d_rl[p], io.d_rl_idx[p] = mem_rl[p].data_ptr(), idx_rl[p].data_ptr()
            io.d_sl[p], io.d_sl_idx[p] = mem_sl[p].data_ptr(), idx_sl[p].data_ptr()
        io.row0, io.rows, io.gamma, io.net_mask = row0, rows, self.gamma, mask
        io.terminal_bootstraps = int(self.terminal_bootstraps)
        io.others_to_target = int(self.others_to_target)
        io.d_grad, io.d_stats = self.flat.data_ptr(), self.flat[GRAD:].data_ptr()
        return io

    def _fit_args(self, idx_rl, idx_sl, mask, w_in=None, row0=0, rows=None):
        """The nfsp_learner_io of sampled rows [row0, row0 + rows) (default: all) and the lrs in net order avg0, br0, avg1, br1."""
        io = self._io(idx_rl, idx_sl, row0, self.minibatch if rows is None else rows, mask, w_in)
        return io, (self.lr_ar, self.lr_br[0], self.lr_ar, self.lr_br[1])

    def _sample_positions(self, snapshot=False, which="both"):
        """sample_batch positions of the four memories (agent.py:217,260) in one launch; the same draws as four
        sample_slots() calls.  Returns ([rl0, rl1], [sl0, sl1]) index tensors of `minibatch` storage slots.
        snapshot: the launch also copies the sampled slots out of the memories; the fit then reads those copies.
        which = "rl" / "sl": only the two rings / the two reservoirs (the pipelined trainer samples the rings as soon as
        the rollout has written them and the reservoirs after the insert launch); "rl" returns nothing."""
        b = self.minibatch
        lo, hi = self._sample_requests(snapshot, which)
        g_rl, g_sl, rows = self._snapshot_buffers() if snapshot else (None, None, None)
        first = C.cast(C.byref(self._pos_reqs, lo * C.sizeof(_lib.SampleReq)), C.POINTER(_lib.SampleReq))
        check(lib().nfsp_sample_minibatches(first, hi - lo, b, _ptr(self._pos[lo:]), None, _stream(self.device)))
        if which == "rl":
            return None
        if snapshot:  # the sampled slots are rows 0 .. b-1 of the snapshots
            self._mems = (g_rl, g_sl)
            return [rows, rows], [rows, rows]
        self._mems = None
        return [self._pos[0], self._pos[1]], [self._pos[2], self._pos[3]]

    def _sample_requests(self, snapshot=False, which="both"):
        """The sampling requests of _sample_positions (self._pos_reqs, rows rl0, rl1, sl0, sl1), their memories' draw
        counters advanced; nothing is launched.  Returns the range [lo, hi) of the requests `which` names."""
        sp, b = self.sp, self.minibatch
        mems = (sp.rl[0], sp.rl[1], sp.sl[0], sp.sl[1])
        if not hasattr(self, "_pos"):
            self._pos = torch.empty((4, b), dtype=torch.int64, device=self.device)   # rows: rl0, rl1, sl0, sl1
            self._pos_reqs = (_lib.SampleReq * 4)(*(mem.sample_req(_lib.SampleReq()) for mem in mems))
        g_rl, g_sl, rows = self._snapshot_buffers() if snapshot else (None, None, None)
        lo, hi = {"both": (0, 4), "rl": (0, 2), "sl": (2, 4)}[which]
        for k in range(lo, hi):
            r = self._pos_reqs[k]
            r.call_idx = mems[k].next_call()
            r.d_rec_out = None if not snapshot else (g_rl[k] if k < 2 else g_sl[k - 2]).data_ptr()
        return lo, hi

    def presample_rings(self):
        """First half of an update for the pipelined trainer: draw the RL minibatches of both players and snapshot their
        records (what update(presampled_rings=True) then trains on).  With direct_rings this is all of an update that
        reads the rings, so the next rollout -- which writes them in place -- only waits for this launch."""
        self._sample_positions(snapshot=True, which="rl")

    # ---- several GPUs of one box: the all-reduce of every SGD step inside the fit kernel, over peer memory ----
    def _agree(self, ok: bool) -> bool:
        """True iff every rank says ok: one MIN all-reduce, so that all ranks take the same branch."""
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        return bool(int(flag.item()))

    def _no_peers(self, why):
        self._peers = None
        self._peer_note = "peer exchange unavailable: %s" % (why,)
        import warnings

        warnings.warn("nfsp_b200 learner: %s; using one NCCL all-reduce per SGD step" % self._peer_note, RuntimeWarning)

    def _setup_peers(self):
        """One exchange buffer per rank that every rank can address.  Two transports, tried in this order (or the one
        `peer_transport` names): "symm" -- torch symmetric memory, which also offers the NVLS multicast mapping -- and
        "ipc" -- buffers the library allocates itself and shares as plain CUDA IPC handles (no private torch module
        involved).  Falls back to the NCCL path (one all-reduce per SGD step) if neither works.

        Collective-safe: each phase that can fail on one rank only runs under its own try, and the ranks AGREE on its
        outcome with an all-reduce before anybody enters the next collective -- no rank can sit in rendezvous / barrier
        while another has already fallen back."""
        if dist.get_world_size() > _lib.MAX_PEERS:  # the same on every rank
            return self._no_peers("more than %d ranks" % _lib.MAX_PEERS)
        notes = []
        for transport in (("symm", "ipc") if self.peer_transport == "auto" else (self.peer_transport,)):
            why = self._setup_peers_symm() if transport == "symm" else self._setup_peers_ipc()
            if why is None:
                self._peer_transport = transport
                return
            notes.append("%s: %s" % (transport, why))
        self._no_peers("; ".join(notes))

    def _finish_peers(self, ptrs, mc, keep):
        p = _lib.Peers()
        p.world, p.rank = dist.get_world_size(), dist.get_rank()
        for r in range(p.world):
            p.d_buf[r] = int(ptrs[r])
        self._peer_err = torch.zeros(1, dtype=torch.int32, device=self.device)
        p.d_err = self._peer_err.data_ptr()
        p.d_mc = mc or None
        self._multicast = bool(mc)
        self._peers, self._peer_keep, self._epoch = p, keep, 0

    def _setup_peers_symm(self):
        """torch symmetric memory; returns None on success, else why not (the same answer on every rank)."""
        symm_mem, buf, why = None, None, None
        try:  # phase 1, local only: the import and the allocation
            import torch.distributed._symmetric_memory as symm_mem

            buf = symm_mem.empty(_lib.PEER_BUF_FLOATS, dtype=torch.float32, device=self.device)
            buf.zero_()
            torch.cuda.synchronize(self.device)
        except Exception as e:  # noqa: BLE001
            why = repr(e)
        if not self._agree(why is None):
            return why or "another rank could not allocate symmetric memory"
        hdl = None
        try:  # phase 2, collective: every rank is here
            hdl = symm_mem.rendezvous(buf, dist.group.WORLD)
        except Exception as e:  # noqa: BLE001
            why = repr(e)
        if not self._agree(why is None):
            return why or "another rank could not map the peers' buffers"
        dist.barrier()  # every buffer is zero before anybody's first word can arrive
        # NVLS: a multicast mapping of the same buffers, when the fabric has one -- a push then leaves the SM once.  Every
        # rank decides alike
        mc = int(getattr(hdl, "multicast_ptr", 0) or 0) if self.use_multicast else 0
        mc_ok = mc != 0 and buf.data_ptr() == int(hdl.buffer_ptrs[dist.get_rank()])
        self._finish_peers(hdl.buffer_ptrs, mc if self._agree(mc_ok) else 0, (buf, hdl))
        return None

    def _setup_peers_ipc(self):
        """Buffers allocated by the library and shared as CUDA IPC handles (nfsp_peer_buffer_*); no multicast mapping."""
        world, rank, dev = dist.get_world_size(), dist.get_rank(), self.device.index
        mine, handle, why = C.c_void_p(), C.create_string_buffer(64), None
        try:
            check(lib().nfsp_peer_buffer_create(dev, C.byref(mine), handle))
        except Exception as e:  # noqa: BLE001
            why = repr(e)
        if not self._agree(why is None):
            if mine.value:
                lib().nfsp_peer_buffer_destroy(dev, mine)
            return why or "another rank could not create its exchange buffer"
        handles = [None] * world
        dist.all_gather_object(handles, handle.raw)  # collective: every rank is here
        ptrs, opened = [0] * world, []
        try:
            for r in range(world):
                if r == rank:
                    ptrs[r] = mine.value
                    continue
                q = C.c_void_p()
                check(lib().nfsp_peer_buffer_open(dev, handles[r], C.byref(q)))
                ptrs[r] = q.value
                opened.append(q)
        except Exception as e:  # noqa: BLE001
            why = repr(e)
        if not self._agree(why is None):
            for q in opened:
                lib().nfsp_peer_buffer_close(dev, q)
            dist.barrier()  # nobody maps a buffer any more: its owner may free it
            lib().nfsp_peer_buffer_destroy(dev, mine)
            return why or "another rank could not map the peers' buffers"
        dist.barrier()
        self._finish_peers(ptrs, 0, ("ipc", mine, opened))
        return None

    def close_peers(self):
        """Collective: unmap and free the exchange buffers (the IPC transport owns raw CUDA allocations; symmetric memory
        is released with its tensors).  The learner continues on the NCCL path afterwards."""
        keep = getattr(self, "_peer_keep", None)
        if getattr(self, "_peers", None) is None or keep is None:
            return
        torch.cuda.synchronize(self.device)
        dist.barrier()  # no fit kernel of any rank still polls or pushes
        if keep[0] == "ipc":
            dev = self.device.index
            for q in keep[2]:
                lib().nfsp_peer_buffer_close(dev, q)
            dist.barrier()  # nobody maps a buffer any more: its owner may free it
            lib().nfsp_peer_buffer_destroy(dev, keep[1])
        self._peers = self._peer_keep = None
        self._peer_note = "peer exchange closed"

    def check_peers(self):
        """Raises if a peer GPU failed to answer during any gradient exchange so far (the kernel then gave up after ~2 s,
        skipped that net's remaining SGD steps and wrote NaN weights for it, so the failure cannot go unnoticed; the
        replicas are no longer identical and the run must be resumed from its last checkpoint, `checkpoint.load` /
        `main.py --resume DIR`).  Reads one device word (syncs):
        called by update(sync=True), by PipelinedTrainer.finish() and every `peer_check_every` updates."""
        if self._peers is not None and int(self._peer_err.item()):
            raise RuntimeError("a peer GPU did not answer during the gradient exchange: the weights of this update are "
                               "invalid (NaN) and the replicas have diverged; resume the run from its last checkpoint "
                               "(main.py --resume DIR, with the --checkpoint DIR it was trained with)")

    @property
    def fit_steps(self) -> int:
        """SGD (or Adam) steps of one fit: `epochs` passes over the minibatch in slices of `fit_batch` rows."""
        return self.epochs * ((self.minibatch + self.fit_batch - 1) // self.fit_batch)

    # ---- Adam's state ----
    def adam_state(self, out=None):
        """The nfsp_adam_state of this learner (moments and steps so far), written into `out` if given."""
        s = _lib.AdamState() if out is None else out
        s.d_m, s.d_v = self.adam_m.data_ptr(), self.adam_v.data_ptr()
        for k in range(4):
            s.t0[k] = self.adam_t[k]
        return s

    def _adam_advance(self, mask, steps):
        """The nets in `mask` have taken `steps` more Adam steps (the others none: they did not move)."""
        for k in range(4):
            if (mask >> k) & 1:
                self.adam_t[k] += steps

    # ---- the whole fit() in one launch: one GPU, or several with the all-reduce of every SGD step inside it ----
    def _fit_one_launch(self, idx_rl, idx_sl, mask, w_in=None, w_out=None):
        io, lr = self._fit_args(idx_rl, idx_sl, mask, w_in)
        args = (C.byref(io), self.minibatch, self.fit_batch, self.epochs, (C.c_float * 4)(*lr),
                _ptr(self.sp.weights if w_out is None else w_out))
        adam = self.optimizer == "adam"
        if self._peers is None:
            if adam:
                # the moments are updated in place on this stream.  Beside the pipelined trainer's next rollout that is
                # safe: a rollout reads the acting images and the memories, never the learner's moments
                check(lib().nfsp_learner_fit_adam(*args, C.byref(self.adam_state()), _stream(self.device)))
                self._adam_advance(mask, self.fit_steps)
                return
            return check(lib().nfsp_learner_fit(*args, _stream(self.device)))
        self._peers.epoch0 = self._epoch & 0xFFFFFFFF
        if adam:
            check(lib().nfsp_learner_fit_peers_adam(*args, C.byref(self._peers), C.byref(self.adam_state()),
                                                    _stream(self.device)))
            self._adam_advance(mask, self.fit_steps)
        else:
            check(lib().nfsp_learner_fit_peers(*args, C.byref(self._peers), _stream(self.device)))
        self._epoch += self.fit_steps

    # ---- one SGD step for all four nets -------------------------------------------------------------
    def _step(self, idx_rl, idx_sl, row0, rows, mask):
        sp = self.sp
        io, lr = self._fit_args(idx_rl, idx_sl, mask, row0=row0, rows=rows)
        check(lib().nfsp_learner_grads(C.byref(io), _stream(self.device)))
        world = self._world()
        if world > 1:  # C1 (gradients) + C2 (exploitability stats) in one collective
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)
        lr = (C.c_float * 4)(*lr)
        if self.optimizer == "adam":
            check(lib().nfsp_adam_apply(_ptr(sp.weights), _ptr(self.flat), C.byref(lr), 1.0 / world, mask,
                                        C.byref(self.adam_state()), _stream(self.device)))
            self._adam_advance(mask, 1)
            return
        check(lib().nfsp_sgd_apply(_ptr(sp.weights), _ptr(self.flat), C.byref(lr), 1.0 / world, _stream(self.device)))

    def _ready_mask(self):
        """agent.py:215,259: a net trains only once its memory holds more than a minibatch.  Memories never shrink,
        so once all four are ready the (host-synchronising) size reads stop."""
        if getattr(self, "_all_ready", False):
            return 15
        sp = self.sp
        mask = 0
        for p in range(2):
            if sp.sl[p].size() > self.minibatch:
                mask |= 1 << (2 * p)
            if sp.rl[p].size() > self.minibatch:
                mask |= 1 << (2 * p + 1)
        if self._world() > 1:  # every rank must take the same decision or the replicas diverge
            m = torch.tensor([(mask >> k) & 1 for k in range(4)], dtype=torch.int32, device=self.device)
            dist.all_reduce(m, op=dist.ReduceOp.MIN)
            mask = sum(int(v) << k for k, v in enumerate(m.tolist()))
        self._all_ready = mask == 15
        return mask

    def update(self, sync=True, weights_in=None, weights_out=None, pack=True, on_gathered=None, presampled_rings=False):
        """update_strategy() of both agents.  Returns a dict of statistics; with sync=False nothing is read back
        from the device (the loss / exploitability-proxy entries are then the previous synchronised values).
        weights_in / weights_out (float32 [4, 2179] device tensors): train FROM / INTO these instead of the acting
        weights of the SelfPlay object, and with pack=False leave the acting nets alone -- what PipelinedTrainer needs
        to run this update beside the next rollout.  Only the one-launch fit supports it.
        on_gathered: a callable; the sampled records are first copied out of the memories and the callable is invoked
        right after that copy is enqueued (PipelinedTrainer records an event there: from then on the memories may change).
        presampled_rings: presample_rings() has already drawn and copied the RL minibatches of this update."""
        sp = self.sp
        mask = self._ready_mask()
        if (weights_in is not None or weights_out is not None) and not self.one_launch:
            raise ValueError("weights_in / weights_out need the one-launch fit (fused=True; peers when world > 1)")
        w_new = sp.weights if weights_out is None else weights_out
        if mask == 0:
            if weights_out is not None:
                weights_out.copy_(sp.weights if weights_in is None else weights_in)
            return {"trained": 0}
        self._begin_update(mask)
        if presampled_rings and on_gathered is None:
            raise ValueError("presampled_rings belongs to the snapshot path (on_gathered)")
        idx_rl, idx_sl = self._sample_positions(snapshot=on_gathered is not None, which="sl" if presampled_rings else "both")
        if on_gathered is not None:
            on_gathered()
        stats = None
        if self.one_launch:
            # one launch for the 8 SGD steps; with peers the per-step all-reduce happens inside it over NVLink
            self._fit_one_launch(idx_rl, idx_sl, mask, weights_in, weights_out)
            stats = self.flat[GRAD:].clone()     # statistics of the first step, as below
        else:
            for _ in range(self.epochs):         # Keras fit(epochs=2), batch_size 32 (agent.py:243,261)
                for row0 in range(0, self.minibatch, self.fit_batch):
                    self._step(idx_rl, idx_sl, row0, min(self.fit_batch, self.minibatch - row0), mask)
                    if stats is None:            # exploitability proxy of the sampled batch, first pass
                        stats = self.flat[GRAD:].clone()
        return self._finish_update(mask, stats, sync, w_new, pack)

    def _begin_update(self, mask):
        """First half of update() once the ready mask is known (non-zero): agent.py:216's iteration step.  The sampling
        and the fit follow; _finish_update() is the second half."""
        for p in range(2):
            if (mask >> (2 * p + 1)) & 1:
                self.iteration[p] += 1          # agent.py:216

    def _finish_update(self, mask, stats, sync, w_new, pack):
        """Second half of update(), after the fit wrote w_new and its first step's statistics `stats` (a device tensor):
        the statistics (read back with sync), then each player's schedules -- iteration, temperature, target-net copy,
        learning-rate decay, epsilon -- and (pack) the acting images rebuilt."""
        sp = self.sp
        if sync:
            self._loss = stats.cpu().tolist()
        if sync or (self._peers is not None and (self.updates + 1) % self.peer_check_every == 0):
            self.check_peers()
        s = getattr(self, "_loss", [0.0] * N_STATS)
        for p in range(2):
            if (mask >> (2 * p + 1)) & 1:
                if sync:
                    self.exploitability[p] = s[p] / max(s[2 + p], 1.0)   # agent.py:234-238 (mean over ranks too)
                self.iteration[p] += 1                               # agent.py:245
                it = self.iteration[p]
                self.temp[p] = (1 + 0.02 * math.sqrt(it)) ** (-1)    # agent.py:247
                if self.target_update_count[p] % self.target_update_rate == 0:   # agent.py:266-273
                    self.target[p].copy_(w_new[2 * p + 1])
                self.target_update_count[p] += 1
                self.lr_br[p] = self.lr_br0 / (1 + 0.003 * math.sqrt(it))        # agent.py:251
        for p in range(2):
            if (mask >> (2 * p + 1)) & 1:   # each agent decays its own epsilon by its own iteration count
                sp.epsilons[p] = sp.epsilons[p] ** 1 / self.iteration[p]         # agent.py:253 (sic)
        if pack:
            sp.set_weights(sp.weights)  # rebuild the kernels' weight images
        self.updates += 1
        return {"trained": mask, "exploitability": sum(self.exploitability), "loss": s[4:8], "epsilon": sp.epsilon,
                "lr_br": list(self.lr_br)}

    # ---- checkpoint / resume (the SelfPlay it trains has its own state dict) ----
    def _shape(self):
        d = dict(minibatch=self.minibatch, fit_batch=self.fit_batch, epochs=self.epochs,
                 terminal_bootstraps=self.terminal_bootstraps, others_to_target=self.others_to_target, fused=self.fused)
        if self.optimizer != "sgd":  # an SGD learner's state is what it was before Adam existed: old checkpoints load
            d["optimizer"] = self.optimizer
        return d

    _SCALARS = dict(gamma=float, lr_br0=float, lr_ar=float, target_update_rate=int, iteration=(int, 2),
                    target_update_count=(int, 2), temp=(float, 2), lr_br=(float, 2), exploitability=(float, 2), updates=int)

    def state_dict(self) -> dict:
        """Host copy of the target nets, the schedules and the last read-back statistics, with the learner's shape.
        Synchronises the device.  The peer exchange's epoch is not part of it: a learner maps fresh, zeroed exchange
        buffers and starts at epoch 0."""
        torch.cuda.synchronize(self.device)
        d = dict(shape=self._shape(), target=self.target.cpu(), loss=list(getattr(self, "_loss", [])) or None)
        for k in self._SCALARS:
            v = getattr(self, k)
            d[k] = list(v) if isinstance(v, list) else v
        if self.optimizer == "adam":
            d.update(adam_m=self.adam_m.cpu(), adam_v=self.adam_v.cpu(), adam_t=list(self.adam_t))
        return d

    def check_state_dict(self, d):
        """Raises ValueError, naming the field, if load_state_dict(d) would refuse d."""
        check_fields(d, "Learner")
        check_fields(d.get("shape"), "Learner", **self._shape())
        saved = d["shape"].get("optimizer", "sgd")
        if saved != self.optimizer:  # check_fields does not see a shape key this learner lacks
            raise ValueError("Learner: optimizer is %r in the state but %r here" % (saved, self.optimizer))
        if self.optimizer == "adam":
            for k in ("adam_m", "adam_v"):
                check_tensor(d.get(k), k, "Learner", tuple(self.adam_m.shape), torch.float32)
            check_numbers(d, "Learner", adam_t=(int, 4))
            if any(t > 2 ** 62 for t in d["adam_t"]):  # nfsp_adam_state.t0 holds at most 2^62
                raise ValueError("Learner: adam_t must be at most 2**62, got %r" % (d["adam_t"],))
        check_tensor(d.get("target"), "target", "Learner", tuple(self.target.shape), torch.float32)
        check_numbers(d, "Learner", **self._SCALARS)
        if d.get("loss") is not None:
            check_numbers(d, "Learner", loss=(float, N_STATS))
        if d["target_update_rate"] < 1:
            raise ValueError("Learner: target_update_rate must be at least 1")

    def load_state_dict(self, d):
        """Validates d, then restores it.  Learning rates, gamma and the target update rate come from d."""
        self.check_state_dict(d)
        torch.cuda.synchronize(self.device)
        self.target.copy_(d["target"])
        if self.optimizer == "adam":
            self.adam_m.copy_(d["adam_m"])
            self.adam_v.copy_(d["adam_v"])
            self.adam_t = list(d["adam_t"])
        for k, kind in self._SCALARS.items():
            setattr(self, k, list(d[k]) if isinstance(kind, tuple) else d[k])
        self.gamma, self.lr_br0, self.lr_ar = float(self.gamma), float(self.lr_br0), float(self.lr_ar)
        self.__dict__.pop("_loss", None)
        if d["loss"] is not None:
            self._loss = list(d["loss"])
        self._all_ready = False  # the memories may hold fewer records now: read their sizes again
        torch.cuda.synchronize(self.device)


class PipelinedTrainer:
    """Self-play with the learner BESIDE the actor: update j runs on its own stream while rollout j+1 plays.

    The sequential loop (main.train, agent.py:130-156) is rollout -> memories -> update -> rollout with the new nets.
    Here rollout j+1 starts right after the memories of step j are written, with the nets that update j is still
    reading (W_j); update j's result W_{j+1} is picked up by rollout j+2.  So the acting nets lag ONE update behind the
    sequential loop -- NFSP learns off-policy from its memories, the reference's own update cadence is arbitrary
    (every 128 decisions of a batch-1 game) -- and in exchange the learner's time (and, with several GPUs, its gradient
    exchange) disappears behind the rollout.  Mechanics: the fit trains from one weight tensor into another
    (two tensors, alternating), so the acting images can be rebuilt from W_j while update j reads it; the rollout's
    persistent grid leaves `reserve_sms` SMs free (the fit is four CTAs that need an SM each); the update first copies
    its sampled records out of the memories (24 KB) and an event after that copy lets the next rollout -- which writes the
    rings in place with direct_rings -- and the next insert go ahead while the fit runs.  Deterministic: the same weights, memories and games as the
    sequential loop run with that lag (tests/test_gpu_train.py)."""

    def __init__(self, selfplay, learner, reserve_sms=4):
        if not learner.one_launch:
            raise RuntimeError("PipelinedTrainer needs the one-launch fit: fused=True and, with several GPUs, minibatch <= %d, fit batch "
                               "<= %d and peer memory (%s)" % (_lib.FIT_ROWS_MAX_MINIBATCH, _lib.FIT_ROWS_MAX_STEP,
                                                               getattr(learner, "_peer_note", "see Learner._setup_peers")))
        self.sp, self.learner, self.reserve_sms = selfplay, learner, int(reserve_sms)
        self.w = [selfplay.weights.clone(), selfplay.weights.clone()]  # W_j lives in w[j % 2]
        self.stream = torch.cuda.Stream(selfplay.device)
        self.flushed = torch.cuda.Event()
        self.gathered = torch.cuda.Event()                             # update j has copied its sampled records
        self.rolled, self.rings_sampled = torch.cuda.Event(), torch.cuda.Event()
        self.updated = [torch.cuda.Event(), torch.cuda.Event()]        # update j records updated[j % 2]
        self.j = 0

    def step(self, n_steps, sync=False):
        """One iteration; sync=True also reads this update's statistics back (the host then waits for the update)."""
        sp, j = self.sp, self.j
        main = torch.cuda.current_stream(sp.device)
        if j >= 2:
            main.wait_event(self.updated[j % 2])          # update j-2 wrote W_{j-1}
        sp.set_weights(self.w[(j - 1) % 2] if j >= 1 else self.w[0])   # acting nets: W_{j-1} (W_0 for the first two steps)
        # update j-1 works on snapshots of its sampled records: once they exist the memories may change.  The rings'
        # snapshot is taken right after rollout j-1 wrote them (beside the insert launch), so with direct_rings the next
        # rollout -- which writes the rings in place -- finds it done; the reservoirs' snapshot gates the next insert
        if j >= 1 and sp.direct_rings:
            main.wait_event(self.rings_sampled)
        sp.rollout(n_steps, insert=False, reserve_sms=self.reserve_sms)
        early = sp.direct_rings and self.learner._ready_mask() == 15
        if early:
            self.rolled.record(main)
            self.stream.wait_event(self.rolled)
            with torch.cuda.stream(self.stream):
                self.learner.presample_rings()
                self.rings_sampled.record(self.stream)
        if j >= 1:
            main.wait_event(self.gathered)
        sp.flush()
        self.flushed.record(main)
        self.stream.wait_event(self.flushed)
        with torch.cuda.stream(self.stream):
            out = self.learner.update(sync=sync, weights_in=self.w[j % 2], weights_out=self.w[(j + 1) % 2], pack=False,
                                      on_gathered=lambda: self.gathered.record(self.stream), presampled_rings=early)
            if not early:
                self.rings_sampled.record(self.stream)
            self.updated[j % 2].record(self.stream)
        self.j = j + 1
        return out

    def finish(self):
        """Wait for the last update and make its weights the acting nets; returns them."""
        torch.cuda.current_stream(self.sp.device).wait_stream(self.stream)
        self.learner.check_peers()
        self.sp.set_weights(self.w[self.j % 2])
        return self.w[self.j % 2]

    def state_dict(self) -> dict:
        """Host copies of the two weight tensors (W_j and W_{j-1}: the next step acts with one and trains from the
        other) and j, once the update in flight has written its result.  The SelfPlay and the Learner have their own
        state dicts."""
        torch.cuda.current_stream(self.sp.device).wait_stream(self.stream)
        torch.cuda.synchronize(self.sp.device)
        return dict(w=[w.cpu() for w in self.w], j=self.j)

    def check_state_dict(self, d):
        """Raises ValueError, naming the field, if load_state_dict(d) would refuse d."""
        check_fields(d, "PipelinedTrainer")
        check_numbers(d, "PipelinedTrainer", j=int)
        if not (isinstance(d.get("w"), list) and len(d["w"]) == 2):
            raise ValueError("PipelinedTrainer: w must be a list of two weight tensors")
        for k in range(2):
            check_tensor(d["w"][k], "w[%d]" % k, "PipelinedTrainer", tuple(self.w[k].shape), torch.float32)

    def load_state_dict(self, d):
        """Validates d, then restores it: the next step() acts with the nets the saved trainer's next step would."""
        self.check_state_dict(d)
        torch.cuda.current_stream(self.sp.device).wait_stream(self.stream)
        for w, src in zip(self.w, d["w"]):
            w.copy_(src)
        self.j = d["j"]
        torch.cuda.synchronize(self.sp.device)


# ---- single-game drop-in: agent.Agent.update_*_network ----------------------------------------------------
def _agent_fit(agent, net):
    """Keras fit(epochs=2, batch 32) of one of the agent's nets on a fresh sample of its own memory."""
    dev = agent.device
    zeros = torch.zeros(_lib.NET_PARAMS, dtype=torch.float32, device=dev)
    w = torch.stack([agent.weights[agent.AVG], agent.weights[agent.BR], zeros, zeros]).contiguous()
    target = torch.stack([agent.weights[agent.TARGET], zeros]).contiguous()
    flat = torch.zeros(GRAD + N_STATS, dtype=torch.float32, device=dev)
    mem = agent._rl_memory.memory if net == 1 else agent._sl_memory.memory
    idx = mem.sample_slots(agent.minibatch_size)[0]
    io = _lib.LearnerIO()
    io.d_weights, io.d_target_weights = w.data_ptr(), target.data_ptr()
    io.d_rl[0], io.d_rl_idx[0] = agent._rl_memory.memory.store.data_ptr(), idx.data_ptr()
    io.d_sl[0], io.d_sl_idx[0] = agent._sl_memory.memory.store.data_ptr(), idx.data_ptr()
    io.gamma, io.net_mask, io.terminal_bootstraps = agent.gamma, 1 << net, 0
    io.d_grad, io.d_stats = flat.data_ptr(), flat[GRAD:].data_ptr()
    lr = (C.c_float * 4)(agent.lr_ar, agent.lr_br_now, 0.0, 0.0)
    first = None
    for _ in range(2):
        for row0 in range(0, agent.minibatch_size, 32):
            io.row0, io.rows = row0, min(32, agent.minibatch_size - row0)
            check(lib().nfsp_learner_grads(C.byref(io), _stream(dev)))
            if first is None:
                first = flat[GRAD:].clone()
            check(lib().nfsp_sgd_apply(_ptr(w), _ptr(flat), C.byref(lr), 1.0, _stream(dev)))
    agent.weights[agent.AVG], agent.weights[agent.BR] = w[0].clone(), w[1].clone()
    agent._upload()
    return first.cpu().tolist()


def update_best_response(agent):
    """agent.py:209-253."""
    if not hasattr(agent, "lr_br_now"):
        agent.lr_br_now = agent.lr_br
    agent.iteration += 1
    s = _agent_fit(agent, 1)
    agent.exploitability = s[0] / max(s[2], 1.0)
    agent.iteration += 1
    agent.temp = (1 + 0.02 * math.sqrt(agent.iteration)) ** (-1)
    agent.update_br_target_network()
    agent.lr_br_now = agent.lr_br / (1 + 0.003 * math.sqrt(agent.iteration))
    agent.epsilon = agent.epsilon ** 1 / agent.iteration


def update_average_policy(agent):
    """agent.py:255-264."""
    if not hasattr(agent, "lr_br_now"):
        agent.lr_br_now = agent.lr_br
    _agent_fit(agent, 0)
