"""Batched engines over the C ABI: N independent Leduc games per call, tensors stay on the GPU.

These are the classes the single-game drop-ins (leduc/env.py, leduc/newenv.py, agent/agent.py,
utils/*.py of this package) are thin batch-of-1 views of.  Names follow the reference's domain:
games, hands, deals, transitions, memories.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import check, lib


def _device(device) -> torch.device:
    if not torch.cuda.is_available():
        raise _lib.NfspError("no CUDA device: this package has no CPU path")
    d = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if d.type != "cuda":
        raise _lib.NfspError("device must be a CUDA device, got %s" % d)
    return torch.device("cuda", d.index if d.index is not None else torch.cuda.current_device())


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream(dev: torch.device):
    """The caller's current CUDA stream on `dev` as a raw handle (asked for on every call: streams change under
    `torch.cuda.stream(...)`).  torch's raw getter when there is one: the Stream object costs ~3 us per call on the
    host path of every step."""
    if _raw_stream is not None and dev.index is not None:
        return C.c_void_p(_raw_stream(dev.index))
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _as(t, dtype, dev, shape=None):
    """Host or device array-like -> contiguous device tensor of `dtype` (a copy only when needed)."""
    if t is None:
        return None
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(np.asarray(t))
    t = t.to(device=dev, dtype=dtype).contiguous()
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise ValueError("expected shape %s, got %s" % (tuple(shape), tuple(t.shape)))
    return t


def check_fields(d, where, **expected):
    """State-dict validation: raises ValueError naming the first field whose saved value differs from `expected`."""
    if not isinstance(d, dict):
        raise ValueError("%s: the state is a %s, not a dict" % (where, type(d).__name__))
    for k, v in expected.items():
        if k not in d:
            raise ValueError("%s: the state has no field %r" % (where, k))
        if type(d[k]) is not type(v) or d[k] != v:
            raise ValueError("%s: %s is %r in the state but %r here" % (where, k, d[k], v))


def check_tensor(t, name, where, shape, dtype):
    """State-dict validation: t (the field `name`) is a host tensor of `shape` and `dtype`."""
    if not (isinstance(t, torch.Tensor) and t.device.type == "cpu" and t.dtype == dtype and tuple(t.shape) == tuple(shape)):
        got = "%s %s" % (t.dtype, tuple(t.shape)) if isinstance(t, torch.Tensor) else type(t).__name__
        raise ValueError("%s: %s must be a host %s tensor of shape %s, got %s" % (where, name, dtype, tuple(shape), got))


def check_numbers(d, where, below=None, **kinds):
    """State-dict validation of a dict: each named field holds a non-negative int (kind int), a number (kind float) or a
    list of n of them (kind (int, n) / (float, n)).  `below` maps an int field to the exclusive bound of what holds it
    (2**64 for a uint64 counter, 2**63 for an int64 tensor), so a counter that cannot be stored is refused up front."""
    for k, bound in (below or {}).items():
        v = d.get(k)
        if type(v) is int and v >= bound:
            raise ValueError("%s: %s must be below 2**%d, got %r" % (where, k, bound.bit_length() - 1, v))
    for k, kind in kinds.items():
        kind, n = kind if isinstance(kind, tuple) else (kind, None)
        v = d.get(k)
        if n is None:
            vals = [v]
        else:
            vals = v if isinstance(v, list) and len(v) == n else None
        if kind is int:
            ok = vals is not None and all(type(x) is int and x >= 0 for x in vals)
        else:
            ok = vals is not None and all(type(x) in (int, float) for x in vals)
        if not ok:
            raise ValueError("%s: %s must be %s%s, got %r" % (where, k, "a list of %d " % n if n else "a ",
                                                             "non-negative int" if kind is int else "number", v))


def expand_obs(masks: torch.Tensor) -> torch.Tensor:
    """30-bit observation masks -> float32 [n, 30] (the reference's state vector, newenv.py:118-122)."""
    m = masks.contiguous().view(torch.int32).reshape(-1)
    out = torch.empty((m.numel(), _lib.OBS_DIM), dtype=torch.float32, device=m.device)
    check(lib().nfsp_expand_obs(_ptr(m), m.numel(), _ptr(out), _stream(m.device)))
    return out


def obs_to_mask(x) -> torch.Tensor:
    """float 0/1 state vectors [..., 30] -> int32 masks [...]; raises on non-binary input (the packed
    record formats only hold the reference's binary observations)."""
    x = torch.as_tensor(x)
    if x.shape[-1] != _lib.OBS_DIM:
        raise ValueError("state vectors must have 30 entries")
    if not bool(((x == 0) | (x == 1)).all()):
        raise ValueError("state vectors must be 0/1 (newenv.py:118 encoding)")
    w = (2 ** torch.arange(_lib.OBS_DIM, dtype=torch.int64, device=x.device))
    return (x.to(torch.int64) * w).sum(-1).to(torch.int32)


class _EnvBase:
    rules = None

    def __init__(self, n_games: int, seed: int = 1234, game0: int = 0, device=None):
        self.device = _device(device)
        self.n = int(n_games)
        self._h = C.c_void_p()
        check(lib().nfsp_env_create(self.rules, self.n, seed & (2 ** 64 - 1), game0, self.device.index,
                                    C.byref(self._h)))
        self.seed, self.game0 = seed, game0

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().nfsp_env_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def step_counter(self) -> int:
        return int(lib().nfsp_env_step_counter(self._h))

    @step_counter.setter
    def step_counter(self, v: int):
        check(lib().nfsp_env_set_step_counter(self._h, int(v)))

    def state_words(self) -> torch.Tensor:
        """A copy of the packed 64-bit game words (checkpointing, multi-GPU invariance tests)."""
        out = torch.empty(self.n, dtype=torch.int64, device=self.device)
        check(lib().nfsp_env_save_state(self._h, _ptr(out), _stream(self.device)))
        return out

    def load_state_words(self, words: torch.Tensor):
        w = _as(words, torch.int64, self.device, (self.n,))
        check(lib().nfsp_env_load_state(self._h, _ptr(w), _stream(self.device)))


class BatchedNfspEnv(_EnvBase):
    """N games of leduc/newenv.py.  `step` is newenv.Env.step for every game in one kernel launch."""

    rules = _lib.RULES_NFSP

    def __init__(self, n_games, seed=1234, game0=0, device=None, eta=0.1):
        super().__init__(n_games, seed, game0, device)
        self.eta = float(eta)

    def reset(self, dealer=None):
        """newenv.Env.reset(dealer) for every game; dealer: None (game id & 1), int, or [n] array."""
        if dealer is not None and not isinstance(dealer, torch.Tensor) and np.ndim(dealer) == 0:
            dealer = torch.full((self.n,), int(dealer), dtype=torch.int8)
        d = _as(dealer, torch.int8, self.device, (self.n,))
        check(lib().nfsp_env_reset(self._h, _ptr(d), self.eta, _stream(self.device)))

    def set_hands(self, dealer, cards, policy=None):
        if not (isinstance(cards, torch.Tensor) and cards.is_cuda):  # host input: ranks are 0 (Ace), 1, 2 (deck.py:21-33)
            chk = np.asarray(cards)
            if chk.size and (chk.min() < 0 or chk.max() > 2):
                raise ValueError("card ranks must be 0, 1 or 2")
        d = _as(dealer, torch.int8, self.device, (self.n,))
        c = _as(cards, torch.int8, self.device, (self.n, 3))
        p = _as(policy, torch.int8, self.device, (self.n, 2))
        check(lib().nfsp_env_set_hands(self._h, _ptr(d), _ptr(c), _ptr(p), _stream(self.device)))

    def step(self, actions=None, players=None, n_steps=1, auto_reset=True, trace=False):
        """actions: None (uniform Philox) or int8 [n_steps, n] codes 0 fold / 1 call / 2 raise /
        3 all-zero vector / -1 random; players: None = main.train's turn order.  Returns the trace
        planes dict when trace=True."""
        shape = (n_steps, self.n)
        a = _as(actions, torch.int8, self.device)
        p = _as(players, torch.int8, self.device)
        if a is not None:
            a = a.reshape(shape)
        if p is not None:
            p = p.reshape(shape)
        tr = torch.empty((3,) + shape, dtype=torch.int32, device=self.device) if trace else None
        check(lib().nfsp_env_step(self._h, _ptr(a), _ptr(p), n_steps, int(bool(auto_reset)), self.eta, _ptr(tr),
                                  _stream(self.device)))
        return None if tr is None else decode_trace(tr)

    def do_action(self, actions, players):
        """newenv.Env.do_action (newenv.py:131-178) on its own: int8 codes as in step(), one player index per game.
        Returns a bool tensor: the player folded."""
        a = _as(actions, torch.int8, self.device, (self.n,))
        p = _as(players, torch.int8, self.device, (self.n,))
        fold = torch.empty(self.n, dtype=torch.int8, device=self.device)
        check(lib().nfsp_env_do_action(self._h, _ptr(a), _ptr(p), _ptr(fold), _stream(self.device)))
        return fold.bool()

    def get_state(self, player):
        """newenv.Env.get_state(p), packed: (s mask, last action id, reward, s2 mask, terminated)."""
        per_game = isinstance(player, (torch.Tensor, np.ndarray, list, tuple))
        pl = _as(player, torch.int8, self.device, (self.n,)) if per_game else None
        s = torch.empty(self.n, dtype=torch.int32, device=self.device)
        s2 = torch.empty_like(s)
        r = torch.empty(self.n, dtype=torch.float32, device=self.device)
        t = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        a = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        check(lib().nfsp_env_observe(self._h, _ptr(pl), -1 if per_game else int(player), _ptr(s), _ptr(s2), _ptr(r),
                                     _ptr(t), _ptr(a), _stream(self.device)))
        return s, a, r, s2, t

    FIELDS = ("hist", "c0", "c1", "pub", "dealer", "round", "k", "bets0", "bets1", "terminated", "need_reset", "pol0",
              "pol1", "last_a0", "last_a1", "nz0", "nz1", "obs0", "obs1", "snap0", "snap1", "rew0_half", "rew1_half",
              "anomaly")

    def export(self):
        out = torch.empty((self.n, _lib.EXPORT_FIELDS), dtype=torch.int32, device=self.device)
        check(lib().nfsp_env_export(self._h, _ptr(out), _stream(self.device)))
        return {k: out[:, i] for i, k in enumerate(self.FIELDS)}


def decode_trace(tr: torch.Tensor):
    """uint32 planes [3, n_steps, n] -> named fields (DESIGN.md "trace record")."""
    obs, rew, misc = tr[0], tr[1], tr[2]
    return dict(raw=tr, obs=obs & 0x3FFFFFFF, terminated=(obs >> 30) & 1, player=(obs >> 31) & 1,
                reward=rew.view(torch.float32), action=misc & 3, effective=(misc >> 2) & 3, round=(misc >> 4) & 1,
                dealer=(misc >> 5) & 1, c0=(misc >> 6) & 3, c1=(misc >> 8) & 3, pub=(misc >> 10) & 3,
                bets0=(misc >> 13) & 15, bets1=(misc >> 17) & 15, started=(misc >> 21) & 1,
                pol0=(misc >> 22) & 1, pol1=(misc >> 23) & 1)


class BatchedLegacyEnv(_EnvBase):
    """N games of leduc/env.py (the README's documented env)."""

    rules = _lib.RULES_LEGACY
    FIELDS = ("c0", "c1", "left0", "left1", "pot0", "pot1", "term0", "term1", "st_pot0", "st_pot1", "st_act0",
              "st_act1", "rew0", "rew1")

    def reset(self):
        check(lib().nfsp_legacy_reset(self._h, _stream(self.device)))

    def set_hands(self, cards):
        c = _as(cards, torch.int8, self.device, (self.n, 2))
        check(lib().nfsp_legacy_set_hands(self._h, _ptr(c), _stream(self.device)))

    def step(self, actions, player):
        per_game = isinstance(player, (torch.Tensor, np.ndarray, list, tuple))
        pl = _as(player, torch.int8, self.device, (self.n,)) if per_game else None
        a = _as(actions, torch.int8, self.device, (self.n,))
        check(lib().nfsp_legacy_step(self._h, _ptr(a), _ptr(pl), -1 if per_game else int(player),
                                     _stream(self.device)))

    def get_new_state(self, player, want_out=True):
        per_game = isinstance(player, (torch.Tensor, np.ndarray, list, tuple))
        pl = _as(player, torch.int8, self.device, (self.n,)) if per_game else None
        out = torch.empty((self.n, 5), dtype=torch.int32, device=self.device) if want_out else None
        check(lib().nfsp_legacy_get_new_state(self._h, _ptr(pl), -1 if per_game else int(player), _ptr(out),
                                              _stream(self.device)))
        return out

    def rollout(self, n_iters=1, actions=None, trace=False):
        a = _as(actions, torch.int8, self.device)
        if a is not None:
            a = a.reshape(n_iters, self.n, 2)
        rec = torch.empty((3, n_iters, self.n, 2), dtype=torch.int32, device=self.device) if trace else None
        check(lib().nfsp_legacy_rollout(self._h, _ptr(a), n_iters, _ptr(rec), _stream(self.device)))
        if rec is None:
            return None
        w = rec[0]
        sb = lambda x: ((x & 0xFF) ^ 0x80) - 0x80  # noqa: E731  signed byte
        return dict(raw=rec, card=sb(w), pub=sb(w >> 8), pot=sb(w >> 16), terminal=sb(w >> 24), reward=rec[1],
                    action=rec[2] & 3, left=((rec[2] >> 2) & 7) - 1, pot_own=(rec[2] >> 5) & 7,
                    started=(rec[2] >> 8) & 1)

    def export(self):
        out = torch.empty((self.n, _lib.LEGACY_EXPORT_FIELDS), dtype=torch.int32, device=self.device)
        check(lib().nfsp_legacy_export(self._h, _ptr(out), _stream(self.device)))
        return {k: out[:, i] for i, k in enumerate(self.FIELDS)}


# ---------------------------------------------------------------------------------------------
# memories (16-byte packed records in HBM)
# ---------------------------------------------------------------------------------------------
RL_DT = np.dtype([("s", "<u4"), ("s2", "<u4"), ("r", "<f4"), ("a", "u1"), ("t", "u1"), ("player", "u1"),
                  ("flags", "u1")])
SL_DT = np.dtype([("s", "<u4"), ("a", "<f4", (3,))])


class _Memory:
    is_ring = True
    slot_words = 4  # int32 words per storage slot

    def __init__(self, capacity: int, seed: int = 1234, device=None):
        self.device = _device(device)
        self.capacity = int(capacity)
        self.seed = int(seed) & (2 ** 64 - 1)
        self.store = torch.zeros((self.capacity, self.slot_words), dtype=torch.int32, device=self.device)
        self.data = self.store[:, :4]  # the 16-byte records (a strided view for the reservoir's 32-byte slots)
        self.total = torch.zeros(1, dtype=torch.int64, device=self.device)  # records ever inserted
        self._scratch = None
        self.sample_calls = 0

    def scratch(self, n_seg: int) -> torch.Tensor:
        """The insert kernel's barrier words + segment-prefix table (zeroed once, then the library's)."""
        need = int(n_seg) + _lib.INSERT_SCRATCH_WORDS
        if self._scratch is None or self._scratch.numel() < need:
            torch.cuda.current_stream(self.device).synchronize()  # an insert that still uses the old block
            self._scratch = torch.zeros(need, dtype=torch.int64, device=self.device)
        return self._scratch

    def size(self) -> int:
        """count saturates at capacity (replay_buffer.py:36-44).  Reads one device word (syncs)."""
        return int(min(int(self.total.item()), self.capacity))

    def sample_req(self, r):
        """Fills the fields of the nfsp_sample_req r that never change (memory, seed, kind); returns r."""
        r.d_mem, r.d_total, r.cap = self.store.data_ptr(), self.total.data_ptr(), self.capacity
        r.seed, r.is_ring = self.seed, int(self.is_ring)
        return r

    def next_call(self) -> int:
        """The draw counter (Philox key with the seed) of this memory's next sample_batch, advanced."""
        self.sample_calls += 1
        return self.sample_calls - 1

    def sample_slots(self, batch: int):
        idx = torch.empty(batch, dtype=torch.int64, device=self.device)
        n = torch.zeros(1, dtype=torch.int32, device=self.device)
        check(lib().nfsp_sample_indices(self.seed, self.next_call(), _ptr(self.total), self.capacity,
                                        int(self.is_ring), batch, _ptr(idx), _ptr(n), _stream(self.device)))
        return idx, n

    def records(self) -> np.ndarray:
        """Host copy of the stored records in storage-slot order (tests)."""
        dt = RL_DT if self.is_ring else SL_DT
        return np.ascontiguousarray(self.data.cpu().numpy()).view(np.uint8).reshape(-1).view(dt)[: self.size()].copy()

    def clear(self):
        self.total.zero_()

    def _shape(self):
        return dict(kind="ring" if self.is_ring else "reservoir", capacity=self.capacity, seed=self.seed,
                    mode=getattr(self, "mode", 0))

    def state_dict(self) -> dict:
        """Host copy of everything later inserts and draws depend on: the held slots store[:min(total, capacity)]
        (whole storage slots, a reservoir's stamps included), `total` and the draw counter.  Synchronises the device."""
        torch.cuda.synchronize(self.device)
        total = int(self.total.item())
        return dict(self._shape(), total=total, sample_calls=self.sample_calls,
                    slots=self.store[:min(total, self.capacity)].cpu())

    def check_state_dict(self, d, where="memory"):
        """Raises ValueError, naming the field, if load_state_dict(d) would refuse d."""
        check_fields(d, where, **self._shape())
        check_numbers(d, where, below=dict(total=2 ** 63, sample_calls=2 ** 64), total=int, sample_calls=int)
        check_tensor(d.get("slots"), "slots", where, (min(d["total"], self.capacity), self.slot_words), torch.int32)

    def load_state_dict(self, d, where="memory"):
        """Validates d, then restores it; slots past the held ones are zeroed, as in a memory that never reached them."""
        self.check_state_dict(d, where)
        held = d["slots"].shape[0]
        self.store[:held].copy_(d["slots"])
        self.store[held:].zero_()
        self.total.fill_(d["total"])
        self.sample_calls = d["sample_calls"]


class DeviceRing(_Memory):
    """Circular replay memory M_RL: FIFO ring of RL records (utils/replay_buffer.py)."""

    is_ring = True

    def insert(self, recs: torch.Tensor, counts: torch.Tensor, seg_cap: Optional[int] = None):
        """recs int32 [n_seg * seg_cap, 4] staged records, counts int32[n_seg] device counts (the batch is
        consumed: counts are zeroed).  A plain dense batch is n_seg = 1."""
        n_seg = counts.numel()
        seg_cap = recs.shape[0] // n_seg if seg_cap is None else seg_cap
        check(lib().nfsp_ring_insert(_ptr(self.store), self.capacity, _ptr(self.total), _ptr(recs), _ptr(counts),
                                     n_seg, int(seg_cap), _ptr(self.scratch(n_seg)), _stream(self.device)))

    def sample(self, batch: int):
        idx, n = self.sample_slots(batch)
        b = batch
        s = torch.empty((b, 30), dtype=torch.float32, device=self.device)
        s2 = torch.empty_like(s)
        a = torch.empty((b, 3), dtype=torch.float32, device=self.device)
        r = torch.empty(b, dtype=torch.float32, device=self.device)
        t = torch.empty(b, dtype=torch.float32, device=self.device)
        check(lib().nfsp_gather_rl(_ptr(self.store), _ptr(idx), b, _ptr(s), _ptr(a), _ptr(r), _ptr(s2), _ptr(t),
                                   _stream(self.device)))
        return s, a, r, s2, t, idx, n


class DeviceReservoir(_Memory):
    """Reservoir memory M_SL (utils/ReservoirBuffer.py).  mode "R" = Algorithm R (default, what
    BASELINE.json's north_star specifies); mode "reference" = the reference's constant-probability law."""

    is_ring = False
    slot_words = 8  # 32-byte slots: {record, int64 stamp = ticket + 1 of the owning record, int64 unused} = one DRAM sector

    def __init__(self, capacity, seed=1234, device=None, mode="R"):
        super().__init__(capacity, seed, device)
        if mode not in ("R", "reference"):
            raise ValueError("mode must be 'R' or 'reference'")
        self.mode = 0 if mode == "R" else 1

    @property
    def stamp(self) -> torch.Tensor:
        """int64 [capacity] view of the slots' stamps."""
        return self.store.view(torch.int64)[:, 2]

    def insert(self, recs, counts, seg_cap=None):
        n_seg = counts.numel()
        seg_cap = recs.shape[0] // n_seg if seg_cap is None else seg_cap
        check(lib().nfsp_reservoir_insert(_ptr(self.store), self.capacity, _ptr(self.total), _ptr(recs), _ptr(counts),
                                          n_seg, int(seg_cap), self.seed, self.mode, _ptr(self.scratch(n_seg)),
                                          _stream(self.device)))

    def sample(self, batch: int):
        idx, n = self.sample_slots(batch)
        s = torch.empty((batch, 30), dtype=torch.float32, device=self.device)
        a = torch.empty((batch, 3), dtype=torch.float32, device=self.device)
        check(lib().nfsp_gather_sl(_ptr(self.store), _ptr(idx), batch, _ptr(s), _ptr(a), _stream(self.device)))
        return s, a, idx, n

    def clear(self):
        super().clear()
        self.store.zero_()


# ---------------------------------------------------------------------------------------------
# acting nets + fused self-play rollout
# ---------------------------------------------------------------------------------------------
def glorot_nets(seed=1234, device=None) -> torch.Tensor:
    """Four acting nets [player*2 + policy] with Keras' default init (glorot_uniform kernels, zero
    biases; agent.py:101-103,110-112): float32 [4, 2179] = W1[30][64], b1[64], W2[64][3], b2[3]."""
    g = torch.Generator().manual_seed(seed)
    w = torch.zeros((4, _lib.NET_PARAMS), dtype=torch.float32)
    l1, l2 = (6.0 / (30 + 64)) ** 0.5, (6.0 / (64 + 3)) ** 0.5
    for k in range(4):
        w[k, :1920] = (torch.rand(1920, generator=g) * 2 - 1) * l1
        w[k, 1984:2176] = (torch.rand(192, generator=g) * 2 - 1) * l2
    return w.to(_device(device)) if device is not None or torch.cuda.is_available() else w


def split_net(w_row):
    """flat [2179] -> dict W1 (30,64), b1, W2 (64,3), b2 (numpy / tensor views)."""
    return dict(W1=w_row[:1920].reshape(30, 64), b1=w_row[1920:1984], W2=w_row[1984:2176].reshape(64, 3),
                b2=w_row[2176:2179])


class SelfPlay:
    """The fused NFSP rollout: env + acting nets + both players' memories on one GPU.

    One `rollout(n_steps)` call = n_steps Agent.play decisions for every game, records staged by the
    kernel and then moved into the ring (M_RL) / reservoir (M_SL) of the player they belong to."""

    STAT_NAMES = ("a0_fold", "a0_call", "a0_raise", "a1_fold", "a1_call", "a1_raise", "played0", "played1",
                  "reward0_half", "reward1_half", "hands", "transitions", "dropped")

    def __init__(self, n_games, weights=None, seed=1234, game0=0, device=None, eta=0.1, epsilon=0.06,
                 rl_capacity=200000, sl_capacity=2000000, max_steps_per_call=8, reservoir_mode="R",
                 variant="default", direct_rings=False, deterministic=False):
        """direct_rings: the rollout kernel writes the RL records straight into the players' rings (variants "cuda" and
        "sorted"; needs 2 * n_games * max_steps_per_call <= rl_capacity so that one launch cannot lap a ring): no staging
        copy, `flush()` then only moves the SL records into the reservoirs.  "auto" = on when that condition holds.
        deterministic: every block of 32 games stages into a segment of its own, so the order in which the records reach
        the memories -- ring slots, reservoir tickets, the rows a minibatch draws -- is the same in every run (up to
        1 048 576 games per GPU; staged records only, the warp-per-block variants only)."""
        self.variant = variant
        self.env = BatchedNfspEnv(n_games, seed, game0, device, eta)
        self.device, self.n = self.env.device, self.env.n
        self.eta = float(eta)
        # one epsilon per player (each Agent of the reference decays its own, agent.py:253); a scalar sets both
        self.epsilons = [float(e) for e in epsilon] if isinstance(epsilon, (list, tuple)) else [float(epsilon)] * 2
        self.max_steps = int(max_steps_per_call)
        self.rl = [DeviceRing(rl_capacity, seed + 1 + p, self.device) for p in range(2)]
        self.sl = [DeviceReservoir(sl_capacity, seed + 3 + p, self.device, reservoir_mode) for p in range(2)]
        sorted_variant = self.VARIANTS[variant] == 4
        can_direct = self.VARIANTS[variant] in (0, 1, 4, 5, 6) and 2 * self.n * self.max_steps <= int(rl_capacity)
        if direct_rings == "auto":
            direct_rings = can_direct
        if direct_rings and not can_direct:
            raise ValueError("direct_rings needs variant 'cuda' or 'sorted' and 2 * n_games * max_steps_per_call <= rl_capacity")
        self.direct_rings = bool(direct_rings)
        # staging.  Variant "sorted" appends through ONE cursor per memory (a dense array, n_seg = 1); the warp-per-block
        # variants use n_seg segments: the 32 games starting at g append to segment (g/32) % n_seg.  Worst case per
        # player, game and step: 2 RL records (previous + terminal) and 1 SL record.
        blocks = (self.n + 31) // 32
        self.n_seg = 1
        # with direct_rings the only staged records are the SL ones (1/13 of all): 16 cursors per player keep the atomics
        # apart, and a batch of <= 32 segments spares the insert launch its prefix scan and one grid barrier
        # staged rings: up to 256k games 32 segments keep the atomics apart well enough, and a batch of <= 32 segments spares
        # the insert launch its scan and a grid barrier (64k games: step 0.076 -> 0.061 ms); above, 1 024 segments
        max_seg = 16 if self.direct_rings else (32 if blocks <= 8192 else 1024)
        while not sorted_variant and self.n_seg * 2 <= min(blocks, max_seg):
            self.n_seg *= 2
        self.deterministic = bool(deterministic)
        if self.deterministic:
            if self.direct_rings or sorted_variant or blocks > 32768:
                raise ValueError("deterministic needs staged records (direct_rings=False), a warp-per-block variant and "
                                 "at most 1 048 576 games")
            while self.n_seg < blocks:  # one segment per block of 32 games: a single warp appends to it, in step order
                self.n_seg *= 2
        per_seg = ((blocks + self.n_seg - 1) // self.n_seg) * 32   # games that can map to one segment
        self.cap_rl = 2 * per_seg * self.max_steps
        self.cap_sl = per_seg * self.max_steps
        rl_slots = 1 if self.direct_rings else self.n_seg * self.cap_rl
        self.stage_rl = [torch.empty((rl_slots, 4), dtype=torch.int32, device=self.device) for _ in range(2)]
        self.stage_sl = [torch.empty((self.n_seg * self.cap_sl, 4), dtype=torch.int32, device=self.device) for _ in range(2)]
        self.counts = torch.zeros((4, self.n_seg), dtype=torch.int32, device=self.device)
        self.stats = torch.zeros(_lib.STATS_FIELDS, dtype=torch.int64, device=self.device)
        self.set_weights(glorot_nets(seed, self.device) if weights is None else weights)
        self.env.reset()

    @property
    def epsilon(self):
        """Player 0's epsilon (both players' while they are equal); assigning a number sets both."""
        return self.epsilons[0]

    @epsilon.setter
    def epsilon(self, value):
        self.epsilons = [float(value)] * 2

    def set_weights(self, weights):
        """The four acting nets, float32 [4, 2179] (avg0, br0, avg1, br1).  A host tensor (pinned for an asynchronous
        copy) is copied into the device tensor this object already holds: no allocation on the step path."""
        on_host = not (isinstance(weights, torch.Tensor) and weights.is_cuda)
        if on_host and getattr(self, "_own_weights", False) and isinstance(weights, torch.Tensor) \
                and weights.dtype == torch.float32 and weights.is_contiguous() and tuple(weights.shape) == tuple(self.weights.shape):
            # host -> device copy and the rebuild of the weight images in ONE library call (cudaMemcpyAsync on the stream)
            self._host_src = weights  # the copy is asynchronous: keep the source alive until the next hand-over
            check(lib().nfsp_act_set_weights_from_host(self.env._h, C.c_void_p(weights.data_ptr()), _ptr(self.weights),
                                                       _stream(self.device)))
            return
        self.weights = _as(weights, torch.float32, self.device, (4, _lib.NET_PARAMS))
        self._own_weights = on_host  # a device tensor handed in stays the caller's: never written through
        check(lib().nfsp_act_set_weights(self.env._h, _ptr(self.weights), _stream(self.device)))

    def forward(self, obs_masks, net_idx, tensor_cores=False):
        """Batched Model.predict: Q-values (BR nets, odd index) / softmax probabilities (average nets).
        tensor_cores=True runs the first layer as tcgen05.mma tiles (TMEM accumulator)."""
        o = _as(obs_masks, torch.int32, self.device).reshape(-1)
        k = _as(net_idx, torch.int8, self.device).reshape(-1)
        out = torch.empty((o.numel(), 3), dtype=torch.float32, device=self.device)
        fn = lib().nfsp_act_forward_tc if tensor_cores else lib().nfsp_act_forward
        check(fn(self.env._h, _ptr(o), _ptr(k), o.numel(), _ptr(out), _stream(self.device)))
        return out

    VARIANTS = {"default": 0, "cuda": 1, "tcgen05": 2, "tcgen05_ws": 3, "sorted": 4, "pairs": 5, "states": 6}

    def rollout(self, n_steps=1, insert=True, debug=False, forced_vec=None, variant=None, reserve_sms=0, weights_host=None,
                refresh_weights=False):
        """variant: "cuda" (CUDA cores, one warp per 32 games: the default), "sorted" (CUDA cores, warp groups sorted by
        net), "tcgen05" / "tcgen05_ws" (first layer as tensor-core tiles with the accumulator in TMEM) or None =
        self.variant.  reserve_sms: SMs the persistent rollout grid
        leaves to kernels of other streams (the learner beside it, PipelinedTrainer).  weights_host: a pinned float32
        [4, 2179] host tensor with new acting nets -- copied to the device and packed by the same library call that launches
        the rollout (`set_weights(host tensor)` + `rollout()` in one trip through the binding).  refresh_weights: the
        device tensor self.weights has been written in place (a learner update): rebuild the kernels' images from it in the
        same library call (`set_weights(self.weights)` + `rollout()` in one trip)."""
        if n_steps > self.max_steps:
            raise ValueError("n_steps %d exceeds max_steps_per_call %d" % (n_steps, self.max_steps))
        want_debug = debug or forced_vec is not None
        io = self._rollout_io(cache=not want_debug)
        io.variant = self.VARIANTS[variant or self.variant]
        io.epsilon_per_player, io.epsilon_p1 = int(self.epsilons[0] != self.epsilons[1]), self.epsilons[1]
        if self.direct_rings and io.variant not in (0, 1, 4, 5, 6):
            raise ValueError("this SelfPlay was built with direct_rings: only the CUDA-core variants can run on it")
        if (io.variant == 4) != (self.VARIANTS[self.variant] == 4):
            raise ValueError("variant 'sorted' appends through one cursor per memory: build the SelfPlay with variant='sorted'")
        io.reserve_sms = int(reserve_sms)
        dbg = None
        if want_debug:
            tr = torch.empty((3, n_steps, self.n), dtype=torch.int32, device=self.device)
            vec = torch.empty((n_steps, self.n, 3), dtype=torch.float32, device=self.device)
            fv = _as(forced_vec, torch.float32, self.device, (n_steps, self.n, 3))
            io.d_trace, io.d_vec = tr.data_ptr(), vec.data_ptr()
            io.d_forced_vec = None if fv is None else fv.data_ptr()
            dbg = (tr, vec, fv)
        if weights_host is not None and not getattr(self, "_own_weights", False):
            self.set_weights(weights_host)  # first hand-over: the device tensor becomes this object's own
            weights_host = None
        if weights_host is not None:
            if not (weights_host.dtype == torch.float32 and weights_host.is_contiguous() and not weights_host.is_cuda
                    and tuple(weights_host.shape) == tuple(self.weights.shape)):
                raise ValueError("weights_host must be a contiguous float32 [4, 2179] host tensor")
            self._host_src = weights_host  # the copy is asynchronous: keep the source alive until the next hand-over
            check(lib().nfsp_rollout_with_weights(self.env._h, C.c_void_p(weights_host.data_ptr()), _ptr(self.weights), n_steps,
                                                  self.eta, self.epsilons[0], C.byref(io), _stream(self.device)))
        elif refresh_weights:
            check(lib().nfsp_rollout_with_weights(self.env._h, None, _ptr(self.weights), n_steps,
                                                  self.eta, self.epsilons[0], C.byref(io), _stream(self.device)))
        else:
            check(lib().nfsp_rollout(self.env._h, n_steps, self.eta, self.epsilons[0], C.byref(io), _stream(self.device)))
        out = None
        if dbg is not None:
            out = decode_trace(dbg[0])
            out["vec"] = dbg[1]
        if insert:
            self.flush()
        return out

    def _rollout_io(self, cache=True):
        """The rollout's argument block: staging arrays, counters and (direct_rings) the rings.  The production block is
        built once (cache=True); a debug call gets a fresh one."""
        io = getattr(self, "_io", None) if cache else None
        if io is None:
            io = _lib.RolloutIO()
            for p in range(2):
                io.d_rl[p], io.d_sl[p] = self.stage_rl[p].data_ptr(), self.stage_sl[p].data_ptr()
            io.cap_rl, io.cap_sl, io.n_segments = self.cap_rl, self.cap_sl, self.n_seg
            io.d_counts, io.d_stats = self.counts.data_ptr(), self.stats.data_ptr()
            if self.direct_rings:
                for p in range(2):
                    io.d_ring[p], io.d_ring_total[p] = self.rl[p].store.data_ptr(), self.rl[p].total.data_ptr()
                io.ring_cap = self.rl[0].capacity
            if cache:
                self._io = io
        return io

    def staged(self):
        """Host copies of the staged records in batch order (segment by segment): ([rl0, rl1], [sl0, sl1])."""
        c = self.counts.cpu().numpy()

        def take(stage, cnt, cap, dt):
            a = stage.cpu().numpy().reshape(self.n_seg, cap, 4)
            parts = [a[s, : int(cnt[s])] for s in range(self.n_seg)]
            return np.ascontiguousarray(np.concatenate(parts)).view(np.uint8).reshape(-1).view(dt)

        if self.direct_rings:  # the RL records went straight into the rings: nothing of them is staged
            rl = [np.zeros(0, dtype=RL_DT) for _ in range(2)]
        else:
            rl = [take(self.stage_rl[p], c[p], self.cap_rl, RL_DT) for p in range(2)]
        sl = [take(self.stage_sl[p], c[2 + p], self.cap_sl, SL_DT) for p in range(2)]
        return rl, sl

    def flush(self):
        """Move the staged records into the memories (stream-ordered, no host sync): ONE cooperative launch for both
        players' rings and reservoirs (`nfsp_insert_multi`: segment prefixes, ring copies beside the reservoirs' stamp
        pass, their write pass, totals committed and counts cleared).  With direct_rings the rings were written by the
        rollout kernel itself and only the two reservoirs travel."""
        mems_now = self.sl if self.direct_rings else self.sl + self.rl
        if hasattr(self, "_flush_reqs") and any(m._scratch is None or m._scratch.data_ptr() != p_ for m, p_ in zip(mems_now, self._flush_scratch)):
            del self._flush_reqs  # somebody inserted into a memory with a larger geometry: its scratch block moved
        if not hasattr(self, "_flush_reqs"):  # pointers and geometry never change: the request block is built once
            mems = self._insert_mems()
            arr = (_lib.InsertReq * len(mems))()
            for r, m in zip(arr, mems):
                self._insert_req(r, *m)
            self._flush_reqs = (arr, len(mems))
            self._flush_scratch = [m[0]._scratch.data_ptr() for m in mems]
        arr, n = self._flush_reqs
        check(lib().nfsp_insert_multi(arr, n, _stream(self.device)))

    def _insert_mems(self):
        """What flush() moves: (memory, staging array, counts row, segment capacity) -- both reservoirs, then the rings
        unless the rollout writes them directly."""
        mems = [(self.sl[p], self.stage_sl[p], 2 + p, self.cap_sl) for p in range(2)]
        if not self.direct_rings:
            mems += [(self.rl[p], self.stage_rl[p], p, self.cap_rl) for p in range(2)]
        return mems

    def _insert_req(self, r, mem, stage, row, seg_cap):
        """Fills the nfsp_insert_req r of one entry of _insert_mems()."""
        r.d_mem, r.cap, r.d_total = mem.store.data_ptr(), mem.capacity, mem.total.data_ptr()
        r.d_scratch = mem.scratch(self.n_seg).data_ptr()
        r.d_recs, r.d_counts = stage.data_ptr(), self.counts[row].data_ptr()
        r.n_segments, r.seg_cap, r.seed, r.mode = self.n_seg, seg_cap, mem.seed, getattr(mem, "mode", 0)
        r.reservoir = 0 if mem.is_ring else 1

    def sample_minibatches(self, batch=256, to_host=False, with_stats=False):
        """sample_batch(batch) of all four memories (replay_buffer.py:46-59, ReservoirBuffer.py:33-43) into ONE
        float32 slab: per player RL s[b,30] a[b,3] r[b] s2[b,30] t[b], then SL s[b,30] a[b,3].  Returns
        (views, slab); with to_host=True the slab lands in a reused pinned host buffer with a single
        device->host copy (the views then alias the host copy; the caller synchronises the stream).
        with_stats: the rollout counters move to the tail of the slab (self.stats becomes a view of it, the rollout
        kernel accumulates there), so the same copy brings them to the host: the int64 view slab[-26:] of the result."""
        b = int(batch)
        per = b * (65 + 33)
        key = ("slab", b)
        cache = self.__dict__.setdefault("_mb_cache", {})
        if key not in cache:
            tail = 2 * _lib.STATS_FIELDS  # room for the counters (int64 = two float32 words each), 8-byte aligned: per is even
            cache[key] = (torch.empty(2 * per + tail, dtype=torch.float32, device=self.device),
                          torch.empty(2 * per + tail, dtype=torch.float32).pin_memory(),
                          torch.empty((4, b), dtype=torch.int64, device=self.device),
                          torch.zeros(4, dtype=torch.int32, device=self.device))
        slab, host, idx, cnt = cache[key]
        if with_stats and self.stats.data_ptr() != slab[2 * per:].data_ptr():
            home = slab[2 * per:].view(torch.int64)
            home.copy_(self.stats)
            self.stats = home
            self.__dict__.pop("_io", None)  # the rollout's argument block holds the counters' address
        st = _stream(self.device)
        lkey = ("layout", b)
        if lkey not in cache:
            layout = []
            for p in range(2):
                o = p * per
                spec = {}
                for name, cols in (("s", 30), ("a", 3), ("r", 0), ("s2", 30), ("t", 0)):
                    n = b * max(cols, 1)
                    spec[name] = (o, n, (b, cols) if cols else (b,))
                    o += n
                for name, cols in (("sl_s", 30), ("sl_a", 3)):
                    n = b * cols
                    spec[name] = (o, n, (b, cols))
                    o += n
                layout.append(spec)
            # one launch: CTAs of memory m draw its positions and expand its rows into its block of the slab
            reqs = (_lib.SampleReq * 4)()
            for p in range(2):
                for k, mem in ((0, self.rl[p]), (1, self.sl[p])):
                    mem.sample_req(reqs[2 * p + k]).d_out = slab.data_ptr() + 4 * (p * per + k * 65 * b)
            views = {src is host: [{k: src[o:o + n].view(shape) for k, (o, n, shape) in spec.items()} for spec in layout]
                     for src in (slab, host)}
            cache[lkey] = (reqs, views)
        reqs, views = cache[lkey]
        for p in range(2):
            for k, mem in ((0, self.rl[p]), (1, self.sl[p])):
                reqs[2 * p + k].call_idx = mem.next_call()
        check(lib().nfsp_sample_minibatches(reqs, 4, b, _ptr(idx), _ptr(cnt), st))
        if to_host:
            host.copy_(slab, non_blocking=True)
        return views[bool(to_host)], (host if to_host else slab)

    def read_stats(self):
        v = self.stats.cpu().numpy()
        return {k: int(v[i]) for i, k in enumerate(self.STAT_NAMES)}

    def _shape(self):
        return dict(n_games=self.n, game0=self.env.game0, seed=self.env.seed, variant=self.variant,
                    direct_rings=self.direct_rings, deterministic=self.deterministic, max_steps=self.max_steps,
                    n_seg=self.n_seg, rl_capacity=self.rl[0].capacity, sl_capacity=self.sl[0].capacity)

    def state_dict(self) -> dict:
        """Host copy of what the run's later rollouts, inserts and draws depend on: the four memories, game words, step
        counter, acting nets, epsilons, eta and rollout counters, with the shape they need.  Synchronises the device;
        refuses (ValueError) while records are staged but not flushed (rollout(insert=False) without flush())."""
        if int(self.counts.sum().item()):
            raise ValueError("SelfPlay: records are staged but not flushed; flush() before state_dict()")
        torch.cuda.synchronize(self.device)
        return dict(shape=self._shape(), rl=[m.state_dict() for m in self.rl], sl=[m.state_dict() for m in self.sl],
                    words=self.env.state_words().cpu(), step=self.env.step_counter, weights=self.weights.cpu(),
                    epsilons=list(self.epsilons), eta=self.eta, stats=self.stats.cpu())

    def check_state_dict(self, d):
        """Raises ValueError, naming the field, if load_state_dict(d) would refuse d."""
        check_fields(d, "SelfPlay")
        check_fields(d.get("shape"), "SelfPlay", **self._shape())
        for key, mems in (("rl", self.rl), ("sl", self.sl)):
            if not (isinstance(d.get(key), list) and len(d[key]) == 2):
                raise ValueError("SelfPlay: %s must be a list of the two players' memories" % key)
            for p in range(2):
                mems[p].check_state_dict(d[key][p], "SelfPlay %s[%d]" % (key, p))
        check_tensor(d.get("words"), "words", "SelfPlay", (self.n,), torch.int64)
        check_tensor(d.get("weights"), "weights", "SelfPlay", tuple(self.weights.shape), torch.float32)
        check_tensor(d.get("stats"), "stats", "SelfPlay", (_lib.STATS_FIELDS,), torch.int64)
        check_numbers(d, "SelfPlay", below=dict(step=2 ** 64), step=int, epsilons=(float, 2), eta=float)

    def load_state_dict(self, d):
        """Validates d, then restores it into this object's own tensors (stats too, which may be a view into the
        sampling slab); the weight images are rebuilt from the restored nets and nothing stays staged."""
        self.check_state_dict(d)
        for key, mems in (("rl", self.rl), ("sl", self.sl)):
            for p in range(2):
                mems[p].load_state_dict(d[key][p])
        self.env.load_state_words(d["words"])
        self.env.step_counter = d["step"]
        self.weights.copy_(d["weights"])
        check(lib().nfsp_act_set_weights(self.env._h, _ptr(self.weights), _stream(self.device)))
        self.epsilons = [float(e) for e in d["epsilons"]]
        self.eta = self.env.eta = float(d["eta"])
        self.stats.copy_(d["stats"])
        self.counts.zero_()
        torch.cuda.synchronize(self.device)
