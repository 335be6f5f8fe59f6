"""ctypes binding of oracle/liboracle.so -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import
this.  The product package never does (tests/test_boundary.py enforces it).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liboracle.so")


def build(force: bool = False) -> str:
    src = [os.path.join(HERE, f) for f in ("leduc_oracle.c", "leduc_oracle.h")]
    if force or not os.path.exists(LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in src):
        base = ["gcc", "-O2", "-fPIC", "-shared", "-Wall", "-Wno-comment", "-o", LIB_PATH, src[0], "-lm"]
        r = subprocess.run(base[:2] + ["-fopenmp"] + base[2:], cwd=HERE, capture_output=True, text=True)
        if r.returncode != 0:  # no libgomp on this box: single-threaded oracle
            subprocess.run(base, cwd=HERE, check=True)
    return LIB_PATH


class LegacyEnv(C.Structure):
    _fields_ = [("card", C.c_int * 2), ("pub", C.c_int), ("st_pot", C.c_int * 2), ("st_reward", C.c_int * 2),
                ("st_terminal", C.c_int * 2), ("st_action", C.c_int * 2), ("pot", C.c_int * 2),
                ("left", C.c_int * 2), ("penalty", C.c_int), ("choices", C.c_int)]


class NfspEnv(C.Structure):
    _fields_ = [("history", C.c_double * 24), ("specific_cards", C.c_double * 12),
                ("overall_raises", C.c_double * 2), ("raises", C.c_double * 2), ("reward", C.c_double * 2),
                ("last_action", C.c_double * 6), ("s", C.c_double * 60),
                ("round", C.c_int), ("round_raises", C.c_int), ("terminated", C.c_int), ("dealer", C.c_int),
                ("actions_done", C.c_int * 8), ("n_done", C.c_int), ("public_card_index", C.c_int),
                ("deck", C.c_int * 3), ("deck_pos", C.c_int), ("anomalies", C.c_int)]


class Net(C.Structure):
    _fields_ = [("W1", C.c_void_p), ("b1", C.c_void_p), ("W2", C.c_void_p), ("b2", C.c_void_p)]


class RolloutOut(C.Structure):
    _fields_ = [("rl", C.c_void_p * 2), ("n_rl", C.c_int64 * 2), ("cap_rl", C.c_int64 * 2),
                ("sl", C.c_void_p * 2), ("n_sl", C.c_int64 * 2), ("cap_sl", C.c_int64 * 2),
                ("actions", C.c_int64 * 6), ("played", C.c_int64 * 2), ("reward_half", C.c_int64 * 2),
                ("hands", C.c_int64)]


class Ring(C.Structure):
    _fields_ = [("data", C.c_void_p), ("cap", C.c_int64), ("count", C.c_int64), ("total", C.c_int64),
                ("rec_bytes", C.c_int)]


class Reservoir(C.Structure):
    _fields_ = [("data", C.c_void_p), ("cap", C.c_int64), ("count", C.c_int64), ("total", C.c_int64),
                ("rec_bytes", C.c_int), ("seed", C.c_uint64), ("mode", C.c_int)]


TRACE_DT = np.dtype([("obs", "<u4"), ("reward", "<f4"), ("misc", "<u4")])
RL_DT = np.dtype([("s", "<u4"), ("s2", "<u4"), ("r", "<f4"), ("a", "u1"), ("t", "u1"), ("player", "u1"),
                  ("flags", "u1")])
SL_DT = np.dtype([("s", "<u4"), ("a", "<f4", (3,))])
LEGACY_DT = np.dtype([("card", "i1"), ("pub", "i1"), ("pot", "i1"), ("terminal", "i1"), ("reward", "<i4"),
                      ("misc", "<u4")])

_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB_PATH)
        L.orc_nfsp_batch_create.restype = C.c_void_p
        L.orc_nfsp_batch_create.argtypes = [C.c_int, C.c_uint64, C.c_uint64]
        L.orc_nfsp_batch_destroy.argtypes = [C.c_void_p]
        L.orc_nfsp_batch_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32]
        L.orc_nfsp_batch_inject.argtypes = [C.c_void_p] + [C.c_int] * 7
        L.orc_nfsp_batch_rollout_env.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p,
                                                 C.c_uint32, C.c_void_p, C.c_int]
        L.orc_nfsp_batch_rollout_act.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint32,
                                                 C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_int]
        L.orc_nfsp_batch_rollout_act2.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint32, C.c_uint32,
                                                  C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.orc_nfsp_batch_env.restype = C.POINTER(NfspEnv)
        L.orc_nfsp_batch_env.argtypes = [C.c_void_p, C.c_int]
        L.orc_nfsp_batch_flags.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int * 4)]
        L.orc_legacy_batch_create.restype = C.c_void_p
        L.orc_legacy_batch_create.argtypes = [C.c_int, C.c_uint64, C.c_uint64]
        L.orc_legacy_batch_destroy.argtypes = [C.c_void_p]
        L.orc_legacy_batch_reset.argtypes = [C.c_void_p, C.c_uint64]
        L.orc_legacy_batch_rollout.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.orc_legacy_batch_env.restype = C.POINTER(LegacyEnv)
        L.orc_legacy_batch_env.argtypes = [C.c_void_p, C.c_int]
        L.orc_reservoir_slot.restype = C.c_int64
        L.orc_reservoir_slot.argtypes = [C.c_uint64, C.c_int64, C.c_int64, C.c_int]
        L.orc_sample_indices.argtypes = [C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_void_p]
        L.orc_ring_insert.argtypes = [C.POINTER(Ring), C.c_void_p, C.c_int64]
        L.orc_reservoir_insert.argtypes = [C.POINTER(Reservoir), C.c_void_p, C.c_int64]
        L.orc_nfsp_step.argtypes = [C.POINTER(NfspEnv), C.POINTER(C.c_double * 3), C.c_int]
        L.orc_nfsp_reset.argtypes = [C.POINTER(NfspEnv), C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_nfsp_get_state.restype = C.c_int
        L.orc_nfsp_get_state.argtypes = [C.POINTER(NfspEnv), C.c_int, C.c_void_p, C.c_void_p,
                                         C.POINTER(C.c_double), C.c_void_p]
        L.orc_nfsp_state_vector.argtypes = [C.POINTER(NfspEnv), C.c_int, C.c_void_p]
        L.orc_mask30.restype = C.c_uint32
        L.orc_mask30.argtypes = [C.c_void_p]
        L.orc_legacy_step.argtypes = [C.POINTER(LegacyEnv), C.POINTER(C.c_double * 3), C.c_int]
        L.orc_legacy_get_new_state.argtypes = [C.POINTER(LegacyEnv), C.c_int, C.POINTER(C.c_int * 5)]
        L.orc_mlp_br.argtypes = [C.POINTER(Net), C.c_void_p, C.c_void_p]
        L.orc_mlp_avg.argtypes = [C.POINTER(Net), C.c_void_p, C.c_void_p]
        L.orc_philox4x32_10.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def philox(ctr, key):
    c = np.asarray(ctr, np.uint32)
    k = np.asarray(key, np.uint32)
    o = np.zeros(4, np.uint32)
    lib().orc_philox4x32_10(c.ctypes.data, k.ctypes.data, o.ctypes.data)
    return o


def u32_frac(x: float) -> int:
    """eta / epsilon as the u32 threshold both the oracle and the kernels use: floor(x * 2^32)."""
    return min(int(x * 4294967296.0), 0xFFFFFFFF)


# ---------------------------------------------------------------------------------------
class NfspSingle:
    """One newenv.Env restated; object API for golden replay."""

    def __init__(self):
        self.e = NfspEnv()

    def reset(self, dealer, c0, c1, pub):
        lib().orc_nfsp_reset(C.byref(self.e), dealer, c0, c1, pub)

    def step(self, vec, p):
        v = (C.c_double * 3)(*[float(x) for x in vec])
        lib().orc_nfsp_step(C.byref(self.e), C.byref(v), p)

    def obs(self, p) -> int:
        buf = np.zeros(30)
        lib().orc_nfsp_state_vector(C.byref(self.e), p, buf.ctypes.data)
        return int(lib().orc_mask30(buf.ctypes.data))

    def snap(self, p) -> int:
        buf = np.array(self.e.s[p * 30:(p + 1) * 30])
        return int(lib().orc_mask30(buf.ctypes.data))

    def get_state(self, p):
        s, a, s2 = np.zeros(30), np.zeros(3), np.zeros(30)
        r = C.c_double()
        t = lib().orc_nfsp_get_state(C.byref(self.e), p, s.ctypes.data, a.ctypes.data, C.byref(r), s2.ctypes.data)
        return s, a, r.value, s2, bool(t)


class LegacySingle:
    def __init__(self):
        self.e = LegacyEnv()
        lib().orc_legacy_init(C.byref(self.e))

    def reset(self, c0, c1):
        lib().orc_legacy_reset(C.byref(self.e), c0, c1)

    def step(self, a, p):
        v = (C.c_double * 3)(0, 0, 0)
        v[a] = 1.0
        lib().orc_legacy_step(C.byref(self.e), C.byref(v), p)

    def get_new_state(self, p):
        o = (C.c_int * 5)()
        lib().orc_legacy_get_new_state(C.byref(self.e), p, C.byref(o))
        return tuple(o)


class Nets:
    """Four acting nets [player*2 + policy] as fp32 arrays (Keras Dense layout)."""

    def __init__(self, weights):
        # weights: list of 4 dicts {W1 (30,64), b1 (64,), W2 (64,3), b2 (3,)}
        self.keep = []
        arr = (Net * 4)()
        for i, w in enumerate(weights):
            t = [np.ascontiguousarray(w[k], np.float32) for k in ("W1", "b1", "W2", "b2")]
            assert t[0].shape == (30, 64) and t[1].shape == (64,) and t[2].shape == (64, 3) and t[3].shape == (3,)
            self.keep.append(t)
            arr[i].W1, arr[i].b1, arr[i].W2, arr[i].b2 = [x.ctypes.data for x in t]
        self.arr = arr

    def forward(self, net_idx, x, head):
        x = np.ascontiguousarray(x, np.float32).reshape(-1, 30)
        out = np.zeros((x.shape[0], 3), np.float32)
        f = lib().orc_mlp_br if head == "br" else lib().orc_mlp_avg
        for i in range(x.shape[0]):
            f(C.byref(self.arr[net_idx]), x[i].ctypes.data, out[i].ctypes.data)
        return out


class NfspBatch:
    def __init__(self, n, seed, game0=0):
        self.n = n
        self.h = lib().orc_nfsp_batch_create(n, seed, game0)

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_nfsp_batch_destroy(self.h)
            self.h = None

    def reset(self, step, eta_u32, dealer=None):
        d = None if dealer is None else np.ascontiguousarray(dealer, np.int32)
        lib().orc_nfsp_batch_reset(self.h, None if d is None else d.ctypes.data, step, eta_u32)

    def inject(self, g, dealer, cards, policy):
        lib().orc_nfsp_batch_inject(self.h, g, int(dealer), int(cards[0]), int(cards[1]), int(cards[2]),
                                    int(policy[0]), int(policy[1]))

    def rollout_env(self, step0, n_steps, eta_u32, actions=None, players=None, threads=0):
        tr = np.zeros((n_steps, self.n), TRACE_DT)
        a = None if actions is None else np.ascontiguousarray(actions, np.int8)
        p = None if players is None else np.ascontiguousarray(players, np.int8)
        lib().orc_nfsp_batch_rollout_env(self.h, step0, n_steps, None if a is None else a.ctypes.data,
                                         None if p is None else p.ctypes.data, eta_u32, tr.ctypes.data, threads)
        return tr

    def rollout_act(self, step0, n_steps, nets: Nets, eta_u32, eps_u32, forced_vec=None, rec_cap=None, eps1_u32=None):
        n = self.n
        cap = rec_cap or (3 * n * n_steps + 8)
        tr = np.zeros((n_steps, n), TRACE_DT)
        vec = np.zeros((n_steps, n, 3), np.float32)
        rl = [np.zeros(cap, RL_DT) for _ in range(2)]
        sl = [np.zeros(cap, SL_DT) for _ in range(2)]
        out = RolloutOut()
        for p in range(2):
            out.rl[p], out.cap_rl[p] = rl[p].ctypes.data, cap
            out.sl[p], out.cap_sl[p] = sl[p].ctypes.data, cap
        fv = None if forced_vec is None else np.ascontiguousarray(forced_vec, np.float32)
        lib().orc_nfsp_batch_rollout_act2(self.h, step0, n_steps, C.byref(nets.arr), eta_u32, eps_u32,
                                          eps_u32 if eps1_u32 is None else eps1_u32,
                                          None if fv is None else fv.ctypes.data, vec.ctypes.data, tr.ctypes.data,
                                          C.byref(out), 0)
        return dict(trace=tr, vec=vec, rl=[rl[p][:out.n_rl[p]] for p in range(2)],
                    sl=[sl[p][:out.n_sl[p]] for p in range(2)],
                    actions=np.array(list(out.actions)).reshape(2, 3), played=np.array(list(out.played)),
                    reward_half=np.array(list(out.reward_half)), hands=int(out.hands))

    def env(self, g) -> NfspEnv:
        return lib().orc_nfsp_batch_env(self.h, g).contents

    def flags(self, g):
        o = (C.c_int * 4)()
        lib().orc_nfsp_batch_flags(self.h, g, C.byref(o))
        return tuple(o)


class LegacyBatch:
    def __init__(self, n, seed, game0=0):
        self.n = n
        self.h = lib().orc_legacy_batch_create(n, seed, game0)

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_legacy_batch_destroy(self.h)
            self.h = None

    def reset(self, step):
        lib().orc_legacy_batch_reset(self.h, step)

    def rollout(self, step0, n_iters, actions=None, threads=0):
        out = np.zeros((n_iters, self.n, 2), LEGACY_DT)
        a = None if actions is None else np.ascontiguousarray(actions, np.int8)
        lib().orc_legacy_batch_rollout(self.h, step0, n_iters, None if a is None else a.ctypes.data,
                                       out.ctypes.data, threads)
        return out

    def env(self, g) -> LegacyEnv:
        return lib().orc_legacy_batch_env(self.h, g).contents


def ring_insert_all(recs: np.ndarray, cap: int, total0: int = 0, data=None):
    """Sequential FIFO ring fed with `recs` (structured array); returns (data[cap], count, total).  A ring mid-life
    starts at total0 records ever inserted with storage `data` (updated in place)."""
    if data is None:
        data = np.zeros(cap, recs.dtype)
    r = Ring(data.ctypes.data, cap, min(total0, cap), total0, recs.dtype.itemsize)
    recs = np.ascontiguousarray(recs)
    lib().orc_ring_insert(C.byref(r), recs.ctypes.data, len(recs))
    return data, r.count, r.total


def reservoir_insert_all(recs: np.ndarray, cap: int, seed: int, mode: int = 0, total0: int = 0, data=None):
    if data is None:
        data = np.zeros(cap, recs.dtype)
    r = Reservoir(data.ctypes.data, cap, min(total0, cap), total0, recs.dtype.itemsize, seed, mode)
    recs = np.ascontiguousarray(recs)
    lib().orc_reservoir_insert(C.byref(r), recs.ctypes.data, len(recs))
    return data, r.count, r.total


def reservoir_slot(seed, ticket, cap, mode=0):
    """Slot the record with this ticket replaces in a reservoir of `cap` slots, -1 if it is dropped."""
    return int(lib().orc_reservoir_slot(seed, ticket, cap, mode))


def sample_indices(seed, call_idx, count, batch):
    out = np.zeros(min(batch, count), np.int64)
    lib().orc_sample_indices(seed, call_idx, count, batch, out.ctypes.data)
    return out


def hw_threads() -> int:
    return int(lib().orc_hw_threads())
