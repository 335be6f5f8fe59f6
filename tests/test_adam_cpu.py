"""Adam without a GPU: the float64 Adam fit (tests/adam_reference.py) against torch.optim.Adam on autograd gradients, the
C ABI of the Adam entries, the learner's Adam checkpoint fields and main.py's --optimizer."""
import ctypes
import os
import sys
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import adam_reference as ar  # noqa: E402
from oracle import learner_oracle as lo  # noqa: E402


def _losses(W, T, c, k, rows, gamma, terminal_bootstraps, others_to_target):
    """The loss of net k on the sampled rows (the definition test_learner_reference_cpu holds the SGD reference to)."""
    import torch.nn.functional as F

    def net(w, m):
        W1, b1, W2, b2 = w[:1920].reshape(30, 64), w[1920:1984], w[1984:2176].reshape(64, 3), w[2176:2179]
        x = torch.from_numpy(((np.asarray(m, np.uint32)[:, None] >> np.arange(30)) & 1).astype(np.float64))
        return F.relu(x @ W1 + b1) @ W2 + b2

    p = k >> 1
    if k & 1:
        b = c["rl"][p][rows]
        q = F.relu(net(W, b["s"]))
        with torch.no_grad():
            qs = F.relu(net(T[p], b["s"]))
            live = 1.0 if terminal_bootstraps else 1.0 - torch.from_numpy(b["t"].astype(np.float64))
            y = torch.from_numpy(b["r"].astype(np.float64)) + gamma * live * F.relu(net(T[p], b["s2"])).max(1).values
            tgt = qs.clone() if others_to_target else q.detach().clone()
            tgt[torch.arange(len(rows)), torch.from_numpy(b["a"].astype(np.int64))] = y
        err = tgt - q
        return torch.where(err.abs() > 1, err.abs() - 0.5, 0.5 * err * err).mean(dim=1).mean()
    b = c["sl"][p][rows]
    y = torch.from_numpy(b["a"].astype(np.float64))
    return (-(y * F.log_softmax(net(W, b["s"]), dim=1)).sum(1)).mean()


class _TorchAdam:
    """The four nets, each with its own torch.optim.Adam in float64.  torch adds epsilon after the bias correction of
    sqrt(v); Keras before it.  Setting the group's eps to 1e-7 / sqrt(1 - beta2^t) before step t gives Keras' step."""

    def __init__(self, c):
        self.W = [torch.tensor(c["w"][k], dtype=torch.float64, requires_grad=True) for k in range(4)]
        self.T = [torch.from_numpy(c["w_target"][p].copy()) for p in range(2)]
        self.opt = [torch.optim.Adam([self.W[k]], lr=float(c["lr"][k]), betas=(0.9, 0.999), eps=1e-7, foreach=False)
                    for k in range(4)]
        self.t = [0] * 4

    def fit(self, c, minibatch, fit_batch, epochs, gamma, mask, terminal_bootstraps, others_to_target):
        for _ in range(epochs):
            for rows in torch.arange(minibatch).split(fit_batch):
                for k in range(4):
                    if not (mask >> k) & 1:
                        continue
                    self.opt[k].zero_grad()
                    _losses(self.W[k], self.T, c, k, rows.numpy(), gamma, terminal_bootstraps, others_to_target).backward()
                    self.t[k] += 1
                    self.opt[k].param_groups[0]["eps"] = 1e-7 / np.sqrt(1 - 0.999 ** self.t[k])
                    self.opt[k].step()

    def state(self):
        W = torch.stack([w.detach() for w in self.W]).numpy()
        m = np.stack([self.opt[k].state[self.W[k]]["exp_avg"].numpy() if self.W[k] in self.opt[k].state
                      else np.zeros(lo.NET_PARAMS) for k in range(4)])
        v = np.stack([self.opt[k].state[self.W[k]]["exp_avg_sq"].numpy() if self.W[k] in self.opt[k].state
                      else np.zeros(lo.NET_PARAMS) for k in range(4)])
        return W, m, v, list(self.t)


def _close(ref, got, m_ref, m_got, v_ref, v_got):
    assert np.abs(ref - got).max() <= 1e-9
    assert np.allclose(m_got, m_ref, rtol=1e-9, atol=1e-15)
    assert np.allclose(v_got, v_ref, rtol=1e-9, atol=1e-18)


@pytest.mark.parametrize("terminal_bootstraps", [False, True])
@pytest.mark.parametrize("others_to_target", [False, True])
@pytest.mark.parametrize("minibatch,fit_batch,epochs,mask", [
    (128, 32, 2, 0xF),       # the reference's sizes
    (100, 24, 3, 0xF),       # ragged last slice of 4 rows, three epochs
    (33, 8, 1, 0b0101),      # a last slice of one row; only the average-policy nets train
    (70, 64, 2, 0b1010),     # only the best-response nets train
])
def test_adam_reference_matches_torch_adam(minibatch, fit_batch, epochs, mask, terminal_bootstraps, others_to_target):
    c = lo.fit_case(3, minibatch)
    w, m, v, t, stats, _ = ar.fit(c["w"], c["w_target"], c["rl"], c["sl"], minibatch, fit_batch, epochs, c["lr"], 0.95,
                               net_mask=mask, terminal_bootstraps=terminal_bootstraps, others_to_target=others_to_target)
    ta = _TorchAdam(c)
    ta.fit(c, minibatch, fit_batch, epochs, 0.95, mask, terminal_bootstraps, others_to_target)
    w_ref, m_ref, v_ref, t_ref = ta.state()
    _close(w_ref, w, m_ref, m, v_ref, v)
    steps = epochs * -(-minibatch // fit_batch)
    assert t == t_ref == [steps if (mask >> k) & 1 else 0 for k in range(4)]
    for k in range(4):
        if (mask >> k) & 1:
            assert np.abs(w[k] - c["w"][k]).max() > 1e-3
        else:   # a net that does not train keeps its weights and its optimizer state
            assert np.array_equal(w[k], c["w"][k]) and not m[k].any() and not v[k].any()
    # the statistics are those of the SGD reference's first step: the optimizer does not change them
    _, stats_sgd, _, _ = lo.fit(c["w"], c["w_target"], c["rl"], c["sl"], minibatch, fit_batch, epochs, c["lr"], 0.95, mask,
                                terminal_bootstraps, others_to_target)
    assert np.array_equal(np.isnan(stats), np.isnan(stats_sgd))
    ok = ~np.isnan(stats)
    assert np.array_equal(stats[ok], stats_sgd[ok])


def test_chained_adam_fits_carry_the_state():
    """Three fits chained through (w, m, v, t), with the masks changing between them, equal one torch optimizer per net
    that lives through all three: t counts each net's own steps, and Adam's step depends on it."""
    c = lo.fit_case(5, 128)
    ta = _TorchAdam(c)
    w, m, v, t = c["w"], None, None, (0, 0, 0, 0)
    for mask in (0b1010, 0xF, 0b0110):
        w, m, v, t, _, _ = ar.fit(w, c["w_target"], c["rl"], c["sl"], 128, 32, 2, c["lr"], 0.95, m=m, v=v, t=t, net_mask=mask)
        ta.fit(c, 128, 32, 2, 0.95, mask, False, False)
        w_ref, m_ref, v_ref, t_ref = ta.state()
        _close(w_ref, w, m_ref, m, v_ref, v)
        assert t == t_ref
    assert t == [8, 24, 16, 16]


def test_adam_state_mirror_matches_the_header(tmp_path):
    """nfsp_adam_state has the size and offsets of its ctypes mirror (a C program compiled against the header)."""
    import subprocess

    from nfsp_b200 import _lib

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "nfsp_b200.h"', "int main(void) {",
             'printf("size %zu\\n", sizeof(nfsp_adam_state));']
    for field, _ in _lib.AdamState._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(nfsp_adam_state, %s));' % (field, field))
    lines += ["return 0;", "}"]
    (tmp_path / "abi.c").write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(root, "include"), str(tmp_path / "abi.c"), "-o",
                    str(tmp_path / "abi")], check=True)
    got = dict(ln.split() for ln in subprocess.run([str(tmp_path / "abi")], capture_output=True, text=True,
                                                   check=True).stdout.splitlines())
    assert int(got["size"]) == ctypes.sizeof(_lib.AdamState) == 48
    for field, _ in _lib.AdamState._fields_:
        assert int(got[field]) == getattr(_lib.AdamState, field).offset


ADAM_SYMBOLS = ["nfsp_learner_fit_adam", "nfsp_learner_fit_runs_adam", "nfsp_learner_fit_peers_adam", "nfsp_adam_apply"]


def test_adam_symbols_are_exported_and_nothing_else_is_new():
    """The four Adam entries are declared, listed and exported; the rest of the ABI is what it was."""
    import re

    from nfsp_b200 import _lib

    assert all(s in _lib.SYMBOLS for s in ADAM_SYMBOLS)
    L = _lib.lib()
    for s in ADAM_SYMBOLS:
        assert getattr(L, s) is not None
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "nfsp_b200.h")).read()
    assert sorted(set(re.findall(r"\bint\s+(nfsp_[a-z0-9_]+)\s*\(", hdr)) & set(ADAM_SYMBOLS)) == sorted(ADAM_SYMBOLS)
    assert len(_lib.SYMBOLS) == len(set(_lib.SYMBOLS)) == 56 + len(ADAM_SYMBOLS)   # 56 entries before Adam


def test_adam_entries_refuse_a_bad_state():
    """Argument checks run before any device work: no GPU is needed to see them."""
    from nfsp_b200 import _lib

    L = _lib.lib()
    lr = (ctypes.c_float * 4)(0.1, 0.1, 0.1, 0.1)
    buf = ctypes.create_string_buffer(64)
    ok = _lib.AdamState(ctypes.addressof(buf), ctypes.addressof(buf) + 16, (ctypes.c_int64 * 4)(0, 0, 0, 0))
    for bad, why in ((None, "null Adam state"),
                     (_lib.AdamState(None, 1, (ctypes.c_int64 * 4)()), "null Adam state"),
                     (_lib.AdamState(8, 8, (ctypes.c_int64 * 4)()), "separate"),
                     (_lib.AdamState(8, 16, (ctypes.c_int64 * 4)(0, -1, 0, 0)), "t0\\[1\\]"),
                     (_lib.AdamState(8, 16, (ctypes.c_int64 * 4)(0, 0, 0, 2 ** 62 + 1)), "t0\\[3\\]")):
        rc = L.nfsp_adam_apply(8, 8, ctypes.byref(lr), 1.0, 15, None if bad is None else ctypes.byref(bad), None)
        assert rc != 0
        assert why.replace("\\", "") in L.nfsp_last_error().decode()
    assert L.nfsp_adam_apply(8, 8, ctypes.byref(lr), 1.0, 16, ctypes.byref(ok), None) != 0   # bad net_mask
    assert "net_mask" in L.nfsp_last_error().decode()


# ---- the learner's state dict, on a CPU stand-in for the self-play ----
def _learner(optimizer, monkeypatch):
    from nfsp_b200.learner import Learner

    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    sp = types.SimpleNamespace(device=torch.device("cpu"), weights=torch.zeros((4, lo.NET_PARAMS)))
    return Learner(sp, optimizer=optimizer)


def test_sgd_state_dict_is_unchanged(monkeypatch):
    d = _learner("sgd", monkeypatch).state_dict()
    assert sorted(d) == sorted(["shape", "target", "loss", "gamma", "lr_br0", "lr_ar", "target_update_rate", "iteration",
                                "target_update_count", "temp", "lr_br", "exploitability", "updates"])
    assert sorted(d["shape"]) == sorted(["minibatch", "fit_batch", "epochs", "terminal_bootstraps", "others_to_target",
                                         "fused"])


def test_adam_state_dict_round_trip_and_refusals(monkeypatch):
    ln = _learner("adam", monkeypatch)
    ln.adam_m.normal_()
    ln.adam_v.uniform_()
    ln.adam_t = [16, 8, 16, 0]
    d = ln.state_dict()
    assert d["shape"]["optimizer"] == "adam" and d["adam_t"] == [16, 8, 16, 0]
    other = _learner("adam", monkeypatch)
    other.load_state_dict(d)
    assert torch.equal(other.adam_m, ln.adam_m) and torch.equal(other.adam_v, ln.adam_v) and other.adam_t == ln.adam_t
    for field, value in (("adam_m", torch.zeros((4, 2178))), ("adam_v", torch.zeros((4, lo.NET_PARAMS), dtype=torch.float64)),
                         ("adam_m", None), ("adam_t", [1, 2, 3]), ("adam_t", [1, 2, 3, -1]), ("adam_t", [0, 0, 0, 1.0]),
                         ("adam_t", [0, 0, 0, 2 ** 62 + 1])):
        bad = dict(d, **{field: value})
        with pytest.raises(ValueError, match=field):
            other.check_state_dict(bad)
    with pytest.raises(ValueError, match="optimizer"):   # an SGD state into an Adam learner
        other.check_state_dict(_learner("sgd", monkeypatch).state_dict())
    with pytest.raises(ValueError, match="optimizer"):   # an Adam state into an SGD learner
        _learner("sgd", monkeypatch).check_state_dict(d)


def test_learner_refuses_an_unknown_optimizer(monkeypatch):
    with pytest.raises(ValueError, match="optimizer"):
        _learner("rmsprop", monkeypatch)


def test_runs_of_one_batch_share_the_optimizer():
    from nfsp_b200.runs import _learner_shape

    a = types.SimpleNamespace(minibatch=128, fit_batch=32, epochs=2, terminal_bootstraps=False, others_to_target=False,
                              fused=True, optimizer="sgd")
    assert _learner_shape(a) != _learner_shape(types.SimpleNamespace(**dict(vars(a), optimizer="adam")))


# ---- main.py --optimizer ----
def _main_learners(monkeypatch, argv):
    """The optimizer of every Learner main.main(argv) builds, with the device, the self-play and the training loops
    replaced by stand-ins."""
    from nfsp_b200 import main

    made = []

    class FakeLearner:
        def __init__(self, sp, **kw):
            made.append(kw["optimizer"])

    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: None)
    monkeypatch.setattr(torch.cuda, "device_count", lambda: 1)
    monkeypatch.setattr(main, "SelfPlay", lambda *a, **k: types.SimpleNamespace())
    monkeypatch.setattr(main, "Learner", FakeLearner)
    monkeypatch.setattr(main, "RunBatch", lambda sps, lns: None)
    for loop in ("train", "train_runs", "train_sweep"):
        monkeypatch.setattr(main, loop, lambda *a, **k: [])
    for k, v in (("WORLD_SIZE", "1"), ("RANK", "0"), ("LOCAL_RANK", "0")):
        monkeypatch.setenv(k, v)
    main.main(argv)
    return made


@pytest.mark.parametrize("argv,expect", [
    ([], ["sgd"]),
    (["--optimizer", "sgd"], ["sgd"]),
    (["--optimizer", "adam"], ["adam"]),
    (["--optimizer", "adam", "--pipelined"], ["adam"]),
    (["--optimizer", "adam", "--runs", "3"], ["adam"] * 3),
    (["--optimizer", "adam", "--sweep", "LearningRateBR=0.001,0.0001", "--runs", "2"], ["adam"] * 4),
])
def test_optimizer_flag_reaches_every_learner(monkeypatch, argv, expect):
    assert _main_learners(monkeypatch, argv) == expect


def test_a_bad_optimizer_is_refused(capsys, monkeypatch):
    from nfsp_b200 import main

    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: (_ for _ in ()).throw(AssertionError("device touched")))
    with pytest.raises(SystemExit) as e:
        main.main(["--optimizer", "rmsprop"])
    assert e.value.code == 2
    assert "--optimizer" in capsys.readouterr().err
