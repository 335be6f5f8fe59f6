"""-m gpu: checkpoints (nfsp_b200.checkpoint, the state_dict() / load_state_dict() of SelfPlay, Learner,
PipelinedTrainer and RunBatch).

A run saved to a file and loaded into freshly built objects must go on exactly as the run that never stopped: game words,
step counter, rollout counters, all four memories (contents, totals, draw counters), acting and target nets, epsilons and
the learner's schedules, bit for bit, and the same dicts from update()."""
import os
from collections import Counter

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nb():
    import nfsp_b200

    assert torch.cuda.is_available()
    return nfsp_b200


def _assert_same(a, b, la=None, lb=None, tag=""):
    """tests/test_gpu_runs.py's _assert_same_run, with every learner scalar a checkpoint carries."""
    torch.cuda.synchronize()
    assert torch.equal(a.env.state_words(), b.env.state_words()), tag
    assert a.env.step_counter == b.env.step_counter, tag
    assert torch.equal(a.stats, b.stats), tag
    for p in range(2):
        for ma, mb in ((a.rl[p], b.rl[p]), (a.sl[p], b.sl[p])):
            assert torch.equal(ma.total, mb.total), (tag, p)
            assert torch.equal(ma.store, mb.store), (tag, p)
            assert ma.sample_calls == mb.sample_calls, (tag, p)
    assert torch.equal(a.weights, b.weights), tag
    assert a.epsilons == b.epsilons and a.eta == b.eta, tag
    if la is not None:
        assert torch.equal(la.target, lb.target), tag
        for k in ("iteration", "target_update_count", "temp", "lr_br", "exploitability", "updates", "gamma", "lr_br0",
                  "lr_ar", "target_update_rate"):
            assert getattr(la, k) == getattr(lb, k), (tag, k)
        assert getattr(la, "_loss", None) == getattr(lb, "_loss", None), tag


def _same_state(x, y, path="state"):
    """Nested state dicts equal: tensors bit for bit, everything else by ==."""
    assert type(x) is type(y), path
    if isinstance(x, dict):
        assert x.keys() == y.keys(), path
        for k in x:
            _same_state(x[k], y[k], "%s.%s" % (path, k))
    elif isinstance(x, (list, tuple)):
        assert len(x) == len(y), path
        for k, (u, v) in enumerate(zip(x, y)):
            _same_state(u, v, "%s[%d]" % (path, k))
    elif isinstance(x, torch.Tensor):
        assert x.dtype == y.dtype and x.shape == y.shape and torch.equal(x, y), path
    else:
        assert x == y, path


def _make(nb, n=4096, seed=1234, eta=0.3, eps=0.2, lr_br=0.05, lr_ar=0.1, learner=None, **kw):
    from nfsp_b200.learner import Learner

    sp = nb.SelfPlay(n, seed=seed, eta=eta, epsilon=eps, **kw)
    return sp, Learner(sp, lr_br=lr_br, lr_ar=lr_ar, **(learner or {}))


def _iterate(sp, ln, it):
    """One iteration of the sequential loop; statistics read back every other iteration."""
    sp.rollout(8)
    return ln.update(sync=it % 2 == 0)


def _resumed(nb, tmp_path, sp, ln, calls, make):
    """Saves (sp, ln) to a checkpoint file and loads it into the fresh pair make() builds."""
    from nfsp_b200 import checkpoint

    d = str(tmp_path / "ck")
    checkpoint.save(d, calls, selfplay=sp, learner=ln)
    assert os.listdir(d) == ["rank0-of-1.pt"]
    c, lc = make()
    assert checkpoint.load(d, selfplay=c, learner=lc) == {"calls": calls}
    return c, lc


def _resume_and_compare(nb, tmp_path, make, k, K, age=None):
    """a runs K iterations; b runs k, is saved and resumed as c, which runs the rest: c must stay equal to a.  age(sp)
    moves a run's counters before the save (a and b alike)."""
    a, la = make()
    b, lb = make()
    outs = [_iterate(a, la, it) for it in range(k)]
    assert [_iterate(b, lb, it) for it in range(k)] == outs
    if age is not None:
        age(a)
        age(b)
    c, lc = _resumed(nb, tmp_path, b, lb, k, make)
    _assert_same(a, c, la, lc, "resumed")
    for it in range(k, K):
        ra, rc = _iterate(a, la, it), _iterate(c, lc, it)
        assert ra == rc, it
        outs.append(ra)
        _assert_same(a, c, la, lc, "iteration %d" % it)
    return a, la, outs


def test_sequential_resume_with_wrapped_rings_and_replacing_reservoirs(nb, tmp_path):
    """Saved after k iterations, when both rings have wrapped and both reservoirs replace records (Algorithm R); a target
    copy falls after the resume (target_update_rate=3)."""
    kw = dict(rl_capacity=1 << 14, sl_capacity=1 << 11, max_steps_per_call=8, deterministic=True,
              learner=dict(target_update_rate=3))
    k, K = 4, 9                 # five updates after the resume: at least one target copy
    probe, lp = _make(nb, **kw)
    for it in range(k):
        _iterate(probe, lp, it)
    for m in probe.rl + probe.sl:
        assert int(m.total.item()) > m.capacity   # wrapped / replacing when the checkpoint is taken

    def age(sp):
        """A long-lived run: step counter, tickets and draw counters past 2^32 when the checkpoint is taken (the high
        words are carried by the file and key the draws after the resume)."""
        sp.env.step_counter = sp.env.step_counter + 2 ** 32 - 7
        for m in sp.rl + sp.sl:
            m.total.add_(2 ** 32 + 2 ** 33 * (m in sp.sl) + 12345)
            m.sample_calls += 2 ** 32 + 5

    a, _, outs = _resume_and_compare(nb, tmp_path, lambda: _make(nb, **kw), k, K, age=age)
    assert all(o["trained"] == 0xF for o in outs[1:])
    assert a.env.step_counter > 2 ** 32 and all(m.sample_calls > 2 ** 32 and int(m.total.item()) > 2 ** 32
                                                for m in a.rl + a.sl)


def test_sequential_resume_before_every_memory_is_ready(nb, tmp_path):
    """Saved while only some nets train (a partial net_mask: the reservoirs hold too few records at eta = 0.02); all four
    become ready after the resume."""
    kw = dict(n=512, eta=0.02, rl_capacity=1 << 14, sl_capacity=1 << 14, max_steps_per_call=8, deterministic=True,
              learner=dict(target_update_rate=3))
    K = 12
    probe, lp = _make(nb, **kw)
    masks = [_iterate(probe, lp, it)["trained"] for it in range(K)]
    partial = [it for it, m in enumerate(masks) if 0 < m < 0xF]
    assert partial and masks[-1] == 0xF, masks
    k = partial[0] + 1          # the saved learner has trained with a partial mask and has not seen all four ready
    _, _, outs = _resume_and_compare(nb, tmp_path, lambda: _make(nb, **kw), k, K)
    assert [o["trained"] for o in outs] == masks


def test_pipelined_trainer_resume(nb, tmp_path):
    """A PipelinedTrainer saved after step k (finish() first, as main.train does) and loaded into a fresh SelfPlay,
    Learner and trainer acts with the same lagged nets: finish() weights, game words and memories equal the trainer that
    never stopped."""
    from nfsp_b200 import checkpoint
    from nfsp_b200.learner import PipelinedTrainer

    def make():
        sp, ln = _make(nb, seed=21, rl_capacity=1 << 15, sl_capacity=1 << 12, max_steps_per_call=8, deterministic=True,
                       learner=dict(target_update_rate=3))
        for _ in range(3):
            sp.rollout(8)
        return sp, ln, PipelinedTrainer(sp, ln)

    k, K = 3, 8
    a, la, ta = make()
    b, lb, tb = make()
    for j in range(k):
        assert ta.step(8)["trained"] == 0xF and tb.step(8)["trained"] == 0xF
    tb.finish()
    d = str(tmp_path / "ck")
    checkpoint.save(d, k, selfplay=b, learner=lb, trainer=tb)
    c, lc, tc = make()
    assert checkpoint.load(d, selfplay=c, learner=lc, trainer=tc) == {"calls": k}
    assert tc.j == k
    for j in range(k, K):
        assert ta.step(8, sync=j % 2 == 0) == tc.step(8, sync=j % 2 == 0), j
    wa, wc = ta.finish(), tc.finish()
    assert torch.equal(wa, wc) and not torch.equal(wa, b.weights)
    _assert_same(a, c, la, lc, "finish")


CONFIGS = [  # tests/test_gpu_runs.py: seed, eta, epsilon per player, lr_br, lr_ar
    (1234, 0.1, (0.06, 0.06), 0.05, 0.1),
    (77, 0.3, (0.2, 0.05), 0.02, 0.2),
    (4242, 0.05, (0.1, 0.15), 0.1, 0.05),
]


def test_run_batch_resume_and_a_run_moved_out_of_the_batch(nb, tmp_path):
    """Three runs of different seeds, eta, epsilons and learning rates: the batch resumed from file equals the batch that
    never stopped, and run 1's state from the same file, loaded into a standalone SelfPlay / Learner and stepped alone,
    equals run 1 of the batch."""
    from nfsp_b200 import checkpoint
    from nfsp_b200.runs import RunBatch

    kw = dict(rl_capacity=1 << 16, sl_capacity=1 << 16, max_steps_per_call=8, deterministic=True)

    def run(cfg):
        s, e, ep, lb_, la_ = cfg
        return _make(nb, seed=s, eta=e, eps=list(ep), lr_br=lb_, lr_ar=la_, **kw)

    def batch():
        runs = [run(c) for c in CONFIGS]
        return RunBatch([sp for sp, _ in runs], [ln for _, ln in runs])

    def step(rb, it):
        rb.rollout(8)
        return rb.update(sync=it % 2 == 0) if it >= 2 else None

    k, K = 5, 10
    A, B = batch(), batch()
    for it in range(k):
        assert step(A, it) == step(B, it)
    d = str(tmp_path / "ck")
    checkpoint.save(d, k, runs=B)
    C = batch()
    assert checkpoint.load(d, runs=C) == {"calls": k}
    saved = torch.load(os.path.join(d, "rank0-of-1.pt"), weights_only=True)
    solo, lsolo = run(CONFIGS[1])
    solo.load_state_dict(saved["runs"]["runs"][1]["selfplay"])     # the file's RunBatch state: {"runs": [run 0, ...]}
    lsolo.load_state_dict(saved["runs"]["runs"][1]["learner"])
    for it in range(k, K):
        oa, oc = step(A, it), step(C, it)
        solo.rollout(8)
        os_ = lsolo.update(sync=it % 2 == 0)
        assert oa == oc and oa[1] == os_, it
        for r in range(3):
            _assert_same(A.sps[r], C.sps[r], A.learners[r], C.learners[r], "iteration %d run %d" % (it, r))
        _assert_same(A.sps[1], solo, A.learners[1], lsolo, "standalone, iteration %d" % it)
    assert A.exploitability() == C.exploitability()
    # and back: the standalone run's state loaded into a batch
    st = C.state_dict()
    st["runs"][1] = dict(selfplay=solo.state_dict(), learner=lsolo.state_dict())
    D = batch()
    D.load_state_dict(st)
    for it in range(K, K + 2):
        assert step(A, it) == step(D, it)
        for r in range(3):
            _assert_same(A.sps[r], D.sps[r], A.learners[r], D.learners[r], "batch again, iteration %d run %d" % (it, r))


def _rows(a):
    return [bytes(x) for x in np.ascontiguousarray(a).view(np.uint8).reshape(len(a), -1)]


def test_direct_rings_resume(nb, tmp_path):
    """direct_rings: the order of the records inside a launch follows the atomics.  save -> load -> save gives the same
    state; the first rollout after the resume gives the game words, step counter, counters and multiset of new records
    of the run that never stopped; the nets stay finite as training goes on."""
    from nfsp_b200 import checkpoint

    def make():
        return _make(nb, n=8192, seed=3, rl_capacity=1 << 18, sl_capacity=1 << 16, max_steps_per_call=8, direct_rings=True)

    a, la = make()
    for it in range(3):
        _iterate(a, la, it)
    d = str(tmp_path / "ck")
    checkpoint.save(d, 3, selfplay=a, learner=la)
    saved = torch.load(os.path.join(d, "rank0-of-1.pt"), weights_only=True)
    b, lb = make()
    checkpoint.load(d, selfplay=b, learner=lb)
    _same_state(saved["selfplay"], b.state_dict())
    _same_state(saved["learner"], lb.state_dict())
    before = [int(m.total.item()) for m in a.rl + a.sl]
    a.rollout(8)
    b.rollout(8)
    torch.cuda.synchronize()
    assert torch.equal(a.env.state_words(), b.env.state_words())
    assert a.env.step_counter == b.env.step_counter and torch.equal(a.stats, b.stats)
    for k, (ma, mb) in enumerate(zip(a.rl + a.sl, b.rl + b.sl)):
        t0, t1 = before[k], int(mb.total.item())
        assert int(ma.total.item()) == t1 and t0 < t1 <= ma.capacity, k
        assert Counter(_rows(ma.data[t0:t1].cpu().numpy())) == Counter(_rows(mb.data[t0:t1].cpu().numpy())), k
        assert torch.equal(ma.data[:t0], mb.data[:t0]), k
    w0 = b.weights.clone()
    for it in range(3, 8):
        assert _iterate(b, lb, it)["trained"] == 0xF
    assert torch.isfinite(b.weights).all() and torch.isfinite(lb.target).all() and not torch.equal(w0, b.weights)


def test_refusals_leave_the_target_as_it_was(nb, tmp_path, monkeypatch):
    """Mismatched shapes, a wrong format version, records staged at save and a save that fails part-way: ValueError or
    the save's own error, the target objects bit-identical to before, the previous checkpoint still loadable."""
    from nfsp_b200 import checkpoint

    base = dict(n=256, rl_capacity=1 << 13, sl_capacity=1 << 12, max_steps_per_call=8)
    sp, ln = _make(nb, **base)
    for it in range(3):
        _iterate(sp, ln, it)
    d = str(tmp_path / "ck")
    checkpoint.save(d, 3, selfplay=sp, learner=ln)

    def used(**over):
        kw = dict(base, seed=1234)
        kw.update(over)
        t, lt = _make(nb, **kw)
        t.rollout(8)
        lt.update()
        return t, lt

    cases = {
        "n_games": used(n=288),
        "rl_capacity": used(rl_capacity=1 << 14),
        "sl_capacity": used(sl_capacity=1 << 13),
        "variant": used(variant="cuda"),
        "minibatch": used(learner=dict(minibatch=64)),
        "deterministic": used(deterministic=True),
        "seed": used(seed=99),
    }
    for field, (t, lt) in cases.items():
        before = (t.state_dict(), lt.state_dict())
        with pytest.raises(ValueError, match=field):
            checkpoint.load(d, selfplay=t, learner=lt)
        _same_state(before, (t.state_dict(), lt.state_dict()), field)
    # a wrong format version, a file of another world size
    t, lt = used()
    before = (t.state_dict(), lt.state_dict())
    state = torch.load(os.path.join(d, "rank0-of-1.pt"), weights_only=True)
    for name, edit in (("format", dict(format=99)), ("world", dict(world=2))):
        bad = tmp_path / name
        bad.mkdir()
        torch.save(dict(state, **edit), str(bad / "rank0-of-1.pt"))
        with pytest.raises(ValueError, match=name):
            checkpoint.load(str(bad), selfplay=t, learner=lt)
        _same_state(before, (t.state_dict(), lt.state_dict()), name)
    # counters their holders cannot store: a memory total of 2^63 (an int64 tensor), a step counter or a draw counter of
    # 2^64 (uint64) -- refused before anything is written, not wrapped or half-loaded
    sp_state = state["selfplay"]
    for name, field, edit in (("total", "total", lambda s: s["sl"][1].update(total=2 ** 63)),
                              ("step", "step", lambda s: s.update(step=2 ** 64)),
                              ("calls", "sample_calls", lambda s: s["rl"][0].update(sample_calls=2 ** 64))):
        sp_bad = dict(sp_state, rl=[dict(m) for m in sp_state["rl"]], sl=[dict(m) for m in sp_state["sl"]])
        edit(sp_bad)
        bad = tmp_path / name
        bad.mkdir()
        torch.save(dict(state, selfplay=sp_bad), str(bad / "rank0-of-1.pt"))
        with pytest.raises(ValueError, match=field):
            checkpoint.load(str(bad), selfplay=t, learner=lt)
        _same_state(before, (t.state_dict(), lt.state_dict()), name)
    # a single run's file loaded without its learner
    with pytest.raises(ValueError, match="holds"):
        checkpoint.load(d, selfplay=t)
    _same_state(before, (t.state_dict(), lt.state_dict()), "parts")
    # records staged but not flushed: no save, the directory as it was
    files = {f: open(os.path.join(d, f), "rb").read() for f in os.listdir(d)}
    sp.rollout(8, insert=False)
    with pytest.raises(ValueError, match="staged"):
        checkpoint.save(d, 4, selfplay=sp, learner=ln)
    assert {f: open(os.path.join(d, f), "rb").read() for f in os.listdir(d)} == files
    sp.flush()
    ln.update()
    # a save that fails part-way: the old file stays, no temporary file is left behind
    real_save = torch.save

    def failing(obj, f, *a, **k):
        f.write(b"partial")
        raise OSError("disk full")

    monkeypatch.setattr(torch, "save", failing)
    with pytest.raises(OSError, match="disk full"):
        checkpoint.save(d, 5, selfplay=sp, learner=ln)
    monkeypatch.setattr(torch, "save", real_save)
    assert {f: open(os.path.join(d, f), "rb").read() for f in os.listdir(d)} == files
    u, lu = _make(nb, **base)
    assert checkpoint.load(d, selfplay=u, learner=lu) == {"calls": 3}
    _same_state(state["selfplay"], u.state_dict())
    _same_state(state["learner"], lu.state_dict())


def _cli(tmp_path, extra):
    from nfsp_b200 import main as drv

    cfg = tmp_path / "config.ini"
    if not cfg.exists():
        cfg.write_text("[Agent]\nMRLSize = 32768\nMSLSize = 8192\n")
    return drv.main(["--config", str(cfg), "--games", "4096", "--steps-per-call", "8", "--deterministic",
                     "--report-every", "5"] + extra)


def _strip(rows):
    out = []
    for r in rows:
        r = dict(r)
        r.pop("transitions_per_sec")
        out.append(r)
    return out


@pytest.mark.parametrize("runs", [1, 3], ids=["sequential", "runs-3"])
def test_cli_checkpoint_and_resume(nb, tmp_path, runs):
    """main.py --checkpoint DIR --checkpoint-every 5 until --episodes E1, then --resume DIR with a larger --episodes:
    the resumed call reports the rows of the run that never stopped (calls, hands, transitions, actions, the proxy and
    the exact exploitability).  A resume of the finished run at E1 itself has nothing left to do, and a command line of
    another shape is refused, naming the field."""
    extra = ["--runs", str(runs)] if runs > 1 else []
    ref = _strip(_cli(tmp_path, extra + ["--episodes", "250000"]))
    assert len(ref) >= 5
    stop = ref[len(ref) // 2]
    e1 = stop["hands"] if runs == 1 else min(r["hands"] for r in stop["runs"])
    d = str(tmp_path / "ck")
    first = _strip(_cli(tmp_path, extra + ["--episodes", str(e1), "--checkpoint", d, "--checkpoint-every", "5"]))
    assert first == ref[:len(ref) // 2 + 1]
    assert _cli(tmp_path, extra + ["--episodes", str(e1), "--resume", d]) == []
    with pytest.raises(ValueError, match="n_games"):
        _cli(tmp_path, extra + ["--episodes", "250000", "--resume", d, "--games", "2048"])
    rest = _strip(_cli(tmp_path, extra + ["--episodes", "250000", "--resume", d]))
    assert rest == ref[len(ref) // 2 + 1:] and rest


def test_checkpoint_on_two_gpus_when_there_are_two(tmp_path):
    """tests/mgpu_checkpoint_check.py under torchrun: a 2-rank run with the peer exchange, saved and resumed, equals the
    one that never stopped on every rank, and a rank file of the wrong rank is refused on both ranks."""
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533",
                          os.path.join(root, "tests", "mgpu_checkpoint_check.py"), str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "mgpu checkpoint check ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
