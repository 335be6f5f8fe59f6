"""-m gpu: hyperparameter sweeps (main.py --sweep, nfsp_b200.sweep, Learner(data_parallel=False)).

Each run of a sweep is the run main.py trains alone with those settings, bit for bit; the rows a sweep reports do not
depend on how many ranks train it; a resumed sweep reproduces the uninterrupted one.  The multi-rank cases run the real
command line under torch.distributed.run; two ranks share one GPU unless the test is the two-GPU one."""
import json
import os
import signal
import subprocess
import sys

import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = ["--games", "4096", "--steps-per-call", "8", "--deterministic", "--report-every", "3"]
MEMORIES = "[Agent]\nMRLSize = 32768\nMSLSize = 8192\n"   # small memories, as in tests/test_gpu_checkpoint.py
EPISODES = 100000                                       # about nine calls: reports at calls 1, 3, 6, 9
TIMING = ("transitions_per_sec", "rank")               # where and how fast a row was computed, not what


@pytest.fixture(scope="module")
def nb():
    import nfsp_b200

    assert torch.cuda.is_available()
    return nfsp_b200


def _config(path, text=""):
    path.write_text(MEMORIES + text)
    return str(path)


def _cli(args):
    from nfsp_b200 import main as drv

    return drv.main(BASE + args)


def _strip(rows):
    return [{k: v for k, v in r.items() if k not in TIMING} for r in rows]


def _read(path):
    with open(path) as f:
        return [json.loads(ln) for ln in f]


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


SWEEPS = {
    "eta-x-lr-x-seeds": ["--sweep", "Eta=0.1,0.3", "--sweep", "LearningRateBR=0.02,0.1", "--runs", "2"],
    # no other test holds gamma and the target-update rate to a run trained alone; rates 2 and 3 copy the target nets
    # several times in the updates of this sweep
    "gamma-x-target-rate": ["--sweep", "Agent.Gamma=0.8,0.99", "--sweep", "TargetModelUpdateRate=2,3",
                            "--sweep", "Seed=99"],
}


@pytest.mark.parametrize("name", list(SWEEPS))
def test_each_run_equals_its_standalone_run(nb, tmp_path, name):
    """A one-rank sweep, saved when it ends: every run's state in the file -- game words, step counter, rollout counters,
    all four memories, acting and target nets, epsilons, schedules, learning rates -- equals, bit for bit, that of
    main.py trained alone (--runs 1) with the run's seed and hyperparameters written into its config.ini, stopped at the
    same call; and the sweep's rows of that run equal the standalone run's rows."""
    d, res = str(tmp_path / "ck"), str(tmp_path / "sweep.jsonl")
    rows = _cli(SWEEPS[name] + ["--config", _config(tmp_path / "config.ini"), "--episodes", str(EPISODES),
                                "--checkpoint", d, "--results", res])
    assert _read(res) == json.loads(json.dumps(rows))
    runs = [r for r in rows if r["kind"] == "run"]
    last = max(r["calls"] for r in rows)
    saved = torch.load(os.path.join(d, "rank0-of-1.pt"), weights_only=True)
    assert saved["driver"]["calls"] == last and len(saved["driver"]["sweep"]["runs"]) == len(saved["runs"]["runs"])
    copies = []
    for i, state in enumerate(saved["runs"]["runs"]):
        mine = [r for r in runs if r["run"] == i]
        hp, seed = mine[0]["hparams"], mine[0]["seed"]
        cfg = _config(tmp_path / ("run%d.ini" % i), "".join("%s = %r\n" % kv for kv in hp.items()) +
                      "[Utils]\nSeed = %d\n" % seed)
        solo_dir = str(tmp_path / ("solo%d" % i))
        # the sweep ran until every run had played EPISODES hands: this run alone stops at the same call when its own
        # hand count at that call is the goal
        solo = _cli(["--config", cfg, "--episodes", str(mine[-1]["hands"]), "--checkpoint", solo_dir])
        assert len(solo) == len(mine) and solo[-1]["calls"] == last, i
        for a, b in zip(_strip(solo), _strip(mine)):
            assert a == {k: b[k] for k in a}, (i, a["calls"])
        alone = torch.load(os.path.join(solo_dir, "rank0-of-1.pt"), weights_only=True)
        _same_state(state["selfplay"], alone["selfplay"], "run %d selfplay" % i)
        _same_state(state["learner"], alone["learner"], "run %d learner" % i)
        assert alone["learner"]["gamma"] == hp["Gamma"] and alone["selfplay"]["eta"] == hp["Eta"]
        copies.append(alone["learner"]["target_update_count"][0] // alone["learner"]["target_update_rate"])
    if "TargetModelUpdateRate" in " ".join(SWEEPS[name]):
        assert min(copies) >= 2, copies
    # one grid point row per report and point, with the mean and spread of its seeds' exact exploitability
    points = [r for r in rows if r["kind"] == "point" and r["calls"] == last]
    for p in points:
        values = [r["exploitability"]["value"] for r in runs if r["calls"] == last and r["point"] == p["point"]]
        assert p["seeds"] == [r["seed"] for r in runs if r["calls"] == last and r["point"] == p["point"]]
        assert p["exploitability_mean"] == pytest.approx(sum(values) / len(values))


def _torchrun(args, timeout=900, one_gpu=True, script=None):
    """Two ranks under torch.distributed.run in a session of their own; the whole process group is killed if the
    timeout expires.  one_gpu: both ranks see the same GPU.  Returns (exit code, stdout, stderr)."""
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    if one_gpu:
        env["CUDA_VISIBLE_DEVICES"] = os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]
    target = [script] if script is not None else ["-m", "nfsp_b200.main"] + BASE + args
    p = subprocess.Popen([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nnodes=1",
                          "--nproc-per-node", "2"] + target, cwd=ROOT, env=env, stdout=subprocess.PIPE,
                         stderr=subprocess.PIPE, text=True, start_new_session=True)
    try:
        out, err = p.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)
        p.communicate()
        raise
    return p.returncode, out, err


SWEEP = ["--sweep", "Eta=0.1,0.3", "--sweep", "LearningRateBR=0.02,0.1", "--runs", "2"]


@pytest.fixture(scope="module")
def one_rank(nb, tmp_path_factory):
    """The sweep on one rank, in this process: its results file."""
    tmp = tmp_path_factory.mktemp("one-rank")
    res = str(tmp / "one.jsonl")
    _cli(SWEEP + ["--config", _config(tmp / "config.ini"), "--episodes", str(EPISODES), "--results", res])
    return _read(res)


def test_results_do_not_depend_on_world_size_and_resume_reproduces_them(one_rank, tmp_path):
    """The same sweep under two ranks sharing one GPU writes the one-rank results file, line for line (timing and the
    rank that computed a row aside).  Stopped half-way with a checkpoint and resumed -- its results file holding the
    lines of reports after the checkpoint, as one whose process died before its next save would -- it writes that file
    again.  A resume with another --sweep value is refused on both ranks, naming the run and value."""
    cfg = _config(tmp_path / "config.ini")
    ref = _strip(one_rank)
    assert {r["run"]: r["rank"] for r in one_rank if r["kind"] == "run"} == {i: 0 for i in range(8)}
    res = str(tmp_path / "two.jsonl")
    code, out, err = _torchrun(SWEEP + ["--config", cfg, "--episodes", str(EPISODES), "--results", res])
    assert code == 0, out[-3000:] + err[-3000:]
    two = _read(res)
    assert _strip(two) == ref
    assert {r["run"]: r["rank"] for r in two if r["kind"] == "run"} == {i: i // 4 for i in range(8)}
    # interrupted at the second report, resumed
    calls = sorted({r["calls"] for r in ref})
    stop = calls[len(calls) // 2 - 1]
    e1 = min(r["hands"] for r in ref if r["kind"] == "run" and r["calls"] == stop)
    d, part = str(tmp_path / "ck"), str(tmp_path / "part.jsonl")
    code, out, err = _torchrun(SWEEP + ["--config", cfg, "--episodes", str(e1), "--results", part, "--checkpoint", d,
                                        "--checkpoint-every", "2"])
    assert code == 0, out[-3000:] + err[-3000:]
    assert sorted(os.listdir(d)) == ["rank0-of-2.pt", "rank1-of-2.pt"]
    assert _strip(_read(part)) == [r for r in ref if r["calls"] <= stop]
    with open(part, "a") as f:
        f.writelines(json.dumps(r) + "\n" for r in one_rank if r["calls"] > stop)
    code, out, err = _torchrun(SWEEP + ["--config", cfg, "--episodes", str(EPISODES), "--results", part, "--resume", d])
    assert code == 0, out[-3000:] + err[-3000:]
    assert _strip(_read(part)) == ref
    # another Eta: refused on both ranks before anything is loaded
    changed = ["--sweep", "Eta=0.1,0.2"] + SWEEP[2:]
    code, out, err = _torchrun(changed + ["--config", cfg, "--episodes", str(EPISODES), "--resume", d])
    assert code != 0
    for rank in range(2):
        assert "rank %d:" % rank in err and "Eta is 0.3 in the checkpoint but 0.2 here" in err, err[-3000:]


def test_results_on_two_gpus_when_there_are_two(one_rank, tmp_path):
    """The same sweep with one rank per GPU writes the one-rank results file."""
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    res = str(tmp_path / "two.jsonl")
    code, out, err = _torchrun(SWEEP + ["--config", _config(tmp_path / "config.ini"), "--episodes", str(EPISODES),
                                        "--results", res], one_gpu=False)
    assert code == 0, out[-3000:] + err[-3000:]
    assert _strip(_read(res)) == _strip(one_rank)


def test_local_learners_never_wait_on_each_other():
    """tests/sweep_local_check.py: two ranks with learners that train alone run different numbers of updates between
    two barriers and both finish."""
    code, out, err = _torchrun([], timeout=600, script=os.path.join(ROOT, "tests", "sweep_local_check.py"))
    assert code == 0 and "sweep local check ok" in out, out[-3000:] + err[-3000:]
