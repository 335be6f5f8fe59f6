"""CPU checks of hyperparameter sweeps (nfsp_b200.sweep, main.py --sweep): the grid and its seeds, the assignment of runs
to ranks, the checkpoint record, and the command lines the driver refuses before any device is touched."""
import pytest

torch = pytest.importorskip("torch")


@pytest.fixture
def cfg(tmp_path):
    from nfsp_b200.config import load_config

    p = tmp_path / "config.ini"
    p.write_text("[Agent]\nEta = 0.2\nGamma = 0.9\nTargetModelUpdateRate = 150\n[Utils]\nSeed = 100\n")
    return load_config(str(p))


def test_grid_order_and_seeds(cfg):
    from nfsp_b200 import sweep

    axes = sweep.parse_axes(["Eta=0.05,0.1", "Agent.LearningRateBR=0.01,0.02,0.03"])
    assert axes == [("Agent.Eta", [0.05, 0.1]), ("Agent.LearningRateBR", [0.01, 0.02, 0.03])]
    runs = sweep.expand(axes, 2, cfg)
    assert len(runs) == 12 and [r["run"] for r in runs] == list(range(12))
    # the last axis fastest, seeds innermost: run i = (point i // 2, seed 100 + i % 2)
    assert [(r["point"], r["seed"]) for r in runs] == [(i // 2, 100 + i % 2) for i in range(12)]
    assert [(r["hparams"]["Eta"], r["hparams"]["LearningRateBR"]) for r in runs[::2]] == \
        [(e, lr) for e in (0.05, 0.1) for lr in (0.01, 0.02, 0.03)]
    # what is not swept comes from config.ini
    assert all(r["hparams"]["Gamma"] == 0.9 and r["hparams"]["LearningRateAR"] == 0.1 and
               r["hparams"]["TargetModelUpdateRate"] == 150 for r in runs)
    # a swept base seed: each point's seeds start at its own base
    runs = sweep.expand(sweep.parse_axes(["Seed=7,1000", "TargetModelUpdateRate=3"]), 3, cfg)
    assert [r["seed"] for r in runs] == [7, 8, 9, 1000, 1001, 1002]
    assert all(type(r["hparams"]["TargetModelUpdateRate"]) is int and r["hparams"]["Eta"] == 0.2 for r in runs)
    # a seed-only sweep: config.ini's seed, --runs seeds
    assert [r["seed"] for r in sweep.expand(sweep.parse_axes(["Seed=1234"]), 64, cfg)] == list(range(1234, 1298))


@pytest.mark.parametrize("n_runs,world", [(1, 1), (5, 1), (32, 1), (8, 8), (9, 8), (60, 8), (63, 2), (64, 2), (256, 8),
                                          (3, 2)])
def test_assignment_is_contiguous_balanced_and_complete(n_runs, world):
    from nfsp_b200 import _lib, sweep

    sweep.check_layout(n_runs, world)
    blocks = [sweep.rank_runs(n_runs, r, world) for r in range(world)]
    assert [i for b in blocks for i in b] == list(range(n_runs))            # every run once, in order: contiguous blocks
    sizes = [len(b) for b in blocks]
    assert max(sizes) - min(sizes) <= 1 and min(sizes) >= 1 and max(sizes) <= _lib.MAX_RUNS


@pytest.mark.parametrize("n_runs,world,why", [(1, 2, "every rank needs a run"), (33, 1, "at most"), (257, 8, "at most")])
def test_layouts_that_are_refused(n_runs, world, why):
    from nfsp_b200 import sweep

    with pytest.raises(ValueError, match=why):
        sweep.check_layout(n_runs, world)


def test_checkpoint_record_names_what_differs(cfg):
    from nfsp_b200 import sweep

    runs = sweep.expand(sweep.parse_axes(["Eta=0.05,0.1"]), 2, cfg)
    rec = sweep.record(runs, 2)
    assert sweep.record_difference(rec, sweep.record(runs, 2)) is None
    other = sweep.expand(sweep.parse_axes(["Eta=0.05,0.2"]), 2, cfg)
    assert "run 2: Eta is 0.1 in the checkpoint but 0.2 here" == sweep.record_difference(rec, sweep.record(other, 2))
    assert "runs" in sweep.record_difference(rec, sweep.record(sweep.expand(sweep.parse_axes(["Eta=0.05,0.1"]), 3, cfg), 2))
    assert "ranks" in sweep.record_difference(rec, sweep.record(runs, 1))
    assert "no sweep" in sweep.record_difference(None, rec)


def _refused(capsys, monkeypatch, argv, world=1):
    """main.main(argv) exits with code 2 and touches no device; returns its error message."""
    from nfsp_b200 import main

    def no_device(*a, **k):
        raise AssertionError("a device was touched")

    monkeypatch.setattr(torch.cuda, "set_device", no_device)
    monkeypatch.setattr(torch.cuda, "device_count", no_device)
    monkeypatch.setenv("WORLD_SIZE", str(world))
    monkeypatch.setenv("RANK", "0")
    monkeypatch.setenv("LOCAL_RANK", "0")
    with pytest.raises(SystemExit) as e:
        main.main(argv)
    assert e.value.code == 2
    return capsys.readouterr().err


@pytest.mark.parametrize("spec", ["MiniBatchSize=64,128", "Agent.MRLSize=1000", "MSLSize=10", "HiddenLayer=32",
                                  "Environment.Decksize=6", "Environment.Suits=2"])
def test_shared_keys_are_refused(capsys, monkeypatch, spec):
    assert "shared by every run of a batch" in _refused(capsys, monkeypatch, ["--sweep", spec])


@pytest.mark.parametrize("argv,why", [
    (["--sweep", "Temperature=1,2"], "unknown key"),
    (["--sweep", "Agent.Omega=0.1"], "unknown key"),
    (["--sweep", "Eta"], "KEY=V1,V2"),
    (["--sweep", "Eta=0.1", "--sweep", "Agent.Eta=0.2"], "given twice"),
    (["--sweep", "Eta="], "empty value"),
    (["--sweep", "Eta=0.1,,0.2"], "empty value"),
    (["--sweep", "Eta=0.1,"], "empty value"),
    (["--sweep", "Gamma=0.9,high"], "not a number"),
    (["--sweep", "Epsilon=nan"], "not a finite number"),
    (["--sweep", "Seed=1.5"], "not an integer"),
    (["--sweep", "TargetModelUpdateRate=0,5"], "below 1"),
    (["--sweep", "TargetModelUpdateRate=2.5"], "not an integer"),
    (["--sweep", "Eta=0.1", "--pipelined"], "--pipelined"),
    (["--sweep", "Eta=0.1", "--updates-per-call", "2"], "--updates-per-call"),
    (["--sweep", "Eta=0.1", "--variant", "cuda"], "--variant cuda"),
    (["--sweep", "Eta=0.1", "--variant", "tcgen05"], "--variant tcgen05"),
    (["--sweep", "Eta=0.1,0.2,0.3", "--runs", "11"], "at most 32"),
    (["--sweep", "Seed=1", "--runs", "0"], "--runs must be at least 1"),
    (["--results", "out.jsonl"], "--results needs --sweep"),
])
def test_command_lines_that_are_refused(capsys, monkeypatch, argv, why):
    assert why in _refused(capsys, monkeypatch, argv)


def test_rank_layouts_that_are_refused(capsys, monkeypatch):
    assert "every rank needs a run" in _refused(capsys, monkeypatch, ["--sweep", "Eta=0.1,0.2", "--runs", "1"], world=4)
    assert "at most 32" in _refused(capsys, monkeypatch, ["--sweep", "Seed=1", "--runs", "129"], world=4)
    # without --sweep nothing changes: independent runs stay on one rank
    assert "--runs > 1" in _refused(capsys, monkeypatch, ["--runs", "2"], world=2)


def test_a_checkpoint_of_another_world_size_is_refused_naming_it(tmp_path):
    from nfsp_b200 import checkpoint

    torch.save(dict(format=checkpoint.FORMAT, world=2, rank=0, driver=dict(calls=3)), str(tmp_path / "rank0-of-2.pt"))
    with pytest.raises(ValueError, match=r"another number of ranks \(rank0-of-2.pt\) than the 1 here"):
        checkpoint.load(str(tmp_path))
