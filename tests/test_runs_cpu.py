"""CPU checks of the independent-runs interface: the header's run limits and their ctypes mirrors, and the driver's
refusals, which come before any device is touched."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _define(name):
    src = open(os.path.join(ROOT, "include", "nfsp_b200.h")).read()
    return int(re.search(r"#define %s (\d+)" % name, src).group(1))


def test_run_limits_match_the_header():
    from nfsp_b200 import _lib

    assert _define("NFSP_MAX_RUNS") == _lib.MAX_RUNS
    # the four memories of every run of a batch sample in one launch
    assert _define("NFSP_MAX_SAMPLE_REQS") == _lib.MAX_SAMPLE_REQS == 4 * _lib.MAX_RUNS
    # the fit of every run in one wave of 4 CTAs per run on the 148 SMs of a B200
    assert 4 * _lib.MAX_RUNS <= 148
    # the geometry of the row-parallel fit kernel, which the learner checks before it sets up the peer exchange
    assert _define("NFSP_FIT_ROWS_MAX_MINIBATCH") == _lib.FIT_ROWS_MAX_MINIBATCH
    assert _define("NFSP_FIT_ROWS_MAX_STEP") == _lib.FIT_ROWS_MAX_STEP


@pytest.mark.parametrize("extra", [["--pipelined"], ["--runs", "0"]])
def test_main_refuses_runs_it_cannot_train(extra, monkeypatch):
    from nfsp_b200 import main

    args = ["--runs", "2"] + extra if extra[0] != "--runs" else extra
    with pytest.raises(SystemExit) as e:
        main.main(args)
    assert e.value.code == 2


def test_main_refuses_runs_over_several_ranks(monkeypatch):
    from nfsp_b200 import main

    monkeypatch.setenv("WORLD_SIZE", "2")
    monkeypatch.setenv("RANK", "0")
    monkeypatch.setenv("LOCAL_RANK", "0")
    with pytest.raises(SystemExit) as e:
        main.main(["--runs", "2"])
    assert e.value.code == 2
