"""The checkpoint file format without a GPU (nfsp_b200.checkpoint): the driver record round trip, refusals of a wrong
format version, world size, rank or missing file, and a save that fails part-way leaving the previous file in place."""
import os

import pytest

torch = pytest.importorskip("torch")

from nfsp_b200 import checkpoint  # noqa: E402


def test_driver_record_round_trip_and_refusals(tmp_path):
    d = str(tmp_path / "ck")
    checkpoint.save(d, 7)
    assert os.listdir(d) == ["rank0-of-1.pt"]
    assert checkpoint.load(d) == {"calls": 7}
    state = torch.load(os.path.join(d, "rank0-of-1.pt"), weights_only=True)
    assert state == {"format": checkpoint.FORMAT, "world": 1, "rank": 0, "driver": {"calls": 7}}
    for name, edit in (("format", dict(format=checkpoint.FORMAT + 1)), ("world", dict(world=2)), ("rank", dict(rank=1)),
                       ("calls", dict(driver={"calls": -1})), ("holds", dict(learner={}))):
        bad = tmp_path / name
        bad.mkdir()
        torch.save(dict(state, **edit), str(bad / "rank0-of-1.pt"))
        with pytest.raises(ValueError, match=name):
            checkpoint.load(str(bad))
    with pytest.raises(ValueError, match="cannot read"):
        checkpoint.load(str(tmp_path / "missing"))
    (tmp_path / "garbage").mkdir()
    (tmp_path / "garbage" / "rank0-of-1.pt").write_bytes(b"not a checkpoint")
    with pytest.raises(ValueError, match="cannot read"):
        checkpoint.load(str(tmp_path / "garbage"))


def test_a_save_that_fails_part_way_keeps_the_previous_file(tmp_path, monkeypatch):
    d = str(tmp_path / "ck")
    checkpoint.save(d, 3)
    before = open(os.path.join(d, "rank0-of-1.pt"), "rb").read()

    def failing(obj, f, *a, **k):
        f.write(b"partial")
        raise OSError("disk full")

    monkeypatch.setattr(torch, "save", failing)
    with pytest.raises(OSError, match="disk full"):
        checkpoint.save(d, 4)
    monkeypatch.undo()
    assert os.listdir(d) == ["rank0-of-1.pt"]
    assert open(os.path.join(d, "rank0-of-1.pt"), "rb").read() == before
    assert checkpoint.load(d) == {"calls": 3}


def test_counters_are_bounded_by_what_holds_them():
    """A memory's total lives in an int64 tensor, the step and draw counters go to the library as uint64: values they
    cannot hold are refused with the field named, before anything is loaded (torch would refuse total = 2^63 only after
    the slots were overwritten; ctypes would wrap step 2^64 + 5 to 5)."""
    from nfsp_b200.batched import check_numbers

    mem = dict(below=dict(total=2 ** 63, sample_calls=2 ** 64), total=int, sample_calls=int)
    check_numbers(dict(total=2 ** 63 - 1, sample_calls=2 ** 64 - 1), "memory", **mem)
    for field, d in (("total", dict(total=2 ** 63, sample_calls=0)), ("sample_calls", dict(total=0, sample_calls=2 ** 64))):
        with pytest.raises(ValueError, match="%s must be below" % field):
            check_numbers(d, "memory", **mem)
    check_numbers(dict(step=2 ** 64 - 1), "SelfPlay", below=dict(step=2 ** 64), step=int)
    with pytest.raises(ValueError, match="step must be below 2\\*\\*64"):
        check_numbers(dict(step=2 ** 64 + 5), "SelfPlay", below=dict(step=2 ** 64), step=int)
