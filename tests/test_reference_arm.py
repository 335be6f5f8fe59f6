"""-m "not gpu": the CPU legs of bench.py run the REFERENCE'S OWN files (oracle/ref_timing.py).  Here: materialise() copies
the files the drivers execute verbatim (into the git-ignored baseline/_ref), and, where the reference's files are present,
both drivers play hands and count transitions as the reference's own counters do."""
import filecmp
import os

import pytest

from oracle import ref_timing


def test_travelling_copy_is_verbatim(tmp_path):
    src, dst = tmp_path / "reference", tmp_path / "copy"
    for i, rel in enumerate(ref_timing.FILES):  # a stand-in tree: distinct bytes per file, every byte value present
        (src / rel).parent.mkdir(parents=True, exist_ok=True)
        (src / rel).write_bytes(bytes((i + k) % 256 for k in range(256 * (i + 1))))
    assert ref_timing.materialise(str(src), str(dst))
    for rel in ref_timing.FILES:
        assert filecmp.cmp(os.path.join(src, rel), os.path.join(dst, rel), shallow=False), rel
    assert not ref_timing.materialise(str(tmp_path / "absent"), str(tmp_path / "copy2"))
    assert not (tmp_path / "copy2").exists()


@pytest.mark.parametrize("kind", ["legacy", "nfsp"])
def test_drivers_play_and_count(kind):
    if ref_timing.reference_root() is None:
        pytest.skip("no reference tree")
    r = ref_timing.run(kind, 300, 1)
    assert r["hands_per_proc"] == 300 and r["seconds"] > 0
    # a Leduc hand is 1-6 decisions under main.train; the README loop steps both players per iteration (2-10 per hand)
    lo, hi = (2, 10) if kind == "legacy" else (1, 6)
    assert lo * 300 <= r["transitions"] <= hi * 300
    assert r["transitions_per_sec"] == pytest.approx(r["transitions"] / r["seconds"])
