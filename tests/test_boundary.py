"""CPU-only checks of the drop-in boundary: the C-ABI library loads and exports every symbol the header
declares (no compute without a GPU), there is no CPU fallback, and the product never touches oracle/."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "neural-ficititious-self-play-in-imperfect-information-games_b200")
HEADER = os.path.join(ROOT, "include", "nfsp_b200.h")


@pytest.fixture(scope="module")
def nb():
    import __graft_entry__ as g

    if not os.path.exists(os.path.join(PKG, "libnfsp_b200.so")):
        g.build()
    import nfsp_b200

    return nfsp_b200


def header_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(nfsp_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(nb):
    L = nb.lib()
    declared = header_symbols()
    assert declared == sorted(nb.SYMBOLS)
    for name in declared:
        assert hasattr(L, name), name
    assert L.nfsp_version() >= 100
    out = subprocess.run(["nm", "-D", "--defined-only", nb.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (nfsp_\w+)", out))
    assert exported == set(declared)


def test_no_torch_types_in_the_abi():
    src = open(HEADER).read()
    assert 'extern "C"' in src
    code = re.sub(r"/\*.*?\*/", "", src, flags=re.S)  # declarations only, comments stripped
    assert "torch" not in code and "at::" not in code and "Tensor" not in code and "#include <torch" not in src


def test_library_is_sm100a_only(nb):
    out = subprocess.run(["cuobjdump", "--list-elf", nb.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_fails_loudly_without_a_gpu(nb):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(nb.NfspError):
        nb.BatchedNfspEnv(8)
    h = ctypes.c_void_p()
    rc = nb.lib().nfsp_env_create(1, 8, 1, 0, 0, ctypes.byref(h))
    assert rc < 0 and nb.lib().nfsp_last_error()


def test_argument_errors_are_reported(nb):
    h = ctypes.c_void_p()
    assert nb.lib().nfsp_env_create(7, 8, 1, 0, 0, ctypes.byref(h)) == -1
    assert b"rules" in nb.lib().nfsp_last_error()
    assert nb.lib().nfsp_env_create(1, 0, 1, 0, 0, ctypes.byref(h)) == -1
    # game ids past 2^32 would replay the deals of game id - 2^32 (Philox counter word 0 is the low half)
    assert nb.lib().nfsp_env_create(1, 8, 1, 2 ** 32 - 7, 0, ctypes.byref(h)) == -1
    assert b"2^32" in nb.lib().nfsp_last_error()
    assert nb.lib().nfsp_expand_obs(None, 4, None, None) == -1


def test_product_never_uses_the_oracle():
    """oracle/ is test infrastructure: no file of the package, bench's GPU arm aside, may reference it."""
    bad = []
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                if re.search(r"\boracle\b|liboracle|/root/reference", text):
                    bad.append(os.path.join(dirpath, f))
    assert not bad, bad


def test_config_loader_matches_reference_keys(nb, tmp_path):
    cfg = nb.load_config(None)
    assert cfg.getfloat("Agent", "Eta") == 0.1 and cfg.getfloat("Agent", "Epsilon") == 0.06
    assert cfg.getint("Agent", "MRLSize") == 200000 and cfg.getint("Agent", "MSLSize") == 2000000
    assert cfg.getint("Utils", "Buffersize") == 40000 and cfg.getint("Utils", "Seed") == 1234
    p = tmp_path / "config.ini"
    p.write_text("[Agent]\nEta: 0.25\n[Environment]\nChoices: 5\n")
    with pytest.raises(ValueError):
        nb.load_config(str(p))
    p.write_text("[Agent]\nEta: 0.25\n")
    assert nb.load_config(str(p)).getfloat("Agent", "Eta") == 0.25


def test_obs_mask_roundtrip_host(nb):
    import torch

    x = (torch.rand(50, 30) < 0.3).float()
    m = nb.obs_to_mask(x)
    back = ((m[:, None].to(torch.int64) >> torch.arange(30)) & 1).float()
    assert torch.equal(back, x)
    with pytest.raises(ValueError):
        nb.obs_to_mask(torch.full((1, 30), 0.5))


def test_dropin_modules_import_without_gpu(nb):
    nb.install_dropin()
    import agent.agent  # noqa: F401
    import leduc.deck as deck
    import leduc.env  # noqa: F401
    import leduc.newenv as newenv
    import utils.ReservoirBuffer  # noqa: F401
    import utils.replay_buffer  # noqa: F401

    d = deck.Deck(6)
    assert sorted(c.rank for c in d._cards) == [0, 0, 1, 1, 2, 2] and d.fake_pub_card().rank == -1
    d.shuffle()
    assert d.pick_up().rank in (0, 1, 2) and len(d._cards) == 5
    import numpy as np

    assert newenv.action_code(np.array([[0.0, 0.5, 0.5], [0, 0, 0], [0.1, 0.2, 0.9]])).tolist() == [1, 3, 2]


def test_ctypes_mirrors_match_the_header(nb, tmp_path):
    """Every struct of include/nfsp_b200.h has the size and field offsets of its ctypes mirror in _lib.py, and the
    constants agree: a C program compiled against the header (gcc, no CUDA needed) prints them."""
    from nfsp_b200 import _lib

    structs = {"nfsp_rollout_io": _lib.RolloutIO, "nfsp_insert_req": _lib.InsertReq, "nfsp_sample_req": _lib.SampleReq,
               "nfsp_learner_io": _lib.LearnerIO, "nfsp_peers": _lib.Peers}
    consts = {"NFSP_RULES_LEGACY": _lib.RULES_LEGACY, "NFSP_RULES_NFSP": _lib.RULES_NFSP, "NFSP_OBS_DIM": _lib.OBS_DIM,
              "NFSP_ACTIONS": _lib.ACTIONS, "NFSP_HIDDEN": _lib.HIDDEN, "NFSP_NET_PARAMS": _lib.NET_PARAMS,
              "NFSP_EXPORT_FIELDS": _lib.EXPORT_FIELDS, "NFSP_LEGACY_EXPORT_FIELDS": _lib.LEGACY_EXPORT_FIELDS,
              "NFSP_STATS_FIELDS": _lib.STATS_FIELDS, "NFSP_MAX_PEERS": _lib.MAX_PEERS,
              "NFSP_PEER_BUF_FLOATS": _lib.PEER_BUF_FLOATS}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "nfsp_b200.h"', "int main(void) {"]
    for name, cls in structs.items():
        lines.append('printf("%s %%zu\\n", sizeof(%s));' % (name, name))
        for field, _ in cls._fields_:
            lines.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (name, field, name, field))
    for name in consts:
        lines.append('printf("%s %%ld\\n", (long)(%s));' % (name, name))
    lines += ["return 0;", "}"]
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for name, cls in structs.items():
        assert int(got[name]) == ctypes.sizeof(cls), name
        for field, _ in cls._fields_:
            assert int(got["%s.%s" % (name, field)]) == getattr(cls, field).offset, (name, field)
    for name, value in consts.items():
        assert int(got[name]) == value, name


def test_every_entry_point_is_mapped_in_integration_md():
    """INTEGRATION.md must name the reference interface every exported entry replaces (or say that there is none)."""
    import re

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "nfsp_b200.h")).read()
    doc = open(os.path.join(root, "INTEGRATION.md")).read()
    missing = sorted(s for s in set(re.findall(r"\b(nfsp_[a-z0-9_]+)\s*\(", hdr)) if s not in doc)
    assert not missing, missing
