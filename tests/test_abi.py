"""The C-ABI shared library loads on a machine without a GPU, exports every symbol include/talc_b200.h declares,
and refuses to work without CUDA (no CPU fallback).  The `talc` command line exists and parses like the reference."""
import ctypes
import os
import re
import subprocess
import sys

from conftest import ROOT


def _declared_symbols():
    txt = open(os.path.join(ROOT, "include", "talc_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(talc_[a-z_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    from talc_b200 import build
    lib = ctypes.CDLL(build.build_library())
    names = _declared_symbols()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), "missing export: " + n


def test_no_cpu_fallback():
    """Run with the devices hidden (child process), so that it holds on a machine with a GPU as well."""
    code = ("import sys; sys.path.insert(0, %r)\nfrom talc_b200 import api\n"
            "try:\n    api.Talc(api.default_params(21))\n    print('CREATED')\n"
            "except api.TalcError as e:\n    print('REFUSED', e)\n") % ROOT
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True).stdout
    assert "REFUSED" in out and "no CPU path" in out


def test_product_does_not_reference_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/."""
    pkg = os.path.join(ROOT, "talc_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".hpp", ".cpp", ".h")):
                src = open(os.path.join(dp, f), errors="ignore").read()
                assert "pyoracle" not in src and "talc_oracle" not in src and "oracle/" not in src, f


def test_cli_parses_like_the_reference(tmp_path):
    from talc_b200 import build
    cli = build.build_cli()
    run = lambda *a: subprocess.call([cli] + list(a), stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, cwd=tmp_path)
    assert run("--help") == 0                                              # main.cpp:199: non-error parse result -> 0
    assert run("reads.fa", "--SRCounts", "d.dump") == 1                    # -k is required
    assert run("reads.fa", "--SRCounts", "d.dump", "-k", "31") == 1        # main.cpp:115: k <= 30
    assert run("reads.fa", "--SRCounts", "d.dump", "-k", "17") == 1        # main.cpp:116: k >= 18
    assert run("reads.fa", "-k", "21") == 1                                # --SRCounts is required
    assert run("reads.fa", "--SRCounts", "d.dump", "-k", "21", "--MIN_COUNT", "1") == 1
    # unreadable input: the files of Settings/Read are written, then main falls off its end with 0 (main.cpp:323)
    assert run("missing.fa", "--SRCounts", "d.dump", "-k", "21", "-o", "x") == 0
    assert os.path.exists(tmp_path / "x.config.txt") and os.path.exists(tmp_path / "x.stats_basics.txt")
    cfg = open(tmp_path / "x.config.txt").read().splitlines()
    assert cfg[2] == "INPUT=missing.fa" and cfg[6] == "KmerSize=21" and cfg[7] == "Junction mode activated? 0"
