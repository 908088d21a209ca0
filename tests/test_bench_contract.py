"""bench.py without a GPU: the pieces of its output contract that are host logic -- the committed ncu capture it
reads for `roofline.traffic` / `roofline.issue`, the peak it divides by, exactly one JSON line on stdout whatever
the libraries underneath print, and a loud failure (no numbers) when there is no CUDA device."""
import importlib.util
import json
import os
import subprocess
import sys

from conftest import ROOT


def _bench():
    spec = importlib.util.spec_from_file_location("talc_bench", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_committed_capture_is_readable():
    b = _bench()
    t, n = b.measured_traffic(), b.measured_instructions()
    assert t is not None and 30e9 < t < 80e9            # DRAM bytes of one correct_kernel launch of the bench workload
    assert n is not None and 1e11 < n < 5e11            # its warp-instructions
    assert os.path.exists(os.path.join(ROOT, b.TRAFFIC_SOURCE.split(" ")[0]))
    peak, src = b.peaks()
    assert 3000 < peak < 9000 and src


def test_one_json_line_on_stdout_whatever_else_is_printed(tmp_path):
    """_claim_stdout keeps a private duplicate of fd 1 for the JSON line and points fd 1 at stderr: a C library that
    prints to stdout (NCCL's version banner) cannot add lines."""
    code = ("import os, sys, ctypes; sys.path.insert(0, %r); import importlib.util as u;"
            "s = u.spec_from_file_location('b', %r); b = u.module_from_spec(s); s.loader.exec_module(b);"
            "b._claim_stdout(); print('python noise'); ctypes.CDLL(None).puts(b'C stdio noise'); ctypes.CDLL(None).fflush(None);"
            "os.write(1, b'raw fd noise\\n'); b.emit({'metric': 'm', 'value': 1.5})") % (ROOT, os.path.join(ROOT, "bench.py"))
    pr = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert pr.returncode == 0, pr.stderr
    lines = pr.stdout.splitlines()
    assert len(lines) == 1 and json.loads(lines[0]) == {"metric": "m", "value": 1.5}
    assert "python noise" in pr.stderr and "C stdio noise" in pr.stderr and "raw fd noise" in pr.stderr


def test_dump_outputs_writes_the_batch_as_float_arrays(tmp_path):
    """--dump-outputs: offsets, status and a digest of every read of the batch, the corrected bases of a fixed seeded
    sample of reads and the call's counters, as float32 / float64 .npy files; the same outputs give the same files,
    and one changed base anywhere changes the digests."""
    import numpy as np
    import torch
    b = _bench()
    rng = np.random.default_rng(1)
    n = 8000
    off = np.concatenate([[0], np.cumsum(rng.integers(0, 50, n))]).astype(np.int64)
    out = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), int(off[-1]) + 100)  # device buffers are larger than the batch
    st = rng.integers(0, 5, n).astype(np.uint8)
    ctr = {"lookups_walk": 12345678901, "reads": n, "ms_total": 1.5}
    for d in ("a", "b"):
        b.dump_outputs(str(tmp_path / d), torch.from_numpy(out), torch.from_numpy(off), torch.from_numpy(st), n, ctr)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["counter_lookups_walk.npy", "counter_reads.npy", "out_offsets.npy", "read_digests.npy",
                     "sample_bases.npy", "sample_reads.npy", "status.npy"]
    got = {}
    for f in files:
        x = np.load(tmp_path / "a" / f)
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, np.load(tmp_path / "b" / f)), f
        got[f[:-4]] = x
    assert np.array_equal(got["out_offsets"], off) and np.array_equal(got["status"], st)
    assert got["counter_lookups_walk"][0] == 12345678901 and got["counter_reads"][0] == n
    idx = got["sample_reads"].astype(np.int64)
    assert len(idx) == b.DUMP_SAMPLE_READS and (np.diff(idx) > 0).all() and idx[-1] < n
    assert np.array_equal(got["sample_bases"], np.concatenate([out[off[i]:off[i + 1]] for i in idx]))
    r = next(i for i in range(n) if i not in set(idx.tolist()) and off[i + 1] > off[i])  # a read outside the sample
    out[off[r]] ^= 1
    dig = b.read_digests(out, off, n)
    assert len(dig) == n and np.nonzero(dig != got["read_digests"])[0].tolist() == [r]


def test_no_numbers_without_a_gpu():
    # the devices are hidden, so that this holds on a machine with a GPU as well
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True,
                        text=True, cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert pr.returncode != 0 and pr.stdout.strip() == "" and "no CPU fallback" in pr.stderr
