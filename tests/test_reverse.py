"""--reverse (main.cpp:253,285-286): long reads from the strand opposite to the short reads.  Every read is
reverse-complemented before anything else; a corrected read comes back reverse-complemented again (input orientation),
every other read comes back as the reverse complement of its input (SURVEY Q24).  CPU tests pin the command line and the
oracle's own reverse path; GPU tests hold every entry point of the library to that oracle."""
import os
import subprocess
import threading

import numpy as np
import pytest

from conftest import have_gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "tiny_case.npz")
SHARED = ["lookups_seg", "lookups_deg", "lookups_walk", "steps_inner", "steps_border", "frontier_sum", "cells_nw",
          "cells_lcs", "cells_ovl", "cells_xdrop", "gaps", "gaps_bridged", "gap_attempts", "borders",
          "borders_corrected", "ev_gardening", "ev_bridge", "ev_edge", "ev_cycle", "bases_out"]

# Dna5 conversion + SeqAn reverseComplement: ACGT in either case -> complement, anything else -> N
_COMP = np.full(256, ord("N"), dtype=np.uint8)
for _a, _b in zip(b"ACGTacgt", b"TGCATGCA"):
    _COMP[_a] = _b


def rc(s: bytes) -> bytes:
    return _COMP[np.frombuffer(s, dtype=np.uint8)[::-1]].tobytes()


def rc_batch(reads: np.ndarray, off: np.ndarray) -> np.ndarray:
    """Every read of a concatenated batch reverse-complemented in place (offsets unchanged, off[0] == 0)."""
    o = off.astype(np.int64)
    idx = np.repeat(o[:-1] + o[1:] - 1, np.diff(o)) - np.arange(o[-1])
    return _COMP[reads[idx]]


def _records(g):
    """The c3 reads with the drop-in test's `tiny` and `junk` records, plus two that are not their own reverse
    complement: a short one with lower case and N, and an unsolvable long one."""
    reads, off = g["c3_reads"], g["c3_off"]
    recs = []
    for r in range(len(off) - 1):
        recs.append((b"read_%d" % r, reads[int(off[r]):int(off[r + 1])].tobytes()))
        if r == 2:
            recs += [(b"tiny", b"ACGTACGT"), (b"junk", b"ACGT" * 60), (b"short_rc", b"ggcaNtacc"),
                     (b"junk_rc", b"AACGTTTGCCA" * 20)]
    return recs


def _write_inputs(tmp_path, g, recs):
    import torch
    from talc_b200 import synth
    k = int(g["c3_k"][0])
    synth.write_dump(str(tmp_path / "sr.dump"), torch.from_numpy(g["c3_keys"].astype(np.int64)),
                     torch.from_numpy(g["c3_counts"].astype(np.int64)), k)
    synth.write_dump(str(tmp_path / "j.dump"), torch.from_numpy(g["c3_jkeys"].astype(np.int64)),
                     torch.from_numpy(g["c3_jcounts"].astype(np.int64)), k)
    with open(tmp_path / "reads.fa", "wb") as f, open(tmp_path / "reads.fq", "wb") as q, \
            open(tmp_path / "rc.fa", "wb") as fr:
        for name, s in recs:
            f.write(b">" + name + b"\n" + s + b"\n")
            q.write(b"@" + name + b"\n" + s + b"\n+\n" + b"I" * len(s) + b"\n")
            fr.write(b">" + name + b"\n" + rc(s) + b"\n")
    return k, ["--SRCounts", str(tmp_path / "sr.dump"), "--junctions", str(tmp_path / "j.dump"), "-k", str(k)]


def _read_fasta(path):
    recs, name, seq = [], None, []
    for line in open(path, "rb").read().split(b"\n"):
        if line.startswith(b">"):
            if name is not None:
                recs.append((name, b"".join(seq)))
            name, seq = line[1:], []
        elif line:
            seq.append(line)
    if name is not None:
        recs.append((name, b"".join(seq)))
    return recs


def _concat(recs):
    off = np.zeros(len(recs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(s) for _, s in recs])
    return np.frombuffer(b"".join(s for _, s in recs), dtype=np.uint8).copy(), off


# ---------------------------------------------------------------------------------------------------- CPU
def test_cli_accepts_reverse(tmp_path):
    """-rev / --reverse parses (the reference's option) and leaves .config.txt as it is: the reference does not echo it."""
    from talc_b200 import build
    cli = build.build_cli()
    run = lambda *a: subprocess.call([cli] + list(a), stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, cwd=tmp_path)
    assert run("missing.fa", "--SRCounts", "d.dump", "-k", "21", "-o", "x") == 0
    plain = open(tmp_path / "x.config.txt").read()
    for flag in ("--reverse", "-rev"):
        os.remove(tmp_path / "x.config.txt")
        assert run("missing.fa", "--SRCounts", "d.dump", "-k", "21", flag, "-o", "x") == 0, flag
        assert open(tmp_path / "x.config.txt").read() == plain, flag
        assert open(tmp_path / "x.stats_basics.txt").read().startswith("read_name\traw_length\t")


def test_oracle_reverse_is_strand_consistent(tmp_path):
    """The oracle's --reverse path, which the GPU tests below compare against: --reverse on the reverse-complemented
    reads gives, per record, the reverse complement of the forward output when the read was corrected and the forward
    output (the normalised original read) otherwise; the failed-read logs are identical."""
    from oracle import pyoracle as po
    g = np.load(GOLD)
    recs = _records(g)
    k, common = _write_inputs(tmp_path, g, recs)
    ora = lambda reads, *a: subprocess.call([po.BIN, str(tmp_path / reads)] + common + ["-t", "1", "--oracle-table", "hash"]
                                            + list(a), cwd=tmp_path, stdout=subprocess.DEVNULL)
    assert ora("reads.fa", "-o", "fwd") == 0
    assert ora("rc.fa", "-o", "rev", "--reverse") == 0
    reads, off = _concat(recs)
    ot = po.OracleTable(po.make_params(k=k)).build_packed(g["c3_keys"], g["c3_counts"].astype(np.int64), g["c3_jkeys"],
                                                          g["c3_jcounts"].astype(np.int64))
    _, _, status, _, _ = ot.correct(reads, off, threads=2)
    fwd, rev = _read_fasta(tmp_path / "fwd.fa"), _read_fasta(tmp_path / "rev.fa")
    assert [n for n, _ in fwd] == [n for n, _ in rev] == [n for n, _ in recs]
    assert (status == 0).sum() > 0 and (status != 0).sum() >= 3
    for r, (name, s) in enumerate(recs):
        if status[r] == 0:
            assert rev[r][1] == rc(fwd[r][1]), name
        else:
            assert rev[r][1] == fwd[r][1] == rc(rc(s)), name
    assert open(tmp_path / "fwd.log", "rb").read() == open(tmp_path / "rev.log", "rb").read()
    assert b"junk_rc" in open(tmp_path / "rev.log", "rb").read()


# ---------------------------------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    if not have_gpu():
        pytest.fail("GPU tests selected but no CUDA device is visible")
    from talc_b200 import api as _api
    return _api


def _ctx(api, case, reverse=True):
    t = api.Talc(api.default_params(case.cfg.k))
    t.load_packed(case.keys, case.counts, case.jkeys, case.jcounts)
    t.set_reverse(reverse)
    return t


_expected = {}


def _expect(case):
    """What --reverse gives for case.reads: the oracle on the reverse-complemented reads, corrected reads flipped back."""
    key = id(case)
    if key not in _expected:
        n = len(case.off) - 1
        o_out, o_off, o_st, o_ctr, _ = case.otable.correct(rc_batch(case.reads, case.off), case.off, threads=8)
        parts = []
        for r in range(n):
            s = o_out[int(o_off[r]):int(o_off[r + 1])].tobytes()
            parts.append(rc(s) if o_st[r] == 0 else s)
        _expected[key] = (parts, o_off, o_st, o_ctr)
    return _expected[key]


def _assert_reverse(case, out, off, st, ctr=None):
    parts, o_off, o_st, o_ctr = _expect(case)
    assert np.array_equal(st, o_st), "per-read status differs"
    assert np.array_equal(off, o_off), "output offsets differ"
    bad = [r for r in range(len(parts)) if out[int(off[r]):int(off[r + 1])].tobytes() != parts[r]]
    assert not bad, "reverse-mode bytes differ for reads %s" % bad[:10]
    if ctr is not None:
        diff = {k: (o_ctr[k], ctr[k]) for k in SHARED if o_ctr[k] != ctr[k]}
        assert not diff, "algorithmic counters differ: %s" % diff


def _assert_antisense(case, out, off, st, ctr=None):
    """Reverse mode on RC(case.reads) against the oracle's forward run on case.reads: corrected reads are the reverse
    complement of the oracle's, every other read is the (normalised) original, status and counters are the same."""
    assert np.array_equal(st, case.o_status), "per-read status differs"
    assert np.array_equal(off, case.o_off), "output offsets differ"
    bad = [r for r in range(len(case.off) - 1) if out[int(off[r]):int(off[r + 1])].tobytes() !=
           (rc(case.oracle_read(r)) if case.o_status[r] == 0 else case.oracle_read(r))]
    assert not bad, "reverse-mode bytes differ for reads %s" % bad[:10]
    if ctr is not None:
        diff = {k: (case.o_ctr[k], ctr[k]) for k in SHARED if case.o_ctr[k] != ctr[k]}
        assert not diff, "algorithmic counters differ: %s" % diff


@gpu
@pytest.mark.parametrize("name", ["c1", "c3", "c5"])
def test_reverse_matches_oracle(api, name, request):
    case = request.getfixturevalue("case_" + name)
    t = _ctx(api, case)
    out, off, st, ctr = t.correct(case.reads, case.off)
    _assert_reverse(case, out, off, st, ctr)


@gpu
@pytest.mark.parametrize("name", ["c1", "c3", "c5"])
def test_strand_invariance(api, name, request):
    """Reverse mode on RC(reads) does the work forward mode does on reads: same status and counters, failed reads
    byte-identical (the normalised original), corrected reads reverse complements of each other."""
    case = request.getfixturevalue("case_" + name)
    t = _ctx(api, case, reverse=False)
    f_out, f_off, f_st, f_ctr = t.correct(case.reads, case.off)
    t.set_reverse(True)
    r_out, r_off, r_st, r_ctr = t.correct(rc_batch(case.reads, case.off), case.off)
    assert np.array_equal(f_st, r_st) and np.array_equal(f_off, r_off)
    assert {k: f_ctr[k] for k in SHARED} == {k: r_ctr[k] for k in SHARED}
    assert (f_st == 0).any()
    for r in range(len(case.off) - 1):
        a = f_out[int(f_off[r]):int(f_off[r + 1])].tobytes()
        b = r_out[int(r_off[r]):int(r_off[r + 1])].tobytes()
        assert (b == rc(a)) if f_st[r] == 0 else (b == a), r


@gpu
def test_reverse_every_entry_point_and_shape(api, case_c1):
    """Host call, device call (the caller's buffer untouched), the stream with uneven batches, a lane from a second
    thread, the split execution shape and the second tier give the same bytes.  The input is the antisense batch
    RC(reads), so that most reads are corrected and come back through the reversed gather."""
    import torch
    case = case_c1
    n = len(case.off) - 1
    rx = rc_batch(case.reads, case.off)
    t = _ctx(api, case)
    out, off, st, ctr = t.correct(rx, case.off)
    _assert_antisense(case, out, off, st, ctr)
    # device-resident buffers
    d_reads = torch.from_numpy(rx.copy()).cuda()
    d_off = torch.from_numpy(case.off.astype(np.int64)).cuda()
    d_out = torch.empty(2 * len(rx) + 64 * n + 4096, dtype=torch.uint8, device="cuda")
    d_ooff = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    d_st = torch.zeros(n, dtype=torch.uint8, device="cuda")
    dctr = t.correct_device(d_reads, d_off, len(rx), d_out, d_ooff, d_st)
    assert np.array_equal(d_reads.cpu().numpy(), rx), "the caller's device buffer was written"
    doff = d_ooff.cpu().numpy().astype(np.uint64)
    _assert_antisense(case, d_out[: int(doff[-1])].cpu().numpy(), doff, d_st.cpu().numpy(), dctr)
    # the stream: uneven batches, one of them empty; read_stats describe the reverse-complemented reads
    cuts = [0, 1, 1, 40, 41, 130, n]
    s = t.stream(read_stats=True)
    outs, sts, stats = [], [], []
    for a, b in zip(cuts, cuts[1:]):
        s.submit(rx[int(case.off[a]):int(case.off[b])], case.off[a:b + 1] - case.off[a])
        o, f, x, rs, _ = s.next()
        outs.append(o)
        sts.append(x)
        stats.append(rs)
    s.close()
    assert np.array_equal(np.concatenate(outs), out) and np.array_equal(np.concatenate(sts), st)
    assert np.array_equal(np.concatenate(stats), case.otable.read_stats(case.reads, case.off, threads=4))
    # a lane follows its parent's strand and refuses to set its own
    lane = t.create_lane()
    with pytest.raises(api.TalcError):
        lane.set_reverse(False)
    h = n // 2
    res = [None, None]

    def run(i, c, a, b):
        res[i] = c.correct(rx[int(case.off[a]):int(case.off[b])], case.off[a:b + 1] - case.off[a])

    th = [threading.Thread(target=run, args=(0, t, 0, h)), threading.Thread(target=run, args=(1, lane, h, n))]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert np.array_equal(np.concatenate([res[0][0], res[1][0]]), out)
    assert np.array_equal(np.concatenate([res[0][2], res[1][2]]), st)
    lane.close()
    # split execution shape, then the second tier
    t.set_exec(1)
    o2, f2, s2, c2 = t.correct(rx, case.off)
    assert c2["rounds"] > 0
    _assert_antisense(case, o2, f2, s2, c2)
    t2 = _ctx(api, case)
    t2.set_scratch(tier1_bytes=6 * 1024)
    o3, f3, s3, c3 = t2.correct(rx, case.off)
    assert c3["reads_second_tier"] > 0
    _assert_antisense(case, o3, f3, s3, c3)
    t.close()


@gpu
def test_reverse_toggles_back(api, case_c3):
    case = case_c3
    t = _ctx(api, case)
    _assert_reverse(case, *t.correct(case.reads, case.off))
    t.set_reverse(False)
    out, off, st, ctr = t.correct(case.reads, case.off)
    assert np.array_equal(st, case.o_status) and np.array_equal(off, case.o_off) and np.array_equal(out, case.o_out)
    assert {k: ctr[k] for k in SHARED} == {k: case.o_ctr[k] for k in SHARED}


@gpu
def test_reverse_coverage(api, case_c1):
    """Read::reCoverage sees the reverse-complemented read."""
    case = case_c1
    t = _ctx(api, case)
    cov = t.coverage(case.reads, case.off)
    pos = 0
    for r in range(40):
        ocnt, _ = case.otable.coverage(rc(case.read(r)))
        assert np.array_equal(cov[pos:pos + len(ocnt)], ocnt), r
        pos += len(ocnt)


@gpu
def test_cli_reverse_is_a_drop_in(api, tmp_path):
    """`talc --reverse` writes the oracle's --reverse files (.fa, .log, stats header, .config.txt), whatever the
    batching and for FASTQ input; --readStats rows describe the reverse-complemented reads."""
    from oracle import pyoracle as po
    from talc_b200 import build
    g = np.load(GOLD)
    recs = _records(g)
    k, common = _write_inputs(tmp_path, g, recs)
    cli = build.build_cli()
    run = lambda exe, reads, *a: subprocess.call([exe, str(tmp_path / reads)] + common + list(a), cwd=tmp_path,
                                                 stdout=subprocess.DEVNULL)
    assert run(cli, "reads.fa", "-o", "gpu", "--reverse") == 0
    assert run(po.BIN, "reads.fa", "-o", "cpu", "--reverse", "-t", "1", "--oracle-table", "hash") == 0
    for ext in (".fa", ".log", ".stats_basics.txt"):
        assert open(tmp_path / ("gpu" + ext), "rb").read() == open(tmp_path / ("cpu" + ext), "rb").read(), ext
    assert open(tmp_path / "gpu.config.txt").read().replace("gpu", "X") == open(tmp_path / "cpu.config.txt").read().replace("cpu", "X")
    assert b"junk_rc" in open(tmp_path / "gpu.log", "rb").read()
    assert run(cli, "reads.fa", "-o", "many", "--reverse", "--batch-reads", "7", "-t", "3") == 0
    assert run(cli, "reads.fq", "-o", "fq", "-rev", "--batch-reads", "5") == 0
    assert run(cli, "reads.fa", "-o", "stats", "--reverse", "--batch-reads", "11", "--readStats") == 0
    for other in ("many", "fq", "stats"):
        for ext in (".fa", ".log"):
            assert open(tmp_path / (other + ext), "rb").read() == open(tmp_path / ("gpu" + ext), "rb").read(), (other, ext)
    rows = open(tmp_path / "stats.stats_basics.txt").read().split("\n")
    assert rows[0].startswith("read_name\traw_length") and rows[1] == ""
    by_id = {r.split("\t")[0]: [int(x) for x in r.split("\t")[1:]] for r in rows[2:]}
    reads, off = _concat(recs)
    rcr = rc_batch(reads, off)
    ot = po.OracleTable(po.make_params(k=k)).build_packed(g["c3_keys"], g["c3_counts"].astype(np.int64), g["c3_jkeys"],
                                                          g["c3_jcounts"].astype(np.int64))
    st = ot.read_stats(rcr, off, threads=2)
    _, o_off, o_st, _, _ = ot.correct(rcr, off, threads=2)
    assert "tiny" not in by_id and "short_rc" not in by_id
    for r, (name, s) in enumerate(recs):
        if len(s) <= k:
            continue
        corr = int(o_off[r + 1] - o_off[r]) if o_st[r] == 0 else 0
        assert by_id[name.decode()] == [len(s), int(st[r][0]), int(st[r][1]), corr], name


@gpu
def test_cli_reverse_two_gpus_equals_one(api, tmp_path):
    import torch
    from talc_b200 import build, synth
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    cfg = synth.baseline_config(1, 0.05)
    cfg.n_reads = 600
    w = synth.make_workload(cfg)
    synth.write_dump(str(tmp_path / "sr.dump"), w.keys, w.counts, cfg.k)
    reads = rc_batch(w.reads.numpy(), w.read_off.numpy().astype(np.uint64))  # antisense reads: mostly corrected
    synth.write_fasta(str(tmp_path / "reads.fa"), torch.from_numpy(reads), w.read_off, width=80)
    cli = build.build_cli()
    args = [str(tmp_path / "reads.fa"), "--SRCounts", str(tmp_path / "sr.dump"), "-k", str(cfg.k), "--reverse"]
    run = lambda *a: subprocess.call([cli] + args + list(a), cwd=tmp_path, stdout=subprocess.DEVNULL)
    assert run("-o", "one", "--gpus", "1") == 0
    assert run("-o", "two", "--gpus", "2", "--batch-reads", "100") == 0
    assert run("-o", "peer", "--gpus", "2", "--batch-reads", "77", "--replicate", "peer") == 0
    for ext in (".fa", ".log"):
        a = open(tmp_path / ("one" + ext), "rb").read() if os.path.exists(tmp_path / ("one" + ext)) else b""
        for other in ("two", "peer"):
            b = open(tmp_path / (other + ext), "rb").read() if os.path.exists(tmp_path / (other + ext)) else b""
            assert a == b, (other, ext)
    assert len(open(tmp_path / "one.fa", "rb").read()) > int(w.read_off[-1])
