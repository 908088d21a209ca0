"""--strand auto: each long read corrected on the strand where it finds more of the (single-strand) k-mer table, every
read returned in its input orientation.  found_fwd / found_rc = windows of the read / of its Dna5 reverse complement
whose k-mer is in the table; strand 1 iff found_rc > found_fwd.  CPU tests pin the command line, the host emulation of
the device helpers (tests/hostemu/strand_emu.cpp) against numpy and the oracle's table look-ups, and the expected
command-line output built from the oracle's forward run on the oriented reads; GPU tests hold every entry point of the
library to the oracle on the oriented batch (each strand-1 read reverse-complemented)."""
import os
import subprocess
import threading

import numpy as np
import pytest

from conftest import Case, have_gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "tiny_case.npz")
SHARED = ["lookups_seg", "lookups_deg", "lookups_walk", "steps_inner", "steps_border", "frontier_sum", "cells_nw",
          "cells_lcs", "cells_ovl", "cells_xdrop", "gaps", "gaps_bridged", "gap_attempts", "borders",
          "borders_corrected", "ev_gardening", "ev_bridge", "ev_edge", "ev_cycle", "bases_out"]

# Dna5 conversion + SeqAn reverseComplement: ACGT in either case -> complement, anything else -> N
_COMP = np.full(256, ord("N"), dtype=np.uint8)
for _a, _b in zip(b"ACGTacgt", b"TGCATGCA"):
    _COMP[_a] = _b
# base code of the forward read (SeqAn char -> Dna5): ACGT and U either case, anything else N (4)
_CODE = np.full(256, 4, dtype=np.uint8)
for _a, _v in zip(b"ACGTUacgtu", [0, 1, 2, 3, 3] * 2):
    _CODE[_a] = _v


def rc(s: bytes) -> bytes:
    return _COMP[np.frombuffer(s, dtype=np.uint8)[::-1]].tobytes()


def _concat(seqs):
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(s) for s in seqs])
    return np.frombuffer(b"".join(seqs) + b"", dtype=np.uint8).copy(), off


def _split(reads, off):
    return [reads[int(off[r]):int(off[r + 1])].tobytes() for r in range(len(off) - 1)]


def _found(seq: bytes, k: int, table) -> int:
    """windows of seq without N whose packed k-mer is in the table (a sorted uint64 array)"""
    codes = _CODE[np.frombuffer(seq, dtype=np.uint8)]
    if len(codes) < k:
        return 0
    w = np.lib.stride_tricks.sliding_window_view(codes, k)
    ok = (w < 4).all(axis=1)
    shifts = (2 * np.arange(k - 1, -1, -1)).astype(np.uint64)
    keys = np.bitwise_or.reduce((w.astype(np.uint64) & np.uint64(3)) << shifts, axis=1)
    pos = np.minimum(np.searchsorted(table, keys), len(table) - 1)
    return int((ok & (table[pos] == keys)).sum())


def np_orient(seqs, k, table):
    """the decision rule in numpy: (strand, found_fwd, found_rc)"""
    ff = np.array([_found(s, k, table) for s in seqs], dtype=np.uint32)
    fr = np.array([_found(rc(s), k, table) for s in seqs], dtype=np.uint32)
    return (fr > ff).astype(np.uint8), ff, fr


def _table(keys, counts, min_count=2):
    return np.unique(np.asarray(keys, dtype=np.uint64)[np.asarray(counts) >= min_count])


def _mixed(seqs, seed=7):
    """a seeded half of the reads reverse-complemented"""
    flip = np.random.default_rng(seed).random(len(seqs)) < 0.5
    return [rc(s) if f else s for s, f in zip(seqs, flip)], flip


def _crafted(k, source: bytes):
    """short, exact-K, all-N, reverse palindromes, lower case, N and other bytes, on both strands"""
    a = source[:3 * k]
    pal = a[:k] + rc(a[:k])
    out = [b"", a[:k - 1], a[:k], rc(a[:k]), b"N" * (2 * k), pal, pal.lower(), b"ACGT" * k, a.lower(),
           a[:k] + b"N" + a[k + 1:], a[:5] + b"X" + a[6:], rc(a).lower(), rc(a)[:k + 3], a[:2 * k] + b"n" * 3 + a[2 * k:]]
    return out


# ---------------------------------------------------------------------------------------------------- CPU
def test_cli_parses_strand(tmp_path):
    """--strand forward|reverse|auto parse and leave .config.txt as it is; a bad value, a missing value and --reverse with
    another strand are PARSE_ERROR (exit 1)."""
    from talc_b200 import build
    exe = build.build_cli()
    run = lambda *a: subprocess.call([exe, "missing.fa", "--SRCounts", "d.dump", "-k", "21", "-o", "x"] + list(a),
                                     stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, cwd=tmp_path)
    assert run() == 0
    plain = open(tmp_path / "x.config.txt").read()
    for extra in (["--strand", "forward"], ["--strand", "reverse"], ["--strand", "auto"], ["--reverse", "--strand", "reverse"],
                  ["--strand", "reverse", "-rev"]):
        os.remove(tmp_path / "x.config.txt")
        assert run(*extra) == 0, extra
        assert open(tmp_path / "x.config.txt").read() == plain, extra
    for extra in (["--strand", "both"], ["--strand", "Auto"], ["--strand"], ["--reverse", "--strand", "auto"],
                  ["--strand", "auto", "-rev"], ["--strand", "forward", "--reverse"]):
        assert run(*extra) == 1, extra
    out = subprocess.run([exe, "--help"], capture_output=True, text=True).stdout
    assert "--strand forward|reverse|auto" in out


def oracle_orient(otable, reads, off):
    """the decision rule from the oracle's own table look-ups: windows of each read / of its Dna5 reverse complement
    with a count (Read::reCoverage on either strand)"""
    seqs = _split(reads, off)
    ff = np.array([int((otable.coverage(s)[0] != 0).sum()) for s in seqs], dtype=np.uint32)
    fr = np.array([int((otable.coverage(rc(s))[0] != 0).sum()) for s in seqs], dtype=np.uint32)
    return (fr > ff).astype(np.uint8), ff, fr


@pytest.mark.parametrize("k", list(range(18, 32)))
def test_emu_orient_matches_numpy(k):
    """emu_orient_reads (the device's strand_roll_push / strand_decide compiled for the host) against numpy, for every K
    from 18 to 31: mutated sense and antisense reads with N, lower case, U and other bytes, plus the crafted reads."""
    import strand_emu
    rng = np.random.default_rng(100 + k)
    tx = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), 3000).tobytes()
    codes = _CODE[np.frombuffer(tx, dtype=np.uint8)]
    w = np.lib.stride_tricks.sliding_window_view(codes, k)
    shifts = (2 * np.arange(k - 1, -1, -1)).astype(np.uint64)
    keys = np.bitwise_or.reduce(w.astype(np.uint64) << shifts, axis=1)
    counts = rng.integers(1, 6, len(keys))  # count 1 is below MIN_COUNT: not in the table
    seqs = []
    for _ in range(120):
        a = int(rng.integers(0, len(tx) - 400))
        s = bytearray(tx[a:a + int(rng.integers(k - 2, 400))])
        for p in rng.integers(0, len(s), len(s) // 12):
            s[p] = rng.choice(np.frombuffer(b"ACGTNnacgtUuX.", dtype=np.uint8))
        seqs.append(rc(bytes(s)) if rng.random() < 0.5 else bytes(s))
    seqs += _crafted(k, tx[500:])
    reads, off = _concat(seqs)
    got = strand_emu.orient(k, keys, counts, reads, off)
    want = np_orient(seqs, k, _table(keys, counts))
    for g, w_, name in zip(got, want, ("strand", "found_fwd", "found_rc")):
        assert np.array_equal(g, w_), (k, name, np.nonzero(g != w_)[0][:10])
    assert want[0].sum() > 20 and (want[0] == 0).sum() > 20
    n0 = len(seqs) - len(_crafted(k, tx[500:]))
    for r in (n0, n0 + 1, n0 + 4, n0 + 5, n0 + 6):  # empty, len < K, all N, reverse palindromes: ties stay forward
        assert got[0][r] == 0 and got[1][r] == got[2][r], r


def test_emu_orient_on_flipped_c1(case_c1):
    """A seeded mix of flipped c1 reads: host emulation == numpy == the oracle's look-ups, and a flipped read swaps the
    counts."""
    import strand_emu
    case = case_c1
    k = case.cfg.k
    seqs = _split(case.reads, case.off)
    mixed, flip = _mixed(seqs)
    reads, off = _concat(mixed)
    got = strand_emu.orient(k, case.keys, case.counts, reads, off)
    want = np_orient(mixed, k, _table(case.keys, case.counts))
    ora = oracle_orient(case.otable, reads, off)
    for g, w_, o in zip(got, want, ora):
        assert np.array_equal(g, w_) and np.array_equal(g, o)
    plain = np_orient(seqs, k, _table(case.keys, case.counts))
    assert np.array_equal(np.where(flip, plain[2], plain[1]), got[1])
    assert np.array_equal(np.where(flip, plain[1], plain[2]), got[2])
    assert (got[0][flip] == 1).mean() > 0.9 and (got[0][~flip] == 0).mean() > 0.9


def _records(seed=11):
    """the c3 reads with a seeded half flipped, plus reads that are ties or fail on either strand"""
    g = np.load(GOLD)
    reads, off = g["c3_reads"], g["c3_off"]
    seqs, _ = _mixed(_split(reads, off), seed)
    recs = [(b"read_%d" % r, s) for r, s in enumerate(seqs)]
    recs[3:3] = [(b"tiny", b"ACGTACGT"), (b"junk", b"ACGT" * 60), (b"short_rc", b"ggcaNtacc"),
                 (b"junk_rc", b"AACGTTTGCCA" * 20), (b"pal", seqs[0][:30] + rc(seqs[0][:30]))]
    return g, recs


def _write_inputs(tmp_path, g, recs):
    import torch
    from talc_b200 import synth
    k = int(g["c3_k"][0])
    synth.write_dump(str(tmp_path / "sr.dump"), torch.from_numpy(g["c3_keys"].astype(np.int64)),
                     torch.from_numpy(g["c3_counts"].astype(np.int64)), k)
    synth.write_dump(str(tmp_path / "j.dump"), torch.from_numpy(g["c3_jkeys"].astype(np.int64)),
                     torch.from_numpy(g["c3_jcounts"].astype(np.int64)), k)
    with open(tmp_path / "reads.fa", "wb") as f, open(tmp_path / "reads.fq", "wb") as q:
        for name, s in recs:
            f.write(b">" + name + b"\n" + s + b"\n")
            q.write(b"@" + name + b"\n" + s + b"\n+\n" + b"I" * len(s) + b"\n")
    return k, ["--SRCounts", str(tmp_path / "sr.dump"), "--junctions", str(tmp_path / "j.dump"), "-k", str(k)]


def _write_fasta(path, recs):
    with open(path, "wb") as f:
        for name, s in recs:
            f.write(b">" + name + b"\n" + s + b"\n")


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


def _fasta_bytes(recs):
    """70-column FASTA, as the reference writes it (io.cpp:50-75)"""
    out = []
    for name, s in recs:
        out.append(b">" + name + b"\n" + (b"\n" if not s else b"".join(s[i:i + 70] + b"\n" for i in range(0, len(s), 70))))
    return b"".join(out)


def _oracle_auto(tmp_path, recs, common, k, g, prefix):
    """What `talc --strand auto -o prefix` must write, from the oracle's forward command line on the oriented reads
    (each strand-1 read reverse-complemented): prefix.fa with the strand-1 records flipped back, the failed-read log
    and stats header of that run, and prefix.strand.txt.  Returns the strands."""
    from oracle import pyoracle as po
    reads, off = _concat([s for _, s in recs])
    ot = po.OracleTable(po.make_params(k=k)).build_packed(g["c3_keys"], g["c3_counts"].astype(np.int64), g["c3_jkeys"],
                                                          g["c3_jcounts"].astype(np.int64))
    strand, _, _ = oracle_orient(ot, reads, off)
    _write_fasta(tmp_path / (prefix + ".oriented.fa"), [(n, rc(s) if st else s) for (n, s), st in zip(recs, strand)])
    assert subprocess.call([po.BIN, str(tmp_path / (prefix + ".oriented.fa"))] + common +
                           ["-t", "1", "--oracle-table", "hash", "-o", prefix], cwd=tmp_path, stdout=subprocess.DEVNULL) == 0
    fwd = _read_fasta(tmp_path / (prefix + ".fa"))
    with open(tmp_path / (prefix + ".fa"), "wb") as f:
        f.write(_fasta_bytes([(n, rc(s) if st else s) for (n, s), st in zip(fwd, strand)]))
    with open(tmp_path / (prefix + ".strand.txt"), "wb") as f:
        f.write(b"".join(n + (b"\t-\n" if st else b"\t+\n") for (n, _), st in zip(recs, strand)))
    return strand


def test_oracle_strand_auto_expectation(tmp_path):
    """The expectation the command-line test compares against: its strands are the decision rule, its '+' records are
    the oracle's forward output and its corrected '-' records the oracle's --reverse output; failed '-' records are the
    normalised input."""
    from oracle import pyoracle as po
    g, recs = _records()
    k, common = _write_inputs(tmp_path, g, recs)
    strand = _oracle_auto(tmp_path, recs, common, k, g, "auto")
    want, _, _ = np_orient([s for _, s in recs], k, _table(g["c3_keys"], g["c3_counts"]))
    assert np.array_equal(strand, want) and strand.sum() > 20 and (strand == 0).sum() > 20
    ora = lambda *a: subprocess.call([po.BIN, str(tmp_path / "reads.fa")] + common + ["-t", "1", "--oracle-table", "hash"]
                                     + list(a), cwd=tmp_path, stdout=subprocess.DEVNULL)
    assert ora("-o", "fwd") == 0 and ora("-o", "rev", "--reverse") == 0
    auto, fwd, rev = (_read_fasta(tmp_path / (p + ".fa")) for p in ("auto", "fwd", "rev"))
    assert [n for n, _ in auto] == [n for n, _ in fwd] == [n for n, _ in recs]
    assert open(tmp_path / "auto.fa", "rb").read() == _fasta_bytes(auto)
    failed = open(tmp_path / "auto.log", "rb").read()
    n_ok = 0
    for (name, a), (_, f), (_, r), (_, s), st in zip(auto, fwd, rev, recs, strand):
        if not st:
            assert a == f, name
        elif b"[Read: " + name + b" ]" in failed or len(s) <= k:
            assert a == rc(rc(s)), name
        else:
            assert a == r, name
            n_ok += 1
    assert n_ok > 20


# ---------------------------------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    if not have_gpu():
        pytest.fail("GPU tests selected but no CUDA device is visible")
    from talc_b200 import api as _api
    return _api


_k31 = {}


@pytest.fixture(scope="module")
def case_k31():
    if "c" not in _k31:
        _k31["c"] = Case(1, 0.02, 120, k=31)
    return _k31["c"]


def _ctx(api, case, mode="auto"):
    t = api.Talc(api.default_params(case.cfg.k))
    t.load_packed(case.keys, case.counts, case.jkeys, case.jcounts)
    t.set_strand(mode)
    return t


_mixes = {}


def _mix(case):
    """(mixed reads, offsets, strands the oracle chooses, expected output parts, offsets, status, counters)"""
    key = id(case)
    if key not in _mixes:
        seqs, _ = _mixed(_split(case.reads, case.off))
        reads, off = _concat(seqs)
        strand, ff, fr = oracle_orient(case.otable, reads, off)
        oriented, _ = _concat([rc(s) if st else s for s, st in zip(seqs, strand)])
        o_out, o_off, o_st, o_ctr, _ = case.otable.correct(oriented, off, threads=8)
        parts = [rc(x) if st else x for x, st in zip(_split(o_out, o_off), strand)]
        _mixes[key] = dict(reads=reads, off=off, strand=strand, ff=ff, fr=fr, oriented=oriented, parts=parts, o_off=o_off,
                           o_st=o_st, o_ctr=o_ctr)
    return _mixes[key]


def _assert_auto(case, out, off, st, ctr=None):
    m = _mix(case)
    assert np.array_equal(st, m["o_st"]), "per-read status differs"
    assert np.array_equal(off, m["o_off"]), "output offsets differ"
    bad = [r for r in range(len(m["parts"])) if out[int(off[r]):int(off[r + 1])].tobytes() != m["parts"][r]]
    assert not bad, "auto-mode bytes differ for reads %s" % bad[:10]
    if ctr is not None:
        diff = {k: (m["o_ctr"][k], ctr[k]) for k in SHARED if m["o_ctr"][k] != ctr[k]}
        assert not diff, "algorithmic counters differ: %s" % diff


@gpu
@pytest.mark.parametrize("name", ["c1", "c3", "c5", "k31"])
def test_orient_matches_oracle(api, name, request):
    """talc_orient_batch == the oracle's per-read found_fwd, found_rc and strand, on the mixed batch and the crafted
    reads; in forward mode too (it does not depend on the context's mode)."""
    case = request.getfixturevalue("case_" + name)
    seqs, _ = _mixed(_split(case.reads, case.off))
    seqs += _crafted(case.cfg.k, case.read(0) + case.read(1) + case.read(2))
    reads, off = _concat(seqs)
    want = oracle_orient(case.otable, reads, off)
    assert want[0].sum() > 10 and (want[0] == 0).sum() > 10
    for mode in ("forward", "auto"):
        t = _ctx(api, case, mode)
        got = t.orient(reads, off)
        for g, w, what in zip(got, want, ("strand", "found_fwd", "found_rc")):
            assert np.array_equal(g, w), (mode, what, np.nonzero(g != w)[0][:10])
        t.close()


@gpu
@pytest.mark.parametrize("name", ["c1", "c3", "c5"])
def test_auto_matches_oracle(api, name, request):
    case = request.getfixturevalue("case_" + name)
    m = _mix(case)
    t = _ctx(api, case)
    out, off, st, ctr = t.correct(m["reads"], m["off"])
    _assert_auto(case, out, off, st, ctr)
    assert np.array_equal(t.last_strands(len(st)), m["strand"])
    assert (st[m["strand"] == 1] == 0).mean() > 0.5  # the antisense reads are corrected


@gpu
@pytest.mark.parametrize("name", ["c1", "c3", "c5"])
def test_auto_strand_invariance(api, name, request):
    """Auto mode on X and on mixed(X) do the same work: a read that is not a tie is corrected on the same strand, so
    it comes back as the reverse complement of its other orientation's output."""
    case = request.getfixturevalue("case_" + name)
    m = _mix(case)
    t = _ctx(api, case)
    a_out, a_off, a_st, a_ctr = t.correct(case.reads, case.off)
    b_out, b_off, b_st, b_ctr = t.correct(m["reads"], m["off"])
    seqs = _split(case.reads, case.off)
    flipped = np.array([mx != s for mx, s in zip(_split(m["reads"], m["off"]), seqs)])
    ties = m["ff"] == m["fr"]
    assert np.array_equal(a_st[~ties], b_st[~ties])
    assert np.array_equal(np.diff(a_off)[~ties], np.diff(b_off)[~ties])
    if not (ties & (m["ff"] > 0)).any():  # a tie with hits is corrected on the strand it is given: other work
        assert np.array_equal(a_st, b_st) and np.array_equal(a_off, b_off)
        assert {k: a_ctr[k] for k in SHARED} == {k: b_ctr[k] for k in SHARED}
    for r in np.nonzero(~ties)[0]:
        a = a_out[int(a_off[r]):int(a_off[r + 1])].tobytes()
        b = b_out[int(b_off[r]):int(b_off[r + 1])].tobytes()
        assert b == (rc(a) if flipped[r] else a), r


@gpu
def test_auto_every_entry_point_and_shape(api, case_c1):
    """Host call, device call (the caller's buffer untouched, strands to a device buffer), the stream with uneven and
    empty batches (strands and read_stats), a lane from a second thread, the split execution shape and the second tier
    give the same bytes and strands."""
    import torch
    case = case_c1
    m = _mix(case)
    rx, roff, strand = m["reads"], m["off"], m["strand"]
    n = len(roff) - 1
    t = _ctx(api, case)
    out, off, st, ctr = t.correct(rx, roff)
    _assert_auto(case, out, off, st, ctr)
    # device-resident buffers
    d_reads = torch.from_numpy(rx.copy()).cuda()
    d_off = torch.from_numpy(roff.astype(np.int64)).cuda()
    d_out = torch.empty(2 * len(rx) + 64 * n + 4096, dtype=torch.uint8, device="cuda")
    d_ooff = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    d_st = torch.zeros(n, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()  # the library's streams do not wait for torch's
    dctr = t.correct_device(d_reads, d_off, len(rx), d_out, d_ooff, d_st)
    assert np.array_equal(d_reads.cpu().numpy(), rx), "the caller's device buffer was written"
    doff = d_ooff.cpu().numpy().astype(np.uint64)
    _assert_auto(case, d_out[: int(doff[-1])].cpu().numpy(), doff, d_st.cpu().numpy(), dctr)
    d_strand = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    assert np.array_equal(t.last_strands(n, out=d_strand).cpu().numpy(), strand)
    assert np.array_equal(t.last_strands(5), strand[:5])
    with pytest.raises(api.TalcError):
        t.last_strands(n + 1)
    # the stream: uneven batches, one of them empty; read_stats describe the oriented reads
    cuts = [0, 1, 1, 40, 41, 130, n]
    s = t.stream(read_stats=True)
    outs, sts, stats, strs = [], [], [], []
    for a, b in zip(cuts, cuts[1:]):
        s.submit(rx[int(roff[a]):int(roff[b])], roff[a:b + 1] - roff[a])
        o, f, x, rs, _ = s.next()
        outs.append(o)
        sts.append(x)
        stats.append(rs)
        strs.append(s.strands())
        assert strs[-1] is not None and len(strs[-1]) == b - a
    s.close()
    assert np.array_equal(np.concatenate(outs), out) and np.array_equal(np.concatenate(sts), st)
    assert np.array_equal(np.concatenate(strs), strand)
    assert np.array_equal(np.concatenate(stats), case.otable.read_stats(m["oriented"], roff, threads=4))
    # a lane follows its parent's mode and refuses to set its own
    lane = t.create_lane()
    with pytest.raises(api.TalcError):
        lane.set_strand("forward")
    h = n // 2
    res = [None, None]

    def run(i, c, a, b):
        res[i] = c.correct(rx[int(roff[a]):int(roff[b])], roff[a:b + 1] - roff[a]) + (c.last_strands(b - a),)

    th = [threading.Thread(target=run, args=(0, t, 0, h)), threading.Thread(target=run, args=(1, lane, h, n))]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert np.array_equal(np.concatenate([res[0][0], res[1][0]]), out)
    assert np.array_equal(np.concatenate([res[0][2], res[1][2]]), st)
    assert np.array_equal(np.concatenate([res[0][4], res[1][4]]), strand)
    lane.close()
    # split execution shape, then the second tier
    t.set_exec(1)
    o2, f2, s2, c2 = t.correct(rx, roff)
    assert c2["rounds"] > 0
    _assert_auto(case, o2, f2, s2, c2)
    t2 = _ctx(api, case)
    t2.set_scratch(tier1_bytes=6 * 1024)
    o3, f3, s3, c3 = t2.correct(rx, roff)
    assert c3["reads_second_tier"] > 0
    _assert_auto(case, o3, f3, s3, c3)
    assert np.array_equal(t2.last_strands(n), strand)
    t.close()
    t2.close()


@gpu
def test_auto_toggles(api, case_c3):
    """auto -> forward reproduces the forward oracle exactly, auto -> reverse the reverse expectation; strands of a
    batch corrected outside auto mode are all 0, and the stream reports none."""
    case = case_c3
    m = _mix(case)
    t = _ctx(api, case)
    _assert_auto(case, *t.correct(m["reads"], m["off"]))
    t.set_strand("forward")
    out, off, st, ctr = t.correct(case.reads, case.off)
    assert np.array_equal(st, case.o_status) and np.array_equal(off, case.o_off) and np.array_equal(out, case.o_out)
    assert {k: ctr[k] for k in SHARED} == {k: case.o_ctr[k] for k in SHARED}
    assert not t.last_strands(len(st)).any()
    t.set_strand("auto")
    t.correct(m["reads"], m["off"])
    t.set_strand("reverse")
    seqs = _split(case.reads, case.off)
    rcb, _ = _concat([rc(s) for s in seqs])
    o_out, o_off, o_st, o_ctr, _ = case.otable.correct(rcb, case.off, threads=8)
    out, off, st, ctr = t.correct(case.reads, case.off)
    assert np.array_equal(st, o_st) and np.array_equal(off, o_off)
    want = [rc(x) if o_st[r] == 0 else x for r, x in enumerate(_split(o_out, o_off))]
    assert _split(out, off) == want
    assert {k: ctr[k] for k in SHARED} == {k: o_ctr[k] for k in SHARED}
    assert not t.last_strands(len(st)).any()
    s = t.stream()
    s.submit(case.reads, case.off)
    s.next()
    assert s.strands() is None
    s.close()
    with pytest.raises(api.TalcError):
        t.set_strand(3)


@gpu
def test_auto_coverage(api, case_c1):
    """talc_coverage_batch in auto mode: each read's coverage on its chosen strand."""
    case = case_c1
    m = _mix(case)
    t = _ctx(api, case)
    cov = t.coverage(m["reads"], m["off"])
    pos = 0
    for r, s in enumerate(_split(m["oriented"], m["off"])):
        ocnt, _ = case.otable.coverage(s)
        assert np.array_equal(cov[pos:pos + len(ocnt)], ocnt), r
        pos += len(ocnt)
    assert pos == len(cov)


@gpu
def test_cli_strand_auto_is_a_drop_in(api, tmp_path):
    """`talc --strand auto` writes what the oracle's forward run on the oriented reads defines (.fa with the strand-1
    records flipped back, .log, stats header, .strand.txt), whatever the batching and for FASTQ input; --readStats rows
    describe the oriented reads; --strand reverse is --reverse."""
    from oracle import pyoracle as po
    from talc_b200 import build
    g, recs = _records()
    k, common = _write_inputs(tmp_path, g, recs)
    cli = build.build_cli()
    run = lambda exe, reads, *a: subprocess.call([exe, str(tmp_path / reads)] + common + list(a), cwd=tmp_path,
                                                 stdout=subprocess.DEVNULL)
    assert run(cli, "reads.fa", "-o", "gpu", "--strand", "auto") == 0
    _oracle_auto(tmp_path, recs, common, k, g, "cpu")
    for ext in (".fa", ".log", ".strand.txt", ".stats_basics.txt"):
        assert open(tmp_path / ("gpu" + ext), "rb").read() == open(tmp_path / ("cpu" + ext), "rb").read(), ext
    assert open(tmp_path / "gpu.config.txt").read().replace("gpu", "X") == \
        open(tmp_path / "cpu.config.txt").read().replace(str(tmp_path / "cpu.oriented.fa"), str(tmp_path / "reads.fa")).replace("cpu", "X")
    assert b"\t-\n" in open(tmp_path / "gpu.strand.txt", "rb").read()
    assert run(cli, "reads.fa", "-o", "many", "--strand", "auto", "--batch-reads", "7", "-t", "3") == 0
    assert run(cli, "reads.fq", "-o", "fq", "--strand", "auto", "--batch-reads", "5") == 0
    assert run(cli, "reads.fa", "-o", "stats", "--strand", "auto", "--batch-reads", "11", "--readStats") == 0
    for other in ("many", "fq", "stats"):
        for ext in (".fa", ".log", ".strand.txt"):
            assert open(tmp_path / (other + ext), "rb").read() == open(tmp_path / ("gpu" + ext), "rb").read(), (other, ext)
    rows = open(tmp_path / "stats.stats_basics.txt").read().split("\n")
    assert rows[0].startswith("read_name\traw_length") and rows[1] == ""
    by_id = {r.split("\t")[0]: [int(x) for x in r.split("\t")[1:]] for r in rows[2:]}
    reads, off = _concat([s for _, s in recs])
    ot = po.OracleTable(po.make_params(k=k)).build_packed(g["c3_keys"], g["c3_counts"].astype(np.int64), g["c3_jkeys"],
                                                          g["c3_jcounts"].astype(np.int64))
    strand, _, _ = oracle_orient(ot, reads, off)
    oriented, _ = _concat([rc(s) if st else s for (_, s), st in zip(recs, strand)])
    stt = ot.read_stats(oriented, off, threads=2)
    _, o_off, o_st, _, _ = ot.correct(oriented, off, threads=2)
    for r, (name, s) in enumerate(recs):
        if len(s) <= k:
            assert name.decode() not in by_id
            continue
        corr = int(o_off[r + 1] - o_off[r]) if o_st[r] == 0 else 0
        assert by_id[name.decode()] == [len(s), int(stt[r][0]), int(stt[r][1]), corr], name
    assert run(cli, "reads.fa", "-o", "rev1", "--reverse") == 0
    assert run(cli, "reads.fa", "-o", "rev2", "--strand", "reverse") == 0
    assert open(tmp_path / "rev1.fa", "rb").read() == open(tmp_path / "rev2.fa", "rb").read()
    assert not os.path.exists(tmp_path / "rev2.strand.txt")


@gpu
def test_cli_strand_auto_two_gpus_equals_one(api, tmp_path):
    import torch
    from talc_b200 import build, synth
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    cfg = synth.baseline_config(1, 0.05)
    cfg.n_reads = 600
    w = synth.make_workload(cfg)
    synth.write_dump(str(tmp_path / "sr.dump"), w.keys, w.counts, cfg.k)
    seqs, _ = _mixed(_split(w.reads.numpy(), w.read_off.numpy().astype(np.uint64)))
    _write_fasta(tmp_path / "reads.fa", [(b"r%d" % i, s) for i, s in enumerate(seqs)])
    cli = build.build_cli()
    args = [str(tmp_path / "reads.fa"), "--SRCounts", str(tmp_path / "sr.dump"), "-k", str(cfg.k), "--strand", "auto"]
    run = lambda *a: subprocess.call([cli] + args + list(a), cwd=tmp_path, stdout=subprocess.DEVNULL)
    assert run("-o", "one", "--gpus", "1") == 0
    assert run("-o", "two", "--gpus", "2", "--batch-reads", "100") == 0
    assert run("-o", "peer", "--gpus", "2", "--batch-reads", "77", "--replicate", "peer") == 0
    for ext in (".fa", ".log", ".strand.txt"):
        a = open(tmp_path / ("one" + ext), "rb").read() if os.path.exists(tmp_path / ("one" + ext)) else b""
        for other in ("two", "peer"):
            b = open(tmp_path / (other + ext), "rb").read() if os.path.exists(tmp_path / (other + ext)) else b""
            assert a == b, (other, ext)
    assert open(tmp_path / "one.strand.txt", "rb").read().count(b"\t-\n") > 200
