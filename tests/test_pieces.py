"""--trim / --split: the stretches of each corrected read that the k-mer table supports, computed on the GPU.

The rule, restated in numpy below (np_pieces): a window [p, p+K) of a read's OUTPUT is solid when its K bytes are ACGT
(either case, U as T) and its k-mer is in the table -- the reverse complement of that k-mer when the read came back
flipped (reverse mode: status OK; auto mode: strand 1).  A base under a solid window is supported; a stretch is a maximal
run of supported bases.  Split gives one piece per stretch, trim [first supported base, last supported base + 1); pieces
shorter than min_len are dropped.  CPU tests pin the command line, the piece formatter and the numpy rule against a
per-base brute force; GPU tests hold talc_pieces_batch to numpy on crafted reads and every correction entry point to
numpy applied to the oracle's output."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile
import threading

import numpy as np
import pytest

from conftest import have_gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "tiny_case.npz")
SHARED = ["lookups_seg", "lookups_deg", "lookups_walk", "steps_inner", "steps_border", "frontier_sum", "cells_nw",
          "cells_lcs", "cells_ovl", "cells_xdrop", "gaps", "gaps_bridged", "gap_attempts", "borders",
          "borders_corrected", "ev_gardening", "ev_bridge", "ev_edge", "ev_cycle", "bases_out", "reads_ok",
          "reads_overflow", "reads_second_tier"]

# base_code of the device: ACGT and U in either case -> 0..3, anything else 4
_CODE = np.full(256, 4, dtype=np.uint8)
for _a, _v in zip(b"ACGTUacgtu", [0, 1, 2, 3, 3] * 2):
    _CODE[_a] = _v
# Dna5 conversion + reverse complement: ACGT in either case -> complement, anything else -> N
_COMP = np.full(256, ord("N"), dtype=np.uint8)
for _a, _b in zip(b"ACGTacgt", b"TGCATGCA"):
    _COMP[_a] = _b
# a complement that keeps case and IUPAC codes: the raw antisense of a read
_CASE_COMP = np.arange(256, dtype=np.uint8)
for _a, _b in zip(b"ACGTacgtRYry", b"TGCAtgcaYRyr"):
    _CASE_COMP[_a] = _b


def antisense(s: bytes) -> bytes:
    return _CASE_COMP[np.frombuffer(s, dtype=np.uint8)[::-1]].tobytes()


def rc(s: bytes) -> bytes:
    return _COMP[np.frombuffer(s, dtype=np.uint8)[::-1]].tobytes()


def _concat(seqs):
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(s) for s in seqs])
    return np.frombuffer(b"".join(seqs), dtype=np.uint8).copy(), off


def _split(reads, off):
    return [reads[int(off[r]):int(off[r + 1])].tobytes() for r in range(len(off) - 1)]


def _pack(codes, k):
    """packed k-mer of every window of codes (first base most significant), and whether it is all ACGT"""
    w = np.lib.stride_tricks.sliding_window_view(codes, k)
    shifts = (2 * np.arange(k - 1, -1, -1)).astype(np.uint64)
    return np.bitwise_or.reduce((w.astype(np.uint64) & np.uint64(3)) << shifts, axis=1), (w < 4).all(axis=1)


def _revcomp_keys(keys, k):
    r = np.zeros_like(keys)
    x = keys.copy()
    for _ in range(k):
        r = (r << np.uint64(2)) | (np.uint64(3) - (x & np.uint64(3)))
        x >>= np.uint64(2)
    return r


def solid_windows(seq: bytes, k: int, table, flip: bool) -> np.ndarray:
    """bool[max(0, L-K+1)]: the solid windows of one output read; table a sorted uint64 array of the keys present"""
    codes = _CODE[np.frombuffer(seq, dtype=np.uint8)]
    if len(codes) < k:
        return np.zeros(0, dtype=bool)
    keys, ok = _pack(codes, k)
    if flip:
        keys = _revcomp_keys(keys, k)
    return ok & np.isin(keys, table)


def stretches(solid: np.ndarray, k: int, length: int):
    """maximal runs of bases covered by a solid window, from a per-base coverage count"""
    cov = np.zeros(length + 1, dtype=np.int64)
    p = np.nonzero(solid)[0]
    np.add.at(cov, p, 1)
    np.add.at(cov, p + k, -1)
    sup = np.concatenate([[False], np.cumsum(cov[:length]) > 0, [False]])
    edges = np.nonzero(sup[1:] != sup[:-1])[0]
    return [(int(a), int(b)) for a, b in zip(edges[::2], edges[1::2])]


def np_pieces(seq: bytes, k: int, table, flip: bool, mode: str, min_len: int):
    st = stretches(solid_windows(seq, k, table, flip), k, len(seq))
    if mode == "trim":
        st = [(st[0][0], st[-1][1])] if st else []
    return [(a, b) for a, b in st if b - a >= min_len]


def brute_pieces(seq: bytes, k: int, keyset, flip: bool, mode: str, min_len: int):
    """the rule base by base, with a Python set and string k-mers"""
    def solid(p):
        w = seq[p:p + k]
        if any(c not in b"ACGTUacgtu" for c in w):
            return False
        s = w.upper().replace(b"U", b"T")
        if flip:
            s = s[::-1].translate(bytes.maketrans(b"ACGT", b"TGCA"))
        return s in keyset
    L = len(seq)
    sol = [solid(p) for p in range(L - k + 1)]
    sup = [any(sol[p] for p in range(max(0, i - k + 1), min(i, L - k) + 1)) for i in range(L)]
    runs, i = [], 0
    while i < L:
        if sup[i]:
            j = i
            while j < L and sup[j]:
                j += 1
            runs.append((i, j))
            i = j
        else:
            i += 1
    if mode == "trim":
        runs = [(runs[0][0], runs[-1][1])] if runs else []
    return [(a, b) for a, b in runs if b - a >= min_len]


def unpack(keys, k):
    return [bytes(b"ACGT"[(int(x) >> (2 * (k - 1 - j))) & 3] for j in range(k)) for x in keys]


def as_lists(piece_off, bounds):
    return [[tuple(int(v) for v in bounds[i]) for i in range(int(piece_off[r]), int(piece_off[r + 1]))]
            for r in range(len(piece_off) - 1)]


# ---------------------------------------------------------------------------------------------------- crafted reads
def crafted(k: int, seed: int):
    """(reads, flips, table keys, table counts): random reads whose solid windows are chosen through the table itself --
    the table holds exactly the chosen windows' k-mers (their reverse complements for a flipped read) at count 3, plus
    the unchosen ones of some reads at count 1, below MIN_COUNT.  The patterns cover lengths 0, K-1, K, K+1 and around
    the 128-window chunk edges; all solid, none solid, alternating, gaps of exactly one base; runs that cross a chunk
    edge; N, lower case, U and IUPAC bytes."""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs, flips, chosen, weak = [], [], [], []

    def add(length, pick, flip=False, edit=None):
        s = bytearray(rng.choice(acgt, length).tobytes())
        C_ = max(0, length - k + 1)
        sel = sorted({p for p in pick(C_) if 0 <= p < C_})
        for p in sel:
            chosen.append((bytes(s[p:p + k]), flip))
        if rng.random() < 0.3:
            weak.extend((bytes(s[p:p + k]), flip) for p in range(C_) if p not in sel)
        if edit:
            edit(s)
        seqs.append(bytes(s))
        flips.append(flip)

    every = lambda step, start=0: (lambda C_: range(start, C_, step))
    for length in (0, k - 1, k, k + 1, 126 + k, 127 + k, 128 + k, 129 + k, 254 + k, 255 + k, 256 + k, 383 + k, 600):
        for flip in (False, True):
            add(length, every(1), flip)
    add(300, lambda C_: [])
    add(300, every(2))                        # alternating solid windows: one stretch
    add(400, every(k + 1))                    # stretches of exactly K, gaps of exactly one base
    add(400, every(k))                        # windows K apart: one stretch
    add(400, every(k + 2, 5), True)
    add(300, lambda C_: [127, 128 + k])       # a one-base gap across the chunk edge
    add(300, lambda C_: [127, 127 + k])       # touching across the chunk edge: one stretch
    add(300, lambda C_: [100, 255, 256])
    add(300, lambda C_: [0, C_ - 1])
    add(300, lambda C_: range(120, 140))
    add(700, lambda C_: list(range(60, 130)) + list(range(130 + k, 300)) + [511 + k, 512 + k])
    add(200 + k, lambda C_: [127, 128])
    for flip in (False, True):
        # N in place of an A inside solid windows: the window holds no k-mer even though 'A' would match
        def n_for_a(s):
            for p in range(40, 140, 17):
                if s[p] == ord("A"):
                    s[p] = ord("N")
            for p in range(150, 250):
                if s[p] == ord("A"):
                    s[p] = ord("N")
                    break
        add(400, every(1), flip, n_for_a)
        add(400, every(1), flip, lambda s: s.__setitem__(slice(50, 120), bytes(s[50:120]).lower()))
        add(400, every(1), flip, lambda s: [s.__setitem__(p, ord("R") if p % 2 else ord("y")) for p in (30, 200, 333)])
        add(400, every(1), flip, lambda s: s.__setitem__(slice(None), bytes(s).replace(b"T", b"U")))
        add(400, every(1), flip, lambda s: s.__setitem__(slice(260, 262), b"nN"))
    for _ in range(40):
        length = int(rng.integers(0, 900))
        dens = rng.random()
        add(length, lambda C_: np.nonzero(rng.random(C_) < dens * dens)[0], bool(rng.random() < 0.5))
    # table: chosen windows at count 3 (reverse complement for a flipped read), others at 1
    def key_of(w, flip):
        x = 0
        for ch in (rc(w) if flip else w):
            x = (x << 2) | b"ACGT".index(ch)
        return x
    keys = [key_of(w, f) for w, f in chosen] + [key_of(w, f) for w, f in weak]
    counts = [3] * len(chosen) + [1] * len(weak)
    return seqs, np.array(flips, dtype=np.uint8), np.array(keys, dtype=np.uint64), np.array(counts, dtype=np.int64)


def _present(keys, counts, min_count=2):
    return np.unique(np.asarray(keys, dtype=np.uint64)[np.asarray(counts) >= min_count])


# ---------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("k", [18, 21, 31])
def test_numpy_rule_matches_brute_force(k):
    seqs, flips, keys, counts = crafted(k, 500 + k)
    table = _present(keys, counts)
    keyset = set(unpack(table, k))
    n_nonempty = 0
    for s, f in zip(seqs, flips):
        for mode in ("split", "trim"):
            for ml in (1, k + 1, 2 * k + 3):
                want = brute_pieces(s, k, keyset, bool(f), mode, ml)
                assert np_pieces(s, k, table, bool(f), mode, ml) == want, (s[:40], f, mode, ml)
                n_nonempty += bool(want)
    assert n_nonempty > 100
    # the patterns do what they say: gaps of one base, stretches of exactly K
    s = seqs[26 + 2]
    st = np_pieces(s, k, table, False, "split", 1)
    assert len(st) > 3 and all(b - a == k for a, b in st) and all(st[i + 1][0] - st[i][1] == 1 for i in range(len(st) - 1))


def test_cli_parses_pieces(tmp_path):
    """--trim, --split (alone and together) and --minPieceLength with either parse and leave .config.txt as it is;
    --minPieceLength alone, 0, negative, non-numeric or without a value is PARSE_ERROR (exit 1)."""
    from talc_b200 import build
    exe = build.build_cli()
    run = lambda *a: subprocess.call([exe, "missing.fa", "--SRCounts", "d.dump", "-k", "21", "-o", "x"] + list(a),
                                     stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, cwd=tmp_path)
    assert run() == 0
    plain = open(tmp_path / "x.config.txt").read()
    for extra in (["--trim"], ["--split"], ["--trim", "--split"], ["--split", "--minPieceLength", "1"],
                  ["--minPieceLength", "100", "--trim"], ["--trim", "--split", "--minPieceLength", "5000"],
                  ["--trim", "--strand", "auto"], ["--split", "--reverse"]):
        os.remove(tmp_path / "x.config.txt")
        assert run(*extra) == 0, extra
        assert open(tmp_path / "x.config.txt").read() == plain, extra
        assert not os.path.exists(tmp_path / "x.trim.fa") and not os.path.exists(tmp_path / "x.split.fa")
    for extra in (["--minPieceLength", "5"], ["--trim", "--minPieceLength", "0"], ["--split", "--minPieceLength", "-3"],
                  ["--trim", "--minPieceLength", "x"], ["--trim", "--minPieceLength"], ["--split", "--minPieceLength", "2.5"]):
        assert run(*extra) == 1, extra
    out = subprocess.run([exe, "--help"], capture_output=True, text=True).stdout
    assert "--trim" in out and "--split" in out and "--minPieceLength" in out


@pytest.fixture(scope="module")
def pio():
    src = os.path.join(HERE, "hostemu", "pieces_io_test.cpp")
    hdr = os.path.join(HERE, "..", "talc_b200", "csrc", "host", "reads_io.hpp")
    h = hashlib.sha256(open(src, "rb").read() + open(hdr, "rb").read()).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), "talc_pieces_io_%s_%d.so" % (h, os.getuid()))
    if not os.path.exists(so):
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-pthread", "-fPIC", "-shared", src, "-o", tmp])
        os.replace(tmp, so)
    L = C.CDLL(so)
    L.pio_format.restype = C.c_long
    L.pio_format.argtypes = [C.c_char_p, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint,
                             C.c_char_p, C.c_long, C.c_void_p]
    return L


def py_piece_records(names, seqs, pieces, mode, min_len):
    """the --trim / --split records from every stretch of each read, as bytes (70 columns)"""
    out, tally = [], [0, 0, 0]
    for name, s, st in zip(names, seqs, pieces):
        if mode == "trim":
            st = [(st[0][0], st[-1][1])] if st else []
        kept = [(a, b) for a, b in st if b - a >= min_len]
        for a, b in kept:
            if mode == "split":
                cut = min([i for i, ch in enumerate(name) if ch in b" \t"] + [len(name)])
                head = name[:cut] + b"_%d_%d" % (a, b) + name[cut:]
            else:
                head = name
            piece = s[a:b]
            out.append(b">" + head + b"\n" + b"".join(piece[i:i + 70] + b"\n" for i in range(0, len(piece), 70)))
            tally[1] += 1
            tally[2] += b - a
        tally[0] += bool(kept)
    return b"".join(out), tally


def test_piece_formatter(pio):
    """format_pieces against the Python restatement: headers with and without a description (blank or tab), pieces
    ending on and around 70-column boundaries, reads without a piece, min_len above some pieces."""
    rng = np.random.default_rng(3)
    names = [b"r0", b"r1 some description", b"r2\tx=1 y", b"r3", b"r4 ", b"r5", b"r6 d"]
    seqs = [bytes(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), n)) for n in (300, 250, 141, 0, 90, 500, 71)]
    pieces = [[(0, 70), (71, 141), (150, 290)], [(10, 31)], [(0, 141)], [], [(20, 89)], [(0, 140), (141, 211), (300, 371), (429, 500)],
              [(0, 71)]]
    ids = b"\n".join(names)
    out, oo = _concat(seqs)
    po = np.zeros(len(seqs) + 1, dtype=np.uint64)
    po[1:] = np.cumsum([len(p) for p in pieces])
    b = np.array([x for p in pieces for x in p], dtype=np.uint32).reshape(-1, 2)
    for mode in ("trim", "split"):
        for ml in (1, 21, 70, 71, 141, 1000):
            dst = C.create_string_buffer(1 << 16)
            tally = np.zeros(3, dtype=np.uint64)
            n = pio.pio_format(ids, len(names), out.ctypes.data, oo.ctypes.data, po.ctypes.data, b.ctypes.data,
                               1 if mode == "split" else 0, ml, dst, len(dst), tally.ctypes.data)
            want, wt = py_piece_records(names, seqs, pieces, mode, ml)
            assert dst.raw[:n] == want, (mode, ml)
            assert list(tally) == wt, (mode, ml)
    got = C.create_string_buffer(1 << 16)
    tally = np.zeros(3, dtype=np.uint64)
    n = pio.pio_format(ids, len(names), out.ctypes.data, oo.ctypes.data, po.ctypes.data, b.ctypes.data, 1, 1, got,
                       len(got), tally.ctypes.data)
    assert b">r1_10_31 some description\n" in got.raw[:n] and b">r2_0_141\tx=1 y\n" in got.raw[:n]
    assert b">r4_20_89 \n" in got.raw[:n] and b">r3" not in got.raw[:n]


# ---------------------------------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    if not have_gpu():
        pytest.fail("GPU tests selected but no CUDA device is visible")
    from talc_b200 import api as _api
    return _api


@gpu
@pytest.mark.parametrize("k", list(range(18, 32)))
def test_pieces_batch_matches_numpy(api, k):
    """talc_pieces_batch == numpy on the crafted reads, both modes, min_len below, at and above the stretch lengths,
    flip flags as crafted, and with no flags at all."""
    seqs, flips, keys, counts = crafted(k, 900 + k)
    table = _present(keys, counts)
    t = api.Talc(api.default_params(k))
    t.load_packed(keys, counts)
    reads, off = _concat(seqs)
    for fl in (flips, None):
        for mode in ("split", "trim"):
            for ml in (1, k, k + 1, 2 * k, 200):
                po, b = t.pieces(reads, off, fl, mode, ml)
                got = as_lists(po, b)
                want = [np_pieces(s, k, table, bool(fl[r]) if fl is not None else False, mode, ml) for r, s in enumerate(seqs)]
                bad = [r for r in range(len(seqs)) if got[r] != want[r]]
                assert not bad, (k, mode, ml, fl is None, bad[:5], [(got[r], want[r]) for r in bad[:2]])
    assert sum(len(x) for x in want) > 20
    po, b = t.pieces(reads[:0], off[:1])
    assert len(po) == 1 and po[0] == 0 and len(b) == 0
    with pytest.raises(api.TalcError):
        t.pieces(reads, off, None, "off")
    with pytest.raises(api.TalcError):
        t.pieces(reads, off, None, "split", 0)
    t.close()


def _expected(case, mode):
    """(input reads, offsets, expected output parts, status, output offsets, counters, flip flags) of a strand mode, from
    the oracle: forward on the reads as they are; reverse on the antisense of the reads (so that they correct), reverse-
    complemented first and the corrected reads flipped back; auto on each read's better strand (the oracle's coverage of
    both), strand-1 reads flipped back"""
    seqs = _split(case.reads, case.off)
    if mode == "forward":
        parts = _split(case.o_out, case.o_off)
        return case.reads, case.off, parts, case.o_status, case.o_off, case.o_ctr, np.zeros(len(seqs), dtype=np.uint8)
    if mode == "reverse":
        seqs = [antisense(s) for s in seqs]
        flip_in = np.ones(len(seqs), dtype=np.uint8)
    else:
        ff = np.array([int((case.otable.coverage(s)[0] != 0).sum()) for s in seqs])
        fr = np.array([int((case.otable.coverage(rc(s))[0] != 0).sum()) for s in seqs])
        flip_in = (fr > ff).astype(np.uint8)
    oriented, off = _concat([rc(s) if f else s for s, f in zip(seqs, flip_in)])
    o_out, o_off, o_st, o_ctr, _ = case.otable.correct(oriented, off, threads=8)
    flip = (o_st == 0).astype(np.uint8) if mode == "reverse" else flip_in
    parts = [rc(x) if f else x for x, f in zip(_split(o_out, o_off), flip)]
    return _concat(seqs) + (parts, o_st, o_off, o_ctr, flip)


_exp = {}


def expected(case, mode):
    key = (id(case), mode)
    if key not in _exp:
        _exp[key] = _expected(case, mode)
    return _exp[key]


@gpu
@pytest.mark.parametrize("name", ["c1", "c3", "c5"])
@pytest.mark.parametrize("strand", ["forward", "reverse", "auto"])
def test_pieces_of_the_correction_match_oracle(api, name, strand, request):
    """talc_correct_batch with pieces on, both execution shapes: the pieces are numpy applied to the oracle's output
    with the flip flags the oracle implies; bytes, offsets, status, strands and counters equal a run with pieces off."""
    case = request.getfixturevalue("case_" + name)
    k = case.cfg.k
    reads, roff, parts, o_st, o_off, o_ctr, flip = expected(case, strand)
    table = _present(case.keys, case.counts)
    for shape, (pmode, ml) in ((1, ("split", 1)), (2, ("trim", 1)), (1, ("trim", k + 40)), (2, ("split", 2 * k))):
        t = api.Talc(api.default_params(k))
        t.load_packed(case.keys, case.counts, case.jkeys, case.jcounts)
        t.set_strand(strand)
        t.set_exec(shape)
        a_out, a_off, a_st, a_ctr = t.correct(reads, roff)
        a_strand = t.last_strands(len(a_st))
        t.set_pieces(pmode, ml)
        out, off, st, ctr = t.correct(reads, roff)
        assert np.array_equal(st, a_st) and np.array_equal(off, a_off) and np.array_equal(out, a_out)
        assert np.array_equal(t.last_strands(len(st)), a_strand)
        assert {x: ctr[x] for x in SHARED + ["kernel_launches"]} == {x: a_ctr[x] for x in SHARED + ["kernel_launches"]}
        assert np.array_equal(st, o_st) and np.array_equal(off, o_off) and _split(out, off) == parts
        assert {x: ctr[x] for x in SHARED[:-3]} == {x: o_ctr[x] for x in SHARED[:-3]}
        got = as_lists(*t.last_pieces(len(st)))
        want = [np_pieces(s, k, table, bool(f), pmode, ml) for s, f in zip(parts, flip)]
        bad = [r for r in range(len(parts)) if got[r] != want[r]]
        assert not bad, (strand, shape, pmode, ml, bad[:5], [(got[r], want[r]) for r in bad[:2]])
        assert sum(map(len, want)) > 0.5 * len(parts)
        t.set_pieces("off")
        t.correct(case.reads[:0], case.off[:1])
        with pytest.raises(api.TalcError):
            t.last_pieces(0)
        t.close()


@gpu
def test_pieces_through_device_call_lane_and_stream(api, case_c1):
    """talc_correct_batch_device (pieces to host and to a device buffer), a lane from a second thread and a stream with
    uneven batches (one empty) give the pieces of the host call; a lane refuses its own setting."""
    import torch
    case = case_c1
    k = case.cfg.k
    _, _, parts, o_st, o_off, _, flip = expected(case, "auto")
    table = _present(case.keys, case.counts)
    want = [np_pieces(s, k, table, bool(f), "split", 1) for s, f in zip(parts, flip)]
    n = len(parts)
    t = api.Talc(api.default_params(k))
    t.load_packed(case.keys, case.counts)
    t.set_strand("auto")
    t.set_pieces("split")
    out, off, st, _ = t.correct(case.reads, case.off)
    assert as_lists(*t.last_pieces(n)) == want
    po_host, b_host = t.last_pieces(n)
    d_reads = torch.from_numpy(case.reads.copy()).cuda()
    d_off = torch.from_numpy(case.off.astype(np.int64)).cuda()
    d_out = torch.empty(2 * len(case.reads) + 64 * n + 4096, dtype=torch.uint8, device="cuda")
    d_ooff = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    d_st = torch.zeros(n, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    t.correct_device(d_reads, d_off, len(case.reads), d_out, d_ooff, d_st)
    assert as_lists(*t.last_pieces(n)) == want
    total = C.c_uint64(0)
    d_po = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    d_b = torch.zeros(len(b_host) * 2, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    from talc_b200.api import lib
    assert lib().talc_last_pieces(t.h, C.c_void_p(d_po.data_ptr()), C.c_void_p(d_b.data_ptr()), len(b_host), C.byref(total)) == 0
    assert np.array_equal(d_po.cpu().numpy().astype(np.uint64), po_host)
    assert np.array_equal(d_b.cpu().numpy().view(np.uint32).reshape(-1, 2), b_host)
    short = np.zeros((len(b_host), 2), dtype=np.uint32)
    assert lib().talc_last_pieces(t.h, None, short.ctypes.data, len(b_host) - 1, C.byref(total)) == -5
    assert total.value == len(b_host) and not short.any()
    # the stream: uneven batches, one of them empty
    cuts = [0, 1, 1, 40, 41, 130, n]
    s = t.stream()
    got = []
    for a, b in zip(cuts, cuts[1:]):
        s.submit(case.reads[int(case.off[a]):int(case.off[b])], case.off[a:b + 1] - case.off[a])
        o, f, x, _, _ = s.next()
        p = s.pieces()
        assert p is not None and len(p[0]) == b - a + 1
        got += as_lists(*p)
        assert np.array_equal(x, st[a:b])
    s.close()
    assert got == want
    # a lane from a second thread
    lane = t.create_lane()
    with pytest.raises(api.TalcError):
        lane.set_pieces("trim")
    h = n // 2
    res = [None, None]

    def run(i, c, a, b):
        c.correct(case.reads[int(case.off[a]):int(case.off[b])], case.off[a:b + 1] - case.off[a])
        res[i] = as_lists(*c.last_pieces(b - a))

    th = [threading.Thread(target=run, args=(0, t, 0, h)), threading.Thread(target=run, args=(1, lane, h, n))]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert res[0] + res[1] == want
    lane.close()
    # pieces off: the stream reports none
    t.set_pieces("off")
    s = t.stream()
    s.submit(case.reads, case.off)
    s.next()
    assert s.pieces() is None
    s.close()
    t.close()


@gpu
@pytest.mark.parametrize("strand", ["forward", "reverse"])
def test_pieces_of_resource_reads(api, case_c1, strand):
    """Reads that outgrow the second tier (TALC_READ_RESOURCE) get their pieces by the same rule, on the bytes they
    come back as; every other read's pieces are those of the oracle's output."""
    case = case_c1
    k = case.cfg.k
    seqs = []
    for r in range(len(case.off) - 1):
        s = bytearray(case.read(r))
        if r % 3 == 0:
            s[100:160] = s[100:160].lower()
            s[250] = ord("R")
        seqs.append(antisense(bytes(s)) if strand == "reverse" else bytes(s))
    reads, off = _concat(seqs)
    table = _present(case.keys, case.counts)
    for shape in (1, 2):
        t = api.Talc(api.default_params(k))
        t.load_packed(case.keys, case.counts)
        t.set_strand(strand)
        t.set_exec(shape)
        t.set_scratch(6 * 1024, 128 * 1024, 4)
        t.set_pieces("split")
        out, ooff, st, ctr = t.correct(reads, off)
        res = st == api.STATUS_RESOURCE
        assert 0 < res.sum() < len(st) and ctr["reads_overflow"] == res.sum()
        flip = (st == 0) if strand == "reverse" else np.zeros(len(st), dtype=bool)
        got = as_lists(*t.last_pieces(len(st)))
        want = [np_pieces(s, k, table, bool(f), "split", 1) for s, f in zip(_split(out, ooff), flip)]
        assert got == want
        assert any(got[r] for r in np.nonzero(res)[0])
        t.close()


def _records():
    g = np.load(GOLD)
    seqs = _split(g["c3_reads"], g["c3_off"])
    recs = [((b"read_%d" % r) + (b" len=%d sample 1" % len(s) if r % 4 == 1 else b"\tx" if r % 4 == 2 else b""), s)
            for r, s in enumerate(seqs)]
    recs[3:3] = [(b"tiny", b"ACGTACGT"), (b"junk desc", b"ACGT" * 60)]
    return g, recs


def _write_inputs(tmp_path, g, recs, reverse=False):
    import torch
    from talc_b200 import synth
    k = int(g["c3_k"][0])
    synth.write_dump(str(tmp_path / "sr.dump"), torch.from_numpy(g["c3_keys"].astype(np.int64)),
                     torch.from_numpy(g["c3_counts"].astype(np.int64)), k)
    synth.write_dump(str(tmp_path / "j.dump"), torch.from_numpy(g["c3_jkeys"].astype(np.int64)),
                     torch.from_numpy(g["c3_jcounts"].astype(np.int64)), k)
    with open(tmp_path / "reads.fa", "wb") as f:
        for name, s in recs:
            f.write(b">" + name + b"\n" + (antisense(s) if reverse else s) + b"\n")
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


@gpu
@pytest.mark.parametrize("strand", ["forward", "reverse", "auto"])
def test_cli_trim_split(api, tmp_path, strand):
    """`talc --trim --split`: .trim.fa and .split.fa are the numpy rule applied to the .fa (the oracle front end's .fa
    in forward and reverse mode), with the flip flags of the mode; .fa, .log, .config.txt, .stats_basics.txt and
    .strand.txt are byte-identical to a run without the options, whatever the batching and --minPieceLength."""
    from oracle import pyoracle as po
    from talc_b200 import build
    g, recs = _records()
    k, common = _write_inputs(tmp_path, g, recs, reverse=strand == "reverse")
    cli = build.build_cli()
    smode = ["--strand", strand]
    run = lambda *a: subprocess.run([cli, str(tmp_path / "reads.fa")] + common + smode + list(a), cwd=tmp_path,
                                    capture_output=True, text=True)
    r = run("-o", "plain")
    assert r.returncode == 0
    for prefix, extra, ml in (("both", ["--trim", "--split"], 1), ("many", ["--split", "--trim", "--batch-reads", "7"], 1),
                              ("ml", ["--trim", "--split", "--minPieceLength", "150", "--batch-reads", "13"], 150)):
        r = run("-o", prefix, *extra)
        assert r.returncode == 0, r.stderr
        for ext in (".fa", ".log", ".stats_basics.txt", ".strand.txt"):
            a, b = tmp_path / ("plain" + ext), tmp_path / (prefix + ext)
            assert os.path.exists(a) == os.path.exists(b), ext
            if os.path.exists(a):
                assert open(a, "rb").read() == open(b, "rb").read(), (prefix, ext)
        assert open(tmp_path / "plain.config.txt").read().replace("plain", "X") == \
            open(tmp_path / (prefix + ".config.txt")).read().replace(prefix, "X")
        fa = _read_fasta(tmp_path / (prefix + ".fa"))
        if strand == "forward":
            flip = [False] * len(fa)
        elif strand == "reverse":
            log = open(tmp_path / "plain.log", "rb").read() if os.path.exists(tmp_path / "plain.log") else b""
            flip = [len(s) > k and b"[Read: " + n + b" ]" not in log for (n, s) in recs]
        else:
            flip = [line.endswith(b"\t-") for line in open(tmp_path / "plain.strand.txt", "rb").read().split(b"\n") if line]
        table = _present(g["c3_keys"], g["c3_counts"])
        pieces = [np_pieces(s, k, table, f, "split", 1) for (_, s), f in zip(fa, flip)]
        names, seqs = [n for n, _ in fa], [s for _, s in fa]
        for mode in ("trim", "split"):
            want, tally = py_piece_records(names, seqs, pieces, mode, ml)
            assert open(tmp_path / ("%s.%s.fa" % (prefix, mode)), "rb").read() == want, (prefix, mode)
            assert "--%s: %d read(s) kept, %d piece(s), %d bases" % (mode, *tally) in r.stdout
        assert 0 < tally[0] < len(fa)
    assert not os.path.exists(tmp_path / "plain.trim.fa") and not os.path.exists(tmp_path / "plain.split.fa")
    if strand != "auto":  # the .fa the numpy rule was applied to is the oracle front end's
        ora = subprocess.call([po.BIN, str(tmp_path / "reads.fa")] + common + ["-t", "1", "--oracle-table", "hash", "-o", "ora"]
                              + (["--reverse"] if strand == "reverse" else []), cwd=tmp_path, stdout=subprocess.DEVNULL)
        assert ora == 0
        for ext in (".fa", ".log"):
            a = tmp_path / ("ora" + ext)
            assert (open(a, "rb").read() if os.path.exists(a) else b"") == \
                (open(tmp_path / ("plain" + ext), "rb").read() if os.path.exists(tmp_path / ("plain" + ext)) else b""), ext


@gpu
def test_cli_trim_split_two_gpus_equals_one(api, tmp_path):
    import torch
    from talc_b200 import build
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    g, recs = _records()
    k, common = _write_inputs(tmp_path, g, recs)
    cli = build.build_cli()
    run = lambda *a: subprocess.call([cli, str(tmp_path / "reads.fa")] + common + ["--trim", "--split"] + list(a),
                                     cwd=tmp_path, stdout=subprocess.DEVNULL)
    assert run("-o", "one") == 0 and run("-o", "two", "--gpus", "2", "--batch-reads", "9") == 0
    for ext in (".fa", ".trim.fa", ".split.fa"):
        assert open(tmp_path / ("one" + ext), "rb").read() == open(tmp_path / ("two" + ext), "rb").read(), ext
