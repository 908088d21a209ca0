"""The k-mer table from stranded and unstranded short-read libraries: talc_table_count_reads_oriented (one orientation
per file: SENSE counts each window x, ANTISENSE rc(x), BOTH x and rc(x), a reverse palindrome once), canonical dumps
(talc_table_load_dump_ex with TALC_DUMP_CANONICAL: line (x, c) stands for (x, c), (rc(x), c)), the cache flags and the
command line (--SRReads, --SRReads2, --SRLibType, --SRExpected, --SRCanonical).

The numpy restatement below follows the kernel's windows: K consecutive bases that base_code reads as A, C, G or T, so a
U counts as T (oracle/kmer_count.py leaves windows with U out; its readers are reused here).  CPU tests pin the command
line and the identities between the counting modes; GPU tests hold the library and the command line to numpy and to
the oracle."""
import os
import subprocess

import numpy as np
import pytest

from conftest import get_case, have_gpu

SHARED = ["lookups_seg", "lookups_deg", "lookups_walk", "steps_inner", "steps_border", "frontier_sum", "cells_nw",
          "cells_lcs", "cells_ovl", "cells_xdrop", "gaps", "gaps_bridged", "gap_attempts", "borders",
          "borders_corrected", "ev_gardening", "ev_bridge", "ev_edge", "ev_cycle", "bases_out"]
SENSE, ANTISENSE, BOTH = 0, 1, 2
LIBTYPES = {"asis": (SENSE, SENSE), "unstranded": (BOTH, BOTH), "fr-firststrand": (ANTISENSE, SENSE),
            "fr-secondstrand": (SENSE, ANTISENSE)}  # (R1 / single-end, R2)

# base_code of the kernel: ACGT and U in either case, U read as T; anything else breaks the window
_CODE = np.full(256, 4, dtype=np.uint8)
for _a, _v in zip(b"ACGTUacgtu", [0, 1, 2, 3, 3] * 2):
    _CODE[_a] = _v
# reverse complement that keeps every window: U pairs with A like T, anything else stays a break (N)
_COMP = np.full(256, ord("N"), dtype=np.uint8)
for _a, _b in zip(b"ACGTUacgtu", b"TGCAATGCAA"):
    _COMP[_a] = _b


def rc(s: bytes) -> bytes:
    return _COMP[np.frombuffer(s, dtype=np.uint8)[::-1]].tobytes()


def window_keys(seq: bytes, k: int) -> np.ndarray:
    """packed keys (first base most significant) of every window the kernel counts, in read order"""
    c = _CODE[np.frombuffer(seq, dtype=np.uint8)]
    if len(c) < k:
        return np.zeros(0, np.uint64)
    w = np.lib.stride_tricks.sliding_window_view(c, k)
    ok = (w < 4).all(axis=1)
    shifts = (2 * np.arange(k - 1, -1, -1)).astype(np.uint64)
    keys = np.bitwise_or.reduce((w.astype(np.uint64) & np.uint64(3)) << shifts, axis=1)
    return keys[ok]


def revcomp_keys(keys, k: int) -> np.ndarray:
    x = np.asarray(keys, dtype=np.uint64).copy()
    r = np.zeros_like(x)
    for _ in range(k):
        r = (r << np.uint64(2)) | (np.uint64(3) - (x & np.uint64(3)))
        x >>= np.uint64(2)
    return r


def count_kmers_oriented(files_of_seqs, orients, k: int):
    """(sorted distinct keys, counts [int64], count increments) of talc_table_count_reads_oriented"""
    parts = [np.zeros(0, np.uint64)]
    for seqs, o in zip(files_of_seqs, orients):
        for s in seqs:
            x = window_keys(s, k)
            if o == SENSE:
                parts.append(x)
            elif o == ANTISENSE:
                parts.append(revcomp_keys(x, k))
            else:
                r = revcomp_keys(x, k)
                parts += [x, r[r != x]]
    allk = np.concatenate(parts)
    keys, counts = np.unique(allk, return_counts=True)
    return keys, counts.astype(np.int64), int(allk.size)


def canonical_counts(seqs, k: int):
    """`jellyfish count -C`: every window counted under min(x, rc(x)); (sorted keys, counts)"""
    x = np.concatenate([np.zeros(0, np.uint64)] + [window_keys(s, k) for s in seqs])
    keys, counts = np.unique(np.minimum(x, revcomp_keys(x, k)), return_counts=True)
    return keys, counts.astype(np.int64)


def expand_canonical(keys, counts, k: int):
    """line i (x, c) of a canonical dump -> lines 2i (x, c) and 2i+1 (rc(x), c)"""
    keys = np.asarray(keys, dtype=np.uint64)
    ek = np.empty(2 * len(keys), np.uint64)
    ek[0::2], ek[1::2] = keys, revcomp_keys(keys, k)
    return ek, np.repeat(np.asarray(counts, dtype=np.int64), 2)


def table_from_dump(keys, counts, min_count: int = 2):
    """buildCDBG on dump lines: lines with count >= MIN_COUNT, the first line of a k-mer wins; (sorted keys, counts)"""
    keys, counts = np.asarray(keys, dtype=np.uint64), np.asarray(counts, dtype=np.int64)
    keep = counts >= min_count
    u, first = np.unique(keys[keep], return_index=True)
    return u, counts[keep][first]


def read_files(paths):
    from oracle import kmer_count as kc
    return [kc.read_sequences(str(p)) for p in paths]


def write_fastq(path, seqs):
    with open(path, "wb") as f:
        for i, s in enumerate(seqs):
            f.write(b"@r%d\n" % i + s + b"\n+\n" + b"I" * len(s) + b"\n")


def write_fasta_crlf(path, seqs):
    with open(path, "wb") as f:
        for i, s in enumerate(seqs):
            f.write(b">r%d\r\n" % i + s + b"\r\n")


def _mutate(rng, s: bytes, extras: bool = True) -> bytes:
    b = bytearray(s)
    for q in np.nonzero(rng.random(len(b)) < 0.01)[0]:
        b[q] = b"ACGT"[int(rng.integers(0, 4))]
    if extras:
        r = rng.random()
        if r < 0.05 and len(b) > 5:
            b[int(rng.integers(0, len(b)))] = ord("N")
        elif r < 0.08 and len(b) > 5:
            b[int(rng.integers(0, len(b)))] = ord("U" if rng.random() < 0.5 else "u")
        elif r < 0.14:
            b = bytearray(bytes(b).lower())
    return bytes(b)


def _special(k: int):
    """reads shorter than K, reverse palindromes (every window of (ACGT)* and (AT)* at even K has rc(x) == x for half
    of its windows), a read followed by its reverse complement, U, N, lower case"""
    rng = np.random.default_rng(k)
    a = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), 2 * k).tobytes()
    return [b"ACGT", a[:k - 1], b"ACGT" * 12, b"AT" * 30, b"acgt" * 9, a + rc(a), a[:k] + rc(a[:k]), b"ACGU" * 10,
            a.replace(b"T", b"U"), a[:k // 2] + b"N" + a[k // 2:], b"N" * 40, b"A" * 60]


def _pool_reads(seed: int, n: int, k: int):
    """short reads of both strands from a random 'transcriptome', mutated, plus the special reads"""
    rng = np.random.default_rng(seed)
    pool = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), 12000).tobytes()
    out = []
    for _ in range(n):
        L = int(rng.integers(30, 151))
        p = int(rng.integers(0, len(pool) - L))
        s = _mutate(rng, pool[p:p + L])
        out.append(rc(s) if rng.random() < 0.3 else s)
    return out + _special(k)


# ---------------------------------------------------------------------------------------------------- CPU
def test_cli_parses_sr_options(tmp_path):
    """--SRReads / --SRReads2 / --SRLibType / --SRExpected / --SRCanonical parse and leave .config.txt as it is; every
    combination the option rules forbid is PARSE_ERROR (exit 1); --help lists them."""
    from talc_b200 import build
    exe = build.build_cli()
    run = lambda *a: subprocess.call([exe, "missing.fa", "-k", "21", "-o", "x"] + list(a), stdout=subprocess.DEVNULL,
                                     stderr=subprocess.DEVNULL, cwd=tmp_path)
    assert run("--SRCounts", "d.dump") == 0
    plain = open(tmp_path / "x.config.txt").read()
    ok = [["--SRReads", "a.fq"], ["--SRReads", "a.fq", "--SRReads2", "b.fq"],
          ["--SRReads", "a", "--SRReads", "b", "--SRReads2", "c", "--SRReads2", "d", "--SRLibType", "fr-firststrand"],
          ["--SRReads", "a", "--SRExpected", "1000000"], ["--SRCounts", "d.dump", "--SRCanonical"],
          ["--SRCounts", "d.dump", "--SRCanonical", "--tableCache", "t.bin"],
          ["--SRReads", "a", "--SRLibType", "unstranded", "--strand", "auto"]]
    ok += [["--SRReads", "a", "--SRReads2", "b", "--SRLibType", t] for t in LIBTYPES]
    for extra in ok:
        os.remove(tmp_path / "x.config.txt")
        assert run(*extra) == 0, extra
        assert open(tmp_path / "x.config.txt").read() == plain, extra
    assert run("--SRCounts", "d.dump", "--junctions", "j") == 0
    junc = open(tmp_path / "x.config.txt").read()
    assert junc != plain
    assert run("--junctions", "j", "--SRReads", "a", "--SRLibType", "unstranded") == 0
    assert open(tmp_path / "x.config.txt").read() == junc
    bad = [[], ["--SRCanonical"], ["--SRCounts", "d", "--SRReads", "a"], ["--SRReads", "a", "--SRCounts", "d"],
           ["--SRCounts", "d", "--SRLibType", "asis"], ["--SRCounts", "d", "--SRReads2", "b"],
           ["--SRCounts", "d", "--SRExpected", "10"], ["--SRReads2", "b"], ["--SRLibType", "unstranded"],
           ["--SRReads", "a", "--SRReads2", "b", "--SRReads2", "c"], ["--SRReads", "a", "--SRReads", "b", "--SRReads2", "c"],
           ["--SRReads", "a", "--SRCanonical"], ["--SRReads", "a", "--tableCache", "t.bin"],
           ["--SRReads", "a", "--SRLibType", "stranded"], ["--SRReads", "a", "--SRLibType", "Unstranded"],
           ["--SRReads", "a", "--SRLibType"], ["--SRReads"], ["--SRReads", "a", "--SRReads2"],
           ["--SRReads", "a", "--SRExpected", "0"], ["--SRReads", "a", "--SRExpected", "x"], ["--SRReads", "a", "--SRExpected"]]
    for extra in bad:
        assert run(*extra) == 1, extra
    out = subprocess.run([exe, "--help"], capture_output=True, text=True).stdout
    for s in ("--SRCounts <dump>", "--SRReads <fq|fa>", "--SRReads2 <fq|fa>", "--SRCanonical", "--SRExpected <N>",
              "--SRLibType asis|unstranded|fr-firststrand|fr-secondstrand"):
        assert s in out, s


@pytest.mark.parametrize("k", [20, 21])
def test_np_both_is_the_canonical_count_expanded(k):
    """BOTH == the `jellyfish count -C` counts expanded onto both orientations, reverse palindromes counted once."""
    seqs = _pool_reads(k, 400, k)
    keys, counts, n = count_kmers_oriented([seqs], [BOTH], k)
    ck, cc = canonical_counts(seqs, k)
    ek, ec = table_from_dump(*expand_canonical(ck, cc, k), min_count=1)
    assert np.array_equal(keys, ek) and np.array_equal(counts, ec)
    sense_k, sense_c, n_sense = count_kmers_oriented([seqs], [SENSE], k)
    occ = dict(zip(sense_k.tolist(), sense_c.tolist()))
    pal = keys == revcomp_keys(keys, k)
    assert n == 2 * n_sense - sum(occ[x] for x in keys[pal].tolist())
    want = [occ.get(x, 0) + (0 if p else occ.get(r, 0)) for x, r, p in zip(keys.tolist(), revcomp_keys(keys, k).tolist(), pal)]
    assert np.array_equal(counts, np.array(want, dtype=np.int64))
    if k % 2 == 0:  # (ACGT)* and (AT)* hold palindromes at even K; each occurrence counts once
        for rep in (b"ACGT", b"AT"):
            x = window_keys(rep * (k // len(rep) + 1), k)[0]
            assert int(revcomp_keys([x], k)[0]) == int(x)
            assert counts[np.searchsorted(keys, x)] == occ[int(x)]
    else:
        assert not pal.any()


@pytest.mark.parametrize("k", [20, 31])
def test_np_antisense_is_sense_of_the_reverse_complements(k):
    seqs = _pool_reads(100 + k, 300, k)
    a = count_kmers_oriented([seqs], [ANTISENSE], k)
    s = count_kmers_oriented([[rc(x) for x in seqs]], [SENSE], k)
    assert np.array_equal(a[0], s[0]) and np.array_equal(a[1], s[1]) and a[2] == s[2]
    mixed = count_kmers_oriented([seqs[:150], seqs[150:]], [ANTISENSE, SENSE], k)
    s2 = count_kmers_oriented([[rc(x) for x in seqs[:150]] + seqs[150:]], [SENSE], k)
    assert np.array_equal(mixed[0], s2[0]) and np.array_equal(mixed[1], s2[1])


def test_np_expanded_canonical_dump_rule():
    """the table of an expanded dump: lines (x, c), (rc(x), c); MIN_COUNT per line, first line wins -- also for a dump
    that is not canonical (a k-mer and its reverse complement on two lines with different counts)"""
    k = 21
    keys = np.array([5, 7, 5, 9, 11], dtype=np.uint64)
    r = revcomp_keys(keys, k)
    keys[3] = r[1]  # line 3 is the reverse complement of line 1, with another count
    counts = np.array([3, 4, 8, 6, 1], dtype=np.int64)
    tk, tc = table_from_dump(*expand_canonical(keys, counts, k))
    want = {5: 3, int(r[0]): 3, 7: 4, int(r[1]): 4}  # line 2 repeats line 0; line 3 lost to line 1; line 4 below MIN
    assert dict(zip(tk.tolist(), tc.tolist())) == want


# ---------------------------------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    if not have_gpu():
        pytest.fail("GPU tests selected but no CUDA device is visible")
    from talc_b200 import api as _api
    return _api


def _check_lookups(t, keys, counts, probe, min_count=2):
    """every probe answers as the numpy table (keys, counts) filtered to count >= MIN_COUNT"""
    kept = counts >= min_count
    kk, kc = keys[kept], counts[kept]
    cnt, _, found = t.lookup(probe)
    pos = np.minimum(np.searchsorted(kk, probe), max(len(kk) - 1, 0))
    hit = (kk[pos] == probe) if len(kk) else np.zeros(len(probe), bool)
    assert np.array_equal(found.astype(bool), hit)
    assert np.array_equal(cnt[hit], kc[pos[hit]].astype(np.uint32)) and not cnt[~hit].any()


def _probe(keys, k, seed=0):
    rng = np.random.default_rng(seed)
    return np.concatenate([keys, revcomp_keys(keys, k),
                           rng.integers(0, 1 << (2 * k), 3000, dtype=np.uint64)]).astype(np.uint64)


@gpu
@pytest.mark.parametrize("k", [20, 21, 30, 31])
def test_count_reads_oriented(api, k, tmp_path):
    """each orientation and per-file mixes against numpy: (increments, distinct, kept) and look-ups of every key, its
    reverse complement and random keys; all-SENSE against talc_table_count_reads"""
    a, b = _pool_reads(k, 3000, k), _pool_reads(50 + k, 2000, k)
    write_fastq(tmp_path / "a.fq", a)
    write_fasta_crlf(tmp_path / "b.fa", b)
    paths = [str(tmp_path / "a.fq"), str(tmp_path / "b.fa")]
    files = read_files(paths)
    assert files[0] == a and files[1] == b
    t = api.Talc(api.default_params(k))
    for orient in ([SENSE, SENSE], [ANTISENSE, ANTISENSE], [BOTH, BOTH], [ANTISENSE, SENSE], [BOTH, SENSE], [SENSE, BOTH]):
        keys, counts, n = count_kmers_oriented(files, orient, k)
        got = t.count_reads(paths, orient)
        assert got == (n, len(keys), int((counts >= 2).sum())), orient
        assert got[2] > 1000
        _check_lookups(t, keys, counts, _probe(keys, k))
    keys, counts, n = count_kmers_oriented(files, [SENSE, SENSE], k)
    old = api.Talc(api.default_params(k))
    assert old.count_reads(paths) == t.count_reads(paths, [SENSE, SENSE])
    probe = _probe(keys, k, 1)
    for x, y in zip(old.lookup(probe), t.lookup(probe)):
        assert np.array_equal(x, y)
    with pytest.raises(api.TalcError):
        t.count_reads(paths, [SENSE, 3])
    with pytest.raises(api.TalcError):  # too small a counting table is an error in every mode
        t.count_reads(paths, [BOTH, BOTH], expected_distinct=1000)


@gpu
@pytest.mark.parametrize("k", [20, 21, 30, 31])
def test_canonical_dump(api, k, tmp_path):
    """BOTH counting == load_dump_ex(canonical) of the numpy canonical dump of the same reads; load_dump_ex(canonical)
    == load_packed of the interleaved expansion, for a dump that is not canonical too; the cache flags"""
    seqs = _pool_reads(200 + k, 3000, k)
    write_fastq(tmp_path / "a.fq", seqs)
    t = api.Talc(api.default_params(k))
    _, _, kept = t.count_reads([str(tmp_path / "a.fq")], [BOTH])
    ck, cc = canonical_counts(seqs, k)
    perm = np.random.default_rng(k).permutation(len(ck))  # jellyfish dumps in hash order
    api.write_dump(str(tmp_path / "can.dump"), ck[perm], cc[perm], k)
    d = api.Talc(api.default_params(k))
    assert d.load_dump(str(tmp_path / "can.dump"), canonical=True) == (len(ck), kept)
    keys, counts, _ = count_kmers_oriented([seqs], [BOTH], k)
    probe = _probe(keys, k)
    for x, y in zip(t.lookup(probe), d.lookup(probe)):
        assert np.array_equal(x, y)
    # a dump that is not canonical: reverse complements on lines of their own, repeated lines, counts below MIN_COUNT
    rng = np.random.default_rng(k + 1)
    pick = rng.integers(0, len(ck), 500)
    nk = np.concatenate([ck[:2000], revcomp_keys(ck[pick], k), ck[pick[:100]], ck[2000:]])
    nc = np.concatenate([cc[:2000], rng.integers(1, 9, 600), cc[2000:]]).astype(np.int64)
    api.write_dump(str(tmp_path / "mixed.dump"), nk, nc, k)
    assert d.load_dump(str(tmp_path / "mixed.dump"), canonical=True)[0] == len(nk)
    p = api.Talc(api.default_params(k))
    ek, ec = expand_canonical(nk, nc, k)
    assert p.load_packed(ek, ec) == d.table_info()["entries"] == len(table_from_dump(ek, ec)[0])
    probe = _probe(nk, k, 2)
    for x, y in zip(p.lookup(probe), d.lookup(probe)):
        assert np.array_equal(x, y)
    # the cache: flags recorded at byte 36 of the header, checked by load_cache_for(_ex)
    dump = str(tmp_path / "can.dump")
    d.load_dump(dump, canonical=True)
    d.table_save(str(tmp_path / "can.bin"))
    d2 = api.Talc(api.default_params(k))
    d2.load_dump(dump)
    d2.table_save(str(tmp_path / "plain.bin"))
    hdr = lambda f: open(tmp_path / f, "rb").read(40)[36:40]
    assert hdr("can.bin") == b"\1\0\0\0" and hdr("plain.bin") == b"\0\0\0\0"
    u = api.Talc(api.default_params(k))
    with pytest.raises(api.TalcError, match=r"\(-7\)"):
        u.table_load_cache_for(str(tmp_path / "can.bin"), dump)
    with pytest.raises(api.TalcError, match=r"\(-7\)"):
        u.table_load_cache_for(str(tmp_path / "plain.bin"), dump, canonical=True)
    assert u.table_load_cache_for(str(tmp_path / "can.bin"), dump, canonical=True) == d.table_info()["entries"]
    for x, y in zip(u.lookup(probe), d.lookup(probe)):
        assert np.array_equal(x, y)
    assert u.table_load_cache_for(str(tmp_path / "plain.bin"), dump) == d2.table_info()["entries"]
    assert u.table_load_cache(str(tmp_path / "can.bin")) == d.table_info()["entries"]
    # a copy carries the flag
    v = api.Talc(api.default_params(k))
    api.table_copy(v, d)
    v.table_save(str(tmp_path / "copy.bin"))
    assert hdr("copy.bin") == b"\1\0\0\0"
    assert u.table_load_cache_for(str(tmp_path / "copy.bin"), dump, canonical=True) == d.table_info()["entries"]
    # a cache whose flags word is 0 (every cache written before the flags existed) is a directional one
    raw = bytearray(open(tmp_path / "can.bin", "rb").read())
    raw[36:40] = b"\0\0\0\0"
    open(tmp_path / "old.bin", "wb").write(bytes(raw))
    assert u.table_load_cache_for(str(tmp_path / "old.bin"), dump) == d.table_info()["entries"]


@gpu
@pytest.mark.parametrize("name", ["c1", "c3", "c5"])
def test_canonical_table_corrects_as_the_oracle(api, name, tmp_path):
    """correction with a table loaded from a dump read as canonical == the oracle on the expanded dump: bytes,
    offsets, status and every shared counter (c3 with junctions)"""
    from oracle import pyoracle as po
    case = get_case(name)
    k = case.cfg.k
    api.write_dump(str(tmp_path / "sr.dump"), case.keys, case.counts, k)
    j = None
    if case.jkeys is not None:
        j = str(tmp_path / "j.dump")
        api.write_dump(j, case.jkeys, case.jcounts, k)
    t = api.Talc(api.default_params(k))
    t.load_dump(str(tmp_path / "sr.dump"), j, canonical=True)
    ek, ec = expand_canonical(case.keys, case.counts, k)
    ot = po.OracleTable(po.make_params(k=k)).build_packed(ek, ec, case.jkeys, case.jcounts)
    assert t.table_info()["entries"] == ot.size() > len(table_from_dump(case.keys, case.counts)[0])
    o_out, o_off, o_st, o_ctr, _ = ot.correct(case.reads, case.off, threads=8)
    out, off, st, ctr = t.correct(case.reads, case.off)
    assert np.array_equal(st, o_st) and np.array_equal(off, o_off) and np.array_equal(out, o_out)
    diff = {c: (o_ctr[c], ctr[c]) for c in SHARED if o_ctr[c] != ctr[c]}
    assert not diff, diff


def _fragments(case, n, seed):
    """paired reads of fr-firststrand (dUTP) fragments of the case's transcripts: R1 = the reverse complement of the
    fragment's 3' end, R2 = its 5' end (sense); and the sense pieces they come from"""
    rng = np.random.default_rng(seed)
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)
    tb, toff = case.w.t_bases.numpy(), case.w.t_off.numpy()
    r1, r2 = [], []
    for _ in range(n):
        t = int(rng.integers(0, len(toff) - 1))
        a, b = int(toff[t]), int(toff[t + 1])
        F = min(b - a, int(rng.integers(150, 400)))
        p = int(rng.integers(a, b - F + 1))
        frag = letters[tb[p:p + F]].tobytes()
        L = min(F, int(rng.integers(60, 126)))
        r2.append(_mutate(rng, frag[:L], extras=False))
        r1.append(rc(_mutate(rng, frag[F - L:], extras=False)))
    return r1, r2


@gpu
def test_fr_firststrand_table_is_the_sense_table(api, case_c1, tmp_path):
    """fr-firststrand pairs ([ANTISENSE, SENSE]) give the table SENSE counting gives on the fragments' sense pieces, and
    correct as the oracle on that table; an unstranded count of the same pairs holds both strands, so talc_orient_batch
    finds every long read equally on both (found_fwd == found_rc, strand 0)"""
    from oracle import pyoracle as po
    case = case_c1
    k = case.cfg.k
    r1, r2 = _fragments(case, 6000, 3)
    write_fastq(tmp_path / "r1.fq", r1)
    write_fasta_crlf(tmp_path / "r2.fa", r2)
    write_fastq(tmp_path / "sense.fq", [rc(s) for s in r1] + r2)
    pe = [str(tmp_path / "r1.fq"), str(tmp_path / "r2.fa")]
    t = api.Talc(api.default_params(k))
    s = api.Talc(api.default_params(k))
    got = t.count_reads(pe, LIBTYPES["fr-firststrand"])
    assert got == s.count_reads([str(tmp_path / "sense.fq")])
    keys, counts, n = count_kmers_oriented([[rc(x) for x in r1] + r2], [SENSE], k)
    assert got == (n, len(keys), int((counts >= 2).sum()))
    probe = _probe(keys, k)
    for x, y in zip(t.lookup(probe), s.lookup(probe)):
        assert np.array_equal(x, y)
    _check_lookups(t, keys, counts, probe)
    ot = po.OracleTable(po.make_params(k=k)).build_packed(keys, counts)
    o_out, o_off, o_st, o_ctr, _ = ot.correct(case.reads, case.off, threads=8)
    out, off, st, ctr = t.correct(case.reads, case.off)
    assert (o_st == 0).sum() > 20
    assert np.array_equal(st, o_st) and np.array_equal(off, o_off) and np.array_equal(out, o_out)
    diff = {c: (o_ctr[c], ctr[c]) for c in SHARED if o_ctr[c] != ctr[c]}
    assert not diff, diff
    # a table that holds both strands: no read prefers either (the long reads hold no U)
    t.count_reads(pe, LIBTYPES["unstranded"])
    strand, ff, fr = t.orient(case.reads, case.off)
    assert not strand.any() and np.array_equal(ff, fr) and (ff > 0).sum() > 100


# ---- the command line
def _cli_inputs(tmp_path, seed=5):
    """long reads and junctions of a small c1-like workload, fr-firststrand pairs of its transcripts with N, U-free"""
    from talc_b200 import synth
    cfg = synth.baseline_config(1, 0.05)
    cfg.n_reads = 60
    w = synth.make_workload(cfg)

    class W:
        pass
    case = W()
    case.w = w
    r1, r2 = _fragments(case, 5000, seed)
    rng = np.random.default_rng(seed)
    for lst in (r1, r2):
        for i in rng.integers(0, len(lst), 200):
            s = bytearray(lst[i])
            s[int(rng.integers(0, len(s)))] = ord("N")
            lst[i] = bytes(s).lower() if i % 3 == 0 else bytes(s)
    write_fastq(tmp_path / "r1.fq", r1)
    write_fasta_crlf(tmp_path / "r2.fa", r2)
    reads, off = w.reads.numpy(), w.read_off.numpy()
    with open(tmp_path / "reads.fa", "wb") as f:
        for i in range(len(off) - 1):
            f.write(b">lr%d\n" % i + reads[int(off[i]):int(off[i + 1])].tobytes() + b"\n")
    synth.write_dump(str(tmp_path / "j.dump"), w.jkeys, w.jcounts, cfg.k)
    return cfg.k, r1, r2


def _same_files(tmp_path, a, b, exts=(".fa", ".log", ".stats_basics.txt")):
    for ext in exts:
        pa, pb = tmp_path / (a + ext), tmp_path / (b + ext)
        ra = open(pa, "rb").read() if os.path.exists(pa) else None
        rb = open(pb, "rb").read() if os.path.exists(pb) else None
        assert ra == rb, (a, b, ext)


@gpu
def test_cli_sr_reads_is_the_dump_of_its_counts(api, tmp_path):
    """For every --SRLibType, `talc --SRReads r1 --SRReads2 r2` writes the .fa, .log and stats header of `talc --SRCounts`
    on the numpy dump of the same oriented counts and of the oracle's command line on that dump, whatever the batch
    size; single-end files follow R1; --SRCanonical matches the oracle on the expanded dump; --SRExpected too small
    exits 2; --strand auto on a table of both strands prints a note."""
    from oracle import pyoracle as po
    from talc_b200 import build
    k, r1, r2 = _cli_inputs(tmp_path)
    cli = build.build_cli()
    common = ["-k", str(k), "--junctions", str(tmp_path / "j.dump")]
    run = lambda exe, *a: subprocess.run([exe, str(tmp_path / "reads.fa")] + common + list(a), cwd=tmp_path,
                                         capture_output=True, text=True)
    sr = ["--SRReads", str(tmp_path / "r1.fq"), "--SRReads2", str(tmp_path / "r2.fa")]
    for lt, orient in LIBTYPES.items():
        keys, counts, n = count_kmers_oriented([r1, r2], orient, k)
        api.write_dump(str(tmp_path / (lt + ".dump")), keys, counts, k)
        p = run(cli, *sr, "--SRLibType", lt, "-o", "gpu_" + lt)
        assert p.returncode == 0, p.stderr
        line = [l for l in p.stdout.split("\n") if l.startswith("[TALC]: counted ")]
        assert len(line) == 1 and ("counted %d k-mer occurrences" % n) in line[0], p.stdout
        assert ("%d distinct, %d with count >= 2" % (len(keys), int((counts >= 2).sum()))) in line[0]
        assert run(cli, "--SRCounts", str(tmp_path / (lt + ".dump")), "-o", "dump_" + lt).returncode == 0
        assert run(po.BIN, "--SRCounts", str(tmp_path / (lt + ".dump")), "-t", "1", "--oracle-table", "hash",
                   "-o", "ora_" + lt).returncode == 0
        _same_files(tmp_path, "gpu_" + lt, "dump_" + lt)
        _same_files(tmp_path, "gpu_" + lt, "ora_" + lt)
        assert open(tmp_path / ("gpu_" + lt + ".config.txt")).read().replace("gpu_" + lt, "X") == \
            open(tmp_path / ("ora_" + lt + ".config.txt")).read().replace("ora_" + lt, "X")
        assert run(cli, *sr, "--SRLibType", lt, "-o", "b7_" + lt, "--batch-reads", "7", "-t", "3").returncode == 0
        _same_files(tmp_path, "gpu_" + lt, "b7_" + lt, (".fa", ".log"))
    # asis is the default; the long reads do find the table
    assert run(cli, *sr, "-o", "default").returncode == 0
    _same_files(tmp_path, "gpu_asis", "default")
    assert open(tmp_path / "gpu_fr-firststrand.fa", "rb").read() != open(tmp_path / "gpu_fr-secondstrand.fa", "rb").read()
    # a single-end file follows R1
    keys, counts, _ = count_kmers_oriented([r1], [ANTISENSE], k)
    api.write_dump(str(tmp_path / "se.dump"), keys, counts, k)
    assert run(cli, "--SRReads", str(tmp_path / "r1.fq"), "--SRLibType", "fr-firststrand", "-o", "se").returncode == 0
    assert run(po.BIN, "--SRCounts", str(tmp_path / "se.dump"), "-t", "1", "--oracle-table", "hash", "-o", "ora_se").returncode == 0
    _same_files(tmp_path, "se", "ora_se")
    # --SRCanonical: the oracle on the expanded dump; it is also the unstranded table
    ck, cc = canonical_counts(r1 + r2, k)
    api.write_dump(str(tmp_path / "can.dump"), ck, cc, k)
    api.write_dump(str(tmp_path / "exp.dump"), *expand_canonical(ck, cc, k), k)
    assert run(cli, "--SRCounts", str(tmp_path / "can.dump"), "--SRCanonical", "-o", "can").returncode == 0
    assert run(po.BIN, "--SRCounts", str(tmp_path / "exp.dump"), "-t", "1", "--oracle-table", "hash", "-o", "ora_can").returncode == 0
    _same_files(tmp_path, "can", "ora_can")
    _same_files(tmp_path, "can", "gpu_unstranded")
    assert run(cli, "--SRCounts", str(tmp_path / "can.dump"), "--SRCanonical", "-o", "can5", "--batch-reads", "5",
               "--tableCache", str(tmp_path / "t.bin")).returncode == 0
    p = run(cli, "--SRCounts", str(tmp_path / "can.dump"), "--SRCanonical", "-o", "can6", "--tableCache", str(tmp_path / "t.bin"))
    assert p.returncode == 0 and "rebuilding" not in p.stdout
    p = run(cli, "--SRCounts", str(tmp_path / "can.dump"), "-o", "notcan", "--tableCache", str(tmp_path / "t.bin"))
    assert p.returncode == 0 and "rebuilding" in p.stdout
    for other in ("can5", "can6"):
        _same_files(tmp_path, "can", other, (".fa", ".log"))
    # too small a counting table: exit 2 with the library's message
    p = run(cli, *sr, "--SRExpected", "1000", "-o", "small")
    assert p.returncode == 2 and "counting table is full" in p.stderr
    # --strand auto on a table of both strands: a note, every read '+'
    p = run(cli, *sr, "--SRLibType", "unstranded", "--strand", "auto", "-o", "auto")
    assert p.returncode == 0 and "[TALC]: note: the k-mer table holds both strands" in p.stdout
    assert b"\t-\n" not in open(tmp_path / "auto.strand.txt", "rb").read()
    _same_files(tmp_path, "auto", "gpu_unstranded", (".fa", ".log"))
    p = run(cli, *sr, "--SRLibType", "fr-firststrand", "--strand", "auto", "-o", "auto2")
    assert p.returncode == 0 and "note:" not in p.stdout


@gpu
def test_cli_sr_reads_two_gpus_equals_one(api, tmp_path):
    import torch
    from talc_b200 import build
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    k, _, _ = _cli_inputs(tmp_path)
    cli = build.build_cli()
    args = [str(tmp_path / "reads.fa"), "-k", str(k), "--SRReads", str(tmp_path / "r1.fq"), "--SRReads2",
            str(tmp_path / "r2.fa"), "--SRLibType", "fr-firststrand"]
    run = lambda *a: subprocess.call([cli] + args + list(a), cwd=tmp_path, stdout=subprocess.DEVNULL)
    assert run("-o", "one", "--gpus", "1") == 0
    assert run("-o", "two", "--gpus", "2", "--batch-reads", "9") == 0
    assert run("-o", "peer", "--gpus", "2", "--batch-reads", "7", "--replicate", "peer") == 0
    for other in ("two", "peer"):
        _same_files(tmp_path, "one", other, (".fa", ".log"))
