"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on the same seeded
inputs.  Integer / byte work, so the bar is bit-exact: identical corrected sequences, identical per-read
status (= identical failed-read log), identical algorithmic counters."""
import os

import numpy as np
import pytest

from conftest import ROOT, have_gpu

pytestmark = pytest.mark.gpu

SHARED = ["lookups_seg", "lookups_deg", "lookups_walk", "steps_inner", "steps_border", "frontier_sum", "cells_nw",
          "cells_lcs", "cells_ovl", "cells_xdrop", "gaps", "gaps_bridged", "gap_attempts", "borders",
          "borders_corrected", "ev_gardening", "ev_bridge", "ev_edge", "ev_cycle", "bases_out"]


@pytest.fixture(scope="module")
def api():
    if not have_gpu():
        pytest.fail("GPU tests selected but no CUDA device is visible")
    from talc_b200 import api as _api
    return _api


def _ctx(api, case, **kw):
    t = api.Talc(api.default_params(case.cfg.k, **kw))
    t.load_packed(case.keys, case.counts, case.jkeys, case.jcounts)
    return t


def _assert_same(case, out, off, status, ctr=None):
    assert np.array_equal(status, case.o_status), "per-read status (failed-read log) differs"
    bad = [r for r in range(len(case.off) - 1)
           if out[int(off[r]):int(off[r + 1])].tobytes() != case.oracle_read(r)]
    assert not bad, "corrected sequence differs for reads %s" % bad[:10]
    if ctr is not None:
        diff = {k: (case.o_ctr[k], ctr[k]) for k in SHARED if case.o_ctr[k] != ctr[k]}
        assert not diff, "algorithmic counters differ: %s" % diff


def test_table_matches_oracle(api, case_c3):
    case = case_c3
    t = _ctx(api, case)
    info = t.table_info()
    assert info["entries"] == case.otable.size()
    from talc_b200 import synth
    rng = np.random.default_rng(0)
    idx = rng.integers(0, len(case.keys), 4000)
    probe = np.concatenate([case.keys[idx], rng.integers(0, 1 << 42, 500).astype(np.uint64)])
    cnt, col, found = t.lookup(probe)
    for i, key in enumerate(probe):
        f, c, l = case.otable.lookup(synth.unpack_kmer(int(key), case.cfg.k))
        assert (bool(found[i]), int(cnt[i]), int(col[i])) == (f, c, l)
    assert (col > 0).any(), "junction colours must be exercised"


def test_table_cache_round_trip(api, case_c3, tmp_path):
    """talc_table_save / talc_table_load_cache (SURVEY row f1): the cached table answers every look-up like the
    table built from the dump (junction colours included), corrects to the same bytes, and a cache made for
    another k-mer size is refused."""
    case = case_c3
    t = _ctx(api, case)
    path = str(tmp_path / "table.bin")
    t.table_save(path)
    t2 = api.Talc(api.default_params(case.cfg.k))
    assert t2.table_load_cache(path) == t.table_info()["entries"]
    probe = np.concatenate([case.keys[:5000], case.keys[:5000] ^ np.uint64(5)])
    c1, l1, f1 = t.lookup(probe)
    c2, l2, f2 = t2.lookup(probe)
    assert np.array_equal(c1, c2) and np.array_equal(l1, l2) and np.array_equal(f1, f2)
    out, off, st, ctr = t2.correct(case.reads, case.off)
    _assert_same(case, out, off, st, ctr)
    t3 = api.Talc(api.default_params(case.cfg.k + 2))
    with pytest.raises(api.TalcError):
        t3.table_load_cache(path)


def test_coverage_matches_oracle(api, case_c1):
    case = case_c1
    t = _ctx(api, case)
    cov = t.coverage(case.reads, case.off)
    pos = 0
    for r in range(40):
        ocnt, _ = case.otable.coverage(case.read(r))
        assert np.array_equal(cov[pos:pos + len(ocnt)], ocnt)
        pos += len(ocnt)


def test_correction_config1(api, case_c1):
    t = _ctx(api, case_c1)
    out, off, st, ctr = t.correct(case_c1.reads, case_c1.off)
    _assert_same(case_c1, out, off, st, ctr)


def test_correction_junctions_config3(api, case_c3):
    t = _ctx(api, case_c3)
    out, off, st, ctr = t.correct(case_c3.reads, case_c3.off)
    _assert_same(case_c3, out, off, st, ctr)


def test_correction_stress_config5(api, case_c5):
    """k=30, 15% errors, low-complexity inserts: frontier > 50 aborts, gardening with ties."""
    assert case_c5.o_ctr["ev_gardening"] > 0 and case_c5.o_ctr["ev_frontier_over50"] > 0
    t = _ctx(api, case_c5)
    out, off, st, ctr = t.correct(case_c5.reads, case_c5.off)
    _assert_same(case_c5, out, off, st, ctr)


def test_second_tier_is_result_neutral(api, case_c1):
    """A tiny first-tier scratch slice pushes most reads through the second tier; bytes must not change."""
    t = _ctx(api, case_c1)
    t.set_scratch(tier1_bytes=6 * 1024)
    out, off, st, ctr = t.correct(case_c1.reads, case_c1.off)
    assert ctr["reads_second_tier"] > 0
    _assert_same(case_c1, out, off, st, ctr)


def test_batch_is_idempotent_and_order_independent(api, case_c1):
    case = case_c1
    t = _ctx(api, case)
    out1, off1, st1, _ = t.correct(case.reads, case.off)
    out2, off2, st2, _ = t.correct(case.reads, case.off)
    assert np.array_equal(out1, out2) and np.array_equal(off1, off2) and np.array_equal(st1, st2)
    # reversed read order gives the same per-read answers
    n = len(case.off) - 1
    parts = [case.reads[int(case.off[r]):int(case.off[r + 1])] for r in range(n)][::-1]
    roff = np.zeros(n + 1, dtype=np.uint64)
    roff[1:] = np.cumsum([len(p) for p in parts])
    out3, off3, st3, _ = t.correct(np.concatenate(parts), roff)
    for r in range(n):
        a = out1[int(off1[r]):int(off1[r + 1])].tobytes()
        b = out3[int(off3[n - 1 - r]):int(off3[n - r])].tobytes()
        assert a == b


def test_edge_cases(api, case_c1):
    """Empty batch, empty read, reads <= K, reads with N, lower case, all-unknown read."""
    case = case_c1
    t = _ctx(api, case)
    k = case.cfg.k
    base = case.read(0)
    reads = [b"", b"ACGT", base[:k], base[:k + 1], base.lower(), base[:200] + b"NNNN" + base[200:], b"N" * 300,
             base[:90] + b"R" + base[91:]]
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(r) for r in reads])
    data = np.frombuffer(b"".join(reads), dtype=np.uint8)
    out, ooff, st, _ = t.correct(data, off)
    o_out, o_off, o_st, _, _ = case.otable.correct(data, off, threads=1)
    assert np.array_equal(st, o_st)
    assert np.array_equal(out, o_out) and np.array_equal(ooff, o_off)
    e_out, e_off, e_st, _ = t.correct(np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.uint64))
    assert len(e_out) == 0 and len(e_st) == 0


def test_alignment_primitives_on_device(api, case_c1):
    from oracle import pyoracle as po
    case = case_c1
    t = _ctx(api, case)
    rng = np.random.default_rng(7)

    def mutate(s: bytes, rate: float) -> bytes:
        out = bytearray()
        for ch in s:
            u = rng.random()
            if u < rate * 0.4:
                out.append(rng.choice(list(b"ACGT")))
            elif u < rate * 0.7:
                out.append(ch)
                out.append(rng.choice(list(b"ACGT")))
            elif u < rate:
                continue
            else:
                out.append(ch)
        return bytes(out) or b"A"

    a_list, b_list = [], []
    for i in range(120):
        n = int(rng.integers(1, 700))
        s = bytes(rng.choice(list(b"ACGT"), n).tolist())
        a = mutate(s, 0.15)
        if i % 7 == 0:
            a = a[: len(a) // 2] + b"N" + a[len(a) // 2:]
        a_list.append(a)
        b_list.append(s)
    for n in (2300, 3100, 4200):  # more than 32 blocks of 64 rows: the striped path
        s = bytes(rng.choice(list(b"ACGT"), n).tolist())
        a_list.append(mutate(s, 0.12))
        b_list.append(s)
    nw = t.test_align(0, a_list, b_list)
    lcs = t.test_align(1, a_list, b_list)
    ovl = t.test_align(2, a_list, b_list)
    fused = t.test_align(5, a_list, b_list)
    for i, (a, b) in enumerate(zip(a_list, b_list)):
        assert nw[i] == po.nw(a, b)
        assert lcs[i] == po.lcs(a, b)
        assert ovl[i] == po.overlap(a, b, True)
        assert (int(fused[i][0]), int(fused[i][1])) == (nw[i], lcs[i])
    # seed-and-extension (X-drop end positions + NW of the extensions), both directions
    k = case.cfg.k
    refs, cands = [], []
    for i in range(80):
        n = int(rng.integers(k + 5, 400))
        s = bytes(rng.choice(list(b"ACGT"), n).tolist())
        c = s[:k] + mutate(s[k:], 0.12)
        if i % 3 == 0:
            c = c[: max(k + 1, len(c) // 2)]
        refs.append(s)
        cands.append(c if len(c) >= k else s)
    for x in (-1, 0, 2, 4, 9, 30):
        res = t.test_align(3, refs, cands, aux=x, aux2=1)
        for i, (r, c) in enumerate(zip(refs, cands)):
            re_, ce_, pos, sc, stop = po.seed_extend(r, c, x, True, k)
            assert tuple(res[i]) == (re_, ce_, int(sc), int(stop)), (i, x)
        # LEFT: the strings end in the shared anchor k-mer (Trail.cpp:383-391 seeds at their last K bases) and the
        # device works on the reversed strings (walk order).  The anchor is common to both strings by construction
        # in the pipeline, and the device relies on it: the score is read off the X-drop end cell.
        res = t.test_align(3, refs, cands, aux=x, aux2=0)
        for i, (r, c) in enumerate(zip(refs, cands)):
            re_, ce_, pos, sc, stop = po.seed_extend(r[::-1], c[::-1], x, False, k)
            assert tuple(res[i]) == (re_, ce_, int(sc), int(stop)), (i, x)


def test_config2_scale_sampled_parity_and_split_invariance(api):
    """A config-2-like workload two orders of magnitude above the other cases (0.76 M-entry table, 6 000 reads): the
    oracle checks a random sample of reads byte for byte, and the whole batch is checked through properties that do
    not need the oracle -- correcting the batch in two halves, or in reverse order, changes no read and no counter
    (the processing order inside the kernel is cost-driven and must not leak into the results)."""
    from oracle import pyoracle as po
    from talc_b200 import synth
    cfg = synth.baseline_config(2, 0.02)
    cfg.n_reads = 6000
    w = synth.make_workload(cfg)
    keys, counts = w.keys.numpy().astype(np.uint64), w.counts.numpy().astype(np.int64)
    reads, off = w.reads.numpy(), w.read_off.numpy().astype(np.uint64)
    n = len(off) - 1
    t = api.Talc(api.default_params(cfg.k))
    t.load_packed(keys, counts)
    out, ooff, st, ctr = t.correct(reads, off)
    assert ctr["reads_ok"] > 0.95 * n and ctr["gaps_bridged"] > 0

    def sub(idx):
        parts = [reads[int(off[r]):int(off[r + 1])] for r in idx]
        so = np.zeros(len(idx) + 1, dtype=np.uint64)
        so[1:] = np.cumsum([len(x) for x in parts])
        return np.concatenate(parts), so

    # (1) oracle on a sample
    rng = np.random.default_rng(4)
    sample = sorted(rng.choice(n, 150, replace=False).tolist())
    ot = po.OracleTable(po.make_params(k=cfg.k)).build_packed(keys, counts)
    sr, so = sub(sample)
    o_out, o_off, o_st, _, _ = ot.correct(sr, so, threads=8)
    for i, r in enumerate(sample):
        assert st[r] == o_st[i], r
        assert out[int(ooff[r]):int(ooff[r + 1])].tobytes() == o_out[int(o_off[i]):int(o_off[i + 1])].tobytes(), r
    # (2) two halves == whole, counters add up
    half = n // 2
    a_r, a_o = sub(range(half))
    b_r, b_o = sub(range(half, n))
    oa, fa, sa, ca = t.correct(a_r, a_o)
    ob, fb, sb, cb = t.correct(b_r, b_o)
    assert np.array_equal(np.concatenate([sa, sb]), st)
    assert np.array_equal(np.concatenate([oa[: int(fa[-1])], ob[: int(fb[-1])]]), out[: int(ooff[-1])])
    for k2 in SHARED:
        assert ca[k2] + cb[k2] == ctr[k2], k2
    # (3) reversed input order == reversed output
    rev = list(range(n - 1, -1, -1))
    r_r, r_o = sub(rev)
    orr, frr, srr, crr = t.correct(r_r, r_o)
    assert np.array_equal(srr, st[::-1])
    for i in (0, 1, n // 3, n - 1):
        r = rev[i]
        assert orr[int(frr[i]):int(frr[i + 1])].tobytes() == out[int(ooff[r]):int(ooff[r + 1])].tobytes()
    assert {k2: crr[k2] for k2 in SHARED} == {k2: ctr[k2] for k2 in SHARED}


def test_xdrop_register_band_on_device(api, case_c1):
    """The register-resident X-drop (csrc/xdrop.cuh, S = 1, 2, 4, 8 diagonals per lane, scalar beyond 255) against the
    oracle's cell-by-cell restatement: end positions for every drop-off, sequence ends reached, N, low complexity."""
    from oracle import pyoracle as po
    t = _ctx(api, case_c1)
    rng = np.random.default_rng(17)
    qs, ds = [], []
    for i in range(1500):
        n = int(rng.integers(1, 30 if i % 3 == 0 else 400))
        alpha = list(b"AC") if i % 5 == 0 else list(b"ACGT")
        s = bytes(rng.choice(alpha, n).tolist())
        rate = float(rng.random()) * 0.3
        b = bytearray()
        for ch in s:
            u = rng.random()
            if u < rate / 3:
                continue
            b.append(int(rng.choice(alpha)) if u < 2 * rate / 3 else ch)
            if rng.random() < rate / 3:
                b.append(int(rng.choice(alpha)))
        b = bytes(b) or b"A"
        if i % 4 == 0:
            b = b[: int(rng.integers(1, len(b) + 1))]
        if i % 11 == 0:
            b += b"A" * int(rng.integers(0, 40))
        if i % 37 == 0:
            s = s[: n // 2] + b"N" + s[n // 2:]
        if i % 2:
            s, b = b, s
        qs.append(s)
        ds.append(b)
    for x in (-1, 0, 1, 2, 3, 5, 8, 13, 21, 31, 32, 47, 63, 64, 100, 127, 128, 200, 255, 256, 300):
        res = t.test_align(4, qs, ds, aux=x)
        for i, (q, d) in enumerate(zip(qs, ds)):
            assert (int(res[i][0]), int(res[i][1])) == po.xdrop(q, d, False, x), (i, x, q, d)


def test_std_sort_replica_on_device(api, case_c1):
    from oracle import pyoracle as po
    t = _ctx(api, case_c1)
    rng = np.random.default_rng(3)
    for n in (1, 2, 5, 16, 17, 33, 64, 100, 207):
        for hi in (2, 4, 50, 10 ** 9):
            keys = rng.integers(0, hi, n)
            assert np.array_equal(t.test_sort(keys), po.std_sort_perm(keys)), (n, hi)
    keys = np.arange(200)[::-1].copy()
    assert np.array_equal(t.test_sort(keys), po.std_sort_perm(keys))


def test_cli_is_a_drop_in(api, tmp_path):
    """The `talc` command line on the GPU writes the same .fa / .log / .config.txt as the oracle's front end
    (reference order: -t 1), from the same text inputs, junction dump included."""
    import os
    import subprocess
    import torch
    from oracle import pyoracle as po
    from talc_b200 import build, synth
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "tiny_case.npz"))
    k = int(g["c3_k"][0])
    synth.write_dump(str(tmp_path / "sr.dump"), torch.from_numpy(g["c3_keys"].astype(np.int64)),
                     torch.from_numpy(g["c3_counts"].astype(np.int64)), k)
    synth.write_dump(str(tmp_path / "j.dump"), torch.from_numpy(g["c3_jkeys"].astype(np.int64)),
                     torch.from_numpy(g["c3_jcounts"].astype(np.int64)), k)
    # reads: wrapped FASTA with one unsolvable read and one short read mixed in, so that the log is exercised
    reads, off = g["c3_reads"], g["c3_off"]
    with open(tmp_path / "reads.fa", "wb") as f:
        for r in range(len(off) - 1):
            s = reads[int(off[r]):int(off[r + 1])].tobytes()
            f.write(b">read_%d some description\n" % r)
            for j in range(0, len(s), 60):
                f.write(s[j:j + 60] + b"\n")
            if r == 3:
                f.write(b">junk\n" + b"ACGT" * 60 + b"\n>tiny\nACGTACGT\n")
    cli = build.build_cli()
    args = [str(tmp_path / "reads.fa"), "--SRCounts", str(tmp_path / "sr.dump"), "--junctions", str(tmp_path / "j.dump"),
            "-k", str(k)]
    assert subprocess.call([cli] + args + ["-o", "gpu", "-t", "4"], cwd=tmp_path, stdout=subprocess.DEVNULL) == 0
    assert subprocess.call([po.BIN] + args + ["-o", "cpu", "-t", "1", "--oracle-table", "hash"], cwd=tmp_path,
                           stdout=subprocess.DEVNULL) == 0
    for ext in (".fa", ".log", ".stats_basics.txt"):
        assert open(tmp_path / ("gpu" + ext), "rb").read() == open(tmp_path / ("cpu" + ext), "rb").read(), ext
    a = open(tmp_path / "gpu.config.txt").read().replace("gpu", "X")
    b = open(tmp_path / "cpu.config.txt").read().replace("cpu", "X")
    assert a == b
    assert b"junk" in open(tmp_path / "gpu.log", "rb").read()


def _write_case_files(tmp_path, g, fastq=False):
    import torch
    from talc_b200 import synth
    k = int(g["c3_k"][0])
    synth.write_dump(str(tmp_path / "sr.dump"), torch.from_numpy(g["c3_keys"].astype(np.int64)),
                     torch.from_numpy(g["c3_counts"].astype(np.int64)), k)
    synth.write_dump(str(tmp_path / "j.dump"), torch.from_numpy(g["c3_jkeys"].astype(np.int64)),
                     torch.from_numpy(g["c3_jcounts"].astype(np.int64)), k)
    reads, off = g["c3_reads"], g["c3_off"]
    with open(tmp_path / "reads.fa", "wb") as f, open(tmp_path / "reads.fq", "wb") as q:
        for r in range(len(off) - 1):
            s = reads[int(off[r]):int(off[r + 1])].tobytes()
            f.write(b">read_%d\n" % r + s + b"\n")
            q.write(b"@read_%d\n" % r + s + b"\n+\n" + b"I" * len(s) + b"\n")
            if r == 2:
                f.write(b">tiny\nACGTACGT\n>junk\n" + b"ACGT" * 60 + b"\n")
                q.write(b"@tiny\nACGTACGT\n+\nIIIIIIII\n@junk\n" + b"ACGT" * 60 + b"\n+\n" + b"I" * 240 + b"\n")
    return k


def test_cli_streams_batches_fastq_and_stats_rows(api, tmp_path):
    """Row f2 / f4: the streamed command line gives the same files whether the input goes through in one batch or in
    many small ones (--batch-reads 7: batch boundaries, the ring of slots, the in-order writer), FASTQ input equals
    FASTA input, and --readStats appends the per-read rows of Read.cpp:418-433 (checked against the oracle)."""
    import os
    import subprocess
    from oracle import pyoracle as po
    from talc_b200 import build
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "tiny_case.npz"))
    k = _write_case_files(tmp_path, g)
    cli = build.build_cli()
    common = ["--SRCounts", str(tmp_path / "sr.dump"), "--junctions", str(tmp_path / "j.dump"), "-k", str(k)]
    run = lambda reads, *a: subprocess.call([cli, str(tmp_path / reads)] + common + list(a), cwd=tmp_path, stdout=subprocess.DEVNULL)
    assert run("reads.fa", "-o", "one") == 0
    assert run("reads.fa", "-o", "many", "--batch-reads", "7", "-t", "3") == 0
    assert run("reads.fq", "-o", "fq", "--batch-reads", "5") == 0
    assert run("reads.fa", "-o", "stats", "--batch-reads", "11", "--readStats") == 0
    one = open(tmp_path / "one.fa", "rb").read()
    assert one.count(b">") == len(g["c3_off"]) - 1 + 2
    for other in ("many", "fq", "stats"):
        assert open(tmp_path / (other + ".fa"), "rb").read() == one, other
        assert open(tmp_path / (other + ".log"), "rb").read() == open(tmp_path / "one.log", "rb").read(), other
    assert not os.path.exists(tmp_path / "one.fa.partial")
    # stats rows: header, then "\n" id raw_length span regions corrected_length per read longer than K
    rows = open(tmp_path / "stats.stats_basics.txt").read().split("\n")
    assert rows[0].startswith("read_name\traw_length") and rows[1] == ""
    rows = [r.split("\t") for r in rows[2:]]
    ot = po.OracleTable(po.make_params(k=k)).build_packed(g["c3_keys"], g["c3_counts"].astype(np.int64), g["c3_jkeys"],
                                                          g["c3_jcounts"].astype(np.int64))
    st = ot.read_stats(g["c3_reads"], g["c3_off"], threads=2)
    by_id = {r[0]: r for r in rows}
    assert "tiny" not in by_id and by_id["junk"][1:] == ["240", "0", "0", "0"]
    off, ooff = g["c3_off"], g["c3_ooff"]
    for r in range(len(off) - 1):
        row = by_id["read_%d" % r]
        corr = int(ooff[r + 1] - ooff[r]) if g["c3_status"][r] == 0 else 0
        assert [int(x) for x in row[1:]] == [int(off[r + 1] - off[r]), int(st[r][0]), int(st[r][1]), corr], r


def test_no_cpu_fallback_on_the_gpu_box(api):
    """With the devices hidden the library must refuse to work, not fall back (run in a child process)."""
    import os
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r)\nfrom talc_b200 import api\n"
            "try:\n    api.Talc(api.default_params(21))\n    print('CREATED')\n"
            "except api.TalcError as e:\n    print('REFUSED', e)\n") % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True).stdout
    assert "REFUSED" in out and "no CPU path" in out


def test_stream_api_matches_single_calls(api, case_c1):
    """talc_stream_*: the same reads cut into uneven batches (one of them empty) come back in submission order with
    the bytes, status and counters of one talc_correct_batch call."""
    case = case_c1
    t = _ctx(api, case)
    out, off, st, ctr = t.correct(case.reads, case.off)
    _assert_same(case, out, off, st, ctr)
    n = len(case.off) - 1
    cuts = [0, 1, 1, 40, 41, 130, n]
    s = t.stream(read_stats=True)
    outs, sts, stats, tot = [], [], [], None
    spans = list(zip(cuts, cuts[1:]))

    def fetch(a, b):
        nonlocal tot
        o, f, x, rs, c = s.next()
        assert len(x) == b - a and len(f) == b - a + 1 and rs.shape == (b - a, 2)
        outs.append(o)
        sts.append(x)
        stats.append(rs)
        tot = c if tot is None else {k2: tot[k2] + c[k2] for k2 in c}

    fetched = 0
    for i, (a, b) in enumerate(spans):  # at most three batches in flight: the ring has four slots
        sub = case.reads[int(case.off[a]):int(case.off[b])]
        s.submit(sub, case.off[a:b + 1] - case.off[a])
        if i - fetched >= 2:
            fetch(*spans[fetched])
            fetched += 1
    assert s.pending() == len(spans) - fetched
    while fetched < len(spans):
        fetch(*spans[fetched])
        fetched += 1
    s.close()
    assert np.array_equal(np.concatenate(outs), out) and np.array_equal(np.concatenate(sts), st)
    assert {k2: tot[k2] for k2 in SHARED} == {k2: ctr[k2] for k2 in SHARED}
    ostats = case.otable.read_stats(case.reads, case.off, threads=4)
    assert np.array_equal(np.concatenate(stats), ostats)


def test_lane_overlaps_batches_with_identical_results(api, case_c1):
    """talc_ctx_create_lane: a context and its lane correct different halves of the reads at the same time from two
    host threads (their kernels overlap on the device); bytes, status and counters equal the one-call result, a lane
    refuses to load a table, and it follows a setting changed on its parent."""
    import threading
    case = case_c1
    t = _ctx(api, case)
    out, off, st, ctr = t.correct(case.reads, case.off)
    _assert_same(case, out, off, st, ctr)
    lane = t.create_lane()
    with pytest.raises(Exception):
        lane.load_packed(np.zeros(1, np.uint64), np.ones(1, np.uint32))
    n = len(case.off) - 1
    h = n // 2
    spans = [(0, h), (h, n)]
    res = [None, None]

    def run(i, c):
        a, b = spans[i]
        for _ in range(3):  # several rounds so that the two threads really run side by side
            res[i] = c.correct(case.reads[int(case.off[a]):int(case.off[b])], case.off[a:b + 1] - case.off[a])

    for shape in ((0, 0, 0), (1, 64, 7)):  # default execution shape, then the split shape set on the parent only
        if shape[0]:
            t.set_exec(*shape)
        th = [threading.Thread(target=run, args=(0, t)), threading.Thread(target=run, args=(1, lane))]
        for x in th:
            x.start()
        for x in th:
            x.join()
        assert res[0] is not None and res[1] is not None
        assert np.array_equal(np.concatenate([res[0][0], res[1][0]]), out)
        assert np.array_equal(np.concatenate([res[0][2], res[1][2]]), st)
        tot = {k2: res[0][3][k2] + res[1][3][k2] for k2 in SHARED}
        assert tot == {k2: ctr[k2] for k2 in SHARED}
        if shape[0]:
            assert res[1][3]["rounds"] > 0  # the lane ran the split shape although only the parent was told to
    lane.close()
    t.close()


def test_gpu_dump_parser_semantics(api, case_c3, tmp_path):
    """Row f1: the dump text is parsed on the GPU.  (1) line semantics of buildCDBG on a hand-made file (first line
    wins, MIN_COUNT filter, malformed lines, lower case, CR LF, trailing tokens, negative and out-of-range counts,
    k-mers of the wrong length, no final newline) against the oracle reading the same file; (2) a whole workload written
    as text builds the table load_packed builds, the host parser of round 1 builds the same one, and the reads
    correct to the oracle's bytes."""
    from oracle import pyoracle as po
    k = 5
    text = ("ACGTA 5\nACGTA 9\nCCCCC 7\r\nGGGGA 1\n  TTTTT\t3 trailing tokens\nbad_line\n\nAAAAA 4\nTACGT 6\nacgtc 8\n"
            "ACG 9\nACGTAC 9\nACGTN 9\nGGGGG x9\nGGGGT -1\nGGGTT 99999999999\nGGTTT +12\nGTTTT 12abc\nCATCA 2")
    (tmp_path / "d.dump").write_text(text)
    (tmp_path / "j.dump").write_text("ACGTA 2\nTACGT 4\nACGTA 3\nAAAAA 5\nCCCCC 10000\nACGTC 0\njunk\nCATCA 17\n")
    t = api.Talc(api.default_params(k))
    nl, nk = t.load_dump(str(tmp_path / "d.dump"), str(tmp_path / "j.dump"))
    h = api.Talc(api.default_params(k))
    assert h.load_dump_host(str(tmp_path / "d.dump"), str(tmp_path / "j.dump")) == (nl, nk)
    ot = po.OracleTable(po.make_params(k=k)).load_dump(str(tmp_path / "d.dump"), str(tmp_path / "j.dump"))
    # the reference's map also holds 'ACG', 'ACGTAC' and 'ACGTN' (no length or alphabet check, Jellyfish.cpp:262): keys
    # that no 5-mer of a read can ever equal; the 2-bit table drops them
    assert nk == ot.size() - 3 == 10
    from itertools import product
    allk = ["".join(x) for x in product("ACGT", repeat=k)]
    keys = np.array([sum("ACGT".index(ch) << (2 * (k - 1 - i)) for i, ch in enumerate(s_)) for s_ in allk], dtype=np.uint64)
    cnt, col, found = t.lookup(keys)
    cnt2, col2, found2 = h.lookup(keys)
    assert np.array_equal(cnt, cnt2) and np.array_equal(col, col2) and np.array_equal(found, found2)
    for i, s_ in enumerate(allk):
        f, c, l = ot.lookup(s_)
        assert (bool(found[i]), int(cnt[i]), int(col[i])) == (f, c, l), s_
    assert int(found.sum()) == nk
    # (2) a real workload through text
    case = case_c3
    api.write_dump(str(tmp_path / "sr.dump"), case.keys, case.counts, case.cfg.k)
    api.write_dump(str(tmp_path / "jj.dump"), case.jkeys, case.jcounts, case.cfg.k)
    a = api.Talc(api.default_params(case.cfg.k))
    nl, nk = a.load_dump(str(tmp_path / "sr.dump"), str(tmp_path / "jj.dump"))
    b = _ctx(api, case)
    assert nl == len(case.keys) and nk == b.table_info()["entries"] == case.otable.size()
    rng = np.random.default_rng(5)
    probe = np.concatenate([case.keys[rng.integers(0, len(case.keys), 20000)], rng.integers(0, 1 << 42, 2000).astype(np.uint64)])
    for x, y in zip(a.lookup(probe), b.lookup(probe)):
        assert np.array_equal(x, y)
    out, off, st, ctr = a.correct(case.reads, case.off)
    _assert_same(case, out, off, st, ctr)
    # the cache written from this table is refused for other inputs and accepted for the same ones
    a.table_save(str(tmp_path / "t.bin"))
    c2 = api.Talc(api.default_params(case.cfg.k))
    assert c2.table_load_cache_for(str(tmp_path / "t.bin"), str(tmp_path / "sr.dump"), str(tmp_path / "jj.dump")) == nk
    with pytest.raises(api.TalcError):
        c2.table_load_cache_for(str(tmp_path / "t.bin"), str(tmp_path / "sr.dump"), None)
    with pytest.raises(api.TalcError):
        c2.table_load_cache_for(str(tmp_path / "t.bin"), str(tmp_path / "jj.dump"), str(tmp_path / "jj.dump"))
    with open(tmp_path / "t.bin", "r+b") as f:  # truncated file
        f.truncate(os.path.getsize(tmp_path / "t.bin") - 16)
    with pytest.raises(api.TalcError):
        c2.table_load_cache(str(tmp_path / "t.bin"))


def test_gpu_kmer_counting_from_short_reads(api, case_c1, tmp_path):
    """Row f3: talc_table_count_reads counts the k-mers of short-read files on the GPU and builds the table `jellyfish
    count | jellyfish dump -c | buildCDBG` would have built: checked against the numpy restatement of the counting rule
    (oracle/kmer_count.py), against the dump route (counts written as text, parsed, filtered), and end to end."""
    from oracle import kmer_count as kc
    case = case_c1
    k = case.cfg.k
    rng = np.random.default_rng(11)
    tb = case.w.t_bases.numpy()
    toff = case.w.t_off.numpy()
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)

    def short_reads(n):
        out = []
        for _ in range(n):
            t = int(rng.integers(0, len(toff) - 1))
            a, b = int(toff[t]), int(toff[t + 1])
            L = int(rng.integers(30, 151))
            p = int(rng.integers(a, max(a + 1, b - L)))
            s = letters[tb[p:min(b, p + L)]].copy()
            for q in np.nonzero(rng.random(len(s)) < 0.01)[0]:
                s[q] = letters[int(rng.integers(0, 4))]
            r = rng.random()
            if r < 0.05 and len(s) > 5:
                s[int(rng.integers(0, len(s)))] = ord("N")
            elif r < 0.10:
                s = np.frombuffer(s.tobytes().lower(), dtype=np.uint8).copy()
            out.append(s.tobytes())
        out.append(b"ACGT")                    # shorter than K
        out.append(b"A" * 70)                  # homopolymer: 70-K+1 occurrences of one k-mer
        return out

    r1, r2 = short_reads(30000), short_reads(20000)
    with open(tmp_path / "sr_1.fq", "wb") as f:
        for i, s_ in enumerate(r1):
            f.write(b"@r%d/1\n" % i + s_ + b"\n+\n" + b"I" * len(s_) + b"\n")
    with open(tmp_path / "sr_2.fa", "wb") as f:
        for i, s_ in enumerate(r2):
            f.write(b">r%d/2\r\n" % i + s_ + b"\r\n")
    okeys, ocounts, occ = kc.count_kmers(kc.read_sequences(str(tmp_path / "sr_1.fq")) + kc.read_sequences(str(tmp_path / "sr_2.fa")), k)
    assert occ > 2_000_000 and len(okeys) > 100_000
    t = api.Talc(api.default_params(k))
    n_kmers, n_distinct, n_kept = t.count_reads([str(tmp_path / "sr_1.fq"), str(tmp_path / "sr_2.fa")])
    keep = ocounts >= 2
    assert (n_kmers, n_distinct, n_kept) == (occ, len(okeys), int(keep.sum()))
    cnt, col, found = t.lookup(okeys)
    assert np.array_equal(found.astype(bool), keep)
    assert np.array_equal(cnt[keep], ocounts[keep].astype(np.uint32)) and not cnt[~keep].any() and not col.any()
    # the dump route: the same counts as text -> parser -> MIN_COUNT filter
    api.write_dump(str(tmp_path / "sr.dump"), okeys, ocounts, k)
    d = api.Talc(api.default_params(k))
    assert d.load_dump(str(tmp_path / "sr.dump")) == (len(okeys), n_kept)
    probe = np.concatenate([okeys[::7], rng.integers(0, 1 << 42, 3000).astype(np.uint64)])
    for x, y in zip(t.lookup(probe), d.lookup(probe)):
        assert np.array_equal(x, y)
    # too small a counting table is an error, not a silent loss
    with pytest.raises(api.TalcError):
        api.Talc(api.default_params(k)).count_reads([str(tmp_path / "sr_1.fq")], expected_distinct=1000)
    # end to end: long reads corrected with the counted table == with the table from the dump of the same counts
    sub_r, sub_o = case.reads[: int(case.off[60])], case.off[:61]
    a = t.correct(sub_r, sub_o)
    b = d.correct(sub_r, sub_o)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    assert a[3]["gaps"] == b[3]["gaps"] and a[3]["lookups_walk"] == b[3]["lookups_walk"]


@pytest.mark.parametrize("shape", [(2, 0, 0), (1, 5, 1), (1, 64, 7), (1, 0, 0)])
def test_execution_shapes_give_identical_results(api, case_c1, case_c5, case_c3, shape):
    """The suspendable per-read program + lane-per-trail walk kernel (split_walk = 1) against the monolithic kernel
    (split_walk = 2) and the oracle: bytes, status and every algorithmic counter, whatever the number of read contexts
    in flight (5: every context is reused dozens of times) and wherever the walk rounds are cut (cap 1: a frontier
    comes back after every single step)."""
    for case in (case_c1, case_c5, case_c3):
        t = _ctx(api, case)
        t.set_exec(*shape)
        out, off, st, ctr = t.correct(case.reads, case.off)
        _assert_same(case, out, off, st, ctr)
        if shape[0]:
            assert (ctr["rounds"] > 0) == (shape[0] == 1)
    # a tiny first tier pushes reads through the second tier in split mode as well
    t = _ctx(api, case_c1)
    t.set_exec(*shape)
    t.set_scratch(tier1_bytes=6 * 1024)
    out, off, st, ctr = t.correct(case_c1.reads, case_c1.off)
    assert ctr["reads_second_tier"] > 0
    _assert_same(case_c1, out, off, st, ctr)


@pytest.mark.parametrize("steps", [2, 3])
def test_bench_dumps_what_its_last_timed_step_computed(api, tmp_path, steps):
    """bench.py --dump-outputs against one correct_device call on the slice of the last timed step, generated here as
    bench.py generates it.  With two lanes the last step runs on lane 1 (2 steps) or on lane 0 (3 steps)."""
    import importlib.util
    import subprocess
    import sys
    import torch
    from talc_b200 import synth
    B, warmup, dev = 1500, 1, "cuda:0"
    d = tmp_path / "dump"
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                         "--scale", "0.02", "--batch-reads", str(B), "--lanes", "2", "--no-table-load", "--no-cpu-baseline",
                         "--dump-outputs", str(d)], capture_output=True, text=True, cwd=ROOT)
    assert pr.returncode == 0, pr.stderr[-3000:]
    cfg = synth.baseline_config(2, 0.02)
    tr = synth.make_transcriptome(cfg, dev)
    keys, counts, _, _ = synth.make_counts(cfg, tr, dev)
    reads, roff = synth.make_reads(cfg, tr, B * (warmup + steps + 1), dev, seed_offset=3)
    roff = roff.to(torch.int64)
    lo = (warmup + steps - 1) * B
    b0, b1 = int(roff[lo]), int(roff[lo + B])
    t = api.Talc(api.default_params(cfg.k))
    t.load_packed(keys.cpu().numpy().astype(np.uint64), counts.cpu().numpy())
    d_out = torch.empty(2 * (b1 - b0) + 64 * B + 4096, dtype=torch.uint8, device=dev)
    d_ooff = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    d_st = torch.zeros(B, dtype=torch.uint8, device=dev)
    ctr = t.correct_device(reads[b0:b1].contiguous(), (roff[lo:lo + B + 1] - roff[lo]).contiguous(), b1 - b0, d_out, d_ooff, d_st)
    off = d_ooff.cpu().numpy()
    out = d_out[: int(off[-1])].cpu().numpy()
    spec = importlib.util.spec_from_file_location("talc_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert np.array_equal(np.load(d / "out_offsets.npy"), off)
    assert np.array_equal(np.load(d / "status.npy"), d_st.cpu().numpy())
    assert np.array_equal(np.load(d / "read_digests.npy"), bench.read_digests(out, off, B))
    idx = np.load(d / "sample_reads.npy").astype(np.int64)
    assert np.array_equal(np.load(d / "sample_bases.npy"), np.concatenate([out[off[r]:off[r + 1]] for r in idx]))
    for k in SHARED + ["reads", "bases_in", "reads_ok"]:
        assert np.load(d / ("counter_%s.npy" % k))[0] == ctr[k], k
