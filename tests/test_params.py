"""The correction at the reference's tunables other than their defaults, and at every k-mer size the command line accepts,
against the oracle.

The command line passes --MIN_COUNT, --WINDOW_SIZE, --MAX_NB_BRANCHES, --ALPHA_FOR_PRED, --SR_ERROR_RATE,
--MIN_INNER_SCORE, --MIN_BORDER_SCORE and -k straight to the kernels, and the library also reaches cycle_mode,
q11_zero_init and the bounds of sr_error_rate.  Several device-only paths depend on them: the fast walk's eligibility
bound (nCur <= 7 && nCur <= max_branches), the trail-slot sizing from max_branches, the warp overlap scoring bounded by
the window, the model tables a context (and each of its lanes) fills for its alpha, the MIN_COUNT filters of the table
build, the cost key, the successor mask and the table cache.  Each grid point below is pinned to a workload on which it
changes the oracle's answer, so that a device that ignored the parameter would be caught.

MIN_BORDER_SCORE 0.5 is not in the grid.  A border is accepted on the LCS identity of its X-drop extension, which
ends at its best-scoring cell; no border of 64 seeded workloads (the c1, c3 and c5 families, long-read error rates from
0.1 to 0.45) scored in [0.5, 0.7), so 0.5 and the default 0.7 gave the same answer on all of them."""
import os
import subprocess

import numpy as np
import pytest

from conftest import Case, have_gpu

SHARED = ["lookups_seg", "lookups_deg", "lookups_walk", "steps_inner", "steps_border", "frontier_sum", "cells_nw",
          "cells_lcs", "cells_ovl", "cells_xdrop", "gaps", "gaps_bridged", "gap_attempts", "borders",
          "borders_corrected", "ev_gardening", "ev_bridge", "ev_edge", "ev_cycle", "bases_out"]

# po.make_params keyword -> talc_params field
TALC_FIELD = {"min_count": "min_count", "window": "window_size", "max_branches": "max_nb_branches", "alpha": "alpha",
              "sr_error": "sr_error_rate", "min_inner": "min_inner_score", "min_border": "min_border_score",
              "cycle_mode": "cycle_mode", "q11": "q11_zero_init"}

# c5: K = 30, 15 % errors, low-complexity inserts: frontiers above 7 trails and gardening (walk and gardening
# parameters).  c1: K = 21, many gaps and borders (the scores).  c3: junction colours, which change the tagging (the
# count model and the table).
WORKLOADS = {"c5": lambda: Case(5, 0.5, 80), "c1": lambda: Case(1, 0.05, 120),
             "c3": lambda: Case(3, 0.004, 120, junctions=True)}

# (workload, parameters, counters that must differ from the default run; None: the bytes or the status must differ)
GRID = [
    ("c5", dict(max_branches=5), ("frontier_sum", "ev_gardening")),
    ("c5", dict(max_branches=6), ("frontier_sum", "ev_gardening")),
    ("c5", dict(max_branches=8), None),
    ("c5", dict(max_branches=12), None),
    ("c5", dict(max_branches=60), None),
    ("c5", dict(max_branches=1000), None),  # pruning never triggers
    ("c5", dict(window=6), None),
    ("c5", dict(window=40), None),
    ("c5", dict(window=500), None),
    ("c5", dict(q11=0), None),
    ("c5", dict(cycle_mode=1), None),
    ("c1", dict(min_inner=0.3), None),
    ("c1", dict(min_inner=0.9), None),
    ("c1", dict(min_border=0.9), None),
    ("c3", dict(alpha=0.67), None),
    ("c3", dict(alpha=6.0), None),
    ("c3", dict(sr_error=0.01), None),
    ("c3", dict(sr_error=0.1), None),
    ("c3", dict(sr_error=0.0), None),  # the bounds talc_ctx_create accepts
    ("c3", dict(sr_error=0.5), None),
    ("c3", dict(min_count=3), None),
    ("c3", dict(min_count=5), None),
    # the lower bound talc_ctx_create accepts: count-1 k-mers (error variants) enter the table and the walk's masks
    ("c3", dict(min_count=1), None),
    ("c5", dict(min_count=1), None),
]
GRID_IDS = ["%s-%s" % (w, "-".join("%s=%s" % kv for kv in kw.items())) for w, kw, _ in GRID]
K_SWEEP = [18, 19, 22, 25, 27, 29]

_workloads, _points = {}, {}


def workload(name):
    if name not in _workloads:
        _workloads[name] = WORKLOADS[name]() if name in WORKLOADS else Case(1, 0.05, 120, k=int(name[1:]))
    return _workloads[name]


class Point:
    """A workload, or some of its reads, and the oracle's answer at the given parameters (conftest.Case runs the
    oracle at defaults)."""

    def __init__(self, name, kw, rows=None):
        from oracle import pyoracle as po
        c = workload(name)
        self.name, self.kw, self.case = name, kw, c
        self.cfg, self.keys, self.counts, self.jkeys, self.jcounts = c.cfg, c.keys, c.counts, c.jkeys, c.jcounts
        self.reads, self.off = c.reads, c.off
        if rows is not None:
            self.reads, self.off = _concat([c.read(r) for r in rows])
        self.op = po.make_params(k=c.cfg.k, **kw)
        self.otable = po.OracleTable(self.op).build_packed(c.keys, c.counts, c.jkeys, c.jcounts)
        self.o_out, self.o_off, self.o_status, self.o_ctr, _ = self.otable.correct(self.reads, self.off, threads=8)

    def oracle_read(self, r):
        return self.o_out[int(self.o_off[r]):int(self.o_off[r + 1])].tobytes()


def _concat(parts):
    off = np.zeros(len(parts) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(p) for p in parts])
    return np.frombuffer(b"".join(parts), dtype=np.uint8).copy(), off


def point(name, kw=None):
    kw = kw or {}
    key = (name, tuple(sorted(kw.items())))
    if key not in _points:
        _points[key] = Point(name, kw)
    return _points[key]


def _assert_same(pt, out, off, status, ctr=None, what=""):
    assert np.array_equal(status, pt.o_status), "%s: per-read status differs" % what
    bad = [r for r in range(len(pt.off) - 1) if out[int(off[r]):int(off[r + 1])].tobytes() != pt.oracle_read(r)]
    assert not bad, "%s: corrected sequence differs for reads %s" % (what, bad[:10])
    if ctr is not None:
        diff = {k: (pt.o_ctr[k], ctr[k]) for k in SHARED if pt.o_ctr[k] != ctr[k]}
        assert not diff, "%s: algorithmic counters differ: %s" % (what, diff)


def _emu_answer(pt):
    from test_hostemu import _emu_correct
    return _emu_correct(pt.op, pt.keys, pt.counts, pt.jkeys, pt.jcounts, pt.reads, pt.off)


# Reads of c3 whose correction at sr_error_rate 0 depends on how the anchors' sort centre, 0 / 0, is converted to int
ZERO_RATE_READS = [32, 45, 62, 69]


# ---------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name,kw,ctrs", GRID, ids=GRID_IDS)
def test_grid_point_changes_the_oracle_answer(name, kw, ctrs):
    """A parameter point proves nothing on a workload where it changes nothing."""
    base, pt = point(name), point(name, kw)
    if ctrs is None:
        assert not (np.array_equal(pt.o_status, base.o_status) and np.array_equal(pt.o_off, base.o_off) and
                    np.array_equal(pt.o_out, base.o_out)), "the corrected reads do not depend on %s here" % kw
    else:
        for k in ctrs:
            assert pt.o_ctr[k] != base.o_ctr[k], "%s does not change %s here" % (kw, k)


@pytest.mark.parametrize("name,kw,ctrs", GRID, ids=GRID_IDS)
def test_host_emulation_matches_oracle_off_defaults(name, kw, ctrs):
    pt = point(name, kw)
    out, off, st, ctr = _emu_answer(pt)
    _assert_same(pt, out, off, st, ctr, "host emulation")


@pytest.mark.parametrize("k", K_SWEEP)
def test_host_emulation_matches_oracle_across_k(k):
    pt = point("k%d" % k)
    assert pt.cfg.k == k
    assert pt.o_ctr["gaps_bridged"] > 0 and pt.o_ctr["borders_corrected"] > 0, "the walk must really run"
    out, off, st, ctr = _emu_answer(pt)
    _assert_same(pt, out, off, st, ctr, "host emulation")


def test_anchor_sort_centre_at_zero_error_rate():
    """At sr_error_rate 0 the anchors' sort centre is 0 / 0 = NaN, which the reference's x86-64 build converts to
    INT_MIN; the distance then wraps, so anchors of count 0 sort first and the others by descending count.  The
    conversion of NaN is undefined in C++ and gives 0 on the device, so the device code spells the x86 result out."""
    sub = Point("c3", dict(sr_error=0.0), ZERO_RATE_READS)
    assert (sub.o_status == 0).all()
    out, off, st, ctr = _emu_answer(sub)
    _assert_same(sub, out, off, st, ctr, "host emulation at sr_error_rate 0")


# ---------------------------------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    if not have_gpu():
        pytest.fail("GPU tests selected but no CUDA device is visible")
    from talc_b200 import api as _api
    return _api


def _talc_params(api, pt):
    return api.default_params(pt.cfg.k, **{TALC_FIELD[k]: v for k, v in pt.kw.items()})


def _ctx(api, pt):
    t = api.Talc(_talc_params(api, pt))
    t.load_packed(pt.keys, pt.counts, pt.jkeys, pt.jcounts)
    return t


@gpu
@pytest.mark.parametrize("name,kw,ctrs", GRID, ids=GRID_IDS)
def test_gpu_matches_oracle_off_defaults(api, name, kw, ctrs):
    """Both execution shapes (split_walk 1: suspendable reads and the walk kernel; 2: one monolithic kernel) bit for bit,
    counters included; for the branch limit also with a first tier so small that reads go through the second."""
    pt = point(name, kw)
    t = _ctx(api, pt)
    for shape in (1, 2):
        t.set_exec(split_walk=shape)
        out, off, st, ctr = t.correct(pt.reads, pt.off)
        _assert_same(pt, out, off, st, ctr, "split_walk %d" % shape)
    if "max_branches" in kw:
        for shape in (1, 2):
            t2 = _ctx(api, pt)
            t2.set_exec(split_walk=shape)
            t2.set_scratch(tier1_bytes=6 * 1024)
            out, off, st, ctr = t2.correct(pt.reads, pt.off)
            assert ctr["reads_second_tier"] > 0
            _assert_same(pt, out, off, st, ctr, "split_walk %d, second tier" % shape)
            t2.close()
    t.close()


@gpu
@pytest.mark.parametrize("k", K_SWEEP)
def test_gpu_matches_oracle_across_k(api, k):
    pt = point("k%d" % k)
    assert pt.o_ctr["gaps_bridged"] > 0 and pt.o_ctr["borders_corrected"] > 0, "the walk must really run"
    t = _ctx(api, pt)
    for shape in (1, 2):
        t.set_exec(split_walk=shape)
        out, off, st, ctr = t.correct(pt.reads, pt.off)
        _assert_same(pt, out, off, st, ctr, "split_walk %d" % shape)
    t.close()


@gpu
@pytest.mark.parametrize("kw", [dict(alpha=0.67), dict(min_count=3)], ids=["alpha=0.67", "min_count=3"])
def test_lane_and_stream_off_defaults(api, kw):
    """A lane fills its own model tables and follows its parent's table and settings; talc_stream corrects through
    lanes.  Both must correct like the oracle at the parent's parameters, a model (alpha) and a table (MIN_COUNT) point."""
    pt = point("c3", kw)
    t = _ctx(api, pt)
    n = len(pt.off) - 1
    for shape in (1, 2):
        t.set_exec(split_walk=shape)
        lane = t.create_lane()
        out, off, st, ctr = lane.correct(pt.reads, pt.off)
        _assert_same(pt, out, off, st, ctr, "lane, split_walk %d" % shape)
        lane.close()
        spans = list(zip([0, 1, 1, 17, 18, 70], [1, 1, 17, 18, 70, n]))
        s = t.stream()
        outs, lens, sts, tot = [], [], [], None
        fetched = 0

        def fetch():
            nonlocal tot, fetched
            a, b = spans[fetched]
            o, f, x, _, c = s.next()
            assert len(x) == b - a
            outs.append(o)
            lens.append(np.diff(f))
            sts.append(x)
            tot = c if tot is None else {k2: tot[k2] + c[k2] for k2 in c}
            fetched += 1

        for i, (a, b) in enumerate(spans):  # at most three batches in flight: the ring has four slots
            s.submit(pt.reads[int(pt.off[a]):int(pt.off[b])], pt.off[a:b + 1] - pt.off[a])
            if i - fetched >= 2:
                fetch()
        while fetched < len(spans):
            fetch()
        s.close()
        off = np.zeros(n + 1, dtype=np.uint64)
        off[1:] = np.cumsum(np.concatenate(lens))
        _assert_same(pt, np.concatenate(outs), off, np.concatenate(sts), tot, "stream, split_walk %d" % shape)
    t.close()


@gpu
def test_gpu_anchor_sort_centre_at_zero_error_rate(api):
    sub = Point("c3", dict(sr_error=0.0), ZERO_RATE_READS)
    t = _ctx(api, sub)
    for shape in (1, 2):
        t.set_exec(split_walk=shape)
        out, off, st, ctr = t.correct(sub.reads, sub.off)
        _assert_same(sub, out, off, st, ctr, "split_walk %d at sr_error_rate 0" % shape)
    t.close()


# Dna5 normalisation and reverse complement of the reference (SeqAn): ACGT in either case, anything else -> N
_NORM = np.full(256, ord("N"), dtype=np.uint8)
_COMP = np.full(256, ord("N"), dtype=np.uint8)
_CASE_COMP = np.arange(256, dtype=np.uint8)  # a complement that keeps case and IUPAC codes: raw antisense input
for _a, _b in zip(b"ACGTacgt", b"ACGTACGT"):
    _NORM[_a] = _b
for _a, _b in zip(b"ACGTacgt", b"TGCATGCA"):
    _COMP[_a] = _b
for _a, _b in zip(b"ACGTacgtRYry", b"TGCAtgcaYRyr"):
    _CASE_COMP[_a] = _b


def _resource_reads(reverse):
    """c1 reads, every third one with a lower-case stretch and IUPAC codes, so that some of the reads passed through
    uncorrected carry bytes the pass-through must normalise.  In reverse mode their antisense, case and codes kept, so
    that the table (of the sense strand) corrects them as in forward mode."""
    c = workload("c1")
    parts = []
    for r in range(len(c.off) - 1):
        s = bytearray(c.read(r))
        if r % 3 == 0:
            s[100:160] = s[100:160].lower()
            s[250] = ord("R")
            s[300] = ord("y")
        parts.append(_CASE_COMP[np.frombuffer(bytes(s), dtype=np.uint8)[::-1]].tobytes() if reverse else bytes(s))
    return parts


@gpu
@pytest.mark.parametrize("reverse", [False, True], ids=["forward", "reverse"])
def test_reads_that_outgrow_the_second_tier_pass_through(api, reverse):
    """TALC_READ_RESOURCE: with a 6 KiB first tier and a 128 KiB second tier on 4 warps some reads outgrow both.  They
    come back as their Dna5-normalised input (upper case, anything else N), reverse-complemented in reverse mode, and
    are counted in reads_overflow; every other read is the oracle's."""
    parts = _resource_reads(reverse)
    reads, off = _concat(parts)
    c = workload("c1")
    n = len(parts)
    # what the correction sees: the reads, or in reverse mode their reverse complement
    seen = [(_COMP[np.frombuffer(p, dtype=np.uint8)[::-1]] if reverse else _NORM[np.frombuffer(p, dtype=np.uint8)]).tobytes()
            for p in parts]
    o_out, o_off, o_st, _, _ = point("c1").otable.correct(*_concat(seen), threads=8)
    for shape in (1, 2):
        t = api.Talc(api.default_params(c.cfg.k))
        t.load_packed(c.keys, c.counts)
        if reverse:
            t.set_reverse(True)
        t.set_exec(split_walk=shape)
        t.set_scratch(6 * 1024, 128 * 1024, 4)
        out, ooff, st, ctr = t.correct(reads, off)
        res = np.nonzero(st == api.STATUS_RESOURCE)[0]
        assert 0 < len(res) < n, "split_walk %d: %d of %d reads outgrew the second tier" % (shape, len(res), n)
        assert ctr["reads_overflow"] == len(res)
        assert any(r % 3 == 0 for r in res), "a read with lower case and IUPAC codes must pass through"
        for r in range(n):
            got = out[int(ooff[r]):int(ooff[r + 1])].tobytes()
            if st[r] == api.STATUS_RESOURCE:
                want = seen[r]
                assert got == want, "split_walk %d: read %d passed through as %r" % (shape, r, got[:80])
            else:
                assert st[r] == o_st[r], (shape, r)
                want = o_out[int(o_off[r]):int(o_off[r + 1])].tobytes()
                if reverse and o_st[r] == 0:
                    want = _COMP[np.frombuffer(want, dtype=np.uint8)[::-1]].tobytes()
                assert got == want, "split_walk %d: read %d differs from the oracle" % (shape, r)
        t.close()


# -k stays at the K of the dumps: a table of other k-mers would not be the same workload (the K sweep covers -k)
CLI_TUNABLES = ["--MIN_COUNT", "3", "--WINDOW_SIZE", "12", "--MAX_NB_BRANCHES", "9", "--ALPHA_FOR_PRED", "3.5",
                "--SR_ERROR_RATE", "0.04", "--MIN_INNER_SCORE", "0.65", "--MIN_BORDER_SCORE", "0.8", "--cycle-mode", "1"]


@gpu
def test_cli_with_every_tunable_set(api, tmp_path):
    """`talc` with every tunable off its default writes the .fa, .log, .stats_basics.txt and .config.txt of the oracle's
    front end given the same flags; a --tableCache written at MIN_COUNT 2 is refused as stale at MIN_COUNT 3, rebuilt,
    and then reused."""
    from oracle import pyoracle as po
    from talc_b200 import build
    from test_gpu_parity import _write_case_files
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "tiny_case.npz"))
    k = _write_case_files(tmp_path, g)
    cli = build.build_cli()
    common = [str(tmp_path / "reads.fa"), "--SRCounts", str(tmp_path / "sr.dump"), "--junctions", str(tmp_path / "j.dump"),
              "-k", str(k)]

    def talc(*a):
        pr = subprocess.run([cli] + common + list(a), cwd=tmp_path, capture_output=True, text=True)
        assert pr.returncode == 0, pr.stderr
        return pr.stdout

    def oracle(*a):
        assert subprocess.call([po.BIN] + common + ["-t", "1", "--oracle-table", "hash"] + list(a), cwd=tmp_path,
                               stdout=subprocess.DEVNULL) == 0

    def same(a, b):
        for ext in (".fa", ".log", ".stats_basics.txt"):
            assert open(tmp_path / (a + ext), "rb").read() == open(tmp_path / (b + ext), "rb").read(), (a, b, ext)
        x = open(tmp_path / (a + ".config.txt")).read().replace(a, "X")
        y = open(tmp_path / (b + ".config.txt")).read().replace(b, "X")
        assert x == y, (a, b)

    talc("-o", "gpu", *CLI_TUNABLES)
    oracle("-o", "cpu", *CLI_TUNABLES)
    oracle("-o", "cpu_default")
    same("gpu", "cpu")
    assert open(tmp_path / "cpu.fa", "rb").read() != open(tmp_path / "cpu_default.fa", "rb").read()
    assert "MIN_SR_COUNT=3" in open(tmp_path / "gpu.config.txt").read()
    # the table cache remembers the MIN_COUNT it was built with
    cache = str(tmp_path / "table.bin")
    out = talc("-o", "c2", "--tableCache", cache)
    assert "rebuilding" not in out and os.path.exists(cache)
    oracle("-o", "o3", "--MIN_COUNT", "3")
    out = talc("-o", "c3", "--tableCache", cache, "--MIN_COUNT", "3")
    assert "rebuilding" in out, out
    same("c3", "o3")
    out = talc("-o", "c3again", "--tableCache", cache, "--MIN_COUNT", "3")
    assert "rebuilding" not in out
    same("c3again", "o3")
    assert open(tmp_path / "o3.fa", "rb").read() != open(tmp_path / "c2.fa", "rb").read()
