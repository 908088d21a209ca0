"""The device scoring primitives and the coverage kernel on the inputs the pipeline gives them: read slices at every
offset in both walk directions, trail slots with stale bits, the length boundaries of each kernel, the X-drop's score
and cell tally at every register-band width, the stripe reuse of gardening, and coverage at every k-mer size.  The
reference is the plain DP of tests/test_primitive_slices.py; the oracle stays the reference for the SeqAn-defined
X-drop end positions and the seed-and-extension result."""
import numpy as np
import pytest

from conftest import have_gpu
from test_primitive_slices import (SEED_X, Views, boundary_pairs, check_scores, check_seed_extension, edit_distance_rows,
                                   mutate, overlap_score, placement, seed_extension_pairs)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def talc():
    if not have_gpu():
        pytest.fail("GPU tests selected but no CUDA device is visible")
    from talc_b200 import api
    t = api.Talc(api.default_params(21))
    yield t
    t.close()


def test_scores_on_slices_at_the_boundaries(talc):
    """NW, LCS, overlap and the fused pass at lengths 0 .. 4097 crossed (either side the longer, so both the fused
    and the striped forms), both steps, 2-bit and 4-bit reads, every start residue, flush slices, trail slots."""
    reads, desc, strings = boundary_pairs(seed=1)
    check_scores(talc.test_align_slices, reads, desc, strings)
    reads, desc, strings = boundary_pairs(seed=2, trails=False)
    check_scores(talc.test_align_slices, reads, desc, strings)


def _frontiers(rng, v, cn):
    """Frontiers of trails of length cn against one reference slice: consecutive trails share prefixes of 0, 127,
    128, 129, 255, 256, 257 and cn bases; then a trail that shares a short prefix with its predecessor followed by one
    that shares a long prefix with it (but a short one with the trail before), and an identical pair."""
    def branch(t, p):
        if p >= cn:
            return t
        alt = bytes([int(rng.choice([c for c in b"ACGT" if c != t[p]]))])
        return t[:p] + alt + v.pad(cn - p - 1)

    groups = []
    for rn, step, four in ((300, 1, False), (129, -1, True), (450, -1, False), (cn, 1, True)):
        ref = v.pad(rn)
        if four:
            ref = ref[: rn // 2] + b"N" + ref[rn // 2 + 1:]
        trails = [mutate(rng, ref.replace(b"N", b"A"), 0.1)[:cn]]  # trails hold A, C, G, T only
        trails[0] = trails[0] + v.pad(cn - len(trails[0]))
        for p in (0, 127, 128, 129, 255, 256, 257, cn, cn):
            trails.append(branch(trails[-1], p))
        trails.append(branch(trails[-1], 10))
        trails.append(branch(trails[-1], min(300, cn)))
        trails.append(trails[-1])
        a = placement(v, ref, step, len(groups), four)
        groups.append((ref, trails, [a + v.side(t, 0, int(rng.integers(0, 40)), int(rng.integers(0, 40))) for t in trails]))
    return groups


@pytest.mark.parametrize("cn", [128, 300, 384])
def test_frontier_scores_with_stripe_reuse(talc, cn):
    """Gardening scores a whole frontier against one reference and skips the stripes inside the prefix a trail shares
    with its predecessor, capped so that the last stripe is always computed.  Every score equals the plain DP and the
    score of the same pair without reuse."""
    rng = np.random.default_rng(cn)
    v = Views(rng)
    groups = _frontiers(rng, v, cn)
    g = len(groups[0][1])
    desc = np.array([d for _, _, ds in groups for d in ds], dtype=np.int32)
    got = talc.test_align_slices(6, v.reads, desc, aux=g)
    alone = talc.test_align_slices(2, v.reads, desc)
    i = 0
    for ref, trails, _ in groups:
        for j, t in enumerate(trails):
            want = overlap_score(ref, t)
            assert alone[i] == want, (cn, len(ref), j)
            assert got[i] == want, (cn, len(ref), j)
            i += 1


def _xdrop_pairs(rng, v):
    pairs, desc = [], []
    for i in range(36):
        n = int(rng.integers(1, 60)) if i % 6 == 0 else int(rng.integers(200, 3000))
        alpha = b"AC" if i % 9 == 4 else b"ACGT"
        d = bytes(rng.choice(list(alpha), n).tolist())
        if i % 4 == 3:
            q = bytes(rng.choice(list(alpha), int(rng.integers(1, n + 40))).tolist())  # unrelated: the band at full width
        else:
            q = mutate(rng, d, float(rng.choice([0.03, 0.15, 0.3])), alpha) or b"A"
        if i % 8 == 5:
            q = q[: len(q) // 2] + b"N" + q[len(q) // 2 + 1:]
        if i % 2:
            q, d = d, q
        sq = (1, -1)[i % 2]
        sd = (1, -1, 0)[i % 3] if b"N" not in d else -1
        desc.append(placement(v, q, sq, i, b"N" in q or i % 5 == 0) + placement(v, d, sd, i + 2, b"N" in d))
        pairs.append((q, d))
    return pairs, np.array(desc, dtype=np.int32)


def test_xdrop_end_score_and_cell_tally(talc):
    """Op 4 returns the end position, the cells visited and the end score.  The end position and the tally must be the
    oracle's; the end score must be minus the edit distance of the two extended prefixes (what replaces the NW call of
    the seed extension) for the register bands S = 1, 2, 4, 8 and the scalar form beyond X = 255."""
    from oracle import pyoracle as po
    rng = np.random.default_rng(23)
    v = Views(rng)
    pairs, desc = _xdrop_pairs(rng, v)
    xs = (31, 32, 63, 64, 127, 128, 255, 256, 300)
    res = {x: talc.test_align_slices(4, v.reads, desc, aux=x) for x in xs}
    for i, (q, d) in enumerate(pairs):
        dist = edit_distance_rows(q, d)
        for x in xs:
            er, ec, cells = po.xdrop_counted(q, d, False, x)
            r = res[x][i]
            assert (int(r[0]), int(r[1]), int(r[2])) == (er, ec, cells), (i, x, len(q), len(d))
            assert r[3] == -dist[ec][er], (i, x, len(q), len(d))


@pytest.mark.parametrize("right", [True, False])
def test_seed_extension_on_slices(talc, right):
    reads, desc, strings = seed_extension_pairs(right, 21)
    for x in SEED_X:
        res = talc.test_align_slices(3, reads, desc, aux=x, aux2=1 if right else 0)
        check_seed_extension(res, strings, x, right, 21)


def _coverage_case(rng, K):
    lens = [K - 1, K, K + 1, K + 2, K + 3] + [K - 1 + c for c in range(1, 257)]  # C = len - K + 1 at every residue mod 128
    rng.shuffle(lens)
    reads = []
    for j, n in enumerate(lens):
        s = bytearray(rng.choice(list(b"ACGT"), n).tolist())
        if j % 3 == 0:
            s[j % n] = ord("N")
        if j % 4 == 1:  # near the edges of the 128-k-mer windows of a warp and of a lane's 4 k-mers
            for e in (128, 256):
                p = e + K - 1 + (j // 4) % 9 - 4
                if p < n:
                    s[p] = ord("N")
        if j % 6 == 2:
            a = int(rng.integers(0, n))
            s[a:a + 40] = bytes(s[a:a + 40]).lower()
        if j % 10 == 7:
            s[int(rng.integers(0, n))] = int(rng.choice(list(b"XRu.-")))
        reads.append(bytes(s))
    return reads


def _kmers(read: bytes, K: int):
    """(key or None) per position: 2-bit, first base most significant; None when the window holds a non-base."""
    codes = [{"A": 0, "C": 1, "G": 2, "T": 3, "U": 3}.get(chr(c).upper(), 4) for c in read]
    out = []
    for p in range(len(read) - K + 1):
        w = codes[p:p + K]
        if max(w) > 3:
            out.append(None)
        else:
            key = 0
            for c in w:
                key = (key << 2) | c
            out.append(key)
    return out


def test_coverage_at_every_k(talc):
    """coverage_kernel for K = 18 .. 31 against a dictionary: reads of K-1 .. K+3 bases and of every length mod 128,
    starting at every output offset mod 4 (the 16-byte store and the scalar tail), N at every lane position and near the
    window edges, lowercase and non-ACGTN bytes; the table holds random keys and k-mers of the reads, some below
    MIN_COUNT, some listed twice (the first entry that passes MIN_COUNT wins)."""
    from talc_b200 import api
    rng = np.random.default_rng(31)
    for K in range(18, 32):
        reads = _coverage_case(rng, K)
        kms = [_kmers(r, K) for r in reads]
        pool = sorted({x for ks in kms for x in ks if x is not None})
        pick = [x for x in pool if rng.random() < 0.7]
        keys = pick + [int(x) for x in rng.integers(0, 1 << (2 * K), 3000, dtype=np.uint64)]
        keys += [pick[i] for i in rng.integers(0, len(pick), len(pick) // 8)]  # listed again, later
        counts = [int(c) for c in rng.choice([1, 1, 2, 3, 9, 200, 70000], len(keys))]
        t = api.Talc(api.default_params(K))
        try:
            t.load_packed(np.array(keys, dtype=np.uint64), np.array(counts, dtype=np.int64))
            m = t.params.min_count
            table = {}
            for k_, c in zip(keys, counts):
                if c >= m and k_ not in table:
                    table[k_] = c
            want = np.array([table.get(x, 0) if x is not None else 0 for ks in kms for x in ks], dtype=np.uint32)
            off = np.zeros(len(reads) + 1, dtype=np.uint64)
            off[1:] = np.cumsum([len(r) for r in reads])
            cov = t.coverage(np.frombuffer(b"".join(reads), dtype=np.uint8), off)
        finally:
            t.close()
        starts = np.cumsum([0] + [len(ks) for ks in kms])[:-1]
        assert {int(s) % 4 for s, ks in zip(starts, kms) if len(ks) >= 4} == {0, 1, 2, 3}
        assert len(cov) == len(want)
        bad = np.nonzero(cov != want)[0]
        assert not len(bad), (K, bad[:10], cov[bad[:10]], want[bad[:10]])
