"""The scoring primitives on the views the correction builds, against plain dynamic programming in numpy.

In the pipeline a reference string is a slice of the packed read (2 bits per base, 4 when the read holds an N) that
starts at any base and walks with step +1 or -1, and the other string is often a 2-bit trail slot whose bits past its
end are stale.  The cases below put every string at such a view, at the length boundaries of the kernels (64-row
blocks, the 2048-base switch between the fused and the striped forms, 128-column overlap stripes), and compare with
row-wise recurrences written here, independent of both the oracle and csrc.  This file runs the host emulation (the
scalar forms, g++); tests/test_gpu_primitives.py runs the same table on the device."""
import numpy as np
import pytest

LENGTHS = (0, 1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 2047, 2048, 2049, 4097)
CODE = np.full(256, 4, dtype=np.int8)
for _ch, _c in zip(b"ACGTUacgtu", (0, 1, 2, 3, 3, 0, 1, 2, 3, 3)):
    CODE[_ch] = _c


# ---------------------------------------------------------------- plain DP (rows = the first string)
def _codes(s: bytes) -> np.ndarray:
    return CODE[np.frombuffer(s, dtype=np.uint8)].astype(np.int64)


def _rows(a: bytes, b: bytes):
    """The shorter string on the rows: every score below is symmetric in its two arguments."""
    return (a, b) if len(a) <= len(b) else (b, a)


def edit_distance_rows(a: bytes, b: bytes) -> np.ndarray:
    """D[i][j] = unit-cost edit distance of a[:i] and b[:j], all rows (for prefix look-ups)."""
    x, y = _codes(a), _codes(b)
    m = len(y)
    ar = np.arange(m + 1)
    D = np.empty((len(x) + 1, m + 1), dtype=np.int32)
    D[0] = ar
    for i in range(1, len(x) + 1):
        p = D[i - 1]
        t = np.empty(m + 1, dtype=np.int64)
        t[0] = i
        t[1:] = np.minimum(p[1:] + 1, p[:-1] + (y != x[i - 1]))
        D[i] = np.minimum.accumulate(t - ar) + ar  # the left neighbour + 1, folded in by a running minimum
    return D


def edit_distance(a: bytes, b: bytes) -> int:
    a, b = _rows(a, b)
    x, y = _codes(a), _codes(b)
    ar = np.arange(len(y) + 1)
    row = ar.copy()
    for i in range(1, len(x) + 1):
        t = np.empty(len(y) + 1, dtype=np.int64)
        t[0] = i
        t[1:] = np.minimum(row[1:] + 1, row[:-1] + (y != x[i - 1]))
        row = np.minimum.accumulate(t - ar) + ar
    return int(row[-1])


def lcs_length(a: bytes, b: bytes) -> int:
    a, b = _rows(a, b)
    x, y = _codes(a), _codes(b)
    row = np.zeros(len(y) + 1, dtype=np.int64)
    for i in range(len(x)):
        t = np.empty_like(row)
        t[0] = 0
        t[1:] = np.maximum(row[1:], row[:-1] + (y == x[i]))
        row = np.maximum.accumulate(t)
    return int(row[-1])


def overlap_score(a: bytes, b: bytes) -> int:
    """match 4, mismatch -3, gap -2; leading gaps of both strings free, trailing gaps charged."""
    a, b = _rows(a, b)
    x, y = _codes(a), _codes(b)
    ar2 = 2 * np.arange(len(y) + 1)
    row = np.zeros(len(y) + 1, dtype=np.int64)
    for i in range(len(x)):
        t = np.empty_like(row)
        t[0] = 0
        t[1:] = np.maximum(row[:-1] + np.where(y == x[i], 4, -3), row[1:] - 2)
        row = np.maximum.accumulate(t + ar2) - ar2
    return int(row[-1])


# ---------------------------------------------------------------- views
class Views:
    """Collects reads and {read, start, step, len} descriptors that present a walk-order string as a view."""

    def __init__(self, rng):
        self.rng = rng
        self.reads = []

    def pad(self, n: int) -> bytes:
        return bytes(self.rng.choice(list(b"ACGT"), n).tolist()) if n > 0 else b""

    def side(self, w: bytes, step: int, lead: int, tail: int, four_bit: bool = False):
        """w in walk order at step +1 / -1 (a slice of a read) or 0 (a trail slot); `lead` / `tail` bases of
        the read lie before / after the slice.  four_bit: the read holds an N (outside the slice if w has none)."""
        body = w[::-1] if step < 0 else w
        lp, tp = bytearray(self.pad(lead)), bytearray(self.pad(tail))
        if four_bit and b"N" not in w:
            assert lead or tail
            if lead:
                lp[self.rng.integers(0, lead)] = ord("N")
            else:
                tp[self.rng.integers(0, tail)] = ord("N")
        start = lead + len(w) - 1 if (step < 0 and w) else lead
        self.reads.append(bytes(lp) + body + bytes(tp))
        return [len(self.reads) - 1, start, step, len(w)]


def placement(v: Views, w: bytes, step: int, i: int, four_bit: bool):
    """The i-th placement of w: starts at every residue mod 32 (2-bit) or 16 (4-bit), flush against base 0 or the
    last base, in reads whose length is or is not a multiple of 32."""
    per = 16 if four_bit else 32
    kind = i % 4
    if kind == 0:    # flush against base 0
        lead = 0
    elif kind == 1:  # flush against the last base
        lead = None
    else:
        lead = (i // 4) % per + per * (i % 3)
    mult32 = (i // 2) % 2 == 0
    if lead is None:
        lead = (-len(w)) % 32 + (0 if mult32 else 5) + (32 if four_bit else 0)
        return v.side(w, step, lead, 0, four_bit)
    tail = (-(lead + len(w))) % 32 if mult32 else (-(lead + len(w))) % 32 + 7
    if four_bit and not lead and not tail and b"N" not in w:
        tail = 32
    return v.side(w, step, lead, tail, four_bit)


def mutate(rng, s: bytes, rate: float, alpha=b"ACGT") -> bytes:
    out = bytearray()
    for ch in s:
        u = rng.random()
        if u < rate / 3:
            continue
        out.append(int(rng.choice(list(alpha))) if u < 2 * rate / 3 else ch)
        if rng.random() < rate / 3:
            out.append(int(rng.choice(list(alpha))))
    return bytes(out)


def boundary_pairs(seed: int = 1, trails: bool = True):
    """Pairs (walk-order strings and their views) at the length table crossed with itself, both steps, 2-bit and
    4-bit reads, trail slots, plus N in either string, identical strings and disjoint alphabets."""
    rng = np.random.default_rng(seed)
    v = Views(rng)
    strings, desc = [], []
    base = bytes(rng.choice(list(b"ACGT"), 5000).tolist())
    i = 0
    for la in LENGTHS:
        for lb in LENGTHS:
            a = base[:la]
            b = mutate(rng, base[: lb + lb // 10], 0.12)[:lb]
            b = b + v.pad(lb - len(b))
            fa, fb = (i % 3 == 1), (i % 5 == 2)
            if fa and la and i % 2:
                a = a[: la // 2] + b"N" + a[la // 2 + 1:]
            if fb and lb and i % 4 == 2:
                b = b[: lb // 3] + b"N" + b[lb // 3 + 1:]
            sa = (1, -1)[i % 2]
            sb = (1, -1, 0)[i % 3] if trails else (1, -1)[(i // 2) % 2]
            if sb == 0 and (fb or b"N" in b):
                sb = -1
            desc.append(placement(v, a, sa, i, fa) + placement(v, b, sb, i + 1, fb))
            strings.append((a, b))
            i += 1
    for n in (1, 64, 65, 129, 2048, 2049):
        s = bytes(rng.choice(list(b"ACGTN"), n, p=[0.24, 0.24, 0.24, 0.24, 0.04]).tolist())
        t = s.replace(b"N", b"A")
        for (x, y, f) in ((s, s, True), (t, t, False), (b"A" * n, b"C" * n, False), (b"A" * n, b"C" * (n + 3), False)):
            for step_b in ((1, -1, 0) if trails and b"N" not in y else (1, -1)):
                desc.append(placement(v, x, -step_b if step_b else 1, i, f) + placement(v, y, step_b, i + 3, f))
                strings.append((x, y))
                i += 1
    return v.reads, np.array(desc, dtype=np.int32), strings


def check_scores(run, reads, desc, strings, ops=(0, 1, 2, 5)):
    """run(op, reads, desc) -> results of talc_test_align_slices (or its host emulation) for ops 0, 1, 2, 5."""
    res = {op: run(op, reads, desc) for op in ops}
    for i, (a, b) in enumerate(strings):
        want_nw, want_lcs = -edit_distance(a, b), lcs_length(a, b)
        where = (i, len(a), len(b), list(desc[i]))
        if 0 in res:
            assert res[0][i] == want_nw, ("distance",) + where
        if 1 in res:
            assert res[1][i] == want_lcs, ("lcs",) + where
        if 2 in res:
            assert res[2][i] == overlap_score(a, b), ("overlap",) + where
        if 5 in res:
            assert (int(res[5][i][0]), int(res[5][i][1])) == (want_nw, want_lcs), ("fused",) + where


# ---------------------------------------------------------------- the host emulation
def test_reference_dp_agrees_with_the_oracle():
    """The numpy recurrences restate the oracle's global / local / overlap scores on non-empty strings."""
    from oracle import pyoracle as po
    rng = np.random.default_rng(3)
    for _ in range(60):
        a = bytes(rng.choice(list(b"ACGTN"), int(rng.integers(1, 90))).tolist())
        b = mutate(rng, a, 0.3, b"ACGTN") or b"A"
        assert -edit_distance(a, b) == po.nw(a, b)
        assert lcs_length(a, b) == po.lcs(a, b)
        assert overlap_score(a, b) == po.overlap(a, b, True)
        D = edit_distance_rows(a, b)
        assert D[len(a)][len(b)] == edit_distance(a, b) and D[len(a)][0] == len(a) and D[0][len(b)] == len(b)


def test_scalar_forms_on_slices_at_the_boundaries():
    import pyemu
    reads, desc, strings = boundary_pairs(seed=1)
    check_scores(lambda op, r, d: pyemu.align_slices(op, r, d), reads, desc, strings)


def test_scalar_distance_of_an_empty_string_is_the_other_length():
    import pyemu
    v = Views(np.random.default_rng(2))
    desc, strings = [], []
    for n in (0, 1, 4, 64, 65, 3000):
        s = v.pad(n)
        for step in (1, -1, 0):
            desc.append(v.side(b"", 1, 3, 5) + v.side(s, step, 2, 9))
            desc.append(v.side(s, step if step else 1, 0, 4, True) + v.side(b"", -1, 7, 0))
            strings += [(b"", s), (s, b"")]
    reads = v.reads
    d = np.array(desc, dtype=np.int32)
    nw = pyemu.align_slices(0, reads, d)
    assert [int(x) for x in nw] == [-max(len(a), len(b)) for a, b in strings]
    check_scores(lambda op, r, dd: pyemu.align_slices(op, r, dd), reads, d, strings)


SEED_X = (3, 31, 32, 63, 64, 127, 128, 255, 256, 300)


def seed_extension_pairs(right: bool, k: int, n_pairs: int = 40):
    """Pairs as the corrector hands them to seed_and_extension: a read slice (step +1 for a search to the right, -1 to
    the left) and a trail slot, in either order, sharing the anchor k-mer at the start of the walk."""
    rng = np.random.default_rng(5 if right else 6)
    v = Views(rng)
    desc, strings = [], []
    for i in range(n_pairs):
        n = int(rng.integers(k + 1, 700 if i % 4 else 2600))
        r = v.pad(n)
        c = r[:k] + mutate(rng, r[k:], float(rng.choice([0.02, 0.1, 0.3])))
        if i % 5 == 0:
            c = c[: max(k + 1, len(c) // 3)]
        if i % 7 == 3:
            c = r[:k] + v.pad(len(c) - k)  # unrelated past the anchor
        step = 1 if right else -1
        if i % 2:
            desc.append(placement(v, r, step, i, i % 3 == 0) + placement(v, c, 0, i + 1, False))
            strings.append((r, c))
        else:
            desc.append(placement(v, c, 0, i, False) + placement(v, r, step, i + 1, i % 3 == 0))
            strings.append((c, r))
    return v.reads, np.array(desc, dtype=np.int32), strings


@pytest.mark.parametrize("right", [True, False])
def test_scalar_seed_extension_on_slices(right):
    """seed_and_extension on those views against the oracle, and its score against the plain edit distance of the
    two extended prefixes."""
    import pyemu
    k = 21
    reads, d, strings = seed_extension_pairs(right, k)
    for x in SEED_X:
        res = pyemu.align_slices(3, reads, d, aux=x, aux2=1 if right else 0, k=k)
        check_seed_extension(res, strings, x, right, k)


def check_seed_extension(res, strings, x, right, k):
    from oracle import pyoracle as po
    for i, (r, c) in enumerate(strings):
        want = po.seed_extend(r, c, x, True, k) if right else po.seed_extend(r[::-1], c[::-1], x, False, k)
        re_, ce_, _, sc, stop = want
        assert tuple(int(t) for t in res[i]) == (re_, ce_, int(sc), int(stop)), (i, x, right)
        if not stop:
            assert res[i][2] == -edit_distance(r[:re_], c[:ce_]), (i, x, right)
