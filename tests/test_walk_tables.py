"""The walk's device-only lookups and decisions against plain references.

Every walk step decides from three pieces that exist only on the device: the successor tables (one bucket per (K-1)-mer
context with the counts of its four successors, table.cuh), the count-model tables (model_tabs_kernel) and the fast
walks' child choice (fast_step_child, model.cuh).  The host emulation asks the k-mer table four times and runs without
model tables, so only the self-test entries talc_test_successors / talc_test_model reach them.  References here:

- the count model restated in Python floats (Python never contracts a multiply-add, so this is the separate mul / add
  double arithmetic of the reference) and in fractions.Fraction, to find alphas where a contracted (fused) bound decides
  otherwise than the reference's unfused one;
- a dictionary of the key set for the successor tables, and Python restatements of hash_kmer, hash_ctx and both
  capacity rules, used only to build layouts whose probe chains wrap around the end of the tables.
"""
import math
from fractions import Fraction

import numpy as np
import pytest

from conftest import have_gpu

E, U, B = 0, 1, 2  # model.cuh Tag
M64 = (1 << 64) - 1
TAB_N = 16384  # kModelTabN


# ---------------------------------------------------------------------------------------------------- count model
def lower_bound(cc, a):
    if cc <= 3:
        x = float(cc) - 0.5
        return math.nan if x < 0 else x + (1 - a) * math.sqrt(x)
    y = a / 2 - math.sqrt(float(cc) + 0.02)
    return y * y


def upper_bound(cc, a):
    if cc <= 3:
        x = float(cc) + 0.5
        return x + a * math.sqrt(x)
    y = a / 2 + math.sqrt(float(cc) + 0.96)
    return y * y


def upper_bound_fused(cc, a):
    """the same with (cc + 0.5) + alpha * sqrt(cc + 0.5) contracted: the correctly rounded exact value"""
    if cc <= 3:
        x = float(cc) + 0.5
        return float(Fraction(x) + Fraction(a) * Fraction(math.sqrt(x)))
    return upper_bound(cc, a)


def upper_exact_holds(nextc, cc, a):
    """nextc <= (cc + 0.5) + alpha * sqrt(cc + 0.5) in exact arithmetic (cc <= 3)"""
    x = Fraction(cc) + Fraction(1, 2)
    d = Fraction(nextc) - x
    return d <= 0 or (a >= 0 and d * d <= Fraction(a) ** 2 * x)


class Model:
    def __init__(self, alpha, sr, min_count=2, upper=upper_bound):
        self.a, self.sr, self.mc, self.upper = alpha, sr, min_count, upper

    def step_bounds(self, count):
        lam = int(float(count) * self.sr)
        noise = lam >= self.mc
        return (lower_bound(count, self.a), self.upper(lam, self.a) if noise else 0.0, math.sqrt(float(count)), lam,
                noise)

    def tags(self, c4, cm, count, complex_=False):
        lower, up, sq, lam, noise = self.step_bounds(count)
        counter = sum(c >= self.mc for c in c4)
        if counter == 0:
            return 0, [U] * 4, [0.0] * 4
        tag, nE, nB, nU = [U] * 4, 0, 0, 0
        for b in range(4):
            c = c4[b]
            if c >= self.mc:
                if c >= lower or counter == 1:
                    tag[b] = E
                    nE += 1
                elif noise:
                    if not (c <= up) or (cm >> b) & 1:
                        tag[b] = B
                        nB += 1
                    else:
                        tag[b] = U
                        nU += 1
                else:
                    tag[b] = B
                    nB += 1
        if nE == 0 and nB == 1:
            tag = [E if t == B else t for t in tag]
        if nE == 1 and nU > 0 and not complex_:
            s, index = 0, 0
            for i in range(4):
                if tag[i] == U:
                    if s == 0:
                        index = i
                    s += c4[i]
                    if c4[index] < c4[i]:
                        index = i
            if not (float(s & 0xFFFFFFFF) <= up):
                tag[index] = B
        dist = []
        for c in c4:
            num = abs(float(count) - float(c))
            dist.append(num / sq if sq else (math.inf if num else math.nan))
        return 4, tag, dist

    def child(self, c4, cm, count):
        m = [c >= self.mc for c in c4]
        if sum(m) == 1:
            return m.index(True)
        if sum(m) == 0:
            return -1
        n, tag, _ = self.tags(c4, cm, count, False)
        kids = [i for i in range(4) if tag[i] != U]
        return kids[0] if len(kids) == 1 else -1

    def row(self, op, a):
        """the uint64[9] result of selftest_model_op for args a"""
        out = [0] * 9
        if op == 0:
            lo, up, sq, lam, noise = self.step_bounds(a[0])
            out[:5] = [dbits(lo), dbits(up), dbits(sq), lam, int(noise)]
        elif op == 1:
            n, tag, dist = self.tags(a[1:5], a[5], a[0], bool(a[6]))
            if n:
                out = [n] + tag + [dbits(d) for d in dist]
        elif op == 2:
            out[0] = self.child(a[1:5], a[5], a[0]) & M64
        elif op == 3:
            out[0] = int(a[0] <= self.upper(a[1], self.a))
        elif op == 4:
            out[0] = int(a[0] <= self.upper(a[1], self.a) and a[0] >= lower_bound(a[1], self.a))
        return out


def dbits(x):
    return int(np.array([x], dtype=np.float64).view(np.uint64)[0])


DOUBLE_COLS = {0: (0, 1, 2), 1: (5, 6, 7, 8), 2: (), 3: (), 4: ()}


def assert_rows(op, got, want, what):
    """bit for bit, except that any NaN equals any NaN (x86 and the GPU make NaNs of different sign)"""
    got = np.asarray(got, dtype=np.uint64)
    want = np.asarray(want, dtype=np.uint64).reshape(got.shape)
    g, w = got.copy(), want.copy()
    for c in DOUBLE_COLS[op]:
        gn, wn = np.isnan(got[:, c].view(np.float64)), np.isnan(want[:, c].view(np.float64))
        both = gn & wn
        g[both, c] = w[both, c] = 0
    bad = np.nonzero((g != w).any(axis=1))[0]
    assert len(bad) == 0, "%s op %d: %d rows differ, first %d: got %s want %s" % (
        what, op, len(bad), bad[0], [hex(int(x)) for x in got[bad[0]]], [hex(int(x)) for x in want[bad[0]]])


def fused_near_ties(lo=0.67, max_bound=40):
    """(cc, nextc, alpha): alphas >= lo where the unfused bound of cc in {1, 2, 3} lands on the integer nextc and the
    fused one does not (or the reverse); found by walking a few ulps around nextc = (cc + 0.5) + alpha * sqrt(cc + .5)"""
    out = []
    for cc in (1, 2, 3):
        x = cc + 0.5
        s = math.sqrt(x)
        for n in range(cc + 1, max_bound + 1):
            a0 = (n - x) / s
            for k in range(-4, 5):
                a = a0
                for _ in range(abs(k)):
                    a = math.nextafter(a, math.inf if k > 0 else -math.inf)
                if a >= lo and (n <= upper_bound(cc, a)) != (n <= upper_bound_fused(cc, a)):
                    out.append((cc, n, a))
    return out


TIES = fused_near_ties()
ALPHAS = [2.57, 0.67] + sorted({a for _, _, a in TIES})
# (alpha, sr_error_rate) of the model tests: every alpha at the default rate, the edges of the accepted rates at 2.57
PARAMS = [(a, 0.025) for a in ALPHAS] + [(2.57, 0.0), (2.57, 0.5)]


def tie_case(cc, n, a):
    """(min_count, sr, args) of a step whose tags and child hinge on the tie: count 10000 with lambda = cc, successors
    {10000, n, 0, 0}; n lies far below the lower bound of 10000, so only the noise interval of lambda decides it"""
    return (1 if cc < 2 else 2), (cc + 0.5) / 10000, [10000, 10000, n, 0, 0, 0, 0, 0]


def model_counts(alpha, sr):
    """counts where model kernels go wrong: the cc <= 3 branch, the table edge, lambda around MIN_COUNT, count * sr
    within an ulp of an integer, the top of int and of u32, and a random sweep"""
    cs = list(range(0, 5)) + list(range(TAB_N - 2, TAB_N + 3)) + [79, 80, 81, 119, 120, 121, (1 << 31) - 1, M64 >> 32]
    if sr > 0:
        near = [c for c in range(1, 200000) if abs(c * sr - round(c * sr)) <= math.ulp(c * sr) and c * sr >= 1]
        cs += near[:40]
    rng = np.random.default_rng(int(alpha * 1000) + int(sr * 1e6))
    cs += [int(x) for x in rng.integers(0, 1 << 32, 60, dtype=np.uint64)]
    cs += [int(x) for x in rng.integers(0, 40000, 60)]
    return sorted(set(cs))


def model_vectors(alpha, sr):
    """args of ops 0-4: successor counts around both bounds of every count, with every colour mask and complex flag"""
    m = Model(alpha, sr)
    rng = np.random.default_rng(7)
    v0, v1, v34 = [], [], []
    for c in model_counts(alpha, sr):
        v0.append([c])
        lo, up, _, lam, _ = m.step_bounds(c)
        near = {0, 1, 2, 3, c, c // 2, lam, lam + 1}
        for b in (lo, up):
            if math.isfinite(b) and 0 <= b < 2 ** 32:
                near |= {int(b), int(b) + 1, max(int(b) - 1, 0)}
        near = sorted(x for x in near if 0 <= x <= M64 >> 32)
        for x in near:
            v1.append([c, c, x, 0, 0, 0, 0])
            v1.append([c, x, 0, x, 1, 2, 0])
            v1.append([c, x, x, x, x, int(rng.integers(0, 16)), 1])
            v1.append([c, 0, x, 0, lam, 0, 0])
            v34.append([x, c])
        v1.append([c, c, lam, lam, 0, 0, 0])  # two UNEXPECTED successors whose sum may leave the noise interval
        v1.append([c, c, lam, lam, 0, 0, 1])
        v1.append([c] + [int(y) for y in rng.integers(0, min(2 * c + 8, 1 << 32), 4)] + [int(rng.integers(0, 16)), int(rng.integers(0, 2))])
        v1.append([c, 1, 1, 1, 1, 15, 0])
        v1.append([c, 0, 0, 0, 0, 0, 0])
    return {0: v0, 1: v1, 2: [r[:6] for r in v1], 3: v34, 4: v34}


# ---------------------------------------------------------------------------------------------------- tables
def hash_kmer(k):
    k = np.asarray(k, dtype=np.uint64).copy()
    with np.errstate(over="ignore"):
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xff51afd7ed558ccd)
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xc4ceb9fe1a85ec53)
        k ^= k >> np.uint64(33)
    return k


def hash_ctx(c):
    c = np.asarray(c, dtype=np.uint64).copy()
    with np.errstate(over="ignore"):
        c *= np.uint64(0x9E3779B97F4A7C15)
    return c ^ (c >> np.uint64(32))


def kmer_capacity(n):  # build_table_device: slots for n kept entries (load <= 1/2)
    cap = 2
    while cap < 2 * n + 2:
        cap <<= 1
    return cap


def ctx_capacity(n):  # build_ctx_tables: buckets for n entries (load <= 1/3)
    cap = 4
    while cap < 3 * n + 4:
        cap <<= 1
    return cap


def kmask(k):
    return np.uint64((1 << (2 * k)) - 1)


class Ref:
    """the dictionary reference: keys (sorted, distinct), counts (u32) and colours of the sealed k-mer table"""

    def __init__(self, k, keys, counts, colours=None):
        o = np.argsort(keys)
        self.k, self.keys = k, np.asarray(keys, dtype=np.uint64)[o]
        self.counts = np.asarray(counts, dtype=np.uint32)[o]
        self.colours = (np.zeros(len(o), np.uint32) if colours is None else np.asarray(colours, np.uint32)[o])

    def get(self, q):
        q = np.asarray(q, dtype=np.uint64)
        pos = np.minimum(np.searchsorted(self.keys, q), len(self.keys) - 1)
        hit = self.keys[pos] == q
        return np.where(hit, self.counts[pos], 0).astype(np.uint32), np.where(hit, self.colours[pos], 0), hit

    def successors(self, kmers, right):
        """counts and colour bits of c+b (right) or b+c (left) for the context c of each k-mer"""
        k = self.k
        kmers = np.asarray(kmers, dtype=np.uint64)
        cnt = np.zeros((len(kmers), 4), np.uint32)
        cm = np.zeros(len(kmers), np.uint32)
        for b in range(4):
            if right:
                succ = ((kmers << np.uint64(2)) | np.uint64(b)) & kmask(k)
            else:
                succ = (kmers >> np.uint64(2)) | (np.uint64(b) << np.uint64(2 * (k - 1)))
            c, col, _ = self.get(succ)
            cnt[:, b] = c
            cm |= (col > 0).astype(np.uint32) << np.uint32(b)
        return cnt, cm


def ctx_of(kmers, right, k):
    kmers = np.asarray(kmers, dtype=np.uint64)
    return kmers & kmask(k - 1) if right else kmers >> np.uint64(2)


def kmer_with_ctx(ctx, right):
    """a k-mer whose walk context is ctx (first base A on the right, last base A on the left)"""
    ctx = np.asarray(ctx, dtype=np.uint64)
    return ctx if right else ctx << np.uint64(2)


def pick_ctx(rng, k, cap, home, n, exclude=()):
    """n distinct (K-1)-mer contexts whose bucket is `home` in a table of cap buckets"""
    got, ex = [], set(int(x) for x in exclude)
    while len(got) < n:
        c = rng.integers(0, 1 << (2 * (k - 1)), 1 << 21, dtype=np.uint64)
        c = c[(hash_ctx(c) & np.uint64(cap - 1)) == np.uint64(home)]
        for x in c.tolist():
            if x not in ex:
                ex.add(x)
                got.append(x)
    return np.array(got[:n], dtype=np.uint64)


def pick_kmers_home_sector(rng, k, cap, sector, n, exclude=()):
    got, ex = [], set(int(x) for x in exclude)
    while len(got) < n:
        x = rng.integers(0, 1 << (2 * k), 1 << 21, dtype=np.uint64)
        x = x[(hash_kmer(x) & np.uint64(cap - 1) & ~np.uint64(1)) == np.uint64(sector)]
        for y in x.tolist():
            if y not in ex:
                ex.add(y)
                got.append(y)
    return np.array(got[:n], dtype=np.uint64)


def adversarial_layout(k, ctx_cap, seed=0):
    """k-mers (count 2..5) for a table whose successor tables have ctx_cap buckets: per direction 40 present contexts
    in the last bucket (the chain crosses into bucket 0) and 30 in one mid bucket (far past the home pair); 40 k-mers
    with their home sector at cap - 2 in the k-mer table; random fill up to the most entries that keep ctx_cap.
    Returns (keys, counts, absent contexts {right: [...], left: [...]}, k-mers homed at cap - 2)."""
    rng = np.random.default_rng(seed + 1000 * k + ctx_cap)
    n = (ctx_cap - 4) // 3
    kcap = kmer_capacity(n)
    keys, absent = [], {}
    top = np.uint64(2 * (k - 1))
    used = set()
    for right in (True, False):
        homes = [ctx_cap - 1, ctx_cap // 2 + 3]
        present = [pick_ctx(rng, k, ctx_cap, homes[0], 40, used), pick_ctx(rng, k, ctx_cap, homes[1], 30, used)]
        ab = [pick_ctx(rng, k, ctx_cap, h, 6, used | set(np.concatenate(present).tolist())) for h in homes]
        for arr in present + ab:
            used |= set(arr.tolist())
        absent[right] = np.concatenate(ab)
        for grp in present:
            for i, c in enumerate(grp):
                for b in range(1 + i % 4):  # 1..4 successors
                    keys.append(int((c << np.uint64(2)) | np.uint64(b)) if right else int((np.uint64(b) << top) | c))
    wrap = pick_kmers_home_sector(rng, k, kcap, kcap - 2, 40, keys)
    keys = list(dict.fromkeys(keys + wrap.tolist()))
    fill = rng.integers(0, 1 << (2 * k), 3 * n, dtype=np.uint64).tolist()
    seen = set(keys)
    for x in fill:
        if len(keys) >= n:
            break
        if x not in seen:
            seen.add(x)
            keys.append(x)
    keys = np.array(keys[:n], dtype=np.uint64)
    counts = rng.integers(2, 6, len(keys)).astype(np.int64)
    # the absent contexts must really be absent from the final key set
    ref = Ref(k, keys, counts)
    for right in (True, False):
        cnt, _ = ref.successors(kmer_with_ctx(absent[right], right), right)
        absent[right] = absent[right][cnt.sum(axis=1) == 0]
    return keys, counts, absent, wrap


def probe_layout(keys, k, ctx_cap, right):
    """bucket of every present context after sequential linear probing in key order (the device's CAS order differs,
    but the chains wrap and run long in every order)"""
    ctx = np.unique(keys >> np.uint64(2) if right else keys & kmask(k - 1))
    occ = np.zeros(ctx_cap, bool)
    where = {}
    for c, h in zip(ctx.tolist(), (hash_ctx(ctx) & np.uint64(ctx_cap - 1)).tolist()):
        i = h
        while occ[i]:
            i = (i + 1) % ctx_cap
        occ[i] = True
        where[c] = (h, i)
    return where, occ


def test_near_ties_are_not_vacuous():
    """the Fraction search finds the alphas of the issue (10 alphas >= 0.67), and at each the unfused, fused and exact
    decisions do not all agree; at tag level the unfused and fused tags and children differ"""
    assert len(TIES) >= 10
    assert (2, 4, 0.9486832980505135) in TIES
    for cc, n, a in TIES:
        unf, fus, ex = n <= upper_bound(cc, a), n <= upper_bound_fused(cc, a), upper_exact_holds(n, cc, a)
        assert unf != fus
        mc, sr, args = tie_case(cc, n, a)
        mu, mf = Model(a, sr, mc), Model(a, sr, mc, upper_bound_fused)
        assert mu.step_bounds(10000)[3] == cc
        assert mu.tags(args[1:5], 0, 10000)[1] != mf.tags(args[1:5], 0, 10000)[1]
        assert mu.child(args[1:5], 0, 10000) != mf.child(args[1:5], 0, 10000)
        assert (unf, fus, ex).count(True) in (1, 2)
    # the example of the issue: {100, 4, 0, 0} at count 100 and the default rate
    m = Model(0.9486832980505135, 0.025)
    assert m.tags([100, 4, 0, 0], 0, 100)[1] == [E, U, U, U]
    assert Model(0.9486832980505135, 0.025, upper=upper_bound_fused).tags([100, 4, 0, 0], 0, 100)[1] == [E, B, U, U]


@pytest.mark.parametrize("alpha,sr", PARAMS[:4] + PARAMS[-2:])
def test_python_model_is_the_oracle(alpha, sr):
    """the Python model tags as the oracle's tagNextNodes on every vector of the model tests"""
    from oracle import pyoracle as po
    p = po.make_params(k=21, alpha=alpha, sr_error=sr)
    m = Model(alpha, sr)
    for a in model_vectors(alpha, sr)[1]:
        n, tags, dist = po.tag_next_nodes(p, a[1:5], [(a[5] >> b) & 1 for b in range(4)], a[0], bool(a[6]))
        wn, wt, wd = m.tags(a[1:5], a[5], a[0], bool(a[6]))
        assert n == wn, a
        if n:
            assert [{0: E, 1: U, 7: B}[int(t)] for t in tags] == wt, a
            for i in range(4):
                if wt[i] != U and not (math.isnan(dist[i]) and math.isnan(wd[i])):
                    assert dist[i] == wd[i], a


@pytest.mark.parametrize("use_tabs", [False, True])
def test_emu_model_is_the_python_model(use_tabs):
    """talc_test_model in the host emulation, computed path and tabulated path, bit for bit against the Python model,
    the near-tie steps included"""
    import pyemu
    from oracle import pyoracle as po
    for alpha, sr in PARAMS:
        ep = pyemu.params_from(po.make_params(k=21, alpha=alpha, sr_error=sr))
        m = Model(alpha, sr)
        for op, vecs in model_vectors(alpha, sr).items():
            got = pyemu.test_model(ep, op, vecs, use_tabs)
            assert_rows(op, got, [m.row(op, v) for v in vecs], "emu alpha %r sr %r" % (alpha, sr))
    for cc, n, a in TIES:
        mc, sr, args = tie_case(cc, n, a)
        ep = pyemu.params_from(po.make_params(k=21, min_count=mc, alpha=a, sr_error=sr))
        m = Model(a, sr, mc)
        for op in (1, 2):
            assert_rows(op, pyemu.test_model(ep, op, [args], use_tabs), [m.row(op, args)], "emu tie %r" % a)


@pytest.mark.parametrize("k,cap", [(21, 1 << 10), (31, 1 << 14)])
def test_adversarial_layouts_collide_and_wrap(k, cap):
    """the layouts used on the GPU really put dozens of contexts in the last bucket (so chains cross into bucket 0),
    chains far past the home pair, absent contexts homed on long chains and on empty buckets, and k-mer home sectors at
    cap - 2, under the restated hashes and capacity rules"""
    keys, counts, absent, wrap = adversarial_layout(k, cap)
    n = len(keys)
    assert ctx_capacity(n) == cap
    kcap = kmer_capacity(n)
    assert ((hash_kmer(wrap) & np.uint64(kcap - 1) & ~np.uint64(1)) == np.uint64(kcap - 2)).all() and len(wrap) == 40
    for right in (True, False):
        where, occ = probe_layout(keys, k, cap, right)
        homes = np.array([h for h, _ in where.values()])
        assert (homes == cap - 1).sum() >= 40
        assert any(h == cap - 1 and i < 30 for h, i in where.values())  # wrapped
        assert max((i - h) % cap for h, i in where.values()) >= 30  # far past the home pair
        ah = hash_ctx(absent[right]) & np.uint64(cap - 1)
        assert len(absent[right]) >= 10 and (ah == np.uint64(cap - 1)).any()


def test_sr_error_rate_is_refused_at_context_creation():
    """NaN and rates outside [0, 0.5] are refused before any device call (TALC_ERR_ARG with a message); the accepted
    rates pass the check (on a machine without a GPU they then fail for want of a device, which is not TALC_ERR_ARG)"""
    from talc_b200 import api
    for bad in (math.nan, -0.01, 0.51, 2.0, math.inf):
        with pytest.raises(api.TalcError, match=r"\(-1\).*sr_error_rate"):
            api.Talc(api.default_params(21, sr_error_rate=bad))
    if not have_gpu():
        for ok in (0.0, 0.025, 0.5):
            with pytest.raises(api.TalcError, match=r"\(-2\)"):
                api.Talc(api.default_params(21, sr_error_rate=ok))


# ---------------------------------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    if not have_gpu():
        pytest.fail("GPU tests selected but no CUDA device is visible")
    from talc_b200 import api as _api
    return _api


@gpu
def test_sr_error_rate_accepted_range(api):
    for ok in (0.0, 0.025, 0.5):
        api.Talc(api.default_params(21, sr_error_rate=ok)).close()
    with pytest.raises(api.TalcError):
        api.Talc(api.default_params(21, sr_error_rate=0.5000000000000001))


@gpu
def test_model_ops_are_the_python_model(api):
    """ops 0-4 on the device's own model tables (and the computed path past them) bit for bit against the Python
    float64 model, for the default alpha, 0.67, every FMA-sensitive alpha and the edge rates"""
    for alpha, sr in PARAMS:
        t = api.Talc(api.default_params(21, alpha=alpha, sr_error_rate=sr))
        m = Model(alpha, sr)
        for op, vecs in model_vectors(alpha, sr).items():
            assert_rows(op, t.test_model(op, vecs), [m.row(op, v) for v in vecs], "alpha %r sr %r" % (alpha, sr))
        t.close()


@gpu
def test_model_near_ties_take_the_unfused_answer(api):
    """at every FMA-sensitive alpha the device tags and picks the child as the unfused reference, not as a fused
    (contracted) or exact evaluation would"""
    for cc, n, a in TIES:
        mc, sr, args = tie_case(cc, n, a)
        t = api.Talc(api.default_params(21, min_count=mc, alpha=a, sr_error_rate=sr))
        mu, mf = Model(a, sr, mc), Model(a, sr, mc, upper_bound_fused)
        for op in (1, 2):
            got = t.test_model(op, [args])
            assert_rows(op, got, [mu.row(op, args)], "tie alpha %r" % a)
            assert list(got[0]) != mf.row(op, args)
        for nextc in (n - 1, n, n + 1):  # op 3 at lambda itself
            assert int(t.test_model(3, [[nextc, cc]])[0, 0]) == int(nextc <= upper_bound(cc, a))
        t.close()
    # the example: {100, 4, 0, 0} at count 100 and the default rate
    t = api.Talc(api.default_params(21, alpha=0.9486832980505135))
    assert list(t.test_model(1, [[100, 100, 4, 0, 0, 0, 0]])[0, :5]) == [4, E, U, U, U]
    assert int(t.test_model(2, [[100, 100, 4, 0, 0, 0]])[0, 0]) == 0


@gpu
def test_fast_child_in_complex_regions(api):
    """op 2 is the unique non-UNEXPECTED tag of the reference with complex = false, else -1.  The fast walk always tags
    with complex = false; in a complex region the reference can only tag fewer successors BREAKPOINT (the last rule is
    skipped), so where op 2 picks a child, complex = true tags at most as many children: the fast walk never takes a
    step that the general step would not, and where they differ it falls back to the general step."""
    t = api.Talc(api.default_params(21))
    m = Model(2.57, 0.025)
    vecs = model_vectors(2.57, 0.025)[1]
    child = t.test_model(2, [v[:6] for v in vecs])[:, 0].astype(np.int64)
    tc = t.test_model(1, [v[:6] + [1] for v in vecs])
    tn = t.test_model(1, [v[:6] + [0] for v in vecs])
    differ = 0
    for v, ch, rc, rn in zip(vecs, child, tc, tn):
        n, tags, _ = m.tags(v[1:5], v[5], v[0], False)
        kids = [i for i in range(4) if n and tags[i] != U]
        assert ch == (kids[0] if len(kids) == 1 else -1), v
        kc = [i for i in range(4) if rc[0] and rc[1 + i] != U]
        kn = [i for i in range(4) if rn[0] and rn[1 + i] != U]
        assert set(kc) <= set(kn)
        differ += kc != kn
    assert differ > 0  # the complex flag does decide some of these vectors


def _check_successors(t, ref, queries_right, queries_left, what, cap=None):
    for right, q in ((True, queries_right), (False, queries_left)):
        q = np.asarray(q, dtype=np.uint64)
        cnt, cm, c = t.test_successors(q, right)
        wc, wm = ref.successors(q, right)
        bad = np.nonzero((cnt != wc).any(axis=1) | (cm != wm))[0]
        assert len(bad) == 0, "%s %s: %d of %d differ, e.g. kmer %#x got %s/%d want %s/%d" % (
            what, "right" if right else "left", len(bad), len(q), int(q[bad[0]]), cnt[bad[0]], cm[bad[0]], wc[bad[0]],
            wm[bad[0]])
        if cap is not None:
            assert c == cap, (what, c, cap)


def _all_queries(ref, absent_r=(), absent_l=()):
    k = ref.k
    r = np.concatenate([kmer_with_ctx(ref.keys >> np.uint64(2), True), kmer_with_ctx(np.asarray(absent_r, np.uint64), True)])
    lft = np.concatenate([kmer_with_ctx(ref.keys & kmask(k - 1), False),
                          kmer_with_ctx(np.asarray(absent_l, np.uint64), False)])
    # every stored k-mer as the walk holds it too: its own successors
    return np.concatenate([r, ref.keys]), np.concatenate([lft, ref.keys])


@gpu
@pytest.mark.parametrize("k,cap", [(21, 1 << 10), (21, 1 << 12), (31, 1 << 14), (17, 1 << 13)])
def test_successor_tables_on_adversarial_layouts(api, k, cap):
    """chains that wrap, run far past the home pair, and absent contexts homed on them and on empty buckets; the same
    for the k-mer table (talc_table_lookup) with home sectors at cap - 2"""
    keys, counts, absent, wrap = adversarial_layout(k, cap)
    ref = Ref(k, keys, counts)
    t = api.Talc(api.default_params(k))
    assert t.load_packed(keys, counts) == len(keys)
    rng = np.random.default_rng(k)
    rnd = rng.integers(0, 1 << (2 * (k - 1)), 4000, dtype=np.uint64)
    qr, ql = _all_queries(ref, np.concatenate([absent[True], rnd]), np.concatenate([absent[False], rnd]))
    _check_successors(t, ref, qr, ql, "layout", ctx_capacity(len(keys)))
    assert t.table_info()["capacity"] == kmer_capacity(len(keys))
    probe = np.concatenate([keys, wrap ^ np.uint64(1), rng.integers(0, 1 << (2 * k), 4000, dtype=np.uint64)])
    c, _, f = t.lookup(probe)
    wc, _, hit = ref.get(probe)
    assert np.array_equal(c, wc) and np.array_equal(f.astype(bool), hit)


def _value_table(k):
    """every colour bit alone and all four together; counts 1, 0x7FFFFFFF and -1 (0xFFFFFFFF, kept by the unsigned
    MIN_COUNT compare); a k-mer that is its own successor (poly-A, poly-T: colour cleared as a homopolymer)"""
    rng = np.random.default_rng(k + 5)
    top = 2 * (k - 1)
    keys, counts, jkeys = [], [], []
    ctxs = rng.integers(1, 1 << (2 * (k - 1)) - 1, 12, dtype=np.uint64).tolist()
    for i, c in enumerate(ctxs[:6]):
        for b in range(4):
            x = (c << 2) | b
            keys.append(x)
            counts.append([1, 0x7FFFFFFF, -1, 7][b])
            if i < 4 and b == i or i == 4:
                jkeys.append(x)
    for i, c in enumerate(ctxs[6:]):
        for b in range(4):
            x = (b << top) | c
            keys.append(x)
            counts.append([3, -1, 1, 0x7FFFFFFF][(b + i) % 4])
            if i < 4 and b == i or i == 4:
                jkeys.append(x)
    poly_a, poly_t = 0, (1 << (2 * k)) - 1
    keys += [poly_a, poly_t, 1]  # 1 = A..AC: poly-A's right successor C and left successor of itself
    counts += [9, 4, 5]
    jkeys += [poly_a]
    keys = np.array(keys, dtype=np.uint64)
    _, first = np.unique(keys, return_index=True)
    keys, counts = keys[np.sort(first)], np.array(counts, dtype=np.int64)[np.sort(first)]
    jkeys = np.array([x for x in jkeys if x in set(keys.tolist())], dtype=np.uint64)
    jcounts = np.arange(1, len(jkeys) + 1, dtype=np.int64) * 37
    rcs = set(_revcomp(jkeys, k).tolist())
    colours = np.array([0 if x in (poly_a, poly_t) else (int(jcounts[list(jkeys).index(x)]) if x in set(jkeys.tolist())
                        else 0) for x in keys.tolist()], dtype=np.uint32)
    assert not (rcs & set(keys.tolist())) - {poly_a, poly_t}  # no colour lands on a reverse complement
    return keys, counts, jkeys, jcounts, colours


def _revcomp(x, k):
    x = np.asarray(x, dtype=np.uint64).copy()
    r = np.zeros_like(x)
    for _ in range(k):
        r = (r << np.uint64(2)) | (np.uint64(3) - (x & np.uint64(3)))
        x >>= np.uint64(2)
    return r


@gpu
@pytest.mark.parametrize("k", [16, 21, 31])
def test_successor_values(api, k):
    keys, counts, jkeys, jcounts, colours = _value_table(k)
    ref = Ref(k, keys, counts.astype(np.uint64) & np.uint64(0xFFFFFFFF), colours)
    t = api.Talc(api.default_params(k, min_count=1))
    t.load_packed(keys, counts, jkeys, jcounts)
    c, col, f = t.lookup(keys)
    assert np.array_equal(c, ref.get(keys)[0]) and np.array_equal(col, ref.get(keys)[1]) and f.all()
    qr, ql = _all_queries(ref)
    _check_successors(t, ref, qr, ql, "values")
    masks = set(ref.successors(qr, True)[1].tolist()) | set(ref.successors(ql, False)[1].tolist())
    assert {1, 2, 4, 8, 15} <= masks
    cnt, _, _ = t.test_successors(np.array([0], np.uint64), True)  # poly-A: its own successor, and A..AC
    assert list(cnt[0]) == [9, 5, 0, 0]


@gpu
@pytest.mark.parametrize("k", [2, 3, 16, 17, 21, 30, 31])
def test_successor_tables_every_k(api, k):
    """all contexts of a random table (every k-mer at K = 2, 3) and absent ones; at K = 31 keys with the top bits set,
    so that contexts use 60 bits and the LEFT base is key >> 60"""
    rng = np.random.default_rng(100 + k)
    if k <= 3:
        keys = np.arange(1 << (2 * k), dtype=np.uint64)
        keys = keys[rng.random(len(keys)) < 0.6]
    else:
        keys = np.unique(rng.integers(0, 1 << (2 * k), 6000, dtype=np.uint64))
        if k == 31:
            keys = np.unique(keys | np.uint64(3 << 60))
    counts = rng.integers(2, 1000, len(keys)).astype(np.int64)
    ref = Ref(k, keys, counts)
    t = api.Talc(api.default_params(k))
    t.load_packed(keys, counts)
    absent = rng.integers(0, 1 << (2 * (k - 1)), 3000, dtype=np.uint64)
    qr, ql = _all_queries(ref, absent, absent)
    _check_successors(t, ref, qr, ql, "K=%d" % k, ctx_capacity(len(keys)))
    if k == 31:
        assert (ref.keys >> np.uint64(60) == 3).all()


def _seal_paths(api, k, keys, counts, tmp_path):
    """the same table sealed every way the library seals one"""
    p = api.default_params(k)
    out = {}
    t = api.Talc(p)
    t.load_packed(keys, counts)
    out["load_packed"] = t
    dump = str(tmp_path / "d.txt")
    api.write_dump(dump, keys, counts, k)
    d = api.Talc(p)
    d.load_dump(dump)
    out["load_dump"] = d
    fa = tmp_path / "r.fa"  # one K-base record per occurrence: counting gives back the counts
    alpha = np.frombuffer(b"ACGT", np.uint8)
    with open(fa, "wb") as f:
        for x, c in zip(keys.tolist(), counts.tolist()):
            s = alpha[[(x >> (2 * (k - 1 - i))) & 3 for i in range(k)]].tobytes()
            f.write((b">r\n" + s + b"\n") * c)
    r = api.Talc(p)
    r.count_reads([str(fa)])
    out["count_reads"] = r
    cache = str(tmp_path / "t.cache")
    t.table_save(cache)
    cc = api.Talc(p)
    cc.table_load_cache(cache)
    out["table_load_cache"] = cc
    cp = api.Talc(p)
    api.table_copy(cp, t)
    out["table_copy"] = cp
    import torch
    info = t.table_info()
    buf = torch.empty(info["bytes"], dtype=torch.uint8, device="cuda:0")
    t.table_export_device(buf)
    im = api.Talc(p)
    im.table_import_device(buf, info["capacity"], info["entries"])
    out["table_import_device"] = im
    out["lane"] = t.create_lane()
    return out


@gpu
def test_every_seal_path_gives_the_same_answers(api, tmp_path):
    k, cap = 21, 1 << 11
    keys, counts, absent, wrap = adversarial_layout(k, cap, seed=3)
    ref = Ref(k, keys, counts)
    qr, ql = _all_queries(ref, absent[True], absent[False])
    paths = _seal_paths(api, k, keys, counts, tmp_path)
    for name, t in paths.items():
        _check_successors(t, ref, qr, ql, name, ctx_capacity(len(keys)))
        c, _, f = t.lookup(np.concatenate([keys, wrap ^ np.uint64(2)]))
        wc, _, hit = ref.get(np.concatenate([keys, wrap ^ np.uint64(2)]))
        assert np.array_equal(c, wc) and np.array_equal(f.astype(bool), hit), name
    paths["lane"].close()


def _slot_image(keys, counts, cap):
    """a k-mer table of cap slots built on the host by pair-aligned linear probing (table.cuh)"""
    img = np.zeros((cap, 2), dtype=np.uint64)
    img[:, 0] = np.uint64(M64)
    for x, c, h in zip(keys.tolist(), counts.tolist(), (hash_kmer(keys) & np.uint64(cap - 1) & ~np.uint64(1)).tolist()):
        i = h
        while img[i, 0] != np.uint64(M64):
            i = (i + 1) & (cap - 1)
        img[i, 0], img[i, 1] = x, c
    return img


@gpu
def test_import_at_half_load(api):
    """a table imported at exactly half load is sealed and answers like the dictionary; one entry more is refused"""
    import torch
    k, cap = 21, 1 << 12
    rng = np.random.default_rng(11)
    keys = np.unique(rng.integers(0, 1 << (2 * k), 3 * cap, dtype=np.uint64))[: cap // 2 + 1]
    keys = np.concatenate([keys[:-40], pick_kmers_home_sector(rng, k, cap, cap - 2, 40, keys)])[: cap // 2 + 1]
    assert len(np.unique(keys)) == cap // 2 + 1
    counts = rng.integers(2, 100, len(keys)).astype(np.int64)
    for n, ok in ((cap // 2, True), (cap // 2 + 1, False)):
        img = _slot_image(keys[:n], counts[:n], cap)
        buf = torch.from_numpy(img.view(np.int64).copy()).to("cuda:0")
        t = api.Talc(api.default_params(k))
        if not ok:
            with pytest.raises(api.TalcError, match="half full"):
                t.table_import_device(buf, cap, n)
            continue
        t.table_import_device(buf, cap, n)
        ref = Ref(k, keys[:n], counts[:n])
        probe = np.concatenate([keys, rng.integers(0, 1 << (2 * k), 4000, dtype=np.uint64)])
        c, _, f = t.lookup(probe)
        assert np.array_equal(c, ref.get(probe)[0]) and np.array_equal(f.astype(bool), ref.get(probe)[2])
        qr, ql = _all_queries(ref, keys[n:] >> np.uint64(2), keys[n:] & kmask(k - 1))
        _check_successors(t, ref, qr, ql, "half load", ctx_capacity(n))


@gpu
def test_successor_tables_at_scale(api):
    """about 4 M random entries at K = 31: every context of every key and 1 M absent contexts, against numpy"""
    k = 31
    rng = np.random.default_rng(31)
    keys = np.unique(rng.integers(0, 1 << (2 * k), 4_200_000, dtype=np.uint64))
    counts = rng.integers(2, 1 << 20, len(keys)).astype(np.int64)
    ref = Ref(k, keys, counts)
    t = api.Talc(api.default_params(k))
    t.load_packed(keys, counts)
    absent = rng.integers(0, 1 << (2 * (k - 1)), 1_000_000, dtype=np.uint64)
    qr, ql = _all_queries(ref, absent, absent)
    _check_successors(t, ref, qr, ql, "scale", ctx_capacity(len(keys)))
