"""The block-join overflow redo (csrc/join.cu k_join, gkd_api.cu run_pairs and its forms, intersect.cu
k_nearest_absorb), forced and checked against exact oracles.

Kernel 4's block join flags a task when the rows of one key range would fill more than 62.5 % of its shared-memory
table; the host then discards the chunk and redoes it with the merge kernel.  Two inputs reach that without any hook:

* coarse tables (recipe A): a large GKD_TABLE_TMAX leaves every set at its floor level (0 for DNA K <= 16 and for
  64-bit keys), so `range_run` hands a row's whole set to every range and ~2,000-key rows overflow any block;
* skewed imported sets (recipe B): keys whose mixed values h = mix(key) fall in one 2^16-wide band put a row's whole
  run into one key range; a block holding enough such rows overflows with the default switches.

Every forcing case first proves that the redo ran (`redo`: the number of kernel-4 launches and the kernel of the last
one), then compares the result with the exact oracle (numpy arithmetic on the imported keys, orc.IntSet on text)
and with the same call on a context pinned to the merge kernel, doubles by their bits.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import sparse

import genome.distance_b200 as gkd

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")
COARSE = str(1 << 24)  # GKD_TABLE_TMAX that leaves every set of these tests at its floor level

# ---- numpy port of the key mix (gkd_internal.cuh mix_key / unmix_key / make_mix) --------------------------------
MIX_C1, MIX_C2 = 0xFF51AFD7ED558CCD, 0xC4CEB9FE1A85EC53
MIX_I1, MIX_I2 = 0x4F74430C22A54005, 0x9CB4B2F8129337DB


def make_mix(bits):
    """(mask, fix, shift) of a key space of `bits` bits"""
    mask = (1 << 64) - 1 if bits >= 64 else (1 << bits) - 1
    shift = min(max((bits + 1) // 2, 1), 63)
    fix = int(_mix_rounds(np.array([mask], dtype=np.uint64), mask, shift)[0]) ^ mask
    return mask, fix, shift


def _mix_rounds(x, mask, shift):
    x = np.array(x, dtype=np.uint64)
    m, s = np.uint64(mask), np.uint64(shift)
    x ^= x >> s
    x = (x * np.uint64(MIX_C1)) & m
    x ^= x >> s
    x = (x * np.uint64(MIX_C2)) & m
    x ^= x >> s
    return x


def mix(keys, p):
    mask, fix, shift = p
    return _mix_rounds(keys, mask, shift) ^ np.uint64(fix)


def unmix(h, p):
    mask, fix, shift = p
    m, s = np.uint64(mask), np.uint64(shift)
    x = np.array(h, dtype=np.uint64) ^ np.uint64(fix)
    x ^= x >> s
    x = (x * np.uint64(MIX_I2)) & m
    x ^= x >> s
    x = (x * np.uint64(MIX_I1)) & m
    x ^= x >> s
    return x


def revcomp(keys, k):
    """reverse complement of 2-bit DNA keys of K bases (a=0 c=1 g=2 t=3)"""
    x = np.array(keys, dtype=np.uint64)
    out = np.zeros_like(x)
    two, three = np.uint64(2), np.uint64(3)
    for _ in range(k):
        out = (out << two) | (three - (x & three))
        x = x >> two
    return out


def canonical_only(keys, k):
    keys = np.asarray(keys, dtype=np.uint64)
    return keys[keys <= revcomp(keys, k)]


# ---- exact oracle of imported key sets (both-strand DNA) ---------------------------------------------------------
class KeySets:
    """|C| from the unique keys, P from key == revcomp(key) (even K), sizes 2|C| - P, I = 2|C_A n C_B| - P(C_A n C_B)
    as sparse products over the shared key pool, the double from orc.distance"""

    def __init__(self, orc, sets, k):
        self.orc = orc
        sets = [np.unique(np.asarray(s, dtype=np.uint64)) for s in sets]
        pool = np.unique(np.concatenate(sets))
        pal = revcomp(pool, k) == pool if k % 2 == 0 else np.zeros(pool.size, dtype=bool)
        cols = np.concatenate([np.searchsorted(pool, s) for s in sets])
        rows = np.repeat(np.arange(len(sets)), [s.size for s in sets])
        self.M = sparse.csr_matrix((np.ones(cols.size, dtype=np.int64), (rows, cols)), shape=(len(sets), pool.size))
        self.Mp = self.M[:, np.flatnonzero(pal)].tocsr()
        self.count = np.array([s.size for s in sets], dtype=np.int64)
        self.pal = np.asarray(self.Mp.sum(axis=1)).ravel().astype(np.int64)
        self.size = 2 * self.count - self.pal

    def inter(self, rows, cols):
        c = (self.M[rows] @ self.M[cols].T).toarray()
        p = (self.Mp[rows] @ self.Mp[cols].T).toarray()
        return (2 * c - p).astype(np.uint64)

    def block(self, rows, cols):
        """(I, dist) of every rows x cols pair"""
        rows, cols = np.asarray(rows), np.asarray(cols)
        I = self.inter(rows, cols)
        return I, _distances(self.orc, I, self.size[rows][:, None], self.size[cols][None, :])


def _distances(orc, I, sa, sb):
    I, sa, sb = np.broadcast_arrays(I, sa, sb)
    out = np.empty(I.shape)
    for x in np.ndindex(I.shape):
        out[x] = orc.distance(int(I[x]), int(sa[x]), int(sb[x]))
    return out


def _text_oracle(orc, seqs, k, alphabet):
    """(I, dist) n x n of orc.IntSet on text"""
    osets = [orc.IntSet(s, k, alphabet) for s in seqs]
    n = len(seqs)
    I, D = np.zeros((n, n), dtype=np.uint64), np.zeros((n, n))
    for i in range(n):
        for j in range(i, n):
            I[i, j] = I[j, i] = osets[i].similarity(osets[j])
            D[i, j] = D[j, i] = osets[i].distance(osets[j])
    return I, D


# ---- helpers ---------------------------------------------------------------------------------------------------
def redo(e, call):
    """(result, kernel-4 launches of the call, kernel of the last launch).  A single-chunk call that took the redo
    shows 2 launches and kernel 3 (32-bit lows) or 4 (64-bit keys); the join alone shows 1 launch and kernel 5."""
    before = e.metrics()["intersect_launches"]
    out = call()
    m = e.metrics()
    return out, m["intersect_launches"] - before, m["intersect_kernel"]


def _merge_kernel(k, alphabet=gkd.DNA):
    bits = 8 * k if alphabet == gkd.PROT else 2 * k
    return 3 if bits <= 42 else 4


def _redone(e, call, k, alphabet=gkd.DNA, launches=2):
    out, n, kern = redo(e, call)
    assert (n, kern) == (launches, _merge_kernel(k, alphabet)), "the block join did not overflow and redo"
    return out


def _check(got, want, what=None):
    for g, w in zip(got, want):
        g, w = np.asarray(g), np.asarray(w)
        assert g.shape == w.shape, what
        if g.dtype == np.float64:
            assert np.array_equal(g.view(np.uint64), w.view(np.uint64)), what  # bit-exact
        else:
            assert np.array_equal(g, w), what


def _thresholds(dist):
    """1.0 (every pair), an attained distance below 1 (inclusive boundary), and one below every distance (no hit)"""
    dist = np.asarray(dist).ravel()
    below = sorted(set(float(x) for x in dist if x < 1.0))
    out = [1.0, float(np.nextafter(float(np.min(dist)), -np.inf))]
    if below:
        out.append(below[len(below) // 2])
    return out


def _nearest_ref(gi, gd, q, r, k, D, exclude_self):
    """numpy: every row stably sorted by (dist, position), filtered by D (and self pairs), cut to k"""
    nq, nr = len(q), len(r)
    pos = np.full((nq, k), 0xFFFFFFFF, dtype=np.uint32)
    inter = np.zeros((nq, k), dtype=np.uint64)
    dist = np.full((nq, k), -1.0)
    found = np.zeros(nq, dtype=np.uint32)
    ra = np.asarray(r)
    for x in range(nq):
        idx = np.arange(nr)
        ok = gd[x] <= D
        if exclude_self:
            ok &= ra != q[x]
        idx = idx[ok]
        if idx.size > k:  # only distances up to the k-th smallest can make the cut (ties included)
            vals = gd[x][idx]
            idx = idx[vals <= np.partition(vals, k - 1)[k - 1]]
        idx = idx[np.lexsort((idx, gd[x][idx]))][:k]
        found[x] = idx.size
        pos[x, :idx.size] = idx
        inter[x, :idx.size] = gi[x][idx]
        dist[x, :idx.size] = gd[x][idx]
    return pos, inter, dist, found


def _hits_ref(pa, pb, gi, gd, D):
    keep = gd <= D
    return pa[keep], pb[keep], gi[keep], gd[keep]


def _engine(monkeypatch, algo, seqs=None, k=21, alphabet=gkd.DNA, keysets=None, coarse=False):
    """a context pinned to one kernel-4 form (switches are read when a context is created)"""
    monkeypatch.setenv("GKD_ISECT_ALGO", algo)
    if coarse:
        monkeypatch.setenv("GKD_TABLE_TMAX", COARSE)
    else:
        monkeypatch.delenv("GKD_TABLE_TMAX", raising=False)
    e = gkd.Engine(k=k, alphabet=alphabet)
    if seqs is not None:
        for s in seqs:
            e.add(s)
        e.build()
    if keysets is not None:
        offs = np.r_[0, np.cumsum([len(s) for s in keysets])]
        assert e.import_sets(np.concatenate(keysets).astype(np.uint64), offs) == 0
    return e


# ---- recipe A: text whose sets stay at the floor level ------------------------------------------------------------
def _text(seed, lens, protein=False, palindromes=False, families=3):
    """related families (members mutated at 0, 0.2, 3 and 15 %); with `palindromes`, shared x + revcomp(x) inserts give
    every set reverse-palindromic 16-mers"""
    rng = np.random.default_rng(seed)
    comp = bytes.maketrans(b"acgt", b"tgca")
    inserts = [rng.choice(np.frombuffer(b"acgt", dtype=np.uint8), 12).tobytes() for _ in range(6)]
    out = []
    for g, n in enumerate(lens):
        a = np.empty(n, dtype=np.uint8)
        mem = g // families
        gkd.synth(a, seed, g % families, mem, [0.0, 0.002, 0.03, 0.15][mem % 4] if mem else 0.0, protein=protein)
        s = a.tobytes()
        if palindromes and n:
            for x in (inserts[g % 6], inserts[(g * 5 + 1) % 6]):
                s += b"n" + x + x[::-1].translate(comp)
        out.append(s)
    return out


LENS_A = [2000] * 36 + [2600, 1400, 30, 0]
CASES_A = [(16, gkd.DNA), (25, gkd.DNA), (8, gkd.PROT)]


def _recipe_a(k, alphabet):
    prot = alphabet == gkd.PROT
    seqs = _text(7, LENS_A, protein=prot, palindromes=(k == 16))
    seqs[20] = seqs[3]  # ties
    seqs[33] = seqs[3]
    return seqs


def _upper(I, D):
    iu = np.triu_indices(I.shape[0], 1)
    return I[iu], D[iu]


def _row_start(n, i):
    return i * (2 * n - i - 1) // 2


@pytest.mark.parametrize("k,alphabet", CASES_A)
def test_dense_coarse_tables(orc, monkeypatch, k, alphabet):
    seqs = _recipe_a(k, alphabet)
    n = len(seqs)
    I, D = _text_oracle(orc, seqs, k, alphabet)
    ui, ud = _upper(I, D)
    total = n * (n - 1) // 2
    with _engine(monkeypatch, "merge", seqs, k, alphabet, coarse=True) as m, \
            _engine(monkeypatch, "join", seqs, k, alphabet, coarse=True) as e:
        got = _redone(e, lambda: e.all_vs_all(), k, alphabet)
        _check(got, (ui, ud))
        _check(got, m.all_vs_all())
        # ranges that start and end inside rows
        for first, count in ((37, 511), (total - 400, 400), (_row_start(n, 4) + 3, _row_start(n, 17) - _row_start(n, 4))):
            got = _redone(e, lambda: e.all_vs_all_range(n, first, count), k, alphabet)
            _check(got, (ui[first:first + count], ud[first:first + count]), (first, count))
            _check(got, m.all_vs_all_range(n, first, count), (first, count))
        # many query rows; fewer than 32 (the join puts the reference side on the table); duplicate ids
        for q, r in ((list(range(0, 35)), list(range(2, n))), ([5, 30, 7], list(range(n))),
                     ([3, 3, 0, 20, 3, 33] * 6, [9, 3, 3, 39, 20])):
            got = _redone(e, lambda: e.query_vs_ref(q, r), k, alphabet)
            _check(got, (I[np.ix_(q, r)], D[np.ix_(q, r)]), (q, r))
            _check(got, m.query_vs_ref(q, r), (q, r))


# ---- recipe B: imported keys in one narrow band of h ------------------------------------------------------------
def _band(k, start, width=1 << 16):
    """the canonical keys whose mixed values are start .. start + width - 1"""
    p = make_mix(2 * k)
    keys = unmix(np.arange(start, start + width, dtype=np.uint64), p)
    keys = canonical_only(keys, k)
    return keys[keys != np.uint64(p[0])]


def _uniform(rng, k, n):
    keys = rng.integers(0, 1 << (2 * k), size=2 * n + 64, dtype=np.uint64)
    keys = np.unique(canonical_only(keys, k))
    keys = keys[keys != np.uint64((1 << (2 * k)) - 1)]
    return rng.permutation(keys)[:n]


def _families(rng, pool, n_sets, base, n_fam, extra_pool=None, extra=0):
    """set i belongs to family i % n_fam (a base of `base` pool keys) and keeps 85 to 95 % of it (so the rows of a
    context fall in one size class of the join plan), plus `extra` keys of extra_pool"""
    bases = [rng.choice(pool, base, replace=False) for _ in range(n_fam)]
    out = []
    for i in range(n_sets):
        b = bases[i % n_fam]
        s = b[rng.random(b.size) < rng.uniform(0.85, 0.95)]
        if extra:
            s = np.concatenate([s, rng.choice(extra_pool, extra)])
        out.append(np.unique(s))
    return out


BAND_M = {21: 1234, 25: 0x2B5C3}  # band start / 2^31: a range boundary at every usable level


def _mixed(k, seed=11, n=140, crafted=range(64, 84)):
    """ordinary sets (uniform h, plus 20 band keys each) with crafted rows (every key in the band) inside the second
    64-row block; copies give ties"""
    rng = np.random.default_rng(seed)
    band = _band(k, BAND_M[k] << 31)
    uni = _uniform(rng, k, 60_000)
    ordinary = _families(rng, uni, n, 780, 8, band, 20)
    craft = _families(rng, band, len(crafted), 800, 4)
    sets = list(ordinary)
    for i, c in zip(crafted, craft):
        sets[i] = c
    for i in (66, 90, 131):
        sets[i] = sets[64]
    for i in (5, 100):
        sets[i] = sets[3]
    return sets


@pytest.mark.parametrize("k", [21, 25])
def test_dense_skewed_imports(orc, monkeypatch, k):
    sets = _mixed(k)
    n = len(sets)
    ks = KeySets(orc, sets, k)
    I, D = ks.block(np.arange(n), np.arange(n))
    ui, ud = _upper(I, D)
    with _engine(monkeypatch, "merge", k=k, keysets=sets) as m, _engine(monkeypatch, "join", k=k, keysets=sets) as e:
        for i in (0, 64, 130):
            assert e.set_size(i) == (int(ks.size[i]), int(ks.count[i]), int(ks.pal[i]))
        got = _redone(e, lambda: e.all_vs_all(), k)
        _check(got, (ui, ud))
        _check(got, m.all_vs_all())
        first = _row_start(n, 60) + 5
        count = _row_start(n, 82) - 3 - first
        got = _redone(e, lambda: e.all_vs_all_range(n, first, count), k)
        _check(got, (ui[first:first + count], ud[first:first + count]))
        for q, r in ((list(range(60, 101)), list(range(n))), ([70, 5, 130], list(range(n))),
                     ([64, 65, 64, 3] * 10, [64, 3, 3, 139, 70])):
            got = _redone(e, lambda: e.query_vs_ref(q, r), k)
            _check(got, (I[np.ix_(q, r)], D[np.ix_(q, r)]), (q, r))
            _check(got, m.query_vs_ref(q, r), (q, r))


def test_within_skewed_imports(orc, monkeypatch):
    k = 21
    sets = _mixed(k)
    n = len(sets)
    I, D = KeySets(orc, sets, k).block(np.arange(n), np.arange(n))
    ui, ud = _upper(I, D)
    iu_a, iu_b = (x.astype(np.uint32) for x in np.triu_indices(n, 1))
    total = n * (n - 1) // 2
    with _engine(monkeypatch, "merge", k=k, keysets=sets) as m, _engine(monkeypatch, "join", k=k, keysets=sets) as e:
        first = _row_start(n, 60) + 5
        count = _row_start(n, 82) - 3 - first
        for D_ in _thresholds(ud):
            got = _redone(e, lambda: e.all_vs_all_within(D_), k)
            _check(got, _hits_ref(iu_a, iu_b, ui, ud, D_), D_)
            _check(got, m.all_vs_all_within(D_), D_)
            s = slice(first, first + count)
            got = _redone(e, lambda: e.all_vs_all_range_within(n, first, count, D_), k)
            _check(got, _hits_ref(iu_a[s], iu_b[s], ui[s], ud[s], D_), D_)
            _check(got, m.all_vs_all_range_within(n, first, count, D_), D_)
            for q, r in ((list(range(60, 101)), list(range(n))), ([70, 5, 130], list(range(n)))):
                pa = np.repeat(np.arange(len(q), dtype=np.uint32), len(r))
                pb = np.tile(np.arange(len(r), dtype=np.uint32), len(q))
                got = _redone(e, lambda: e.query_vs_ref_within(q, r, D_), k)
                _check(got, _hits_ref(pa, pb, I[np.ix_(q, r)].ravel(), D[np.ix_(q, r)].ravel(), D_), (q, D_))
                _check(got, m.query_vs_ref_within(q, r, D_), (q, D_))
        # through the C ABI with room for fewer hits than there are: the total stays exact, the prefix is the first
        # hits, and no hit is written twice
        D_ = 1.0
        L = e._L
        for cap in (0, 1000, total - 1):
            ha, hb = np.empty(cap, dtype=np.uint32), np.empty(cap, dtype=np.uint32)
            hi, hd = np.empty(cap, dtype=np.uint64), np.empty(cap, dtype=np.float64)
            h = gkd._lib.GkdHits(ha.ctypes.data, hb.ctypes.data, hi.ctypes.data, hd.ctypes.data, cap, 0)
            _redone(e, lambda: e._ck(L.gkd_all_vs_all_range_within(e._h, n, 0, total, D_, C.byref(h))), k)
            assert h.n == total, cap
            _check((ha, hb, hi, hd), (iu_a[:cap], iu_b[:cap], ui[:cap], ud[:cap]), cap)
            assert np.unique(ha.astype(np.uint64) << np.uint64(32) | hb).size == cap


def test_nearest_skewed_imports(orc, monkeypatch):
    k = 21
    sets = _mixed(k)
    n = len(sets)
    ids = list(range(n))
    I, D = KeySets(orc, sets, k).block(np.arange(n), np.arange(n))
    with _engine(monkeypatch, "merge", k=k, keysets=sets) as m, _engine(monkeypatch, "join", k=k, keysets=sets) as e:
        for kk in (1, 5, 256):
            for D_ in _thresholds(_upper(I, D)[1]):
                got = _redone(e, lambda: e.all_vs_all_nearest(kk, D_), k)
                _check(got, _nearest_ref(I, D, ids, ids, kk, D_, True), (kk, D_))
                _check(got, m.all_vs_all_nearest(kk, D_), (kk, D_))
                _check(got, _redone(e, lambda: e.query_vs_ref_nearest(ids, ids, kk, D_, exclude_self=True), k),
                       (kk, D_))
        assert list(e.all_vs_all_nearest(3, 1.0)[0][66]) == [64, 90, 131]  # ties by the smaller id
        for q, r, excl in ((list(range(60, 101)), list(range(3, n)), False), ([70, 5, 130], ids, True),
                           ([64, 65, 64, 3] * 10, [64, 3, 3, 139, 70], False)):
            for kk, D_ in ((1, 1.0), (5, 0.9), (256, 1.0)):
                want_q = _nearest_ref(I[np.ix_(q, r)], D[np.ix_(q, r)], q, r, kk, D_, excl)
                want_r = _nearest_ref(I[np.ix_(r, q)], D[np.ix_(r, q)], r, q, kk, D_, excl)
                got = _redone(e, lambda: e.query_vs_ref_nearest(q, r, kk, D_, exclude_self=excl), k)
                _check(got, want_q, (q, kk, D_))
                qs, rs = _redone(e, lambda: e.query_vs_ref_nearest_ex(q, r, kk, D_, exclude_self=excl), k)
                _check(qs, want_q, (q, kk, D_))
                _check(rs, want_r, (q, kk, D_))
                mq, mr = m.query_vs_ref_nearest_ex(q, r, kk, D_, exclude_self=excl)
                _check(qs, mq, (q, kk, D_))
                _check(rs, mr, (q, kk, D_))


def test_nearest_ex_redone_in_every_launch(orc, monkeypatch):
    """2^19 references: a launch holds 128 query rows, so 260 rows take three, and the reference side's lists are built
    across them.  Even ids are crafted; the query rows alternate, so every 64-row block of the first two launches
    overflows, and so does every block of the third, whose 4 rows put the references on the table."""
    k = 21
    rng = np.random.default_rng(3)
    band = _band(k, BAND_M[k] << 31)
    uni = _uniform(rng, k, 40_000)
    craft = _families(rng, band, 24, 800, 6)
    ordinary = _families(rng, uni, 24, 800, 6, band, 10)
    sets = [craft[i // 2] if i % 2 == 0 else ordinary[i // 2] for i in range(48)]
    n = len(sets)
    r = np.tile(np.arange(n, dtype=np.uint32), (1 << 19) // n + 1)[: 1 << 19]
    q = (rng.integers(0, n // 2, 260) * 2 + np.arange(260) % 2).astype(np.uint32)
    I, D = KeySets(orc, sets, k).block(np.arange(n), np.arange(n))
    with _engine(monkeypatch, "merge", k=k, keysets=sets) as m, _engine(monkeypatch, "join", k=k, keysets=sets) as e:
        for kk, D_, excl in ((1, 1.0, False), (16, 0.6, True)):
            qs, rs = _redone(e, lambda: e.query_vs_ref_nearest_ex(q, r, kk, D_, exclude_self=excl), k, launches=6)
            mq, mr = m.query_vs_ref_nearest_ex(q, r, kk, D_, exclude_self=excl)
            _check(qs, mq, kk)
            _check(rs, mr, kk)
            # the exact oracle on sampled rows of both sides
            for x in (0, 127, 128, 200, 259):
                _check([g[x:x + 1] for g in qs],
                       _nearest_ref(I[q[x:x + 1]][:, r], D[q[x:x + 1]][:, r], q[x:x + 1], r, kk, D_, excl), (kk, x))
            for y in (0, 1, 47, 1000, (1 << 19) - 1):
                _check([g[y:y + 1] for g in rs],
                       _nearest_ref(I[r[y:y + 1]][:, q], D[r[y:y + 1]][:, q], r[y:y + 1], q, kk, D_, excl), (kk, y))


def test_overflow_only_in_the_second_chunk(orc, monkeypatch):
    """~12,000 small sets: 7.2e7 pairs, two 64 Mi-pair chunks; the boundary lies inside row 8,873.  Rows before it are
    ordinary, the 3,000 rows from 9,000 on are crafted, so only the second chunk overflows: the lists the absorb epilogue
    kept from the first chunk must survive the redo of the second, and the discarded attempt must add nothing."""
    k = 21
    n, first_crafted = 12_000, 9_000
    rng = np.random.default_rng(29)
    band = _band(k, BAND_M[k] << 31)
    uni = _uniform(rng, k, 200_000)
    sets = _families(rng, uni, first_crafted, 330, 200, band, 20) + \
        _families(rng, band, n - first_crafted, 330, 100)
    dup = [40, 3_000, 8_800, 8_871, 8_873, 8_900, 10_000, 11_999]
    for i in dup[1:]:
        sets[i] = sets[dup[0]]
    sets[11_998] = sets[9_001]
    total = n * (n - 1) // 2
    assert _row_start(n, 8873) < 64 << 20 < _row_start(n, 8874)
    ks = KeySets(orc, sets, k)
    sample = np.array([0, 40, 3_000, 8_800, 8_872, 8_873, 8_874, 8_999, 9_000, 9_001, 10_000, 11_998, 11_999])
    sI, sD = ks.block(sample, np.arange(n))
    kk, D_ = 8, 0.5
    with _engine(monkeypatch, "join", k=k, keysets=sets) as e:
        near = _redone(e, lambda: e.all_vs_all_nearest(kk, 1.0), k, launches=3)
        assert e.metrics()["pairs"] == total
        hits = _redone(e, lambda: e.all_vs_all_within(D_), k, launches=3)
        _check([g[sample] for g in near], _nearest_ref(sI, sD, sample, np.arange(n), kk, 1.0, True))
        _check([g[sample] for g in near], e.query_vs_ref_nearest(sample, np.arange(n), kk, 1.0, exclude_self=True))
        assert list(near[0][8_873][:4]) == [40, 3_000, 8_800, 8_871]
        ra, rb, ri, rd = e.query_vs_ref_within(sample, np.arange(n), D_)
    a, b = hits[0], hits[1]
    assert a.size and np.all((a[1:] > a[:-1]) | ((a[1:] == a[:-1]) & (b[1:] > b[:-1])))  # enumeration order, no repeat
    assert (a >= 8_873).any() and (a < 8_873).any()
    for x_at, x in enumerate(sample):
        mine = (a == x) | (b == x)
        other = np.where(a[mine] == x, b[mine], a[mine])
        want = np.flatnonzero((sD[x_at] <= D_) & (np.arange(n) != x))
        assert np.array_equal(other, want), x
        assert np.array_equal(hits[2][mine], sI[x_at][want]), x
        assert np.array_equal(hits[3][mine].view(np.uint64), sD[x_at][want].view(np.uint64)), x
        row = (ra == x_at) & (rb != x)
        assert np.array_equal(rb[row], want), x
    with _engine(monkeypatch, "merge", k=k, keysets=sets) as m:
        _check(near, m.all_vs_all_nearest(kk, 1.0))
        _check(hits, m.all_vs_all_within(D_))


def test_group_equals_redone_single_context(monkeypatch):
    import torch

    k = 25
    seqs = _recipe_a(k, gkd.DNA)
    n = len(seqs)
    with _engine(monkeypatch, "join", seqs, k, coarse=True) as e:
        want = {"dense": _redone(e, lambda: e.all_vs_all(), k)}
        dist = want["dense"][1]
        for D_ in _thresholds(dist):
            want[("within", D_)] = _redone(e, lambda: e.all_vs_all_within(D_), k)
        for kk in (1, 5, 256):
            want[("nearest", kk)] = _redone(e, lambda: e.all_vs_all_nearest(kk, 1.0), k)
    ndev = torch.cuda.device_count()
    for members in (2, 3, 4):
        devices = [x % ndev for x in range(members)]
        with gkd.Group(devices, k=k, workspace_bytes=4 << 20, panel=2) as g:
            per = (n + members - 1) // members
            for i, s in enumerate(seqs):
                assert g.add(min(i // per, members - 1), s) == i
            g.build()
            for key, w in want.items():
                if key == "dense":
                    got = g.all_vs_all()
                elif key[0] == "within":
                    got = g.all_vs_all_within(key[1])
                else:
                    got = g.all_vs_all_nearest(key[1], 1.0)
                for x, y in zip(got, w):
                    assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)), (members, key)


def test_cli_reports_do_not_change_when_the_join_overflows(tmp_path):
    seqs = _recipe_a(25, gkd.DNA)[:38]  # records of 1.4 kbp and more
    fa = tmp_path / "in.fa"
    with open(fa, "w") as f:
        for i, s in enumerate(seqs):
            f.write(">r%04d rec %d\n%s\n" % (i, i, s.decode()))
    plain = {k: v for k, v in os.environ.items() if k not in ("GKD_ISECT_ALGO", "GKD_TABLE_TMAX")}
    forced = dict(plain, GKD_ISECT_ALGO="join", GKD_TABLE_TMAX=COARSE)
    for opts in (["--nearest", "5"], ["--maxDist", "0.5"]):
        outs = []
        for env in (plain, forced):
            p = subprocess.run([GKD, "fastaDist", "-i", str(fa), "-K", "25"] + opts, capture_output=True, env=env,
                               timeout=600)
            assert p.returncode == 0, p.stderr
            outs.append(p.stdout)
        assert outs[0].count(b"\n") > 1 and outs[0] == outs[1], opts


def test_range_boundaries_and_import_contract(orc, monkeypatch):
    """h at the first and last value of key ranges (multiples of 2^31 are range boundaries at every usable level for
    K = 21; the first value's low word differs from the table's EMPTY pattern only in bit 31), h = 0, and sets that
    straddle two adjacent ranges; exact under both kernel-4 forms"""
    k = 21
    p = make_mix(2 * k)
    ms = np.arange(1, 1 << 11, dtype=np.uint64)
    firsts = unmix(ms << np.uint64(31), p)
    lasts = unmix((ms << np.uint64(31)) - np.uint64(1), p)
    edge = np.concatenate([firsts[firsts <= revcomp(firsts, k)][:60], lasts[lasts <= revcomp(lasts, k)][:60],
                           unmix(np.array([0], dtype=np.uint64), p)])
    assert np.array_equal(np.sort(mix(unmix(np.arange(1000, dtype=np.uint64), p), p)), np.arange(1000, dtype=np.uint64))
    straddle = np.concatenate([_band(k, (m << 31) - 400, 800) for m in (5, 6, 700)])
    rng = np.random.default_rng(17)
    uni = _uniform(rng, k, 5_000)
    sets = []
    for i in range(40):
        s = [rng.choice(edge, 50, replace=False), rng.choice(straddle, 150, replace=False), rng.choice(uni, 30)]
        sets.append(np.unique(np.concatenate(s)))
    sets[7] = np.unique(np.concatenate([edge, straddle]))
    n = len(sets)
    ks = KeySets(orc, sets, k)
    I, D = ks.block(np.arange(n), np.arange(n))
    ui, ud = _upper(I, D)
    for algo, kernel in (("join", 5), ("merge", 3)):
        with _engine(monkeypatch, algo, k=k, keysets=sets) as e:
            got, launches, kern = redo(e, lambda: e.all_vs_all())
            assert (launches, kern) == (1, kernel), algo
            _check(got, (ui, ud), algo)
            got, launches, kern = redo(e, lambda: e.query_vs_ref([7, 0, 7], list(range(n))))
            assert (launches, kern) == (1, kernel), algo
            _check(got, (I[[7, 0, 7]], D[[7, 0, 7]]), algo)
            # the import contract: values outside the key space and the all-ones key are dropped
            junk = np.array([1 << (2 * k), (1 << (2 * k)) - 1, 1 << 63, (1 << 64) - 1], dtype=np.uint64)
            x = e.import_set(np.concatenate([sets[7], junk, sets[7][:9]]))
            assert e.set_size(x) == (2 * sets[7].size, sets[7].size, 0)
            assert np.array_equal(e.export_set(x), sets[7])
            assert e.import_set(junk) == x + 1 and e.set_size(x + 1) == (0, 0, 0)
