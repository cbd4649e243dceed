"""GKD_STRAND_CANONICAL: plain Jaccard over canonical k-mers, |S| = |C| and I = |C_A n C_B|, on every call.

The mode is read at separate sites: set sizes and the host completion (both_size), the `both` flag every kernel-5 form
gets from run_pairs (pair_result in k_epilogue, k_select_within, k_select_nearest, k_nearest_absorb, k_cluster_link and
the linkage compaction), the greedy pass, and the sketch filter (one strand hashed instead of two).  For odd K the two
modes give bit-identical distances (I, |A| and |B| all double), and for even K they differ only through
reverse-palindromic k-mers, which random genomes hardly have at the usual K.  So the selection tests here run at
K = 4, 6 and 8 on records built from palindromic 6-mer words, with thresholds chosen strictly between the two modes'
distances of chosen pairs, and assert that a both-strand context gives a different answer at the same thresholds: a
path that ignored the mode fails.  The dense calls discriminate at every K through I (c against 2c - P_I).

Oracles: orc.IntSet (canonical count, palindromes, IntSet.intersect's (c, P_I)) and orc.distance for the dense values;
the ranked-row, component, rectangle and spanning-forest oracles of the selection test files applied to the canonical
dense matrix; py_hash_set over orc.py_canonical_set for the sketches.  tests/test_strand_canonical_cpu.py checks on the
CPU that the recipes below keep separating the modes.
"""
import itertools
import os
import sys

import numpy as np
import pytest

import genome.distance_b200 as gkd

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_gpu_clusters as tc  # noqa: E402  (component and rectangle oracles)
import test_gpu_join_redo as jr  # noqa: E402  (ranked rows, hits, the overflow recipes)
import test_gpu_linkage as tl  # noqa: E402  (spanning-forest oracles)

pytestmark = pytest.mark.gpu

CAN, BOTH = gkd.STRAND_CANONICAL, gkd.STRAND_BOTH
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kat_survey_8c.json")

# ---- inputs (numpy only, so the CPU test can rebuild them) ---------------------------------------------------------
_ACGT = np.frombuffer(b"acgt", dtype=np.uint8)
_COMP = bytes.maketrans(b"acgt", b"tgca")
WORDS = [bytes(x) + bytes(x)[::-1].translate(_COMP) for x in itertools.product(b"acgt", repeat=3)]  # 64 palindromes


def _random(rng, n):
    return rng.choice(_ACGT, n).tobytes()


def _mutate(rng, s, rate):
    a = np.frombuffer(s, dtype=np.uint8).copy()
    hit = rng.random(a.size) < rate
    a[hit] = rng.choice(_ACGT, int(hit.sum()))
    return a.tobytes()


def _spliced(rng, s, every=40):
    """a palindromic word after every `every` bases"""
    return b"".join(s[i:i + every] + WORDS[int(rng.integers(len(WORDS)))] for i in range(0, len(s), every))


def pal_records(seed=5):
    """records built from palindromic 6-mer words (three families with their own 16-word vocabularies; members redraw
    0, 5, 15 and 40 % of their 250 words), a random genome with words spliced in and two mutants of it, two plain random
    genomes and an empty record"""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(3):
        vocab = rng.choice(len(WORDS), 16, replace=False)
        base = rng.choice(vocab, 250)
        for rate in (0.0, 0.05, 0.15, 0.4):
            w = base.copy()
            hit = rng.random(w.size) < rate
            w[hit] = rng.choice(vocab, int(hit.sum()))
            out.append(b"".join(WORDS[i] for i in w))
    g = _spliced(rng, _random(rng, 3000))
    out += [g, _mutate(rng, g, 0.01), _mutate(rng, g, 0.06), _random(rng, 3000), _random(rng, 800), b""]
    return out


def dense_inputs(seed=9):
    """genomes (lists of contigs) for the set and dense checks: random, upper case, mixed case with N runs and IUPAC
    letters, contigs that are empty or shorter than K, every palindromic word, word records, an empty genome, a copy"""
    rng = np.random.default_rng(seed)
    g = _random(rng, 5000)
    mixed = np.frombuffer(_mutate(rng, g, 0.08), dtype=np.uint8).copy()
    for _ in range(12):
        p, run = int(rng.integers(0, mixed.size - 30)), int(rng.integers(1, 25))
        mixed[p:p + run] = rng.choice(np.frombuffer(b"nNRy-", dtype=np.uint8))
    mixed[(np.arange(mixed.size) % 3 == 0) & (mixed >= ord("a")) & (mixed <= ord("z"))] -= 32
    mixed = mixed.tobytes()
    recs = pal_records(seed)
    return [[g], [_mutate(rng, g, 0.02).upper()], [mixed],
            [_random(rng, 700), b"", _random(rng, 31), _random(rng, 19), _random(rng, 3), _random(rng, 33)],
            [b"".join(WORDS)], [recs[0]], [recs[2], recs[5]], [recs[12]], [b""], [g]]


def to_rna(genome):
    return [c.replace(b"t", b"u").replace(b"T", b"U") for c in genome]


# ---- the oracle of both modes ------------------------------------------------------------------------------------
class Modes:
    """full n x n (I, D) of both modes from orc.IntSet: canonical I = c over sizes |C|; both-strand I = 2c - P_I over
    sizes 2|C| - P (protein: c over |C| in both)"""

    def __init__(self, orc, seqs, k, alphabet=gkd.DNA):
        self.sets = [orc.IntSet(s, k, alphabet) for s in seqs]
        n = len(seqs)
        self.count = np.array([o.count for o in self.sets], dtype=np.int64)
        self.pal = np.array([o.palindromes for o in self.sets], dtype=np.int64)
        self.IC, self.IB, self.PI = (np.zeros((n, n), dtype=np.uint64) for _ in range(3))
        self.DC, self.DB = np.zeros((n, n)), np.zeros((n, n))
        for i in range(n):
            for j in range(i, n):
                c, p = self.sets[i].intersect(self.sets[j])
                ib = c if alphabet == gkd.PROT else 2 * c - p
                self.IC[i, j] = self.IC[j, i] = c
                self.PI[i, j] = self.PI[j, i] = p
                self.IB[i, j] = self.IB[j, i] = ib
                self.DC[i, j] = self.DC[j, i] = orc.distance(c, int(self.count[i]), int(self.count[j]))
                self.DB[i, j] = self.DB[j, i] = orc.distance(ib, len(self.sets[i]), len(self.sets[j]))
        iu = np.triu_indices(n, 1)
        self.n, self.iu = n, iu
        self.ic, self.dc, self.ib, self.db = self.IC[iu], self.DC[iu], self.IB[iu], self.DB[iu]


def between(dc, db):
    """thresholds strictly between the two modes' distances of three pairs whose distances differ: the midpoints for
    the smallest, a middle and the largest canonical distance among those pairs"""
    t = np.flatnonzero(dc != db)
    t = t[np.argsort(dc[t], kind="stable")]
    return [float((dc[x] + db[x]) / 2) for x in t[[0, t.size // 2, -1]]]


def _spread(xs, pick):
    return xs[:: max(1, len(xs) // pick)][:pick]


def splitting(n, dc, db, pick=3):
    """midpoints of differing pairs at which the two modes' single-linkage clusters differ"""
    cands = sorted({float((dc[x] + db[x]) / 2) for x in np.flatnonzero(dc != db)})
    return _spread([t for t in cands if not np.array_equal(tc._oracle(n, dc, t)[0], tc._oracle(n, db, t)[0])], pick)


def greedy(D, order, t):
    """the greedy representative pass over a full distance matrix: 1 where order[i] became a representative"""
    reps, out = [], []
    for g in order:
        found = any(D[r, g] <= t for r in reps)
        out.append(0 if found else 1)
        if not found:
            reps.append(g)
    return out


def greedy_splitting(DC, DB, order, pick=3):
    """midpoints of differing pairs at which the two modes' greedy passes pick different representatives"""
    iu = np.triu_indices(DC.shape[0], 1)
    dc, db = DC[iu], DB[iu]
    cands = sorted({float((dc[x] + db[x]) / 2) for x in np.flatnonzero(dc != db)})
    return _spread([t for t in cands if greedy(DC, order, t) != greedy(DB, order, t)], pick)


# ---- helpers -------------------------------------------------------------------------------------------------------
def _engine(monkeypatch, seqs, k, mode=CAN, alphabet=gkd.DNA, algo=None, coarse=False, **kw):
    """a context of one strand mode; `algo` pins the kernel-4 form (switches are read when a context is created)"""
    if algo:
        monkeypatch.setenv("GKD_ISECT_ALGO", algo)
    else:
        monkeypatch.delenv("GKD_ISECT_ALGO", raising=False)
    if coarse:
        monkeypatch.setenv("GKD_TABLE_TMAX", jr.COARSE)
    else:
        monkeypatch.delenv("GKD_TABLE_TMAX", raising=False)
    e = gkd.Engine(k=k, alphabet=alphabet, strand_mode=mode, **kw)
    for s in seqs:
        e.add(s)
    e.build()
    return e


def _bits(x):
    x = np.atleast_1d(np.asarray(x))
    return x.shape, x.dtype, x.view(np.uint8)


def _same(x, y):
    """bit-equal result tuples"""
    return all(_bits(a)[:2] == _bits(b)[:2] and np.array_equal(_bits(a)[2], _bits(b)[2]) for a, b in zip(x, y))


def _doubled(can, both, inter_at):
    """the both-strand result of an odd-K call: every array bit-equal except the intersections, which are doubled"""
    assert len(can) == len(both)
    for i, (c, b) in enumerate(zip(can, both)):
        if i == inter_at:
            assert np.asarray(c).dtype == np.asarray(b).dtype and np.array_equal(b, 2 * np.asarray(c)), i
        else:
            assert _same([c], [b]), i


# ---- 1. known answers ----------------------------------------------------------------------------------------------
def _kats():
    import json

    with open(GOLD) as f:
        return [p for p in json.load(f)["pairs"] if "canonical" in p]


@pytest.mark.parametrize("kat", _kats(), ids=lambda p: p["name"])
def test_known_answers(orc, kat):
    ca, cb, I = kat["canonical"]
    with gkd.Engine(k=kat["k"], strand_mode=CAN) as e:
        a, b = e.add(kat["a"]), e.add(kat["b"])
        e.build()
        pa, pb = (orc.IntSet(kat[x], kat["k"]).palindromes for x in "ab")
        if "palindromes" in kat:
            assert [pa, pb] == kat["palindromes"][:2]
        assert e.set_size(a) == (ca, ca, pa) and e.set_size(b) == (cb, cb, pb)
        assert e.pair(a, b) == (I, ca + cb - I, orc.distance(I, ca, cb))
        assert e.pair(b, a) == (I, ca + cb - I, orc.distance(I, ca, cb))


# ---- 2. sets and dense calls against the oracle (3. for the dense calls: how the modes relate) -------------------
DENSE_CASES = [(k, gkd.DNA) for k in (2, 4, 5, 6, 8, 11, 12, 16, 20, 21, 22, 32)] + [(8, gkd.RNA)]
DIFFERING_K = (4, 6, 8, 12)  # dense_inputs() has distances that differ between the modes (at K = 2 every set is full)


@pytest.mark.parametrize("algo", ["merge", "join"])
@pytest.mark.parametrize("k,alphabet", DENSE_CASES, ids=lambda x: str(x))
def test_sets_and_dense_calls(orc, monkeypatch, algo, k, alphabet):
    genomes = dense_inputs()
    if alphabet == gkd.RNA:
        genomes = [to_rna(g) if i % 2 else g for i, g in enumerate(genomes)]
    m = Modes(orc, genomes, k, alphabet)
    n = m.n
    with _engine(monkeypatch, genomes, k, CAN, alphabet, algo) as e, \
            _engine(monkeypatch, genomes, k, BOTH, alphabet, algo) as f:
        for i in range(n):
            assert e.set_size(i) == (m.count[i], m.count[i], m.pal[i]), i
            keys = e.export_set(i)
            assert np.array_equal(keys, m.sets[i].keys()) and np.array_equal(keys, f.export_set(i)), i
        got = e.all_vs_all()
        if algo == "join":
            assert e.metrics()["intersect_kernel"] == 5
        jr._check(got, (m.ic, m.dc))
        total = n * (n - 1) // 2
        for first, count in ((0, total), (3, 17), (total - 8, 8), (jr._row_start(n, 2) + 1, 11)):
            jr._check(e.all_vs_all_range(n, first, count), (m.ic[first:first + count], m.dc[first:first + count]))
        for q, r in ((list(range(n)), list(range(n))), ([4, 4, 0, 9], [9, 1, 4, 4, 7]), ([6], list(range(n)))):
            jr._check(e.query_vs_ref(q, r), (m.IC[np.ix_(q, r)], m.DC[np.ix_(q, r)]), (q, r))
        a = np.array([0, 9, 4, 6, 6, 2, 8, 3, 1], dtype=np.uint32)
        b = np.array([9, 0, 4, 7, 5, 3, 8, 2, 6], dtype=np.uint32)
        jr._check(e.pairs(a, b), (m.IC[a, b], m.DC[a, b]))
        inter, dist, ca, cb = e.pairs_ex(a, b)
        jr._check((inter, dist), (m.IC[a, b], m.DC[a, b]))
        cnt = m.count.astype(np.float64)
        want_a = np.where(cnt[a] > 0, m.IC[a, b] / np.maximum(cnt[a], 1), 0.0)
        want_b = np.where(cnt[b] > 0, m.IC[a, b] / np.maximum(cnt[b], 1), 0.0)
        jr._check((ca, cb), (want_a, want_b))
        # the both-strand context on the same input: I = 2c - P_I, identical doubles for odd K
        fi, fd = f.all_vs_all()
        jr._check((fi, fd), (m.ib, m.db))
        assert np.array_equal(fi, 2 * m.ic - m.PI[m.iu])
        if k % 2:
            assert np.array_equal(fd.view(np.uint64), got[1].view(np.uint64))
            assert not m.PI.any()
        elif k in DIFFERING_K:
            assert (fd != got[1]).any()


# ---- 3. odd K: every output of the two modes agrees --------------------------------------------------------------
@pytest.mark.parametrize("k", [5, 21])
def test_odd_k_outputs_agree_across_modes(orc, monkeypatch, k):
    seqs = pal_records(3)
    n = len(seqs)
    ids = list(range(n))
    q, r = [0, 5, 5, 13, 16], [1, 14, 5, 12, 0, 2]
    with _engine(monkeypatch, seqs, k, CAN) as e, _engine(monkeypatch, seqs, k, BOTH) as f:
        ci, cd = e.all_vs_all()
        _doubled((ci, cd), f.all_vs_all(), 0)
        below = sorted(set(cd[cd < 1.0].tolist()))
        ts = [below[0], below[len(below) // 2], below[-1], 1.0]
        for t in ts:
            _doubled(e.all_vs_all_within(t), f.all_vs_all_within(t), 2)
            _doubled(e.query_vs_ref_within(q, r, t), f.query_vs_ref_within(q, r, t), 2)
            for kk in (1, 4):
                _doubled(e.all_vs_all_nearest(kk, t), f.all_vs_all_nearest(kk, t), 1)
                _doubled(e.query_vs_ref_nearest(q, r, kk, t), f.query_vs_ref_nearest(q, r, kk, t), 1)
                for cs, bs in zip(e.query_vs_ref_nearest_ex(q, r, kk, t), f.query_vs_ref_nearest_ex(q, r, kk, t)):
                    _doubled(cs, bs, 1)
            _doubled(e.all_vs_all_clusters(t), f.all_vs_all_clusters(t), None)
            _doubled(e.query_vs_ref_clusters(q, r, t), f.query_vs_ref_clusters(q, r, t), None)
            _doubled(e.all_vs_all_linkage(t), f.all_vs_all_linkage(t), 2)
            _doubled(e.query_vs_ref_linkage(q, r, t), f.query_vs_ref_linkage(q, r, t), 2)
            for order in (ids, ids[::-1]):
                assert np.array_equal(e.greedy_reps(order, t), f.greedy_reps(order, t))


# ---- 4. selections on input that separates the modes -------------------------------------------------------------
@pytest.mark.parametrize("algo", ["merge", "join"])
@pytest.mark.parametrize("k", [4, 6, 8])
def test_selections_separate_the_modes(orc, monkeypatch, algo, k):
    seqs = pal_records()
    m = Modes(orc, seqs, k)
    n = m.n
    ids = list(range(n))
    ts = between(m.dc, m.db)
    splits = splitting(n, m.dc, m.db)
    assert ts and splits
    rects = [(ids, ids), ([0, 4, 4, 9, 13, 17], [1, 5, 2, 4, 12, 14, 14, 8]), ([2, 13], ids)]
    with _engine(monkeypatch, seqs, k, CAN, algo=algo) as e, _engine(monkeypatch, seqs, k, BOTH, algo=algo) as f:
        jr._check(e.all_vs_all(), (m.ic, m.dc))
        ia, ib = (x.astype(np.uint32) for x in m.iu)
        for t in ts:
            got = e.all_vs_all_within(t)
            jr._check(got, jr._hits_ref(ia, ib, m.ic, m.dc, t), t)
            assert not _same(got, f.all_vs_all_within(t)), t
            first, count = 5, n * (n - 1) // 2 - 40
            s = slice(first, first + count)
            jr._check(e.all_vs_all_range_within(n, first, count, t), jr._hits_ref(ia[s], ib[s], m.ic[s], m.dc[s], t), t)
            for q, r in rects:
                pa = np.repeat(np.arange(len(q), dtype=np.uint32), len(r))
                pb = np.tile(np.arange(len(r), dtype=np.uint32), len(q))
                jr._check(e.query_vs_ref_within(q, r, t),
                          jr._hits_ref(pa, pb, m.IC[np.ix_(q, r)].ravel(), m.DC[np.ix_(q, r)].ravel(), t), (q, t))
            for kk in (1, 3):
                got = e.all_vs_all_nearest(kk, t)
                jr._check(got, jr._nearest_ref(m.IC, m.DC, ids, ids, kk, t, True), (kk, t))
                assert not _same(got, f.all_vs_all_nearest(kk, t)), (kk, t)
                for q, r in rects:
                    for excl in (False, True):
                        want_q = jr._nearest_ref(m.IC[np.ix_(q, r)], m.DC[np.ix_(q, r)], q, r, kk, t, excl)
                        want_r = jr._nearest_ref(m.IC[np.ix_(r, q)], m.DC[np.ix_(r, q)], r, q, kk, t, excl)
                        got = e.query_vs_ref_nearest(q, r, kk, t, exclude_self=excl)
                        jr._check(got, want_q, (q, kk, t))
                        if q is ids:
                            assert not _same(got, f.query_vs_ref_nearest(q, r, kk, t, exclude_self=excl)), (kk, t)
                        qs, rs = e.query_vs_ref_nearest_ex(q, r, kk, t, exclude_self=excl)
                        jr._check(qs, want_q, (q, kk, t))
                        jr._check(rs, want_r, (q, kk, t))
                        if q is ids:
                            fq, fr = f.query_vs_ref_nearest_ex(q, r, kk, t, exclude_self=excl)
                            assert not _same(qs, fq) and not _same(rs, fr), (kk, t)
            got = e.all_vs_all_linkage(t)
            tl._eq(got, tl._oracle(n, m.ic, m.dc, t), t)
            assert not _same(got, f.all_vs_all_linkage(t)), t
            for q, r in rects:
                tl._eq(e.query_vs_ref_linkage(q, r, t), tl._rect_oracle(m.IC, m.DC, q, r, t), (q, t))
        rect_differs = False
        for t in splits:
            got = e.all_vs_all_clusters(t)
            tc._eq(got, tc._oracle(n, m.dc, t), t)
            assert not np.array_equal(got[0], f.all_vs_all_clusters(t)[0]), t
            for q, r in rects:
                ql, rl = e.query_vs_ref_clusters(q, r, t)
                wq, wr = tc._rect_oracle(m.DC, q, r, t)
                assert np.array_equal(ql, wq) and np.array_equal(rl, wr), (q, t)
                fq, fr = f.query_vs_ref_clusters(q, r, t)
                rect_differs |= not (np.array_equal(ql, fq) and np.array_equal(rl, fr))
            got = e.all_vs_all_linkage(t)
            tl._eq(got, tl._oracle(n, m.ic, m.dc, t), t)
        assert rect_differs


# ---- 5. the block-join overflow redo -----------------------------------------------------------------------------
def test_redo_coarse_tables(orc, monkeypatch):
    """recipe A of test_gpu_join_redo at K = 16 (palindromic inserts): the dense call and the linkage form"""
    k = 16
    seqs = jr._recipe_a(k, gkd.DNA)
    m = Modes(orc, seqs, k)
    n = m.n
    assert (m.dc != m.db).any()
    with _engine(monkeypatch, seqs, k, CAN, algo="join", coarse=True) as e:
        jr._check(jr._redone(e, lambda: e.all_vs_all(), k), (m.ic, m.dc))
        q, r = [3, 3, 0, 20, 3, 33] * 6, [9, 3, 3, 39, 20]
        jr._check(jr._redone(e, lambda: e.query_vs_ref(q, r), k), (m.IC[np.ix_(q, r)], m.DC[np.ix_(q, r)]))
        for t in between(m.dc, m.db) + [1.0]:
            tl._eq(jr._redone(e, lambda: e.all_vs_all_linkage(t), k), tl._oracle(n, m.ic, m.dc, t), t)


def test_redo_skewed_imports(orc, monkeypatch):
    """recipe B of test_gpu_join_redo (K = 21): imported sets are counted as they are, |S| = |C|; the dense call and the
    absorb form"""
    k = 21
    sets = jr._mixed(k)
    n = len(sets)
    ks = jr.KeySets(orc, sets, k)
    I = (ks.M @ ks.M.T).toarray().astype(np.uint64)
    D = jr._distances(orc, I, ks.count[:, None], ks.count[None, :])
    ui, ud = jr._upper(I, D)
    monkeypatch.setenv("GKD_ISECT_ALGO", "join")
    monkeypatch.delenv("GKD_TABLE_TMAX", raising=False)
    with gkd.Engine(k=k, strand_mode=CAN) as e:
        offs = np.r_[0, np.cumsum([len(s) for s in sets])]
        assert e.import_sets(np.concatenate(sets).astype(np.uint64), offs) == 0
        for i in (0, 64, 130):
            assert e.set_size(i) == (int(ks.count[i]), int(ks.count[i]), 0)
        jr._check(jr._redone(e, lambda: e.all_vs_all(), k), (ui, ud))
        ids = list(range(n))
        for kk, t in ((1, 1.0), (5, 0.9), (256, 1.0)):
            got = jr._redone(e, lambda: e.all_vs_all_nearest(kk, t), k)
            jr._check(got, jr._nearest_ref(I, D, ids, ids, kk, t, True), (kk, t))


# ---- 6. more than one 64 Mi-pair chunk ---------------------------------------------------------------------------
def test_absorb_over_two_chunks(orc, monkeypatch):
    """~12,000 gene-sized records (7.2e7 pairs, two chunks, the boundary inside row 8,873); copies of one record on
    both sides of the boundary.  The triangle's lists must equal the rectangle's and the oracle on sampled rows."""
    n = 12_000
    seqs = tc._seqs(77, [900 + (i * 37) % 400 for i in range(n)], families=40)
    dup = [40, 3_000, 8_800, 8_873, 11_999]
    for i in dup[1:]:
        seqs[i] = seqs[dup[0]]
    k, kk = 20, 4
    ids = np.arange(n, dtype=np.uint32)
    sample = np.array([0, 40, 8_872, 8_873, 8_874, 11_998, 11_999])
    osets = [orc.IntSet(s, k) for s in seqs]
    I = np.array([[osets[x].intersect(o)[0] for o in osets] for x in sample], dtype=np.uint64)
    D = np.array([[orc.distance(int(I[a, y]), osets[x].count, osets[y].count) for y in range(n)]
                  for a, x in enumerate(sample)])
    with _engine(monkeypatch, seqs, k, CAN) as e:
        before = e.metrics()["intersect_launches"]
        got = e.all_vs_all_nearest(kk, 1.0)
        assert e.metrics()["pairs"] == n * (n - 1) // 2 and e.metrics()["intersect_launches"] - before == 2
        jr._check(got, e.query_vs_ref_nearest(ids, ids, kk, 1.0, exclude_self=True))
        jr._check([g[sample] for g in got], jr._nearest_ref(I, D, sample, ids, kk, 1.0, True))
        assert list(got[0][8_873]) == [40, 3_000, 8_800, 11_999]


# ---- 7. group ----------------------------------------------------------------------------------------------------
def test_group_equals_single_canonical_context(orc, monkeypatch):
    k = 8
    seqs = pal_records(11)
    m = Modes(orc, seqs, k)
    n = m.n
    ts = between(m.dc, m.db)
    splits = splitting(n, m.dc, m.db)
    with _engine(monkeypatch, seqs, k, CAN) as e:
        want = {"dense": e.all_vs_all()}
        jr._check(want["dense"], (m.ic, m.dc))
        for t in ts:
            want[("within", t)] = e.all_vs_all_within(t)
            want[("nearest", t)] = e.all_vs_all_nearest(3, t)
            want[("linkage", t)] = e.all_vs_all_linkage(t)
        for t in splits:
            want[("clusters", t)] = e.all_vs_all_clusters(t)
    for members in (2, 3):
        with gkd.Group([0] * members, k=k, strand_mode=CAN, workspace_bytes=4 << 20, panel=2) as g:
            per = (n + members - 1) // members
            for i, s in enumerate(seqs):
                assert g.add(min(i // per, members - 1), s) == i
            g.build()
            for key, w in want.items():
                if key == "dense":
                    got = g.all_vs_all()
                else:
                    got = {"within": g.all_vs_all_within, "nearest": lambda t: g.all_vs_all_nearest(3, t),
                           "linkage": g.all_vs_all_linkage, "clusters": g.all_vs_all_clusters}[key[0]](key[1])
                if key[0] == "clusters":
                    tc._eq(got, w, (members, key))
                else:
                    assert _same(got, w), (members, key)


# ---- 8. sketches -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", [gkd.HASH_JAVA_STRING, gkd.HASH_MURMUR3])
def test_sketches(orc, kind):
    rng = np.random.default_rng(21 + kind)
    g = _random(rng, 12_000)
    recs = pal_records(13)
    seqs = [g, _mutate(rng, g, 0.03), _spliced(rng, _random(rng, 6000), 20), b"".join(WORDS) * 3, recs[0], recs[1],
            _random(rng, 60), b"acgtn"]
    for k, width in ((21, 400), (9, 1000), (8, 300), (4, 4096), (6, 120)):
        want = [orc.py_hash_set(orc.py_canonical_set(s.decode(), k), width, kind) for s in seqs]
        both = [orc.py_hash_set(orc.py_kmer_set(s.decode(), k), width, kind) for s in seqs]
        with gkd.Engine(k=k, strand_mode=CAN) as e, gkd.Engine(k=k) as f:
            for s in seqs:
                e.add(s)
                f.add(s)
            e.build()
            f.build()
            got = [e.hash_set(i, width, kind).tolist() for i in range(len(seqs))]
            assert got == want, (k, width)
            assert [f.hash_set(i, width, kind).tolist() for i in range(len(seqs))] == both, (k, width)
            # the palindrome-heavy set, the word records and the dwarf; the random genomes' bottom codes can coincide
            # (String.hashCode ranks strings that start with "a", which are canonical, first)
            assert all(x != y for x, y in zip(got[3:7], both[3:7])), (k, width)
            assert len(want[6]) < width  # a dwarf
            if k == 4:  # "acgtn" holds one k-mer, the palindrome acgt: one code in either mode
                assert len(got[7]) == 1 and got[7] == both[7]
            a = [i for i in range(len(seqs)) for j in range(len(seqs))]
            b = [j for i in range(len(seqs)) for j in range(len(seqs))]
            d = e.sketch_distances(width, a, b, kind)
            assert d.tolist() == [orc.py_sketch_distance(want[i], want[j]) for i, j in zip(a, b)], (k, width)


# ---- 9. greedy representatives -----------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [4, 8])
def test_greedy_reps(orc, monkeypatch, k):
    seqs = pal_records(17)
    m = Modes(orc, seqs, k)
    n = m.n
    orders = [list(range(n)), list(range(n))[::-1], [int(x) for x in np.random.default_rng(k).permutation(n)]]
    with _engine(monkeypatch, seqs, k, CAN) as e, _engine(monkeypatch, seqs, k, BOTH) as f:
        for order in orders:
            ts = greedy_splitting(m.DC, m.DB, order)
            for t in ts + [0.3, 1.0]:
                got = e.greedy_reps(order, t).tolist()
                assert got == greedy(m.DC, order, t), (order, t)
                if t in ts:
                    assert got != f.greedy_reps(order, t).tolist(), (order, t)
        assert any(greedy_splitting(m.DC, m.DB, o) for o in orders)


# ---- 10. sets move between modes ---------------------------------------------------------------------------------
def test_sets_move_between_modes(orc, monkeypatch, tmp_path):
    """the .kset header records K and the alphabet, not the mode, and even-K sets carry palindrome lists in both
    modes: a set saved or adopted in one mode answers as the loading context's mode"""
    import torch

    from genome.distance_b200 import sharding

    k = 8
    seqs = pal_records(19)
    m = Modes(orc, seqs, k)
    n = m.n
    t = between(m.dc, m.db)[1]
    want = {CAN: (m.ic, m.dc), BOTH: (m.ib, m.db)}
    for src, dst in ((BOTH, CAN), (CAN, BOTH)):
        path = str(tmp_path / ("from%d.kset" % src))
        with _engine(monkeypatch, seqs, k, src, workspace_bytes=4 << 20) as e, \
                _engine(monkeypatch, seqs, k, dst) as ref, gkd.Engine(k=k, strand_mode=dst) as f, \
                gkd.Engine(k=k, strand_mode=dst) as h:
            e.save_sets(path)
            assert f.load_sets(path) == (0, n)
            bufs = []
            for p in sharding.plan_panels(e.arena_meta(), 0, n, 5):
                buf = e.arena_view(p["arena"], p["begin"], p["end"]).clone()
                torch.cuda.synchronize()
                assert h.adopt_sets(buf, p["table"]) == p["first"]
                bufs.append(buf)
            for x in (f, h):
                assert [x.set_size(i) for i in range(n)] == [ref.set_size(i) for i in range(n)]
                got = x.all_vs_all()
                jr._check(got, want[dst], (src, dst))
                jr._check(got, ref.all_vs_all(), (src, dst))
                assert not _same(got, e.all_vs_all())
                assert _same(x.all_vs_all_within(t), ref.all_vs_all_within(t)), (src, dst)
                assert _same(x.all_vs_all_nearest(3, t), ref.all_vs_all_nearest(3, t)), (src, dst)


# ---- 11. the protein alphabet has one strand ---------------------------------------------------------------------
def test_protein_is_the_same_in_both_modes(orc, monkeypatch):
    rng = np.random.default_rng(23)
    aa = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWY", dtype=np.uint8)
    base = rng.choice(aa, 3000)
    seqs = []
    for i in range(10):
        a = base.copy()
        hit = rng.random(a.size) < 0.03 * i
        a[hit] = rng.choice(aa, int(hit.sum()))
        seqs.append(a.tobytes())
    seqs += [rng.choice(aa, 500).tobytes(), b"MKV", b""]
    k = 4
    m = Modes(orc, seqs, k, gkd.PROT)
    with _engine(monkeypatch, seqs, k, CAN, gkd.PROT) as e, _engine(monkeypatch, seqs, k, BOTH, gkd.PROT) as f:
        got = e.all_vs_all()
        jr._check(got, (m.ic, m.dc))
        assert _same(got, f.all_vs_all())
        assert [e.set_size(i) for i in range(m.n)] == [f.set_size(i) for i in range(m.n)]
        for t in (0.2, 0.6, 1.0):
            assert _same(e.all_vs_all_within(t), f.all_vs_all_within(t))
            assert _same(e.all_vs_all_nearest(3, t), f.all_vs_all_nearest(3, t))
            assert _same(e.all_vs_all_clusters(t), f.all_vs_all_clusters(t))
            assert _same(e.all_vs_all_linkage(t), f.all_vs_all_linkage(t))
            assert _same([e.greedy_reps(list(range(m.n)), t)], [f.greedy_reps(list(range(m.n)), t)])
        for kind in (gkd.HASH_JAVA_STRING, gkd.HASH_MURMUR3):
            assert e.hash_set(0, 200, kind).tolist() == f.hash_set(0, 200, kind).tolist()
