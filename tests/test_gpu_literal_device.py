"""GKD_AMBIG_LITERAL contexts on the device.  The literal k-mers of a set (windows with a character outside acgt) live
on the host; per chunk the host counts the literal k-mers each pair shares, and kernel 5 (csrc/intersect.cu
PairCounts::value) adds them, and each set's literal k-mers, to the counts of kernel 4.  Every form then runs its device
kernels as in a skip context.

Checked here: a selection copies what it copies in a skip context; the block-join overflow redo (recipe A of
test_gpu_join_redo.py) under every form; a call of two chunks.  Every form is compared with the dense result of the same
context or of one pinned to the merge kernel, and the dense result with the oracle's literal string sets.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import genome.distance_b200 as gkd

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_gpu_clusters as tc  # noqa: E402  (inputs, thresholds, component oracle)
import test_gpu_join_redo as jr  # noqa: E402  (the overflow recipe, redo counter, nearest and hits oracles)
import test_gpu_linkage as tl  # noqa: E402  (the forest oracle)

pytestmark = pytest.mark.gpu


def _n_runs(seqs, seed, every=1):
    """runs of 1 to 29 n in every `every`-th sequence of 40 bases or more"""
    rng = np.random.default_rng(seed)
    out = []
    for i, s in enumerate(seqs):
        a = np.frombuffer(s, dtype=np.uint8).copy()
        if i % every == 0 and a.size >= 40:
            for _ in range(3):
                p = int(rng.integers(0, a.size - 30))
                a[p:p + int(rng.integers(1, 30))] = ord("n")
        out.append(a.tobytes())
    return out


def _engine(monkeypatch, algo, seqs, k, coarse=False):
    """a literal context pinned to one kernel-4 form (switches are read when a context is created)"""
    monkeypatch.setenv("GKD_ISECT_ALGO", algo)
    if coarse:
        monkeypatch.setenv("GKD_TABLE_TMAX", jr.COARSE)
    else:
        monkeypatch.delenv("GKD_TABLE_TMAX", raising=False)
    e = gkd.Engine(k=k, ambig_policy=gkd.AMBIG_LITERAL)
    for s in seqs:
        e.add(s)
    e.build()
    return e


def _check_oracle(orc, seqs, k, pairs, inter, dist):
    """(I, dist) of the pairs (i, j) against orc.StrSet(ambig=LITERAL), doubles by their bits"""
    ss = {}
    for t, (i, j) in enumerate(pairs):
        for x in (i, j):
            if x not in ss:
                ss[x] = orc.StrSet(seqs[x], k, orc.DNA, orc.AMBIG_LITERAL)
        I = ss[i].similarity(ss[j])
        want = orc.distance(I, len(ss[i]), len(ss[j]))
        assert int(inter[t]) == I and np.float64(dist[t]).view(np.uint64) == np.float64(want).view(np.uint64), (i, j)


def test_selection_copies_what_a_skip_context_copies():
    """the within selection reads back 8 bytes per chunk and 24 per hit written, as in a skip context"""
    seqs = _n_runs(tc._seqs(40, [60_000] * 12), 9)
    seqs[7] = seqs[2]
    n = len(seqs)
    total = n * (n - 1) // 2
    iu_a, iu_b = (x.astype(np.uint32) for x in np.triu_indices(n, 1))
    with tc._engine(seqs, 21, ambig_policy=gkd.AMBIG_LITERAL) as e:
        gi, gd = e.all_vs_all()
        L = e._L
        for D in tc._thresholds(gd):
            ha, hb = np.empty(total, dtype=np.uint32), np.empty(total, dtype=np.uint32)
            hi, hd = np.empty(total, dtype=np.uint64), np.empty(total, dtype=np.float64)
            h = gkd._lib.GkdHits(ha.ctypes.data, hb.ctypes.data, hi.ctypes.data, hd.ctypes.data, total, 0)
            before = e.metrics()["d2h_bytes"]
            e._ck(L.gkd_all_vs_all_range_within(e._h, n, 0, total, float(D), C.byref(h)))
            assert e.metrics()["d2h_bytes"] - before == 8 + 24 * h.n, D
            jr._check((ha[:h.n], hb[:h.n], hi[:h.n], hd[:h.n]), jr._hits_ref(iu_a, iu_b, gi, gd, D), D)


@pytest.mark.parametrize("k", [16, 25])
def test_overflow_redo(orc, monkeypatch, k):
    """recipe A with runs of n: every form of the join-forced context takes the redo and equals the dense result of a
    context pinned to the merge kernel"""
    seqs = _n_runs(jr._recipe_a(k, gkd.DNA), 5, every=2)
    seqs[20] = seqs[33] = seqs[4]  # ties between sets with literal k-mers
    n = len(seqs)
    ids = list(range(n))
    iu_a, iu_b = (x.astype(np.uint32) for x in np.triu_indices(n, 1))
    with _engine(monkeypatch, "merge", seqs, k, coarse=True) as m, \
            _engine(monkeypatch, "join", seqs, k, coarse=True) as e:
        ui, ud = m.all_vs_all()
        fi, fd = m.query_vs_ref(ids, ids)
        _check_oracle(orc, seqs, k, list(zip(iu_a.tolist(), iu_b.tolist())), ui, ud)
        jr._check((fi[iu_a, iu_b], fd[iu_a, iu_b]), (ui, ud))
        jr._check(jr._redone(e, lambda: e.all_vs_all(), k), (ui, ud))
        for D in jr._thresholds(ud):
            jr._check(jr._redone(e, lambda: e.all_vs_all_within(D), k), jr._hits_ref(iu_a, iu_b, ui, ud, D), D)
            for kk in (1, 5):
                jr._check(jr._redone(e, lambda: e.all_vs_all_nearest(kk, D), k),
                          jr._nearest_ref(fi, fd, ids, ids, kk, D, True), (kk, D))
            tc._eq(jr._redone(e, lambda: e.all_vs_all_clusters(D), k), tc._oracle(n, ud, D), D)
            tl._eq(jr._redone(e, lambda: e.all_vs_all_linkage(D), k), tl._oracle(n, ui, ud, D), D)
        q, r = list(range(0, 35)), list(range(2, n))
        for kk, D in ((1, 1.0), (5, 0.9)):
            qs, rs = jr._redone(e, lambda: e.query_vs_ref_nearest_ex(q, r, kk, D), k)
            jr._check(qs, jr._nearest_ref(fi[np.ix_(q, r)], fd[np.ix_(q, r)], q, r, kk, D, False), (kk, D))
            jr._check(rs, jr._nearest_ref(fi[np.ix_(r, q)], fd[np.ix_(r, q)], r, q, kk, D, False), (kk, D))


def test_two_chunks(orc):
    """~12,000 gene-sized records, every third with runs of n: 7.2e7 pairs, two 64 Mi-pair chunks.  Copies of a record
    at 5, 40 and 11,999 tie at distance 0 across the boundary."""
    n = 12_000
    seqs = _n_runs(tc._seqs(77, [900 + (i * 37) % 400 for i in range(n)], families=40), 13, every=3)
    seqs[40] = seqs[11_999] = seqs[5]
    total = n * (n - 1) // 2

    def two(e, call):
        before = e.metrics()["intersect_launches"]
        out = call()
        m = e.metrics()
        assert m["pairs"] == total and m["intersect_launches"] - before == 2
        return out

    with tc._engine(seqs, 21, ambig_policy=gkd.AMBIG_LITERAL) as e:
        gi, gd = two(e, lambda: e.all_vs_all())
        # sampled pairs through a single-chunk pair list, and a handful through the oracle
        rng = np.random.default_rng(5)
        t = np.concatenate([rng.integers(0, total, 400), [0, total - 1, (64 << 20) - 1, 64 << 20]])
        pa, pb = tc._upper_ids(n, t)
        pi, pd = e.pairs(pa, pb)
        jr._check((pi, pd), (gi[t], gd[t]))
        ci, cd = e.pairs([5, 5, 0], [40, 11_999, 3])
        _check_oracle(orc, seqs, 21, list(zip(pa[:8].tolist(), pb[:8].tolist())) + [(5, 40), (5, 11_999), (0, 3)],
                      np.r_[gi[t[:8]], ci], np.r_[gd[t[:8]], cd])
        assert cd[0] == cd[1] == 0.0
        below = np.unique(gd[gd < 1.0])
        D = float(below[below.size // 3])
        keep = np.flatnonzero(gd <= D)
        i, j = tc._upper_ids(n, keep)
        jr._check(e.all_vs_all_within(D), (i.astype(np.uint32), j.astype(np.uint32), gi[keep], gd[keep]))
        tc._eq(two(e, lambda: e.all_vs_all_clusters(D)), tc._oracle(n, gd, D))
        tl._eq(two(e, lambda: e.all_vs_all_linkage(D)), tl._oracle(n, gi, gd, D))
        near = two(e, lambda: e.all_vs_all_nearest(8, 1.0))
        sample = np.array([0, 5, 40, 8_872, 8_873, 8_874, 11_000, 11_999])
        si, sd = e.query_vs_ref(sample, np.arange(n))
        for x_at, x in enumerate(sample):  # the rectangle's rows are the dense triangle's
            others = np.delete(np.arange(n), x)
            lo, hi = np.minimum(x, others), np.maximum(x, others)
            tt = lo * (2 * n - lo - 1) // 2 + hi - lo - 1
            jr._check((si[x_at][others], sd[x_at][others]), (gi[tt], gd[tt]), x)
        jr._check([g[sample] for g in near], jr._nearest_ref(si, sd, sample, np.arange(n), 8, 1.0, True))
