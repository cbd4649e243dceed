"""The single-linkage hierarchy on the device (csrc/intersect.cu k_link_*): after kernel 4 each 64 Mi-pair chunk's
pairs within max_dist are compacted, and Boruvka rounds replace the call's forest F (in HBM) with MSF(F u chunk) under
the strict order (distance bits, min key, max key).  Only the forest leaves the device.

The oracle ranks the dense result's edges <= D with np.lexsort by (distance bits, min key, max key) and runs
scipy.sparse.csgraph.minimum_spanning_tree on weights rank + 1 (raw distances would read zeros as missing edges and
break ties arbitrarily).  The comparison is exact: equal a, b, inter and dist arrays with their dtypes.  For every
threshold t <= D the components of the edges with dist <= t must also be the labels of all_vs_all_clusters(t).
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest
from scipy import sparse
from scipy.sparse.csgraph import minimum_spanning_tree

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_gpu_clusters as tc  # noqa: E402  (inputs, thresholds, component oracle, FASTA helpers)
import test_gpu_join_redo as jr  # noqa: E402  (the overflow recipes)

pytestmark = pytest.mark.gpu


# ---- oracle ------------------------------------------------------------------------------------------------------
def _msf(nodes, na, nb, a, b, inter, dist, ka=None, kb=None):
    """(a, b, inter, dist) of the minimum spanning forest of the edges na -- nb (reported as a, b) in ascending order of
    (distance bits, min key, max key); keys default to the nodes"""
    na, nb = np.asarray(na, dtype=np.int64), np.asarray(nb, dtype=np.int64)
    ka = na if ka is None else np.asarray(ka, dtype=np.int64)
    kb = nb if kb is None else np.asarray(kb, dtype=np.int64)
    dist = np.ascontiguousarray(dist, dtype=np.float64)
    order = np.lexsort((np.maximum(ka, kb), np.minimum(ka, kb), dist.view(np.uint64)))
    rank = np.empty(order.size, dtype=np.float64)
    rank[order] = np.arange(1, order.size + 1)
    t = minimum_spanning_tree(sparse.csr_matrix((rank, (na, nb)), shape=(nodes, nodes)))
    sel = order[np.sort(t.data).astype(np.int64) - 1]
    return (np.asarray(a)[sel].astype(np.uint32), np.asarray(b)[sel].astype(np.uint32),
            np.asarray(inter)[sel].astype(np.uint64), dist[sel])


def _oracle(n, gi, gd, D, m=None):
    """the forest of the first m (default n) sets from the dense triangle (gi, gd) of n sets"""
    t = np.flatnonzero(np.asarray(gd) <= D)
    i, j = tc._upper_ids(n, t)
    if m is not None:
        keep = j < m
        i, j, t, n = i[keep], j[keep], t[keep], m
    return _msf(n, i, j, i, j, np.asarray(gi)[t], np.asarray(gd)[t])


def _rect_oracle(fi, fd, q, r, D, q_key=None, r_key=None):
    """the forest of the rectangle q x r from the full matrices (fi, fd): node i is q[i], node len(q) + j is r[j]"""
    q, r = np.asarray(q, dtype=np.int64), np.asarray(r, dtype=np.int64)
    nq, nr = q.size, r.size
    js = [np.flatnonzero(fd[x][r] <= D) for x in q]  # row by row: q x r can be 10^8 pairs
    i = np.repeat(np.arange(nq), [x.size for x in js])
    j = np.concatenate(js) if js else np.zeros(0, dtype=np.int64)
    ka = i if q_key is None else np.asarray(q_key, dtype=np.int64)[i]
    kb = nq + j if r_key is None else np.asarray(r_key, dtype=np.int64)[j]
    return _msf(nq + nr, i, nq + j, i, j, fi[q[i], r[j]], fd[q[i], r[j]], ka, kb)


def _eq(got, want, what=None):
    for g, w, dt in zip(got, want, (np.uint32, np.uint32, np.uint64, np.float64)):
        assert g.dtype == dt and w.dtype == dt, what
        assert g.shape == w.shape and np.array_equal(g, w), what


def _consistent(e, got, D, n):
    """the clusters at every threshold t <= D are the components of the forest edges with dist <= t"""
    a, b, _, d = got
    ts = sorted(set(float(x) for x in d))
    for t in [t for t in tc._thresholds(d if d.size else np.array([1.0])) if t <= D] + ts[:: max(1, len(ts) // 6)]:
        keep = d <= t
        assert np.array_equal(e.all_vs_all_clusters(t, n=n)[0], tc._components(n, a[keep], b[keep])[0]), t


# ---- tests -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", ["merge", "join"])
@pytest.mark.parametrize("k,alphabet", [(21, gkd.DNA), (16, gkd.DNA), (25, gkd.DNA), (8, gkd.PROT)])
def test_forms_and_alphabets(monkeypatch, algo, k, alphabet):
    monkeypatch.setenv("GKD_ISECT_ALGO", algo)
    prot = alphabet == gkd.PROT
    seqs = tc._seqs(31, [max(n // 4, 8) if n else 0 for n in tc.LENS] if prot else tc.LENS, protein=prot)
    seqs[33] = seqs[36] = seqs[5]  # identical copies: the tie order decides which edges are kept
    n = len(seqs)
    with tc._engine(seqs, k, alphabet) as e:
        gi, gd = e.all_vs_all()
        sizes = set()
        for D in tc._thresholds(gd):
            got = e.all_vs_all_linkage(D)
            if algo == "join":
                assert e.metrics()["intersect_kernel"] == 5
            assert e.metrics()["pairs"] == n * (n - 1) // 2
            _eq(got, _oracle(n, gi, gd, D), D)
            assert got[0].size == n - e.all_vs_all_clusters(D)[1]
            sizes.add(got[0].size)
            _eq(e.all_vs_all_linkage(D, n=17), _oracle(n, gi, gd, D, m=17), (17, D))
            if D >= 0:
                _consistent(e, got, D, n)
        assert {0, n - 1} <= sizes and len(sizes) > 2  # no edge, a spanning tree, and something in between
        for m in (0, 1):
            assert all(x.size == 0 for x in e.all_vs_all_linkage(1.0, n=m))
        assert e.all_vs_all_linkage(1.0, n=2)[0].tolist() == [0]


def test_chain_and_copies():
    """a mutation chain s0 -> ... -> s5, unrelated records, an empty one, one shorter than K and copies of s2: the
    spanning tree at 1.0 ties at distance 1.0 for every unrelated pair"""
    rng = np.random.default_rng(8)
    chain = [tc._random(rng, 30_000)]
    for _ in range(5):
        chain.append(tc._mutate(rng, chain[-1], 0.012))
    seqs = chain + [tc._random(rng, 30_000) for _ in range(4)] + [b"", b"acgtacgtac", chain[2], chain[2], chain[2]]
    n = len(seqs)
    with tc._engine(seqs, 21) as e:
        gi, gd = e.all_vs_all()
        for D in tc._thresholds(gd) + [max(e.pair(i, i + 1)[2] for i in range(5))]:
            got = e.all_vs_all_linkage(D)
            _eq(got, _oracle(n, gi, gd, D), D)
            if D >= 0:
                _consistent(e, got, D, n)
        a, b, _, d = e.all_vs_all_linkage(0.0)
        assert list(zip(a, b)) == [(2, 12), (2, 13), (2, 14)] and not d.any()


def test_null_arrays_cap_and_device_memory():
    import torch

    seqs = tc._seqs(5, [40_000] * 24)
    seqs[20] = seqs[3]
    n = len(seqs)
    with tc._engine(seqs, 21) as e:
        want = e.all_vs_all_linkage(0.9)
        w = want[0].size
        assert w > 4

        def raw(cap, arrays):
            ptr = [None if x is None else (x.data_ptr() if torch.is_tensor(x) else x.ctypes.data) for x in arrays]
            h = _lib.GkdHits(*ptr, cap, 0)
            e._ck(e._L.gkd_all_vs_all_linkage(e._h, n, 0.9, C.byref(h)))
            return h.n

        host = [np.zeros(w, dtype=dt) for dt in (np.uint32, np.uint32, np.uint64, np.float64)]
        for cap in (0, 1, w - 1):
            out = [np.full(w, 7, dtype=x.dtype) for x in host]
            assert raw(cap, out) == w
            for o, x in zip(out, want):
                assert np.array_equal(o[:cap], x[:cap]) and (o[cap:] == 7).all(), cap
        for drop in range(4):  # each array NULL in turn
            out = [None if i == drop else np.zeros(w, dtype=x.dtype) for i, x in enumerate(host)]
            assert raw(w, out) == w
            for o, x in zip(out, want):
                assert o is None or np.array_equal(o, x)
        assert raw(0, [None] * 4) == w
        dev = [torch.zeros(w, dtype=t, device="cuda:0") for t in (torch.int32, torch.int32, torch.int64, torch.float64)]
        assert raw(w, dev) == w
        got = [dev[0].cpu().numpy().view(np.uint32), dev[1].cpu().numpy().view(np.uint32),
               dev[2].cpu().numpy().view(np.uint64), dev[3].cpu().numpy()]
        _eq(got, want)


def test_more_than_one_chunk():
    """~12,000 gene-sized records: two 64 Mi-pair chunks.  Copies of one record at 5 and 40 (first chunk) and 11,999
    (second chunk) tie at distance 0 across the boundary; records 11,000 and 11,500 link only in the second chunk."""
    n = 12_000
    seqs = tc._seqs(77, [900 + (i * 37) % 400 for i in range(n)], families=40)
    rng = np.random.default_rng(2)
    seqs[11_000] = seqs[11_500] = tc._random(rng, 1_100)
    seqs[40] = seqs[11_999] = seqs[5]
    total = n * (n - 1) // 2
    with tc._engine(seqs, 21) as e:
        gi, gd = e.all_vs_all()
        below = np.unique(gd[gd < 1.0])
        for D in (float(below[below.size // 3]), float(below[-1])):
            before = e.metrics()["intersect_launches"]
            got = e.all_vs_all_linkage(D)
            m = e.metrics()
            assert m["pairs"] == total and m["intersect_launches"] - before == 2
            _eq(got, _oracle(n, gi, gd, D), D)
            pairs = set(zip(got[0].tolist(), got[1].tolist()))
            assert {(5, 40), (5, 11_999), (11_000, 11_500)} <= pairs and (40, 11_999) not in pairs
            assert np.array_equal(e.all_vs_all_clusters(D)[0], tc._components(n, got[0], got[1])[0])


def test_rectangle_default_and_explicit_keys():
    seqs = tc._seqs(12, tc.LENS)
    seqs[30] = seqs[4]
    n = len(seqs)
    rng = np.random.default_rng(3)
    with tc._engine(seqs, 21) as e:
        fi, fd = e.query_vs_ref(list(range(n)), list(range(n)))
        cases = [([4, 4, 9, 0, 23, 4, 30], [1, 4, 4, 7, 1, 9, 23, 23, 0, 30]),  # ids on both sides, repeated
                 (list(range(0, 35)), list(range(3, n))),
                 ([5, 30, 7], list(range(n)))]  # fewer than 32 query rows: the join puts r on the table
        for q, r in cases:
            keys = rng.permutation(10 * (len(q) + len(r)))[: len(q) + len(r)].astype(np.uint32)
            for D in tc._thresholds(fd[np.ix_(q, r)]):
                _eq(e.query_vs_ref_linkage(q, r, D), _rect_oracle(fi, fd, q, r, D), (q, D))
                qk, rk = keys[: len(q)], keys[len(q):]
                _eq(e.query_vs_ref_linkage(q, r, D, qk, rk), _rect_oracle(fi, fd, q, r, D, qk, rk), (q, D, "keys"))
                qk = qk + np.uint32(len(q) + len(r))  # clear of the default reference keys len(q) + j
                _eq(e.query_vs_ref_linkage(q, r, D, q_key=qk), _rect_oracle(fi, fd, q, r, D, q_key=qk), (q, D, "q"))
        assert all(x.size == 0 for x in e.query_vs_ref_linkage([2], [], 1.0))
        with pytest.raises(RuntimeError, match="not distinct"):
            e.query_vs_ref_linkage([1, 2], [3], 0.5, [5, 6], [6])


def test_rectangle_rows_over_three_launches():
    """2^19 references (repeated ids of small records): a launch holds 128 query rows, so 260 rows take three and the
    forest lasts across them.  Repeated ids tie at distance 0 everywhere."""
    seqs = tc._seqs(3, [300 + 7 * i for i in range(48)], families=24)
    n = len(seqs)
    rng = np.random.default_rng(5)
    r = rng.permutation(np.tile(np.arange(n, dtype=np.uint32), (1 << 19) // n + 1)[: 1 << 19]).astype(np.uint32)
    q = rng.integers(0, n, 260).astype(np.uint32)
    keys = rng.permutation(1 << 21)[: q.size + r.size].astype(np.uint32)
    with tc._engine(seqs, 21) as e:
        fi, fd = e.query_vs_ref(list(range(n)), list(range(n)))
        below = np.unique(fd[fd < 1.0])
        assert below.size > 1
        for D in (float(below[-1]), 0.0):
            before = e.metrics()["intersect_launches"]
            got = e.query_vs_ref_linkage(q, r, D)
            assert e.metrics()["intersect_launches"] - before == 3
            _eq(got, _rect_oracle(fi, fd, q, r, D), D)
            got = e.query_vs_ref_linkage(q, r, D, keys[: q.size], keys[q.size:])
            _eq(got, _rect_oracle(fi, fd, q, r, D, keys[: q.size], keys[q.size:]), (D, "keys"))


# ---- the forced block-join redo (recipes of test_gpu_join_redo.py) ------------------------------------------------
def test_redo_coarse_tables(monkeypatch):
    k = 25
    seqs = jr._recipe_a(k, gkd.DNA)
    n = len(seqs)
    q, r = [3, 3, 0, 20, 3, 33] * 6, [9, 3, 3, 39, 20]
    with jr._engine(monkeypatch, "merge", seqs, k, coarse=True) as m, \
            jr._engine(monkeypatch, "join", seqs, k, coarse=True) as e:
        gi, gd = m.all_vs_all()
        fi, fd = m.query_vs_ref(list(range(n)), list(range(n)))
        for D in tc._thresholds(gd):
            got = jr._redone(e, lambda: e.all_vs_all_linkage(D), k)
            _eq(got, _oracle(n, gi, gd, D), D)
            _eq(got, m.all_vs_all_linkage(D), D)
            got = jr._redone(e, lambda: e.query_vs_ref_linkage(q, r, D), k)
            _eq(got, _rect_oracle(fi, fd, q, r, D), (q, D))


def test_redo_skewed_imports(monkeypatch):
    k = 21
    sets = jr._mixed(k)
    n = len(sets)
    with jr._engine(monkeypatch, "merge", k=k, keysets=sets) as m, jr._engine(monkeypatch, "join", k=k, keysets=sets) as e:
        gi, gd = m.all_vs_all()
        fi, fd = m.query_vs_ref(list(range(n)), list(range(n)))
        for D in tc._thresholds(gd):
            got = jr._redone(e, lambda: e.all_vs_all_linkage(D), k)
            _eq(got, _oracle(n, gi, gd, D), D)
            for q, r in ((list(range(60, 101)), list(range(n))), ([64, 65, 64, 3] * 10, [64, 3, 3, 139, 70])):
                got = jr._redone(e, lambda: e.query_vs_ref_linkage(q, r, D), k)
                _eq(got, _rect_oracle(fi, fd, q, r, D), (q, D))


def test_redo_only_in_the_second_chunk(monkeypatch):
    """12,000 imported sets whose rows from 9,000 on are crafted: only the second chunk overflows (join, join, merge
    redo).  The forest of the first chunk must survive the redo, and the discarded attempt must add nothing."""
    k = 21
    n, first_crafted = 12_000, 9_000
    rng = np.random.default_rng(29)
    band = jr._band(k, jr.BAND_M[k] << 31)
    uni = jr._uniform(rng, k, 200_000)
    sets = jr._families(rng, uni, first_crafted, 330, 200, band, 20) + \
        jr._families(rng, band, n - first_crafted, 330, 100)
    for i in (3_000, 8_873, 10_000, 11_999):
        sets[i] = sets[40]
    with jr._engine(monkeypatch, "merge", k=k, keysets=sets) as m:
        gi, gd = m.all_vs_all()
        want = m.all_vs_all_linkage(0.5)
    _eq(want, _oracle(n, gi, gd, 0.5))
    assert 0 < want[0].size < n - 1
    with jr._engine(monkeypatch, "join", k=k, keysets=sets) as e:
        _eq(jr._redone(e, lambda: e.all_vs_all_linkage(0.5), k, launches=3), want)


def test_literal_ambiguous_context():
    """GKD_AMBIG_LITERAL with runs of N: kernel 5 adds the shared literal k-mers, counted on the host, and the forest is
    built on the device; a rectangle of sets without literals runs as in a skip context"""
    rng = np.random.default_rng(9)
    seqs = []
    for i, s in enumerate(tc._seqs(40, [60_000] * 12)):
        a = np.frombuffer(s, dtype=np.uint8).copy()
        if i not in (1, 5, 9):
            for _ in range(4):
                p = int(rng.integers(0, a.size - 40))
                a[p:p + int(rng.integers(1, 30))] = ord("n")
        seqs.append(a.tobytes())
    seqs[7] = seqs[2]
    seqs[10] = seqs[2]
    n = len(seqs)
    ids = list(range(n))
    with tc._engine(seqs, 21, ambig_policy=gkd.AMBIG_LITERAL) as e:
        gi, gd = e.all_vs_all()
        fi, fd = e.query_vs_ref(ids, ids)
        for D in tc._thresholds(gd):
            _eq(e.all_vs_all_linkage(D), _oracle(n, gi, gd, D), D)
            for q, r in (([0, 3, 3, 11, 7], ids), ([1, 5], [9, 1, 5, 5]), ([2, 7, 1], [10, 5, 9, 2])):
                _eq(e.query_vs_ref_linkage(q, r, D), _rect_oracle(fi, fd, q, r, D), (q, D))


def test_group_equals_single_context():
    """16 sets on 2 to 4 members.  On 4 members (ids 0-3, 4-7, 8-11, 12-15) copies 3, 8, 9 and 13 are identical:
    member 2's ring call has rows 8..11 and the columns 12..15 then 2..3, so its columns span peers on both sides of
    its own ids.  The 4-cycle 8, 9 x 13, 3 at distance 0 is broken in that call, and only global-id keys make it drop
    the edge one context drops."""
    import torch

    seqs = tc._seqs(21, [150_000] * 9 + [0, 40_000, 220_000, 100_000, 60_000, 80_000, 30_000])
    rng = np.random.default_rng(4)
    seqs[1] = seqs[14] = tc._random(rng, 120_000)
    for i in (8, 9, 13):
        seqs[i] = seqs[3]
    n = len(seqs)
    with tc._engine(seqs, 20) as e:
        gi, gd = e.all_vs_all()
        want = {D: e.all_vs_all_linkage(D) for D in tc._thresholds(gd)}
    for D, w in want.items():
        _eq(w, _oracle(n, gi, gd, D), D)
    tree = set(zip(want[1.0][0].tolist(), want[1.0][1].tolist()))
    assert {(3, 8), (3, 9), (3, 13)} <= tree and not {(8, 9), (8, 13), (9, 13)} & tree
    ndev = torch.cuda.device_count()
    for members in (2, 3, 4):
        devices = [m % ndev for m in range(members)]
        with gkd.Group(devices, k=20, workspace_bytes=4 << 20, panel=2) as g:
            per = (n + members - 1) // members
            for i, s in enumerate(seqs):
                assert g.add(min(i // per, members - 1), s) == i
            g.build()
            for D, w in want.items():
                _eq(g.all_vs_all_linkage(D), w, (members, D))


def test_cli_fastadist_linkage(tmp_path):
    import torch

    rng = np.random.default_rng(6)
    seqs = tc._seqs(61, [30_000] * 14 + [5_000, 200])
    seqs[9] = seqs[2]
    seqs[3] = seqs[15] = tc._random(rng, 8_000)
    fa = tmp_path / "in.fa"
    tc._fasta(fa, seqs)
    n = len(seqs)
    full = tc._run(["fastaDist", "-i", str(fa)]).split("\n")
    rows = [ln.split("\t") for ln in full[1:] if ln]
    assert len(rows) == n * (n - 1) // 2
    with tc._engine(seqs, 21) as e:
        gi, gd = e.all_vs_all()
    head = "seq1\tname1\tseq2\tname2\tdistance\n"
    group = ["--gpus", "2"] if torch.cuda.device_count() >= 2 else ["--devices", "0,0"]
    dists = sorted(set(float(x) for x in gd[gd < 1.0]))
    for D in (None, dists[len(dists) // 2], 0.5):
        a, b, _, d = _oracle(n, gi, gd, 1.0 if D is None else D)
        t = [int(i) * (2 * n - int(i) - 1) // 2 + int(j) - int(i) - 1 for i, j in zip(a, b)]
        want = head + "".join("\t".join(rows[x]) + "\n" for x in t)
        args = ["fastaDist", "-i", str(fa), "--linkage"] + ([] if D is None else ["--maxDist", repr(D)])
        got = tc._run(args)
        assert got == want, D
        assert tc._run(args + group) == got, D
        if D is not None:
            assert set(got.split("\n")[1:]) <= set(tc._run(["fastaDist", "-i", str(fa), "--maxDist", repr(D)]).split("\n"))
    assert tc._run(["fastaDist", "-i", str(fa), "--linkage"]).count("\n") == n  # header + n - 1 merges
