"""Single-linkage clusters on the device (csrc/intersect.cu k_cluster_link / k_cluster_flatten): every pair within
max_dist links its two sets in a union-find forest kept in HBM across the 64 Mi-pair chunks of a call, and only the
labels leave the device.  label[i] is the smallest id of i's cluster.

The oracle is the dense result thresholded at D (the comparison of gkd_*_within) followed by
scipy.sparse.csgraph.connected_components, relabelled to the smallest index of each component.  Labels and counts must
be equal arrays on every path: both kernel-4 forms, chunks, the forced block-join redo, the rectangle, the literal
policy, groups and the command line.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy import sparse
from scipy.sparse.csgraph import connected_components

import genome.distance_b200 as gkd

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_gpu_join_redo as jr  # noqa: E402  (the overflow recipes)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")


# ---- oracle ------------------------------------------------------------------------------------------------------
def _components(n, a, b):
    """(labels, count) of the graph on n nodes with edges (a, b): each label is the smallest node of its component"""
    a, b = np.asarray(a, dtype=np.int64), np.asarray(b, dtype=np.int64)
    g = sparse.coo_matrix((np.ones(a.size, dtype=np.int8), (a, b)), shape=(n, n))
    nc, comp = connected_components(g, directed=False)
    first = np.full(nc, n, dtype=np.int64)
    np.minimum.at(first, comp, np.arange(n))
    return first[comp].astype(np.uint32), nc


def _upper_ids(n, t):
    """(i, j) of linear indices t of the row-major strict upper triangle of n sets"""
    t = np.asarray(t, dtype=np.int64)
    rows = np.arange(n, dtype=np.int64)
    starts = rows * (2 * n - rows - 1) // 2
    i = np.searchsorted(starts, t, side="right") - 1
    return i, t - starts[i] + i + 1


def _oracle(n, gd, D, m=None):
    """clusters of the first m (default n) sets from the dense triangle gd of n sets"""
    gd = np.asarray(gd)
    if m is None and n > 1 and (gd <= D).all():  # every pair links (no need to list 7e7 edges)
        return np.zeros(n, dtype=np.uint32), 1
    i, j = _upper_ids(n, np.flatnonzero(gd <= D))
    if m is not None:
        keep = j < m
        i, j, n = i[keep], j[keep], m
    return _components(n, i, j)


def _rect_oracle(full, q, r, D):
    """(q_label, r_label) of the bipartite graph q[i] -- r[j] with full[q[i], r[j]] <= D; node i is q[i] and node
    len(q) + j is r[j].  Positions that share an id and have a link end up in one component, so the graph is solved on
    the distinct ids and every position without a link stays alone."""
    q, r = np.asarray(q, dtype=np.int64), np.asarray(r, dtype=np.int64)
    nq, nr = q.size, r.size
    uq, qi = np.unique(q, return_inverse=True)
    ur, ri = np.unique(r, return_inverse=True)
    adj = full[np.ix_(uq, ur)] <= D
    a, b = np.nonzero(adj)
    nu = uq.size + ur.size
    nc, comp = connected_components(sparse.coo_matrix((np.ones(a.size, dtype=np.int8), (a, uq.size + b)),
                                                      shape=(nu, nu)), directed=False)
    node = np.concatenate([np.where(adj.any(1)[qi], comp[qi], nc + np.arange(nq)),
                           np.where(adj.any(0)[ri], comp[uq.size + ri], nc + nq + np.arange(nr))])
    first = np.full(nc + nq + nr, nq + nr, dtype=np.int64)
    np.minimum.at(first, node, np.arange(nq + nr))
    lab = first[node].astype(np.uint32)
    return lab[:nq], lab[nq:]


def _eq(got, want, what=None):
    assert got[1] == want[1], what
    assert got[0].dtype == np.uint32 and np.array_equal(got[0], want[0]), what


def _thresholds(dist):
    """an attained distance below 1 (inclusive boundary) and the double just below it, one below every distance
    (singletons), 1.0 (one cluster) and a negative one (singletons)"""
    dist = np.asarray(dist).ravel()
    below = sorted(set(float(x) for x in dist if x < 1.0))
    out = [float(np.nextafter(float(np.min(dist)), -np.inf)), 1.0, -0.5]
    if below:
        hit = below[len(below) // 2]
        out += [hit, float(np.nextafter(hit, -np.inf))]
    return out


# ---- inputs ------------------------------------------------------------------------------------------------------
def _seqs(seed, lens, protein=False, families=3):
    """related families (members mutated at 0, 0.2, 3 and 15 %) next to unrelated ones"""
    out = []
    for g, n in enumerate(lens):
        a = np.empty(n, dtype=np.uint8)
        mem = g // families
        gkd.synth(a, seed, g % families, mem, [0.0, 0.002, 0.03, 0.15][mem % 4] if mem else 0.0, protein=protein)
        out.append(a.tobytes())
    return out


def _random(rng, n):
    return rng.choice(np.frombuffer(b"acgt", dtype=np.uint8), n).tobytes()


def _mutate(rng, s, rate):
    a = np.frombuffer(s, dtype=np.uint8).copy()
    hit = rng.random(a.size) < rate
    a[hit] = rng.choice(np.frombuffer(b"acgt", dtype=np.uint8), int(hit.sum()))
    return a.tobytes()


def _engine(seqs, k, alphabet=gkd.DNA, **kw):
    e = gkd.Engine(k=k, alphabet=alphabet, **kw)
    for s in seqs:
        e.add(s)
    e.build()
    return e


LENS = [200_000] * 20 + [250_000, 90_000, 25, 0, 600_000, 9_000, 300_000] + [180_000] * 13


@pytest.mark.parametrize("algo", ["merge", "join"])
@pytest.mark.parametrize("k,alphabet", [(21, gkd.DNA), (16, gkd.DNA), (25, gkd.DNA), (8, gkd.PROT)])
def test_forms_and_alphabets(monkeypatch, algo, k, alphabet):
    monkeypatch.setenv("GKD_ISECT_ALGO", algo)
    prot = alphabet == gkd.PROT
    seqs = _seqs(31, [max(n // 4, 8) if n else 0 for n in LENS] if prot else LENS, protein=prot)
    n = len(seqs)
    with _engine(seqs, k, alphabet) as e:
        _, gd = e.all_vs_all(want_inter=False)
        counts = set()
        for D in _thresholds(gd):
            got = e.all_vs_all_clusters(D)
            if algo == "join":
                assert e.metrics()["intersect_kernel"] == 5
            assert e.metrics()["pairs"] == n * (n - 1) // 2
            _eq(got, _oracle(n, gd, D), D)
            counts.add(got[1])
            _eq(e.all_vs_all_clusters(D, n=17), _oracle(n, gd, D, m=17), (17, D))
        assert {1, n} <= counts and len(counts) > 2  # one cluster, singletons, and something in between
        assert e.all_vs_all_clusters(0.5, n=0)[1] == 0
        assert np.array_equal(e.all_vs_all_clusters(1.0, n=1)[0], [0])


def test_chain_is_one_cluster():
    """s0 -> s1 -> ... -> s5, each mutated from the previous one: consecutive distances are <= D while d(s0, s5) > D,
    so the chain is one cluster although the greedy pass splits it.  Identical copies, an empty record and one shorter
    than K sit next to it."""
    rng = np.random.default_rng(8)
    chain = [_random(rng, 30_000)]
    for _ in range(5):
        chain.append(_mutate(rng, chain[-1], 0.012))
    seqs = chain + [_random(rng, 30_000) for _ in range(4)] + [b"", b"acgtacgtac", chain[2], chain[2]]
    n = len(seqs)
    with _engine(seqs, 21) as e:
        _, gd = e.all_vs_all(want_inter=False)
        step = [e.pair(i, i + 1)[2] for i in range(5)]
        D = max(step)
        assert e.pair(0, 5)[2] > D and e.pair(0, 2)[2] > D
        labels, count = e.all_vs_all_clusters(D)
        _eq((labels, count), _oracle(n, gd, D))
        assert list(labels[:6]) == [0] * 6 and labels[12] == labels[13] == 0
        assert list(labels[6:12]) == [6, 7, 8, 9, 10, 11] and count == 7
        assert e.greedy_reps(list(range(6)), D).sum() > 1  # the greedy pass does not join the ends
        assert e.all_vs_all_clusters(float(np.nextafter(D, -np.inf)))[1] > count
        for D_ in _thresholds(gd):
            _eq(e.all_vs_all_clusters(D_), _oracle(n, gd, D_), D_)


def test_more_than_one_chunk():
    """~12,000 gene-sized records: 7.2e7 pairs, two 64 Mi-pair chunks (the boundary lies inside row 8,873).  Records
    11,000 and 11,500 are copies of an unrelated sequence: their only link is in the second chunk."""
    n = 12_000
    seqs = _seqs(77, [900 + (i * 37) % 400 for i in range(n)], families=40)
    rng = np.random.default_rng(2)
    seqs[11_000] = seqs[11_500] = _random(rng, 1_100)
    seqs[40] = seqs[11_999]  # a first-chunk member joined to a second-chunk one
    total = n * (n - 1) // 2
    assert total > 64 << 20
    with _engine(seqs, 21) as e:
        _, gd = e.all_vs_all(want_inter=False)
        below = np.unique(gd[gd < 1.0])
        for D in (float(below[below.size // 3]), 1.0):
            before = e.metrics()["intersect_launches"]
            labels, count = e.all_vs_all_clusters(D)
            m = e.metrics()
            assert m["pairs"] == total and m["intersect_launches"] - before == 2
            _eq((labels, count), _oracle(n, gd, D), D)
            if D < 1.0:
                assert labels[11_500] == 11_000 and (labels == 11_000).sum() == 2
                assert labels[11_999] == labels[40] and count > 1
            else:
                assert count == 1


def test_rectangle():
    seqs = _seqs(12, LENS)
    n = len(seqs)
    with _engine(seqs, 21) as e:
        full = e.query_vs_ref(list(range(n)), list(range(n)))[1]
        cases = [([4, 4, 9, 0, 23, 4], [1, 4, 4, 7, 1, 9, 23, 23, 0]),  # the same id on both sides, repeated
                 (list(range(0, 35)), list(range(3, n))),
                 ([5, 30, 7], list(range(n))),  # fewer than 32 query rows: the join puts r on the table
                 ([2], [])]
        for q, r in cases:
            for D in _thresholds(full[np.ix_(q, r)] if r else full):
                got = e.query_vs_ref_clusters(q, r, D)
                want = _rect_oracle(full, q, r, D)
                assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (q, r, D)
        ql, rl = e.query_vs_ref_clusters([4, 9], [4, 9], 0.0)  # the same id on both sides is one component
        assert list(ql) == [0, 1] and list(rl) == [0, 1]


def test_rectangle_rows_over_three_launches():
    """2^19 references (repeated ids of small records): a launch holds 128 query rows, so 260 rows take three and the
    forest lasts across them"""
    seqs = _seqs(3, [300 + 7 * i for i in range(48)], families=4)
    n = len(seqs)
    rng = np.random.default_rng(5)
    r = rng.permutation(np.tile(np.arange(n, dtype=np.uint32), (1 << 19) // n + 1)[: 1 << 19]).astype(np.uint32)
    q = rng.integers(0, n, 260).astype(np.uint32)
    with _engine(seqs, 21) as e:
        full = e.query_vs_ref(list(range(n)), list(range(n)))[1]
        below = np.unique(full[full < 1.0])
        for D in (float(below[below.size // 2]), float(below[0]) - 1e-9, 1.0):
            before = e.metrics()["intersect_launches"]
            got = e.query_vs_ref_clusters(q, r, D)
            assert e.metrics()["intersect_launches"] - before == 3
            want = _rect_oracle(full, q, r, D)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), D


# ---- the forced block-join redo (recipes of test_gpu_join_redo.py) ------------------------------------------------
def test_redo_coarse_tables(monkeypatch):
    k = 25
    seqs = jr._recipe_a(k, gkd.DNA)
    n = len(seqs)
    q, r = [3, 3, 0, 20, 3, 33] * 6, [9, 3, 3, 39, 20]
    with jr._engine(monkeypatch, "merge", seqs, k, coarse=True) as m, \
            jr._engine(monkeypatch, "join", seqs, k, coarse=True) as e:
        _, gd = m.all_vs_all(want_inter=False)
        full = m.query_vs_ref(list(range(n)), list(range(n)))[1]
        for D in _thresholds(gd):
            got = jr._redone(e, lambda: e.all_vs_all_clusters(D), k)
            _eq(got, _oracle(n, gd, D), D)
            _eq(got, m.all_vs_all_clusters(D), D)
            ql, rl = jr._redone(e, lambda: e.query_vs_ref_clusters(q, r, D), k)
            wq, wr = _rect_oracle(full, q, r, D)
            assert np.array_equal(ql, wq) and np.array_equal(rl, wr), D


def test_redo_skewed_imports(monkeypatch):
    k = 21
    sets = jr._mixed(k)
    n = len(sets)
    with jr._engine(monkeypatch, "merge", k=k, keysets=sets) as m, jr._engine(monkeypatch, "join", k=k, keysets=sets) as e:
        _, gd = m.all_vs_all(want_inter=False)
        full = m.query_vs_ref(list(range(n)), list(range(n)))[1]
        for D in _thresholds(gd):
            got = jr._redone(e, lambda: e.all_vs_all_clusters(D), k)
            _eq(got, _oracle(n, gd, D), D)
            _eq(got, m.all_vs_all_clusters(D), D)
            for q, r in ((list(range(60, 101)), list(range(n))), ([64, 65, 64, 3] * 10, [64, 3, 3, 139, 70])):
                ql, rl = jr._redone(e, lambda: e.query_vs_ref_clusters(q, r, D), k)
                wq, wr = _rect_oracle(full, q, r, D)
                assert np.array_equal(ql, wq) and np.array_equal(rl, wr), (q, D)


def test_redo_only_in_the_second_chunk(monkeypatch):
    """12,000 imported sets whose rows from 9,000 on are crafted: only the second chunk overflows (join, join, merge
    redo).  The links of the first chunk must survive the redo, and the discarded attempt must add none."""
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
        _, gd = m.all_vs_all(want_inter=False)
        want = {D: m.all_vs_all_clusters(D) for D in (0.5, 1.0)}
    with jr._engine(monkeypatch, "join", k=k, keysets=sets) as e:
        for D, w in want.items():
            got = jr._redone(e, lambda: e.all_vs_all_clusters(D), k, launches=3)
            _eq(got, _oracle(n, gd, D), D)
            _eq(got, w, D)
        assert got[1] == 1
    labels = want[0.5][0]
    assert labels[11_999] == labels[8_873] == labels[40] and 1 < want[0.5][1] < n


def test_literal_ambiguous_context():
    """GKD_AMBIG_LITERAL with runs of N: kernel 5 adds the shared literal k-mers, counted on the host, and links on the
    device; a rectangle of sets without literals runs as in a skip context"""
    rng = np.random.default_rng(9)
    seqs = []
    for i, s in enumerate(_seqs(40, [60_000] * 12)):
        a = np.frombuffer(s, dtype=np.uint8).copy()
        if i not in (1, 5, 9):
            for _ in range(4):
                p = int(rng.integers(0, a.size - 40))
                a[p:p + int(rng.integers(1, 30))] = ord("n")
        seqs.append(a.tobytes())
    seqs[7] = seqs[2]
    n = len(seqs)
    ids = list(range(n))
    with _engine(seqs, 21, ambig_policy=gkd.AMBIG_LITERAL) as e:
        _, gd = e.all_vs_all(want_inter=False)
        full = e.query_vs_ref(ids, ids)[1]
        for D in _thresholds(gd):
            _eq(e.all_vs_all_clusters(D), _oracle(n, gd, D), D)
            for q, r in (([0, 3, 3, 11], ids), ([1, 5], [9, 1, 5, 5])):
                ql, rl = e.query_vs_ref_clusters(q, r, D)
                wq, wr = _rect_oracle(full, q, r, D)
                assert np.array_equal(ql, wq) and np.array_equal(rl, wr), (q, D)


def test_group_equals_single_context():
    """13 sets on 2 to 4 members (4 members: the last one holds a single set).  Sets 1 and 11 are copies of an
    unrelated sequence on different members, so their component has only a cross-member link; copies of set 3 on
    every member join components through ring calls."""
    import torch

    seqs = _seqs(21, [150_000] * 9 + [0, 40_000, 220_000, 100_000])
    rng = np.random.default_rng(4)
    seqs[1] = seqs[11] = _random(rng, 120_000)
    for i in (6, 9, 12):
        seqs[i] = seqs[3]
    n = len(seqs)
    with _engine(seqs, 20) as e:
        _, gd = e.all_vs_all(want_inter=False)
        want = {D: e.all_vs_all_clusters(D) for D in _thresholds(gd)}
    for D, w in want.items():
        _eq(w, _oracle(n, gd, D), D)
    D_mid = max(D for D in want if D < 1.0)
    assert want[D_mid][0][11] == 1 and (want[D_mid][0] == 1).sum() == 2
    ndev = torch.cuda.device_count()
    for members in (2, 3, 4):
        devices = [m % ndev for m in range(members)]
        with gkd.Group(devices, k=20, workspace_bytes=4 << 20, panel=2) as g:
            per = (n + members - 1) // members
            for i, s in enumerate(seqs):
                assert g.add(min(i // per, members - 1), s) == i
            g.build()
            for D, w in want.items():
                _eq(g.all_vs_all_clusters(D), w, (members, D))


def _fasta(path, seqs):
    with open(path, "w") as f:
        for i, s in enumerate(seqs):
            f.write(">r%04d rec %d\n" % (i, i))
            t = s.decode()
            for x in range(0, len(t), 80):
                f.write(t[x:x + 80] + "\n")


def _run(args):
    p = subprocess.run([GKD] + args, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    return p.stdout


def test_cli_fastadist_clusters(tmp_path):
    import torch

    rng = np.random.default_rng(6)
    seqs = _seqs(61, [30_000] * 14 + [5_000, 200])
    seqs[9] = seqs[2]
    seqs[3] = seqs[15] = _random(rng, 8_000)
    fa = tmp_path / "in.fa"
    _fasta(fa, seqs)
    n = len(seqs)
    full = _run(["fastaDist", "-i", str(fa)]).split("\n")
    rows = [ln.split("\t") for ln in full[1:] if ln]
    assert len(rows) == n * (n - 1) // 2
    gd = np.array([float(r[4]) for r in rows])
    dists = sorted(set(float(x) for x in gd[gd < 1.0]))
    group = ["--gpus", "2"] if torch.cuda.device_count() >= 2 else ["--devices", "0,0"]
    for D in (dists[len(dists) // 2], 0.5, 1.0):
        labels, _ = _oracle(n, gd, D)
        want = "seq\tname\tcluster\n" + "".join("r%04d\trec %d\tr%04d\n" % (i, i, labels[i]) for i in range(n))
        args = ["fastaDist", "-i", str(fa), "--clusters", "--maxDist", repr(D)]
        assert _run(args) == want, D
        assert _run(args + group) == want, D
