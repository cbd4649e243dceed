"""The k-nearest-neighbour graph from the upper triangle (csrc/intersect.cu k_nearest_absorb): every pair i < j is
intersected once and offered to both of its rows, and each row keeps a top-k list on the device across the 64 Mi-pair
chunks.  The result must equal, bit for bit, the rectangle q = r = all sets with exclude_self (k_select_nearest) and a
numpy ranking of the dense matrix made symmetric: ascending distance, ties by the smaller id.

The same accumulator gives the reference side of gkd_query_vs_ref_nearest_ex, and the group form merges the members'
partial lists by (distance, global id).

Join-overflow redo: the device-side guard of the absorb kernel (it reads the overflow flag on the stream and writes
nothing when it is set) is forced in tests/test_gpu_join_redo.py, with coarse set tables and skewed imported key sets,
including an overflow in the second chunk only.
"""
import os
import subprocess

import numpy as np
import pytest

import genome.distance_b200 as gkd

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")


def _seqs(seed, lens, protein=False, families=3):
    """related families (members mutated at 0, 0.2, 3 and 15 %) next to unrelated ones"""
    out = []
    for g, n in enumerate(lens):
        a = np.empty(n, dtype=np.uint8)
        mem = g // families
        gkd.synth(a, seed, g % families, mem, [0.0, 0.002, 0.03, 0.15][mem % 4] if mem else 0.0, protein=protein)
        out.append(a.tobytes())
    return out


def _engine(seqs, k, alphabet=gkd.DNA, **kw):
    e = gkd.Engine(k=k, alphabet=alphabet, **kw)
    for s in seqs:
        e.add(s)
    e.build()
    return e


def _thresholds(dist):
    """1.0 (every pair), an attained distance below 1 (inclusive boundary), and one below every distance (no hit)"""
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
        idx = idx[np.lexsort((idx, gd[x][idx]))][:k]
        found[x] = idx.size
        pos[x, :idx.size] = idx
        inter[x, :idx.size] = gi[x][idx]
        dist[x, :idx.size] = gd[x][idx]
    return pos, inter, dist, found


def _check(got, want, what=None):
    for g, w in zip(got, want):
        assert g.shape == w.shape, what
        if g.dtype == np.float64:
            assert np.array_equal(g.view(np.uint64), w.view(np.uint64)), what  # bit-exact
        else:
            assert np.array_equal(g, w), what


def _symmetric(n, gi, gd):
    """the dense triangle of the first n sets as full n x n matrices (the diagonal is never read: exclude_self)"""
    I = np.zeros((n, n), dtype=np.uint64)
    Dm = np.zeros((n, n))
    iu = np.triu_indices(n, 1)
    I[iu], Dm[iu] = gi, gd
    return I + I.T, Dm + Dm.T


LENS = [200_000] * 20 + [250_000, 90_000, 25, 0, 600_000, 9_000, 300_000] + [180_000] * 13


@pytest.mark.parametrize("algo", ["merge", "join"])
@pytest.mark.parametrize("k,alphabet", [(21, gkd.DNA), (16, gkd.DNA), (25, gkd.DNA), (8, gkd.PROT)])
def test_triangle_equals_rectangle_and_dense(monkeypatch, algo, k, alphabet):
    monkeypatch.setenv("GKD_ISECT_ALGO", algo)
    prot = alphabet == gkd.PROT
    seqs = _seqs(31, [max(n // 4, 8) if n else 0 for n in LENS] if prot else LENS, protein=prot)
    n = len(seqs)
    with _engine(seqs, k, alphabet) as e:
        gi, gd = e.all_vs_all()
        I, Dm = _symmetric(n, np.asarray(gi), np.asarray(gd))
        for m in (n, 17):  # every set, and the first m < n
            ids = list(range(m))
            for kk in (1, 5, 256):
                for D in _thresholds(np.asarray(gd)):
                    got = e.all_vs_all_nearest(kk, D, n=m)
                    if algo == "join" and m == n:
                        assert e.metrics()["intersect_kernel"] == 5
                    assert e.metrics()["pairs"] == m * (m - 1) // 2
                    _check(got, _nearest_ref(I[:m, :m], Dm[:m, :m], ids, ids, kk, D, True), (m, kk, D))
                    _check(got, e.query_vs_ref_nearest(ids, ids, kk, D, exclude_self=True), (m, kk, D))


def test_ties_are_broken_by_id():
    """byte-identical copies of two genomes: distance-0 groups, and groups at one equal distance from every other set;
    k cuts through them"""
    seqs = _seqs(44, [120_000] * 24)
    for i in (3, 8, 11, 17, 22):
        seqs[i] = seqs[0]
    for i in (6, 14, 20):
        seqs[i] = seqs[1]
    n = len(seqs)
    ids = list(range(n))
    with _engine(seqs, 21) as e:
        gi, gd = e.all_vs_all()
        I, Dm = _symmetric(n, np.asarray(gi), np.asarray(gd))
        for kk in (1, 2, 3, 4, 7):
            for D in (1.0, 0.0):
                got = e.all_vs_all_nearest(kk, D)
                _check(got, _nearest_ref(I, Dm, ids, ids, kk, D, True), (kk, D))
                _check(got, e.query_vs_ref_nearest(ids, ids, kk, D, exclude_self=True), (kk, D))
        pos, _, dist, found = e.all_vs_all_nearest(3, 1.0)
        assert list(pos[17]) == [0, 3, 8] and (dist[17] == 0.0).all()
        assert list(pos[0]) == [3, 8, 11]


def test_more_than_one_chunk():
    """~12,000 gene-sized records: 7.2e7 pairs, two 64 Mi-pair chunks.  Copies of one record sit on both sides of the
    chunk boundary (inside row 8,873), so equal-distance neighbours of one row arrive in different chunks and from both the
    row and the column side.  The oracle is the rectangle call."""
    n = 12_000
    seqs = _seqs(77, [900 + (i * 37) % 400 for i in range(n)], families=40)
    dup = [40, 3_000, 8_800, 8_871, 8_873, 8_900, 10_000, 11_999]
    for i in dup[1:]:
        seqs[i] = seqs[dup[0]]
    total = n * (n - 1) // 2
    assert total > 64 << 20
    ids = np.arange(n, dtype=np.uint32)
    with _engine(seqs, 21) as e:
        for kk, D in ((1, 1.0), (4, 1.0), (16, 0.6), (256, 1.0)):
            got = e.all_vs_all_nearest(kk, D)
            assert e.metrics()["pairs"] == total
            want = e.query_vs_ref_nearest(ids, ids, kk, D, exclude_self=True)
            _check(got, want, (kk, D))
        pos = e.all_vs_all_nearest(4, 1.0)[0]
        for x in dup:
            assert list(pos[x]) == [y for y in dup if y != x][:4], x


def test_ex_both_directions():
    seqs = _seqs(12, LENS)
    n = len(seqs)
    with _engine(seqs, 21) as e:
        cases = [([4, 4, 9, 0, 23, 4], [1, 4, 4, 7, 1, 9, 23, 23, 0], False),  # duplicate ids on both sides
                 ([2, 2, 5], [2, 2, 5, 5], True),
                 (list(range(0, 35)), list(range(3, n)), False),
                 ([5, 30, 7], list(range(n)), True)]  # fewer than 32 query rows: the join puts r on the table
        for q, r, excl in cases:
            gi, gd = e.query_vs_ref(q, r)
            for kk in (1, 5, 256):
                for D in _thresholds(gd.ravel()):
                    qs, rs = e.query_vs_ref_nearest_ex(q, r, kk, D, exclude_self=excl)
                    _check(qs, e.query_vs_ref_nearest(q, r, kk, D, exclude_self=excl), (q, kk, D))
                    _check(rs, e.query_vs_ref_nearest(r, q, kk, D, exclude_self=excl), (q, kk, D))
                    _check(rs, _nearest_ref(gi.T.copy(), gd.T.copy(), r, q, kk, D, excl), (q, kk, D))
        qs, rs = e.query_vs_ref_nearest_ex([1, 2], [], 3, 1.0)
        assert (qs[0] == 0xFFFFFFFF).all() and (qs[2] == -1.0).all() and (qs[3] == 0).all() and rs[0].shape == (0, 3)


def test_ex_reference_side_accumulates_over_launches():
    """2^19 references (repeated ids of small records): a launch holds 128 query rows, so 260 rows take three and every
    reference's list is built across them"""
    seqs = _seqs(3, [300 + 7 * i for i in range(48)], families=4)
    n = len(seqs)
    rng = np.random.default_rng(5)
    r = rng.permutation(np.tile(np.arange(n, dtype=np.uint32), (1 << 19) // n + 1)[: 1 << 19]).astype(np.uint32)
    q = rng.integers(0, n, 260).astype(np.uint32)
    with _engine(seqs, 21) as e:
        for kk, D, excl in ((1, 1.0, False), (16, 0.6, True)):
            qs, rs = e.query_vs_ref_nearest_ex(q, r, kk, D, exclude_self=excl)
            _check(qs, e.query_vs_ref_nearest(q, r, kk, D, exclude_self=excl), kk)
            _check(rs, e.query_vs_ref_nearest(r, q, kk, D, exclude_self=excl), kk)


def test_literal_ambiguous_context():
    """GKD_AMBIG_LITERAL with runs of N: kernel 5 adds the shared literal k-mers, counted on the host, and the lists
    are kept on the device"""
    rng = np.random.default_rng(9)
    seqs = []
    for s in _seqs(40, [60_000] * 12):
        a = np.frombuffer(s, dtype=np.uint8).copy()
        for _ in range(4):
            p = int(rng.integers(0, a.size - 40))
            a[p:p + int(rng.integers(1, 30))] = ord("n")
        seqs.append(a.tobytes())
    seqs[7] = seqs[2]
    n = len(seqs)
    ids = list(range(n))
    with _engine(seqs, 21, ambig_policy=gkd.AMBIG_LITERAL) as e:
        gi, gd = e.all_vs_all()
        I, Dm = _symmetric(n, np.asarray(gi), np.asarray(gd))
        q, r = [0, 3, 3, 11], ids
        for D in _thresholds(np.asarray(gd)):
            for kk in (1, 4, 256):
                _check(e.all_vs_all_nearest(kk, D), _nearest_ref(I, Dm, ids, ids, kk, D, True), (kk, D))
                qs, rs = e.query_vs_ref_nearest_ex(q, r, kk, D, exclude_self=True)
                _check(qs, _nearest_ref(I[q], Dm[q], q, r, kk, D, True), (kk, D))
                _check(rs, _nearest_ref(I[:, q], Dm[:, q], r, q, kk, D, True), (kk, D))


def test_group_equals_single_context():
    """Copies of one genome on every member of a 4-member group (ids 3, 6, 9, 12): member 2's ring call spans member 3
    and the second half of member 0, so its columns are not in ascending global id and ties must still go to the
    smaller id"""
    import torch

    seqs = _seqs(21, [150_000] * 9 + [0, 40_000, 220_000, 100_000])
    for i in (6, 9, 12):
        seqs[i] = seqs[3]
    n = len(seqs)
    with _engine(seqs, 20) as e:
        gi, gd = e.all_vs_all()
        want = {(kk, D): e.all_vs_all_nearest(kk, D) for kk in (1, 2, 3, 256) for D in _thresholds(np.asarray(gd))}
    assert list(want[(1, 1.0)][0][9]) == [3]
    ndev = torch.cuda.device_count()
    for members in (2, 3, 4):
        devices = [m % ndev for m in range(members)]
        with gkd.Group(devices, k=20, workspace_bytes=4 << 20, panel=2) as g:
            per = (n + members - 1) // members
            for i, s in enumerate(seqs):
                assert g.add(min(i // per, members - 1), s) == i
            g.build()
            for key, w in want.items():
                got = g.all_vs_all_nearest(*key)
                for x, y in zip(got, w):
                    assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), (members, key)


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


def test_cli_fastadist_nearest_is_the_full_report_ranked(tmp_path):
    seqs = _seqs(61, [30_000] * 14 + [5_000, 200])
    seqs[9] = seqs[2]
    seqs[13] = seqs[2]
    fa = tmp_path / "in.fa"
    _fasta(fa, seqs)
    full = _run(["fastaDist", "-i", str(fa)]).split("\n")
    rows = [ln.split("\t") for ln in full[1:] if ln]
    index = {}
    for r in rows:
        index.setdefault(r[0], (len(index), r[1]))
        index.setdefault(r[2], (len(index), r[3]))
    labels = sorted(index, key=lambda x: index[x][0])
    dists = sorted(set(float(r[4]) for r in rows))
    for N, D in ((1, None), (3, None), (2, dists[len(dists) // 3]), (256, 0.5)):
        want = [full[0]]
        for me in labels:
            mine = [(r[2], r[4]) if r[0] == me else (r[0], r[4]) for r in rows if me in (r[0], r[2])]
            mine = [x for x in mine if D is None or float(x[1]) <= D]
            mine.sort(key=lambda x: (float(x[1]), index[x[0]][0]))
            want += ["\t".join([me, index[me][1], o, index[o][1], d]) for o, d in mine[:N]]
        want = "\n".join(want) + "\n"
        args = ["fastaDist", "-i", str(fa), "--nearest", str(N)] + ([] if D is None else ["--maxDist", repr(D)])
        assert _run(args) == want, (N, D)
        assert _run(args + ["--devices", "0,0"]) == want, (N, D)
