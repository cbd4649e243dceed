"""Selections on the device (csrc/intersect.cu k_select_within / k_select_nearest): only the chosen pairs leave the
GPU, and each one must be exactly the dense call's entry.

* within:  (a, b, inter, dist) = the dense all_vs_all_range / query_vs_ref entries with dist <= D, bit-exact and in
           enumeration order, under both kernel-4 forms, for K = 21, 16 (palindrome sub-sets), 25 (64-bit keys) and
           protein 8, at D = 1.0, at an attained distance (the comparison is inclusive) and below every distance;
* nearest: each query row = a stable sort of the dense row by (distance, position in r), filtered and cut to k.

Join-overflow redo: a block-join table is flagged (and the chunk redone by the merge kernel) when the rows of one key
range fill more than 62.5 % of its slots.  With uniform keys that does not happen: GKD_JOIN_FILL is clamped to 45 % and
every row's range count keeps its expected share under that target (the 45 % fill is covered below).  Coarse set
tables and skewed imported key sets do overflow; tests/test_gpu_join_redo.py forces the redo that way and checks that
the within and nearest selections of a redone chunk are copied and counted once (run_pairs and the Within /
Nearest forms in gkd_api.cu).
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import genome.distance_b200 as gkd

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")


def _seqs(seed, lens, protein=False, families=3):
    """related families (members mutated at 0, 0.2, 3 and 15 %) next to unrelated ones, so thresholds fall on both
    sides of real distances"""
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


def _check_hits(got, want_a, want_b, gi, gd, D):
    a, b, i, d = got
    keep = gd <= D
    assert np.array_equal(a, want_a[keep]) and np.array_equal(b, want_b[keep]), D
    assert np.array_equal(i, gi[keep]), D
    assert np.array_equal(d.view(np.uint64), gd[keep].view(np.uint64)), D  # bit-exact


LENS = [200_000] * 20 + [250_000, 90_000, 25, 0, 600_000, 9_000, 300_000] + [180_000] * 13


@pytest.mark.parametrize("algo", ["merge", "join"])
@pytest.mark.parametrize("k,alphabet", [(21, gkd.DNA), (16, gkd.DNA), (25, gkd.DNA), (8, gkd.PROT)])
def test_within_equals_dense_filtered(monkeypatch, algo, k, alphabet):
    monkeypatch.setenv("GKD_ISECT_ALGO", algo)
    prot = alphabet == gkd.PROT
    seqs = _seqs(31, [max(n // 4, 8) if n else 0 for n in LENS] if prot else LENS, protein=prot)
    n = len(seqs)
    total = n * (n - 1) // 2
    iu_a, iu_b = (x.astype(np.uint32) for x in np.triu_indices(n, 1))
    with _engine(seqs, k, alphabet) as e:
        # the whole triangle and ranges that start and end inside rows
        for first, count in ((0, total), (37, 511), (total - 400, 400), (0, 60)):
            gi, gd = e.all_vs_all_range(n, first, count)
            gi, gd = np.asarray(gi), np.asarray(gd)
            for D in _thresholds(gd):
                got = e.all_vs_all_range_within(n, first, count, D)
                _check_hits(got, iu_a[first:first + count], iu_b[first:first + count], gi, gd, D)
                if algo == "join" and count == total:
                    assert e.metrics()["intersect_kernel"] == 5
        # rectangles with many and few query rows (the join puts the longer side on the table below 32 rows)
        for q, r in ((list(range(0, 30)), list(range(5, n))), ([5, 30, 7], list(range(n))), ([3, 3, 0], [9, 3, 3, 39])):
            gi, gd = e.query_vs_ref(q, r)
            gi, gd = gi.ravel(), gd.ravel()
            pa = np.repeat(np.arange(len(q), dtype=np.uint32), len(r))
            pb = np.tile(np.arange(len(r), dtype=np.uint32), len(q))
            for D in _thresholds(gd):
                _check_hits(e.query_vs_ref_within(q, r, D), pa, pb, gi, gd, D)


def test_within_at_the_largest_join_fill(monkeypatch):
    monkeypatch.setenv("GKD_ISECT_ALGO", "join")
    monkeypatch.setenv("GKD_JOIN_FILL", "45")
    seqs = _seqs(5, [200_000] * 34 + [1_500_000, 30_000, 2_000, 800_000], families=2)
    n = len(seqs)
    iu_a, iu_b = (x.astype(np.uint32) for x in np.triu_indices(n, 1))
    with _engine(seqs, 21) as e:
        gi, gd = e.all_vs_all()
        for D in _thresholds(gd):
            _check_hits(e.all_vs_all_within(D), iu_a, iu_b, gi, gd, D)
        assert e.metrics()["intersect_kernel"] == 5


def test_within_crosses_chunk_boundaries_and_caps():
    """~12,000 gene-sized records: 7.2e7 pairs, more than one 64 Mi-pair launch.  Then cap < n: the first cap hits
    are the prefix and n is still the full total."""
    n = 12_000
    seqs = _seqs(77, [900 + (i * 37) % 400 for i in range(n)], families=40)
    total = n * (n - 1) // 2
    assert total > 64 << 20
    with _engine(seqs, 21) as e:
        D = 0.5
        a, b, i, d = e.all_vs_all_within(D)
        gi, gd = e.all_vs_all()
        gd = np.asarray(gd)
        keep = np.flatnonzero(gd <= D)
        assert 0 < keep.size < total
        assert keep[-1] >= 64 << 20, "no hit after the first chunk"
        # pair index -> (i, j) of the row-major triangle
        row_start = np.cumsum(np.r_[0, np.arange(n - 1, 0, -1, dtype=np.int64)])
        ra = (np.searchsorted(row_start, keep, side="right") - 1).astype(np.uint32)
        rb = (keep - row_start[ra] + ra + 1).astype(np.uint32)
        assert np.array_equal(a, ra) and np.array_equal(b, rb)
        assert np.array_equal(i, np.asarray(gi)[keep]) and np.array_equal(d.view(np.uint64), gd[keep].view(np.uint64))
        del gi, gd
        L = e._L
        for cap in (0, 1000, keep.size - 1):
            ha, hb = np.empty(cap, dtype=np.uint32), np.empty(cap, dtype=np.uint32)
            hi, hd = np.empty(cap, dtype=np.uint64), np.empty(cap, dtype=np.float64)
            h = gkd._lib.GkdHits(ha.ctypes.data, hb.ctypes.data, hi.ctypes.data, hd.ctypes.data, cap, 0)
            e._ck(L.gkd_all_vs_all_range_within(e._h, n, 0, total, D, C.byref(h)))
            assert h.n == keep.size
            assert np.array_equal(ha, a[:cap]) and np.array_equal(hb, b[:cap]) and np.array_equal(hi, i[:cap])
            assert np.array_equal(hd.view(np.uint64), d[:cap].view(np.uint64))
        m = e.metrics()
        assert m["pairs"] == total and m["epilogue_ms"] > 0


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


def _check_nearest(got, want):
    for g, w in zip(got, want):
        assert g.shape == w.shape
        if g.dtype == np.float64:
            assert np.array_equal(g.view(np.uint64), w.view(np.uint64))
        else:
            assert np.array_equal(g, w)


@pytest.mark.parametrize("algo", ["merge", "join"])
def test_nearest_equals_stable_sort_of_dense_rows(monkeypatch, algo):
    monkeypatch.setenv("GKD_ISECT_ALGO", algo)
    seqs = _seqs(12, LENS)
    n = len(seqs)
    with _engine(seqs, 21) as e:
        cases = [(list(range(n)), list(range(n)), True),              # each set's neighbours
                 (list(range(0, 35)), list(range(3, n)), False),
                 ([4, 4, 9, 0, 23, 4], [1, 4, 4, 7, 1, 9, 23, 23, 0], False),  # duplicate ids on both sides
                 ([2, 2, 5], [2, 2, 5, 5], True)]
        for q, r, excl in cases:
            gi, gd = e.query_vs_ref(q, r)
            for k in (1, 5, 256):
                for D in _thresholds(gd.ravel()):
                    got = e.query_vs_ref_nearest(q, r, k, D, exclude_self=excl)
                    _check_nearest(got, _nearest_ref(gi, gd, q, r, k, D, excl))
        # no reference at all: every slot is unused
        pos, inter, dist, found = e.query_vs_ref_nearest([1, 2], [], 3, 1.0)
        assert (pos == 0xFFFFFFFF).all() and (inter == 0).all() and (dist == -1.0).all() and (found == 0).all()


def test_nearest_over_several_launches():
    """2^19 references (repeated ids of small records): a launch holds 128 query rows, so 260 rows take three"""
    seqs = _seqs(3, [300 + 7 * i for i in range(48)], families=4)
    n = len(seqs)
    r = np.tile(np.arange(n, dtype=np.uint32), (1 << 19) // n + 1)[: 1 << 19]
    rng = np.random.default_rng(5)
    r = rng.permutation(r).astype(np.uint32)
    q = rng.integers(0, n, 260).astype(np.uint32)
    with _engine(seqs, 21) as e:
        for k, D in ((1, 1.0), (16, 0.6)):
            got = e.query_vs_ref_nearest(q, r, k, D)
            for x0 in range(0, len(q), 40):  # the dense rows in blocks, to bound host memory
                gi, gd = e.query_vs_ref(q[x0:x0 + 40], r)
                want = _nearest_ref(gi, gd, q[x0:x0 + 40], r, k, D, False)
                _check_nearest([g[x0:x0 + 40] for g in got], want)


def test_literal_ambiguous_context():
    """GKD_AMBIG_LITERAL with runs of N: kernel 5 adds the shared literal k-mers, counted on the host, and selects on
    the device"""
    rng = np.random.default_rng(9)
    seqs = []
    for s in _seqs(40, [60_000] * 12):
        a = np.frombuffer(s, dtype=np.uint8).copy()
        for _ in range(4):
            p = int(rng.integers(0, a.size - 40))
            a[p:p + int(rng.integers(1, 30))] = ord("n")
        seqs.append(a.tobytes())
    n = len(seqs)
    iu_a, iu_b = (x.astype(np.uint32) for x in np.triu_indices(n, 1))
    with _engine(seqs, 21, ambig_policy=gkd.AMBIG_LITERAL) as e:
        gi, gd = e.all_vs_all()
        for D in _thresholds(gd):
            _check_hits(e.all_vs_all_within(D), iu_a, iu_b, gi, gd, D)
        q, r = [0, 3, 3, 11], list(range(n))
        qi, qd = e.query_vs_ref(q, r)
        pa = np.repeat(np.arange(len(q), dtype=np.uint32), n)
        pb = np.tile(np.arange(n, dtype=np.uint32), len(q))
        for D in _thresholds(qd.ravel()):
            _check_hits(e.query_vs_ref_within(q, r, D), pa, pb, qi.ravel(), qd.ravel(), D)
            for k in (1, 4):
                _check_nearest(e.query_vs_ref_nearest(q, r, k, D, exclude_self=True),
                               _nearest_ref(qi, qd, q, r, k, D, True))


def test_group_within_equals_single_context():
    import torch

    seqs = _seqs(21, [150_000] * 9 + [0, 40_000, 220_000, 100_000])
    n = len(seqs)
    with _engine(seqs, 20) as e:
        gi, gd = e.all_vs_all()
        want = {D: e.all_vs_all_within(D) for D in _thresholds(gd)}
    ndev = torch.cuda.device_count()
    for members in (2, 3, 4):
        devices = [m % ndev for m in range(members)]
        with gkd.Group(devices, k=20, workspace_bytes=4 << 20, panel=2) as g:
            per = (n + members - 1) // members
            for i, s in enumerate(seqs):
                assert g.add(min(i // per, members - 1), s) == i
            g.build()
            for D, w in want.items():
                got = g.all_vs_all_within(D)
                for x, y in zip(got, w):
                    assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), (members, D)


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


def test_cli_fastadist_maxdist_is_the_full_report_filtered(tmp_path):
    fa = tmp_path / "in.fa"
    _fasta(fa, _seqs(61, [30_000] * 14 + [5_000, 200]))
    full = _run(["fastaDist", "-i", str(fa)]).split("\n")
    dists = sorted(set(float(ln.rsplit("\t", 1)[1]) for ln in full[1:] if ln))
    for D in (1.0, dists[len(dists) // 3], 0.05):
        want = [full[0]] + [ln for ln in full[1:] if ln and float(ln.rsplit("\t", 1)[1]) <= D]
        want = "\n".join(want) + "\n"
        assert _run(["fastaDist", "-i", str(fa), "--maxDist", repr(D)]) == want, D
        assert _run(["fastaDist", "-i", str(fa), "--maxDist", repr(D), "--devices", "0,0"]) == want, D


def test_cli_genomes_nearest_is_the_dense_matrix_ranked(tmp_path):
    seqs = _seqs(62, [20_000] * 9)
    bdir, qdir = tmp_path / "base", tmp_path / "query"
    bdir.mkdir()
    qdir.mkdir()
    for i, s in enumerate(seqs[:6]):
        (bdir / ("b%d.fa" % i)).write_text(">c\n" + s.decode() + "\n")
    for i, s in enumerate(seqs[6:] + seqs[:2]):
        (qdir / ("q%d.fa" % i)).write_text(">c\n" + s.decode() + "\n")
    full = _run(["genomes", "-t", "FASTA", str(bdir), str(qdir)]).split("\n")
    rows = [ln.split("\t") for ln in full[1:] if ln]
    base = sorted("b%d" % i for i in range(6))
    for N, m in ((1, "1.0"), (3, "0.9"), (256, "0.5")):
        want = [full[0]]
        for qid in sorted(set(r[0] for r in rows)):
            mine = [r for r in rows if r[0] == qid and float(r[2]) <= float(m)]
            mine.sort(key=lambda r: (float(r[2]), base.index(r[1])))
            want += ["\t".join(r) for r in mine[:N]]
        got = _run(["genomes", "-t", "FASTA", "-m", m, "--nearest", str(N), str(bdir), str(qdir)])
        assert got == "\n".join(want) + "\n", (N, m)
