"""Complete- and average-linkage hierarchies on the device (csrc/agglomerate.cu): the distances stay in an n x n matrix in
HBM and reciprocal nearest neighbours merge in parallel rounds; only the merges leave the device.

The oracle is oracle/agglomerate.py's exact sequential agglomeration of the dense result.  (a, b, height, size) must be
equal arrays on every path: both kernel-4 forms, chunks, the forced block-join redo, the literal and canonical contexts,
the caller's triangle (host or device), groups and the command line.
"""
import ctypes as C
import os
import sys
from fractions import Fraction

import numpy as np
import pytest

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib
from oracle import agglomerate as agg

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_gpu_clusters as tc  # noqa: E402  (inputs, engine, CLI helpers)
import test_gpu_join_redo as jr  # noqa: E402  (the overflow recipes)

pytestmark = pytest.mark.gpu

METHODS = (gkd.LINK_COMPLETE, gkd.LINK_AVERAGE)
NAMES = {gkd.LINK_COMPLETE: "complete", gkd.LINK_AVERAGE: "average"}


def _arrays(merges):
    return (np.array([m[0] for m in merges], dtype=np.uint32), np.array([m[1] for m in merges], dtype=np.uint32),
            np.array([m[2] for m in merges], dtype=np.float64), np.array([m[3] for m in merges], dtype=np.uint32))


class Oracle:
    """the whole agglomeration of the first m sets of the triangle gd over n, once; any threshold is a prefix of it"""

    def __init__(self, n, gd, method, m=None):
        gd = np.asarray(gd)
        if m is not None:
            i, j = np.triu_indices(n, 1)
            gd, n = gd[(i < m) & (j < m)], m
        self.values = []
        self.merges = agg.sequential(gd, n, method, 2.0, self.values)

    def __call__(self, D):
        return _arrays(agg.prefix(self.merges, self.values, D))


def _eq(got, want, what=None):
    assert len(got) == 4 and got[0].dtype == np.uint32 and got[3].dtype == np.uint32, what
    for g, w in zip(got, want):
        assert g.shape == w.shape, what
        assert np.array_equal(g.view(np.uint64) if g.dtype == np.float64 else g,
                              w.view(np.uint64) if w.dtype == np.float64 else w), what


def _square(n, gd):
    full = np.zeros((n, n))
    i, j = np.triu_indices(n, 1)
    full[i, j] = full[j, i] = gd
    return full


def _properties(full, got, method, cuts):
    """each height against the dense matrix, complete-linkage diameters at the cuts, and the cluster counts"""
    n = full.shape[0]
    a, b, h, size = got
    members = {x: [x] for x in range(n)}
    w = np.round(full * 2.0 ** 53).astype(np.uint64)
    for t in range(a.size):
        A, B = members[int(a[t])], members.pop(int(b[t]))
        blk = w[np.ix_(A, B)]
        if method == gkd.LINK_COMPLETE:
            assert h[t] == full[np.ix_(A, B)].max(), t
        else:  # exact sum of the 2^-53 words, split so that uint64 sums cannot wrap
            s = (int((blk >> np.uint64(32)).sum()) << 32) + int((blk & np.uint64(0xFFFFFFFF)).sum())
            assert h[t] == float(Fraction(s, len(A) * len(B) << 53)), t
        assert size[t] == len(A) + len(B)
        members[int(a[t])] = A + B
    if method != gkd.LINK_COMPLETE:
        return
    for D in cuts:  # complete heights are the exact values: the clusters at D have diameter <= D
        keep = h <= D
        lab = agg.labels(list(zip(a[keep], b[keep], h[keep], size[keep])), n)
        assert len(set(lab)) == n - int(keep.sum())
        for c in set(lab):
            idx = [x for x in range(n) if lab[x] == c]
            assert full[np.ix_(idx, idx)].max() <= D


def _cuts(gd):
    return [t for t in tc._thresholds(gd) if t >= 0]


def _check_call(e, n, gd, method, want_full, D):
    got = e.all_vs_all_agglomerate(method, D)
    _eq(got, want_full(D), (NAMES[method], D))
    return got


@pytest.mark.parametrize("algo", ["merge", "join"])
@pytest.mark.parametrize("k,alphabet", [(21, gkd.DNA), (16, gkd.DNA), (25, gkd.DNA), (8, gkd.PROT)])
def test_forms_and_alphabets(monkeypatch, algo, k, alphabet):
    import torch

    monkeypatch.setenv("GKD_ISECT_ALGO", algo)
    prot = alphabet == gkd.PROT
    seqs = tc._seqs(31, [max(n // 4, 8) if n else 0 for n in tc.LENS] if prot else tc.LENS, protein=prot)
    seqs[33] = seqs[36] = seqs[5]
    n = len(seqs)
    with tc._engine(seqs, k, alphabet) as e:
        _, gd = e.all_vs_all(want_inter=False)
        full = _square(n, gd)
        for method in METHODS:
            want = Oracle(n, gd, method)
            sizes = set()
            for D in tc._thresholds(gd):
                got = _check_call(e, n, gd, method, want, D)
                if algo == "join":
                    assert e.metrics()["intersect_kernel"] == 5
                assert e.metrics()["pairs"] == n * (n - 1) // 2
                sizes.add(got[0].size)
                _eq(e.all_vs_all_agglomerate(method, D, n=17), Oracle(n, gd, method, m=17)(D), (17, D))
            assert {0, n - 1} <= sizes and len(sizes) > 2
            whole = e.all_vs_all_agglomerate(method, 1.0)
            _properties(full, whole, method, _cuts(gd))
            # the caller's triangle, from the host and from the device, is read and left as it was
            host = gd.copy()
            _eq(e.agglomerate(host, method, 1.0), whole)
            assert np.array_equal(host, gd)
            dev = torch.from_numpy(gd).to("cuda:0")
            _eq(e.agglomerate(dev, method, 1.0), whole)
            assert np.array_equal(dev.cpu().numpy(), gd)
            for m in (0, 1):
                assert all(x.size == 0 for x in e.all_vs_all_agglomerate(method, 1.0, n=m))
            got = e.all_vs_all_agglomerate(method, 1.0, n=2)
            assert got[0].tolist() == [0] and got[1].tolist() == [1] and got[2][0] == gd[0] and got[3].tolist() == [2]


def test_ties_and_chains():
    """a mutation chain (many rounds), unrelated records (ties at 1.0), an empty one, one shorter than K and identical
    copies (ties at 0.0)"""
    rng = np.random.default_rng(8)
    chain = [tc._random(rng, 30_000)]
    for _ in range(9):
        chain.append(tc._mutate(rng, chain[-1], 0.012))
    seqs = chain + [tc._random(rng, 30_000) for _ in range(6)] + [b"", b"acgtacgtac", chain[2], chain[2], chain[7]]
    n = len(seqs)
    with tc._engine(seqs, 21) as e:
        _, gd = e.all_vs_all(want_inter=False)
        full = _square(n, gd)
        for method in METHODS:
            want = Oracle(n, gd, method)
            for D in tc._thresholds(gd) + [max(e.pair(i, i + 1)[2] for i in range(9))]:
                _check_call(e, n, gd, method, want, D)
            whole = e.all_vs_all_agglomerate(method, 1.0)
            assert e.metrics()["agglomerate_rounds"] >= 2
            _properties(full, whole, method, _cuts(gd))
            a, b, h, _ = e.all_vs_all_agglomerate(method, 0.0)
            assert list(zip(a, b)) == [(2, 18), (2, 19), (7, 20)] and not h.any()


def test_arguments_cap_and_device_outputs():
    import torch

    seqs = tc._seqs(5, [40_000] * 24)
    seqs[20] = seqs[3]
    n = len(seqs)
    with tc._engine(seqs, 21) as e:
        want = e.all_vs_all_agglomerate(gkd.LINK_AVERAGE, 0.9)
        w = want[0].size
        assert w > 4

        def raw(cap, arrays, method=gkd.LINK_AVERAGE, D=0.9, nn=n):
            ptr = [None if x is None else (x.data_ptr() if torch.is_tensor(x) else x.ctypes.data) for x in arrays]
            m = _lib.GkdMerges(*ptr, cap, 0)
            rc = e._L.gkd_all_vs_all_agglomerate(e._h, nn, method, D, C.byref(m))
            return rc, m.n

        dts = (np.uint32, np.uint32, np.float64, np.uint32)
        for cap in (0, 1, w - 1):
            out = [np.full(w, 7, dtype=dt) for dt in dts]
            assert raw(cap, out) == (0, w)
            for o, x in zip(out, want):
                assert np.array_equal(o[:cap], x[:cap]) and (o[cap:] == 7).all(), cap
        assert raw(0, [None] * 4) == (0, w)
        dev = [torch.zeros(w, dtype=t, device="cuda:0") for t in (torch.int32, torch.int32, torch.float64, torch.int32)]
        assert raw(w, dev) == (0, w)
        _eq([dev[0].cpu().numpy().view(np.uint32), dev[1].cpu().numpy().view(np.uint32), dev[2].cpu().numpy(),
             dev[3].cpu().numpy().view(np.uint32)], want)
        for bad in ((float("nan"), gkd.LINK_AVERAGE, n), (0.5, 0, n), (0.5, 7, n), (0.5, gkd.LINK_COMPLETE, n + 1)):
            D, method, nn = bad
            assert raw(4, [None] * 4, method, D, nn)[0] == _lib.GKD_EINVAL, bad
        assert e._L.gkd_all_vs_all_agglomerate(e._h, n, gkd.LINK_COMPLETE, 0.5, None) == _lib.GKD_EINVAL
        assert all(x.size == 0 for x in e.all_vs_all_agglomerate(gkd.LINK_COMPLETE, -0.5))
        # a triangle off the 2^-53 grid is refused
        with pytest.raises(gkd.GkdError, match="2\\^-53"):
            e.agglomerate(np.array([0.1, 0.5, 0.25]), gkd.LINK_COMPLETE, 1.0)
        with pytest.raises(gkd.GkdError, match="2\\^-53"):
            e.agglomerate(np.array([0.5, 2.5, 0.25]), gkd.LINK_AVERAGE, 1.0)


def test_more_than_one_chunk():
    """~12,000 gene-sized records: two 64 Mi-pair chunks.  The call equals gkd_agglomerate on the dense triangle."""
    import torch

    n = 12_000
    seqs = tc._seqs(77, [900 + (i * 37) % 400 for i in range(n)], families=40)
    seqs[40] = seqs[11_999] = seqs[5]
    total = n * (n - 1) // 2
    with tc._engine(seqs, 21) as e:
        _, gd = e.all_vs_all(want_inter=False)
        dev = torch.from_numpy(gd).to("cuda:0")
        for method in METHODS:
            before = e.metrics()["intersect_launches"]
            got = e.all_vs_all_agglomerate(method, 1.0)
            m = e.metrics()
            assert m["pairs"] == total and m["intersect_launches"] - before == 2
            assert got[0].size == n - 1
            _eq(got, e.agglomerate(gd, method, 1.0))
            _eq(got, e.agglomerate(dev, method, 1.0))
            assert (got[2][1:] >= got[2][:-1]).all()
            assert (5, 40) in set(zip(got[0].tolist(), got[1].tolist()))
            below = float(np.unique(gd[gd < 1.0])[100])
            cut = e.all_vs_all_agglomerate(method, below)
            _eq(cut, tuple(x[:cut[0].size] for x in got))
            # properties on the small clusters (every merge of two clusters of at most 8 records)
            small = set(np.flatnonzero(got[3] <= 8).tolist())
            members = {}
            for t in range(got[0].size):
                A = members.get(int(got[0][t]), [int(got[0][t])])
                B = members.pop(int(got[1][t]), [int(got[1][t])])
                if t in small:
                    i, j = np.meshgrid(A, B, indexing="ij")
                    lo, hi = np.minimum(i, j).ravel(), np.maximum(i, j).ravel()
                    d = gd[lo * (2 * n - lo - 1) // 2 + hi - lo - 1]
                    if method == gkd.LINK_COMPLETE:
                        assert got[2][t] == d.max()
                    else:
                        s = sum(int(x) for x in np.round(d * 2.0 ** 53).astype(np.uint64))
                        assert got[2][t] == float(Fraction(s, len(A) * len(B) << 53))
                members[int(got[0][t])] = A + B


# ---- the forced block-join redo (recipes of test_gpu_join_redo.py) ------------------------------------------------
def test_redo_coarse_tables(monkeypatch):
    k = 25
    seqs = jr._recipe_a(k, gkd.DNA)
    with jr._engine(monkeypatch, "merge", seqs, k, coarse=True) as m, \
            jr._engine(monkeypatch, "join", seqs, k, coarse=True) as e:
        _, gd = m.all_vs_all()
        for method in METHODS:
            want = Oracle(len(seqs), gd, method)
            for D in tc._thresholds(gd):
                got = jr._redone(e, lambda: e.all_vs_all_agglomerate(method, D), k)
                _eq(got, want(D), D)
                _eq(got, m.all_vs_all_agglomerate(method, D), D)


def test_redo_skewed_imports(monkeypatch):
    k = 21
    sets = jr._mixed(k)
    with jr._engine(monkeypatch, "merge", k=k, keysets=sets) as m, jr._engine(monkeypatch, "join", k=k, keysets=sets) as e:
        _, gd = m.all_vs_all()
        for method in METHODS:
            want = Oracle(len(sets), gd, method)
            for D in tc._thresholds(gd):
                _eq(jr._redone(e, lambda: e.all_vs_all_agglomerate(method, D), k), want(D), D)


def test_redo_only_in_the_second_chunk(monkeypatch):
    """12,000 imported sets whose rows from 9,000 on are crafted: only the second chunk overflows (join, join, merge
    redo); the discarded attempt must write nothing the redo does not rewrite"""
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
        want = {meth: m.all_vs_all_agglomerate(meth, 0.5) for meth in METHODS}
    with jr._engine(monkeypatch, "join", k=k, keysets=sets) as e:
        for meth in METHODS:
            assert 0 < want[meth][0].size < n - 1
            _eq(jr._redone(e, lambda: e.all_vs_all_agglomerate(meth, 0.5), k, launches=3), want[meth], meth)


# ---- other contexts ---------------------------------------------------------------------------------------------
def test_literal_and_canonical_contexts():
    rng = np.random.default_rng(9)
    seqs = []
    for i, s in enumerate(tc._seqs(40, [60_000] * 12)):
        a = np.frombuffer(s, dtype=np.uint8).copy()
        if i not in (1, 5, 9):
            for _ in range(4):
                p = int(rng.integers(0, a.size - 40))
                a[p:p + int(rng.integers(1, 30))] = ord("n")
        seqs.append(a.tobytes())
    seqs[7] = seqs[10] = seqs[2]
    n = len(seqs)
    for kw in ({"ambig_policy": gkd.AMBIG_LITERAL}, {"strand_mode": gkd.STRAND_CANONICAL}):
        with tc._engine(seqs, 20, **kw) as e:
            _, gd = e.all_vs_all(want_inter=False)
            for method in METHODS:
                want = Oracle(n, gd, method)
                for D in tc._thresholds(gd):
                    _check_call(e, n, gd, method, want, D)
                if "ambig_policy" in kw:  # host outputs only
                    import torch

                    dev = torch.zeros(n, dtype=torch.int32, device="cuda:0")
                    m = _lib.GkdMerges(dev.data_ptr(), None, None, None, n, 0)
                    assert e._L.gkd_all_vs_all_agglomerate(e._h, n, method, 1.0, C.byref(m)) == _lib.GKD_EINVAL


def test_group_equals_single_context():
    import torch

    seqs = tc._seqs(21, [150_000] * 9 + [0, 40_000, 220_000, 100_000, 60_000, 80_000, 30_000])
    rng = np.random.default_rng(4)
    seqs[1] = seqs[14] = tc._random(rng, 120_000)
    for i in (8, 9, 13):
        seqs[i] = seqs[3]
    n = len(seqs)
    with tc._engine(seqs, 20) as e:
        _, gd = e.all_vs_all(want_inter=False)
        want = {(m, D): e.all_vs_all_agglomerate(m, D) for m in METHODS for D in tc._thresholds(gd)}
    for (m, D), w in want.items():
        _eq(w, Oracle(n, gd, m)(D), (m, D))
    ndev = torch.cuda.device_count()
    for members in (2, 3, 4):
        devices = [x % ndev for x in range(members)]
        with gkd.Group(devices, k=20, workspace_bytes=4 << 20, panel=2) as g:
            per = (n + members - 1) // members
            for i, s in enumerate(seqs):
                assert g.add(min(i // per, members - 1), s) == i
            g.build()
            for (m, D), w in want.items():
                _eq(g.all_vs_all_agglomerate(m, D), w, (members, m, D))


def test_cli_fastadist_method(tmp_path):
    import torch

    rng = np.random.default_rng(6)
    seqs = tc._seqs(61, [30_000] * 14 + [5_000, 200])
    seqs[9] = seqs[2]
    seqs[3] = seqs[15] = tc._random(rng, 8_000)
    fa = tmp_path / "in.fa"
    tc._fasta(fa, seqs)
    n = len(seqs)
    with tc._engine(seqs, 21) as e:
        _, gd = e.all_vs_all(want_inter=False)
    labels = ["r%04d" % i for i in range(n)]  # as tc._fasta writes them
    comments = ["rec %d" % i for i in range(n)]
    group = ["--gpus", "2"] if torch.cuda.device_count() >= 2 else ["--devices", "0,0"]
    dists = sorted(set(float(x) for x in gd[gd < 1.0]))
    base = ["fastaDist", "-i", str(fa)]
    for method in METHODS:
        want_all = Oracle(n, gd, method)
        for D in (None, dists[len(dists) // 2], 0.5):
            a, b, h, _ = want_all(1.0 if D is None else D)
            want = "seq1\tname1\tseq2\tname2\tdistance\n" + "".join(
                f"{labels[x]}\t{comments[x]}\t{labels[y]}\t{comments[y]}\t{gkd.format_double(float(z))}\n"
                for x, y, z in zip(a, b, h))
            args = base + ["--linkage", "--method", NAMES[method]] + ([] if D is None else ["--maxDist", repr(D)])
            got = tc._run(args)
            assert got == want, (method, D)
            assert tc._run(args + group) == got, (method, D)
            if D is None:
                continue
            lab = agg.labels(list(zip(a, b, h, h)), n)
            want = "seq\tname\tcluster\n" + "".join(f"{labels[x]}\t{comments[x]}\t{labels[lab[x]]}\n" for x in range(n))
            args = base + ["--clusters", "--maxDist", repr(D), "--method", NAMES[method]]
            got = tc._run(args)
            assert got == want, (method, D)
            assert tc._run(args + group) == got, (method, D)
    for args in (["--linkage"], ["--linkage", "--maxDist", "0.5"], ["--clusters", "--maxDist", "0.5"]):
        assert tc._run(base + args + ["--method", "single"]) == tc._run(base + args), args
