"""Complete linkage from the pairs within a distance (gkd_*_complete_linkage): the pairs within max_dist are collected on
the device, sorted into one row per set, and merged by the rounds of csrc/agglomerate.cu; device memory grows with the
pairs instead of n^2.

(a, b, height, size) must be equal arrays, bit for bit, to the dense gkd_all_vs_all_agglomerate(GKD_LINK_COMPLETE) and
to oracle/agglomerate.py's sequential agglomeration: both kernel-4 forms, chunks, the forced block-join redo, literal and
canonical contexts, the caller's pair list (host or device), groups and the command line when the dense matrix does
not fit (GKD_AGG_MAX_BYTES caps it).
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_gpu_agglomerate as ta  # noqa: E402  (oracle and equality helpers)
import test_gpu_clusters as tc  # noqa: E402  (inputs, engine, CLI helpers)
import test_gpu_join_redo as jr  # noqa: E402  (the overflow recipes)

pytestmark = pytest.mark.gpu

COMPLETE = gkd.LINK_COMPLETE


def _attained(gd, count=6):
    """a spread of attained distances below 1.0 (each a tie threshold: the inclusive boundary)"""
    d = sorted(set(float(x) for x in np.asarray(gd) if x < 1.0))
    return [d[int(t)] for t in np.linspace(0, len(d) - 1, min(count, len(d)))] if d else []


def _same(e, D, n=None, want=None):
    """the sparse call equals the dense call (and want, when given), merges and rounds"""
    got = e.all_vs_all_complete_linkage(D, n)
    rounds = e.metrics()["agglomerate_rounds"]
    dense = e.all_vs_all_agglomerate(COMPLETE, D, n)
    ta._eq(got, dense, D)
    assert rounds == e.metrics()["agglomerate_rounds"], D
    if want is not None:
        ta._eq(got, want, D)
    return got


@pytest.mark.parametrize("algo", ["merge", "join"])
@pytest.mark.parametrize("k,alphabet", [(21, gkd.DNA), (16, gkd.DNA), (25, gkd.DNA), (8, gkd.PROT)])
def test_forms_and_alphabets(monkeypatch, algo, k, alphabet):
    monkeypatch.setenv("GKD_ISECT_ALGO", algo)
    prot = alphabet == gkd.PROT
    seqs = tc._seqs(31, [max(n // 4, 8) if n else 0 for n in tc.LENS] if prot else tc.LENS, protein=prot)
    seqs[33] = seqs[36] = seqs[5]
    n = len(seqs)
    with tc._engine(seqs, k, alphabet) as e:
        _, gd = e.all_vs_all(want_inter=False)
        want = ta.Oracle(n, gd, COMPLETE)
        sizes = set()
        for D in tc._thresholds(gd) + _attained(gd):
            got = _same(e, D, want=want(D))
            if algo == "join":
                assert e.metrics()["intersect_kernel"] == 5
            sizes.add(got[0].size)
            _same(e, D, n=17, want=ta.Oracle(n, gd, COMPLETE, m=17)(D))
        assert {0, n - 1} <= sizes and len(sizes) > 2
        e.all_vs_all_complete_linkage(1.0)
        m = e.metrics()
        assert m["pairs"] == n * (n - 1) // 2 and m["epilogue_ms"] > 0
        for small in (0, 1):
            assert all(x.size == 0 for x in e.all_vs_all_complete_linkage(1.0, n=small))


def test_identical_records_at_zero_and_one_family():
    """D = 0 merges exactly the identical copies; a family whose every pair is within D gives rows of degree n - 1"""
    rng = np.random.default_rng(12)
    base = tc._random(rng, 40_000)
    fam = [base] + [tc._mutate(rng, base, 0.001 * (1 + i % 5)) for i in range(70)]
    seqs = fam + [fam[3], fam[3], fam[40]]
    n = len(seqs)
    with tc._engine(seqs, 21) as e:
        _, gd = e.all_vs_all(want_inter=False)
        want = ta.Oracle(n, gd, COMPLETE)
        a, b, h, _ = _same(e, 0.0, want=want(0.0))
        assert list(zip(a, b)) == [(3, 71), (3, 72), (40, 73)] and not h.any()
        for D in (float(gd.max()), 0.5, 1.0) + tuple(_attained(gd, 4)):
            got = _same(e, D, want=want(D))
        assert got[0].size == n - 1 and e.metrics()["agglomerate_rounds"] >= 2


def test_cap_device_outputs_and_arguments():
    import torch

    seqs = tc._seqs(5, [40_000] * 24)
    seqs[20] = seqs[3]
    n = len(seqs)
    with tc._engine(seqs, 21) as e:
        want = e.all_vs_all_agglomerate(COMPLETE, 0.9)
        w = want[0].size
        assert w > 4

        def raw(cap, arrays, D=0.9, nn=n):
            ptr = [None if x is None else (x.data_ptr() if torch.is_tensor(x) else x.ctypes.data) for x in arrays]
            m = _lib.GkdMerges(*ptr, cap, 0)
            return e._L.gkd_all_vs_all_complete_linkage(e._h, nn, D, C.byref(m)), m.n

        dts = (np.uint32, np.uint32, np.float64, np.uint32)
        for cap in (0, 1, w - 1):
            out = [np.full(w, 7, dtype=dt) for dt in dts]
            assert raw(cap, out) == (0, w)
            for o, x in zip(out, want):
                assert np.array_equal(o[:cap], x[:cap]) and (o[cap:] == 7).all(), cap
        assert raw(0, [None] * 4) == (0, w)
        dev = [torch.zeros(w, dtype=t, device="cuda:0") for t in (torch.int32, torch.int32, torch.float64, torch.int32)]
        assert raw(w, dev) == (0, w)
        ta._eq([dev[0].cpu().numpy().view(np.uint32), dev[1].cpu().numpy().view(np.uint32), dev[2].cpu().numpy(),
                dev[3].cpu().numpy().view(np.uint32)], want)
        assert raw(4, [None] * 4, float("nan"))[0] == _lib.GKD_EINVAL
        assert raw(4, [None] * 4, 0.5, n + 1)[0] == _lib.GKD_EINVAL
        assert e._L.gkd_all_vs_all_complete_linkage(e._h, n, 0.5, None) == _lib.GKD_EINVAL
        assert all(x.size == 0 for x in e.all_vs_all_complete_linkage(-0.5))


def test_more_than_one_chunk():
    """~12,000 gene-sized records: two 64 Mi-pair chunks"""
    n = 12_000
    seqs = tc._seqs(77, [900 + (i * 37) % 400 for i in range(n)], families=40)
    seqs[40] = seqs[11_999] = seqs[5]
    with tc._engine(seqs, 21) as e:
        _, gd = e.all_vs_all(want_inter=False)
        below = sorted(set(float(x) for x in gd[gd < 1.0]))
        for D in (below[100], below[len(below) // 2], 1.0):
            before = e.metrics()["intersect_launches"]
            got = e.all_vs_all_complete_linkage(D)
            assert e.metrics()["intersect_launches"] - before == 2
            ta._eq(got, e.all_vs_all_agglomerate(COMPLETE, D), D)
        assert got[0].size == n - 1 and (5, 40) in set(zip(got[0].tolist(), got[1].tolist()))


# ---- the forced block-join redo (recipes of test_gpu_join_redo.py) ------------------------------------------------
def test_redo_coarse_tables(monkeypatch):
    k = 25
    seqs = jr._recipe_a(k, gkd.DNA)
    with jr._engine(monkeypatch, "merge", seqs, k, coarse=True) as m, \
            jr._engine(monkeypatch, "join", seqs, k, coarse=True) as e:
        _, gd = m.all_vs_all()
        want = ta.Oracle(len(seqs), gd, COMPLETE)
        for D in tc._thresholds(gd) + _attained(gd, 3):
            ta._eq(jr._redone(e, lambda: e.all_vs_all_complete_linkage(D), k), want(D), D)


def test_redo_skewed_imports(monkeypatch):
    k = 21
    sets = jr._mixed(k)
    with jr._engine(monkeypatch, "merge", k=k, keysets=sets) as m, jr._engine(monkeypatch, "join", k=k, keysets=sets) as e:
        _, gd = m.all_vs_all()
        want = ta.Oracle(len(sets), gd, COMPLETE)
        for D in tc._thresholds(gd):
            ta._eq(jr._redone(e, lambda: e.all_vs_all_complete_linkage(D), k), want(D), D)


def test_redo_only_in_the_second_chunk(monkeypatch):
    """only the second chunk overflows (join, join, merge redo): the discarded attempt must append nothing"""
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
        want = m.all_vs_all_agglomerate(COMPLETE, 0.5)
        ta._eq(m.all_vs_all_complete_linkage(0.5), want)
    with jr._engine(monkeypatch, "join", k=k, keysets=sets) as e:
        assert 0 < want[0].size < n - 1
        ta._eq(jr._redone(e, lambda: e.all_vs_all_complete_linkage(0.5), k, launches=3), want)


# ---- other contexts ---------------------------------------------------------------------------------------------
def test_literal_and_canonical_contexts():
    import torch

    seqs = _literal_inputs()
    n = len(seqs)
    for kw in ({"ambig_policy": gkd.AMBIG_LITERAL}, {"strand_mode": gkd.STRAND_CANONICAL}):
        with tc._engine(seqs, 20, **kw) as e:
            _, gd = e.all_vs_all(want_inter=False)
            want = ta.Oracle(n, gd, COMPLETE)
            for D in tc._thresholds(gd) + _attained(gd, 3):
                _same(e, D, want=want(D))
            if "ambig_policy" in kw:  # host outputs only
                dev = torch.zeros(n, dtype=torch.int32, device="cuda:0")
                m = _lib.GkdMerges(dev.data_ptr(), None, None, None, n, 0)
                assert e._L.gkd_all_vs_all_complete_linkage(e._h, n, 1.0, C.byref(m)) == _lib.GKD_EINVAL


def _literal_inputs():
    """the inputs of test_gpu_agglomerate's literal test: runs of n in most records, three identical ones"""
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
    return seqs


# ---- a caller's pair list -----------------------------------------------------------------------------------------
def test_pair_list():
    import torch

    seqs = tc._seqs(17, [60_000] * 30)
    seqs[25] = seqs[4]
    n = len(seqs)
    with tc._engine(seqs, 21) as e:
        _, gd = e.all_vs_all(want_inter=False)
        ia, ib = np.triu_indices(n, 1)
        ia, ib = ia.astype(np.uint32), ib.astype(np.uint32)
        rng = np.random.default_rng(3)
        for D in tc._thresholds(gd) + _attained(gd, 4):
            want = e.all_vs_all_agglomerate(COMPLETE, D)
            keep = gd <= D
            a, b, d = ia[keep], ib[keep], gd[keep]
            ta._eq(e.complete_linkage(n, a, b, d, D), want, D)
            # any order and either orientation; pairs beyond D take part in nothing
            p = rng.permutation(a.size)
            flip = rng.random(a.size) < 0.5
            ta._eq(e.complete_linkage(n, np.where(flip, b, a)[p], np.where(flip, a, b)[p], d[p], D), want, D)
            ta._eq(e.complete_linkage(n, ib, ia, gd, D), want, D)
            dev = [torch.from_numpy(x.view(np.int32) if x.dtype == np.uint32 else x).to("cuda:0") for x in (a, b, d)]
            ta._eq(e.complete_linkage(n, *dev, D), want, D)
        ta._eq(e.complete_linkage(n, ia[:0], ib[:0], gd[:0], 1.0), tuple(np.empty(0, dt) for dt in
                                                                        (np.uint32, np.uint32, np.float64, np.uint32)))
        a, b, d = ia[:40].copy(), ib[:40].copy(), gd[:40].copy()
        for bad, match in (("dup", "more than once"), ("swapdup", "more than once"), ("self", "two equal ids"),
                           ("range", "not below n"), ("grid", "2\\^-53"), ("big", "2\\^-53")):
            x, y, z = a.copy(), b.copy(), d.copy()
            if bad == "dup":
                x[7], y[7] = x[3], y[3]
            elif bad == "swapdup":
                x[7], y[7] = y[3], x[3]
            elif bad == "self":
                y[5] = x[5]
            elif bad == "range":
                y[9] = n
            elif bad == "grid":
                z[2] = 0.1
            else:
                z[2] = 2.5
            with pytest.raises(gkd.GkdError, match=match) as ex:
                e.complete_linkage(n, x, y, z, 1.0)
            assert ex.value.code == _lib.GKD_EINVAL, bad
        # the context stays usable
        ta._eq(e.complete_linkage(n, a, b, d, 1.0), e.complete_linkage(n, a[::-1], b[::-1], d[::-1], 1.0))


# ---- groups ---------------------------------------------------------------------------------------------------------
def _group_seqs():
    seqs = tc._seqs(21, [150_000] * 9 + [0, 40_000, 220_000, 100_000, 60_000, 80_000, 30_000])
    rng = np.random.default_rng(4)
    seqs[1] = seqs[14] = tc._random(rng, 120_000)
    for i in (8, 9, 13):
        seqs[i] = seqs[3]
    return seqs


def _group(seqs, members, ndev):
    g = gkd.Group([x % ndev for x in range(members)], k=20, workspace_bytes=4 << 20, panel=2)
    per = (len(seqs) + members - 1) // members
    for i, s in enumerate(seqs):
        assert g.add(min(i // per, members - 1), s) == i
    g.build()
    return g


def test_group_equals_single_context():
    import torch

    seqs = _group_seqs()
    n = len(seqs)
    with tc._engine(seqs, 20) as e:
        _, gd = e.all_vs_all(want_inter=False)
        want = {D: _same(e, D, want=ta.Oracle(n, gd, COMPLETE)(D)) for D in tc._thresholds(gd) + _attained(gd, 3)}
    ndev = torch.cuda.device_count()
    for members in (2, 3, 4):
        with _group(seqs, members, ndev) as g:
            for D, w in want.items():
                ta._eq(g.all_vs_all_complete_linkage(D), w, (members, D))


def test_dense_group_fails_before_the_ring(monkeypatch):
    """under a cap on the dense matrix the group call returns GKD_ENOMEM, naming the bytes, before any pair is
    intersected; the sparse group call still answers"""
    import torch

    seqs = _group_seqs()
    n = len(seqs)
    ndev = torch.cuda.device_count()
    with _group(seqs, 2, ndev) as g:
        want = g.all_vs_all_agglomerate(COMPLETE, 0.5)
        need = agg_state_bytes_complete(n)
        monkeypatch.setenv("GKD_AGG_MAX_BYTES", str(need - 1))
        m0 = g._L.gkd_group_member(g._h, 0)

        def launches():
            m = _lib.GkdMetrics()
            assert g._L.gkd_get_metrics(m0, C.byref(m)) == 0
            return m.intersect_launches

        before = launches()
        for method in (COMPLETE, gkd.LINK_AVERAGE):
            with pytest.raises(gkd.GkdError) as ex:
                g.all_vs_all_agglomerate(method, 0.5)
            assert ex.value.code == _lib.GKD_ENOMEM and "bytes" in ex.value.msg
        assert launches() == before
        ta._eq(g.all_vs_all_complete_linkage(0.5), want)
        monkeypatch.setenv("GKD_AGG_MAX_BYTES", str(need))
        ta._eq(g.all_vs_all_agglomerate(COMPLETE, 0.5), want)
    with tc._engine(seqs, 20) as e:
        monkeypatch.setenv("GKD_AGG_MAX_BYTES", str(need - 1))
        with pytest.raises(gkd.GkdError) as ex:
            e.all_vs_all_agglomerate(COMPLETE, 0.5)
        assert ex.value.code == _lib.GKD_ENOMEM and e.metrics()["pairs"] == 0
        ta._eq(e.all_vs_all_complete_linkage(0.5), want)


def agg_state_bytes_complete(n):
    """agg_state_bytes(n, complete) of csrc/agglomerate.cu: the matrix and the O(n) state"""
    return n * n * 8 + n * (5 * 4 + 2 * 8) + n * 32 + 7 * 8 + 256


# ---- the command line -----------------------------------------------------------------------------------------------
def test_cli_uses_the_sparse_form_when_the_matrix_does_not_fit(tmp_path):
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
    dists = sorted(set(float(x) for x in gd[gd < 1.0]))
    group = ["--gpus", "2"] if torch.cuda.device_count() >= 2 else ["--devices", "0,0"]
    capped = dict(os.environ, GKD_AGG_MAX_BYTES=str(agg_state_bytes_complete(n) - 1))

    def run(args, env=None):
        p = subprocess.run([tc.GKD] + args, capture_output=True, text=True, timeout=600, env=env)
        assert p.returncode == 0, p.stderr
        return p.stdout, p.stderr

    base = ["fastaDist", "-i", str(fa), "--method", "complete"]
    for args in (["--linkage"], ["--linkage", "--maxDist", repr(dists[len(dists) // 2])],
                 ["--clusters", "--maxDist", repr(dists[len(dists) // 3])], ["--clusters", "--maxDist", "0.5"]):
        for extra in ([], group):
            want, log = run(base + args + extra)
            assert "pairs within distance" not in log
            got, log = run(base + args + extra, capped)
            assert got == want, (args, extra)
            assert "merging from the pairs within distance" in log, (args, extra)
    # average linkage has no sparse form: the capped call fails as before
    p = subprocess.run([tc.GKD] + ["fastaDist", "-i", str(fa), "--linkage", "--method", "average"], capture_output=True,
                       text=True, timeout=600, env=dict(os.environ, GKD_AGG_MAX_BYTES="1000"))
    assert p.returncode != 0 and "bytes" in p.stderr
