"""BIONJ trees on the device (csrc/nj.cu, gkd_*_bionj): NJ's matrix with d above the diagonal and the variances V below
it, every round queued without a host read; only the n - 1 rows leave the device.

The oracle is oracle/bionj.py, the definition of include/gkd.h in numpy float64.  (a, b, len_a, len_b) must be equal
arrays, bit for bit, on every path: both kernel-4 forms, chunks, the forced block-join redo, the literal and canonical
contexts, the caller's triangle (host or device), the inputs that reach each branch of lambda, groups and the command
line.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib
from oracle import bionj, nj

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_bionj_cpu as tb  # noqa: E402  (the crafted lambda inputs)
import test_gpu_clusters as tc  # noqa: E402  (inputs, engine, CLI helpers)
import test_gpu_join_redo as jr  # noqa: E402  (the overflow recipes)
import test_gpu_nj as tg  # noqa: E402  (row arrays, bit comparison, additive inputs)

pytestmark = pytest.mark.gpu

_eq = tg._eq


def _oracle(n, gd, m=None):
    gd = np.asarray(gd)
    if m is not None:
        i, j = np.triu_indices(n, 1)
        gd, n = gd[(i < m) & (j < m)], m
    return tg._arrays(bionj.bionj(gd, n)[0])


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
        got = e.all_vs_all_bionj()
        if algo == "join":
            assert e.metrics()["intersect_kernel"] == 5
        m = e.metrics()
        assert m["pairs"] == n * (n - 1) // 2 and m["agglomerate_rounds"] == n - 1
        _eq(got, _oracle(n, gd))
        _eq(e.all_vs_all_bionj(n=17), _oracle(n, gd, m=17), 17)
        # the caller's triangle, from the host and from the device, is read and left as it was
        host = gd.copy()
        _eq(e.bionj(host), got)
        assert np.array_equal(host, gd)
        dev = torch.from_numpy(gd).to("cuda:0")
        _eq(e.bionj(dev), got)
        assert np.array_equal(dev.cpu().numpy(), gd)
        for small in (0, 1):
            assert all(x.size == 0 for x in e.all_vs_all_bionj(n=small))
        for small in (2, 3):
            _eq(e.all_vs_all_bionj(n=small), _oracle(n, gd, m=small), small)


def test_caller_triangle_multi_cta_and_lambda_branches():
    """n = 1,000: the multi-CTA pick and the packed move over 998 rounds; every Q tied; each branch of lambda"""
    import torch

    n = 1000
    gd = tg._additive_noise(n, 5)
    with tc._engine(tc._seqs(3, [20_000] * 4), 21) as e:
        want = _oracle(n, gd)
        _eq(e.bionj(gd), want)
        _eq(e.bionj(torch.from_numpy(gd).to("cuda:0")), want)
        assert e.metrics()["agglomerate_rounds"] == n - 1
        # it is not NJ on the same triangle
        assert not np.array_equal(e.nj(gd)[2], want[2])
        for v in (0.0, 1.0):
            _eq(e.bionj(np.full(300 * 299 // 2, v)), _oracle(300, np.full(300 * 299 // 2, v)), v)
        for name, (m, d) in tb.crafted().items():
            _eq(e.bionj(d), _oracle(m, d), name)
        d = tb.noisy_additive(200, 2002)  # unclamped lambdas and clamps to 0 and 1
        _eq(e.bionj(d), _oracle(200, d))


def test_arguments_cap_and_device_outputs():
    import torch

    seqs = tc._seqs(5, [40_000] * 24)
    seqs[20] = seqs[3]
    n = len(seqs)
    with tc._engine(seqs, 21) as e:
        want = e.all_vs_all_bionj()
        w = n - 1

        def raw(cap, arrays):
            ptr = [None if x is None else (x.data_ptr() if torch.is_tensor(x) else x.ctypes.data) for x in arrays]
            j = _lib.GkdJoins(*ptr, cap, 0)
            return e._L.gkd_all_vs_all_bionj(e._h, n, C.byref(j)), j.n

        dts = (np.uint32, np.uint32, np.float64, np.float64)
        for cap in (0, 1, w - 1):
            out = [np.full(w, 7, dtype=dt) for dt in dts]
            assert raw(cap, out) == (0, w)
            for o, x in zip(out, want):
                assert np.array_equal(o[:cap], x[:cap]) and (o[cap:] == 7).all(), cap
        assert raw(0, [None] * 4) == (0, w)
        dev = [torch.zeros(w, dtype=t, device="cuda:0") for t in (torch.int32, torch.int32, torch.float64, torch.float64)]
        assert raw(w, dev) == (0, w)
        _eq([dev[0].cpu().numpy().view(np.uint32), dev[1].cpu().numpy().view(np.uint32), dev[2].cpu().numpy(),
             dev[3].cpu().numpy()], want)
        j = _lib.GkdJoins(None, None, None, None, 0, 0)
        assert e._L.gkd_all_vs_all_bionj(e._h, n + 1, C.byref(j)) == _lib.GKD_EINVAL
        # a device triangle with an invalid value is refused by the scatter, naming the pair
        bad = torch.full((n * (n - 1) // 2,), 0.5, dtype=torch.float64, device="cuda:0")
        bad[30] = float("nan")
        i, k = np.triu_indices(n, 1)
        with pytest.raises(gkd.GkdError, match=r"gkd_bionj: the distance of pair \(%d, %d\) is not a finite value"
                                               % (i[30], k[30])):
            e.bionj(bad)
        _eq(e.all_vs_all_bionj(), want)


def test_more_than_one_chunk():
    """~12,000 gene-sized records: two 64 Mi-pair chunks.  The call equals gkd_bionj on the dense triangle."""
    n = 12_000
    seqs = tc._seqs(77, [900 + (i * 37) % 400 for i in range(n)], families=40)
    seqs[40] = seqs[11_999] = seqs[5]
    total = n * (n - 1) // 2
    with tc._engine(seqs, 21) as e:
        _, gd = e.all_vs_all(want_inter=False)
        before = e.metrics()["intersect_launches"]
        got = e.all_vs_all_bionj()
        m = e.metrics()
        assert m["pairs"] == total and m["intersect_launches"] - before == 2
        assert got[0].size == n - 1
        _eq(got, e.bionj(gd))


# ---- the forced block-join redo (recipes of test_gpu_join_redo.py) ------------------------------------------------
def test_redo_coarse_tables(monkeypatch):
    k = 25
    seqs = jr._recipe_a(k, gkd.DNA)
    with jr._engine(monkeypatch, "merge", seqs, k, coarse=True) as m, \
            jr._engine(monkeypatch, "join", seqs, k, coarse=True) as e:
        _, gd = m.all_vs_all()
        got = jr._redone(e, lambda: e.all_vs_all_bionj(), k)
        _eq(got, _oracle(len(seqs), gd))
        _eq(got, m.all_vs_all_bionj())


def test_redo_skewed_imports(monkeypatch):
    k = 21
    sets = jr._mixed(k)
    with jr._engine(monkeypatch, "merge", k=k, keysets=sets) as m, jr._engine(monkeypatch, "join", k=k, keysets=sets) as e:
        _, gd = m.all_vs_all()
        _eq(jr._redone(e, lambda: e.all_vs_all_bionj(), k), _oracle(len(sets), gd))


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
        want = m.all_vs_all_bionj()
    with jr._engine(monkeypatch, "join", k=k, keysets=sets) as e:
        _eq(jr._redone(e, lambda: e.all_vs_all_bionj(), k, launches=3), want)


# ---- other contexts ---------------------------------------------------------------------------------------------
def test_literal_and_canonical_contexts():
    import torch

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
            _eq(e.all_vs_all_bionj(), _oracle(n, gd), kw)
            if "ambig_policy" in kw:  # host outputs only
                dev = torch.zeros(n, dtype=torch.int32, device="cuda:0")
                j = _lib.GkdJoins(dev.data_ptr(), None, None, None, n, 0)
                assert e._L.gkd_all_vs_all_bionj(e._h, n, C.byref(j)) == _lib.GKD_EINVAL


# ---- memory and launches ------------------------------------------------------------------------------------------
def bionj_state_bytes(n):
    """bionj_state_bytes(n) of csrc/nj.cu: NJ's matrix and state, plus S (8 B per set) and lambda"""
    return tg.nj_state_bytes(n) + 8 * n + 8


def test_memory_cap(monkeypatch):
    import torch

    seqs = tc._seqs(13, [30_000] * 10)
    n = len(seqs)
    need = bionj_state_bytes(n)
    with tc._engine(seqs, 20) as e:
        want = e.all_vs_all_bionj()
        monkeypatch.setenv("GKD_AGG_MAX_BYTES", str(need - 1))
        with pytest.raises(gkd.GkdError) as ex:
            e.all_vs_all_bionj()
        assert ex.value.code == _lib.GKD_ENOMEM and "BIONJ of %d sets needs %d bytes" % (n, need) in ex.value.msg
        assert e.metrics()["pairs"] == 0
        monkeypatch.setenv("GKD_AGG_MAX_BYTES", str(need))
        _eq(e.all_vs_all_bionj(), want)
    monkeypatch.delenv("GKD_AGG_MAX_BYTES")
    ndev = torch.cuda.device_count()
    with gkd.Group([0, 1 % ndev], k=20, workspace_bytes=4 << 20, panel=2) as g:
        for i, s in enumerate(seqs):
            g.add(0 if i < n // 2 else 1, s)
        g.build()
        m0 = g._L.gkd_group_member(g._h, 0)

        def launches():
            m = _lib.GkdMetrics()
            assert g._L.gkd_get_metrics(m0, C.byref(m)) == 0
            return m.intersect_launches

        before = launches()
        monkeypatch.setenv("GKD_AGG_MAX_BYTES", str(need - 1))
        with pytest.raises(gkd.GkdError) as ex:
            g.all_vs_all_bionj()
        assert ex.value.code == _lib.GKD_ENOMEM and "%d bytes" % need in ex.value.msg
        assert launches() == before
        monkeypatch.setenv("GKD_AGG_MAX_BYTES", str(need))
        _eq(g.all_vs_all_bionj(), want)


def test_launches_are_pinned():
    """the fill (one scatter per staged piece) and 3 (n - 2) + 2 launches of the start and the rounds, as NJ"""
    n = 40
    d = tb.noisy_additive(n, 7)
    with tc._engine(tc._seqs(3, [20_000] * 4), 21) as e:
        for call in (e.nj, e.bionj):
            before = e.metrics()["launches"]
            call(d)
            assert e.metrics()["launches"] - before == 1 + 3 * (n - 2) + 2


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
        want = e.all_vs_all_bionj()
    _eq(want, _oracle(n, gd))
    ndev = torch.cuda.device_count()
    for members in (2, 3, 4):
        devices = [x % ndev for x in range(members)]
        with gkd.Group(devices, k=20, workspace_bytes=4 << 20, panel=2) as g:
            per = (n + members - 1) // members
            for i, s in enumerate(seqs):
                assert g.add(min(i // per, members - 1), s) == i
            g.build()
            _eq(g.all_vs_all_bionj(), want, members)


# ---- the command line ---------------------------------------------------------------------------------------------
def test_cli_fastadist_tree_method(tmp_path):
    import torch

    rng = np.random.default_rng(6)
    seqs = tc._seqs(61, [30_000] * 14 + [5_000, 200])
    seqs[9] = seqs[2]
    seqs[3] = seqs[15] = tc._random(rng, 8_000)
    fa = tmp_path / "in.fa"
    tc._fasta(fa, seqs)
    n = len(seqs)
    with tc._engine(seqs, 21) as e:
        rows = list(zip(*e.all_vs_all_bionj()))
    labels = ["r%04d" % i for i in range(n)]  # as tc._fasta writes them
    want = nj.newick(rows, labels, gkd.format_double)
    group = ["--gpus", "2"] if torch.cuda.device_count() >= 2 else ["--devices", "0,0"]
    base = ["fastaDist", "-i", str(fa), "--tree", "--treeMethod", "bionj"]
    p = subprocess.run([tc.GKD] + base, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout == want, p.stderr
    assert "joins in the BIONJ tree" in p.stderr
    assert tc._run(base + group) == want
    assert tc._run(base + ["--devices", "0,0"]) == want
    out = tmp_path / "tree.nwk"
    assert tc._run(base + ["-o", str(out)]) == ""
    assert out.read_text() == want
    # nj is the default: the same bytes as --tree alone, and not BIONJ's
    nj_tree = tc._run(["fastaDist", "-i", str(fa), "--tree"])
    assert tc._run(["fastaDist", "-i", str(fa), "--tree", "--treeMethod", "nj"]) == nj_tree != want
    p = subprocess.run([tc.GKD, "fastaDist", "-i", str(fa), "--tree", "--treeMethod", "nj"], capture_output=True,
                       text=True, timeout=600)
    assert "joins in the neighbor-joining tree" in p.stderr
    for extra in (["--maxDist", "0.5"], ["--nearest", "3"], ["--clusters"], ["--linkage"], ["--method", "average"]):
        rc, err = tg._run_fail(base + extra)
        assert rc == 1 and err.startswith("--tree and %s cannot be combined.\n" % extra[0]), (extra, err)
    rc, err = tg._run_fail(["fastaDist", "-i", str(fa), "--treeMethod", "bionj"])
    assert rc == 1 and err.startswith("--treeMethod needs --tree.\n"), err
    rc, err = tg._run_fail(["fastaDist", "-i", str(fa), "--tree", "--treeMethod", "upgma"])
    assert rc == 1 and err.startswith("Tree method must be nj or bionj.\n"), err
