"""Balanced minimum-evolution NNIs on the device (csrc/bme.cu, gkd_*_bme, gkd_bme_nni): the table of subtree averages
in HBM, built by levels and updated after every swap only where a side holds the swapped edge; only the rows leave the
device.

The oracle is oracle/bme.py, the definition of include/gkd.h, which recomputes the whole table after every swap.
(a, b, len_a, len_b) and the swap count must be equal, bit for bit, on every path: both kernel-4 forms, both start
trees, crafted start trees, the forced block-join redo, the literal and canonical contexts, the caller's triangle (host
or device), groups and the command line.
"""
import ctypes as C
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib
from oracle import bme, nj

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_bme_cpu as tbc  # noqa: E402  (crafted inputs, perturbed starts)
import test_bionj_cpu as tb  # noqa: E402  (noisy tree-shaped inputs)
import test_gpu_clusters as tc  # noqa: E402  (inputs, engine, CLI helpers)
import test_gpu_join_redo as jr  # noqa: E402  (the overflow recipes)
import test_gpu_nj as tg  # noqa: E402  (row arrays, bit comparison)
import test_nj_cpu as tn  # noqa: E402  (random additive trees)

pytestmark = pytest.mark.gpu

_eq = tg._eq


def _oracle(n, gd, start="bionj", m=None):
    gd = np.asarray(gd)
    if m is not None:
        i, j = np.triu_indices(n, 1)
        gd, n = gd[(i < m) & (j < m)], m
    rows, swaps = bme.bme(gd, n, start)
    return tg._arrays(rows), swaps


def _same(got, want, what=None):
    _eq(got[0], want[0], what)
    assert got[1] == want[1], what


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
        for start in ("nj", "bionj"):
            got = e.all_vs_all_bme(start)
            if algo == "join":
                assert e.metrics()["intersect_kernel"] == 5
            assert e.metrics()["pairs"] == n * (n - 1) // 2
            _same(got, _oracle(n, gd, start), start)
            _same(e.all_vs_all_bme(start, n=17), _oracle(n, gd, start, m=17), 17)
            host = gd.copy()
            _same(e.bme(host, start), got)
            assert np.array_equal(host, gd)
            dev = torch.from_numpy(gd).to("cuda:0")
            _same(e.bme(dev, start), got)
        for small in (0, 1):
            rows, swaps = e.all_vs_all_bme(n=small)
            assert all(x.size == 0 for x in rows) and swaps == 0
        for small in (2, 3, 4):
            _same(e.all_vs_all_bme(n=small), _oracle(n, gd, m=small), small)
        _eq(e.all_vs_all_bme("nj", n=2)[0], e.all_vs_all_nj(n=2))


def test_caller_triangles_and_crafted_trees():
    """noisy tree-shaped triangles from both starts, additive triangles from perturbed starts, the crafted tie and
    root-edge inputs, every one against the oracle; crafted trees on the device"""
    import torch

    with tc._engine(tc._seqs(3, [20_000] * 4), 21) as e:
        for seed, n in [(1, 5), (2, 9), (3, 30), (4, 60)]:
            tri = tb.noisy_additive(n, seed)
            for start in ("nj", "bionj"):
                _same(e.bme(tri, start), _oracle(n, tri, start), (seed, start))
        for seed in range(6):
            rng = random.Random(seed)
            n = 24
            tri = tn._path_sums(tn._random_tree(rng, n), n)[np.triu_indices(n, 1)]
            start = tbc._nni_rows(nj.nj(tri, n), n, rng, 1 + seed % 3)
            a, b = [r[0] for r in start], [r[1] for r in start]
            rows, swaps = bme.bme_nni(tri, n, start)
            _same(e.bme_nni(tri, a, b), (tg._arrays(rows), swaps), seed)
            ta = torch.tensor(np.array(a, dtype=np.int32), device="cuda:0")
            tb_ = torch.tensor(np.array(b, dtype=np.int32), device="cuda:0")
            tree = _lib.GkdJoins(ta.data_ptr(), tb_.data_ptr(), None, None, n - 1, n - 1)
            out = [np.zeros(n - 1, dtype=dt) for dt in (np.uint32, np.uint32, np.float64, np.float64)]
            j = _lib.GkdJoins(*[x.ctypes.data for x in out], n - 1, 0)
            w = C.c_uint64(0)
            assert e._L.gkd_bme_nni(e._h, n, tri.ctypes.data, C.byref(tree), C.byref(j), C.byref(w)) == 0
            _same((tuple(out), w.value), (tg._arrays(rows), swaps))
        for name, (n, tri, start) in tbc.crafted().items():
            a, b = [r[0] for r in start], [r[1] for r in start]
            rows, swaps = bme.bme_nni(tri, n, start)
            assert swaps >= 1
            _same(e.bme_nni(np.asarray(tri), a, b), (tg._arrays(rows), swaps), name)


def test_many_swaps():
    """starts far from the best tree (the NJ tree of much noisier distances): n = 80 takes hundreds of swaps, each with
    its incremental update, and equals the oracle, which rebuilds the table after every swap; n = 2,000 ends at a fixed
    point of the device's own search"""
    with tc._engine(tc._seqs(3, [20_000] * 4), 21) as e:
        for n, noise in [(80, 0.6), (2000, 0.1)]:
            tri = tb.noisy_additive(n, 11)
            g = np.random.default_rng(12)
            start = nj.nj(np.clip(tri * (1 + noise * g.standard_normal(tri.size)), 0.0, 2.0), n)
            rows, swaps = e.bme_nni(tri, [r[0] for r in start], [r[1] for r in start])
            assert 50 < swaps < bme.max_swaps(n), (n, swaps)
            if n <= 80:
                _same((rows, swaps), (tg._arrays(bme.bme_nni(tri, n, start)[0]), swaps))
            again, swaps2 = e.bme_nni(tri, rows[0], rows[1])
            assert swaps2 == 0
            _eq(again, rows)


def _max_height(rows, n):
    """the largest height of a side of the rows' tree"""
    t = bme.Tree(n, rows)
    memo = {}

    def h(x):
        if x not in memo:
            memo[x] = 0 if t.is_leaf_side(x) else 1 + max(h(c) for c in t.children(x))
        return memo[x]

    return max(h(x) for x in tbc._sides(t))


def test_launches_are_pinned():
    """a search that takes no swap: the scatter, the leaf block, 2 x (largest side height) level launches of the build,
    one pick and the lengths; a search that swaps adds per swap one pick and at most one launch per level of its marked
    cells, far below the build's launches"""
    n = 60
    tri = tb.noisy_additive(n, 7)
    with tc._engine(tc._seqs(3, [20_000] * 4), 21) as e:
        (rows, swaps) = e.bme(tri, "nj")
        before = e.metrics()["launches"]
        again, zero = e.bme_nni(tri, rows[0], rows[1])
        assert zero == 0
        build = 2 * _max_height(list(zip(rows[0], rows[1])), n)
        assert e.metrics()["launches"] - before == 1 + 1 + build + 1 + 1
        g = np.random.default_rng(3)
        start = nj.nj(np.clip(tri * (1 + 0.5 * g.standard_normal(tri.size)), 0.0, 2.0), n)
        before = e.metrics()["launches"]
        _, swaps = e.bme_nni(tri, [r[0] for r in start], [r[1] for r in start])
        used = e.metrics()["launches"] - before
        first = 1 + 1 + 2 * _max_height(start, n) + 1
        assert swaps > 10
        assert first + swaps <= used <= first + swaps * (1 + 2 * (n - 1))
        assert (used - first) / swaps < build


def test_more_than_one_chunk():
    """~12,000 gene-sized records: two 64 Mi-pair chunks.  The call equals gkd_bme on the dense triangle."""
    n = 12_000
    seqs = tc._seqs(77, [900 + (i * 37) % 400 for i in range(n)], families=40)
    seqs[40] = seqs[11_999] = seqs[5]
    with tc._engine(seqs, 21) as e:
        _, gd = e.all_vs_all(want_inter=False)
        before = e.metrics()["intersect_launches"]
        got = e.all_vs_all_bme("nj")
        m = e.metrics()
        assert m["pairs"] == n * (n - 1) // 2 and m["intersect_launches"] - before == 2
        _same(got, e.bme(gd, "nj"))


def test_arguments_cap_and_device_outputs():
    import torch

    seqs = tc._seqs(5, [40_000] * 24)
    seqs[20] = seqs[3]
    n = len(seqs)
    with tc._engine(seqs, 21) as e:
        want, swaps = e.all_vs_all_bme()
        w = n - 1

        def raw(cap, arrays, sw=True):
            ptr = [None if x is None else (x.data_ptr() if torch.is_tensor(x) else x.ctypes.data) for x in arrays]
            j = _lib.GkdJoins(*ptr, cap, 0)
            s = C.c_uint64(99)
            rc = e._L.gkd_all_vs_all_bme(e._h, n, _lib.TREE_BIONJ, C.byref(j), C.byref(s) if sw else None)
            return rc, j.n, s.value

        dts = (np.uint32, np.uint32, np.float64, np.float64)
        for cap in (0, 1, w - 1):
            out = [np.full(w, 7, dtype=dt) for dt in dts]
            assert raw(cap, out) == (0, w, swaps)
            for o, x in zip(out, want):
                assert np.array_equal(o[:cap], x[:cap]) and (o[cap:] == 7).all(), cap
        assert raw(0, [None] * 4, sw=False) == (0, w, 99)
        dev = [torch.zeros(w, dtype=t, device="cuda:0") for t in (torch.int32, torch.int32, torch.float64, torch.float64)]
        assert raw(w, dev)[0] == 0
        _eq([dev[0].cpu().numpy().view(np.uint32), dev[1].cpu().numpy().view(np.uint32), dev[2].cpu().numpy(),
             dev[3].cpu().numpy()], want)
        bad = torch.full((n * (n - 1) // 2,), 0.5, dtype=torch.float64, device="cuda:0")
        bad[30] = float("nan")
        i, k = np.triu_indices(n, 1)
        with pytest.raises(gkd.GkdError, match=r"gkd_bme: the distance of pair \(%d, %d\) is not a finite value"
                                               % (i[30], k[30])):
            e.bme(bad)
        _eq(e.all_vs_all_bme()[0], want)


# ---- the forced block-join redo (recipes of test_gpu_join_redo.py) ------------------------------------------------
def test_redo_coarse_tables(monkeypatch):
    k = 25
    seqs = jr._recipe_a(k, gkd.DNA)
    with jr._engine(monkeypatch, "merge", seqs, k, coarse=True) as m, \
            jr._engine(monkeypatch, "join", seqs, k, coarse=True) as e:
        _, gd = m.all_vs_all()
        got = jr._redone(e, lambda: e.all_vs_all_bme(), k)
        _same(got, _oracle(len(seqs), gd))


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
            _same(e.all_vs_all_bme("nj"), _oracle(n, gd, "nj"), kw)


# ---- memory and groups ----------------------------------------------------------------------------------------------
def bme_state_bytes(n):
    """bme_state_bytes(n) of csrc/bme.cu"""
    N, M = n, 2 * n - 2
    nj_bytes = tg.nj_state_bytes(n) + 8 * n + 8
    table = (max(M * M * 8, N * M * 8 + nj_bytes) + 255) & ~255
    return table + 16 * M * 4 + 256 + M * 64 + M * 8 + 24 + 256 + min(1 << 20, M * M) * 8


def test_memory_cap(monkeypatch):
    import torch

    seqs = tc._seqs(13, [30_000] * 10)
    n = len(seqs)
    need = bme_state_bytes(n)
    with tc._engine(seqs, 20) as e:
        want = e.all_vs_all_bme()
        monkeypatch.setenv("GKD_AGG_MAX_BYTES", str(need - 1))
        with pytest.raises(gkd.GkdError) as ex:
            e.all_vs_all_bme()
        assert ex.value.code == _lib.GKD_ENOMEM and "balanced minimum evolution of %d sets needs %d bytes" % (n, need) in ex.value.msg
        assert e.metrics()["pairs"] == 0
        monkeypatch.setenv("GKD_AGG_MAX_BYTES", str(need))
        _same(e.all_vs_all_bme(), want)
    monkeypatch.delenv("GKD_AGG_MAX_BYTES")
    ndev = torch.cuda.device_count()
    with gkd.Group([0, 1 % ndev], k=20, workspace_bytes=4 << 20, panel=2) as g:
        for i, s in enumerate(seqs):
            g.add(0 if i < n // 2 else 1, s)
        g.build()
        monkeypatch.setenv("GKD_AGG_MAX_BYTES", str(need - 1))
        with pytest.raises(gkd.GkdError) as ex:
            g.all_vs_all_bme()
        assert ex.value.code == _lib.GKD_ENOMEM and "%d bytes" % need in ex.value.msg
        monkeypatch.setenv("GKD_AGG_MAX_BYTES", str(need))
        _same(g.all_vs_all_bme(), want)


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
        want = e.all_vs_all_bme()
    _same(want, _oracle(n, gd))
    ndev = torch.cuda.device_count()
    for members in (2, 3, 4):
        devices = [x % ndev for x in range(members)]
        with gkd.Group(devices, k=20, workspace_bytes=4 << 20, panel=2) as g:
            per = (n + members - 1) // members
            for i, s in enumerate(seqs):
                assert g.add(min(i // per, members - 1), s) == i
            g.build()
            _same(g.all_vs_all_bme(), want, members)


# ---- the command line ---------------------------------------------------------------------------------------------
def test_cli_fastadist_nni(tmp_path):
    import torch

    rng = np.random.default_rng(6)
    seqs = tc._seqs(61, [30_000] * 14 + [5_000, 200])
    seqs[9] = seqs[2]
    seqs[3] = seqs[15] = tc._random(rng, 8_000)
    fa = tmp_path / "in.fa"
    tc._fasta(fa, seqs)
    n = len(seqs)
    labels = ["r%04d" % i for i in range(n)]
    group = ["--gpus", "2"] if torch.cuda.device_count() >= 2 else ["--devices", "0,0"]
    for method in ("nj", "bionj"):
        with tc._engine(seqs, 21) as e:
            rows, swaps = e.all_vs_all_bme(method)
            plain = list(zip(*(e.all_vs_all_nj() if method == "nj" else e.all_vs_all_bionj())))
        want = nj.newick(list(zip(*rows)), labels, gkd.format_double)
        base = ["fastaDist", "-i", str(fa), "--tree", "--treeMethod", method]
        p = subprocess.run([tc.GKD] + base + ["--nni"], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0 and p.stdout == want, p.stderr
        assert "%d balanced NNIs applied" % swaps in p.stderr
        assert tc._run(base + ["--nni"] + group) == want
        # without --nni the bytes are the start tree's, as before
        assert tc._run(base) == nj.newick(plain, labels, gkd.format_double)
    rc, err = tg._run_fail(["fastaDist", "-i", str(fa), "--nni"])
    assert rc == 1 and err.startswith("--nni needs --tree.\n"), err
    rc, err = tg._run_fail(["fastaDist", "-i", str(fa), "--tree", "--nni", "--maxDist", "0.5"])
    assert rc == 1 and err.startswith("--tree and --maxDist cannot be combined.\n"), err
