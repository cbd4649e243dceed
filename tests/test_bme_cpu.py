"""CPU-side checks of the balanced minimum-evolution NNI search (gkd_*_bme, gkd_bme_nni): the definition's Delta and
gains equal the closed forms of BME (path weights and Pauplin's length), its output is NNI-locally optimal and never
longer than its start, it recovers additive trees from perturbed starts, it lowers the Robinson-Foulds distance of
BIONJ on noisy inputs, crafted inputs reach the tie rule, a swap across the root edge, the cap and the small cases,
and the argument, row and command-line checks come before any device is used."""
import ctypes as C
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib
from oracle import bionj, bme, nj

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_bionj_cpu as tb  # noqa: E402  (noisy tree-shaped inputs)
import test_nj_cpu as tn  # noqa: E402  (random additive trees and their splits)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")


def _sides(t: bme.Tree):
    out = [(v, 0) for v in range(t.root)]
    out += [(v, 1) for v in range(t.root) if t.par[v] != t.root]
    return out


def _disjoint(t, X, Y):
    a = {x for x, _ in t.leaves(t.canon(X))}
    b = {x for x, _ in t.leaves(t.canon(Y))}
    return not (a & b)


def _nni_rows(rows, n, rng, k):
    """the tree of rows after k random NNIs"""
    t = bme.Tree(n, rows)
    for _ in range(k):
        where, groups = rng.choice(t.edges())
        A, B, C_, D = t.name(groups)
        bme.apply(t, (1.0, 0, 0, rng.randint(0, 1), where, groups))
    return bme.rows_of(t, {v: 0.0 for v in range(t.root)} | {"root": 0.0})


@pytest.mark.parametrize("seed", range(4))
def test_definition_equals_direct_form(seed):
    n = 9
    tri = tb.noisy_additive(n, seed)
    d = nj.square(tri, n)
    t = bme.Tree(n, bionj.bionj(tri, n)[0])
    D = bme.Table(t, d)
    for X in _sides(t):
        for Y in _sides(t):
            if X < Y and _disjoint(t, X, Y):
                assert abs(D(X, Y) - bme.direct_delta(t, d, X, Y)) < 1e-12
    L0 = bme.pauplin_length(t, d)
    for c in bme.gains(t, D):
        t2 = bme.Tree(n, bionj.bionj(tri, n)[0])
        c2 = [x for x in bme.gains(t2, bme.Table(t2, d)) if x[1:4] == c[1:4]][0]
        bme.apply(t2, c2)
        assert abs(c[0] - (L0 - bme.pauplin_length(t2, d))) < 1e-12


@pytest.mark.parametrize("seed", range(6))
def test_output_is_locally_optimal_and_not_longer(seed):
    n = 14
    tri = tb.noisy_additive(n, 100 + seed)
    d = nj.square(tri, n)
    start = bionj.bionj(tri, n)[0]
    rows, swaps = bme.bme_nni(tri, n, start)
    t = bme.Tree(n, rows)
    assert bme.pauplin_length(t, d) <= bme.pauplin_length(bme.Tree(n, start), d) + 1e-12
    L = bme.pauplin_length(t, d)
    for where, groups in t.edges():
        for sw in (0, 1):
            t2 = bme.Tree(n, rows)
            g2 = dict(t2.edges())[where] if where != "root" else [e for e in t2.edges() if e[0] == "root"][0][1]
            bme.apply(t2, (1.0, 0, 0, sw, where, g2))
            assert L - bme.pauplin_length(t2, d) <= bme.EPS + 1e-12


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("k", [1, 2])
def test_additive_recovered_from_perturbed_start(seed, k):
    rng = random.Random(seed)
    n = 10
    adj = tn._random_tree(rng, n)
    d = tn._path_sums(adj, n)
    tri = d[np.triu_indices(n, 1)]
    start = _nni_rows(nj.nj(tri, n), n, rng, k)
    rows, swaps = bme.bme_nni(tri, n, start)
    assert set(tn._splits_of_rows(rows, n)) == set(tn._splits_of_tree(adj, n))
    assert (swaps > 0) == (set(tn._splits_of_rows(start, n)) != set(tn._splits_of_tree(adj, n)))
    # the lengths are the tree's: the path sums of the rows equal d
    want, _ = bme.bme_nni(tri, n, nj.nj(tri, n))
    assert _path_sums_of_rows(rows, n) == pytest.approx(d, abs=1e-12)
    assert _path_sums_of_rows(want, n) == pytest.approx(d, abs=1e-12)


def _path_sums_of_rows(rows, n):
    """the leaf-to-leaf path sums of the rows' tree"""
    out = np.zeros((n, n))
    cur = {i: {i: 0.0} for i in range(n)}
    for a, b, la, lb in rows:
        A, B = cur[a], cur.pop(b)
        for x, u in A.items():
            for y, w in B.items():
                out[x, y] = out[y, x] = u + la + w + lb
        cur[a] = {x: v + la for x, v in A.items()} | {y: v + lb for y, v in B.items()}
    return out


@pytest.mark.parametrize("seed", range(4))
def test_nj_start_on_additive_input_takes_no_swap(seed):
    rng = random.Random(seed)
    n = 12
    tri = tn._path_sums(tn._random_tree(rng, n), n)[np.triu_indices(n, 1)]
    assert bme.bme(tri, n, "nj")[1] == 0


def test_noisy_inputs_come_closer_to_the_true_tree():
    before = after = 0
    for seed in range(30):
        n = 16
        rng = random.Random(seed)
        adj = tn._random_tree(rng, n)
        d = tn._path_sums(adj, n)[np.triu_indices(n, 1)]
        g = np.random.default_rng(seed)
        tri = np.clip(d * (1 + 0.25 * g.standard_normal(d.size)), 0.0, 2.0)
        true = set(tn._splits_of_tree(adj, n))
        start = bionj.bionj(tri, n)[0]
        rows, _ = bme.bme_nni(tri, n, start)
        before += len(true ^ set(tn._splits_of_rows(start, n)))
        after += len(true ^ set(tn._splits_of_rows(rows, n)))
    assert after < before


def crafted():
    """{name: (n, triangle, start rows)}"""
    out = {}
    # four leaves: a square, every quartet split equally long, so both swaps of the one edge gain the same: the tie
    # goes to swap B <-> C
    sq = np.full((4, 4), 0.25)
    np.fill_diagonal(sq, 0.0)
    sq[0, 1] = sq[1, 0] = sq[2, 3] = sq[3, 2] = 0.5  # {0,1 | 2,3} is the longest of the three splits
    out["tie"] = (4, sq[np.triu_indices(4, 1)], [(0, 1), (2, 3), (0, 2)])
    # an additive tree over six leaves ((0,1),(2,3)) | ((4,5)) rooted across its middle edge, started with 1 and 2
    # exchanged across the root edge
    adj = {6: {0: .1, 1: .1, 8: .2}, 7: {2: .1, 3: .1, 8: .2}, 8: {6: .2, 7: .2, 9: .3}, 9: {8: .3, 4: .1, 5: .1}}
    for v, nb in list(adj.items()):
        for w, x in nb.items():
            adj.setdefault(w, {})[v] = x
    d6 = tn._path_sums(adj, 6)
    out["root_edge"] = (4, d6[np.ix_([0, 1, 2, 3], [0, 1, 2, 3])][np.triu_indices(4, 1)], [(0, 2), (1, 3), (0, 1)])
    # six leaves from a caterpillar: the two best swaps are at two different edges with equal gains; the one of the
    # smaller edge key (label 2 before label 3) is taken
    out["edge_tie"] = (6, np.array([0.25, 0.375, 0.125, 0.5, 0.125, 0.25, 0.125, 0.375, 0.375, 0.375, 0.125, 0.5, 0.375,
                                    0.125, 0.125]), [(0, 1), (0, 2), (0, 3), (0, 4), (0, 5)])
    return out


def test_tie_between_two_edges():
    n, tri, start = crafted()["edge_tie"]
    t = bme.Tree(n, start)
    cands = sorted(bme.gains(t, bme.Table(t, nj.square(tri, n))), key=lambda c: (-c[0], c[1], c[2], c[3]))
    assert cands[0][0] == cands[1][0] > bme.EPS and cands[0][4] != cands[1][4]
    assert (cands[0][1], cands[1][1]) == (2, 3)
    assert bme.best(cands) is cands[0]


def test_tie_rule():
    n, tri, start = crafted()["tie"]
    t = bme.Tree(n, start)
    cands = bme.gains(t, bme.Table(t, nj.square(tri, n)))
    assert len(cands) == 2 and cands[0][0] == cands[1][0] > bme.EPS
    assert bme.best(cands)[3] == 0


def test_swap_across_the_root_edge():
    n, tri, start = crafted()["root_edge"]
    t = bme.Tree(n, start)
    assert [w for w, _ in t.edges()] == ["root"]
    rows, swaps = bme.bme_nni(tri, n, start)
    assert swaps == 1
    assert {frozenset(s) for s in bme.tree_splits(bme.Tree(n, rows))} == {frozenset({2, 3})}


def test_cap():
    rng = random.Random(3)
    n = 10
    tri = tn._path_sums(tn._random_tree(rng, n), n)[np.triu_indices(n, 1)]
    start = _nni_rows(nj.nj(tri, n), n, rng, 3)
    full, swaps = bme.bme_nni(tri, n, start)
    assert swaps >= 2
    capped, k = bme.bme_nni(tri, n, start, cap=1)
    assert k == 1 and capped != full
    assert bme.max_swaps(n) == 4 * n


def test_small_n():
    assert bme.bme_nni([], 0, []) == ([], 0)
    assert bme.bme_nni([], 1, []) == ([], 0)
    assert bme.bme([0.375], 2, "nj") == ([(0, 1, 0.1875, 0.1875)], 0)
    assert bme.bme([0.375], 2, "nj")[0] == nj.nj([0.375], 2)
    tri = [0.3, 0.5, 0.4]
    rows, swaps = bme.bme(tri, 3, "bionj")
    assert swaps == 0 and len(rows) == 2
    # the pendant lengths of a star: 0.5 ((d_iA + d_iB) - d_AB)
    la = {0: 0.5 * ((0.3 + 0.5) - 0.4), 1: 0.5 * ((0.3 + 0.4) - 0.5), 2: 0.5 * ((0.5 + 0.4) - 0.3)}
    a, b, x, y = rows[0]
    assert (x, y) == (la[a], la[b])


# ---- the checks before any device is used --------------------------------------------------------------------------


def _contextless_engine():
    e = gkd.Engine.__new__(gkd.Engine)
    e._L, e._h = gkd.load(), None
    return e


def test_bme_arguments_are_einval_before_device_use():
    lib = gkd.load()
    tri = np.full(3, 0.5)
    j = _lib.GkdJoins(None, None, None, None, 0, 0)
    assert lib.gkd_bme(None, 3, tri.ctypes.data, 1, None, None) == _lib.GKD_EINVAL
    assert b"gkd_bme: null out" in lib.gkd_last_error(None)
    assert lib.gkd_bme(None, 3, tri.ctypes.data, 3, C.byref(j), None) == _lib.GKD_EINVAL
    assert b"gkd_bme: start 3 is not" in lib.gkd_last_error(None)
    assert lib.gkd_all_vs_all_bme(None, 3, 1, None, None) == _lib.GKD_EINVAL
    assert b"gkd_all_vs_all_bme: null out" in lib.gkd_last_error(None)
    assert lib.gkd_all_vs_all_bme(None, 3, 0, C.byref(j), None) == _lib.GKD_EINVAL
    assert lib.gkd_group_all_vs_all_bme(None, 1, None, None) == _lib.GKD_EINVAL
    assert b"gkd_group_all_vs_all_bme: null out" in lib.gkd_group_last_error(None)
    assert lib.gkd_group_all_vs_all_bme(None, 5, C.byref(j), None) == _lib.GKD_EINVAL
    assert lib.gkd_bme(None, 3, None, 1, C.byref(j), None) == _lib.GKD_EINVAL
    assert b"gkd_bme: null dist" in lib.gkd_last_error(None)
    e = _contextless_engine()
    with pytest.raises(ValueError):
        e.bme(tri, start="upgma")
    n = 5
    i, k = np.triu_indices(n, 1)
    d = np.full(n * (n - 1) // 2, 0.5)
    d[7] = float("nan")
    with pytest.raises(gkd.GkdError, match=r"gkd_bme: the distance of pair \(%d, %d\)" % (i[7], k[7])):
        e.bme(d)
    with pytest.raises(gkd.GkdError, match=r"gkd_bme_nni: the distance of pair \(%d, %d\)" % (i[7], k[7])):
        e.bme_nni(d, [0, 0, 0, 0], [1, 2, 3, 4])


@pytest.mark.parametrize("a,b,msg", [
    ([0, 2], [1, 3], r"the tree has 2 rows; a tree of 4 sets has 3"),
    ([0, 2, 0], [1, 4, 2], r"row 1: label 4 is not below n = 4"),
    ([0, 3, 0], [1, 2, 2], r"row 1: labels 3, 2 are not a < b"),
    ([0, 1, 0], [1, 2, 3], r"row 1: label 1 was joined by an earlier row"),
    ([0, 2, 0], [1, 3, 3], r"row 2: label 3 was joined by an earlier row"),
])
def test_malformed_rows_are_einval_before_device_use(a, b, msg):
    e = _contextless_engine()
    tri = np.full(6, 0.5)
    with pytest.raises(gkd.GkdError, match="gkd_bme_nni: " + msg) as err:
        e.bme_nni(tri, a, b)
    assert err.value.code == _lib.GKD_EINVAL
    # a well-formed tree passes the checks and reaches the context check
    with pytest.raises(gkd.GkdError) as err:
        e.bme_nni(tri, [0, 2, 0], [1, 3, 2])
    assert err.value.code == _lib.GKD_EINVAL


def test_nni_parse_errors(tmp_path):
    fa = tmp_path / "in.fa"
    fa.write_text(">a\nACGTACGTACGTACGTACGTACGT\n>b\nACGTACGTACGTACGTACGTACGA\n")
    for args, msg in [(["--nni"], "--nni needs --tree."), (["--nni", "--maxDist", "0.5"], "--nni needs --tree.")]:
        r = subprocess.run([GKD, "fastaDist", "-i", str(fa)] + args, capture_output=True, text=True,
                           env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
        assert r.returncode != 0 and msg in (r.stdout + r.stderr)
    r = subprocess.run([GKD, "fastaDist", "-i", str(fa), "--tree", "--nni", "--linkage"], capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode != 0 and "--tree and --linkage cannot be combined." in (r.stdout + r.stderr)
