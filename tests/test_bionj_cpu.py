"""CPU-side checks of BIONJ (gkd_*_bionj): the packed layout the device keeps (d above the diagonal, V below) gives the
definition's rows bit for bit, the definition recovers additive trees, it agrees with Gascuel's algorithm summed
directly every round and differs from NJ, every branch of lambda is reached, and the argument and command-line checks
that come before any device is used."""
import ctypes as C
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib
from oracle import bionj, nj

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_nj_cpu as tn  # noqa: E402  (random additive trees, their splits, tie-heavy inputs)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")


def _bits(rows):
    return [(a, b, np.float64(x).view(np.uint64), np.float64(y).view(np.uint64)) for a, b, x, y in rows]


def noisy_additive(n, seed):
    """the path sums of a random tree over n leaves, each times (1 + 0.1 N(0, 1)) and clipped into [0, 2]: noise that
    grows with the distance, as in Mash-style distances.  The noise breaks the triangle inequality here and there."""
    rng = random.Random(seed)
    d = tn._path_sums(tn._random_tree(rng, n), n)[np.triu_indices(n, 1)]
    g = np.random.default_rng(seed)
    return np.clip(d * (1 + 0.1 * g.standard_normal(d.size)), 0.0, 2.0)


def crafted():
    """{name: (n, triangle)}: inputs on which lambda takes each of its branches in a known round.  Clamping needs a
    triangle that breaks the triangle inequality: records 0 and 1 are 0.01 apart, one of them is 1.9 from the others
    and the other 0.1, so they join first with lambda clamped towards the near one."""

    def clamp(far):
        d = np.full((5, 5), 0.3)
        np.fill_diagonal(d, 0.0)
        d[0, 1] = d[1, 0] = 0.01
        d[far, 2:] = d[2:, far] = 1.9
        d[1 - far, 2:] = d[2:, 1 - far] = 0.1
        return d[np.triu_indices(5, 1)]

    dup = np.full((8, 8), 0.75)
    for i in range(8):
        for j in range(8):
            dup[i, j] = 0.5 + 0.0625 * ((i * 5 + j * 3) % 7) if i != j else 0.0
    dup = np.minimum(dup, dup.T)
    dup[1, :], dup[:, 1] = dup[0, :], dup[:, 0]  # records 0 and 1 are identical: d(0, 1) = V(0, 1) = 0
    dup[0, 1] = dup[1, 0] = 0.0
    return {
        "clamp_to_1": (5, clamp(1)),
        "clamp_to_0": (5, clamp(0)),
        "duplicates": (8, dup[np.triu_indices(8, 1)]),
        "zeros": (6, np.zeros(15)),
    }


# ---- the packed layout --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(12))
def test_packed_layout_equals_definition_bit_for_bit(seed):
    rng = random.Random(seed)
    n = 3 + seed * 37 // 11  # 3 .. 40
    m = n * (n - 1) // 2
    few = np.array([rng.choice((0.125, 0.25, 0.5)) for _ in range(m)])
    for d in (tn._tie_heavy(rng, n), np.zeros(m), np.ones(m), few, np.array([rng.random() for _ in range(m)]),
              noisy_additive(n, seed)):
        rows, lams = bionj.bionj(d, n)
        srows, slams = bionj.bionj_slot_rounds(d, n)
        assert _bits(srows) == _bits(rows), n
        assert np.array_equal(np.array(slams).view(np.uint64), np.array(lams).view(np.uint64)), n
        assert len(rows) == n - 1 and len(lams) == n - 2
        assert all(a < b for a, b, _, _ in rows)


def test_small_n():
    assert bionj.bionj(np.zeros(0), 0) == ([], []) and bionj.bionj(np.zeros(0), 1) == ([], [])
    assert bionj.bionj(np.array([0.75]), 2) == ([(0, 1, 0.375, 0.375)], [])
    # at r = 3 NJ's pick and lengths; the last row is NJ's midpoint
    d = np.array([0.5, 0.25, 0.125])
    rows, lams = bionj.bionj(d, 3)
    assert [r[:2] for r in rows] == [(0, 1), (0, 2)] and rows[0] == nj.nj(d, 3)[0] and len(lams) == 1


# ---- it is BIONJ --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(6))
def test_recovers_additive_trees(seed):
    """on additive distances every lambda in [0, 1] reduces to the same tree: the splits exactly, the lengths to 1e-12
    (lambda is not dyadic, so the lengths are not exact)"""
    rng = random.Random(100 + seed)
    n = rng.randint(4, 40)
    adj = tn._random_tree(rng, n)
    d = tn._path_sums(adj, n)
    rows, lams = bionj.bionj(d[np.triu_indices(n, 1)], n)
    want, got = tn._splits_of_tree(adj, n), tn._splits_of_rows(rows, n)
    assert set(got) == set(want)
    for k in want:
        assert abs(got[k] - want[k]) < 1e-12, (k, got[k], want[k])
    assert any(0.0 < x < 1.0 and x != 0.5 for x in lams)


@pytest.mark.parametrize("n", [10, 50, 200])
def test_equals_gascuel_summed_directly(n):
    """the running sums R and S drift from direct sums by rounding only: up to the round at r = 4 the two forms join the
    same pairs with lengths within 1e-12 and lambdas within 1e-10.  At r = 4 the two complementary pairs' Q are equal
    in exact arithmetic, so rounding may pick either; both give the same unrooted tree, which is compared by its
    splits"""
    for seed in range(3):
        d = noisy_additive(n, 10 * n + seed)
        rows, lams = bionj.bionj(d, n)
        trows, tlams = bionj.bionj_textbook(d, n)
        h = n - 4
        assert [r[:2] for r in rows[:h]] == [r[:2] for r in trows[:h]], seed
        assert np.abs(np.array([r[2:] for r in rows[:h]]) - np.array([r[2:] for r in trows[:h]])).max() < 1e-12
        assert np.abs(np.array(lams[:h]) - np.array(tlams[:h])).max() < 1e-10
        assert set(tn._splits_of_rows(rows, n)) == set(tn._splits_of_rows(trows, n)), seed
        # and it is not NJ
        assert rows != nj.nj(d, n), seed


def test_every_lambda_branch_is_reached():
    c = crafted()
    rows, lams = bionj.bionj(*c["clamp_to_1"][::-1])
    assert rows[0][:2] == (0, 1) and lams[0] == 1.0
    rows, lams = bionj.bionj(*c["clamp_to_0"][::-1])
    assert rows[0][:2] == (0, 1) and lams[0] == 0.0
    # V(f, g) == 0: the identical records join first with lambda 0.5 (the formula would give 0 / 0)
    rows, lams = bionj.bionj(*c["duplicates"][::-1])
    assert rows[0] == (0, 1, 0.0, 0.0) and lams[0] == 0.5
    rows, lams = bionj.bionj(*c["zeros"][::-1])
    assert lams == [0.5] * 4 and [r[:2] for r in rows] == [(0, 1), (0, 2), (0, 3), (0, 4), (0, 5)]
    # unclamped, and clamps on noisy Mash-like inputs
    lams = bionj.bionj(noisy_additive(200, 2002), 200)[1]
    assert sum(0.0 < x < 1.0 and x != 0.5 for x in lams) > 100 and 1.0 in lams and 0.0 in lams


# ---- arguments ----------------------------------------------------------------------------------------------------
def _contextless_engine():
    """an Engine whose context is NULL: its calls reach the checks that come before a context is used"""
    e = gkd.Engine.__new__(gkd.Engine)
    e._L, e._h = gkd.load(), None
    return e


def test_bionj_arguments_are_einval_before_device_use():
    lib = gkd.load()
    tri = np.full(3, 0.5)
    assert lib.gkd_bionj(None, 3, tri.ctypes.data, None) == _lib.GKD_EINVAL
    assert b"gkd_bionj: null out" in lib.gkd_last_error(None)
    assert lib.gkd_all_vs_all_bionj(None, 3, None) == _lib.GKD_EINVAL
    assert b"gkd_all_vs_all_bionj: null out" in lib.gkd_last_error(None)
    assert lib.gkd_group_all_vs_all_bionj(None, None) == _lib.GKD_EINVAL
    assert b"gkd_group_all_vs_all_bionj: null out" in lib.gkd_group_last_error(None)
    j = _lib.GkdJoins(None, None, None, None, 0, 0)
    assert lib.gkd_bionj(None, 3, None, C.byref(j)) == _lib.GKD_EINVAL
    assert b"gkd_bionj: null dist" in lib.gkd_last_error(None)
    e = _contextless_engine()
    n = 5
    i, k = np.triu_indices(n, 1)
    for bad in (float("nan"), -0.25, 2.5, float("inf")):
        d = np.full(n * (n - 1) // 2, 0.5)
        d[7] = bad
        with pytest.raises(gkd.GkdError, match=r"gkd_bionj: the distance of pair \(%d, %d\) is not a finite value in "
                                               r"\[0, 2\]" % (i[7], k[7])):
            e.bionj(d)
    # valid values pass the checks and reach the context check, which sets no message
    assert lib.gkd_bionj(None, 2, None, None) == _lib.GKD_EINVAL
    with pytest.raises(gkd.GkdError) as err:
        e.bionj(np.array([0.0, 2.0, -0.0]))
    assert err.value.code == _lib.GKD_EINVAL and "null out" in err.value.msg
    with pytest.raises(ValueError):
        e.bionj(np.zeros(4))


# ---- the command line ---------------------------------------------------------------------------------------------
def _run(args):
    p = subprocess.run([GKD] + args, capture_output=True, text=True, timeout=120, stdin=subprocess.DEVNULL)
    return p.returncode, p.stderr


def test_fastadist_tree_method_is_checked_before_any_device():
    assert os.path.exists(GKD), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    missing = ["-i", "/nonexistent/in.fa"]
    for method in ("nj", "bionj"):
        rc, err = _run(["fastaDist", "--treeMethod", method] + missing)
        assert rc == 1 and err.startswith("--treeMethod needs --tree.\n"), err
    for method in ("upgma", "BIONJ", ""):
        rc, err = _run(["fastaDist", "--tree", "--treeMethod", method] + missing)
        assert rc == 1 and err.startswith("Tree method must be nj or bionj.\n"), (method, err)
    for extra in (["--maxDist", "0.5"], ["--nearest", "3"], ["--clusters"], ["--linkage"], ["--method", "average"]):
        rc, err = _run(["fastaDist", "--tree", "--treeMethod", "bionj"] + extra + missing)
        assert rc == 1 and err.startswith("--tree and %s cannot be combined.\n" % extra[0]), (extra, err)
    # a valid method passes the checks and reaches the input
    rc, err = _run(["fastaDist", "--tree", "--treeMethod", "bionj"] + missing)
    assert rc == 1 and "/nonexistent/in.fa" in err, err
