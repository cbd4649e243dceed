"""CPU-side checks of complete- and average-linkage agglomeration (gkd_*_agglomerate): the exact oracle against scipy, the
reciprocal-nearest-neighbour rounds the device runs against the sequential definition on tie-heavy inputs, the 2^-53
grid of kernel 5's distances, and the argument checks that come before any context, group or device is used."""
import ctypes as C
import os
import random
import subprocess
from fractions import Fraction

import numpy as np
import pytest
from scipy.cluster import hierarchy

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib
from oracle import agglomerate as agg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")
METHODS = {agg.COMPLETE: "complete", agg.AVERAGE: "average"}


def _grid(rng, m):
    """m distinct-ish random distances on the 2^-53 grid in [0, 1]"""
    return np.array([rng.getrandbits(53) / 2.0 ** 53 for _ in range(m)])


def _topology(merges, n):
    """the merges as (frozenset of the two clusters' members) -- comparable with scipy's cluster ids"""
    members = {x: frozenset([x]) for x in range(n)}
    out = []
    for a, b, _, size in merges:
        out.append(frozenset([members[a], members[b]]))
        members[a] = members[a] | members[b]
        assert len(members[a]) == size
        del members[b]
    return out


def _scipy_topology(Z, n):
    members = {x: frozenset([x]) for x in range(n)}
    out = []
    for t, (p, q, _, _) in enumerate(Z):
        out.append(frozenset([members[int(p)], members[int(q)]]))
        members[n + t] = members.pop(int(p)) | members.pop(int(q))
    return out


@pytest.mark.parametrize("method", sorted(METHODS))
@pytest.mark.parametrize("n", [2, 3, 9, 30])
def test_oracle_equals_scipy_without_ties(method, n):
    rng = random.Random(n * 7 + method)
    d = _grid(rng, n * (n - 1) // 2)
    merges = agg.sequential(d, n, method, 1.0)
    Z = hierarchy.linkage(d, method=METHODS[method])
    assert len(merges) == n - 1
    assert _topology(merges, n) == _scipy_topology(Z, n)
    h = np.array([m[2] for m in merges])
    if method == agg.COMPLETE:
        assert np.array_equal(h, Z[:, 2])
    else:
        assert np.allclose(h, Z[:, 2], rtol=0, atol=1e-12)
    assert [m[3] for m in merges] == Z[:, 3].astype(int).tolist()


def _tie_heavy(rng, n):
    """small integers x 2^-53, blocks of identical records (0.0) and of unrelated ones (1.0)"""
    w = np.empty((n, n))
    for i in range(n):
        for j in range(i + 1, n):
            r = rng.random()
            w[i, j] = 0.0 if r < 0.15 else 1.0 if r < 0.5 else rng.randint(1, 6) / 2.0 ** 53
    blk = rng.randrange(n)
    for i in range(blk, min(n, blk + 4)):
        for j in range(i + 1, min(n, blk + 4)):
            w[i, j] = 0.0
    return w[np.triu_indices(n, 1)]


@pytest.mark.parametrize("method", sorted(METHODS))
@pytest.mark.parametrize("seed", range(6))
def test_rnn_rounds_equal_sequential_on_ties(method, seed):
    rng = random.Random(seed)
    n = rng.randint(2, 24)
    d = _tie_heavy(rng, n)
    for max_dist in (-1.0, 0.0, 3 / 2.0 ** 53, 0.5, 1.0):
        seq = agg.sequential(d, n, method, max_dist)
        par, rounds = agg.rnn_rounds(d, n, method, max_dist)
        assert par == seq, (max_dist, n)
        assert rounds <= len(seq)
        # the keys strictly increase in the sequential order
        assert all(h1 <= h2 for (_, _, h1, _), (_, _, h2, _) in zip(seq, seq[1:]))


def test_mutation_chain_takes_many_rounds():
    n = 12
    full = np.array([[abs(i - j) / 2.0 ** 53 if i != j else 0 for j in range(n)] for i in range(n)])
    d = full[np.triu_indices(n, 1)]
    seq = agg.sequential(d, n, agg.COMPLETE, 1.0)
    par, rounds = agg.rnn_rounds(d, n, agg.COMPLETE, 1.0)
    assert par == seq and rounds >= 3


def test_kernel5_distances_are_on_the_2_53_grid():
    rng = random.Random(5)
    for _ in range(200000):
        sa, sb = rng.randint(1, 1 << 28), rng.randint(1, 1 << 28)
        inter = rng.randint(0, min(sa, sb))
        d = agg.pair_result(inter, sa, sb)
        assert 0.0 <= d <= 1.0
        assert (Fraction(d) * (1 << 53)).denominator == 1, (inter, sa, sb)


def test_average_height_rounds_to_nearest_even():
    assert agg.height(3, 2) == 1.5 / 2.0 ** 53
    for s, n in ((1, 3), (10 ** 20 + 7, 3 ** 30), (2 ** 60 - 1, 2 ** 40 + 1)):
        assert agg.height(s, n) == float(Fraction(s, n << 53))
    with pytest.raises(ValueError):
        agg.to_words([0.1])  # not a multiple of 2^-53
    with pytest.raises(ValueError):
        agg.to_words([2.5])


def _merges(cap=4):
    a, b = np.zeros(cap, dtype=np.uint32), np.zeros(cap, dtype=np.uint32)
    h, s = np.zeros(cap, dtype=np.float64), np.zeros(cap, dtype=np.uint32)
    return (a, b, h, s), _lib.GkdMerges(a.ctypes.data, b.ctypes.data, h.ctypes.data, s.ctypes.data, cap, 0)


def test_agglomerate_arguments_are_einval_before_device_use():
    """NaN max_dist, an unknown method and a NULL out are refused with a message even with no context or group (and no
    GPU); arguments that pass reach the NULL-handle check, still GKD_EINVAL."""
    lib = gkd.load()
    keep, m = _merges()
    tri = np.zeros(1)
    calls = {
        "all_vs_all": (lambda meth, D, out: lib.gkd_all_vs_all_agglomerate(None, 2, meth, D, out), lib.gkd_last_error),
        "triangle": (lambda meth, D, out: lib.gkd_agglomerate(None, 2, tri.ctypes.data, meth, D, out), lib.gkd_last_error),
        "group": (lambda meth, D, out: lib.gkd_group_all_vs_all_agglomerate(None, meth, D, out), lib.gkd_group_last_error),
    }
    for name, (call, err) in calls.items():
        assert call(gkd.LINK_COMPLETE, float("nan"), C.byref(m)) == _lib.GKD_EINVAL, name
        assert b"NaN" in err(None), name
        for bad in (0, 3, -1):
            assert call(bad, 0.5, C.byref(m)) == _lib.GKD_EINVAL, name
            assert b"unknown method" in err(None), name
        assert call(gkd.LINK_AVERAGE, 0.5, None) == _lib.GKD_EINVAL, name
        assert b"null out" in err(None), name
        for meth in (gkd.LINK_COMPLETE, gkd.LINK_AVERAGE):
            for D in (0.5, -1.0, 1.0):
                assert call(meth, D, C.byref(m)) == _lib.GKD_EINVAL, (name, D)
    assert lib.gkd_agglomerate(None, 3, None, gkd.LINK_COMPLETE, 0.5, C.byref(m)) == _lib.GKD_EINVAL
    assert b"null dist" in lib.gkd_last_error(None)


def _run(args):
    p = subprocess.run([GKD] + args, capture_output=True, text=True, timeout=120, stdin=subprocess.DEVNULL)
    return p.returncode, p.stdout, p.stderr


def test_fastadist_method_messages_before_input():
    assert os.path.exists(GKD), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    for method in ("complete", "average", "single"):
        rc, out, err = _run(["fastaDist", "--method", method, "-i", "/nonexistent/in.fa"])
        assert rc == 1 and err.startswith("--method needs --linkage or --clusters.\n"), err
    for bad in ("ward", "", "Complete"):
        rc, out, err = _run(["fastaDist", "--linkage", "--method", bad, "-i", "/nonexistent/in.fa"])
        assert rc == 1 and err.startswith("Linkage method must be single, complete or average.\n"), (bad, err)
    rc, out, err = _run(["fastaDist", "--clusters", "--method", "average", "-i", "/nonexistent/in.fa"])
    assert rc == 1 and err.startswith("--clusters needs --maxDist.\n"), err
    rc, out, err = _run(["fastaDist", "--linkage", "--method", "average", "-i", "/nonexistent/in.fa"])
    assert rc == 1 and "not found or unreadable" in err, err
    rc, out, err = _run(["fastaDist", "--help"])
    assert rc == 0 and "--method" in err and "average" in err
