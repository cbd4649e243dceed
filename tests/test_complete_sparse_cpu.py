"""CPU-side checks of complete linkage from the pairs within a distance (gkd_*_complete_linkage): a Python copy of the
sparse rounds of csrc/agglomerate.cu against the exact sequential agglomeration of the dense triangle, on tie-heavy
inputs at every tie value as the threshold, and the argument checks that come before any context or group is used.

`sparse_rounds` follows the device step by step: CSR rows sorted by neighbour, tombstones that keep their neighbour,
the scan / pair / update / finalize rounds.  Its update records, per device thread, the value words it reads and
writes, and fails when two threads of one launch touch one word other than through the barrier between the two phases
of one CTA: the concurrency argument of the update, checked on every input."""
import bisect
import ctypes as C
import os
import random
import sys
from fractions import Fraction

import numpy as np
import pytest

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib
from oracle import agglomerate as agg

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_agglomerate_cpu as tac  # noqa: E402  (the tie-heavy inputs)

TOMB = (1 << 64) - 1


def pairs_within(dist, n, max_dist):
    """(a, b, w) of the condensed triangle's pairs with d <= max_dist, in (a, b) order"""
    w = agg.to_words(dist)
    limit = Fraction(max_dist) * agg.SCALE
    i, j = np.triu_indices(n, 1)
    return [(int(a), int(b), x) for a, b, x in zip(i, j, w) if x <= limit]


class _Launch:
    """the words one kernel launch reads and writes, per thread (cta, phase, entry)"""

    def __init__(self):
        self.reads, self.writes = {}, {}

    def read(self, t, word):
        self.reads.setdefault(word, set()).add(t)

    def write(self, t, word):
        self.writes.setdefault(word, set()).add(t)

    def check(self):
        def ordered(t, u):  # the barrier between the phases of one CTA orders them
            return t[0] == u[0] and t[1] != u[1]

        for word, ws in self.writes.items():
            ws = sorted(ws)
            for x in range(len(ws)):
                for y in range(x + 1, len(ws)):
                    assert ordered(ws[x], ws[y]), ("two threads write", word, ws)
            for r in self.reads.get(word, ()):
                for t in ws:
                    assert r == t or ordered(r, t), ("read of a word another thread writes", word, r, t)


def sparse_rounds(n, pairs, max_dist, rng=None):
    """the device's rounds over the rows of `pairs` ((a, b, w), any order): (merges sorted by key, rounds that merged).
    rng, when given, shuffles the order in which survivors and entries are processed."""
    nbr = [[] for _ in range(n)]
    for a, b, w in sorted([(a, b, w) for a, b, w in pairs] + [(b, a, w) for a, b, w in pairs]):
        nbr[a].append((b, w))
    w_of = [[w for _, w in r] for r in nbr]
    nbr = [[k for k, _ in r] for r in nbr]
    limit = Fraction(max_dist) * agg.SCALE
    size = [1] * n
    nn = [None] * n  # (w, k)
    stale = list(range(n))
    merges, rounds = [], 0

    def find(x, k):
        p = bisect.bisect_left(nbr[x], k)
        return p if p < len(nbr[x]) and nbr[x][p] == k else None

    while True:
        for i in stale:  # scan
            best = None
            for p, k in enumerate(nbr[i]):
                if w_of[i][p] != TOMB and size[k] and (best is None or (w_of[i][p], k) < best):
                    best = (w_of[i][p], k)
            nn[i] = best
        mate = [None] * n  # pair
        surv = []
        for x in range(n):
            if size[x] and nn[x] is not None and nn[nn[x][1]] is not None and nn[nn[x][1]][1] == x and nn[x][0] <= limit:
                mate[x] = nn[x][1]
                if x < mate[x]:
                    merges.append(((nn[x][0], x, mate[x]), x, mate[x], float(Fraction(nn[x][0], agg.SCALE)),
                                   size[x] + size[mate[x]]))
                    surv.append(x)
        if not surv:
            return [m[1:] for m in sorted(merges)], rounds
        rounds += 1
        if rng:
            rng.shuffle(surv)
        launch, pending = _Launch(), []

        def word(t, x, k):
            p = find(x, k)
            if p is None:
                return TOMB
            launch.read(t, (x, p))
            return w_of[x][p]

        def put(t, x, p, v):
            launch.write(t, (x, p))
            pending.append((x, p, v))

        for phase in (1, 2):  # update: every CTA's phase 1, then every CTA's phase 2
            for i in surv:
                j = mate[i]
                row = j if phase == 1 else i
                order = list(range(len(nbr[row])))
                if rng:
                    rng.shuffle(order)
                for e in order:
                    t = (i, phase, e)
                    launch.read(t, (row, e))
                    v = w_of[row][e]
                    if v == TOMB:
                        continue
                    k = nbr[row][e]
                    if phase == 1:
                        if k == i or mate[k] is not None or not size[k]:
                            continue
                        if word(t, i, k) == TOMB:
                            put(t, k, find(k, j), TOMB)
                        continue
                    if k == j:
                        put(t, i, e, TOMB)
                        continue
                    mk = mate[k]
                    if mk is not None:
                        if mk < k:
                            continue
                        put(t, i, e, max(v, word(t, j, k), word(t, i, mk), word(t, j, mk)))
                        continue
                    if not size[k]:
                        continue
                    v = max(v, word(t, j, k))
                    put(t, i, e, v)
                    put(t, k, find(k, i), v)
                    p = find(k, j)
                    if p is not None:
                        put(t, k, p, TOMB)
            for x, p, v in pending:
                w_of[x][p] = v
            pending.clear()
        launch.check()
        for i in surv:
            size[i] += size[mate[i]]
            size[mate[i]] = 0
        stale = [x for x in range(n) if size[x] and (mate[x] is not None or (nn[x] is not None and mate[nn[x][1]] is not None))]


def _ties(d):
    return sorted(set(float(x) for x in d)) + [-1.0]


@pytest.mark.parametrize("seed", range(8))
def test_sparse_rounds_equal_sequential_at_every_tie(seed):
    rng = random.Random(seed)
    n = rng.randint(2, 22)
    d = tac._tie_heavy(rng, n)
    for max_dist in _ties(d):
        want = agg.sequential(d, n, agg.COMPLETE, max_dist)
        pairs = pairs_within(d, n, max_dist)
        got, rounds = sparse_rounds(n, pairs, max_dist)
        assert got == want, (n, max_dist)
        assert got == agg.rnn_rounds(d, n, agg.COMPLETE, max_dist)[0]
        # any processing order, and the pairs in any order, give the same merges
        shuffled = list(pairs)
        rng.shuffle(shuffled)
        assert sparse_rounds(n, shuffled, max_dist, rng)[0] == want


def test_pairs_beyond_the_threshold_change_nothing():
    rng = random.Random(11)
    n = 18
    d = tac._tie_heavy(rng, n)
    every = pairs_within(d, n, 2.0)
    for max_dist in _ties(d):
        assert sparse_rounds(n, every, max_dist)[0] == agg.sequential(d, n, agg.COMPLETE, max_dist), max_dist


def test_one_family_and_a_chain():
    """rows of degree n - 1 (every pair within the threshold), and a mutation chain that takes many rounds"""
    n = 16
    rng = random.Random(3)
    d = np.array([rng.randint(1, 40) / 2.0 ** 53 for _ in range(n * (n - 1) // 2)])
    got, _ = sparse_rounds(n, pairs_within(d, n, 1.0), 1.0)
    assert got == agg.sequential(d, n, agg.COMPLETE, 1.0) and len(got) == n - 1
    full = np.array([[abs(i - j) / 2.0 ** 53 for j in range(n)] for i in range(n)])
    d = full[np.triu_indices(n, 1)]
    for D in (3 / 2.0 ** 53, 7 / 2.0 ** 53, 1.0):
        got, rounds = sparse_rounds(n, pairs_within(d, n, D), D)
        assert got == agg.sequential(d, n, agg.COMPLETE, D)
    assert rounds >= 3


def _merges(cap=4):
    a, b = np.zeros(cap, dtype=np.uint32), np.zeros(cap, dtype=np.uint32)
    h, s = np.zeros(cap, dtype=np.float64), np.zeros(cap, dtype=np.uint32)
    return (a, b, h, s), _lib.GkdMerges(a.ctypes.data, b.ctypes.data, h.ctypes.data, s.ctypes.data, cap, 0)


def test_arguments_are_einval_before_device_use():
    """NaN max_dist, a NULL out, NULL pairs and NULL pair arrays are refused with a message with no context or group
    (and no GPU); arguments that pass reach the NULL-handle check, still GKD_EINVAL."""
    lib = gkd.load()
    keep, m = _merges()
    a, b, d = np.array([0], dtype=np.uint32), np.array([1], dtype=np.uint32), np.array([0.5])
    h = _lib.GkdHits(a.ctypes.data, b.ctypes.data, None, d.ctypes.data, 1, 1)
    calls = {
        "all_vs_all": (lambda D, out: lib.gkd_all_vs_all_complete_linkage(None, 2, D, out), lib.gkd_last_error),
        "list": (lambda D, out: lib.gkd_complete_linkage(None, 2, C.byref(h), D, out), lib.gkd_last_error),
        "group": (lambda D, out: lib.gkd_group_all_vs_all_complete_linkage(None, D, out), lib.gkd_group_last_error),
    }
    for name, (call, err) in calls.items():
        assert call(float("nan"), C.byref(m)) == _lib.GKD_EINVAL, name
        assert b"NaN" in err(None), name
        assert call(0.5, None) == _lib.GKD_EINVAL, name
        assert b"null out" in err(None), name
        for D in (0.5, -1.0, 1.0):
            assert call(D, C.byref(m)) == _lib.GKD_EINVAL, (name, D)
    assert lib.gkd_complete_linkage(None, 2, None, 0.5, C.byref(m)) == _lib.GKD_EINVAL
    assert b"null pairs" in lib.gkd_last_error(None)
    for hole in ("a", "b", "dist"):
        bad = _lib.GkdHits(a.ctypes.data, b.ctypes.data, None, d.ctypes.data, 1, 1)
        setattr(bad, hole, None)
        assert lib.gkd_complete_linkage(None, 2, C.byref(bad), 0.5, C.byref(m)) == _lib.GKD_EINVAL, hole
        assert b"null pair array" in lib.gkd_last_error(None), hole
    # an empty list needs no arrays: it passes the checks and reaches the NULL-handle check
    empty = _lib.GkdHits(None, None, None, None, 0, 0)
    assert lib.gkd_complete_linkage(None, 2, C.byref(empty), 0.5, C.byref(m)) == _lib.GKD_EINVAL
