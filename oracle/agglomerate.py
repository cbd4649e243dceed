"""Exact pure-Python oracle of complete- and average-linkage agglomeration (gkd_*_agglomerate).

Distances are integer multiples of 2^-53 (every value SequenceKmers.distance can take), so a cluster distance is held
exactly: complete = the max of w = d * 2^53, average = S / (|A| |B|) with S the integer sum of w.  Pairs of current
clusters are ranked by the strict key (v, min label, max label); a cluster's label is its smallest id.

`sequential` is the definition: repeatedly merge the pair with the smallest key while v <= max_dist.  `rnn_rounds` is the
parallel reciprocal-nearest-neighbour form the device runs, kept here so that the equivalence can be checked on the
CPU; it returns the same merges and its number of rounds."""
from __future__ import annotations

from fractions import Fraction
from typing import List, Tuple

import numpy as np

COMPLETE, AVERAGE = 1, 2
SCALE = 1 << 53

Merge = Tuple[int, int, float, int]  # (a, b, height, size)


def pair_result(inter: int, size_a: int, size_b: int) -> float:
    """SequenceKmers.distance from I, |A| and |B| (kernel 5's formula: a Java int sum, then double arithmetic)"""
    if inter <= 0:
        return 1.0
    s = (size_a + size_b) & 0xFFFFFFFF
    s = s - (1 << 32) if s >= 1 << 31 else s
    return 1.0 - float(inter) / (float(s) - float(inter))


def to_words(dist) -> List[int]:
    """d * 2^53 of every entry, as exact integers; ValueError for a value that is not a multiple of 2^-53 in [0, 2]"""
    out = []
    for d in np.asarray(dist, dtype=np.float64).tolist():
        w = Fraction(d) * SCALE
        if not (0 <= d <= 2) or w.denominator != 1:
            raise ValueError(f"distance {d!r} is not a multiple of 2^-53 in [0, 2]")
        out.append(int(w))
    return out


def height(s: int, n: int) -> float:
    """S / (N 2^53) rounded to the nearest double, ties to even"""
    return float(Fraction(s, n * SCALE))


def _value(method: int, e: int, size_a: int, size_b: int) -> Fraction:
    return Fraction(e) if method == COMPLETE else Fraction(e, size_a * size_b)


def _setup(dist, n: int):
    w = to_words(dist)
    if len(w) != n * (n - 1) // 2:
        raise ValueError("dist is not the strict upper triangle of n")
    e = [[0] * n for _ in range(n)]
    t = 0
    for i in range(n):
        for j in range(i + 1, n):
            e[i][j] = e[j][i] = w[t]
            t += 1
    return e


def _merge(method: int, e, i: int, j: int, active):
    for k in active:
        if k != i and k != j:
            v = max(e[i][k], e[j][k]) if method == COMPLETE else e[i][k] + e[j][k]
            e[i][k] = e[k][i] = v


def _limit(max_dist: float) -> Fraction:
    return Fraction(max_dist) * SCALE


def sequential(dist, n: int, method: int, max_dist: float, values: list = None) -> List[Merge]:
    """the sequential agglomeration of the condensed triangle `dist` over n records, up to max_dist; `values`, when
    given, receives every merge's exact value v * 2^53 (a Fraction)"""
    e = _setup(dist, n)
    size = [1] * n
    active = list(range(n))
    limit = _limit(max_dist)
    out: List[Merge] = []
    while len(active) > 1:
        best = None
        for x in range(len(active)):
            i = active[x]
            for j in active[x + 1:]:
                key = (_value(method, e[i][j], size[i], size[j]), i, j)
                if best is None or key < best:
                    best = key
        v, i, j = best
        if v > limit:
            break
        out.append((i, j, float(v / SCALE), size[i] + size[j]))
        if values is not None:
            values.append(v)
        _merge(method, e, i, j, active)
        size[i] += size[j]
        active.remove(j)
    return out


def rnn_rounds(dist, n: int, method: int, max_dist: float) -> Tuple[List[Merge], int]:
    """the reciprocal-nearest-neighbour rounds of the device engine: (merges sorted by key, rounds that merged)"""
    e = _setup(dist, n)
    size = [1] * n
    active = set(range(n))
    limit = _limit(max_dist)
    merges = []
    rounds = 0
    while True:
        nn = {}
        for i in active:
            best = None
            for k in active:
                if k != i:
                    key = (_value(method, e[i][k], size[i], size[k]), k)
                    if best is None or key < best:
                        best = key
            nn[i] = best
        pairs = [(i, nn[i][1], nn[i][0]) for i in active
                 if nn[i] is not None and i < nn[i][1] and nn[nn[i][1]][1] == i and nn[i][0] <= limit]
        if not pairs:
            return [m[1:] for m in sorted(merges)], rounds
        rounds += 1
        mate = {}
        for i, j, _ in pairs:
            mate[i], mate[j] = j, i
        new = {}
        for i, j, v in pairs:
            merges.append(((v, i, j), i, j, float(v / SCALE), size[i] + size[j]))
            for k in active:
                if k in (i, j) or (k in mate and mate[k] < k):
                    continue
                if k in mate:  # another survivor: all four entries of the two merging pairs
                    parts = [e[i][k], e[j][k], e[i][mate[k]], e[j][mate[k]]]
                else:
                    parts = [e[i][k], e[j][k]]
                new[(i, k)] = max(parts) if method == COMPLETE else sum(parts)
        for (i, k), v in new.items():
            e[i][k] = e[k][i] = v
        for i, j, _ in pairs:
            size[i] += size[j]
            active.remove(j)


def prefix(merges: List[Merge], values: list, max_dist: float) -> List[Merge]:
    """the agglomeration up to max_dist from a longer one: its merges with exact value <= max_dist (they come first)"""
    limit = _limit(max_dist)
    return [m for m, v in zip(merges, values) if v <= limit]


def labels(merges, n: int, t=None, exact=None) -> List[int]:
    """the smallest id of every record's cluster after the merges (those with height <= t when t is given; `exact`
    is then a list of the merges' exact values to test instead of the rounded heights)"""
    root = list(range(n))

    def find(x):
        while root[x] != x:
            x = root[x]
        return x

    for idx, (a, b, h, _) in enumerate(merges):
        if t is not None and (exact[idx] if exact is not None else h) > t:
            continue
        x, y = find(a), find(b)
        root[max(x, y)] = min(x, y)
    return [find(x) for x in range(n)]
