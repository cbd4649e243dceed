"""Numpy float64 oracle of neighbour joining (gkd_*_nj), and the Newick text `fastaDist --tree` writes.

`nj` is the definition in include/gkd.h: every step is one IEEE double operation in the order written there, so its
rows equal the device's bit for bit.  Clusters are indexed by label (the smallest id) in a full n x n array.
`slot_rounds` is the same computation in the layout the device keeps (the active clusters in a compact prefix of slots,
the last slot moved into the slot g leaves, each pair of the corner scanned once from its smaller slot), kept here so
that the layout can be checked against the definition on the CPU."""
from __future__ import annotations

from typing import List, Tuple

import numpy as np

Row = Tuple[int, int, float, float]  # (a, b, len_a, len_b)


def square(dist, n: int) -> np.ndarray:
    d = np.zeros((n, n))
    i, j = np.triu_indices(n, 1)
    d[i, j] = d[j, i] = np.asarray(dist, dtype=np.float64)
    return d


def start_sums(d: np.ndarray) -> np.ndarray:
    """R_i = (((0 + d(i, 0)) + d(i, 1)) + ...): one sequential sum per row (np.sum would sum pairwise)"""
    R = np.zeros(d.shape[0])
    for k in range(d.shape[0]):
        R = R + d[:, k]
    return R


def _join(d, R, f, g, others, r):
    """the round's branch lengths, and d(u, k), R_k, R_u written into d and R (u takes f's place)"""
    dfg = d[f, g]
    t = (R[f] - R[g]) / np.float64(2 * (r - 2))
    la = np.float64(0.5) * dfg + t
    lb = dfg - la
    du = np.float64(0.5) * ((d[f, others] + d[g, others]) - dfg)
    R[others] = ((R[others] - d[f, others]) - d[g, others]) + du
    R[f] = np.float64(0.5) * ((R[f] + R[g]) - np.float64(r) * dfg)
    d[f, others] = du
    d[others, f] = du
    return float(la), float(lb)


def nj(dist, n: int) -> List[Row]:
    """the rows of the neighbour-joining tree of the condensed triangle `dist` over n records"""
    if n < 2:
        return []
    d = square(dist, n)
    R = start_sums(d)
    active = list(range(n))  # ascending labels
    rows: List[Row] = []
    while len(active) >= 3:
        r = len(active)
        A = np.array(active)
        sub = d[np.ix_(A, A)]
        Q = (np.float64(r - 2) * sub - R[A][:, None]) - R[A][None, :]
        Q[np.tril_indices(r)] = np.inf
        x, y = divmod(int(np.argmin(Q)), r)  # the first minimum in row-major order: the smallest (Q, a, b)
        f, g = active[x], active[y]
        others = np.array([k for k in active if k != f and k != g], dtype=np.int64)
        la, lb = _join(d, R, f, g, others, r)
        rows.append((f, g, la, lb))
        active.remove(g)
    a, b = active
    h = float(np.float64(0.5) * d[a, b])
    rows.append((a, b, h, h))
    return rows


def slot_rounds(dist, n: int) -> List[Row]:
    """nj() in the device's layout: slots 0 .. r - 1 hold the active clusters, label[s] their labels"""
    if n < 2:
        return []
    d = square(dist, n)
    R = start_sums(d)
    label = list(range(n))
    rows: List[Row] = []
    for r in range(n, 2, -1):
        best = None
        for i in range(r - 1):
            for j in range(i + 1, r):
                li, lj = label[i], label[j]
                x = np.float64(r - 2) * d[i, j]
                if li < lj:
                    c = ((x - R[i]) - R[j], li, lj, i, j)
                else:
                    c = ((x - R[j]) - R[i], lj, li, j, i)
                if best is None or c[:3] < best[:3]:
                    best = c
        _, a, b, sf, sg = best
        others = np.array([k for k in range(r) if k != sf and k != sg], dtype=np.int64)
        la, lb = _join(d, R, sf, sg, others, r)
        rows.append((a, b, la, lb))
        last = r - 1
        if sg != last:
            keep = np.array([k for k in range(last) if k != sg], dtype=np.int64)
            d[sg, keep] = d[last, keep]
            d[keep, sg] = d[keep, last]
            R[sg], label[sg] = R[last], label[last]
    h = float(np.float64(0.5) * d[0, 1])
    rows.append((min(label[0], label[1]), max(label[0], label[1]), h, h))
    return rows


_SPECIAL = set("()[]':;,")


def quote(label: str) -> str:
    """a Newick label: single-quoted, with any ' doubled, when it holds whitespace or one of ()[]':;,"""
    if any(ch.isspace() or ch in _SPECIAL for ch in label):
        return "'" + label.replace("'", "''") + "'"
    return label


def newick(rows, labels, fmt) -> str:
    """the tree of the rows as one Newick line: row t is the node (A:len_a,B:len_b) of the current subtrees of labels a
    and b; the last row's node is the root.  fmt formats a length (gkd_format_double); n = 1: `label;`, n = 0: ''"""
    if len(labels) == 0:
        return ""
    sub = {i: quote(x) for i, x in enumerate(labels)}
    for a, b, la, lb in rows:
        sub[int(a)] = "(%s:%s,%s:%s)" % (sub[int(a)], fmt(float(la)), sub.pop(int(b)), fmt(float(lb)))
    return sub[0] + ";\n"
