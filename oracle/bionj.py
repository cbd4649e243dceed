"""Numpy float64 oracle of BIONJ (gkd_*_bionj), Gascuel's variant of neighbour joining (Mol. Biol. Evol. 14:685-695,
1997).

`bionj` is the definition in include/gkd.h: every step is one IEEE double operation in the order written there, so its
rows equal the device's bit for bit.  Clusters are indexed by label (the smallest id) in full n x n arrays d and V.
`bionj_slot_rounds` is the same computation in the layout the device keeps: one n x n array with d(x, y) above the
diagonal and V(x, y) below it, the active clusters in a compact prefix of slots and the last slot moved into the slot g
leaves, so that the packed layout can be checked against the definition on the CPU.
`bionj_textbook` is Gascuel's algorithm as usually stated: the row sums and lambda's sum over the other clusters are
summed directly every round.  It is not bit-exact and serves only to show that the definition is BIONJ."""
from __future__ import annotations

from typing import List, Tuple

import numpy as np

from oracle.nj import Row, square, start_sums


def _lambda(Sf, Sg, vfg, r: int) -> float:
    """0.5 when V(f, g) == 0, else clamp(0.5 + ((S_g - S_f) / ((double)(2 (r - 2)) V(f, g))), 0, 1)"""
    if vfg == 0.0:
        return np.float64(0.5)
    x = np.float64(0.5) + ((np.float64(Sg) - np.float64(Sf)) / (np.float64(2 * (r - 2)) * np.float64(vfg)))
    return np.float64(0.0) if x < 0.0 else np.float64(1.0) if x > 1.0 else x


def _lengths(dfg, Rf, Rg, r: int):
    """NJ's branch lengths"""
    t = (Rf - Rg) / np.float64(2 * (r - 2))
    la = np.float64(0.5) * dfg + t
    return la, dfg - la


def _reduce(lam, la, lb, dfg, vfg, dfk, dgk, vfk, vgk, Rk, Sk, Rf, Rg, Sf, Sg, r: int):
    """the round's d(u, k), V(u, k), R_k, S_k over the other clusters k (arrays), and R_u, S_u"""
    mu = np.float64(1.0) - lam
    w = lam * mu
    du = (lam * (dfk - la)) + (mu * (dgk - lb))
    vu = ((lam * vfk) + (mu * vgk)) - (w * vfg)
    Rk = ((Rk - dfk) - dgk) + du
    Sk = ((Sk - vfk) - vgk) + vu
    rm2 = np.float64(r - 2)
    Ru = (lam * ((Rf - dfg) - rm2 * la)) + (mu * ((Rg - dfg) - rm2 * lb))
    Su = ((lam * (Sf - vfg)) + (mu * (Sg - vfg))) - (rm2 * (w * vfg))
    return du, vu, Rk, Sk, Ru, Su


def bionj(dist, n: int) -> Tuple[List[Row], List[float]]:
    """(rows, lambdas): the rows of the BIONJ tree of the condensed triangle `dist` over n records, and the lambda of
    each round (n - 2 of them)"""
    if n < 2:
        return [], []
    d = square(dist, n)
    V = d.copy()
    R = start_sums(d)
    S = R.copy()
    active = list(range(n))  # ascending labels
    rows: List[Row] = []
    lams: List[float] = []
    while len(active) >= 3:
        r = len(active)
        A = np.array(active)
        Q = (np.float64(r - 2) * d[np.ix_(A, A)] - R[A][:, None]) - R[A][None, :]
        Q[np.tril_indices(r)] = np.inf
        x, y = divmod(int(np.argmin(Q)), r)  # the first minimum in row-major order: the smallest (Q, a, b)
        f, g = active[x], active[y]
        k = np.array([c for c in active if c != f and c != g], dtype=np.int64)
        la, lb = _lengths(d[f, g], R[f], R[g], r)
        lam = _lambda(S[f], S[g], V[f, g], r)
        du, vu, R[k], S[k], R[f], S[f] = _reduce(lam, la, lb, d[f, g], V[f, g], d[f, k], d[g, k], V[f, k], V[g, k], R[k],
                                                 S[k], R[f], R[g], S[f], S[g], r)
        d[f, k] = d[k, f] = du
        V[f, k] = V[k, f] = vu
        rows.append((f, g, float(la), float(lb)))
        lams.append(float(lam))
        active.remove(g)
    a, b = active
    h = float(np.float64(0.5) * d[a, b])
    rows.append((a, b, h, h))
    return rows, lams


def bionj_slot_rounds(dist, n: int) -> Tuple[List[Row], List[float]]:
    """bionj() in the device's layout: D[min, max] = d, D[max, min] = V; slots 0 .. r - 1 hold the active clusters,
    label[s] their labels"""
    if n < 2:
        return [], []
    D = square(dist, n)  # both triangles hold d, so V starts equal to d
    R = start_sums(D)
    S = R.copy()
    label = list(range(n))
    rows: List[Row] = []
    lams: List[float] = []
    for r in range(n, 2, -1):
        best = None
        for i in range(r - 1):  # the scan reads row i from column i + 1 on: the upper triangle, d
            for j in range(i + 1, r):
                li, lj = label[i], label[j]
                x = np.float64(r - 2) * D[i, j]
                c = ((x - R[i]) - R[j], li, lj, i, j) if li < lj else ((x - R[j]) - R[i], lj, li, j, i)
                if best is None or c[:3] < best[:3]:
                    best = c
        _, a, b, sf, sg = best
        lo, hi = min(sf, sg), max(sf, sg)
        dfg, vfg = D[lo, hi], D[hi, lo]
        la, lb = _lengths(dfg, R[sf], R[sg], r)
        lam = _lambda(S[sf], S[sg], vfg, r)
        k = np.array([s for s in range(r) if s != sf and s != sg], dtype=np.int64)
        flo, fhi = np.minimum(sf, k), np.maximum(sf, k)
        glo, ghi = np.minimum(sg, k), np.maximum(sg, k)
        du, vu, R[k], S[k], R[sf], S[sf] = _reduce(lam, la, lb, dfg, vfg, D[flo, fhi], D[glo, ghi], D[fhi, flo],
                                                   D[ghi, glo], R[k], S[k], R[sf], R[sg], S[sf], S[sg], r)
        D[flo, fhi] = du
        D[fhi, flo] = vu
        rows.append((a, b, float(la), float(lb)))
        lams.append(float(lam))
        last = r - 1
        if sg != last:  # d(last, k) from [k, last] into g's upper entry, V(last, k) from [last, k] into its lower one
            keep = np.array([s for s in range(last) if s != sg], dtype=np.int64)
            dv, vv = D[keep, last].copy(), D[last, keep].copy()
            mlo, mhi = np.minimum(sg, keep), np.maximum(sg, keep)
            D[mlo, mhi] = dv
            D[mhi, mlo] = vv
            R[sg], S[sg], label[sg] = R[last], S[last], label[last]
    h = float(np.float64(0.5) * D[0, 1])
    rows.append((min(label[0], label[1]), max(label[0], label[1]), h, h))
    return rows, lams


def bionj_textbook(dist, n: int) -> Tuple[List[Row], List[float]]:
    """Gascuel's BIONJ with direct sums every round: R_i = sum of d(i, k) over the active k, and
    lambda = 1/2 + sum over k != f, g of (V(g, k) - V(f, k)) / (2 (r - 2) V(f, g)), clamped to [0, 1]"""
    if n < 2:
        return [], []
    d = square(dist, n)
    V = d.copy()
    active = list(range(n))
    rows: List[Row] = []
    lams: List[float] = []
    while len(active) >= 3:
        r = len(active)
        A = np.array(active)
        sub = d[np.ix_(A, A)]
        R = sub.sum(axis=1)
        Q = (r - 2) * sub - R[:, None] - R[None, :]
        Q[np.tril_indices(r)] = np.inf
        x, y = divmod(int(np.argmin(Q)), r)
        f, g = active[x], active[y]
        k = np.array([c for c in active if c != f and c != g], dtype=np.int64)
        la = 0.5 * d[f, g] + (R[x] - R[y]) / (2 * (r - 2))
        lb = d[f, g] - la
        if V[f, g] == 0.0:
            lam = 0.5
        else:
            lam = min(1.0, max(0.0, 0.5 + (V[g, k] - V[f, k]).sum() / (2 * (r - 2) * V[f, g])))
        du = lam * (d[f, k] - la) + (1 - lam) * (d[g, k] - lb)
        vu = lam * V[f, k] + (1 - lam) * V[g, k] - lam * (1 - lam) * V[f, g]
        d[f, k] = d[k, f] = du
        V[f, k] = V[k, f] = vu
        rows.append((f, g, float(la), float(lb)))
        lams.append(float(lam))
        active.remove(g)
    a, b = active
    rows.append((a, b, 0.5 * d[a, b], 0.5 * d[a, b]))
    return rows, lams
