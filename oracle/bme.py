"""Python float oracle of the balanced minimum-evolution (BME) NNI search (gkd_*_bme, gkd_bme_nni).

`bme_nni` is the definition in include/gkd.h: every Delta is one IEEE double operation per step, in the order written
there, and the whole table is recomputed from scratch after every swap, so its rows are what the device's incremental
update must equal bit for bit.  `direct_delta` and `pauplin_length` are the closed forms (path weights 2^-depth, and
Pauplin's length sum 2^(1 - tau_ij) d_ij) used only to show that the definition is BME.

A tree is held rooted at the midpoint of its root edge: nodes 0 .. n - 1 are the leaves, row t of the rows builds node
n + t, and the last row's node (2n - 2) is the root, whose two children c0, c1 are the root edge's ends.  A side is
(v, 0), the leaves below v, or (v, 1), the leaves above v; (c, 1) for a root child c is the side (sibling of c, 0).
An NNI at the edge above v swaps one child of v with v's sibling; at the root edge one child of c0 with one of c1.
The edge towards the root is never moved, so the root edge stays the edge between c0 and c1."""
from __future__ import annotations

import sys
from typing import Dict, List, Tuple

import numpy as np

from oracle.nj import Row, square

EPS = 2.0 ** -40  # GKD_BME_EPS: a swap is taken only when its gain exceeds this


def max_swaps(n: int) -> int:
    """GKD_BME_MAX_SWAPS(n)"""
    return 4 * n


class Tree:
    """the binary tree of gkd_joins rows (only a and b are read)"""

    def __init__(self, n: int, rows):
        self.n = n
        self.root = 2 * n - 2
        self.par = [-1] * (2 * n - 1)
        self.kids: List[List[int]] = [[] for _ in range(2 * n - 1)]
        cur = list(range(n))
        for t, r in enumerate(rows):
            a, b = int(r[0]), int(r[1])
            v = n + t
            self.kids[v] = [cur[a], cur[b]]
            self.par[cur[a]] = self.par[cur[b]] = v
            cur[a] = v
        self._cache()

    def _cache(self):
        self._size: Dict = {}
        self._label: Dict = {}

    def leaf(self, v: int) -> bool:
        return v < self.n

    def sib(self, v: int) -> int:
        k = self.kids[self.par[v]]
        return k[1] if k[0] == v else k[0]

    def canon(self, s):
        v, up = s
        if up and self.par[v] == self.root:
            return (self.sib(v), 0)
        return s

    def children(self, s):
        """the two child sides of a non-leaf side, in label order"""
        v, up = s
        if up:
            c = [(self.sib(v), 0), self.canon((self.par[v], 1))]
        else:
            c = [(k, 0) for k in self.kids[v]]
        return sorted(c, key=self.label)

    def is_leaf_side(self, s) -> bool:
        return s[1] == 0 and self.leaf(s[0])

    def size(self, s) -> int:
        if s not in self._size:
            self._size[s] = 1 if self.is_leaf_side(s) else sum(self.size(c) for c in self.children(s))
        return self._size[s]

    def label(self, s) -> int:
        if s not in self._label:
            self._label[s] = s[0] if self.is_leaf_side(s) else min(self.label(c) for c in self.children(s))
        return self._label[s]

    def leaves(self, s) -> List[Tuple[int, int]]:
        """(leaf, depth below the side's attachment) of every leaf of the side"""
        if self.is_leaf_side(s):
            return [(s[0], 0)]
        return [(x, k + 1) for c in self.children(s) for x, k in self.leaves(c)]

    def edges(self):
        """the internal edges as (where, [[x1, x2], [y1, y2]]): where is v for the edge above v, or 'root'"""
        out = []
        c0, c1 = self.kids[self.root]
        for v in range(self.n, self.root):
            if self.par[v] != self.root:
                out.append((v, [[(k, 0) for k in self.kids[v]], [(self.sib(v), 0), self.canon((self.par[v], 1))]]))
        if not self.leaf(c0) and not self.leaf(c1):
            out.append(("root", [[(k, 0) for k in self.kids[c0]], [(k, 0) for k in self.kids[c1]]]))
        return out

    def name(self, groups):
        """A, B, C, D: A the side of the smallest label, B its partner, C and D the other two in label order"""
        g0, g1 = groups
        if min(self.label(s) for s in g1) < min(self.label(s) for s in g0):
            g0, g1 = g1, g0
        A, B = sorted(g0, key=self.label)
        C, D = sorted(g1, key=self.label)
        return A, B, C, D

    def swap(self, where, groups, partner_of_x1):
        """make the split in which the first side of groups[0] is paired with partner_of_x1"""
        (x1, x2), (y1, y2) = groups
        if where == "root":
            self._exchange(x2[0], y1[0] if partner_of_x1 == y1 else y2[0])
        else:  # y1 is v's sibling; the side above v's parent stays
            self._exchange(x2[0] if partner_of_x1 == y1 else x1[0], y1[0])
        self._cache()

    def _exchange(self, a: int, b: int):
        pa, pb = self.par[a], self.par[b]
        self.kids[pa][self.kids[pa].index(a)] = b
        self.kids[pb][self.kids[pb].index(b)] = a
        self.par[a], self.par[b] = pb, pa


class Table:
    """Delta of the definition over one tree, memoised (the table recomputed from scratch)"""

    def __init__(self, tree: Tree, d: np.ndarray):
        self.t, self.d = tree, d
        self.memo: Dict = {}

    def __call__(self, X, Y) -> float:
        t = self.t
        X, Y = t.canon(X), t.canon(Y)
        key = (X, Y) if X < Y else (Y, X)
        v = self.memo.get(key)
        if v is not None:
            return v
        if t.is_leaf_side(X) and t.is_leaf_side(Y):
            v = float(self.d[X[0], Y[0]])
        else:
            Z, W = (X, Y) if (t.size(X), t.label(X)) > (t.size(Y), t.label(Y)) else (Y, X)
            z1, z2 = t.children(Z)
            v = 0.5 * (self(z1, W) + self(z2, W))
        self.memo[key] = v
        return v


def gains(tree: Tree, D) -> List[Tuple[float, int, int, int, object, list]]:
    """(gain, key label, key size, swap, where, groups) of both swaps at every internal edge; swap 0 exchanges B and C,
    swap 1 B and D"""
    out = []
    for where, groups in tree.edges():
        A, B, C, Dd = tree.name(groups)
        ab_cd = D(A, B) + D(C, Dd)
        g0 = 0.25 * (ab_cd - (D(A, C) + D(B, Dd)))
        g1 = 0.25 * (ab_cd - (D(A, Dd) + D(B, C)))
        key = (tree.label(C), tree.size(C) + tree.size(Dd))
        out.append((g0, key[0], key[1], 0, where, groups))
        out.append((g1, key[0], key[1], 1, where, groups))
    return out


def best(cands):
    """the largest gain; ties to the smaller edge key, then to swap 0"""
    return min(cands, key=lambda c: (-c[0], c[1], c[2], c[3])) if cands else None


def apply(tree: Tree, c):
    g, _, _, sw, where, groups = c
    A, B, C, Dd = tree.name(groups)
    pairs = [{A, C}, {B, Dd}] if sw == 0 else [{A, Dd}, {B, C}]  # the new split
    x1 = groups[0][0]
    partner = next(iter((p - {x1}) for p in pairs if x1 in p)).pop()
    tree.swap(where, groups, partner)


def lengths(tree: Tree, D) -> Dict:
    """{v: length of the edge above v} for every non-root node but the root children, and 'root': the root edge"""
    out = {}
    c0, c1 = tree.kids[tree.root]

    def internal(groups):
        A, B, C, Dd = tree.name(groups)
        return 0.25 * (((D(A, C) + D(A, Dd)) + D(B, C)) + D(B, Dd)) - 0.5 * (D(A, B) + D(C, Dd))

    def pendant(i):
        A, B = tree.children(tree.canon((i, 1)))
        return 0.5 * ((D((i, 0), A) + D((i, 0), B)) - D(A, B))

    for v in range(tree.root):
        if tree.par[v] == tree.root:
            continue
        if tree.leaf(v):
            out[v] = pendant(v)
        else:
            out[v] = internal([[(k, 0) for k in tree.kids[v]], [(tree.sib(v), 0), tree.canon((tree.par[v], 1))]])
    if tree.leaf(c0) and tree.leaf(c1):
        out["root"] = float(D((c0, 0), (c1, 0)))
    elif tree.leaf(c1) or tree.leaf(c0):
        out["root"] = pendant(c1 if tree.leaf(c1) else c0)
    else:
        out["root"] = internal([[(k, 0) for k in tree.kids[c0]], [(k, 0) for k in tree.kids[c1]]])
    return out


def rows_of(tree: Tree, ln: Dict) -> List[Row]:
    """the post-order rows: the child of the smaller label first, the root row (a, b, l/2, l/2) last"""
    rows: List[Row] = []
    lab = lambda v: tree.label((v, 0))  # noqa: E731

    def emit(v):
        if tree.leaf(v):
            return
        k = sorted(tree.kids[v], key=lab)
        emit(k[0])
        emit(k[1])
        rows.append((lab(k[0]), lab(k[1]), float(ln[k[0]]), float(ln[k[1]])))

    k = sorted(tree.kids[tree.root], key=lab)
    emit(k[0])
    emit(k[1])
    h = 0.5 * ln["root"]
    rows.append((lab(k[0]), lab(k[1]), h, h))
    return rows


def bme_nni(dist, n: int, start_rows, cap: int = None) -> Tuple[List[Row], int]:
    """(rows, swaps): the BME NNI search from the tree of start_rows over the condensed triangle dist"""
    if n < 2:
        return [], 0
    sys.setrecursionlimit(max(sys.getrecursionlimit(), 20 * n + 1000))
    cap = max_swaps(n) if cap is None else cap
    d = square(dist, n)
    tree = Tree(n, start_rows)
    swaps = 0
    while swaps < cap:
        c = best(gains(tree, Table(tree, d)))
        if c is None or not c[0] > EPS:
            break
        apply(tree, c)
        swaps += 1
    return rows_of(tree, lengths(tree, Table(tree, d))), swaps


def bme(dist, n: int, start: str = "bionj", cap: int = None) -> Tuple[List[Row], int]:
    """gkd_bme: the search from the NJ or BIONJ tree"""
    from oracle import bionj, nj

    rows = nj.nj(dist, n) if start == "nj" else bionj.bionj(dist, n)[0]
    return bme_nni(dist, n, rows, cap)


# ---- closed forms, used only to show that the definition is BME ----------------------------------------------------


def direct_delta(tree: Tree, d: np.ndarray, X, Y) -> float:
    """sum over x in X, y in Y of 2^-(depth x + depth y) d(x, y)"""
    return float(sum(2.0 ** -(i + j) * d[x, y] for x, i in tree.leaves(tree.canon(X)) for y, j in tree.leaves(tree.canon(Y))))


def pauplin_length(tree: Tree, d: np.ndarray) -> float:
    """Pauplin's balanced tree length: the sum over leaf pairs of 2^(1 - tau_ij) d_ij, tau_ij the edges between them"""
    n = tree.n
    adj: Dict[int, List[int]] = {v: [] for v in range(2 * n - 1)}
    for v in range(2 * n - 2):
        if tree.par[v] >= 0:
            adj[v].append(tree.par[v])
            adj[tree.par[v]].append(v)
    c0, c1 = tree.kids[tree.root]  # the root is not a node of the unrooted tree
    adj[c0] = [x for x in adj[c0] if x != tree.root] + [c1]
    adj[c1] = [x for x in adj[c1] if x != tree.root] + [c0]
    total = 0.0
    for i in range(n):
        dep = {i: 0}
        stack = [i]
        while stack:
            u = stack.pop()
            for w in adj[u]:
                if w != tree.root and w not in dep:
                    dep[w] = dep[u] + 1
                    stack.append(w)
        for j in range(i + 1, n):
            total += 2.0 ** (1 - dep[j]) * d[i, j]
    return total


def tree_splits(tree: Tree) -> set:
    """the nontrivial splits, each as the frozenset of the side without leaf 0"""
    n = tree.n
    full = frozenset(range(n))
    out = set()
    for v in range(n, tree.root):
        s = frozenset(x for x, _ in tree.leaves((v, 0)))
        s = full - s if 0 in s else s
        if 1 < len(s) < n - 1:
            out.add(s)
    return out
