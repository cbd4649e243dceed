"""CPU-side checks of neighbour joining (gkd_*_nj): the numpy oracle recovers random additive trees, the slot layout the
device keeps gives the oracle's rows bit for bit on tie-heavy inputs, the argument checks that come before any context
is used, the gkd_joins mirror, and the Newick text of `fastaDist --tree`."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib
from oracle import nj

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- additive trees -----------------------------------------------------------------------------------------------
def _random_tree(rng, n):
    """a random unrooted binary tree over leaves 0 .. n-1 (n >= 3) with dyadic branch lengths: {node: {neighbour: len}}"""
    adj = {0: {}, 1: {}, 2: {}, n: {}}
    for leaf in range(3):
        w = rng.randint(1, 16) / 64.0
        adj[leaf][n] = adj[n][leaf] = w
    nxt = n + 1
    for leaf in range(3, n):
        # split a random edge (x, y) with a new inner node and hang the leaf there
        x = rng.choice(sorted(adj))
        y = rng.choice(sorted(adj[x]))
        w = adj[x].pop(y)
        del adj[y][x]
        cut = rng.randint(1, 15)
        wx = w * cut / 16.0
        m = nxt
        nxt += 1
        adj[m] = {x: wx, y: w - wx}
        adj[x][m], adj[y][m] = wx, w - wx
        adj[leaf] = {m: rng.randint(1, 16) / 64.0}
        adj[m][leaf] = adj[leaf][m]
    return adj


def _path_sums(adj, n):
    d = np.zeros((n, n))
    for s in range(n):
        seen, stack = {s: 0.0}, [s]
        while stack:
            x = stack.pop()
            for y, w in adj[x].items():
                if y not in seen:
                    seen[y] = seen[x] + w
                    stack.append(y)
        for t in range(n):
            d[s, t] = seen[t]
    return d


def _splits_of_tree(adj, n):
    """{frozenset of the side without leaf 0: length} of every edge"""
    out = {}
    for x in adj:
        for y, w in adj[x].items():
            if x < y:
                side, stack = {y}, [y]
                while stack:
                    z = stack.pop()
                    for v in adj[z]:
                        if v not in side and v != x:
                            side.add(v)
                            stack.append(v)
                leaves = frozenset(v for v in side if v < n)
                key = leaves if 0 not in leaves else frozenset(range(n)) - leaves
                out[key] = out.get(key, 0.0) + w
    return out


def _splits_of_rows(rows, n):
    """the same of the rows' tree; the root's two edges are one edge of the unrooted tree"""
    members = {x: frozenset([x]) for x in range(n)}
    out = {}

    def add(leaves, w):
        key = leaves if 0 not in leaves else frozenset(range(n)) - leaves
        out[key] = out.get(key, 0.0) + w

    for a, b, la, lb in rows:
        add(members[a], la)
        add(members[b], lb)
        members[a] = members[a] | members.pop(b)
    return out


@pytest.mark.parametrize("seed", range(8))
def test_oracle_recovers_additive_trees(seed):
    rng = random.Random(seed)
    n = rng.randint(3, 40)
    adj = _random_tree(rng, n)
    d = _path_sums(adj, n)
    rows = nj.nj(d[np.triu_indices(n, 1)], n)
    assert len(rows) == n - 1
    want, got = _splits_of_tree(adj, n), _splits_of_rows(rows, n)
    assert set(got) == set(want)
    for k in want:
        assert abs(got[k] - want[k]) < 1e-9, (k, got[k], want[k])


def test_small_n():
    assert nj.nj(np.zeros(0), 0) == [] and nj.nj(np.zeros(0), 1) == []
    assert nj.nj(np.array([0.75]), 2) == [(0, 1, 0.375, 0.375)]
    # at r = 3 every Q is -(d01 + d02 + d12): the smallest labels join
    assert [r[:2] for r in nj.nj(np.array([0.5, 0.25, 0.125]), 3)] == [(0, 1), (0, 2)]


def test_start_sums_are_sequential():
    """np.sum sums pairwise; the definition sums each row in ascending order"""
    rng = np.random.default_rng(3)
    d = rng.random((300, 300))
    R = nj.start_sums(d)
    for i in (0, 7, 299):
        s = 0.0
        for k in range(300):
            s += float(d[i, k])
        assert R[i] == s


# ---- the device layout ---------------------------------------------------------------------------------------------
def _tie_heavy(rng, n):
    """blocks of identical records (0.0), unrelated ones (1.0) and a few small values"""
    w = np.empty((n, n))
    for i in range(n):
        for j in range(i + 1, n):
            r = rng.random()
            w[i, j] = 0.0 if r < 0.2 else 1.0 if r < 0.6 else rng.randint(1, 6) / 64.0
    blk = rng.randrange(n)
    for i in range(blk, min(n, blk + 5)):
        for j in range(i + 1, min(n, blk + 5)):
            w[i, j] = 0.0
    return w[np.triu_indices(n, 1)]


def _bits(rows):
    return [(a, b, np.float64(x).view(np.uint64), np.float64(y).view(np.uint64)) for a, b, x, y in rows]


@pytest.mark.parametrize("seed", range(10))
def test_slot_layout_equals_oracle_bit_for_bit(seed):
    rng = random.Random(seed)
    n = rng.randint(2, 26)
    for d in (_tie_heavy(rng, n), np.zeros(n * (n - 1) // 2), np.ones(n * (n - 1) // 2),
              np.array([rng.random() for _ in range(n * (n - 1) // 2)])):
        want = nj.nj(d, n)
        assert _bits(nj.slot_rounds(d, n)) == _bits(want), n
        assert len(want) == n - 1
        assert all(a < b for a, b, _, _ in want)


def test_identical_records_join_by_label():
    """every Q ties: the smallest labels join first"""
    rows = nj.nj(np.zeros(10), 5)
    assert [r[:2] for r in rows] == [(0, 1), (0, 2), (0, 3), (0, 4)]
    assert all(x == 0.0 for r in rows for x in r[2:])


# ---- arguments ----------------------------------------------------------------------------------------------------
def test_joins_mirror_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gkd.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu\\n", sizeof(gkd_joins), offsetof(gkd_joins, len_b),'
                   ' offsetof(gkd_joins, cap), offsetof(gkd_joins, n));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    J = _lib.GkdJoins
    assert got == [C.sizeof(J), J.len_b.offset, J.cap.offset, J.n.offset]


def _contextless_engine():
    """an Engine whose context is NULL: its calls reach the checks that come before a context is used"""
    e = gkd.Engine.__new__(gkd.Engine)
    e._L, e._h = gkd.load(), None
    return e


def test_nj_arguments_are_einval_before_device_use():
    lib = gkd.load()
    tri = np.full(3, 0.5)
    assert lib.gkd_nj(None, 3, tri.ctypes.data, None) == _lib.GKD_EINVAL
    assert b"null out" in lib.gkd_last_error(None)
    assert lib.gkd_all_vs_all_nj(None, 3, None) == _lib.GKD_EINVAL
    assert b"null out" in lib.gkd_last_error(None)
    assert lib.gkd_group_all_vs_all_nj(None, None) == _lib.GKD_EINVAL
    assert b"null out" in lib.gkd_group_last_error(None)
    j = _lib.GkdJoins(None, None, None, None, 0, 0)
    assert lib.gkd_nj(None, 3, None, C.byref(j)) == _lib.GKD_EINVAL
    assert b"null dist" in lib.gkd_last_error(None)
    e = _contextless_engine()
    n = 5
    i, k = np.triu_indices(n, 1)
    for bad in (float("nan"), -0.25, 2.5, float("inf")):
        d = np.full(n * (n - 1) // 2, 0.5)
        d[7] = bad
        with pytest.raises(gkd.GkdError, match=r"pair \(%d, %d\) is not a finite value in \[0, 2\]" % (i[7], k[7])):
            e.nj(d)
    # valid values pass the checks and reach the context check, which sets no message
    assert lib.gkd_nj(None, 2, None, None) == _lib.GKD_EINVAL
    with pytest.raises(gkd.GkdError) as err:
        e.nj(np.array([0.0, 2.0, -0.0]))
    assert err.value.code == _lib.GKD_EINVAL and "null out" in err.value.msg
    with pytest.raises(ValueError):
        e.nj(np.zeros(4))


# ---- Newick -------------------------------------------------------------------------------------------------------
def test_newick_label_quoting():
    assert nj.quote("r0001") == "r0001"
    assert nj.quote("NC_000913.3|x") == "NC_000913.3|x"
    assert nj.quote("a b") == "'a b'"
    assert nj.quote("a\tb") == "'a\tb'"
    for ch in "()[]':;,":
        assert nj.quote("x%sy" % ch) == "'x%sy'" % (ch * 2 if ch == "'" else ch)
    assert nj.quote("it's") == "'it''s'"


def _parse(text):
    """a small Newick parser: (tree, rest) with tree = label or [(subtree, length), (subtree, length)]"""
    assert text.endswith(";\n")
    s, pos = text[:-2], 0

    def label():
        nonlocal pos
        if s[pos] == "'":
            out, pos = [], pos + 1
            while True:
                if s[pos] == "'" and s[pos + 1:pos + 2] == "'":
                    out.append("'")
                    pos += 2
                elif s[pos] == "'":
                    pos += 1
                    return "".join(out)
                else:
                    out.append(s[pos])
                    pos += 1
        start = pos
        while pos < len(s) and s[pos] not in "():,;":
            pos += 1
        return s[start:pos]

    def node():
        nonlocal pos
        if s[pos] != "(":
            return label()
        pos += 1
        kids = []
        while True:
            sub = node()
            assert s[pos] == ":"
            pos += 1
            start = pos
            while s[pos] not in ",)":
                pos += 1
            kids.append((sub, float(s[start:pos])))
            if s[pos] == ")":
                pos += 1
                return kids
            pos += 1

    tree = node()
    assert pos == len(s)
    return tree


def _leaves(tree):
    return [tree] if isinstance(tree, str) else [x for sub, _ in tree for x in _leaves(sub)]


@pytest.mark.parametrize("seed", range(4))
def test_newick_round_trips(seed):
    rng = random.Random(seed)
    n = rng.randint(3, 30)
    adj = _random_tree(rng, n)
    d = _path_sums(adj, n)
    rows = nj.nj(d[np.triu_indices(n, 1)], n)
    labels = ["r%d" % i for i in range(n)]
    labels[1], labels[2] = "with space", "it's (odd):[x],y;"
    text = nj.newick(rows, labels, repr)
    assert text.count("\n") == 1
    tree = _parse(text)
    assert sorted(_leaves(tree)) == sorted(labels)
    # the lengths read back are the rows' lengths, node by node
    members = {x: labels[x] for x in range(n)}
    for a, b, la, lb in rows:
        members[a] = [(members[a], la), (members.pop(b), lb)]
    assert tree == members[0]


def test_newick_small():
    assert nj.newick([], [], repr) == ""
    assert nj.newick([], ["only one"], repr) == "'only one';\n"
    assert nj.newick([(0, 1, 0.25, 0.25)], ["a", "b"], gkd.format_double) == "(a:0.25,b:0.25);\n"
