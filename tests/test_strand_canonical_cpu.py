"""The canonical strand mode on the CPU: orc.py_canonical_set (the set {min(s, revcomp(s))} that GKD_STRAND_CANONICAL
counts) pinned to the known answers and to orc.IntSet; the input recipes of tests/test_gpu_strand_canonical.py checked
to separate the two modes (so a later change to them cannot make the GPU tests vacuous); and the refusal of the literal
ambiguity policy, which is made before any device is touched."""
import json
import os
import sys

import numpy as np
import pytest

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_gpu_strand_canonical as sc  # noqa: E402  (recipes and threshold choices)

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kat_survey_8c.json")
_CODE = {"a": 0, "c": 1, "g": 2, "t": 3}


def _key(s):
    v = 0
    for ch in s:
        v = (v << 2) | _CODE[ch]
    return v


def test_canonical_set_known_answers(orc):
    with open(GOLD) as f:
        kats = [p for p in json.load(f)["pairs"] if "canonical" in p]
    assert len(kats) == 4
    for p in kats:
        a, b = (orc.py_canonical_set(p[x], p["k"]) for x in "ab")
        assert [len(a), len(b), len(a & b)] == p["canonical"], p["name"]
        oa, ob = orc.IntSet(p["a"], p["k"]), orc.IntSet(p["b"], p["k"])
        assert [oa.count, ob.count, oa.intersect(ob)[0]] == p["canonical"], p["name"]


def _rand(rng, n, letters="acgt"):
    return "".join(rng.choice(list(letters), n))


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6, 8, 11, 12, 16, 21, 22, 32])
def test_canonical_set_equals_intset(orc, k):
    """count, keys in 2-bit order, palindromes and (c, P_I) of IntSet.intersect, on random, mixed-case, N-run, RNA
    and palindromic-word input"""
    rng = np.random.default_rng(40 + k)
    g = _rand(rng, 2000)
    mixed = "".join(ch.upper() if i % 3 == 0 else ch for i, ch in enumerate(_rand(rng, 1500, "acgtnNRy")))
    words = "".join(w.decode() for w in sc.WORDS)
    genomes = [[g], [g[:900].upper() + "n" * 30 + g[900:]], [mixed, "", g[:k - 1]], [words, g[:300]],
               [sc.pal_records()[1].decode()]]
    rna = [g.replace("t", "u")[:1200], mixed.replace("t", "u")]
    cases = [(x, orc.DNA) for x in genomes] + [(rna, orc.RNA)]
    sets = [(orc.py_canonical_set(x, k, al), orc.IntSet(x, k, al)) for x, al in cases]
    for (x, al), (ps, o) in zip(cases, sets):
        assert len(ps) == o.count
        assert np.array_equal(np.array(sorted(_key(s) for s in ps), dtype=np.uint64), o.keys())
        assert sum(s == orc.py_revcomp(s) for s in ps) == o.palindromes
        assert ps == {min(s, orc.py_revcomp(s)) for s in orc.py_kmer_set(x, k, al)}
    for (pa, oa) in sets:
        for (pb, ob) in sets:
            both = pa & pb
            assert oa.intersect(ob) == (len(both), sum(s == orc.py_revcomp(s) for s in both))


def test_protein_sets_are_not_folded(orc):
    s = "MKVLAAGIVGLLLAQWERTY"
    assert orc.py_canonical_set(s, 3, orc.PROT) == orc.py_kmer_set(s, 3, orc.PROT)


@pytest.mark.parametrize("k", [4, 6, 8])
def test_recipes_separate_the_modes(orc, k):
    """the distances of the selection inputs differ between the modes, every threshold lies strictly between the two
    distances of a pair, and the cluster and greedy thresholds change the answer"""
    for seed in (3, 5, 11, 17, 19):
        m = sc.Modes(orc, sc.pal_records(seed), k)
        n = m.n
        differ = np.flatnonzero(m.dc != m.db)
        assert differ.size > n, seed
        ts = sc.between(m.dc, m.db)
        assert len(ts) == 3 and all(t < 1.0 for t in ts)
        lo, hi = np.minimum(m.dc, m.db), np.maximum(m.dc, m.db)
        for t in ts:
            assert ((lo < t) & (t < hi)).any(), (seed, t)
            assert not np.array_equal(m.dc <= t, m.db <= t), (seed, t)
        splits = sc.splitting(n, m.dc, m.db)
        assert splits, seed
        for t in splits:
            assert ((lo < t) & (t < hi)).any()
            assert not np.array_equal(sc.tc._oracle(n, m.dc, t)[0], sc.tc._oracle(n, m.db, t)[0])
        orders = [list(range(n)), list(range(n))[::-1], [int(x) for x in np.random.default_rng(k).permutation(n)]]
        assert any(sc.greedy_splitting(m.DC, m.DB, o) for o in orders), seed
        # canonical distances are I/|C| Jaccard: both-strand I = 2c - P_I exactly
        assert np.array_equal(m.ib, 2 * m.ic - m.PI[m.iu])


def test_odd_k_modes_have_identical_doubles(orc):
    for k in (5, 21):
        m = sc.Modes(orc, sc.pal_records(3), k)
        assert np.array_equal(m.dc.view(np.uint64), m.db.view(np.uint64)) and np.array_equal(m.ib, 2 * m.ic)


def test_dense_inputs_have_palindromes_and_edges(orc):
    genomes = sc.dense_inputs()
    assert any(c == b"" for g in genomes for c in g) and [b""] in genomes
    assert any(ch in c for g in genomes for c in g for ch in (b"N", b"n")) and any(c.isupper() for g in genomes for c in g)
    for k in sc.DIFFERING_K:
        for alphabet in (gkd.DNA, gkd.RNA):
            gs = [sc.to_rna(g) if i % 2 else g for i, g in enumerate(genomes)] if alphabet == gkd.RNA else genomes
            m = sc.Modes(orc, gs, k, alphabet)
            assert (m.dc != m.db).any() and m.PI.any(), (k, alphabet)


def test_literal_policy_is_refused_in_canonical_mode():
    """GKD_AMBIG_LITERAL is defined for the both-strand sets only; protein has no strands"""
    for alphabet in (gkd.DNA, gkd.RNA):
        with pytest.raises(gkd.GkdError) as e:
            gkd.Engine(k=21, alphabet=alphabet, strand_mode=gkd.STRAND_CANONICAL, ambig_policy=gkd.AMBIG_LITERAL)
        assert e.value.code == _lib.GKD_EINVAL
        assert "literal ambiguous k-mers are defined for the both-strand sets only" in e.value.msg
