"""ctypes loader for oracle/libgkd_oracle.so plus a literal pure-Python restatement.

TEST INFRASTRUCTURE ONLY (see oracle/gkd_oracle.h).  PARITY UNPINNED: the reference ships no golden
vectors; the known answers this is pinned to are the hand-derived ones of SURVEY.md section 8(c).

Three restatements of the same contract are kept so they can check each other:
  * ``py_*``      -- Python ``set`` of literal substrings; the most direct reading of
                    ``HashSet<String>`` (reference: KmerCountProcessor.java:76-77); tiny inputs only.
  * ``StrSet``    -- C hash set of literal substrings (Java String.hashCode); timed CPU baseline.
  * ``IntSet``    -- C sorted canonical uint64 keys; the representation the CUDA path uses.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Iterable, List, Sequence, Tuple

import numpy as np

DNA, PROT, RNA = 0, 1, 2
AMBIG_SKIP, AMBIG_LITERAL = 0, 1
_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libgkd_oracle.so")
_lib = None


def build(force: bool = False) -> str:
    """Compile the C oracle (gcc, seconds)."""
    src = os.path.join(_HERE, "gkd_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return _LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(_LIB_PATH)
    vp, sz, u64, i32, dbl = C.c_void_p, C.c_size_t, C.c_uint64, C.c_int, C.c_double
    L.orc_strset_new.restype = vp
    L.orc_strset_new.argtypes = [i32, i32, i32]
    L.orc_strset_add.argtypes = [vp, C.c_char_p, sz]
    L.orc_strset_size.restype = sz
    L.orc_strset_size.argtypes = [vp]
    L.orc_strset_similarity.restype = sz
    L.orc_strset_similarity.argtypes = [vp, vp]
    L.orc_strset_free.argtypes = [vp]
    L.orc_intset_new.restype = vp
    L.orc_intset_new.argtypes = [i32, i32]
    L.orc_intset_add.argtypes = [vp, C.c_char_p, sz]
    L.orc_intset_finish.argtypes = [vp]
    for f in ("orc_intset_count", "orc_intset_palindromes", "orc_intset_size_both"):
        getattr(L, f).restype = sz
        getattr(L, f).argtypes = [vp]
    L.orc_intset_keys.restype = C.POINTER(u64)
    L.orc_intset_keys.argtypes = [vp]
    L.orc_intset_intersect.restype = sz
    L.orc_intset_intersect.argtypes = [vp, vp, C.POINTER(sz)]
    L.orc_intset_free.argtypes = [vp]
    L.orc_dna_canonical.restype = u64
    L.orc_dna_canonical.argtypes = [C.c_char_p, i32, C.POINTER(i32)]
    L.orc_dna_revcomp_key.restype = u64
    L.orc_dna_revcomp_key.argtypes = [u64, i32]
    L.orc_distance.restype = dbl
    L.orc_distance.argtypes = [u64, u64, u64]
    L.orc_double_to_string.argtypes = [dbl, C.c_char_p, sz]
    L.orc_fasta_dist.argtypes = [C.POINTER(C.c_char_p), C.POINTER(sz), sz, i32, i32, i32, i32, i32, i32,
                                 C.POINTER(u64), C.POINTER(dbl)]
    L.orc_query_vs_ref.argtypes = [C.POINTER(C.c_char_p), C.POINTER(sz), sz, C.POINTER(C.c_char_p),
                                   C.POINTER(sz), sz, i32, i32, i32, i32, i32, C.POINTER(u64), C.POINTER(dbl)]
    L.orc_max_threads.restype = i32
    _lib = L
    return L


def _b(s) -> bytes:
    return s if isinstance(s, (bytes, bytearray)) else (s.tobytes() if isinstance(s, np.ndarray) else s.encode("latin-1"))


class StrSet:
    """HashSet<String> analogue (DnaKmers / GenomeKmers / ProteinKmers)."""

    def __init__(self, contigs: Iterable, k: int, alphabet: int = DNA, ambig: int = AMBIG_SKIP):
        self._h = lib().orc_strset_new(alphabet, k, ambig)
        if not self._h:
            raise ValueError("bad k")
        for c in ([contigs] if isinstance(contigs, (str, bytes, np.ndarray)) else contigs):
            b = _b(c)
            if lib().orc_strset_add(self._h, b, len(b)):
                raise MemoryError

    def __len__(self):
        return lib().orc_strset_size(self._h)

    def similarity(self, other: "StrSet") -> int:
        return lib().orc_strset_similarity(self._h, other._h)

    def distance(self, other: "StrSet") -> float:
        return distance(self.similarity(other), len(self), len(other))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_strset_free(self._h)
            self._h = None


class IntSet:
    """Sorted canonical uint64 keys + palindrome count."""

    def __init__(self, contigs: Iterable, k: int, alphabet: int = DNA):
        self.alphabet = alphabet
        self._h = lib().orc_intset_new(alphabet, k)
        if not self._h:
            raise ValueError("bad k")
        for c in ([contigs] if isinstance(contigs, (str, bytes, np.ndarray)) else contigs):
            b = _b(c)
            if lib().orc_intset_add(self._h, b, len(b)):
                raise MemoryError
        lib().orc_intset_finish(self._h)

    @property
    def count(self) -> int:
        return lib().orc_intset_count(self._h)

    @property
    def palindromes(self) -> int:
        return lib().orc_intset_palindromes(self._h)

    def __len__(self):  # the both-strand size the reference's set would have
        return lib().orc_intset_size_both(self._h)

    def keys(self) -> np.ndarray:
        n = self.count
        if n == 0:
            return np.zeros(0, dtype=np.uint64)
        return np.ctypeslib.as_array(lib().orc_intset_keys(self._h), shape=(n,)).copy()

    def intersect(self, other: "IntSet") -> Tuple[int, int]:
        pal = C.c_size_t(0)
        c = lib().orc_intset_intersect(self._h, other._h, C.byref(pal))
        return c, pal.value

    def similarity(self, other: "IntSet") -> int:
        c, pal = self.intersect(other)
        return c if self.alphabet == PROT else 2 * c - pal

    def distance(self, other: "IntSet") -> float:
        return distance(self.similarity(other), len(self), len(other))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_intset_free(self._h)
            self._h = None


def distance(inter: int, size_a: int, size_b: int) -> float:
    return lib().orc_distance(inter, size_a, size_b)


def java_double(v: float) -> str:
    buf = C.create_string_buffer(64)
    lib().orc_double_to_string(v, buf, 64)
    return buf.value.decode()


def _cstr_array(seqs: Sequence):
    bs = [_b(s) for s in seqs]
    arr = (C.c_char_p * len(bs))(*bs)
    lens = (C.c_size_t * len(bs))(*[len(b) for b in bs])
    return bs, arr, lens


def fasta_dist(seqs: Sequence, k: int, alphabet: int = DNA, batch: int = 20, threads: int = 0, mode: int = 0,
               ambig: int = AMBIG_SKIP):
    """FastaDistanceProcessor restatement: (inter, dist) over the strict upper triangle, row-major."""
    n = len(seqs)
    npairs = n * (n - 1) // 2
    keep, arr, lens = _cstr_array(seqs)
    inter = np.zeros(max(npairs, 1), dtype=np.uint64)
    dist = np.zeros(max(npairs, 1), dtype=np.float64)
    rc = lib().orc_fasta_dist(arr, lens, n, alphabet, k, batch, threads, mode, ambig,
                              inter.ctypes.data_as(C.POINTER(C.c_uint64)), dist.ctypes.data_as(C.POINTER(C.c_double)))
    if rc:
        raise MemoryError("oracle fasta_dist failed")
    return inter[:npairs], dist[:npairs]


def query_vs_ref(queries: Sequence, refs: Sequence, k: int, alphabet: int = DNA, threads: int = 0, mode: int = 0,
                 ambig: int = AMBIG_SKIP):
    """GenomeProcessor restatement: (inter, dist) as (nq, nr) arrays."""
    kq, qa, ql = _cstr_array(queries)
    kr, ra, rl = _cstr_array(refs)
    nq, nr = len(queries), len(refs)
    inter = np.zeros(max(nq * nr, 1), dtype=np.uint64)
    dist = np.zeros(max(nq * nr, 1), dtype=np.float64)
    rc = lib().orc_query_vs_ref(qa, ql, nq, ra, rl, nr, alphabet, k, threads, mode, ambig,
                                inter.ctypes.data_as(C.POINTER(C.c_uint64)), dist.ctypes.data_as(C.POINTER(C.c_double)))
    if rc:
        raise MemoryError("oracle query_vs_ref failed")
    return inter[: nq * nr].reshape(nq, nr), dist[: nq * nr].reshape(nq, nr)


def max_threads() -> int:
    return lib().orc_max_threads()


# ----------------------------------------------------------------------------------------------
# literal pure-Python restatement (tiny inputs)
# ----------------------------------------------------------------------------------------------
_COMP = {"a": "t", "c": "g", "g": "c", "t": "a"}


def py_revcomp(s: str) -> str:
    return "".join(_COMP.get(ch, "n") for ch in reversed(s))


def py_kmer_set(contigs, k: int, alphabet: int = DNA, ambig: int = AMBIG_SKIP) -> set:
    """DnaKmers/GenomeKmers (both strands, lower-cased) or ProteinKmers (literal, one strand)."""
    if isinstance(contigs, str):
        contigs = [contigs]
    out = set()
    for seq in contigs:
        if alphabet == PROT:
            strands = [seq]
        else:
            s = seq.lower()
            if alphabet == RNA:
                s = s.replace("u", "t")
            strands = [s, py_revcomp(s)]
        for s in strands:
            for i in range(len(s) - k + 1):
                km = s[i:i + k]
                if alphabet != PROT and ambig == AMBIG_SKIP and any(ch not in "acgt" for ch in km):
                    continue
                out.add(km)
    return out


def py_canonical_set(contigs, k: int, alphabet: int = DNA) -> set:
    """the set GKD_STRAND_CANONICAL counts: min(s, revcomp(s)) of every k-mer of py_kmer_set (lower-case
    lexicographic order is the 2-bit key order a < c < g < t); protein sets are returned as they are"""
    kmers = py_kmer_set(contigs, k, alphabet)
    return kmers if alphabet == PROT else {min(s, py_revcomp(s)) for s in kmers}


def py_distance(a: set, b: set) -> Tuple[int, float]:
    inter = sum(1 for x in b if x in a)
    if inter == 0:
        return 0, 1.0
    return inter, 1.0 - float(inter) / float((len(a) + len(b)) - float(inter))


def parse_fasta(text: str) -> List[Tuple[str, str, str]]:
    """FastaInputStream restatement: (label, comment, sequence) per record.

    label = header up to the first whitespace, comment = remainder (trimmed); sequence lines are
    concatenated with surrounding whitespace removed (FastaDistanceProcessor.java:104-108,189-190).
    """
    recs = []
    label = comment = None
    chunks: List[str] = []
    for line in text.splitlines():
        if line.startswith(">"):
            if label is not None:
                recs.append((label, comment, "".join(chunks)))
            hdr = line[1:].strip()
            parts = hdr.split(None, 1)
            label = parts[0] if parts else ""
            comment = parts[1].strip() if len(parts) > 1 else ""
            chunks = []
        elif label is not None:
            chunks.append(line.strip())
    if label is not None:
        recs.append((label, comment, "".join(chunks)))
    return recs


# ------------------------------------------------------------------------------------------------
# MinHash sketches (SURVEY 8f row 4).  UNPINNED: SequenceKmers.hashSet / Sketch.distance live in the external
# org.theseed.sequence module; restated here as "the `width` smallest distinct hash codes of the set's k-mer
# strings, ascending as Java ints" and the bottom-w estimator, with the string hash as a switch
# (call sites: SketchProcessor.java:91, WidthProcessor.java:177-183, MashProcessor.java:116-150).
# ------------------------------------------------------------------------------------------------
HASH_JAVA_STRING, HASH_MURMUR3 = 0, 1


def _s32(x: int) -> int:
    x &= 0xFFFFFFFF
    return x - (1 << 32) if x & 0x80000000 else x


def java_string_hash(s) -> int:
    """java.lang.String.hashCode of a Latin-1 string, as a signed 32-bit int"""
    h = 0
    for ch in (s.encode("latin-1") if isinstance(s, str) else s):
        h = (31 * h + ch) & 0xFFFFFFFF
    return _s32(h)


def murmur3_32(data, seed: int = 0) -> int:
    """murmur3_x86_32 of the bytes, as a signed 32-bit int"""
    data = data.encode("latin-1") if isinstance(data, str) else bytes(data)
    c1, c2, h, n = 0xCC9E2D51, 0x1B873593, seed & 0xFFFFFFFF, len(data)

    def rotl(x, r):
        return ((x << r) | (x >> (32 - r))) & 0xFFFFFFFF

    for i in range(0, n - n % 4, 4):
        k = int.from_bytes(data[i:i + 4], "little")
        k = (k * c1) & 0xFFFFFFFF
        k = rotl(k, 15)
        k = (k * c2) & 0xFFFFFFFF
        h ^= k
        h = rotl(h, 13)
        h = (h * 5 + 0xE6546B64) & 0xFFFFFFFF
    tail = data[n - n % 4:]
    k = 0
    if len(tail) >= 3:
        k ^= tail[2] << 16
    if len(tail) >= 2:
        k ^= tail[1] << 8
    if len(tail) >= 1:
        k ^= tail[0]
        k = (k * c1) & 0xFFFFFFFF
        k = rotl(k, 15)
        k = (k * c2) & 0xFFFFFFFF
        h ^= k
    h ^= n
    h ^= h >> 16
    h = (h * 0x85EBCA6B) & 0xFFFFFFFF
    h ^= h >> 13
    h = (h * 0xC2B2AE35) & 0xFFFFFFFF
    h ^= h >> 16
    return _s32(h)


def py_hash_set(kmers: set, width: int, kind: int = HASH_JAVA_STRING) -> List[int]:
    """SequenceKmers.hashSet(width) over a literal k-mer string set (py_kmer_set)"""
    fn = java_string_hash if kind == HASH_JAVA_STRING else murmur3_32
    return sorted({fn(k) for k in kmers})[:width]


def py_sketch_distance(a: Sequence[int], b: Sequence[int]) -> float:
    """Sketch.distance: over the w = min(|a|,|b|) smallest codes of the union, m are in both; 1 - m/w"""
    w = min(len(a), len(b))
    if w == 0:
        return 1.0
    i = j = m = 0
    for _ in range(w):
        x, y = a[i], b[j]
        m += x == y
        i, j = i + (x <= y), j + (y <= x)
        if i >= len(a) or j >= len(b):
            break
    return 1.0 - float(m) / float(w)
