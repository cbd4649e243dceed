"""Thin Python host layer over the C ABI: device memory plumbing for tests, bench and multi-GPU
sharding.  The product is libgkd.so; nothing here computes."""
from __future__ import annotations

import ctypes as C
from typing import List, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import (AMBIG_LITERAL, AMBIG_SKIP, DNA, PROT, RNA, STRAND_BOTH, STRAND_CANONICAL, GkdConfig, GkdHits,
                   GkdMerges, GkdMetrics, GkdNeighbors, GkdOutputs, GkdPackedSet)

PACKED_DTYPE = np.dtype([("offs_off", "<u8"), ("lows_off", "<u8"), ("pal_offs_off", "<u8"), ("pal_lows_off", "<u8"),
                         ("n", "<u4"), ("n_pal", "<u4"), ("level", "<u4"), ("pal_level", "<u4")])
assert PACKED_DTYPE.itemsize == C.sizeof(GkdPackedSet)


# Selections (gkd_hits) are sized by count-then-fetch: the first call offers room for min(pairs, FIRST_HITS_CAP) hits;
# when the call reports more (n > cap) it is made once more with cap = n.  A selection that keeps few pairs -- the
# use it exists for -- costs one call and host memory for its hits only.
FIRST_HITS_CAP = 1 << 20


def _select(call, pairs: int, cap: int = None):
    """(a, b, inter, dist) numpy arrays of a gkd_hits call `call(hits)` (count-then-fetch, see FIRST_HITS_CAP; a cap
    known to suffice, such as nodes - 1 for a spanning forest, makes it one call)"""
    cap = min(pairs, FIRST_HITS_CAP) if cap is None else cap
    while True:
        a, b = np.empty(cap, dtype=np.uint32), np.empty(cap, dtype=np.uint32)
        inter, dist = np.empty(cap, dtype=np.uint64), np.empty(cap, dtype=np.float64)
        h = GkdHits(a.ctypes.data, b.ctypes.data, inter.ctypes.data, dist.ctypes.data, cap, 0)
        call(h)
        if h.n <= cap:
            n = h.n
            return a[:n], b[:n], inter[:n], dist[:n]
        cap = h.n


def _neighbors(rows: int, k: int):
    """host arrays (pos, inter, dist, n_found) of `rows` k-nearest lists and the gkd_neighbors that points at them"""
    k = max(int(k), 0)
    pos, inter = np.empty((rows, k), dtype=np.uint32), np.empty((rows, k), dtype=np.uint64)
    dist, found = np.empty((rows, k), dtype=np.float64), np.empty(rows, dtype=np.uint32)
    return (pos, inter, dist, found), GkdNeighbors(pos.ctypes.data, inter.ctypes.data, dist.ctypes.data, found.ctypes.data)


def _merges(call, n: int):
    """(a, b, height, size) numpy arrays of a gkd_merges call `call(merges)`; n - 1 entries always suffice"""
    cap = max(int(n) - 1, 0)
    a, b = np.empty(cap, dtype=np.uint32), np.empty(cap, dtype=np.uint32)
    height, size = np.empty(cap, dtype=np.float64), np.empty(cap, dtype=np.uint32)
    m = GkdMerges(a.ctypes.data, b.ctypes.data, height.ctypes.data, size.ctypes.data, cap, 0)
    call(m)
    return a[:m.n], b[:m.n], height[:m.n], size[:m.n]


class GkdError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"gkd error {code}: {msg}")
        self.code = code
        self.msg = msg


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


class Engine:
    """One gkd context on one GPU.

    Mirrors the reference objects at batch granularity: `add` = `KmerType.createKmers` /
    `new GenomeKmers(genome)` / `new ProteinKmers(str)`; `all_vs_all` = FastaDistanceProcessor's pair
    loop; `query_vs_ref` = GenomeProcessor's; `pair` = `SequenceKmers.distance`.
    """

    def __init__(self, k: int = 0, alphabet: int = DNA, strand_mode: int = STRAND_BOTH, device: int = 0,
                 workspace_bytes: int = 0, segment_keys: int = 0, ambig_policy: int = AMBIG_SKIP):
        self._L = _lib.load()
        cfg = GkdConfig(device=device, k=k, alphabet=alphabet, strand_mode=strand_mode,
                        workspace_bytes=workspace_bytes, segment_keys=segment_keys, ambig_policy=ambig_policy)
        h = C.c_void_p()
        rc = self._L.gkd_create(C.byref(h), C.byref(cfg))
        if rc:
            raise GkdError(rc, (self._L.gkd_last_error(None) or b"").decode())
        self._h = h
        self.device = device
        self.alphabet = alphabet
        self._keep: List[object] = []
        self._adopted: List[Tuple[int, object]] = []  # (first id, buffer) of adopted panels

    # -- plumbing ---------------------------------------------------------------------------------
    def _ck(self, rc: int):
        if rc:
            raise GkdError(rc, (self._L.gkd_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            self._L.gkd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @staticmethod
    def _ptr_len(x) -> Tuple[int, int, object]:
        """(address, byte length, keep-alive) of str / bytes / numpy uint8 / torch uint8 (cpu or cuda)."""
        if isinstance(x, str):
            x = x.encode("latin-1")
        if isinstance(x, (bytes, bytearray)):
            buf = C.create_string_buffer(bytes(x), len(x)) if len(x) else C.create_string_buffer(1)
            return C.addressof(buf), len(x), buf
        if isinstance(x, np.ndarray):
            a = np.ascontiguousarray(x).view(np.uint8)
            return a.ctypes.data, a.size, a
        if _is_torch(x):
            t = x.contiguous()
            return t.data_ptr(), t.numel() * t.element_size(), t
        raise TypeError(f"unsupported sequence type {type(x)}")

    # -- ingest ------------------------------------------------------------------------------------
    def add(self, contigs) -> int:
        """Add one genome / record; `contigs` is one sequence or a list of contigs (or proteins)."""
        if isinstance(contigs, (str, bytes, bytearray, np.ndarray)) or _is_torch(contigs):
            contigs = [contigs]
        triples = [self._ptr_len(c) for c in contigs]
        n = len(triples)
        ptrs = (C.c_void_p * max(n, 1))(*[t[0] for t in triples])
        lens = (C.c_uint64 * max(n, 1))(*[t[1] for t in triples])
        out = C.c_uint32()
        if any(_is_torch(c) and c.is_cuda for c in contigs):
            import torch

            torch.cuda.synchronize(self.device)  # producers ran on torch's stream
        self._ck(self._L.gkd_add_sequences(self._h, ptrs, lens, n, C.byref(out)))
        # pinned / device text is read asynchronously and must stay alive until build() (gkd.h)
        self._keep.extend(t[2] for t in triples if _is_torch(t[2]))
        return out.value

    def add_fasta(self, path: str, per_record: bool = True) -> Tuple[int, int]:
        first, n = C.c_uint32(), C.c_uint32()
        self._ck(self._L.gkd_add_fasta_file(self._h, path.encode(), 1 if per_record else 0, C.byref(first), C.byref(n)))
        return first.value, n.value

    def label(self, i: int) -> str:
        return self._L.gkd_label(self._h, i).decode("latin-1")

    def comment(self, i: int) -> str:
        return self._L.gkd_comment(self._h, i).decode("latin-1")

    def __len__(self) -> int:
        return self._L.gkd_count(self._h)

    # -- sets --------------------------------------------------------------------------------------
    def build(self):
        self._ck(self._L.gkd_build_sets(self._h))
        self._keep.clear()

    def set_size(self, i: int) -> Tuple[int, int, int]:
        """(reference HashSet size, canonical count, palindromes)"""
        a, b, p = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._ck(self._L.gkd_set_size(self._h, i, C.byref(a), C.byref(b), C.byref(p)))
        return a.value, b.value, p.value

    def export_set(self, i: int) -> np.ndarray:
        n = self.set_size(i)[1]
        out = np.empty(n, dtype=np.uint64)
        got = C.c_uint64()
        self._ck(self._L.gkd_export_set(self._h, i, out.ctypes.data if n else None, n, C.byref(got)))
        return out

    # -- set exchange (multi-GPU) --------------------------------------------------------------------
    def arenas(self) -> List[Tuple[int, int, int, int]]:
        """[(first_id, n_sets, device address, bytes)] of every live set arena, in id order"""
        out = []
        for a in range(self._L.gkd_arena_count(self._h)):
            first, n, base, nbytes = C.c_uint32(), C.c_uint32(), C.c_void_p(), C.c_uint64()
            self._ck(self._L.gkd_arena_info(self._h, a, C.byref(first), C.byref(n), C.byref(base), C.byref(nbytes)))
            out.append((first.value, n.value, base.value or 0, nbytes.value))
        return out

    def describe_sets(self, first_id: int, n_sets: int) -> np.ndarray:
        """packed layout (PACKED_DTYPE, offsets relative to the arena base) of consecutive sets of one arena"""
        table = np.zeros(n_sets, dtype=PACKED_DTYPE)
        self._ck(self._L.gkd_describe_sets(self._h, first_id, n_sets,
                                           table.ctypes.data_as(C.POINTER(GkdPackedSet))))
        return table

    def arena_meta(self):
        """[(first_id, n_sets, bytes, table)] of every live arena: what sharding.plan_panels consumes"""
        return [(first, n, nbytes, self.describe_sets(first, n)) for first, n, _, nbytes in self.arenas()]

    def arena_view(self, arena: int, begin: int, end: int):
        """zero-copy uint8 torch view of bytes [begin, end) of a set arena on this context's device
        (aliases engine memory: send it, do not write it)"""
        import torch

        base = self.arenas()[arena][2]
        size = max(end - begin, 1)

        class _Raw:
            __cuda_array_interface__ = {"shape": (size,), "typestr": "|u1", "data": (base + begin, False), "version": 3}

        return torch.as_tensor(_Raw(), device=f"cuda:{self.device}")

    def adopt_sets(self, buf, table: np.ndarray) -> int:
        """Register the sets described by `table` whose bytes are in `buf` (uint8 torch tensor on this
        device, e.g. a received panel) WITHOUT copying; `buf` is kept alive until truncate()/reset().
        The bytes must already be there (synchronise with the producer first)."""
        t = np.ascontiguousarray(table, dtype=PACKED_DTYPE)
        out = C.c_uint32()  # the caller has synchronised with whatever filled `buf`
        self._ck(self._L.gkd_adopt_sets(self._h, buf.data_ptr(), buf.numel(), t.ctypes.data_as(C.POINTER(GkdPackedSet)),
                                        t.size, C.byref(out)))
        self._adopted.append((out.value, buf))
        return out.value

    def import_set(self, keys) -> int:
        """Add a set from its key array (numpy uint64 on host or torch int64/uint64 on this device); copied."""
        if isinstance(keys, np.ndarray):
            a = np.ascontiguousarray(keys, dtype=np.uint64)
            ptr, n, keep = a.ctypes.data, a.size, a
        else:
            import torch

            t = keys.contiguous()
            if t.is_cuda:
                torch.cuda.synchronize(self.device)
            ptr, n, keep = t.data_ptr(), t.numel(), t
        out = C.c_uint32()
        self._ck(self._L.gkd_import_set(self._h, ptr if n else None, n, C.byref(out)))
        del keep
        return out.value

    def import_sets(self, keys, offsets) -> int:
        """Add many sets from key arrays stored back to back (`keys`: numpy uint64 or torch int64 tensor,
        host or this device; `offsets`: n+1 host integers).  Returns the id of the first new set."""
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        if isinstance(keys, np.ndarray):
            a = np.ascontiguousarray(keys, dtype=np.uint64)
            ptr, keep = a.ctypes.data, a
        else:
            import torch

            t = keys.contiguous()
            if t.is_cuda:
                torch.cuda.synchronize(self.device)
            ptr, keep = t.data_ptr(), t
        out = C.c_uint32()
        self._ck(self._L.gkd_import_sets(self._h, ptr if int(offs[-1]) else None,
                                         offs.ctypes.data_as(C.POINTER(C.c_uint64)), offs.size - 1, C.byref(out)))
        del keep
        return out.value

    # -- distances ---------------------------------------------------------------------------------
    @staticmethod
    def _outs(n: int, inter_out, dist_out, want_inter: bool, want_dist: bool):
        inter = inter_out if inter_out is not None else (np.empty(n, dtype=np.uint64) if want_inter else None)
        dist = dist_out if dist_out is not None else (np.empty(n, dtype=np.float64) if want_dist else None)

        def addr(x):
            if x is None:
                return None
            return x.ctypes.data if isinstance(x, np.ndarray) else x.data_ptr()

        return inter, dist, addr(inter), addr(dist)

    def all_vs_all(self, inter_out=None, dist_out=None, want_inter=True, want_dist=True):
        n = len(self)
        npairs = n * (n - 1) // 2
        inter, dist, pi, pd = self._outs(npairs, inter_out, dist_out, want_inter, want_dist)
        self._ck(self._L.gkd_all_vs_all(self._h, pi, pd))
        return inter, dist

    def all_vs_all_range(self, n: int, first: int, count: int, inter_out=None, dist_out=None):
        inter, dist, pi, pd = self._outs(count, inter_out, dist_out, True, True)
        self._ck(self._L.gkd_all_vs_all_range(self._h, n, first, count, pi, pd))
        return inter, dist

    def query_vs_ref(self, q: Sequence[int], r: Sequence[int]):
        qa, ra = np.ascontiguousarray(q, dtype=np.uint32), np.ascontiguousarray(r, dtype=np.uint32)
        inter, dist, pi, pd = self._outs(qa.size * ra.size, None, None, True, True)
        self._ck(self._L.gkd_query_vs_ref(self._h, qa.ctypes.data, qa.size, ra.ctypes.data, ra.size, pi, pd))
        return inter.reshape(qa.size, ra.size), dist.reshape(qa.size, ra.size)

    # -- selections: only the chosen pairs leave the device ----------------------------------------------------------
    def all_vs_all_range_within(self, n: int, first: int, count: int, max_dist: float):
        """(a, b, inter, dist) of the pairs [first, first+count) of the triangle over the first n sets whose distance is
        <= max_dist, in enumeration order (a < b are set ids); each entry equals the dense call's"""
        return _select(lambda h: self._ck(self._L.gkd_all_vs_all_range_within(self._h, n, first, count, float(max_dist),
                                                                               C.byref(h))), count)

    def all_vs_all_within(self, max_dist: float):
        n = len(self)
        return self.all_vs_all_range_within(n, 0, n * (n - 1) // 2, max_dist)

    def query_vs_ref_within(self, q: Sequence[int], r: Sequence[int], max_dist: float):
        """(a, b, inter, dist) of the query x reference pairs within max_dist in row-major order; a and b are positions
        in q and r"""
        qa, ra = np.ascontiguousarray(q, dtype=np.uint32), np.ascontiguousarray(r, dtype=np.uint32)
        return _select(lambda h: self._ck(self._L.gkd_query_vs_ref_within(self._h, qa.ctypes.data, qa.size, ra.ctypes.data,
                                                                           ra.size, float(max_dist), C.byref(h))),
                       qa.size * ra.size)

    def query_vs_ref_nearest(self, q: Sequence[int], r: Sequence[int], k: int, max_dist: float, exclude_self: bool = False):
        """(ref_pos, inter, dist, n_found): every query's <= k nearest references within max_dist, as (len(q), k)
        arrays in ascending distance, ties by position in r; unused slots hold ref_pos 2**32-1, inter 0, dist -1.0"""
        qa, ra = np.ascontiguousarray(q, dtype=np.uint32), np.ascontiguousarray(r, dtype=np.uint32)
        slots = qa.size * max(int(k), 0)
        pos, inter = np.empty(slots, dtype=np.uint32), np.empty(slots, dtype=np.uint64)
        dist, found = np.empty(slots, dtype=np.float64), np.empty(qa.size, dtype=np.uint32)
        self._ck(self._L.gkd_query_vs_ref_nearest(self._h, qa.ctypes.data, qa.size, ra.ctypes.data, ra.size, int(k),
                                                  float(max_dist), 1 if exclude_self else 0, pos.ctypes.data,
                                                  inter.ctypes.data, dist.ctypes.data, found.ctypes.data))
        shape = (qa.size, max(int(k), 0))
        return pos.reshape(shape), inter.reshape(shape), dist.reshape(shape), found

    def query_vs_ref_nearest_ex(self, q: Sequence[int], r: Sequence[int], k: int, max_dist: float,
                                exclude_self: bool = False):
        """(q_side, r_side) of one query x reference pass: q_side is query_vs_ref_nearest(q, r, ...), r_side every
        reference's <= k nearest queries (positions in q), equal to query_vs_ref_nearest(r, q, ...); each side is a
        (pos, inter, dist, n_found) tuple"""
        qa, ra = np.ascontiguousarray(q, dtype=np.uint32), np.ascontiguousarray(r, dtype=np.uint32)
        q_side, qn = _neighbors(qa.size, k)
        r_side, rn = _neighbors(ra.size, k)
        self._ck(self._L.gkd_query_vs_ref_nearest_ex(self._h, qa.ctypes.data, qa.size, ra.ctypes.data, ra.size, int(k),
                                                     float(max_dist), 1 if exclude_self else 0, C.byref(qn), C.byref(rn)))
        return q_side, r_side

    def all_vs_all_nearest(self, k: int, max_dist: float, n: int = None):
        """(pos, inter, dist, n_found): each of the first n sets' (default: all) <= k nearest other sets within
        max_dist, as (n, k) arrays in ascending distance, ties by the smaller id; every pair is intersected once.  Equal
        to query_vs_ref_nearest(range(n), range(n), k, max_dist, exclude_self=True)"""
        n = len(self) if n is None else int(n)
        out, nb = _neighbors(n, k)
        self._ck(self._L.gkd_all_vs_all_nearest(self._h, n, int(k), float(max_dist), C.byref(nb)))
        return out

    def all_vs_all_clusters(self, max_dist: float, n: int = None):
        """(labels, n_clusters): single-linkage clusters of the first n sets (default: all) at max_dist, i.e. the
        connected components of the pairs with distance <= max_dist; labels[i] (uint32) is the smallest id of i's
        cluster.  Every pair is intersected once and only the labels leave the device"""
        n = len(self) if n is None else int(n)
        labels, count = np.empty(n, dtype=np.uint32), C.c_uint32()
        self._ck(self._L.gkd_all_vs_all_clusters(self._h, n, float(max_dist), labels.ctypes.data, C.byref(count)))
        return labels, count.value

    def query_vs_ref_clusters(self, q: Sequence[int], r: Sequence[int], max_dist: float):
        """(q_label, r_label): the components of the bipartite graph of the query x reference pairs within max_dist;
        node i is q[i] and node len(q) + j is r[j], and each label is the smallest node of its component"""
        qa, ra = np.ascontiguousarray(q, dtype=np.uint32), np.ascontiguousarray(r, dtype=np.uint32)
        ql, rl = np.empty(qa.size, dtype=np.uint32), np.empty(ra.size, dtype=np.uint32)
        self._ck(self._L.gkd_query_vs_ref_clusters(self._h, qa.ctypes.data, qa.size, ra.ctypes.data, ra.size,
                                                   float(max_dist), ql.ctypes.data, rl.ctypes.data))
        return ql, rl

    def all_vs_all_linkage(self, max_dist: float, n: int = None):
        """(a, b, inter, dist): the single-linkage hierarchy of the first n sets (default: all) up to max_dist, i.e. the
        minimum spanning forest of the pairs within max_dist under the order (distance bits, a, b), in ascending order
        (the merge order of single-linkage agglomeration).  Every pair is intersected once; only the forest leaves the
        device"""
        n = len(self) if n is None else int(n)
        return _select(lambda h: self._ck(self._L.gkd_all_vs_all_linkage(self._h, n, float(max_dist), C.byref(h))),
                       max(n - 1, 0), max(n - 1, 0))

    def query_vs_ref_linkage(self, q: Sequence[int], r: Sequence[int], max_dist: float, q_key=None, r_key=None):
        """(a, b, inter, dist): the forest of one query x reference pass; node i is q[i] and node len(q) + j is r[j], an
        edge reports a = i and b = j.  Ties are broken by the nodes' (min key, max key); keys default to the nodes and
        must be distinct"""
        qa, ra = np.ascontiguousarray(q, dtype=np.uint32), np.ascontiguousarray(r, dtype=np.uint32)
        qk = None if q_key is None else np.ascontiguousarray(q_key, dtype=np.uint32)
        rk = None if r_key is None else np.ascontiguousarray(r_key, dtype=np.uint32)
        if (qk is not None and qk.size != qa.size) or (rk is not None and rk.size != ra.size):
            raise ValueError("q_key / r_key must have one entry per query / reference")
        nodes = max(qa.size + ra.size - 1, 0)
        return _select(lambda h: self._ck(self._L.gkd_query_vs_ref_linkage(
            self._h, qa.ctypes.data, qa.size, ra.ctypes.data, ra.size, float(max_dist),
            None if qk is None else qk.ctypes.data, None if rk is None else rk.ctypes.data, C.byref(h))), nodes, nodes)

    def all_vs_all_agglomerate(self, method: int, max_dist: float, n: int = None):
        """(a, b, height, size): the complete- (LINK_COMPLETE) or average-linkage (LINK_AVERAGE) hierarchy of the first
        n sets (default: all) up to max_dist, one entry per merge in the order of the sequential agglomeration; a < b
        are the smallest ids of the two clusters and size the size of the merged cluster.  Every pair is intersected
        once and its distance stays on the device"""
        n = len(self) if n is None else int(n)
        return _merges(lambda m: self._ck(self._L.gkd_all_vs_all_agglomerate(self._h, n, int(method), float(max_dist),
                                                                             C.byref(m))), n)

    def agglomerate(self, dist, method: int, max_dist: float):
        """all_vs_all_agglomerate over a caller's row-major strict upper triangle of distances (a float64 numpy array
        or CUDA tensor of n(n-1)/2 entries, read and not modified), on this context's device"""
        m = int(dist.numel() if _is_torch(dist) else np.asarray(dist).size)
        n = int(round((1 + (1 + 8 * m) ** 0.5) / 2)) if m else 0
        if n * (n - 1) // 2 != m:
            raise ValueError(f"{m} distances are not a strict upper triangle")
        if _is_torch(dist):
            import torch

            if dist.dtype != torch.float64 or not dist.is_contiguous():
                raise ValueError("dist must be a contiguous float64 tensor")
            ptr, keep = dist.data_ptr(), dist
        else:
            keep = np.ascontiguousarray(dist, dtype=np.float64)
            ptr = keep.ctypes.data
        out = _merges(lambda mg: self._ck(self._L.gkd_agglomerate(self._h, n, ptr, int(method), float(max_dist),
                                                                 C.byref(mg))), n)
        del keep
        return out

    def pairs(self, a: Sequence[int], b: Sequence[int], inter_out=None, dist_out=None):
        aa, ba = np.ascontiguousarray(a, dtype=np.uint32), np.ascontiguousarray(b, dtype=np.uint32)
        inter, dist, pi, pd = self._outs(aa.size, inter_out, dist_out, True, True)
        self._ck(self._L.gkd_pairs(self._h, aa.ctypes.data, ba.ctypes.data, aa.size, pi, pd))
        return inter, dist

    def pairs_ex(self, a: Sequence[int], b: Sequence[int]):
        """(inter, dist, contain_a, contain_b) of an explicit pair list (gkd_pairs_ex)"""
        aa, ba = np.ascontiguousarray(a, dtype=np.uint32), np.ascontiguousarray(b, dtype=np.uint32)
        n = aa.size
        inter, dist = np.empty(n, dtype=np.uint64), np.empty(n, dtype=np.float64)
        ca, cb = np.empty(n, dtype=np.float64), np.empty(n, dtype=np.float64)
        o = GkdOutputs(inter.ctypes.data, dist.ctypes.data, ca.ctypes.data, cb.ctypes.data)
        self._ck(self._L.gkd_pairs_ex(self._h, aa.ctypes.data, ba.ctypes.data, n, C.byref(o)))
        return inter, dist, ca, cb

    # -- MinHash sketches --------------------------------------------------------------------------
    def hash_set(self, i: int, width: int, hash_kind: int = 0) -> np.ndarray:
        """SequenceKmers.hashSet(width): the smallest distinct hash codes of set i, ascending, as int32"""
        out = np.empty(width, dtype=np.int32)
        n = C.c_uint32()
        self._ck(self._L.gkd_hash_set(self._h, i, width, hash_kind, out.ctypes.data, C.byref(n)))
        return out[: n.value].copy()

    def sketch_distances(self, width: int, a: Sequence[int], b: Sequence[int], hash_kind: int = 0) -> np.ndarray:
        """Sketch.distance for a pair list (sketches built and compared on the device)"""
        aa, ba = np.ascontiguousarray(a, dtype=np.uint32), np.ascontiguousarray(b, dtype=np.uint32)
        dist = np.empty(aa.size, dtype=np.float64)
        self._ck(self._L.gkd_sketch_distances(self._h, width, hash_kind, aa.ctypes.data, ba.ctypes.data, aa.size,
                                              dist.ctypes.data))
        return dist

    def greedy_reps(self, order: Sequence[int], max_dist: float) -> np.ndarray:
        """greedy representative pass on the device: flags[i] = 1 iff order[i] became a representative"""
        o = np.ascontiguousarray(order, dtype=np.uint32)
        flags = np.zeros(o.size, dtype=np.uint8)
        self._ck(self._L.gkd_greedy_reps(self._h, o.ctypes.data, o.size, float(max_dist), flags.ctypes.data))
        return flags

    def pair(self, a: int, b: int) -> Tuple[int, int, float]:
        i, u, d = C.c_uint64(), C.c_uint64(), C.c_double()
        self._ck(self._L.gkd_pair(self._h, a, b, C.byref(i), C.byref(u), C.byref(d)))
        return i.value, u.value, d.value

    # -- misc --------------------------------------------------------------------------------------
    def reset(self):
        self._ck(self._L.gkd_reset(self._h))
        self._keep.clear()
        self._adopted.clear()

    @property
    def stream_ptr(self) -> int:
        """cudaStream_t of this context (wrap with torch.cuda.ExternalStream to time on it)"""
        return self._L.gkd_stream(self._h) or 0

    def save_sets(self, path: str):
        """write every set (with label and comment) to a .kset cache file"""
        self._ck(self._L.gkd_save_sets(self._h, path.encode()))

    def load_sets(self, path: str) -> Tuple[int, int]:
        """append the sets of a .kset cache file; returns (first id, count)"""
        first, n = C.c_uint32(), C.c_uint32()
        self._ck(self._L.gkd_load_sets(self._h, path.encode(), C.byref(first), C.byref(n)))
        return first.value, n.value

    def truncate(self, n_keep: int):
        """drop the sets with id >= n_keep (a streamed panel) and recycle their arena"""
        self._ck(self._L.gkd_truncate(self._h, n_keep))
        self._adopted = [x for x in self._adopted if x[0] < n_keep]

    def metrics(self) -> dict:
        m = GkdMetrics()
        self._ck(self._L.gkd_get_metrics(self._h, C.byref(m)))
        return {f: getattr(m, f) for f, _ in GkdMetrics._fields_ if not f.startswith("reserved")}


def format_double(v: float) -> str:
    buf = C.create_string_buffer(64)
    _lib.load().gkd_format_double(v, buf, 64)
    return buf.value.decode()


def synth(dst, seed: int, family: int, member: int, rate: float, protein: bool = False, device: int = 0):
    """Fill `dst` (numpy uint8 array or torch uint8 tensor, host or device) with a synthetic sequence."""
    L = _lib.load()
    if isinstance(dst, np.ndarray):
        ptr, n, dev = dst.ctypes.data, dst.size, -1
    else:
        ptr, n, dev = dst.data_ptr(), dst.numel(), (device if dst.is_cuda else -1)
    fn = L.gkd_synth_protein if protein else L.gkd_synth_dna
    rc = fn(dev, ptr, n, seed, family, member, float(rate))
    if rc:
        raise GkdError(rc, "synth failed")
    return dst


class Group:
    """Several devices in one process behind the C ABI (gkd_group_*): one context per listed device ordinal
    (an ordinal may repeat), one host thread per member, peer copies of set arenas, no reduction."""

    def __init__(self, devices: Sequence[int], k: int = 0, alphabet: int = DNA, strand_mode: int = STRAND_BOTH,
                 workspace_bytes: int = 0, panel: int = 0):
        self._L = _lib.load()
        cfg = GkdConfig(device=0, k=k, alphabet=alphabet, strand_mode=strand_mode, workspace_bytes=workspace_bytes)
        devs = (C.c_int32 * len(devices))(*devices)
        h = C.c_void_p()
        rc = self._L.gkd_group_create(C.byref(h), C.byref(cfg), devs, len(devices))
        if rc:
            raise GkdError(rc, (self._L.gkd_group_last_error(None) or b"").decode())
        self._h = h
        if panel:
            self._ck(self._L.gkd_group_set_panel(self._h, panel))

    def _ck(self, rc: int):
        if rc:
            raise GkdError(rc, (self._L.gkd_group_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            self._L.gkd_group_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __len__(self) -> int:
        return self._L.gkd_group_count(self._h)

    def add(self, member: int, contigs) -> int:
        """one genome on one member (members must be filled in ascending order); returns its global id"""
        if isinstance(contigs, (str, bytes, bytearray, np.ndarray)):
            contigs = [contigs]
        triples = [Engine._ptr_len(c) for c in contigs]
        n = len(triples)
        ptrs = (C.c_void_p * max(n, 1))(*[t[0] for t in triples])
        lens = (C.c_uint64 * max(n, 1))(*[t[1] for t in triples])
        out = C.c_uint32()
        self._ck(self._L.gkd_group_add_sequences(self._h, member, ptrs, lens, n, C.byref(out)))
        return out.value

    def add_fasta(self, path: str) -> int:
        n = C.c_uint32()
        self._ck(self._L.gkd_group_add_fasta_file(self._h, path.encode(), C.byref(n)))
        return n.value

    def label(self, i: int) -> str:
        return self._L.gkd_group_label(self._h, i).decode("latin-1")

    def comment(self, i: int) -> str:
        return self._L.gkd_group_comment(self._h, i).decode("latin-1")

    def build(self):
        self._ck(self._L.gkd_group_build(self._h))

    def all_vs_all(self):
        n = len(self)
        npairs = n * (n - 1) // 2
        inter, dist = np.empty(npairs, dtype=np.uint64), np.empty(npairs, dtype=np.float64)
        self._ck(self._L.gkd_group_all_vs_all(self._h, inter.ctypes.data, dist.ctypes.data))
        return inter, dist

    def all_vs_all_within(self, max_dist: float):
        """(a, b, inter, dist) of the pairs within max_dist over all global ids, ordered by (a, b): the single-context
        Engine.all_vs_all_within result"""
        n = len(self)
        return _select(lambda h: self._ck(self._L.gkd_group_all_vs_all_within(self._h, float(max_dist), C.byref(h))),
                       n * (n - 1) // 2)

    def all_vs_all_nearest(self, k: int, max_dist: float):
        """(pos, inter, dist, n_found) over all global ids: the single-context Engine.all_vs_all_nearest result"""
        out, nb = _neighbors(len(self), k)
        self._ck(self._L.gkd_group_all_vs_all_nearest(self._h, int(k), float(max_dist), C.byref(nb)))
        return out

    def all_vs_all_clusters(self, max_dist: float):
        """(labels, n_clusters) over all global ids: the single-context Engine.all_vs_all_clusters result"""
        labels, count = np.empty(len(self), dtype=np.uint32), C.c_uint32()
        self._ck(self._L.gkd_group_all_vs_all_clusters(self._h, float(max_dist), labels.ctypes.data, C.byref(count)))
        return labels, count.value

    def all_vs_all_linkage(self, max_dist: float):
        """(a, b, inter, dist) over all global ids: the single-context Engine.all_vs_all_linkage result"""
        n = max(len(self) - 1, 0)
        return _select(lambda h: self._ck(self._L.gkd_group_all_vs_all_linkage(self._h, float(max_dist), C.byref(h))), n, n)

    def all_vs_all_agglomerate(self, method: int, max_dist: float):
        """(a, b, height, size) over all global ids: the single-context Engine.all_vs_all_agglomerate result"""
        return _merges(lambda m: self._ck(self._L.gkd_group_all_vs_all_agglomerate(self._h, int(method), float(max_dist),
                                                                                   C.byref(m))), len(self))
