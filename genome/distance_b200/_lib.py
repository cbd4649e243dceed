"""ctypes binding of libgkd.so (include/gkd.h).  Fails loudly when the CUDA library is missing:
there is no CPU fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GKD_LIB") or os.path.join(_HERE, "libgkd.so")  # GKD_LIB: tuning builds only

GKD_OK, GKD_EINVAL, GKD_EIO, GKD_ENOMEM, GKD_ECUDA, GKD_ESTATE = 0, -1, -2, -3, -4, -5
DNA, PROT, RNA = 0, 1, 2
STRAND_BOTH, STRAND_CANONICAL = 0, 1
AMBIG_SKIP, AMBIG_LITERAL = 0, 1
HASH_JAVA_STRING, HASH_MURMUR3 = 0, 1
LINK_COMPLETE, LINK_AVERAGE = 1, 2
ABI_VERSION = 2


class GkdConfig(C.Structure):
    _fields_ = [("device", C.c_int32), ("k", C.c_int32), ("alphabet", C.c_int32), ("strand_mode", C.c_int32),
                ("workspace_bytes", C.c_uint64), ("segment_keys", C.c_uint32), ("ambig_policy", C.c_int32),
                ("reserved", C.c_uint32 * 6)]


class GkdPackedSet(C.Structure):
    _fields_ = [("offs_off", C.c_uint64), ("lows_off", C.c_uint64), ("pal_offs_off", C.c_uint64),
                ("pal_lows_off", C.c_uint64), ("n", C.c_uint32), ("n_pal", C.c_uint32), ("level", C.c_uint32),
                ("pal_level", C.c_uint32)]


class GkdOutputs(C.Structure):
    _fields_ = [("inter", C.c_void_p), ("dist", C.c_void_p), ("contain_a", C.c_void_p), ("contain_b", C.c_void_p)]


class GkdHits(C.Structure):
    _fields_ = [("a", C.c_void_p), ("b", C.c_void_p), ("inter", C.c_void_p), ("dist", C.c_void_p), ("cap", C.c_uint64),
                ("n", C.c_uint64)]


class GkdMerges(C.Structure):
    _fields_ = [("a", C.c_void_p), ("b", C.c_void_p), ("height", C.c_void_p), ("size", C.c_void_p), ("cap", C.c_uint64),
                ("n", C.c_uint64)]


class GkdNeighbors(C.Structure):
    _fields_ = [("pos", C.c_void_p), ("inter", C.c_void_p), ("dist", C.c_void_p), ("n_found", C.c_void_p)]


class GkdMetrics(C.Structure):
    _fields_ = [("pack_ms", C.c_double), ("encode_ms", C.c_double), ("sort_ms", C.c_double), ("unique_ms", C.c_double),
                ("intersect_ms", C.c_double), ("epilogue_ms", C.c_double), ("h2d_ms", C.c_double), ("d2h_ms", C.c_double),
                ("residues_packed", C.c_uint64), ("kmer_positions", C.c_uint64), ("keys_sorted", C.c_uint64),
                ("sort_passes", C.c_uint32), ("intersect_kernel", C.c_uint32), ("keys_unique", C.c_uint64), ("pairs", C.c_uint64),
                ("intersect_bytes", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("launches", C.c_uint64), ("intersect_launches", C.c_uint64), ("total_pairs", C.c_uint64),
                ("total_intersect_bytes", C.c_uint64), ("total_intersect_ms", C.c_double), ("agglomerate_rounds", C.c_uint64),
                ("reserved", C.c_uint64 * 2)]


# every symbol include/gkd.h declares: name -> (restype, argtypes)
_vp, _u32, _u64, _i32, _dbl = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int, C.c_double
_pu32, _pu64, _pdbl = C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_double)
SYMBOLS = {
    "gkd_abi_version": (_i32, []),
    "gkd_create": (_i32, [C.POINTER(_vp), C.POINTER(GkdConfig)]),
    "gkd_destroy": (_i32, [_vp]),
    "gkd_reset": (_i32, [_vp]),
    "gkd_truncate": (_i32, [_vp, _u32]),
    "gkd_last_error": (C.c_char_p, [_vp]),
    "gkd_add_sequences": (_i32, [_vp, C.POINTER(_vp), _pu64, _u32, _pu32]),
    "gkd_add_fasta_file": (_i32, [_vp, C.c_char_p, _i32, _pu32, _pu32]),
    "gkd_label": (C.c_char_p, [_vp, _u32]),
    "gkd_comment": (C.c_char_p, [_vp, _u32]),
    "gkd_count": (_u32, [_vp]),
    "gkd_set_label": (_i32, [_vp, _u32, C.c_char_p, C.c_char_p]),
    "gkd_group_create": (_i32, [C.POINTER(_vp), C.POINTER(GkdConfig), C.POINTER(C.c_int32), _u32]),
    "gkd_group_destroy": (_i32, [_vp]),
    "gkd_group_last_error": (C.c_char_p, [_vp]),
    "gkd_group_size": (_u32, [_vp]),
    "gkd_group_count": (_u32, [_vp]),
    "gkd_group_member": (_vp, [_vp, _u32]),
    "gkd_group_set_panel": (_i32, [_vp, _u32]),
    "gkd_group_add_sequences": (_i32, [_vp, _u32, C.POINTER(_vp), _pu64, _u32, _pu32]),
    "gkd_group_add_fasta_file": (_i32, [_vp, C.c_char_p, _pu32]),
    "gkd_group_label": (C.c_char_p, [_vp, _u32]),
    "gkd_group_comment": (C.c_char_p, [_vp, _u32]),
    "gkd_group_build": (_i32, [_vp]),
    "gkd_group_all_vs_all": (_i32, [_vp, _vp, _vp]),
    "gkd_group_all_vs_all_within": (_i32, [_vp, _dbl, C.POINTER(GkdHits)]),
    "gkd_group_all_vs_all_nearest": (_i32, [_vp, _u32, _dbl, C.POINTER(GkdNeighbors)]),
    "gkd_group_all_vs_all_clusters": (_i32, [_vp, _dbl, _vp, _pu32]),
    "gkd_group_all_vs_all_linkage": (_i32, [_vp, _dbl, C.POINTER(GkdHits)]),
    "gkd_group_all_vs_all_agglomerate": (_i32, [_vp, _i32, _dbl, C.POINTER(GkdMerges)]),
    "gkd_build_sets": (_i32, [_vp]),
    "gkd_set_size": (_i32, [_vp, _u32, _pu64, _pu64, _pu64]),
    "gkd_export_set": (_i32, [_vp, _u32, _vp, _u64, _pu64]),
    "gkd_arena_count": (_u32, [_vp]),
    "gkd_arena_info": (_i32, [_vp, _u32, _pu32, _pu32, C.POINTER(_vp), _pu64]),
    "gkd_describe_sets": (_i32, [_vp, _u32, _u32, C.POINTER(GkdPackedSet)]),
    "gkd_adopt_sets": (_i32, [_vp, _vp, _u64, C.POINTER(GkdPackedSet), _u32, _pu32]),
    "gkd_import_set": (_i32, [_vp, _vp, _u64, _pu32]),
    "gkd_import_sets": (_i32, [_vp, _vp, _pu64, _u32, _pu32]),
    "gkd_save_sets": (_i32, [_vp, C.c_char_p]),
    "gkd_load_sets": (_i32, [_vp, C.c_char_p, _pu32, _pu32]),
    "gkd_all_vs_all": (_i32, [_vp, _vp, _vp]),
    "gkd_all_vs_all_range": (_i32, [_vp, _u32, _u64, _u64, _vp, _vp]),
    "gkd_query_vs_ref": (_i32, [_vp, _vp, _u32, _vp, _u32, _vp, _vp]),
    "gkd_pairs": (_i32, [_vp, _vp, _vp, _u64, _vp, _vp]),
    "gkd_all_vs_all_range_ex": (_i32, [_vp, _u32, _u64, _u64, C.POINTER(GkdOutputs)]),
    "gkd_query_vs_ref_ex": (_i32, [_vp, _vp, _u32, _vp, _u32, C.POINTER(GkdOutputs)]),
    "gkd_pairs_ex": (_i32, [_vp, _vp, _vp, _u64, C.POINTER(GkdOutputs)]),
    "gkd_greedy_reps": (_i32, [_vp, _vp, _u32, _dbl, _vp]),
    "gkd_pair": (_i32, [_vp, _u32, _u32, _pu64, _pu64, _pdbl]),
    "gkd_all_vs_all_range_within": (_i32, [_vp, _u32, _u64, _u64, _dbl, C.POINTER(GkdHits)]),
    "gkd_query_vs_ref_within": (_i32, [_vp, _vp, _u32, _vp, _u32, _dbl, C.POINTER(GkdHits)]),
    "gkd_query_vs_ref_nearest": (_i32, [_vp, _vp, _u32, _vp, _u32, _u32, _dbl, _i32, _vp, _vp, _vp, _vp]),
    "gkd_query_vs_ref_nearest_ex": (_i32, [_vp, _vp, _u32, _vp, _u32, _u32, _dbl, _i32, C.POINTER(GkdNeighbors),
                                           C.POINTER(GkdNeighbors)]),
    "gkd_all_vs_all_nearest": (_i32, [_vp, _u32, _u32, _dbl, C.POINTER(GkdNeighbors)]),
    "gkd_all_vs_all_clusters": (_i32, [_vp, _u32, _dbl, _vp, _pu32]),
    "gkd_query_vs_ref_clusters": (_i32, [_vp, _vp, _u32, _vp, _u32, _dbl, _vp, _vp]),
    "gkd_all_vs_all_linkage": (_i32, [_vp, _u32, _dbl, C.POINTER(GkdHits)]),
    "gkd_query_vs_ref_linkage": (_i32, [_vp, _vp, _u32, _vp, _u32, _dbl, _vp, _vp, C.POINTER(GkdHits)]),
    "gkd_all_vs_all_agglomerate": (_i32, [_vp, _u32, _i32, _dbl, C.POINTER(GkdMerges)]),
    "gkd_agglomerate": (_i32, [_vp, _u32, _vp, _i32, _dbl, C.POINTER(GkdMerges)]),
    "gkd_hash_set": (_i32, [_vp, _u32, _u32, _i32, _vp, _pu32]),
    "gkd_sketch_distances": (_i32, [_vp, _u32, _i32, _vp, _vp, _u64, _vp]),
    "gkd_format_double": (_i32, [_dbl, C.c_char_p, C.c_size_t]),
    "gkd_get_metrics": (_i32, [_vp, C.POINTER(GkdMetrics)]),
    "gkd_stream": (_vp, [_vp]),
    "gkd_synth_dna": (_i32, [_i32, _vp, _u64, _u64, _u32, _u32, _dbl]),
    "gkd_synth_protein": (_i32, [_i32, _vp, _u64, _u64, _u32, _u32, _dbl]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen libgkd.so and type every entry point.  Raises if the library or a symbol is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(genome.distance_b200 has no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
