"""genome.distance_b200 -- B200-native (sm_100a) replacement for the k-mer set distance hot path of
SEEDtk/genome.distance.  The product is `libgkd.so` (C ABI in include/gkd.h, CUDA kernels in csrc/);
this package is the host-side plumbing used by tests, bench.py and the multi-GPU sharding."""
from ._lib import (AMBIG_LITERAL, AMBIG_SKIP, HASH_JAVA_STRING, HASH_MURMUR3, LINK_AVERAGE, LINK_COMPLETE, TREE_BIONJ, TREE_NJ, DNA, PROT, RNA, STRAND_BOTH, STRAND_CANONICAL, LIB_PATH, SYMBOLS,  # noqa: F401
                   load)
from .engine import Engine, GkdError, Group, format_double, synth  # noqa: F401
