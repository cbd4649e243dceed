"""CPU-side checks of the selection calls (pairs within a distance, k nearest references): the gkd_hits mirror
against the C compiler's layout, the argument checks that run before any device is touched, and the validation
messages of `fastaDist --maxDist` and `genomes --nearest`."""
import ctypes as C
import os
import subprocess

import numpy as np

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")


def test_hits_struct_matches_header_layout(tmp_path):
    src = tmp_path / "hits.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "gkd.h"\n'
        'int main(void){printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(gkd_hits), offsetof(gkd_hits, a),'
        ' offsetof(gkd_hits, b), offsetof(gkd_hits, inter), offsetof(gkd_hits, dist), offsetof(gkd_hits, cap),'
        ' offsetof(gkd_hits, n));return 0;}\n')
    exe = tmp_path / "hits"
    subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    h = _lib.GkdHits
    assert got == [C.sizeof(h), h.a.offset, h.b.offset, h.inter.offset, h.dist.offset, h.cap.offset, h.n.offset]


def test_bad_k_and_nan_max_dist_are_einval_before_device_use():
    """k outside 1..256, a NaN max_dist and a NULL gkd_hits are refused before the context is looked at, so they are
    GKD_EINVAL with a message even with no context (and no GPU) at all."""
    lib = gkd.load()
    q = np.zeros(2, dtype=np.uint32)
    pos, found = np.zeros(2 * 300, dtype=np.uint32), np.zeros(2, dtype=np.uint32)
    inter, dist = np.zeros(2 * 300, dtype=np.uint64), np.zeros(2 * 300, dtype=np.float64)
    for k in (0, 257, 1000):
        rc = lib.gkd_query_vs_ref_nearest(None, q.ctypes.data, 2, q.ctypes.data, 2, k, 0.5, 0, pos.ctypes.data,
                                          inter.ctypes.data, dist.ctypes.data, found.ctypes.data)
        assert rc == _lib.GKD_EINVAL
        assert b"outside 1..256" in lib.gkd_last_error(None)
    nan = float("nan")
    rc = lib.gkd_query_vs_ref_nearest(None, q.ctypes.data, 2, q.ctypes.data, 2, 4, nan, 0, pos.ctypes.data,
                                      inter.ctypes.data, dist.ctypes.data, found.ctypes.data)
    assert rc == _lib.GKD_EINVAL and b"NaN" in lib.gkd_last_error(None)
    h = _lib.GkdHits(None, None, None, None, 0, 0)
    assert lib.gkd_all_vs_all_range_within(None, 2, 0, 1, nan, C.byref(h)) == _lib.GKD_EINVAL
    assert b"NaN" in lib.gkd_last_error(None)
    assert lib.gkd_query_vs_ref_within(None, q.ctypes.data, 2, q.ctypes.data, 2, nan, C.byref(h)) == _lib.GKD_EINVAL
    assert b"NaN" in lib.gkd_last_error(None)
    assert lib.gkd_all_vs_all_range_within(None, 2, 0, 1, 0.5, None) == _lib.GKD_EINVAL
    assert lib.gkd_query_vs_ref_within(None, q.ctypes.data, 2, q.ctypes.data, 2, 0.5, None) == _lib.GKD_EINVAL
    assert lib.gkd_group_all_vs_all_within(None, nan, C.byref(h)) == _lib.GKD_EINVAL
    assert b"NaN" in lib.gkd_group_last_error(None)
    assert lib.gkd_group_all_vs_all_within(None, 0.5, None) == _lib.GKD_EINVAL


def _run(args):
    p = subprocess.run([GKD] + args, capture_output=True, text=True, timeout=120, stdin=subprocess.DEVNULL)
    return p.returncode, p.stdout, p.stderr


def test_maxdist_and_nearest_validation_messages(tmp_path):
    assert os.path.exists(GKD), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    for bad in ("0", "-0.1", "1.5", "nan"):
        rc, out, err = _run(["fastaDist", "--maxDist", bad])
        assert rc == 1 and err.startswith("Maximum distance must be > 0 and <= 1."), (bad, err)
    rc, out, err = _run(["fastaDist", "--maxDist", "x"])
    assert rc == 1 and 'is not a valid value for "--maxDist"' in err
    d = tmp_path / "g"
    d.mkdir()
    for bad in ("0", "257", "-3"):
        rc, out, err = _run(["genomes", "--nearest", bad, str(d), str(d)])
        assert rc == 1 and "\nNumber of neighbors must be between 1 and 256.\n" in err, (bad, err)
    rc, out, err = _run(["genomes", "--nearest", "two", str(d), str(d)])
    assert rc == 1 and 'is not a valid value for "--nearest"' in err
    # the existing -m check still comes first and is unchanged
    rc, out, err = _run(["genomes", "-m", "1.5", "--nearest", "3", str(d), str(d)])
    assert rc == 1 and "Maximum distance must be > 0 and <= 1." in err and "neighbors" not in err
    # the usage lists the new options
    rc, out, err = _run(["fastaDist", "--help"])
    assert rc == 0 and "--maxDist" in err
    rc, out, err = _run(["genomes", "--help"])
    assert rc == 0 and "--nearest" in err
