"""CPU-side checks of the k-nearest-neighbour calls (gkd_all_vs_all_nearest, gkd_query_vs_ref_nearest_ex and the group
form): the gkd_neighbors mirror against the C compiler's layout, the argument checks that run before any device is
touched, and the validation messages and usage of `fastaDist --nearest`."""
import ctypes as C
import os
import subprocess

import numpy as np

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")


def test_neighbors_struct_matches_header_layout(tmp_path):
    src = tmp_path / "nb.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "gkd.h"\n'
        'int main(void){printf("%zu %zu %zu %zu %zu\\n", sizeof(gkd_neighbors), offsetof(gkd_neighbors, pos),'
        ' offsetof(gkd_neighbors, inter), offsetof(gkd_neighbors, dist), offsetof(gkd_neighbors, n_found));return 0;}\n')
    exe = tmp_path / "nb"
    subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    s = _lib.GkdNeighbors
    assert got == [C.sizeof(s), s.pos.offset, s.inter.offset, s.dist.offset, s.n_found.offset]


def test_nearest_arguments_are_einval_before_device_use():
    """k outside 1..256, a NaN max_dist, a NULL output (or two NULL sides) are refused before the context or group is
    looked at, so they are GKD_EINVAL with a message even with neither (and no GPU) at all."""
    lib = gkd.load()
    q = np.zeros(2, dtype=np.uint32)
    pos, found = np.zeros(2 * 300, dtype=np.uint32), np.zeros(2, dtype=np.uint32)
    inter, dist = np.zeros(2 * 300, dtype=np.uint64), np.zeros(2 * 300, dtype=np.float64)
    nb = _lib.GkdNeighbors(pos.ctypes.data, inter.ctypes.data, dist.ctypes.data, found.ctypes.data)
    nan = float("nan")

    calls = {
        "all_vs_all": (lambda k, D, o: lib.gkd_all_vs_all_nearest(None, 2, k, D, o), lib.gkd_last_error),
        "ex": (lambda k, D, o: lib.gkd_query_vs_ref_nearest_ex(None, q.ctypes.data, 2, q.ctypes.data, 2, k, D, 0, o, o),
               lib.gkd_last_error),
        "group": (lambda k, D, o: lib.gkd_group_all_vs_all_nearest(None, k, D, o), lib.gkd_group_last_error),
    }
    for name, (call, err) in calls.items():
        for k in (0, 257, 1000):
            assert call(k, 0.5, C.byref(nb)) == _lib.GKD_EINVAL, (name, k)
            assert b"outside 1..256" in err(None), (name, k)
        assert call(4, nan, C.byref(nb)) == _lib.GKD_EINVAL, name
        assert b"NaN" in err(None), name
        assert call(4, 0.5, None) == _lib.GKD_EINVAL, name
    # _ex: one side may be NULL, not both
    rc = lib.gkd_query_vs_ref_nearest_ex(None, q.ctypes.data, 2, q.ctypes.data, 2, 4, 0.5, 0, C.byref(nb), None)
    assert rc == _lib.GKD_EINVAL  # refused for the NULL context, after the arguments passed
    rc = lib.gkd_query_vs_ref_nearest_ex(None, q.ctypes.data, 2, q.ctypes.data, 2, 4, 0.5, 0, None, None)
    assert rc == _lib.GKD_EINVAL and b"both sides are NULL" in lib.gkd_last_error(None)


def _run(args):
    p = subprocess.run([GKD] + args, capture_output=True, text=True, timeout=120, stdin=subprocess.DEVNULL)
    return p.returncode, p.stdout, p.stderr


def test_fastadist_nearest_validation_messages_and_usage():
    assert os.path.exists(GKD), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    for bad in ("0", "257", "-3"):
        rc, out, err = _run(["fastaDist", "--nearest", bad])
        assert rc == 1 and err.startswith("Number of neighbors must be between 1 and 256.\n"), (bad, err)
    rc, out, err = _run(["fastaDist", "--nearest", "two"])
    assert rc == 1 and 'is not a valid value for "--nearest"' in err
    # the --maxDist check comes first and is unchanged
    rc, out, err = _run(["fastaDist", "--maxDist", "1.5", "--nearest", "0"])
    assert rc == 1 and err.startswith("Maximum distance must be > 0 and <= 1.") and "neighbors" not in err
    rc, out, err = _run(["fastaDist", "--help"])
    assert rc == 0 and "--nearest" in err and "twice" in err
