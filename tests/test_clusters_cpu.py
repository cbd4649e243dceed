"""CPU-side checks of the single-linkage cluster calls (gkd_all_vs_all_clusters, gkd_query_vs_ref_clusters and the group
form): the argument checks that run before any context, group or device is looked at, and the validation messages,
their order and the usage of `fastaDist --clusters`."""
import ctypes as C
import os
import subprocess

import numpy as np

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")


def test_cluster_arguments_are_einval_before_device_use():
    """A NaN max_dist, a NULL label (or two NULL rectangle outputs) are refused with a message even with no context or
    group (and no GPU); arguments that pass reach the NULL-handle check, still GKD_EINVAL."""
    lib = gkd.load()
    q = np.zeros(2, dtype=np.uint32)
    label, other = np.zeros(4, dtype=np.uint32), np.zeros(4, dtype=np.uint32)
    count = C.c_uint32()
    nan = float("nan")

    calls = {
        "all_vs_all": (lambda D, lab: lib.gkd_all_vs_all_clusters(None, 2, D, lab, C.byref(count)), lib.gkd_last_error),
        "rect": (lambda D, lab: lib.gkd_query_vs_ref_clusters(None, q.ctypes.data, 2, q.ctypes.data, 2, D, lab, lab),
                 lib.gkd_last_error),
        "group": (lambda D, lab: lib.gkd_group_all_vs_all_clusters(None, D, lab, C.byref(count)),
                  lib.gkd_group_last_error),
    }
    for name, (call, err) in calls.items():
        assert call(nan, label.ctypes.data) == _lib.GKD_EINVAL, name
        assert b"NaN" in err(None), name
        assert call(0.5, None) == _lib.GKD_EINVAL, name
        assert b"null label" in err(None) or b"both outputs are NULL" in err(None), name
        # legal arguments, including a negative max_dist (singletons): refused only for the NULL handle
        for D in (0.5, -1.0):
            assert call(D, label.ctypes.data) == _lib.GKD_EINVAL, (name, D)
    assert lib.gkd_all_vs_all_clusters(None, 2, 0.5, None, None) == _lib.GKD_EINVAL
    assert b"null label" in lib.gkd_last_error(None)
    assert lib.gkd_group_all_vs_all_clusters(None, 0.5, None, None) == _lib.GKD_EINVAL
    assert b"null label" in lib.gkd_group_last_error(None)
    # the rectangle: one output may be NULL, not both
    rc = lib.gkd_query_vs_ref_clusters(None, q.ctypes.data, 2, q.ctypes.data, 2, 0.5, label.ctypes.data, None)
    assert rc == _lib.GKD_EINVAL
    rc = lib.gkd_query_vs_ref_clusters(None, q.ctypes.data, 2, q.ctypes.data, 2, 0.5, None, other.ctypes.data)
    assert rc == _lib.GKD_EINVAL
    rc = lib.gkd_query_vs_ref_clusters(None, q.ctypes.data, 2, q.ctypes.data, 2, 0.5, None, None)
    assert rc == _lib.GKD_EINVAL and b"both outputs are NULL" in lib.gkd_last_error(None)


def _run(args):
    p = subprocess.run([GKD] + args, capture_output=True, text=True, timeout=120, stdin=subprocess.DEVNULL)
    return p.returncode, p.stdout, p.stderr


def test_fastadist_clusters_validation_messages_order_and_usage():
    assert os.path.exists(GKD), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    rc, out, err = _run(["fastaDist", "--clusters"])
    assert rc == 1 and err.startswith("--clusters needs --maxDist.\n"), err
    for extra in (["--nearest", "3"], ["--nearest", "256"]):
        rc, out, err = _run(["fastaDist", "--clusters", "--maxDist", "0.5"] + extra)
        assert rc == 1 and err.startswith("--clusters and --nearest cannot be combined.\n"), (extra, err)
    # the --maxDist range check runs first and is unchanged, then the --nearest range check
    for bad in ("0", "1.5", "-0.2"):
        rc, out, err = _run(["fastaDist", "--clusters", "--maxDist", bad])
        assert rc == 1 and err.startswith("Maximum distance must be > 0 and <= 1.\n"), (bad, err)
    rc, out, err = _run(["fastaDist", "--clusters", "--maxDist", "0.5", "--nearest", "0"])
    assert rc == 1 and err.startswith("Number of neighbors must be between 1 and 256.\n"), err
    # a missing --maxDist is reported before the combination
    rc, out, err = _run(["fastaDist", "--clusters", "--nearest", "3"])
    assert rc == 1 and err.startswith("--clusters needs --maxDist.\n"), err
    # the checks run before the input is opened
    rc, out, err = _run(["fastaDist", "--clusters", "-i", "/nonexistent/in.fa"])
    assert rc == 1 and err.startswith("--clusters needs --maxDist.\n"), err
    rc, out, err = _run(["fastaDist", "--help"])
    assert rc == 0 and "--clusters" in err and "single-linkage" in err
