"""CPU-side checks of the single-linkage hierarchy calls (gkd_all_vs_all_linkage, gkd_query_vs_ref_linkage and the group
form): the argument checks that run before any context, group or device is looked at, and the validation messages,
their order and the usage of `fastaDist --linkage`."""
import ctypes as C
import os
import subprocess

import numpy as np

import genome.distance_b200 as gkd
from genome.distance_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")


def _hits(cap=4):
    a, b = np.zeros(cap, dtype=np.uint32), np.zeros(cap, dtype=np.uint32)
    inter, dist = np.zeros(cap, dtype=np.uint64), np.zeros(cap, dtype=np.float64)
    return (a, b, inter, dist), _lib.GkdHits(a.ctypes.data, b.ctypes.data, inter.ctypes.data, dist.ctypes.data, cap, 0)


def test_linkage_arguments_are_einval_before_device_use():
    """A NaN max_dist, a NULL out and duplicate rectangle keys are refused with a message even with no context or group
    (and no GPU); arguments that pass reach the NULL-handle check, still GKD_EINVAL."""
    lib = gkd.load()
    q = np.zeros(2, dtype=np.uint32)
    keep, h = _hits()
    nan = float("nan")
    calls = {
        "all_vs_all": (lambda D, out: lib.gkd_all_vs_all_linkage(None, 2, D, out), lib.gkd_last_error),
        "rect": (lambda D, out: lib.gkd_query_vs_ref_linkage(None, q.ctypes.data, 2, q.ctypes.data, 2, D, None, None, out),
                 lib.gkd_last_error),
        "group": (lambda D, out: lib.gkd_group_all_vs_all_linkage(None, D, out), lib.gkd_group_last_error),
    }
    for name, (call, err) in calls.items():
        assert call(nan, C.byref(h)) == _lib.GKD_EINVAL, name
        assert b"NaN" in err(None), name
        assert call(0.5, None) == _lib.GKD_EINVAL, name
        assert b"null out" in err(None), name
        # legal arguments, including a negative max_dist (no edges): refused only for the NULL handle
        for D in (0.5, -1.0, 1.0):
            assert call(D, C.byref(h)) == _lib.GKD_EINVAL, (name, D)

    def rect(qk, rk):
        return lib.gkd_query_vs_ref_linkage(None, q.ctypes.data, 2, q.ctypes.data, 2, 0.5,
                                            None if qk is None else qk.ctypes.data,
                                            None if rk is None else rk.ctypes.data, C.byref(h))

    u = lambda *v: np.array(v, dtype=np.uint32)
    # duplicates within one side, across the sides, and against the default key of the other side (nq + j)
    for qk, rk in ((u(7, 7), u(1, 2)), (u(1, 2), u(3, 3)), (u(5, 9), u(9, 4)), (u(2, 0), None), (None, u(1, 8))):
        assert lib.gkd_all_vs_all_linkage(None, 2, nan, C.byref(h)) == _lib.GKD_EINVAL
        assert rect(qk, rk) == _lib.GKD_EINVAL
        assert b"not distinct" in lib.gkd_last_error(None), (qk, rk)
    # distinct keys pass the check and reach the NULL-handle check, which leaves the last message as it was
    for qk, rk in ((u(10, 3), u(7, 0)), (u(9, 8), None), (None, u(2, 3)), (None, None)):
        assert lib.gkd_all_vs_all_linkage(None, 2, nan, C.byref(h)) == _lib.GKD_EINVAL
        assert rect(qk, rk) == _lib.GKD_EINVAL
        assert b"NaN" in lib.gkd_last_error(None), (qk, rk)
    # the NaN check comes before the key check
    assert lib.gkd_query_vs_ref_linkage(None, q.ctypes.data, 2, q.ctypes.data, 2, nan, u(1, 1).ctypes.data, None,
                                        C.byref(h)) == _lib.GKD_EINVAL
    assert b"NaN" in lib.gkd_last_error(None)


def _run(args):
    p = subprocess.run([GKD] + args, capture_output=True, text=True, timeout=120, stdin=subprocess.DEVNULL)
    return p.returncode, p.stdout, p.stderr


def test_fastadist_linkage_validation_messages_order_and_usage():
    assert os.path.exists(GKD), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    for extra in (["--nearest", "3"], ["--nearest", "256"], ["--maxDist", "0.5", "--nearest", "1"]):
        rc, out, err = _run(["fastaDist", "--linkage"] + extra)
        assert rc == 1 and err.startswith("--linkage and --nearest cannot be combined.\n"), (extra, err)
    rc, out, err = _run(["fastaDist", "--linkage", "--clusters", "--maxDist", "0.5"])
    assert rc == 1 and err.startswith("--linkage and --clusters cannot be combined.\n"), err
    # the existing checks come first and are unchanged
    for bad in ("0", "1.5", "-0.2"):
        rc, out, err = _run(["fastaDist", "--linkage", "--maxDist", bad])
        assert rc == 1 and err.startswith("Maximum distance must be > 0 and <= 1.\n"), (bad, err)
    rc, out, err = _run(["fastaDist", "--linkage", "--nearest", "0"])
    assert rc == 1 and err.startswith("Number of neighbors must be between 1 and 256.\n"), err
    rc, out, err = _run(["fastaDist", "--linkage", "--clusters"])
    assert rc == 1 and err.startswith("--clusters needs --maxDist.\n"), err
    rc, out, err = _run(["fastaDist", "--linkage", "--clusters", "--maxDist", "0.5", "--nearest", "3"])
    assert rc == 1 and err.startswith("--clusters and --nearest cannot be combined.\n"), err
    # then --nearest before --clusters, and all of it before the input is opened
    rc, out, err = _run(["fastaDist", "--linkage", "--nearest", "3", "-i", "/nonexistent/in.fa"])
    assert rc == 1 and err.startswith("--linkage and --nearest cannot be combined.\n"), err
    rc, out, err = _run(["fastaDist", "--linkage", "--clusters", "--maxDist", "0.5", "-i", "/nonexistent/in.fa"])
    assert rc == 1 and err.startswith("--linkage and --clusters cannot be combined.\n"), err
    rc, out, err = _run(["fastaDist", "--linkage", "-i", "/nonexistent/in.fa"])
    assert rc == 1 and "not found or unreadable" in err and "--linkage" not in err, err
    rc, out, err = _run(["fastaDist", "--help"])
    assert rc == 0 and "--linkage" in err and "single-linkage hierarchy" in err
