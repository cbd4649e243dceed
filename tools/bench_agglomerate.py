#!/usr/bin/env python
"""Complete- and average-linkage hierarchies on the device (gkd_all_vs_all_agglomerate) against the dense triangle
copied to the host (Engine.all_vs_all) followed by scipy.cluster.hierarchy.linkage, on one GPU, in one command, printing
one JSON line.  The workloads of tools/bench_linkage.py:

* config 2: 1000 x 5 Mbp from the synthetic generator of tools/bench_rect.py (499,500 pairs);
* genes: 12,000 gene-sized records (900-1300 bp, 7.2e7 pairs: two 64 Mi-pair chunks), where kernel 4 is cheapest and
  the agglomeration weighs most.

For each method at D = 1.0 (the whole tree), per path: wall time (host clock around the call, which ends in a device
synchronise; median of --repeat for the device path, one call for the host path), kernel-4 ms and kernel-5 ms (the
distance epilogue, the matrix scatter and the rounds) summed over the last library call (CUDA events of the library),
the rounds, and the bytes copied device to host.  The agglomeration alone is also timed with CUDA events on gkd_stream
around gkd_agglomerate on the triangle already in device memory.  The host path's time is split into the dense call and
scipy.  The merges of the two paths are compared in the same run: scipy's cluster ids are mapped to the labels (the
smallest id of each cluster); ties may be broken in another order by scipy, so the result reports whether the topology
and sizes are equal and the largest height difference.  The card's name and power limit are read in the same run.
Writes nothing in the tree (--out also writes the JSON line to a file).
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
from scipy.cluster import hierarchy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import genome.distance_b200 as gkd  # noqa: E402
from bench_select import card, measure  # noqa: E402

METHODS = {"complete": gkd.LINK_COMPLETE, "average": gkd.LINK_AVERAGE}


def scipy_merges(Z, n):
    """(a, b, height, size) of a scipy linkage matrix, with each cluster named by its smallest member"""
    label = list(range(n)) + [0] * max(n - 1, 0)
    a, b = np.empty(n - 1, dtype=np.uint32), np.empty(n - 1, dtype=np.uint32)
    for t, (p, q, _, _) in enumerate(Z):
        x, y = label[int(p)], label[int(q)]
        a[t], b[t] = min(x, y), max(x, y)
        label[n + t] = a[t]
    return a, b, Z[:, 2].copy(), Z[:, 3].astype(np.uint32)


def agglomerate_ms(e, dev, method, repeat):
    """CUDA-event time on gkd_stream of gkd_agglomerate over a triangle in device memory (median of repeat)"""
    s = torch.cuda.ExternalStream(e.stream_ptr)
    times = []
    for _ in range(repeat):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(s)
        e.agglomerate(dev, method, 1.0)
        t1.record(s)
        t1.synchronize()
        times.append(t0.elapsed_time(t1))
    return round(float(np.median(times)), 3)


def compare(e, repeat):
    n = len(e)
    out = {}
    t0 = time.perf_counter()
    _, gd = e.all_vs_all(want_inter=False)
    dense_s = time.perf_counter() - t0
    dense_d2h = int(e.metrics()["d2h_bytes"])
    dev = torch.from_numpy(gd).to("cuda")
    for name, method in METHODS.items():
        e.all_vs_all_agglomerate(method, 1.0)  # warm-up
        got, rd = measure(e, lambda: e.all_vs_all_agglomerate(method, 1.0), repeat)
        rd["rounds"] = int(e.metrics()["agglomerate_rounds"])
        rd["merges"] = int(got[0].size)
        rd["agglomerate_only_ms"] = agglomerate_ms(e, dev, method, repeat)
        rd["equal_to_agglomerate_of_dense"] = all(np.array_equal(x, y) for x, y in zip(got, e.agglomerate(gd, method, 1.0)))
        t0 = time.perf_counter()
        Z = hierarchy.linkage(gd, method=name)
        scipy_s = time.perf_counter() - t0
        ref = scipy_merges(Z, n)
        rh = {"wall_ms": round(1e3 * (dense_s + scipy_s), 3), "dense_ms": round(1e3 * dense_s, 3),
              "scipy_ms": round(1e3 * scipy_s, 3), "d2h_bytes": dense_d2h}
        same = got[0].size == ref[0].size
        rd["equal_to_scipy"] = {
            "topology_and_sizes": bool(same and all(np.array_equal(x, y) for x, y in zip((got[0], got[1], got[3]),
                                                                                       (ref[0], ref[1], ref[3])))),
            "heights_bitwise": bool(same and np.array_equal(got[2], ref[2])),
            "max_height_diff": float(np.max(np.abs(got[2] - ref[2]))) if same and got[2].size else None,
        }
        out[name] = {"device": rd, "dense_then_scipy": rh}
    del dev
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genomes", type=int, default=1000)
    ap.add_argument("--length", type=int, default=5_000_000)
    ap.add_argument("--genes", type=int, default=12_000)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_agglomerate needs a GPU"
    res = {"what": "all_vs_all_agglomerate at D = 1.0 (device) against all_vs_all + scipy linkage (host)", **card()}
    buf = torch.empty((100, a.length), dtype=torch.uint8, device="cuda")
    with gkd.Engine(k=21) as e:
        for g in range(a.genomes):
            # the generator of tools/bench_rect.py: families of 100, members mutated at 0.1 / 1 / 5 / 20 %
            gkd.synth(buf[g % 100], 0x5EED0000, g // 100, g % 100, [0.001, 0.01, 0.05, 0.2][g % 4] if g % 100 else 0.0)
            e.add(buf[g % 100])
            if g % 100 == 99:
                e.build()
        e.build()
        res["config2"] = {"genomes": a.genomes, "length": a.length, **compare(e, a.repeat)}
    del buf
    torch.cuda.empty_cache()
    with gkd.Engine(k=21) as e:
        for g in range(a.genes):
            # the gene-sized records of tests/test_gpu_nearest.py: 40 families, lengths 900-1299
            s = np.empty(900 + (g * 37) % 400, dtype=np.uint8)
            mem = g // 40
            gkd.synth(s, 77, g % 40, mem, [0.0, 0.002, 0.03, 0.15][mem % 4] if mem else 0.0)
            e.add(s.tobytes())
        e.build()
        res["genes"] = {"records": a.genes, **compare(e, a.repeat)}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
