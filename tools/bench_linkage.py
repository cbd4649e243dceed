#!/usr/bin/env python
"""The single-linkage hierarchy on the device (gkd_all_vs_all_linkage) against the pairs within D copied to the host
(Engine.all_vs_all_within) followed by scipy's minimum_spanning_tree, on one GPU, in one command, printing one JSON
line.  The workloads of tools/bench_clusters.py:

* config 2: 1000 x 5 Mbp from the synthetic generator of tools/bench_rect.py (499,500 pairs);
* genes: 12,000 gene-sized records (900-1300 bp, 7.2e7 pairs: two 64 Mi-pair chunks), where kernel 4 is cheapest and
  the linkage epilogue weighs most.

For each threshold (default 0.3, and 1.0, where every pair is an edge: 64 Mi edges per chunk and the most Boruvka
work), per call: wall time (host clock around the call, which ends in a device synchronise; median of --repeat for the
device path, one call for the host path, whose hits can take gigabytes), kernel-4 ms and kernel-5 ms (compaction and
rounds on the device path) summed over the launches of the last library call (CUDA events of the library), bytes
copied device to host over the whole path, the number of forest edges, and whether both paths give equal edge lists
(a, b, inter, dist).  The host path ranks the edges by (distance bits, a, b) so that scipy breaks ties as the library
does; its wall time includes that and the tree (also given alone).  The card's name and power limit are read in the
same run.  Writes nothing in the tree (--out also writes the JSON line to a file).
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
from scipy import sparse
from scipy.sparse.csgraph import minimum_spanning_tree

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import genome.distance_b200 as gkd  # noqa: E402
from bench_select import card, measure  # noqa: E402


def host_linkage(e, D):
    """the forest from the within hits: scipy's minimum spanning tree on weights rank + 1 of (distance bits, a, b)"""
    n = len(e)
    a, b, inter, dist = e.all_vs_all_within(D)
    t0 = time.perf_counter()
    order = np.lexsort((b, a, dist.view(np.uint64)))
    rank = np.empty(order.size, dtype=np.float64)
    rank[order] = np.arange(1, order.size + 1)
    t = minimum_spanning_tree(sparse.csr_matrix((rank, (a.astype(np.int64), b.astype(np.int64))), shape=(n, n)))
    sel = order[np.sort(t.data).astype(np.int64) - 1]
    return (a[sel], b[sel], inter[sel], dist[sel]), time.perf_counter() - t0, a.size


def compare(e, thresholds, repeat):
    e.all_vs_all_linkage(thresholds[0])  # warm-up of both paths
    e.all_vs_all_within(thresholds[0])
    out = {}
    for D in thresholds:
        dev, rd = measure(e, lambda: e.all_vs_all_linkage(D), repeat)
        rd["edges"] = int(dev[0].size)
        (host, tree_s, hits), rh = measure(e, lambda: host_linkage(e, D), 1)
        rh["tree_ms"] = round(1e3 * tree_s, 3)
        rh["hits"] = int(hits)
        rd["equal_to_host"] = all(x.dtype == y.dtype and np.array_equal(x, y) for x, y in zip(dev, host))
        out["D%g" % D] = {"device": rd, "within_then_host": rh}
        del host
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genomes", type=int, default=1000)
    ap.add_argument("--length", type=int, default=5_000_000)
    ap.add_argument("--genes", type=int, default=12_000)
    ap.add_argument("--thresholds", type=float, nargs="+", default=[0.3, 1.0])
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_linkage needs a GPU"
    res = {"what": "all_vs_all_linkage (device) against all_vs_all_within + scipy minimum_spanning_tree (host)", **card()}
    buf = torch.empty((100, a.length), dtype=torch.uint8, device="cuda")
    with gkd.Engine(k=21) as e:
        for g in range(a.genomes):
            # the generator of tools/bench_rect.py: families of 100, members mutated at 0.1 / 1 / 5 / 20 %
            gkd.synth(buf[g % 100], 0x5EED0000, g // 100, g % 100, [0.001, 0.01, 0.05, 0.2][g % 4] if g % 100 else 0.0)
            e.add(buf[g % 100])
            if g % 100 == 99:
                e.build()
        e.build()
        res["config2"] = {"genomes": a.genomes, "length": a.length, **compare(e, a.thresholds, a.repeat)}
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
        res["genes"] = {"records": a.genes, **compare(e, a.thresholds, a.repeat)}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
