#!/usr/bin/env python
"""The k-nearest-neighbour graph from the upper triangle (gkd_all_vs_all_nearest) against the rectangle q = r = all
sets with exclude_self (gkd_query_vs_ref_nearest), on one GPU, in one command, printing one JSON line.  Two workloads:

* config 2: 1000 x 5 Mbp from the synthetic generator (499,500 triangle pairs against 1,000,000 rectangle pairs);
* genes: 12,000 gene-sized records (900-1300 bp, 7.2e7 triangle pairs: two 64 Mi-pair chunks), where kernel 4 is
  cheapest and the selection epilogue weighs most.

For k = 1, 16 and 256 at max_dist 1.0, per call: wall time (host clock around the call, which ends in a device
synchronise; median of --repeat), kernel-4 ms and kernel-5 ms summed over the call's launches (CUDA events of the
library), bytes copied device to host, and whether the two results are equal bit for bit.  The card's name and power
limit are read in the same run.  Writes nothing in the tree (--out also writes the JSON line to a file).
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import genome.distance_b200 as gkd  # noqa: E402
from bench_select import card, measure  # noqa: E402


def same(a, b):
    return all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b))


def compare(e, ks, repeat):
    n = len(e)
    ids = np.arange(n, dtype=np.uint32)
    e.all_vs_all_nearest(ks[0], 1.0)  # warm-up of both paths
    e.query_vs_ref_nearest(ids, ids, ks[0], 1.0, exclude_self=True)
    out = {}
    for k in ks:
        tri, rt = measure(e, lambda: e.all_vs_all_nearest(k, 1.0), repeat)
        rect, rr = measure(e, lambda: e.query_vs_ref_nearest(ids, ids, k, 1.0, exclude_self=True), repeat)
        rt["equal_to_rectangle"] = same(tri, rect)
        rt["found"] = int(tri[3].sum())
        out["k%d" % k] = {"triangle": rt, "rectangle": rr}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genomes", type=int, default=1000)
    ap.add_argument("--length", type=int, default=5_000_000)
    ap.add_argument("--genes", type=int, default=12_000)
    ap.add_argument("--ks", type=int, nargs="+", default=[1, 16, 256])
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_nearest needs a GPU"
    res = {"what": "all_vs_all_nearest (triangle) against query_vs_ref_nearest(all, all, exclude_self) (rectangle)",
           "max_dist": 1.0, **card()}
    buf = torch.empty((100, a.length), dtype=torch.uint8, device="cuda")
    with gkd.Engine(k=21) as e:
        for g in range(a.genomes):
            # the generator of tools/bench_rect.py: families of 100, members mutated at 0.1 / 1 / 5 / 20 %
            gkd.synth(buf[g % 100], 0x5EED0000, g // 100, g % 100, [0.001, 0.01, 0.05, 0.2][g % 4] if g % 100 else 0.0)
            e.add(buf[g % 100])
            if g % 100 == 99:
                e.build()
        e.build()
        res["config2"] = {"genomes": a.genomes, "length": a.length, **compare(e, a.ks, a.repeat)}
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
        res["genes"] = {"records": a.genes, **compare(e, a.ks, a.repeat)}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
