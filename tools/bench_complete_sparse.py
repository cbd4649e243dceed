#!/usr/bin/env python
"""Complete linkage from the pairs within D (gkd_all_vs_all_complete_linkage, "sparse") against the dense matrix form
(gkd_all_vs_all_agglomerate(GKD_LINK_COMPLETE), "dense"), on one GPU, in one command, printing one JSON line.  The
workloads of tools/bench_agglomerate.py:

* config 2: 1000 x 5 Mbp from the synthetic generator of tools/bench_rect.py (499,500 pairs);
* genes: 12,000 gene-sized records (900-1300 bp, 7.2e7 pairs: two 64 Mi-pair chunks);

each at D = 0.05, 0.3, 0.7 and 1.0 (every pair).  Per form: wall time (host clock around the call, which ends in a
device synchronise; median of --repeat), kernel-4 ms and kernel-5 ms (sparse: compaction, row build and rounds; dense:
epilogue, scatter and rounds) of the library's CUDA events, the rounds, the bytes copied device to host, and the peak
device memory of the call, sampled: the largest drop of cudaMemGetInfo's free bytes below its value before the call,
polled every 0.5 ms on a host thread (a short-lived peak between two polls is missed).  hits = the pairs within D, from
the dense triangle.  The merges of both forms are compared in the same run.

Then one collection of --large gene-sized records (default 150,000: 1.1e10 pairs) where the dense matrix does not fit
in the card's memory: the dense call must fail with GKD_ENOMEM before any pair is intersected, and the sparse call at
D = --large-dist runs to the end (wall, kernel-4 and kernel-5 ms, merges, sampled peak).  The card's name and power limit
are read in the same run.  Writes nothing in the tree (--out also writes the JSON line to a file).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import genome.distance_b200 as gkd  # noqa: E402
from bench_select import card, measure  # noqa: E402

THRESHOLDS = (0.05, 0.3, 0.7, 1.0)


class PeakSampler:
    """the largest drop of the device's free bytes below their value at start, polled on a host thread"""

    def __init__(self, period=5e-4):
        self.period, self.stop, self.peak = period, threading.Event(), 0

    def __enter__(self):
        self.base = torch.cuda.mem_get_info(0)[0]
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def _run(self):
        while not self.stop.is_set():
            self.peak = max(self.peak, self.base - torch.cuda.mem_get_info(0)[0])
            time.sleep(self.period)

    def __exit__(self, *a):
        self.stop.set()
        self.t.join()


def timed(e, fn, repeat):
    with PeakSampler() as p:
        out, r = measure(e, fn, repeat)
    r["rounds"] = int(e.metrics()["agglomerate_rounds"])
    r["merges"] = int(out[0].size)
    r["peak_device_bytes_sampled"] = int(p.peak)
    return out, r


def compare(e, repeat):
    _, gd = e.all_vs_all(want_inter=False)
    out = {}
    for D in THRESHOLDS:
        e.all_vs_all_complete_linkage(D)  # warm-up
        sparse, rs = timed(e, lambda: e.all_vs_all_complete_linkage(D), repeat)
        dense, rd = timed(e, lambda: e.all_vs_all_agglomerate(gkd.LINK_COMPLETE, D), repeat)
        equal = all(np.array_equal(x.view(np.uint64) if x.dtype == np.float64 else x,
                                   y.view(np.uint64) if y.dtype == np.float64 else y) for x, y in zip(sparse, dense))
        out[str(D)] = {"hits": int((gd <= D).sum()), "sparse": rs, "dense": rd, "equal": bool(equal)}
    return out


def genes(e, n):
    for g in range(n):
        # the gene-sized records of tests/test_gpu_nearest.py: 40 families, lengths 900-1299
        s = np.empty(900 + (g * 37) % 400, dtype=np.uint8)
        mem = g // 40
        gkd.synth(s, 77, g % 40, mem, [0.0, 0.002, 0.03, 0.15][mem % 4] if mem else 0.0)
        e.add(s.tobytes())
        if g % 20_000 == 19_999:
            e.build()
    e.build()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genomes", type=int, default=1000)
    ap.add_argument("--length", type=int, default=5_000_000)
    ap.add_argument("--genes", type=int, default=12_000)
    ap.add_argument("--large", type=int, default=150_000, help="records of the run the dense form cannot hold (0: skip)")
    ap.add_argument("--large-dist", type=float, default=0.05)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_complete_sparse needs a GPU"
    res = {"what": "all_vs_all_complete_linkage (sparse) against all_vs_all_agglomerate(COMPLETE) (dense)", **card()}
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
        genes(e, a.genes)
        res["genes"] = {"records": a.genes, **compare(e, a.repeat)}
    if a.large:
        with gkd.Engine(k=21) as e:
            genes(e, a.large)
            big = {"records": a.large, "max_dist": a.large_dist}
            try:
                e.all_vs_all_agglomerate(gkd.LINK_COMPLETE, a.large_dist)
                big["dense"] = "completed"
            except gkd.GkdError as ex:
                big["dense"] = {"code": ex.code, "message": ex.msg, "pairs_intersected": int(e.metrics()["pairs"])}
            _, big["sparse"] = timed(e, lambda: e.all_vs_all_complete_linkage(a.large_dist), 1)
            res["large"] = big
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
