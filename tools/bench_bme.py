#!/usr/bin/env python
"""Balanced minimum-evolution NNIs on the device (gkd_bme, gkd_bme_nni) on one GPU, in one command, printing one JSON
line.

Workloads, each a triangle in device memory:
* config 2: the dense triangle of 1000 x 5 Mbp from the synthetic generator of tools/bench_rect.py;
* families: 5,000 x 400 kbp from the same generator (families of 100 near-identical members), whose near-tied joins
  make the BIONJ start take many swaps;
* synthetic: the additive-tree-plus-noise triangle of tools/bench_nj.py at n = 5,000.

On the same triangle, timed with CUDA events on gkd_stream (median of --repeat):
* bionj:  gkd_bionj, the BIONJ rounds (the start tree);
* search: gkd_bme_nni from the BIONJ rows: the table build, every swap and the lengths, and the number of swaps;
* build:  gkd_bme_nni from the searched tree, which takes no swap: the table build, one pick and the lengths.
search - build is the time of the swaps; over their number, the time of one swap.  The call equals gkd_bme(bionj) in
the same run.  The card's name and power limit are read in the same run.  Writes nothing in the tree (--out also
writes the JSON line to a file).
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
from bench_nj import same, synthetic  # noqa: E402
from bench_select import card  # noqa: E402


def timed(e, call, repeat):
    """(result, median ms, launches of one call): CUDA events on gkd_stream around call()"""
    s = torch.cuda.ExternalStream(e.stream_ptr)
    ms, out, launches = [], None, 0
    for _ in range(repeat):
        before = e.metrics()["launches"]
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(s)
        out = call()
        t1.record(s)
        t1.synchronize()
        ms.append(t0.elapsed_time(t1))
        launches = int(e.metrics()["launches"] - before)
    return out, float(np.median(ms)), launches


def families(e, genomes, length):
    """the dense triangle (CUDA tensor) of the generator of tools/bench_rect.py: families of 100, members mutated at
    0.1 / 1 / 5 / 20 %"""
    buf = torch.empty((100, length), dtype=torch.uint8, device="cuda")
    for g in range(genomes):
        gkd.synth(buf[g % 100], 0x5EED0000, g // 100, g % 100, [0.001, 0.01, 0.05, 0.2][g % 4] if g % 100 else 0.0)
        e.add(buf[g % 100])
        if g % 100 == 99:
            e.build()
    e.build()
    _, gd = e.all_vs_all(want_inter=False)
    del buf
    torch.cuda.empty_cache()
    return torch.from_numpy(gd).to("cuda")


def run(e, dev, n, repeat):
    start, bionj_ms, _ = timed(e, lambda: e.bionj(dev), repeat)
    (rows, swaps), search_ms, search_launches = timed(e, lambda: e.bme_nni(dev, start[0], start[1]), repeat)
    (again, zero), build_ms, build_launches = timed(e, lambda: e.bme_nni(dev, rows[0], rows[1]), repeat)
    whole, _ = e.bme(dev, "bionj")
    swap_ms = search_ms - build_ms
    return {"n": n, "bionj_ms": round(bionj_ms, 3), "search_ms": round(search_ms, 3), "swaps": swaps,
            "build_and_lengths_ms": round(build_ms, 3), "swaps_ms": round(swap_ms, 3),
            "ms_per_swap": round(swap_ms / swaps, 4) if swaps else None, "search_launches": search_launches,
            "build_launches": build_launches, "fixed_point": zero == 0 and same(again, rows),
            "equal_to_gkd_bme": same(whole, rows)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genomes", type=int, default=1000)
    ap.add_argument("--length", type=int, default=5_000_000)
    ap.add_argument("--sizes", type=int, nargs="*", default=[5000])
    ap.add_argument("--family-genomes", type=int, default=5000)
    ap.add_argument("--family-length", type=int, default=400_000)
    ap.add_argument("--repeat", type=int, default=2)
    ap.add_argument("--seed", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_bme needs a GPU"
    res = {"what": "BME NNIs on the device from the BIONJ tree: gkd_bionj, gkd_bme_nni (config 2 and synthetic device "
                   "triangles)", **card()}
    with gkd.Engine(k=21) as e:
        dev = families(e, a.genomes, a.length)
        e.bme(dev)  # warm-up
        res["config2"] = {"genomes": a.genomes, "length": a.length, **run(e, dev, a.genomes, a.repeat)}
    with gkd.Engine(k=21) as e:
        dev = families(e, a.family_genomes, a.family_length)
        res["families"] = {"genomes": a.family_genomes, "length": a.family_length,
                           **run(e, dev, a.family_genomes, a.repeat)}
        del dev
        torch.cuda.empty_cache()
    with gkd.Engine(k=21) as e:
        res["synthetic"] = []
        for n in a.sizes:
            dev = synthetic(n, a.seed + n)
            torch.cuda.synchronize()
            res["synthetic"].append(run(e, dev, n, a.repeat))
            del dev
            torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
