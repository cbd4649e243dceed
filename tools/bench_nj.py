#!/usr/bin/env python
"""Neighbour-joining and BIONJ trees on the device (gkd_all_vs_all_nj, gkd_nj, gkd_all_vs_all_bionj, gkd_bionj) on one
GPU, in one command, printing one JSON line.

Workloads:
* config 2: 1000 x 5 Mbp from the synthetic generator of tools/bench_rect.py: the dense call (Engine.all_vs_all, the
  triangle copied to the host) and all_vs_all_nj (the triangle stays on the device), whose rows are compared with
  gkd_nj over the dense triangle in the same run, and likewise all_vs_all_bionj against gkd_bionj;
* synthetic: gkd_nj and gkd_bionj on a triangle already in device memory at n = 5,000 and 20,000: the path sums of a random tree
  (leaves at the ends of 20-bit random paths of a complete binary tree, random pendant edges) plus uniform noise, scaled
  into [0, 1], generated on the device from a seed.

gkd_nj and gkd_bionj run alternately on the same device triangle, so both see the same card state.  Reported per run
and per method: the call time and the rounds time from CUDA events on gkd_stream (the rounds: the library's
epilogue_ms, which spans the start sums and all n - 1 rounds), the bytes the row scans must read (the same for both),
sum over r = 3 .. n of r (r - 1) / 2 x 8, and that figure over the rounds time, and the launches of the call.  The
active r x r corner fits the 126 MB L2 once r is below about 4,000, so the last rounds read from L2.  As a CPU reference,
the numpy oracles (oracle/nj.py, oracle/bionj.py) at n = 1,000.  The card's name and power limit are read in the same run.  Writes nothing
in the tree (--out also writes the JSON line to a file).
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import genome.distance_b200 as gkd  # noqa: E402
from bench_select import card, measure  # noqa: E402
from oracle import bionj, nj  # noqa: E402


def scan_bytes(n):
    r = np.arange(3, n + 1, dtype=np.float64)
    return float((r * (r - 1) / 2 * 8).sum())


def synthetic(n, seed, device="cuda"):
    """the condensed triangle (float64 CUDA tensor) of an additive tree plus noise over n leaves"""
    g = torch.Generator(device=device).manual_seed(seed)
    bits = 20
    code = torch.randint(0, 1 << bits, (n,), generator=g, device=device, dtype=torch.int64)
    pend = torch.randint(1, 64, (n,), generator=g, device=device).double() / 4096.0
    level = torch.randint(1, 16, (bits + 1,), generator=g, device=device).double() / 4096.0
    below = torch.flip(torch.cumsum(torch.flip(level, [0]), 0), [0])  # below[l]: the path from depth l to a leaf
    below[bits] = 0.0
    out = torch.empty(n * (n - 1) // 2, dtype=torch.float64, device=device)
    at, step = 0, 1024
    cols = torch.arange(n, device=device)
    for r0 in range(0, n - 1, step):
        rows = torch.arange(r0, min(r0 + step, n - 1), device=device)
        x = (code[rows, None] ^ code[None, :]).double()
        blen = torch.where(x > 0, torch.frexp(x)[1].double(), torch.zeros_like(x))  # bit length of the xor
        lcp = (bits - blen).long()
        d = pend[rows, None] + pend[None, :] + 2.0 * below[lcp]
        d += torch.rand(d.shape, generator=g, device=device, dtype=torch.float64) / 1024.0
        keep = cols[None, :] > rows[:, None]
        part = d[keep]
        out[at:at + part.numel()] = part
        at += part.numel()
    return out / max(1.0, float(out.max()))


def timed_trees(e, dev, repeat):
    """{"nj": ..., "bionj": ...} of (rows, call ms, rounds ms, launches of one call): CUDA events on gkd_stream around
    gkd_nj and gkd_bionj, called alternately, median of repeat"""
    s = torch.cuda.ExternalStream(e.stream_ptr)
    calls = {"nj": e.nj, "bionj": e.bionj}
    times = {m: ([], [], None, 0) for m in calls}
    for _ in range(repeat):
        for m, call in calls.items():
            c, r, _, _ = times[m]
            before = e.metrics()["launches"]
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(s)
            rows = call(dev)
            t1.record(s)
            t1.synchronize()
            c.append(t0.elapsed_time(t1))
            r.append(e.metrics()["epilogue_ms"])
            times[m] = (c, r, rows, int(e.metrics()["launches"] - before))
    return {m: (rows, float(np.median(c)), float(np.median(r)), launches) for m, (c, r, rows, launches) in times.items()}


def same(x, y):
    return all(np.array_equal(a.view(np.uint64) if a.dtype == np.float64 else a,
                              b.view(np.uint64) if b.dtype == np.float64 else b) for a, b in zip(x, y))


def report(n, rounds_ms, call_ms, launches):
    b = scan_bytes(n)
    return {"n": n, "call_ms": round(call_ms, 3), "rounds_ms": round(rounds_ms, 3), "scan_bytes": b,
            "scan_bytes_per_s": round(b / (rounds_ms * 1e-3), 1) if rounds_ms > 0 else None, "launches": launches}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genomes", type=int, default=1000)
    ap.add_argument("--length", type=int, default=5_000_000)
    ap.add_argument("--sizes", type=int, nargs="*", default=[5000, 20000])
    ap.add_argument("--repeat", type=int, default=2)
    ap.add_argument("--seed", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_nj needs a GPU"
    res = {"what": "neighbour joining and BIONJ on the device: all_vs_all_nj / all_vs_all_bionj (config 2) and gkd_nj / "
                   "gkd_bionj on device triangles", **card()}
    buf = torch.empty((100, a.length), dtype=torch.uint8, device="cuda")
    with gkd.Engine(k=21) as e:
        for g in range(a.genomes):
            # the generator of tools/bench_rect.py: families of 100, members mutated at 0.1 / 1 / 5 / 20 %
            gkd.synth(buf[g % 100], 0x5EED0000, g // 100, g % 100, [0.001, 0.01, 0.05, 0.2][g % 4] if g % 100 else 0.0)
            e.add(buf[g % 100])
            if g % 100 == 99:
                e.build()
        e.build()
        _, dense = measure(e, lambda: e.all_vs_all(want_inter=False), a.repeat)
        _, gd = e.all_vs_all(want_inter=False)
        res["config2"] = {"genomes": a.genomes, "length": a.length, "dense_all_vs_all": dense}
        got = {}
        for m, call in (("nj", e.all_vs_all_nj), ("bionj", e.all_vs_all_bionj)):
            call()  # warm-up
            before = e.metrics()["launches"]
            got[m], rd = measure(e, call, a.repeat)
            rd["launches"] = int(e.metrics()["launches"] - before) // a.repeat
            rd["rounds"] = int(e.metrics()["agglomerate_rounds"])
            res["config2"]["all_vs_all_" + m] = rd
        for m, (rows, call_ms, rounds_ms, launches) in timed_trees(e, torch.from_numpy(gd).to("cuda"), a.repeat).items():
            res["config2"]["all_vs_all_" + m]["equal_to_%s_of_dense" % m] = same(got[m], rows)
            res["config2"][m + "_of_device_triangle"] = report(a.genomes, rounds_ms, call_ms, launches)
    del buf
    torch.cuda.empty_cache()
    res["synthetic"] = []
    with gkd.Engine(k=21) as e:
        for n in a.sizes:
            dev = synthetic(n, a.seed + n)
            torch.cuda.synchronize()
            e.nj(dev)  # warm-up of this shape
            e.bionj(dev)
            for m, (rows, call_ms, rounds_ms, launches) in timed_trees(e, dev, a.repeat).items():
                r = {"method": m, **report(n, rounds_ms, call_ms, launches)}
                r["negative_lengths"] = int((rows[2] < 0).sum() + (rows[3] < 0).sum())
                res["synthetic"].append(r)
            del dev
            torch.cuda.empty_cache()
    # CPU reference: the numpy oracles at n = 1,000
    ref = synthetic(1000, a.seed).cpu().numpy()
    with gkd.Engine(k=21) as e:
        for m, oracle, call in (("nj", nj.nj, e.nj), ("bionj", lambda d, n: bionj.bionj(d, n)[0], e.bionj)):
            t0 = time.perf_counter()
            want = oracle(ref, 1000)
            cpu_s = time.perf_counter() - t0
            got = call(ref)
            eq = all(np.array_equal(np.asarray([w[c] for w in want], dtype=x.dtype).view(np.uint8), x.view(np.uint8))
                     for c, x in enumerate(got))
            res["cpu_oracle_n1000" if m == "nj" else "cpu_bionj_oracle_n1000"] = {"seconds": round(cpu_s, 3),
                                                                                  "equal_to_device": bool(eq)}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
