#!/usr/bin/env python
"""Selections against the dense calls on config-2-sized data (1000 x 5 Mbp from the synthetic generator) on one GPU,
in one command, printing one JSON line:

* dense gkd_all_vs_all against gkd_all_vs_all_range_within over the whole triangle at two thresholds;
* dense gkd_query_vs_ref against gkd_query_vs_ref_nearest (k = 1 and k = 16, max_dist 1.0) on a 500 x 500 rectangle;
* the `gkd fastaDist` command on a FASTA file of the same genomes, with and without --maxDist: wall time and report size.

Per call: wall time (host clock around the call, which ends in a device synchronise; median of --repeat), kernel-4 ms and
kernel-5 ms (dense epilogue or selection, CUDA events of the library), bytes copied device to host, and hits.  The card's
name and power limit are read in the same run.  Writes nothing in the tree; the FASTA file and reports go to a
temporary directory that is removed at the end (--out also writes the JSON line to a file).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import genome.distance_b200 as gkd  # noqa: E402

GKD = os.path.join(ROOT, "genome", "distance_b200", "gkd")


def card():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = q.stdout.strip() or q.stderr.strip()
    except OSError as ex:
        info["nvidia_smi"] = "unavailable: %s" % ex
    return info


def measure(e, fn, repeat):
    """median wall time of `repeat` calls, with the library's metrics and the D2H bytes of the last one"""
    walls, out, m = [], None, None
    for _ in range(repeat):
        before = e.metrics()["d2h_bytes"]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        walls.append(time.perf_counter() - t0)
        m = e.metrics()
        m["d2h_call"] = m["d2h_bytes"] - before
    return out, {"wall_ms": round(1e3 * statistics.median(walls), 3), "kernel4_ms": round(m["intersect_ms"], 3),
                 "kernel5_ms": round(m["epilogue_ms"], 3), "d2h_bytes": int(m["d2h_call"]), "pairs": int(m["pairs"])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genomes", type=int, default=1000)
    ap.add_argument("--length", type=int, default=5_000_000)
    ap.add_argument("--rect", type=int, default=500)
    ap.add_argument("--thresholds", type=float, nargs=2, default=[0.1, 0.9])
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--cli-max-dist", type=float, default=0.5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_select needs a GPU"
    res = {"what": "selection epilogues against the dense calls", "genomes": a.genomes, "length": a.length, **card()}
    n = a.genomes
    with tempfile.TemporaryDirectory(prefix="gkd_bench_select_") as tmp:
        fa = os.path.join(tmp, "genomes.fa")
        buf = torch.empty((100, a.length), dtype=torch.uint8, device="cuda")
        with gkd.Engine(k=21) as e, open(fa, "wb") as f:
            for g in range(n):
                # the generator of tools/bench_rect.py: families of 100, members mutated at 0.1 / 1 / 5 / 20 %
                gkd.synth(buf[g % 100], 0x5EED0000, g // 100, g % 100, [0.001, 0.01, 0.05, 0.2][g % 4] if g % 100 else 0.0)
                e.add(buf[g % 100])
                f.write(b">g%04d synthetic\n" % g)
                f.write(buf[g % 100].cpu().numpy().tobytes())
                f.write(b"\n")
                if g % 100 == 99:
                    e.build()
            e.build()
            total = n * (n - 1) // 2
            e.all_vs_all()  # warm-up of the dense and the selection paths
            e.all_vs_all_within(a.thresholds[0])
            (inter, dist), res["dense_all_vs_all"] = measure(e, e.all_vs_all, a.repeat)
            for D in a.thresholds:
                (wa, wb, wi, wd), r = measure(e, lambda: e.all_vs_all_within(D), a.repeat)
                keep = dist <= D
                r["hits"] = int(wa.size)
                r["equal_to_dense_filtered"] = bool(np.array_equal(wi, inter[keep]) and np.array_equal(wd, dist[keep]))
                res["within_%g" % D] = r
            q = np.arange(a.rect, dtype=np.uint32)
            rr = np.arange(a.rect, min(2 * a.rect, n), dtype=np.uint32)
            e.query_vs_ref(q, rr)
            e.query_vs_ref_nearest(q, rr, 1, 1.0)
            (qi, qd), res["dense_query_vs_ref_%dx%d" % (q.size, rr.size)] = measure(e, lambda: e.query_vs_ref(q, rr), a.repeat)
            for k in (1, 16):
                (pos, _, nd, nf), r = measure(e, lambda: e.query_vs_ref_nearest(q, rr, k, 1.0), a.repeat)
                order = np.lexsort((np.tile(np.arange(rr.size), (q.size, 1)), qd), axis=1)[:, :k]
                r["hits"] = int(nf.sum())
                r["equal_to_dense_sorted"] = bool(np.array_equal(pos, order) and
                                                  np.array_equal(nd, np.take_along_axis(qd, order, axis=1)))
                res["nearest_k%d" % k] = r
        del buf
        torch.cuda.empty_cache()
        for name, extra in (("cli_fastaDist", []), ("cli_fastaDist_maxDist_%g" % a.cli_max_dist, ["--maxDist", repr(a.cli_max_dist)])):
            rep = os.path.join(tmp, "report.tbl")
            t0 = time.perf_counter()
            p = subprocess.run([GKD, "fastaDist", "-i", fa, "-o", rep] + extra, capture_output=True, text=True)
            wall = time.perf_counter() - t0
            assert p.returncode == 0, p.stderr
            with open(rep, "rb") as f:
                lines = sum(1 for _ in f) - 1
            res[name] = {"wall_s": round(wall, 3), "report_bytes": os.path.getsize(rep), "report_lines": lines}
            os.remove(rep)
        res["fasta_bytes"] = os.path.getsize(fa)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
