#!/usr/bin/env python
"""bench.py -- headline benchmark of the k-mer set distance hot path (BASELINE.json metric).

Workload (config.workload): BASELINE configs[1] -- N synthetic 5 Mbp genomes (10 families of mutated
descendants, SURVEY 8d generator), DNA K=21, all-vs-all Jaccard distance = N(N-1)/2 pairs.  Default
N=1000 (499,500 pairs) on one B200.  One "step" = one full pass of the hot path: kernel 1 (pack) ->
2 (canonical encode + mix) -> 3 (MSD bucket sort + unique + bucket tables) -> 4 (block join: 64 row sets per
shared-memory hash table, every column set probed once per row block; the bucket-merge kernel serves small
calls and GKD_ISECT_ALGO=merge) -> 5 (distance epilogue).

  value  : pairs/s with the genome text already resident in HBM when the step starts
  e2e    : pairs/s through the C ABI with HOST (pinned) text buffers in, host result arrays out
  roofline: kernel 4 algorithmic bytes 8*(|A|+|B|) per pair (SURVEY 8d) / CUDA-event time of its launches
  cpu_baseline: the oracle's HashSet<String> port of the reference on a bounded sample (rank 0, N=1)

N>1 (torchrun): strong scaling of the same workload -- rank r builds the sets of its slice of the
genomes and owns a set of rank blocks of the pair matrix; the peers' sets arrive as panels over NCCL
send/recv while earlier blocks are being intersected and are adopted in place
(genome/distance_b200/sharding.py: ring_all_vs_all); no cross-rank reduction.

`--impl reference` times the reference's own CPU algorithm (oracle string-set port of
FastaDistanceProcessor; the Java original cannot run here: no JVM, arithmetic in an un-vendored artifact)
on a bounded sample.  That arm never loads the product library.

`--dump-outputs DIR` writes what the last timed step returned (intersection counts and distances of the
pairs) to DIR as float64 .npy files, so that two builds can be compared output for output on the same
seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "genome pairs/sec all-vs-all k-mer distance"
UNIT = "pairs/s"
SEED = 0x5EED0000
RATES = [0.001, 0.01, 0.05, 0.2]
DUMP_PAIRS = 2_000_000  # --dump-outputs: three float64 arrays of at most this length, 48 MB


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--genomes", type=int, default=int(os.environ.get("GKD_BENCH_GENOMES", "1000")))
    ap.add_argument("--length", type=int, default=int(os.environ.get("GKD_BENCH_LENGTH", "5000000")))
    ap.add_argument("--families", type=int, default=10)
    ap.add_argument("--k", type=int, default=21)
    ap.add_argument("--panel", type=int, default=int(os.environ.get("GKD_BENCH_PANEL", "128")),
                    help="sets per exchanged panel (N>1)")
    ap.add_argument("--cpu-sample", type=int, default=int(os.environ.get("GKD_BENCH_CPU_SAMPLE", "22")),
                    help="largest CPU sample (genomes); the reference arm shrinks it to fit its time budget")
    ap.add_argument("--cpu-budget", type=float, default=float(os.environ.get("GKD_BENCH_CPU_BUDGET_S", "240")),
                    help="wall-clock budget (s) of the whole --impl reference run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--other-configs", action="store_true", default=os.environ.get("GKD_BENCH_OTHER", "0") == "1",
                    help="also run BASELINE configs 1, 3 and 5 at full size (N=1) and report them as other_configs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's results to DIR/{pair_index,intersections,"
                         f"distances}}.npy (float64, pairs in row-major upper-triangle order; a fixed seeded sample "
                         f"of {DUMP_PAIRS} pairs when there are more)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")
    return a


def genome_params(g: int, n_genomes: int, families: int):
    """family / member / substitution rate of genome g (10 families x 100 at the default size)"""
    per = max(1, (n_genomes + families - 1) // families)
    fam, mem = g // per, g % per
    rate = 0.0 if mem == 0 else RATES[mem % len(RATES)]
    return fam, mem, rate


def workload_name(a):
    return (f"{a.genomes} synthetic {a.length / 1e6:g} Mbp genomes all-vs-all DNA k-mer Jaccard, K={a.k} "
            f"({a.genomes * (a.genomes - 1) // 2} pairs)")


def config_dict(a, world):
    """identical in both arms: the workload the metric is quoted on, and the bounded sample of it that the CPU
    arm (reference arm / cpu_baseline) actually runs"""
    n = a.genomes
    return {"workload": workload_name(a), "k": a.k, "genomes": n, "genome_bp": a.length, "pairs": n * (n - 1) // 2,
            "families": a.families,
            "cpu_sample": f"CPU legs run the first n <= {a.cpu_sample} genomes of this workload with the reference's "
                          "batch=20 decomposition; n is chosen to fit the leg's time budget and stated in cpu_baseline.sample",
            "l2": "inputs (21 MB per set, 21 GB total) are far larger than L2; no flush needed"}


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.path = f"/tmp/gkd_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    mx.append(float(p[2]))
                except ValueError:
                    continue
                for name, v in zip(names, p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline (oracle port; the only place bench.py executes oracle/, and this leg never
# imports the product package: inputs come from the oracle's own numpy port of the generator)
# ------------------------------------------------------------------------------------------------
def host_sample(a, n_sample: int):
    from oracle import synth as osynth

    seqs = []
    for g in range(n_sample):
        fam, mem, rate = genome_params(g, a.genomes, a.families)
        seqs.append(osynth.synth(a.length, SEED, fam, mem, rate).tobytes())
    return seqs


def run_cpu_reference(a, n_sample: int, seqs=None, mode: int = 0):
    """FastaDistanceProcessor's algorithm on the first n_sample genomes of the workload with the reference's
    own decomposition: batches of 20 sets cached serially (:151-155), rows of a batch in parallel (:157-158),
    the set of a column outside the batch rebuilt for every pair (:183-184).  mode 0 = HashSet<String> port
    (the reference's representation), mode 1 = sorted canonical uint64 sets + merge (a stronger CPU line).
    Returns (pairs/s, seconds, threads, pairs)."""
    from oracle import oracle as orc

    seqs = seqs if seqs is not None else host_sample(a, n_sample)
    threads = orc.max_threads()
    t0 = time.perf_counter()
    orc.fasta_dist(seqs, a.k, alphabet=orc.DNA, batch=20, threads=threads, mode=mode)
    dt = time.perf_counter() - t0
    pairs = n_sample * (n_sample - 1) // 2
    return pairs / dt, dt, threads, pairs


def cpu_phase_costs(a, seqs):
    """single-thread cost of the two phases of the reference's algorithm (one set build, one probe)"""
    from oracle import oracle as orc

    t0 = time.perf_counter()
    s0 = orc.StrSet(seqs[0], a.k)
    t1 = time.perf_counter()
    s1 = orc.StrSet(seqs[1], a.k)
    t2 = time.perf_counter()
    s0.similarity(s1)
    t3 = time.perf_counter()
    return {"set_build_s_per_genome_1thread": 0.5 * (t2 - t0), "probe_s_per_pair_1thread": t3 - t2,
            "note": "HashSet<String> port; the reference pays one build per uncached column per pair plus one probe"}


def choose_sample(a, budget_s, phases, threads):
    """largest sample (4 .. --cpu-sample genomes) whose modelled step time fits budget_s: the batch cache is
    built serially, the pairs run on the rows' threads at ~50 % parallel efficiency (memory-bound probes)"""
    tb, tp = phases["set_build_s_per_genome_1thread"], phases["probe_s_per_pair_1thread"]
    best = 4
    for n in range(4, max(4, a.cpu_sample) + 1):
        cached = min(n, 20)
        pairs_cached = cached * (cached - 1) // 2
        pairs_rebuilt = n * (n - 1) // 2 - pairs_cached - max(0, n - 20) * (max(0, n - 20) - 1) // 2
        later = max(0, n - 20)  # second batch: its own cache and pairs
        t = cached * tb + later * tb + (pairs_cached * tp + later * (later - 1) // 2 * tp +
                                         pairs_rebuilt * (tb + tp)) / max(1.0, 0.5 * min(threads, cached))
        if t <= budget_s:
            best = n
    return best


def cpu_baseline_block(a, value, dt, threads, pairs, extra=None, n_sample=None):
    n_sample = n_sample or a.cpu_sample
    sample = (f"first {n_sample} genomes of the workload ({pairs} pairs in {dt:.1f} s): reference decomposition, "
              f"batch=20 cached serially, rows in parallel on {threads} threads, uncached columns rebuilt per pair; "
              f"C port of the reference's HashSet<String> algorithm, not the JVM")
    blk = {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
           "pairs_per_s_per_core": value / max(threads, 1)}
    if extra:
        blk.update(extra)
    return blk


def reference_main(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as orc

    # size the per-step sample so that the whole run (warm-up + timed steps) fits the budget
    seqs = host_sample(a, min(a.cpu_sample, 2))
    phases = cpu_phase_costs(a, seqs)
    n_sample = choose_sample(a, a.cpu_budget / max(1, a.warmup + a.steps), phases, orc.max_threads())
    seqs = host_sample(a, n_sample)
    vals = []
    threads = pairs = 0
    for s in range(a.warmup + a.steps):
        v, dt, threads, pairs = run_cpu_reference(a, n_sample, seqs)
        if s >= a.warmup:
            vals.append((v, dt))
    value = sum(p for p, _ in vals) / len(vals)
    ms = 1e3 * sum(d for _, d in vals) / len(vals)
    iv, idt, _, _ = run_cpu_reference(a, n_sample, seqs, mode=1)
    extra = {"integer_mode": {"value": iv, "unit": UNIT, "seconds": idt,
                              "what": "same sample and decomposition on sorted canonical uint64 sets with a linear merge "
                                      "(not the reference's representation; shown so the string sets do not flatter the GPU)"},
             "phases": phases}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic", "config": config_dict(a, a.gpus),
            "cpu_baseline": cpu_baseline_block(a, value, ms / 1e3, threads, pairs, extra, n_sample),
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "product_library_loaded": "genome.distance_b200" in sys.modules}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def dump_outputs(out_dir, inter, dist_out):
    """write one step's per-pair results as float64 .npy files; pair_index holds each entry's row-major index in
    the strict upper triangle (counts and indices stay exact in float64 below 2**53)"""
    import numpy as np

    total = inter.size
    if total > DUMP_PAIRS:
        idx = np.sort(np.random.default_rng(SEED).choice(total, DUMP_PAIRS, replace=False))
    else:
        idx = np.arange(total)
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("pair_index", idx), ("intersections", inter[idx]), ("distances", dist_out[idx])):
        np.save(os.path.join(out_dir, name + ".npy"), arr.astype(np.float64))


def main():
    a = parse_args()
    if a.impl == "reference":
        return reference_main(a)

    import numpy as np
    import torch
    import torch.distributed as dist

    import genome.distance_b200 as gkd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs a single process: at N>1 the pair results stay on their ranks")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: libgkd has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from genome.distance_b200 import sharding

    N, Lg = a.genomes, a.length
    total_pairs = N * (N - 1) // 2
    my_ids = sharding.genome_slice(N, world, rank)

    # synthetic inputs: this rank's genomes as text in HBM, and a pinned host copy for the e2e leg
    d_text = torch.empty((len(my_ids), Lg), dtype=torch.uint8, device=dev)
    for r, g in enumerate(my_ids):
        fam, mem, rate = genome_params(g, N, a.families)
        gkd.synth(d_text[r], SEED, fam, mem, rate, device=local)
    h_text = None
    if not a.no_e2e:
        h_text = torch.empty((len(my_ids), Lg), dtype=torch.uint8, pin_memory=True)
        h_text.copy_(d_text)
    torch.cuda.synchronize()

    # N>1: one build batch (= one set arena = one exchange panel) per `panel` genomes of the slice
    ws = 0 if world == 1 else min(len(my_ids), a.panel) * Lg * 16 + (1 << 24)
    eng = gkd.Engine(k=a.k, device=local, workspace_bytes=ws)
    ext = torch.cuda.ExternalStream(eng.stream_ptr, device=dev)
    inter = np.empty(total_pairs if world == 1 else 0, dtype=np.uint64)
    dist_out = np.empty(total_pairs if world == 1 else 0, dtype=np.float64)
    check = {"pairs": 0, "inter_sum": 0, "related": 0}

    def sink(gi, gj, bi, bd):
        """every block of results lands in host arrays (inside the timed region); keep a checksum"""
        bi = np.asarray(bi).reshape(-1)
        check["pairs"] += bi.size
        check["inter_sum"] += int(bi.sum(dtype=np.uint64))
        check["related"] += int((np.asarray(bd).reshape(-1) < 1.0).sum())

    def one_step(text):
        """one pass of the hot path over the whole workload; returns engine metrics"""
        t_start = time.perf_counter()
        eng.reset()
        for r in range(len(my_ids)):
            eng.add(text[r])
        t_add = time.perf_counter()
        eng.build()
        t_build = time.perf_counter()
        stats = {}
        if world > 1:
            check.update(pairs=0, inter_sum=0, related=0)
            sharding.ring_all_vs_all(eng, N, world, rank, dev, panel_genomes=a.panel, sink=sink, stats=stats)
        else:
            eng.all_vs_all_range(N, 0, total_pairs, inter_out=inter, dist_out=dist_out)
        m = eng.metrics()
        m["wall_add_ms"] = 1e3 * (t_add - t_start)
        m["wall_build_ms"] = 1e3 * (t_build - t_add)
        m["wall_exchange_exposed_ms"] = 1e3 * stats.get("exposed_wait_s", 0.0)
        m["wall_distance_ms"] = 1e3 * (time.perf_counter() - t_build)
        return m

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(text, steps):
        """(max-over-ranks seconds for `steps` steps on the device, per-step metrics)"""
        mets = []
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(ext)
        for _ in range(steps):
            mets.append(one_step(text))
        e1.record(ext)
        barrier()
        wall = time.perf_counter() - t0
        dev_s = e0.elapsed_time(e1) / 1e3
        t = torch.tensor([dev_s, wall], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), mets

    # warm-up (also sizes every pool), then the timed region with the clock sampler running
    for _ in range(a.warmup):
        one_step(d_text)
    launches0 = eng.metrics()["launches"]
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    dev_s, wall_s, mets = timed(d_text, a.steps)
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs:  # before the e2e leg, which writes its results into the same arrays
        dump_outputs(a.dump_outputs, inter, dist_out)
    launches = eng.metrics()["launches"] - launches0
    if world > 1:
        t = torch.tensor([float(launches), float(check["pairs"])], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        launches, pairs_done = int(t[0]), int(t[1])
        assert pairs_done == total_pairs, (pairs_done, total_pairs)

    value = a.steps * total_pairs / dev_s
    ms_per_step = 1e3 * dev_s / a.steps

    # e2e: same step from pinned host text (H2D inside), results to host arrays (D2H inside)
    e2e = None
    if h_text is not None:
        one_step(h_text)  # one warm-up of the host path (pinned staging, pools)
        e_dev, e_wall, emets = timed(h_text, a.steps)
        e_s = max(e_dev, e_wall)
        h2d = sum(m["h2d_bytes"] for m in emets) / a.steps
        d2h = sum(m["d2h_bytes"] for m in emets) / a.steps
        if world > 1:
            t = torch.tensor([h2d, d2h], dtype=torch.float64, device=dev)
            dist.all_reduce(t)
            h2d, d2h = float(t[0]), float(t[1])
        e2e = {"value": a.steps * total_pairs / e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e_s / a.steps}

    # roofline of the dominant kernel (kernel 4), from the engine's CUDA events on its own stream, summed over
    # the launches of a step (one launch at N=1; one per block of the ring at N>1); slowest rank at N>1
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    isect_ms = sum(m["total_intersect_ms"] for m in mets) / len(mets)
    isect_bytes = sum(m["total_intersect_bytes"] for m in mets) / len(mets)
    if world > 1:
        t = torch.tensor([isect_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        isect_ms = float(t[0])
    achieved = isect_bytes / (isect_ms * 1e-3) / 1e9 if isect_ms > 0 else 0.0
    traffic, traffic_src, stored = None, None, None
    kernel_id = int(mets[-1].get("intersect_kernel", 0))
    joined = kernel_id == 5
    tpath = os.path.join(ROOT, "profiles", "intersect_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))["join" if joined else "merge"]
            traffic = tj["dram_bytes_per_algorithmic_byte"] * isect_bytes
            traffic_src = ("ESTIMATED, not measured in this run: ncu dram__bytes_read+write per algorithmic byte of the "
                           f"profiled launch ({tj.get('source', 'profiles/')}) x this run's algorithmic bytes")
            stored = tj.get("stored_bytes_per_algorithmic_byte")
        except Exception:
            traffic = None
    kname = {3: "k_intersect_bucket<uint32_t> (bucket merge, 32-bit low words)",
             4: "k_intersect_bucket<uint64_t> (bucket merge, 64-bit keys)",
             5: "k_join (block join: 64 row sets share one shared-memory hash table per key range; every column set "
                "is probed once per row block)"}
    if joined:
        note = ("achieved = 8*(|A|+|B|) bytes per pair (SURVEY 8d definition: two sorted uint64 sets streamed per pair) / "
                "CUDA-event time of kernel 4.  The block join does NOT stream both sets per pair: one probe of a column key "
                "serves 64 rows, every column set is read once per block of 64 rows (from L2: the tasks run range-major) "
                "and once per step from HBM, so the algorithmic figure is far above the HBM peak and says how much "
                "pair-streaming work was avoided, not how busy HBM is.  moved_frac = bytes actually moved L2->SM / time / "
                "peak (estimated from the committed ncu ratio); the kernel's limiter is SM instruction issue and "
                "shared-memory probe latency (62 % issue slots busy in profiles/r2j_join_ncu_full.txt)")
    else:
        note = ("achieved = 8*(|A|+|B|) bytes per pair (SURVEY 8d definition: sorted uint64 sets) / CUDA-event time "
                "of kernel 4.  The kernel reads the sets in a compressed layout (32-bit low words + bucket table, "
                "~4.25 stored bytes per key) and the row sets are served from L2, so the algorithmic figure can "
                "exceed the HBM peak; stored_frac is the same fraction on the bytes actually stored")
    roofline = {"kernel": kname.get(kernel_id, "k_intersect_bucket"), "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_step": isect_bytes, "ms_per_step": isect_ms, "note": note,
                ("moved_frac" if joined else "stored_frac"): (achieved / peak) * stored if stored else None}
    build_ms = sum(m["encode_ms"] + m["sort_ms"] + m["unique_ms"] for m in mets) / len(mets)
    kpos = sum(m["kmer_positions"] for m in mets) / len(mets)
    stages = {"encode_ms": sum(m["encode_ms"] for m in mets) / len(mets),
              "sort_ms": sum(m["sort_ms"] for m in mets) / len(mets),
              "unique_ms": sum(m["unique_ms"] for m in mets) / len(mets),
              "intersect_ms": isect_ms, "epilogue_ms": sum(m["epilogue_ms"] for m in mets) / len(mets),
              "kmers_hashed_per_s_this_rank": kpos / (build_ms * 1e-3) if build_ms > 0 else 0.0,
              "sort_passes": mets[-1]["sort_passes"],
              "wall_ms": {k: sum(m[k] for m in mets) / len(mets) for k in
                          ("wall_add_ms", "wall_build_ms", "wall_exchange_exposed_ms", "wall_distance_ms")}}

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        seqs = host_sample(a, a.cpu_sample)
        v, dt, threads, pairs = run_cpu_reference(a, a.cpu_sample, seqs)
        iv, idt, _, _ = run_cpu_reference(a, a.cpu_sample, seqs, mode=1)
        cpu = cpu_baseline_block(a, v, dt, threads, pairs,
                                 {"integer_mode": {"value": iv, "unit": UNIT, "seconds": idt,
                                                   "what": "same sample and decomposition on sorted canonical uint64 sets "
                                                           "with a linear merge (not the reference's representation)"},
                                  "phases": cpu_phase_costs(a, seqs)})

    other = None
    if a.other_configs and world == 1:
        eng.close()
        eng = None
        del d_text, h_text
        torch.cuda.empty_cache()
        from tools import run_config

        other = []
        for fn in (run_config.c1, lambda: run_config.c3(10000, 500, 4000), lambda: run_config.c5(2000)):
            try:
                other.append(fn())
            except Exception as ex:  # a failed side config must not lose the headline line
                other.append({"error": repr(ex)})

    if rank == 0:
        cfg = config_dict(a, world)
        cfg["sharding"] = (f"rank blocks of the pair matrix x{world}, peers' sets arrive as panels of <= {a.panel} sets "
                           "over NCCL send/recv and are intersected in groups of up to 1024 sets; the transfers of the "
                           "next group run under kernel 4 of the current one") if world > 1 else "single GPU"
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "u64", "data": "synthetic", "config": cfg,
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
                "clocks": clocks, "stages": stages, "wall_s_timed_region": wall_s}
        if world > 1:
            line["critical_path_collective"] = ("none by construction (point-to-point panels, posted one compute group ahead); what "
                                                "stays exposed when kernel 4 is shorter than the transfer is reported per step as "
                                                "stages.wall_ms.wall_exchange_exposed_ms")
            line["checksum"] = {"pairs": total_pairs, "related_pairs_this_rank": check["related"]}
        if other is not None:
            line["other_configs"] = other
        print(json.dumps(line), flush=True)
    if eng is not None:
        eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
