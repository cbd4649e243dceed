"""bench.py --dump-outputs on a small workload: the files hold what the timed step returned for every pair, equal
to the oracle on the same generated genomes, and do not depend on how many steps ran."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, LENGTH = 30, 300_000


def _bench(out_dir, steps, warmup):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--genomes", str(N), "--length", str(LENGTH),
           "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out_dir)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-4000:]
    line = json.loads([x for x in p.stdout.splitlines() if x.startswith("{")][-1])
    assert line["steps"] == steps and line["config"]["pairs"] == N * (N - 1) // 2
    return {n: np.load(os.path.join(out_dir, n + ".npy")) for n in ("pair_index", "intersections", "distances")}


def test_dump_outputs_hold_every_pair_result(orc, tmp_path):
    import bench
    from oracle import synth as osynth

    a = _bench(tmp_path / "a", 2, 1)
    b = _bench(tmp_path / "b", 1, 0)
    total = N * (N - 1) // 2
    for name in a:
        assert a[name].dtype == np.float64 and a[name].shape == (total,), name
        assert np.array_equal(a[name], b[name]), name
    assert np.array_equal(a["pair_index"], np.arange(total))
    sets = [orc.IntSet(osynth.synth(LENGTH, bench.SEED, *bench.genome_params(g, N, 10)), 21) for g in range(N)]
    t = 0
    for i in range(N):
        for j in range(i + 1, N):
            assert a["intersections"][t] == sets[i].similarity(sets[j]), (i, j)
            assert a["distances"][t] == sets[i].distance(sets[j]), (i, j)
            t += 1
    assert (a["distances"] < 1.0).sum() >= 10 * 3  # the families' related pairs are in the workload
