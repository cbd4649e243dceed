"""The numpy port of the key mix that tests/test_gpu_join_redo.py uses to craft imported key sets must be the header's
mix: a host program compiled against gkd_internal.cuh prints mix_key / unmix_key of random keys, and the port must
give the same values.  Runs without a GPU."""
import os
import shutil
import subprocess

import numpy as np

from test_gpu_join_redo import canonical_only, make_mix, mix, revcomp, unmix

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROGRAM = r"""
#include <cmath>
#include <cstdio>
#include "gkd_internal.cuh"
int main(int argc, char **argv) {
    const gkd::MixParams p = gkd::make_mix(atoi(argv[1]));
    unsigned long long x;
    while (scanf("%llu", &x) == 1)
        printf("%llu %llu\n", (unsigned long long)gkd::mix_key(x, p), (unsigned long long)gkd::unmix_key(x, p));
    return 0;
}
"""


def _cuda_include():
    home = os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH")
    if not home:
        nvcc = shutil.which("nvcc")
        home = os.path.dirname(os.path.dirname(nvcc)) if nvcc else "/usr/local/cuda"
    return os.path.join(home, "include")


def test_numpy_mix_port_equals_the_header(tmp_path):
    src = tmp_path / "mix.cpp"
    src.write_text(PROGRAM)
    exe = tmp_path / "mix"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           "-I", os.path.join(ROOT, "genome", "distance_b200", "csrc"), "-I", _cuda_include(),
                           str(src), "-o", str(exe)])
    rng = np.random.default_rng(1)
    for bits in (16, 32, 42, 50, 64):
        p = make_mix(bits)
        mask = p[0]
        keys = rng.integers(0, mask, size=2000, dtype=np.uint64, endpoint=True)
        keys = np.concatenate([keys, np.array([0, 1, mask - 1, mask], dtype=np.uint64)])
        out = subprocess.run([str(exe), str(bits)], input="\n".join(str(int(x)) for x in keys), capture_output=True,
                             text=True, check=True).stdout.split()
        want = np.array([int(x) for x in out], dtype=np.uint64).reshape(-1, 2)
        assert np.array_equal(mix(keys, p), want[:, 0]), bits
        assert np.array_equal(unmix(keys, p), want[:, 1]), bits
        assert np.array_equal(unmix(mix(keys, p), p), keys), bits
        assert int(mix(np.array([mask], dtype=np.uint64), p)[0]) == mask, bits  # the all-ones key maps to itself


def test_revcomp_port():
    """2-bit reverse complement: an involution; palindromes only for even K; canonical = not above its complement"""
    rng = np.random.default_rng(2)
    assert int(revcomp(np.array([0b00011011], dtype=np.uint64), 4)[0]) == 0b00011011  # acgt is its own complement
    assert int(revcomp(np.array([0b000110], dtype=np.uint64), 3)[0]) == 0b011011  # acg -> cgt
    for k in (5, 16, 21, 25, 32):
        keys = rng.integers(0, 1 << (2 * k), size=5000, dtype=np.uint64, endpoint=False) if k < 32 else \
            rng.integers(0, np.iinfo(np.uint64).max, size=5000, dtype=np.uint64, endpoint=True)
        rc = revcomp(keys, k)
        assert np.array_equal(revcomp(rc, k), keys), k
        if k % 2:
            assert not (rc == keys).any(), k
        c = canonical_only(keys, k)
        assert (c <= revcomp(c, k)).all() and c.size >= keys.size // 2 - 200, k
