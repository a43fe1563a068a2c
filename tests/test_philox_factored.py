"""The fused kernels draw their normals through philox_prefix / philox_lane / philox_finish (sgpmp_rng.cuh), which regroup
the rounds of philox4x32 so that the sample-invariant words are computed once per (t, k).  This checks, on the host (the
functions are __host__ __device__), that the composition gives philox4x32's words exactly, for every round count the build
accepts (SGPMP_PHILOX_ROUNDS >= 3), at the counters the kernels use: every DoF pair including the odd tail pair, time steps
up to 255, samples offset by a nonzero sample_gid0 (split-particle mode), particle ids offset by a problem offset, and draw
indices advanced per iteration."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "stoch_gpmp_b200", "csrc")

PROGRAM = r"""
#include <cstdio>
#include "sgpmp_rng.cuh"
using namespace sgpmp;

int main() {
    const uint64_t seeds[] = {0ull, 1234ull, 0xFFFFFFFFFFFFFFFFull, 0x9E3779B97F4A7C15ull};
    const uint32_t sample_gid0[] = {0u, 256u, 3u * 512u + 17u, 0xFFFFFF00u};
    const uint32_t pgid0[] = {0u, 38u * 16u, 6143u, 0xFFFFFFF0u};
    long n = 0, bad = 0;
    for (uint64_t seed : seeds)
        for (uint32_t it = 0; it < 4; ++it) {
            const RngKey key = make_rng_key(seed, 7u + 1000u * it);
            for (uint32_t g0 : pgid0)
                for (uint32_t pg = 0; pg < 3; ++pg) {
                    const uint32_t pgid = g0 + pg;
                    for (uint32_t t = 0; t < 256; t += 17)
                        for (uint32_t k = 0; k < 4; ++k) {           // k = 3: the tail pair of 7 DoF (and a full pair of 8)
                            const uint32_t x = philox_x(t, k), w = key.draw + it;
                            const uint4 pre = philox_prefix(x, pgid, w, key);
                            for (uint32_t s0 : sample_gid0)
                                for (uint32_t s = 0; s < 600; s += 37) {
                                    const uint32_t sample = s0 + s;
                                    const uint4 a = philox_finish(pre, philox_lane(sample, pgid, key), key);
                                    const uint4 b = philox4x32(make_uint4(x, sample, pgid, w), key);
                                    ++n;
                                    if (a.x != b.x || a.y != b.y || a.z != b.z || a.w != b.w) {
                                        if (++bad <= 5) printf("mismatch seed %llx it %u pgid %u t %u k %u sample %u\n",
                                                               (unsigned long long)seed, it, pgid, t, k, sample);
                                    }
                                }
                        }
                }
        }
    printf("checked %ld counters, %ld mismatches\n", n, bad);
    return bad != 0;
}
"""


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    pytest.skip("nvcc not found")


@pytest.mark.parametrize("rounds", range(3, 13))
def test_factored_philox_equals_philox4x32(tmp_path, rounds):
    src = tmp_path / "philox_factored.cu"
    exe = tmp_path / "philox_factored"
    src.write_text(PROGRAM)
    r = subprocess.run([_nvcc(), "-O2", "-std=c++17", "-DSGPMP_PHILOX_ROUNDS=%d" % rounds, "-I", CSRC,
                        "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "0 mismatches" in r.stdout


def test_factored_philox_needs_three_rounds(tmp_path):
    src = tmp_path / "philox_two_rounds.cu"
    src.write_text('#include "sgpmp_rng.cuh"\nint main() { return 0; }\n')
    r = subprocess.run([_nvcc(), "-std=c++17", "-DSGPMP_PHILOX_ROUNDS=2", "-I", CSRC, "-I", os.path.join(ROOT, "include"),
                        "-c", str(src), "-o", str(tmp_path / "x.o")], capture_output=True, text=True)
    assert r.returncode != 0 and "rounds 0-2 apart" in r.stderr
