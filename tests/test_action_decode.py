"""The random policy's action decode (action_from_word in csrc/philox.cuh) against the Float64 expression it replaces, on all 2^32
words: Float32(fma(1 + u, 2, -3)) with 1 + u = w * 2^-32 assembled in a double's significand.  The harness is compiled from the
shipped header, so the test checks the helper the rollout kernel calls, not a copy of it.  CPU only (nvcc compiles host code)."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "master-thesis-deep-reinforcement-learning-ddpg-in-home-energy-management_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

HARNESS = r"""
#include <math.h>
#include <stdio.h>
#include <string.h>
#include "philox.cuh"

static float old_decode(uint32_t w) {  // the Float64 decode the rollout kernel used before action_from_word
  const uint64_t bits = ((uint64_t)(0x3ff00000u | (w >> 12)) << 32) | (uint32_t)(w << 20);
  double one_plus_u;
  memcpy(&one_plus_u, &bits, 8);
  return (float)fma(one_plus_u, 2.0, -3.0);
}

int main() {
  long long bad = 0;
#pragma omp parallel for reduction(+ : bad) schedule(static)
  for (long long hi = 0; hi < 65536; ++hi) {
    for (uint32_t lo = 0; lo < 65536u; ++lo) {
      const uint32_t w = ((uint32_t)hi << 16) | lo;
      const float a = action_from_word(w), b = old_decode(w);
      if (memcmp(&a, &b, 4) != 0) {
        if (bad < 4) printf("mismatch w=%08x new=%a old=%a\n", w, a, b);
        ++bad;
      }
    }
  }
  printf("mismatches %lld\n", bad);
  return bad != 0;
}
"""


@pytest.mark.skipif(not (os.path.exists(NVCC) or shutil.which("nvcc")), reason="needs nvcc to compile the host harness")
def test_action_decode_all_words(tmp_path):
    src = tmp_path / "decode.cu"
    src.write_text(HARNESS)
    exe = tmp_path / "decode"
    nvcc = NVCC if os.path.exists(NVCC) else shutil.which("nvcc")
    subprocess.check_call([nvcc, "-O2", "-std=c++17", "-I", CSRC, "-Xcompiler", "-fopenmp,-ffp-contract=off", "-ccbin", "/usr/bin/g++",
                           str(src), "-o", str(exe)])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "mismatches 0" in out.stdout, out.stdout + out.stderr
