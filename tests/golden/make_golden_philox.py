"""Writes tests/golden/philox.npz: (ctr, key) -> curand_Philox4x32_10 output rows computed by curand's own header,
compiled for the HOST with plain nvcc (no GPU needed), as an independent check of oracle/sample_oracle.philox.

    python tests/golden/make_golden_philox.py

4096 random (ctr, key) pairs plus the edge cases (all zero, all ones, single set bits, the counters the samplers use).
"""
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

PROGRAM = r"""
#define QUALIFIERS static inline __host__ __device__
#include <curand_philox4x32_x.h>
#include <cstdio>
int main() {
  unsigned in[6];
  while (fread(in, sizeof(unsigned), 6, stdin) == 6) {
    uint4 r = curand_Philox4x32_10(make_uint4(in[0], in[1], in[2], in[3]), make_uint2(in[4], in[5]));
    unsigned out[4] = {r.x, r.y, r.z, r.w};
    fwrite(out, sizeof(unsigned), 4, stdout);
  }
  return 0;
}
"""


def _inputs():
    rng = np.random.default_rng(20261021)
    rows = [rng.integers(0, 1 << 32, (4096, 6), dtype=np.uint64).astype(np.uint32)]
    edge = [[0] * 6, [0xFFFFFFFF] * 6]
    for i in range(6):
        for bit in (0, 31):
            e = [0] * 6
            e[i] = 1 << bit
            edge.append(e)
    edge += [[5, 7, 0, 0, 1, 0], [16073, 127, 0, 1, 0xDEADBEEF, 0x12345678], [0, 0xFFFFFFFF, 0xFFFFFFFF, 2, 1, 1]]
    rows.append(np.array(edge, np.uint32))
    return np.concatenate(rows)


def main():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    inp = _inputs()
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "philox.cu"), os.path.join(tmp, "philox")
        with open(src, "w") as f:
            f.write(PROGRAM)
        subprocess.run([nvcc, "-O2", "-Wno-deprecated-gpu-targets", src, "-o", exe], check=True)
        out = subprocess.run([exe], input=inp.tobytes(), capture_output=True, check=True).stdout
    res = np.frombuffer(out, np.uint32).reshape(-1, 4)
    assert len(res) == len(inp)
    np.savez_compressed(os.path.join(HERE, "philox.npz"), ctr=inp[:, :4], key=inp[:, 4:], out=res)
    print("wrote %d rows" % len(res))


if __name__ == "__main__":
    main()
