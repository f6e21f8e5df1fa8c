"""In-tree build of libfrcnn_b200.so with nvcc for sm_100a (no GPU needed to build).

    python -m faster_rcnn_b200._build [--force]

All translation units are built with -fmad=false: the reference's numpy arithmetic rounds every
multiply and add separately, and none of these kernels is FMA-throughput bound.
"""
import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
OUT = os.path.join(_HERE, "libfrcnn_b200.so")
SOURCES = ["capi.cu", "proposals.cu", "nms.cu", "label.cu", "roi.cu", "roi_bwd.cu", "postproc.cu", "boxes.cu", "losses.cu", "evalmatch.cu", "image.cu",
           "sample.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale():
    if not os.path.isfile(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(_HERE, "..", "include", "frcnn_b200.h"),
                                                               os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source into faster_rcnn_b200/libfrcnn_b200.so.  Returns the path."""
    if not force and not _stale():
        return OUT
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + SOURCES + ["-o", OUT + ".tmp"]
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s" % (res.stdout, res.stderr))
    if verbose:
        sys.stderr.write(res.stderr)
    os.replace(OUT + ".tmp", OUT)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
