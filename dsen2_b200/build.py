"""Build ``dsen2_b200/_lib/libdsen2_b200.so`` in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "_lib", "libdsen2_b200.so")
SOURCES = ["patch_kernels.cu", "prep_kernels.cu", "conv_api.cu", "conv_pair.cu", "conv_tail.cu", "nodata.cu", "train_kernels.cu"]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(SRC, f) for f in os.listdir(SRC)] + [os.path.join(HERE, "..", "include", "dsen2_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "-shared", "-Xcompiler", "-fPIC", "-o", OUT] + [os.path.join(SRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libdsen2_b200.so")
    if verbose:
        sys.stderr.write(r.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
