"""Builds nisqa_b200/libnisqa_b200.so in-tree with nvcc for sm_100a (no GPU needed to build).

    python -m nisqa_b200.build [--force]
"""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libnisqa_b200.so")
STAMP = os.path.join(HERE, ".libnisqa_b200.stamp")
SOURCES = ["engine.cu", "frontend.cu", "conv1.cu", "conv_split.cu", "conv12.cu", "td.cu", "td_tiled.cu", "wavio.cpp", "flac.cpp", "resample.cpp", "resample_gpu.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--shared"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _digest():
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    files.append(os.path.join(os.path.dirname(HERE), "include", "nisqa_b200.h"))
    for f in files:
        with open(f, "rb") as fh:       # (file NAME, not path: the digest must not depend on where the tree is checked out)
            h.update(os.path.basename(f).encode()); h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def kernel_digest():
    """Digest of the kernel sources alone (*.cu, *.cuh except engine.cu, + flags): what a measured per-kernel table (profiles/roofline_traffic.json)
    is tied to - a change to the host-side readers does not invalidate it."""
    h = hashlib.sha256()
    for name in sorted(os.listdir(CSRC)):
        if name.endswith((".cu", ".cuh")) and name != "engine.cu":        # (engine.cu holds the host side: ABI, passes, packing)
            with open(os.path.join(CSRC, name), "rb") as fh:
                h.update(name.encode()); h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    dg = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == dg:
        return LIB
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB, "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libnisqa_b200.so")
    if verbose:
        sys.stderr.write(r.stderr)
    with open(STAMP, "w") as f:
        f.write(dg)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
