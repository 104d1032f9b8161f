"""Builds libb200vton.so (hand-written sm_100a CUDA behind the C ABI of include/b200vton.h) in-tree with nvcc.

The shared object lives next to this file so it travels with the repo snapshot to the GPU box. Rebuilds only when a
source is newer than the library.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libb200vton.so")
SOURCES = ["host.cu", "gemm.cu", "gemm2.cu", "attn.cu", "attn6.cu", "attn_cross.cu", "attn_enc.cu", "conv_tf32.cu", "norm_f32.cu", "vae_f32.cu", "norm.cu", "elementwise.cu", "sched.cu", "capi.cu"]
HEADERS = ["common.cuh", "gemm_common.cuh", "host.h", os.path.join("..", "..", "include", "b200vton.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


STAMP = LIB + ".srchash"


def _source_hash():
    """Content hash of every source/header (mtimes are meaningless after the repo is copied to the GPU box)."""
    import hashlib
    h = hashlib.sha256()
    for s in SOURCES + HEADERS:
        with open(os.path.join(CSRC, s), "rb") as f:
            h.update(s.encode() + b"\0" + f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def needs_build():
    if not os.path.exists(LIB) or not os.path.exists(STAMP):
        return True
    with open(STAMP) as f:
        return f.read().strip() != _source_hash()


def build(force=False, verbose=False):
    """Compile every translation unit for sm_100a and link libb200vton.so. Returns the library path."""
    if not force and not needs_build():
        return LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    procs = []
    objs = []
    for s in SOURCES:
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, s), "-o", obj]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"nvcc failed for {s}:\n{out}\n")
        elif verbose and out:
            sys.stderr.write(f"--- {s}\n{out}\n")
    if failed:
        raise RuntimeError("libb200vton build failed")
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    with open(STAMP, "w") as f:
        f.write(_source_hash())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
