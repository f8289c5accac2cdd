"""Build libtmf_sm100a.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtmf_sm100a.so")
SOURCES = ["api.cu", "conv_direct.cu", "conv_umma.cu", "conv_umma_col.cu", "wgrad_umma.cu", "wgrad_umma_col.cu", "conv1_umma.cu", "conv1_bwd_fused.cu", "conv1_dgrad.cu", "gradcam.cu", "lrp.cu", "ig.cu", "bn_act_pool.cu", "fusion_ops.cu", "attention.cu", "attention_mma.cu", "enc_fused.cu", "eval_ops.cu", "augment.cu", "mnet_ops.cu", "adam.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-DTMF_BUILD", "-Xptxas", "-v"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


HASH_FILE = LIB + ".srchash"


def source_hash():
    """sha256 over every file under csrc/ (sorted by name), include/tmf.h and the nvcc flags: the identity of a build."""
    import hashlib
    h = hashlib.sha256()
    deps = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC)) + [os.path.join(HERE, "..", "include", "tmf.h")]
    for d in deps:
        h.update(os.path.basename(d).encode())
        with open(d, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS + SOURCES).encode())
    return h.hexdigest()


def recorded_hash():
    """The source hash the in-tree .so was built from ('' if unknown)."""
    try:
        with open(HASH_FILE) as f:
            return f.read().strip()
    except OSError:
        return ""


def needs_build():
    """Content-based (not mtime-based): a .so that does not match the sources is never used silently."""
    return not os.path.exists(LIB) or recorded_hash() != source_hash()


def build(force=False, verbose=False):
    """Compile every .cu under csrc/ to objects and link the shared library."""
    if not force and not needs_build():
        return LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for s in SOURCES:
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, s), "-o", obj]
        procs.append((s, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs, log = [], []
    for s, obj, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {s}\n{out}")
        if p.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError(f"nvcc failed on {s}")
        objs.append(obj)
    with open(os.path.join(objdir, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    cmd = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-lcudart", "-lcuda"]
    subprocess.run(cmd, check=True)
    with open(HASH_FILE, "w") as f:
        f.write(source_hash() + "\n")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
