"""Build libfbkst_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python fbk-fairseq-st_b200/build.py [--force] [--verbose]

nvcc cross-compiles without a GPU.  The built .so is git-ignored but travels to the GPU box
with the gpurun snapshot.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "fbkst_b200", "libfbkst_b200.so")
OBJ_DIR = os.path.join(HERE, "build")
SOURCES = ["host_common.cu", "elementwise.cu", "ctc.cu", "ctc_criterion.cu", "augment.cu", "cross_attention.cu", "self_attention.cu", "gemm_tcgen05.cu", "gemm2_tcgen05.cu", "conv2_tcgen05.cu", "conv1_tcgen05.cu",
           "attention_tcgen05.cu", "attention_wide.cu", "attention_train.cu", "train_elementwise.cu", "conv_train.cu", "tf32x3.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
# extra defines for A/B experiments on the GPU box (e.g. FBKST_NVCC_FLAGS="-DFBKST_ATTN_TRACE");
# part of the object digest, so switching them rebuilds
FLAGS += os.environ.get("FBKST_NVCC_FLAGS", "").split()


def _digest(path):
    h = hashlib.sha1()
    for name in sorted(os.listdir(CSRC)) + ["../../include/fbkst_b200.h"]:
        p = os.path.join(CSRC, name)
        if name.endswith((".cuh", ".h")) or p == path:
            with open(p, "rb") as f:
                h.update(f.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    os.makedirs(OBJ_DIR, exist_ok=True)
    objs, rebuilt = [], False
    procs = []
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        stamp = obj + ".sha1"
        dig = _digest(path)
        objs.append(obj)
        if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dig:
            continue
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
        procs.append((src, stamp, dig, subprocess.Popen(cmd, stdout=subprocess.PIPE,
                                                        stderr=subprocess.STDOUT, text=True)))
    for src, stamp, dig, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError("nvcc failed on %s" % src)
        if verbose:
            print(out)
        with open(stamp, "w") as f:
            f.write(dig)
        rebuilt = True
    if rebuilt or not os.path.exists(OUT):
        cmd = [NVCC, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
        subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
