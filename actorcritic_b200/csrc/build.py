"""Build libacx.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "libacx.so")
SOURCES = ["lib.cu", "preprocess.cu", "returns.cu", "gemm.cu", "conv.cu", "layers.cu", "kfac.cu", "kfac_inv.cu", "peer.cu", "learner_core.cu", "learner.cu", "mlp.cu"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--expt-relaxed-constexpr",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-Xcompiler", "-Wno-unused-function",
         "-fmad=true", "-shared", "-lcudart_static", "-lpthread", "-ldl", "-lrt"]


def build(verbose=False, force=False):
    srcs = [os.path.join(HERE, s) for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    deps = srcs + [os.path.join(HERE, "common.cuh"), os.path.join(os.path.dirname(os.path.dirname(HERE)), "include", "acx.h")]
    deps += [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith(".cuh")]
    if not force and os.path.exists(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(d) for d in deps):
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    build_dir = os.path.join(HERE, "build")
    os.makedirs(build_dir, exist_ok=True)
    cflags = [f for f in FLAGS if f not in ("-shared", "-lcudart_static", "-lpthread", "-ldl", "-lrt")]
    for s in srcs:
        o = os.path.join(build_dir, os.path.basename(s) + ".o")
        objs.append(o)
        if (not force and os.path.exists(o)
                and all(os.path.getmtime(o) >= os.path.getmtime(d) for d in [s] + deps[len(srcs):])):
            continue
        cmd = [nvcc] + cflags + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for cmd, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            print(" ".join(cmd))
            print(out)
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", OUT] + objs + ["-lcudart_static", "-lpthread", "-ldl", "-lrt"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
