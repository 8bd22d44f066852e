"""Build libsbr_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python sequence-based-recommendations_b200/build.py [--force] [-v] [--timeline]

--timeline compiles the clock64 phase stamps into the tcgen05 scan kernels (profiling builds only; read them with
SBR_TC_TIMELINE=1).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libsbr_b200.so")
SOURCES = ["model.cu", "gather_scatter.cu", "rnn_cluster.cu", "rnn_tc.cu", "wgrad_tc.cu", "tc_gemm.cu", "tc_scan.cu", "gemm.cu", "loss.cu", "optim.cu", "cluster.cu"]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--use_fast_math=false",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "sbr_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, timeline=False):
    if not force and not timeline and not needs_build():
        return OUT
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")]
    if timeline:
        flags.append("-DSBR_TC_TIMELINE_BUILD")
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", "_tl.o" if timeline else ".o"))
        objs.append(obj)
        cmd = [_nvcc()] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("== %s ==\n%s\n" % (src, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    out = OUT.replace(".so", "_timeline.so") if timeline else OUT
    link = [_nvcc(), "-shared", "-o", out] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl"]
    subprocess.check_call(link)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, timeline="--timeline" in sys.argv))
