"""Builds chessrl_b200/libchessrl_b200.so (sm_100a only) with nvcc.  `python -m chessrl_b200.build`."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libchessrl_b200.so")
SOURCES = ["api.cu", "kernels_rules.cu", "kernels_encode.cu", "kernels_tree.cu", "net.cu", "kernels_ab.cu"]
HEADERS = ["engine.cuh", "chess_core.cuh", "tree_core.cuh", "hash_eval.cuh", "ab_search.cuh", "search_targets.cuh", os.path.join("..", "..", "include", "chessrl_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
         "--fmad=true", "-Xptxas", "-v"]


def stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not stale():
        return OUT
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [NVCC] + FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        log.append("== %s ==\n%s" % (src, out))
        failed = failed or p.returncode != 0
    with open(os.path.join(HERE, "build", "nvcc.log"), "w") as f:
        f.write("\n".join(log))
    if failed or verbose:
        sys.stderr.write("\n".join(log))
    if failed:
        raise RuntimeError("nvcc failed; see chessrl_b200/build/nvcc.log")
    cmd = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT] + objs + ["-lcudart"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
