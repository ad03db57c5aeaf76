"""Builds morna_b200/libmorna_b200.so in-tree with nvcc for sm_100a (no JIT cache)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libmorna_b200.so")
SOURCES = ["api.cu", "index_build.cu", "search_exact.cu", "search_single.cu", "search_batched.cu", "search_sparse.cu", "search_range.cu", "search_capped.cu",
           "search_within.cu",
           "query_build.cu",
           "tokenize.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v"] + os.environ.get("MORNA_NVCC_EXTRA", "").split()


def nvcc_path():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "morna_b200.h"))
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    objs = []
    logs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc_path()] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        logs.append(p.stdout)
        if p.returncode != 0:
            sys.stderr.write(p.stdout)
            raise RuntimeError("nvcc failed on " + src)
        objs.append(obj)
    cmd = [nvcc_path(), "-shared", "-o", OUT] + objs + ["-lcudart", "-lpthread"]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if p.returncode != 0:
        sys.stderr.write(p.stdout)
        raise RuntimeError("link failed")
    with open(os.path.join(CSRC, "ptxas.log"), "w") as fh:
        fh.write("\n".join(logs))
    if verbose:
        sys.stdout.write("\n".join(logs))
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
