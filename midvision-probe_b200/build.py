"""Build libmvmatch.so (the C-ABI CUDA library) in-tree with plain nvcc for sm_100a.

    python midvision-probe_b200/build.py [--force]

The shared object lands in midvision-probe_b200/lib/ so that it travels with the source tree
(it is git-ignored).  No torch headers are involved: the library's boundary is include/mvmatch.h.
"""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libmvmatch.so")
SOURCES = ["api.cu", "k1_sample.cu", "k1_grid.cu", "k2_sim.cu", "lr_gram.cu", "k3_score.cu", "knn_rerank.cu", "spair_batch.cu", "spair_tiled.cu", "stage.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC or put /usr/local/cuda/bin on PATH)")


def _stamp():
    h = hashlib.sha256()
    files = sorted(os.listdir(CSRC)) + [os.path.join("..", "..", "include", "mvmatch.h")]
    for f in files:
        p = os.path.join(CSRC, f)
        if os.path.isfile(p):
            h.update(f.encode())
            h.update(open(p, "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build_lib(force=False, verbose=False):
    """Compile csrc/*.cu into lib/libmvmatch.so unless an up-to-date build exists. Returns the path."""
    os.makedirs(LIBDIR, exist_ok=True)
    stamp_file = os.path.join(LIBDIR, "libmvmatch.stamp")
    stamp = _stamp()
    if not force and os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
    link = [nvcc, "-shared", "-o", LIB] + objs + ["-lpthread"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("linking libmvmatch.so failed")
    open(stamp_file, "w").write(stamp)
    return LIB


if __name__ == "__main__":
    print(build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv))
