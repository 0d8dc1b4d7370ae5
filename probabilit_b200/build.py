"""Build libprobabilit_b200.so in-tree with nvcc for sm_100a (B200).

    python -m probabilit_b200.build [--force] [--verbose]

One object per .cu (compiled in parallel), linked into probabilit_b200/libprobabilit_b200.so.
nvcc cross-compiles without a GPU, so this also runs in the CPU-only build container.
"""
import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "csrc", "_obj")
LIB = os.path.join(HERE, "libprobabilit_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
]


# Per-source flags.  graph.cu (the inverse CDFs and the arithmetic nodes of the modeling graph) is compiled
# without FMA contraction: the reference's values come from NumPy ufuncs and SciPy's C special functions,
# which round every product before the sum; a contracted a*b+c differs in the last place, and the Halley
# iterations / series of gammaincinv amplify that to several ulp.
# stats.cu reproduces NumPy's sums and quantile interpolation bit for bit, so it is compiled the same way.
PER_SOURCE_FLAGS = {"graph.cu": ["-fmad=false"], "stats.cu": ["-fmad=false"]}


def nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found")
    return exe


def sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def newest_input_mtime():
    paths = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    paths.append(os.path.join(os.path.dirname(HERE), "include", "probabilit_b200.h"))
    paths.append(os.path.abspath(__file__))
    return max(os.path.getmtime(p) for p in paths)


def up_to_date():
    return os.path.exists(LIB) and os.path.getmtime(LIB) >= newest_input_mtime()


def build(force=False, verbose=False):
    if not force and up_to_date():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    exe = nvcc()
    extra = ["-Xptxas", "-v"] if verbose else []
    extra += os.environ.get("PBL_EXTRA_NVCC_FLAGS", "").split()  # developer instrumentation (e.g. -DPBL_PASS_PROFILE)

    def compile_one(src):
        obj = os.path.join(OBJ, src[:-3] + ".o")
        cmd = [exe, *NVCC_FLAGS, *PER_SOURCE_FLAGS.get(src, []), *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with cf.ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, sources()))
    cmd = [exe, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
