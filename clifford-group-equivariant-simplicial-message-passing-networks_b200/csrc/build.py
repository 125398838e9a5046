#!/usr/bin/env python
"""Build libcsmpn_b200.so (sm_100a) in-tree with nvcc.  Used by __graft_entry__.build()."""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["api.cu", "elementwise.cu", "linear.cu", "graph.cu", "block_fused.cu", "lift.cu", "tc_block_fwd.cu", "tc_block_bwd.cu"]
LIB = os.path.join(HERE, "libcsmpn_b200.so")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v",
]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _digest(paths):
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode() + b"\0" + f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def generate_tables():
    """algebra_gen.cuh (unrolled sign/index tables of Cl(2,0), Cl(3,0), Cl(5,0)) is GENERATED from algebra/metric.py by
    gen_algebra.py whenever it is missing or older than its generator; it is not tracked in git."""
    out = os.path.join(HERE, "algebra_gen.cuh")
    srcs = [os.path.join(HERE, "gen_algebra.py"), os.path.join(HERE, "..", "algebra", "metric.py")]
    if os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in srcs):
        return out
    r = subprocess.run([sys.executable, os.path.join(HERE, "gen_algebra.py")], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"gen_algebra.py failed:\n{r.stdout}\n{r.stderr}")
    return out


def build(force=False, verbose=False):
    generate_tables()
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    deps = [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith((".cu", ".cuh", ".h"))]
    deps.append(os.path.join(HERE, "..", "..", "include", "csmpn_b200.h"))
    stamp = os.path.join(HERE, "build", "stamp.txt")
    dig = _digest(deps)
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == dig:
        return LIB
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(HERE, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = os.path.join(HERE, "build", src.replace(".cu", ".ptxas.log"))
        with open(log, "w") as f:
            f.write(r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(f"[build] {src} ok", file=sys.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
