"""Build libscrib200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo).

Each .cu is compiled to an object under csrc/_obj/ (only when it or a header changed, all stale ones in parallel), then
linked; `python -m scri_b200.build [-v]` forces a full rebuild."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB = os.path.join(HERE, "libscrib200.so")
SOURCES = ["runtime.cu", "rotate.cu", "synth.cu", "spline_tile.cu", "mix.cu", "analysis.cu", "modes.cu", "product.cu", "codec.cu", "inner.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--fmad=true",
]


def _headers():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".inc"))] + [
        os.path.join(HERE, "..", "include", "scrib200.h")]


def needs_build():
    if not os.path.exists(LIB):
        return True
    mt = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES] + _headers()
    return any(os.path.getmtime(d) > mt for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJ, exist_ok=True)
    hdr_mt = max(os.path.getmtime(h) for h in _headers() if os.path.exists(h))
    jobs = []
    objs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        if not os.path.exists(src):
            continue
        obj = os.path.join(OBJ, s[:-3] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_mt):
            jobs.append([nvcc, "-c", "-o", obj] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + [src])

    def run(cmd):
        return cmd, subprocess.run(cmd, capture_output=True, text=True)

    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 4))) as pool:
        results = list(pool.map(run, jobs))
    for cmd, res in results:
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError(f"nvcc failed on {cmd[-1]}")
        if verbose:
            print(res.stderr)
    res = subprocess.run([nvcc, "-shared", "-o", LIB] + NVCC_FLAGS + objs, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed linking libscrib200.so")
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))
