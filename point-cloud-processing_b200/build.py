"""Build recipe of libpcpx.so (CUDA C++ for sm_100a, explicit nvcc, in-tree output).

    python point-cloud-processing_b200/build.py [--force]

nvcc cross-compiles without a GPU; the resulting lib/libpcpx.so is git-ignored but travels to
the GPU box with the repository snapshot.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(HERE, "build")
LIB = os.path.join(LIBDIR, "libpcpx.so")
UNITS = ["index.cu", "query.cu", "query_normals.cu", "query_mean.cu", "api.cu", "smoothing.cu",
         "orient.cu", "shard.cu", "query_box.cu", "cluster.cu", "icp.cu"]

NVCC_FLAGS = [
    "-std=c++17", "-O3",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-O2",
    "-I", os.path.join(ROOT, "include"), "-I", CSRC,
]


def _sources():
    out = [os.path.join(ROOT, "include", "pcpx.h")]
    for f in os.listdir(CSRC):
        out.append(os.path.join(CSRC, f))
    return out


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(s) > t for s in _sources())


def build(force=False, verbose=False, defines=(), out=None):
    """defines / out: build an experimental variant (e.g. -DPCPX_MIN_BLOCKS=8) next to the
    product library; the product is always built with no extra defines."""
    global LIB, OBJDIR
    if out is not None:
        LIB = os.path.join(LIBDIR, out)
        OBJDIR = os.path.join(HERE, "build", out.replace(".so", ""))
        force = True
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = os.environ.get("NVCC", "nvcc")

    headers = [os.path.join(ROOT, "include", "pcpx.h")] + [
        os.path.join(CSRC, f) for f in os.listdir(CSRC) if not f.endswith(".cu")]
    newest_header = max(os.path.getmtime(h) for h in headers)

    def compile_one(unit):
        obj = os.path.join(OBJDIR, unit.replace(".cu", ".o"))
        src = os.path.join(CSRC, unit)
        # an object newer than its source and every header is kept (query.cu takes minutes)
        if (not defines and not verbose and os.path.exists(obj)
                and os.path.getmtime(obj) > max(newest_header, os.path.getmtime(src))):
            return obj
        cmd = [nvcc] + NVCC_FLAGS + list(defines) + (["-Xptxas", "-v"] if verbose else []) + [
            "-c", os.path.join(CSRC, unit), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (unit, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
        objs = list(ex.map(compile_one, UNITS))
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB


if __name__ == "__main__":
    defs = [a for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a.split("=", 1)[1] for a in sys.argv[1:] if a.startswith("--out=")]
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, defines=defs,
                out=outs[0] if outs else None))
