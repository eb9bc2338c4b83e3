"""Build recipe for lib/libmsacl_b200.so (sm_100a only; nvcc cross-compiles without a GPU).

    python <package dir>/build.py [--force] [--verbose]

The library is built in-tree (`<repo>/lib/`, a short path: the package directory name is ~100 characters long) so
that it travels with the repo snapshot to the GPU box; it is git-ignored (*.so).  Every source is compiled to its
own object (in parallel, re-compiled only when its digest changes) and the objects are linked into one shared
library.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIBDIR = os.path.join(ROOT, "lib")
OBJDIR = os.path.join(LIBDIR, "obj")
LIB = os.path.join(LIBDIR, "libmsacl_b200.so")
STAMP = LIB + ".stamp"
SOURCES = ["env_step.cu", "rollout_fused.cu", "windows.cu", "targets.cu", "tc_selftest.cu", "rollout_tc.cu",
           "mlp_tc.cu", "mlp_bwd.cu", "learner.cu", "certify.cu", "certify_region.cu"]
SOURCES = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith(".cuh")) + [os.path.join(ROOT, "include", "msacl_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false",            # dynamics must round like NumPy scalar math; GEMMs call __fmaf_rn explicitly
    "-Xcompiler", "-fPIC", "-Xcompiler", "-ffp-contract=off",
] + (["-DMSACL_TC_TIMING"] if os.environ.get("MSACL_TC_TIMING") else []) \
  + (["-DMSACL_TC_WATCHDOG"] if os.environ.get("MSACL_TC_WATCHDOG") else [])   # role timers / watchdog: tools/tc_*.py


def _sha(paths, extra=""):
    h = hashlib.sha256()
    for p in paths:
        with open(p, "rb") as fh:
            h.update(fh.read())
    h.update(extra.encode())
    return h.hexdigest()


def _header_paths():
    return [f if os.path.isabs(f) else os.path.join(CSRC, f) for f in HEADERS]


def _digest():
    return _sha([os.path.join(CSRC, s) for s in SOURCES] + _header_paths(), " ".join(NVCC_FLAGS))


def is_current():
    """True when lib/libmsacl_b200.so exists and was built from the sources / flags now in the tree."""
    return os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == _digest()


def _compile_one(nvcc, src, verbose):
    obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
    stamp = obj + ".stamp"
    digest = _sha([os.path.join(CSRC, src)] + _header_paths(), " ".join(NVCC_FLAGS))
    if os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return obj, ""
    cmd = [nvcc, *NVCC_FLAGS, *(["-Xptxas", "-v"] if verbose else []), "-c", os.path.join(CSRC, src), "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    with open(stamp, "w") as fh:
        fh.write(digest)
    return obj, res.stderr


def build(force=False, verbose=False):
    digest = _digest()
    if not force and is_current():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJDIR, exist_ok=True)
    if force:
        for f in os.listdir(OBJDIR):
            os.remove(os.path.join(OBJDIR, f))
    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as ex:
        results = list(ex.map(lambda s: _compile_one(nvcc, s, verbose), SOURCES))
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", *[o for o, _ in results], "-o", LIB]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    with open(STAMP, "w") as fh:
        fh.write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
