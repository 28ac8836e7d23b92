"""Builds libsfcvit.so (all CUDA kernels + the C ABI) for sm_100a with nvcc, in-tree.

    python space-filling-curves-for-vision-transformers_b200/build.py [--force] [--verbose]

Output: space-filling-curves-for-vision-transformers_b200/lib/libsfcvit.so (git-ignored, travels with gpurun).
"""
import concurrent.futures as cf
import glob
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
_TL = bool(os.environ.get("SFC_ATTN_TIMELINE"))               # debug build with clock64 stamps (tools/attn_timeline*.py)
OBJ_DIR = os.path.join(HERE, "build_tl" if _TL else "build")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libsfcvit_tl.so" if _TL else "libsfcvit.so")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
    "-I", os.path.join(ROOT, "include"), "-I", CSRC,
] + (["-DSFC_ATTN_TIMELINE"] if os.environ.get("SFC_ATTN_TIMELINE") else [])   # debug stamps for tools/attn_timeline.py


def _sha(paths, extra=""):
    h = hashlib.sha1(extra.encode())
    for p in sorted(paths):
        h.update(os.path.basename(p).encode())
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _headers():
    return glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.h")) + \
        glob.glob(os.path.join(ROOT, "include", "*.h"))


def _stamp(path):
    try:
        with open(path) as f:
            return f.read().strip()
    except OSError:
        return None


def _compile(src, obj, verbose):
    cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
    return r.stderr


def _plan(force=False):
    """-> (compile jobs, every object, objects of deleted sources). Reads only, so it works in a read-only tree."""
    # staleness by CONTENT hash (source + every header + flags), not mtime: a copied or freshly checked-out tree has new
    # timestamps, and a spurious rebuild would cost minutes
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cu")))
    hdrs = _headers()
    flags = " ".join(FLAGS)
    jobs, objs = [], []
    for s in srcs:
        o = os.path.join(OBJ_DIR, os.path.basename(s)[:-3] + ".o")
        objs.append(o)
        want = _sha([s] + hdrs, flags)
        if force or not os.path.exists(o) or _stamp(o + ".sha") != want:
            jobs.append((s, o, want))
    stale = [o for o in glob.glob(os.path.join(OBJ_DIR, "*.o")) if o not in objs]      # objects of deleted sources
    return jobs, objs, stale


def up_to_date():
    """True when build() would compile and link nothing."""
    jobs, _objs, stale = _plan()
    return not jobs and not stale and os.path.exists(LIB)


def build(force=False, verbose=False):
    os.makedirs(OBJ_DIR, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    jobs, objs, stale = _plan(force)
    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            futs = {ex.submit(_compile, s, o, verbose): (o, want) for s, o, want in jobs}
            for f in cf.as_completed(futs):
                log = f.result()
                o, want = futs[f]
                with open(o + ".sha", "w") as fh:
                    fh.write(want)
                if verbose:
                    sys.stderr.write(log)
    for o in stale:
        os.remove(o)
    if jobs or stale or not os.path.exists(LIB):
        tmp = f"{LIB}.{os.getpid()}.tmp"                     # link aside, then rename: a concurrent loader never sees a partial file
        cmd = [NVCC, "-shared", "-o", tmp] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
        os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
