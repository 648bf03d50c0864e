"""Build librebvo_b200.so (CUDA, sm_100a only) in-tree with nvcc.  No CPU fallback is built."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librebvo_b200.so")
SOURCES = ["dog.cu", "detect.cu", "tracker.cu", "capi.cu", "capi_track.cu", "pipeline.cu", "hostmath.cu",
           "undistort.cu", "imu_track.cu", "netpack.cu", "logfmt.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# -fmad=false: the reference is built without FMA contraction (x86-64 -O2, no -march); bit parity of the
# float32 scale space and of the per-keyline float64 arithmetic depends on it.
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-fmad=false",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fno-fast-math", "-Xcompiler", "-ffp-contract=off"]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "rebvo_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)

    def cc(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(cc, SOURCES))
    # the soname makes programs linked against this file record "librebvo_b200.so" rather than its absolute build path,
    # so that they find it through their rpath wherever the tree is moved to
    cmd = [NVCC, "-shared", "-Xlinker", "-soname=librebvo_b200.so", "-o", LIB] + objs + ["-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
