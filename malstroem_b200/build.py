"""Build libmalstroem_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
import glob
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# MS_BUILD_TAG=_x builds a variant (with MS_NVCC_EXTRA flags) into libmalstroem_b200_x.so; load it with MS_LIB=<path>
TAG = os.environ.get("MS_BUILD_TAG", "")
OBJ = os.path.join(HERE, "csrc", "_obj" + TAG)
LIB = os.path.join(HERE, "libmalstroem_b200%s.so" % TAG)
SOURCES = ["core.cu", "primitives.cu", "fill.cu", "noflats.cu", "flow.cu", "accum.cu", "labels.cu", "pipeline.cu", "synth.cu", "network.cu", "cache.cu", "tiff.cu", "polygon.cu", "flood.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# no --use_fast_math: denormals (ftz=false), exact division and no FMA contraction are part of the contract
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-fmad=false",
         "-Xcompiler", "-fPIC", "-Xptxas", "-v"] + os.environ.get("MS_NVCC_EXTRA", "").split()


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    hdrs = sorted(glob.glob(os.path.join(CSRC, "*.cuh"))) + [os.path.join(HERE, "..", "include", "malstroem_b200.h")]
    jobs = []
    for src in SOURCES:
        sp = os.path.join(CSRC, src)
        op = os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or _stale(op, [sp] + hdrs):
            jobs.append((sp, op))

    def compile_one(job):
        sp, op = job
        r = subprocess.run([NVCC] + FLAGS + ["-c", sp, "-o", op], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                           text=True)
        return sp, r.returncode, r.stdout

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for sp, rc, out in ex.map(compile_one, jobs):
                if verbose or rc != 0:
                    sys.stderr.write(out)
                if rc != 0:
                    raise RuntimeError("nvcc failed on %s" % sp)
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        subprocess.check_call([NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
