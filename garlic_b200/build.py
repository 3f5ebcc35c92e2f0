"""Build libgarlic_b200.so (hand-written sm_100a kernels + the C ABI) in-tree with nvcc."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libgarlic_b200.so")
SOURCES = ["kernels.cu", "squeeze.cu", "wlod.cu", "kde.cu", "ingest.cu", "bed.cu", "vcf.cu", "bcf.cu", "xchg.cu", "capi.cu"]
HEADERS = ["common.cuh", "walk.cuh", "bound.cuh", "vcf_gt.cuh", "bcf_gt.cuh", "bed_select.cuh", "segments.h", "kernels.h", "wlod.h", os.path.join("..", "..", "include", "garlic_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-fmad=false",          # the reference is built without FMA; keep mul/add roundings separate
              "-Xcompiler", "-fPIC", "--shared"]


OBJ_DIR = os.path.join(HERE, "build")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def needs_build():
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return _stale(OUT, deps)


def build(force=False, verbose=False):
    """One object per translation unit (compiled in parallel, only the stale ones), then one link."""
    if not force and not needs_build():
        return OUT
    from concurrent.futures import ThreadPoolExecutor
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJ_DIR, exist_ok=True)
    common = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    flags = [f for f in NVCC_FLAGS if f != "--shared"]

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, os.path.splitext(src)[0] + ".o")
        path = os.path.join(CSRC, src)
        if not force and not _stale(obj, [path] + common):
            return obj, 0, ""
        r = subprocess.run([nvcc] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj],
                           capture_output=True, text=True)
        return obj, r.returncode, r.stdout + r.stderr

    with ThreadPoolExecutor(len(SOURCES)) as ex:
        res = list(ex.map(compile_one, SOURCES))
    for obj, rc, log in res:
        if rc != 0:
            sys.stderr.write(log)
            raise RuntimeError("nvcc failed compiling " + obj)
        if verbose:
            sys.stderr.write(log)
    r = subprocess.run([nvcc, "--shared", "-Xcompiler", "-fPIC"] + [o for o, _, _ in res] + ["-lnccl", "-o", OUT],
                       capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed linking libgarlic_b200.so")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
