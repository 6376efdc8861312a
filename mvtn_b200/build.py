"""Builds libmvr_b200.so (the sm_100a kernels + C ABI) in-tree with plain nvcc.

No torch headers are involved: the ABI is raw pointers + a stream, loaded with ctypes.
-fmad=false is part of the parity contract (see csrc/mvr_common.cuh): fragment-deciding
arithmetic must not be contracted into FMAs; tolerance-level code uses fmaf() explicitly.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmvr_b200.so")
# source -> allow FMA contraction?  The forward units decide fragments and keep the written IEEE operation order
# (-fmad=false); mvr_mesh_bwd.cu only produces tolerance-compared gradients from inputs that are exact by construction
# (intrinsics in mvr_common.cuh / mvr_mesh.cuh) and is compiled with contraction.
SOURCES = {"mvr_util.cu": False, "mvr_camera.cu": False, "mvr_mesh.cu": False, "mvr_mesh_clip.cu": False, "mvr_mesh_soft.cu": False, "mvr_mesh_bwd.cu": True,
           "mvr_points.cu": False, "mvr_augment.cu": False}
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fopenmp",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "mvr_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    base = [_nvcc()] + NVCC_FLAGS
    if os.path.exists("/usr/bin/g++"):
        base += ["-ccbin", "/usr/bin/g++"]
    if verbose:
        base += ["-Xptxas", "-v"]
    objdir = os.path.join(HERE, "_obj")
    os.makedirs(objdir, exist_ok=True)
    from concurrent.futures import ThreadPoolExecutor

    def compile_one(item):
        src, fmad = item
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = base + ["-fmad=true" if fmad else "-fmad=false", "-c", os.path.join(CSRC, src), "-o", obj]
        return obj, subprocess.run(cmd, capture_output=True, text=True)

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(compile_one, SOURCES.items()))
    objs = []
    for obj, res in results:
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("nvcc failed building libmvr_b200.so")
        if verbose:
            sys.stderr.write(res.stderr)
        objs.append(obj)
    res = subprocess.run(base + ["-shared", "-o", LIB] + objs, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed linking libmvr_b200.so")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
