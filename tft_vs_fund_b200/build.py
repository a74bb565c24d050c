"""Build libtvf.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

Each translation unit is compiled to an object file (in parallel, reused while neither the source nor any
header changed) and the objects are linked into tft_vs_fund_b200/libtvf.so."""
import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtvf.so")
OBJ = os.path.join(HERE, "build")
SOURCES = ["tvf_core_kernels.cu", "tvf_large_kernels.cu", "tvf_pose_kernels.cu", "tvf_scene_kernels.cu", "tvf_gh_kernels.cu", "tvf_ba_kernels.cu", "tvf_ba_cov_kernels.cu", "tvf_ransac_kernels.cu", "tvf_api.cu"]
HEADERS = ["tvf_math.cuh", "tvf_pose.cuh", "tvf_warp.cuh", "tvf_async.cuh", "tvf_scene.cuh", "tvf_ba.cuh", "tvf_ransac.cuh", "tvf_kernels.h", os.path.join("..", "..", "include", "tvf.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xptxas=-v", "-Xcompiler", "-fPIC", "-cudart", "shared"]


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(src, defines, obj_dir, force):
    obj = os.path.join(obj_dir, os.path.splitext(src)[0] + ".o")
    deps = [os.path.join(CSRC, src)] + [os.path.join(CSRC, f) for f in HEADERS] + [os.path.abspath(__file__)]
    if not force and os.path.exists(obj) and all(os.path.getmtime(d) <= os.path.getmtime(obj) for d in deps):
        return obj, 0, ""
    cmd = [_nvcc()] + NVCC_FLAGS + list(defines) + ["-I", CSRC, "-c", os.path.join(CSRC, src), "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    return obj, res.returncode, " ".join(cmd) + "\n" + res.stdout + res.stderr


def build(force=False, verbose=False, defines=(), out=None, obj_dir=None):
    """Compile every CUDA source for sm_100a into tft_vs_fund_b200/libtvf.so (or `out`, with extra -D `defines`:
    the compile-time variants tools/build_variants.py times against each other)."""
    lib = out or LIB
    if out is None and not force and not needs_build():
        return LIB
    obj_dir = obj_dir or (OBJ if out is None else os.path.splitext(out)[0] + "_obj")
    os.makedirs(obj_dir, exist_ok=True)
    with ThreadPoolExecutor(len(SOURCES)) as ex:
        results = list(ex.map(lambda s: _compile(s, defines, obj_dir, force), SOURCES))
    log_text = "".join(r[2] for r in results)
    rc = max(r[1] for r in results)
    if rc == 0:
        cmd = [_nvcc(), "-shared", "-cudart", "shared", "-o", lib] + [r[0] for r in results]
        res = subprocess.run(cmd, capture_output=True, text=True)
        log_text += " ".join(cmd) + "\n" + res.stdout + res.stderr
        rc = res.returncode
    log = os.path.join(HERE, "build.log") if out is None else os.path.splitext(out)[0] + ".log"
    with open(log, "w") as f:
        f.write(log_text)
    if verbose or rc != 0:
        print(log_text)
    if rc != 0:
        raise RuntimeError("nvcc failed building %s (see %s)" % (os.path.basename(lib), log))
    return lib


if __name__ == "__main__":
    build(force=True, verbose=True)
