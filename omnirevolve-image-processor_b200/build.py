"""Build libomni_b200.so (hand-written sm_100a CUDA + the C ABI of include/omni_b200.h) in-tree.

    python omnirevolve-image-processor_b200/build.py [--force] [--verbose]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libomni_b200.so")
SOURCES = ["capi.cu", "generic_kernels.cu", "fast_kernels.cu", "edges3.cu", "label_pipe.cu", "resize_tma.cu", "kmeans.cu", "trace.cu", "morph_ellipse.cu", "png_encode.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--fmad=false",                      # float paths must round every product and sum (SURVEY A.1, A.4)
              "-Xcompiler", "-fPIC,-fvisibility=default"]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static", "-Xcompiler", "-fPIC"]
OBJ_DIR = os.path.join(HERE, "build")


def _deps():
    d = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    d.append(os.path.join(os.path.dirname(HERE), "include", "omni_b200.h"))
    return d


def _compile_all(defines=(), verbose=False, obj_dir=OBJ_DIR, only_stale=True):
    """One nvcc per translation unit, in parallel; returns the object files."""
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(obj_dir, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    hdrs = [p for p in _deps() if not p.endswith(".cu")]
    hdr_t = max(os.path.getmtime(p) for p in hdrs)

    def one(src):
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        path = os.path.join(CSRC, src)
        if only_stale and os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(path), hdr_t):
            return obj, 0, ""
        cmd = [nvcc] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, path]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        return obj, r.returncode, r.stdout

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as pool:
        res = list(pool.map(one, SOURCES))
    log = "".join(o for _, _, o in res)
    if verbose or any(rc for _, rc, _ in res):
        print(log)
    if any(rc for _, rc, _ in res):
        raise RuntimeError("nvcc failed building libomni_b200.so")
    return [o for o, _, _ in res]


def _link(objs, out):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    r = subprocess.run([nvcc] + LINK_FLAGS + ["-o", out] + objs, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        print(r.stdout)
        raise RuntimeError("linking libomni_b200.so failed")


def build(force: bool = False, verbose: bool = False, out: str | None = None, defines=()) -> str:
    """out / defines: build an experimental variant (e.g. -DE3V_MINBLOCKS=4) next to the product library."""
    os.makedirs(LIB_DIR, exist_ok=True)
    if out is not None:
        tag = "v_" + "_".join(d.replace("=", "-") for d in defines) if defines else "v_plain"
        objs = _compile_all(defines, verbose, os.path.join(OBJ_DIR, tag), only_stale=False)
        _link(objs, out)
        return out
    if not force and os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(p) for p in _deps()):
        return LIB
    objs = _compile_all((), verbose, OBJ_DIR, only_stale=not force)
    _link(objs, LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
