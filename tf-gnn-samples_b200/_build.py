"""Build librgnn.so (the C-ABI CUDA library) in-tree for sm_100a.

`python -m tf_gnn_samples_b200._build` or `__graft_entry__.build()`.  nvcc cross-compiles without a
GPU.  The library and its source-digest stamp are build products (git-ignored); the digest hashes paths relative to
the repository root, so a built tree stays current when it is copied or moved.
"""
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_DIR = os.path.join(PKG_DIR, "lib")
LIB_PATH = os.environ.get("RGNN_LIB_PATH") or os.path.join(LIB_DIR, "librgnn.so")   # RGNN_LIB_PATH: measurement variants (build_variant)
STAMP = os.path.join(LIB_DIR, "librgnn.stamp")
SOURCES = ["gemm_tcgen05.cu", "gemm_tn_tcgen05.cu", "plan.cu", "halo.cu", "seg_kernels.cu", "layers.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def _source_digest():
    h = hashlib.sha256()
    root = os.path.dirname(PKG_DIR)
    inc = os.path.join(root, "include", "rgnn.h")
    files = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    for path in files + [inc]:
        with open(path, "rb") as f:
            h.update(os.path.relpath(path, root).encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_current():
    if not (os.path.exists(LIB_PATH) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as f:
        return f.read().strip() == _source_digest()


def build_variant(name: str, extra_flags):
    """A second library lib/librgnn_<name>.so compiled with extra nvcc flags (e.g. -DRGNN_GEMM_TRACE for tools/gemm_trace.py).
    Measurement tooling only: the package always loads lib/librgnn.so unless a tool points _build.LIB_PATH elsewhere."""
    nvcc = _nvcc()
    if nvcc is None:
        raise RuntimeError("nvcc not found")
    obj_dir = os.path.join(LIB_DIR, "obj_" + name)
    os.makedirs(obj_dir, exist_ok=True)
    out = os.path.join(LIB_DIR, "librgnn_%s.so" % name)
    objs = []
    for src in [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]:
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        res = subprocess.run([nvcc] + NVCC_FLAGS + list(extra_flags) + ["-c", os.path.join(CSRC, src), "-o", obj], capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, res.stdout, res.stderr))
        objs.append(obj)
    res = subprocess.run([nvcc, "-shared", "-o", out] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"],
                         capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (res.stdout, res.stderr))
    return out


def build(force=False, verbose=False):
    """Compile every .cu under csrc/ and link lib/librgnn.so.  Returns the library path."""
    if not force and is_current():
        return LIB_PATH
    nvcc = _nvcc()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build librgnn.so (and no prebuilt, current library in %s)" % LIB_DIR)
    os.makedirs(LIB_DIR, exist_ok=True)
    obj_dir = os.path.join(LIB_DIR, "obj")
    os.makedirs(obj_dir, exist_ok=True)
    sources = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]

    def compile_one(src):
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, res.stdout, res.stderr))
        if verbose and (res.stdout or res.stderr):
            print(res.stdout, res.stderr, file=sys.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(len(sources), os.cpu_count() or 4)) as ex:
        objs = list(ex.map(compile_one, sources))
    cmd = [nvcc, "-shared", "-o", LIB_PATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (res.stdout, res.stderr))
    with open(STAMP, "w") as f:
        f.write(_source_digest())
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
