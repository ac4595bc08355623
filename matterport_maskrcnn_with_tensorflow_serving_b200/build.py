"""In-tree build of libmrx.so (the C-ABI library declared in include/mrx.h).

nvcc cross-compiles for sm_100a without a GPU; the .so is git-ignored but travels to
the GPU box with the gpurun snapshot.  `python -m matterport_maskrcnn_with_tensorflow_serving_b200.build`
or `__graft_entry__.build()` runs this.  Every .cu is compiled to its own object (in
parallel, rebuilt only when it or a header changed) and the objects are linked into the .so.

Environment (development only): MRX_NVCC_FLAGS = extra nvcc flags (e.g. "-DMRX_DEV"),
MRX_LIB_NAME = another output name (e.g. libmrx_dev.so, picked up by _native via MRX_LIB).
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_DIR = os.path.join(PKG_DIR, "lib")

SOURCES = ["capi.cu", "anchors.cu", "unmold.cu", "expand_team.cu", "expand_bits.cu", "mold.cu",
           "composite.cu", "pack.cu", "rle.cu", "contours.cu", "peer.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "expand.cuh"),
           os.path.join(os.path.dirname(PKG_DIR), "include", "mrx.h")]

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "--cudart", "shared",          # share torch's CUDA runtime instance (device/stream state)
    "-Xcompiler", "-fPIC",
]


def lib_name():
    return os.environ.get("MRX_LIB_NAME", "libmrx.so")


def lib_path():
    return os.path.join(LIB_DIR, lib_name())


LIB_PATH = os.path.join(LIB_DIR, "libmrx.so")


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; libmrx.so cannot be built")
    return exe


def _extra_flags():
    return os.environ.get("MRX_NVCC_FLAGS", "").split()


def _digest(paths, salt):
    h = hashlib.sha256()
    for path in paths:
        with open(path, "rb") as f:
            h.update(f.read())
    h.update(salt.encode())
    return h.hexdigest()


def _fingerprint():
    """Digest of everything the library is built from (sources, headers, flags)."""
    return _digest([os.path.join(CSRC, s) for s in SOURCES] + HEADERS,
                   " ".join(NVCC_FLAGS + _extra_flags()))


def _compile_one(src, obj_dir, verbose):
    path = os.path.join(CSRC, src)
    fp = _digest([path] + HEADERS, " ".join(NVCC_FLAGS + _extra_flags()))
    obj = os.path.join(obj_dir, src[:-3] + ".o")
    stamp = obj + ".stamp"
    if os.path.exists(obj) and os.path.exists(stamp):
        with open(stamp) as f:
            if f.read().strip() == fp:
                return obj, ""
    cmd = [_nvcc()] + NVCC_FLAGS + _extra_flags()
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += ["-c", path, "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src}:\n{res.stdout}{res.stderr}")
    with open(stamp, "w") as f:
        f.write(fp)
    return obj, res.stdout + res.stderr


def build(force=False, verbose=False):
    """Compile csrc/*.cu into lib/libmrx.so (skipped when sources are unchanged)."""
    os.makedirs(LIB_DIR, exist_ok=True)
    out = lib_path()
    stamp_path = out[:-3] + ".stamp"
    fp = _fingerprint()
    if not force and os.path.exists(out) and os.path.exists(stamp_path):
        with open(stamp_path) as f:
            if f.read().strip() == fp:
                return out
    obj_dir = os.path.join(LIB_DIR, "obj_" + lib_name()[:-3])
    if force and os.path.isdir(obj_dir):
        shutil.rmtree(obj_dir)
    os.makedirs(obj_dir, exist_ok=True)
    workers = max(1, min(len(SOURCES), os.cpu_count() or 1))
    with ThreadPoolExecutor(workers) as ex:
        results = list(ex.map(lambda s: _compile_one(s, obj_dir, verbose), SOURCES))
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    cmd = [_nvcc(), "-shared", "--cudart", "shared", "-gencode", "arch=compute_100a,code=sm_100a"]
    cmd += [obj for obj, _ in results]
    cmd += ["-Xlinker", "-rpath=/usr/local/cuda/lib64", "-o", out]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed linking " + out)
    with open(stamp_path, "w") as f:
        f.write(fp)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
