"""Builds libfdt_cuda.so (sm_100a) in-tree with nvcc.  No JIT, no torch extension machinery: the
library is a plain C-ABI shared object (include/fdt_api.h) that Dart (dart:ffi), C++ and Python
(ctypes) bind alike."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libfdt_cuda.so"
OBJ = PKG / "build"

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-std=c++17", "-O3", "-lineinfo", "-Xcompiler", "-fPIC,-fvisibility=hidden", "-I", str(PKG.parent / "include")]
COMMON += os.environ.get("FDT_NVCC_FLAGS", "").split()   # tuning experiments, e.g. -DFDT_MINB=2
SOURCES = {
    "tflite_model.cpp": [],
    "plan.cpp": [],
    "jpeg_host.cpp": [],
    "engine.cu": [],
    "fdt_api.cu": [],
    "kernels_naive.cu": [],
    "kernels_tiled.cu": [],
    "kernels_ws.cu": [],
    "kernels_tail.cu": [],
    "kernels_ts.cu": [],
    "kernels_fc.cu": [],
    "kernels_jpeg.cu": [],
    "kernels_pre.cu": [],
    # f64 geometry must be evaluated operation by operation (no fused multiply-add contraction)
    "kernels_post.cu": ["-fmad=false"],
    "kernels_warp422.cu": ["-fmad=false"],
    "kernels_warp16.cu": ["-fmad=false"],
}


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _stamp() -> str:
    h = hashlib.sha256()
    for p in sorted(list(CSRC.glob("*")) + [PKG.parent / "include" / "fdt_api.h", Path(__file__)]):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    h.update(os.environ.get("FDT_NVCC_FLAGS", "").encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> Path:
    stamp_file = OBJ / "stamp"
    stamp = _stamp()
    if not force and LIB.exists() and stamp_file.exists() and stamp_file.read_text() == stamp:
        return LIB
    OBJ.mkdir(exist_ok=True)
    nvcc = _nvcc()
    objs = []
    procs = []
    for src, extra in SOURCES.items():
        obj = OBJ / (src + ".o")
        cmd = [nvcc, *ARCH, *COMMON, *extra, "-x", "cu", "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(str(obj))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed on %s" % src)
    cmd = [nvcc, *ARCH, "-shared", "-o", str(LIB), *objs, "-Xlinker", "--no-undefined"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    stamp_file.write_text(stamp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
