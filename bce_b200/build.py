"""Build recipes for the native pieces of bce_b200 (all in-tree, nothing JIT-cached).

    libbce_gpu.so    CUDA kernels + C ABI (include/bce_gpu.h), sm_100a only
    libbce_host.so   host side of the compressor: range coders, archive writer/reader (C++)
    bce              command line tool with the reference's interface (bce -c / -d / -ds / -s)
    libbce_synth.so  synthetic input generators (SURVEY.md 8d)

`python -m bce_b200.build` builds whatever is out of date.  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
HOST = CSRC / "host"

GPU_SOURCES = ["api.cu", "radix_sort.cu", "suffix_sort.cu", "wavelet.cu", "cse.cu", "unbwt.cu", "many.cu", "unbwt_many.cu", "code_many.cu", "decode_many.cu"]
GPU_HEADERS = ["common.cuh", "ctx.h", "cse_rule.cuh", "cse_wide.cuh", "cse_slots.cuh", "cse_mid.cuh", "local_sort.cuh", "../../include/bce_gpu.h"]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC", "-cudart", "static",
]
# built here, run on the GPU box's host CPU: no -march=native
HOST_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-march=x86-64-v2", "-mpopcnt", "-Wall", "-Wextra", "-pthread"]

LIB_GPU = PKG / "libbce_gpu.so"
LIB_HOST = PKG / "libbce_host.so"
LIB_SYNTH = PKG / "libbce_synth.so"
BIN_BCE = PKG / "bce"


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built")


def _cxx() -> str:
    for cand in ("/usr/bin/g++", shutil.which("g++")):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("g++ not found")


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).exists() and Path(d).stat().st_mtime > t for d in deps)


def _run(cmd, cwd=None):
    r = subprocess.run([str(c) for c in cmd], cwd=cwd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("build failed: %s\n%s\n%s" % (" ".join(map(str, cmd)), r.stdout, r.stderr))
    return r


def _flavor() -> str:
    """`BCE_GPU_EXPERIMENTS=1 python -m bce_b200.build` compiles the development switches in (environment knobs
    of the level loop for A/B timing, its cycle stamps).  The default build -- the
    one __graft_entry__.build() and the tests use -- has none of them."""
    return "experiments" if os.environ.get("BCE_GPU_EXPERIMENTS", "") not in ("", "0") else "default"


def build_gpu(force: bool = False, verbose: bool = False) -> Path:
    deps = [CSRC / s for s in GPU_SOURCES] + [CSRC / h for h in GPU_HEADERS]
    stamp = PKG / "_build" / "gpu_flavor.txt"
    flavor = _flavor()
    if force or _stale(LIB_GPU, deps) or not stamp.exists() or stamp.read_text().strip() != flavor:
        cmd = [_nvcc(), *NVCC_FLAGS, "-ccbin", _cxx(), "-shared", "-o", LIB_GPU, *GPU_SOURCES]
        if flavor == "experiments":
            cmd[1:1] = ["-DBCE_GPU_EXPERIMENTS"]
        if verbose:
            cmd[1:1] = ["-Xptxas", "-v"]
        r = _run(cmd, cwd=CSRC)
        stamp.parent.mkdir(exist_ok=True)
        stamp.write_text(flavor + "\n")
        if verbose:
            print(r.stderr)
    return LIB_GPU


def build_synth(force: bool = False) -> Path:
    src = HOST / "synth.c"
    if force or _stale(LIB_SYNTH, [src]):
        _run(["/usr/bin/gcc", "-O2", "-fPIC", "-march=x86-64-v2", "-shared", "-o", LIB_SYNTH, src])
    return LIB_SYNTH


def build_host(force: bool = False) -> Path:
    srcs = [HOST / "coders.cpp", HOST / "archive.cpp", HOST / "decode.cpp", HOST / "host_api.cpp"]
    hdrs = [HOST / "coders.hpp", HOST / "archive.hpp", HOST / "decode.hpp", ROOT / "include" / "bce_gpu.h", ROOT / "include" / "bce_host.h"]
    if not all(s.exists() for s in srcs):
        return LIB_HOST
    if force or _stale(LIB_HOST, srcs + hdrs):
        _run([_cxx(), *HOST_FLAGS, "-shared", "-o", LIB_HOST, *srcs, "-I", ROOT / "include",
              "-L", PKG, "-lbce_gpu", "-Wl,-rpath,$ORIGIN"])
    main = HOST / "bce_main.cpp"
    if main.exists() and (force or _stale(BIN_BCE, srcs + hdrs + [main, LIB_GPU])):
        _run([_cxx(), *HOST_FLAGS, "-DBCE_HAVE_DECODER", "-o", BIN_BCE, main, *srcs, "-I", ROOT / "include",
              "-L", PKG, "-lbce_gpu", "-Wl,-rpath,$ORIGIN", "-ldl"])
    return LIB_HOST


def build_all(force: bool = False, verbose: bool = False) -> None:
    build_gpu(force, verbose)
    build_synth(force)
    build_host(force)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print("built:", *(p.name for p in (LIB_GPU, LIB_HOST, LIB_SYNTH, BIN_BCE) if p.exists()))
