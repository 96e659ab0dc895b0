"""Deterministic synthetic inputs (SURVEY.md 8d); thin ctypes wrapper over csrc/host/synth.c."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

KINDS = {"markov2-text": 0, "enwik-shaped": 1, "mixed-binary": 2, "uniform": 3}
_LIB = Path(__file__).resolve().parent / "libbce_synth.so"
_lib = None


def _load():
    global _lib
    if _lib is None:
        if not _LIB.exists():
            from . import build
            build.build_synth()
        lib = C.CDLL(str(_LIB))
        lib.bce_synth.argtypes = [C.c_int, C.c_void_p, C.c_size_t, C.c_uint64]
        _lib = lib          # published only once its signatures are set: another thread must not call it before
    return _lib


def generate(kind: str, n: int, seed: int) -> np.ndarray:
    out = np.empty(n, dtype=np.uint8)
    rc = _load().bce_synth(KINDS[kind], out.ctypes.data, n, seed)
    if rc != 0:
        raise RuntimeError(f"bce_synth({kind}) failed: {rc}")
    return out


# the configs BASELINE.json names: (generator, bytes, seed)
CONFIGS = {
    "markov2-1MB": ("markov2-text", 10**6, 1),
    "enwik-100MB": ("enwik-shaped", 10**8, 2),
    "enwik-1GB": ("enwik-shaped", 10**9, 3),
    "mixed-256MB": ("mixed-binary", 268435456, 4),
    "batch-128MB": ("enwik-shaped", 134217728, 100),
}
