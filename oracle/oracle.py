"""ctypes access to the CPU oracle.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module; nothing under bce_b200/ does (tests/test_no_oracle_in_product.py checks).

  liboracle.so          plain-C restatement of the reference path (oracle/bce_oracle.c)
  _ref/libbce_ref_tap.so the UNMODIFIED reference behind a recording coder (oracle/ref_tap.cpp)
  _ref/bce_ref          the UNMODIFIED reference command line tool
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / "_build" / "liboracle.so"
TAP = HERE / "_ref" / "libbce_ref_tap.so"
REF_BIN = HERE / "_ref" / "bce_ref"
REF_TIME_BIN = HERE / "_ref" / "bce_ref_time"


class CseResult(C.Structure):
    _fields_ = [("tuples", C.c_void_p * 8), ("count", C.c_size_t * 8), ("cap", C.c_size_t * 8),
                ("C", C.c_uint32 * 8), ("visits", C.c_uint64 * 8), ("rounds", C.c_uint64),
                ("peak_frontier", C.c_uint64)]


_lib = None
_tap = None


def lib():
    global _lib
    if _lib is None:
        if not LIB.exists():
            subprocess.run(["make", "-C", str(HERE), "oracle"], check=True, capture_output=True)
        L = C.CDLL(str(LIB))
        L.bceo_least_rotation.argtypes = [C.c_void_p, C.c_size_t]
        L.bceo_least_rotation.restype = C.c_uint32
        L.bceo_bwt.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p]
        L.bceo_wavelet.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
        L.bceo_cse.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(CseResult)]
        L.bceo_cse_free.argtypes = [C.POINTER(CseResult)]
        L.bceo_encode_archive.argtypes = [C.POINTER(CseResult), C.c_uint32, C.c_uint32, C.c_void_p,
                                          C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
        L.bceo_compress.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
        L.bceo_unbwt_bitwise.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_void_p]
        L.bceo_unbwt_bytewise.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_void_p]
        L.bceo_wavelet_to_bytes.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_void_p]
        L.bceo_default_config.restype = C.c_void_p
        L.bceo_free.argtypes = [C.c_void_p]
        L.bceo_call_checksum.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64, C.POINTER(C.c_uint64)]
        L.bceo_word_checksum.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64, C.POINTER(C.c_uint64)]
        # published only once every signature is set: a thread that found it earlier would pass 64-bit pointers as C ints
        _lib = L
    return _lib


def _u8(data) -> np.ndarray:
    if isinstance(data, (bytes, bytearray, memoryview)):
        return np.frombuffer(data, dtype=np.uint8)
    return np.ascontiguousarray(data, dtype=np.uint8)


def least_rotation(data) -> int:
    T = _u8(data)
    return int(lib().bceo_least_rotation(T.ctypes.data, T.size))


def bwt(data, want_sa: bool = False):
    T = _u8(data)
    n = T.size
    L = np.empty(n, dtype=np.uint8)
    sa = np.empty(n, dtype=np.uint32) if want_sa else None
    off = C.c_uint32()
    rc = lib().bceo_bwt(T.ctypes.data, n, L.ctypes.data, C.byref(off), sa.ctypes.data if want_sa else None)
    if rc != 0:
        raise RuntimeError(f"bceo_bwt failed: {rc}")
    return L, int(off.value), sa


def _rank_ptrs(ranks):
    return (C.c_void_p * 8)(*[r.ctypes.data for r in ranks])


def wavelet(L):
    L = _u8(L)
    n = L.size
    ranks = [np.zeros(n // 32 + 1, dtype=np.uint64) for _ in range(8)]
    lib().bceo_wavelet(L.ctypes.data, n, _rank_ptrs(ranks))
    return ranks


def cse(ranks, n: int):
    """Returns dict(C, streams[8] as (E,5) uint32 arrays, visits[8], rounds, peak_frontier)."""
    r = CseResult()
    rc = lib().bceo_cse(_rank_ptrs(ranks), n, C.byref(r))
    if rc != 0:
        raise RuntimeError(f"bceo_cse failed: {rc}")
    streams = []
    for i in range(8):
        cnt = int(r.count[i])
        if cnt:
            a = np.ctypeslib.as_array((C.c_uint32 * (cnt * 5)).from_address(r.tuples[i])).reshape(cnt, 5).copy()
        else:
            a = np.zeros((0, 5), dtype=np.uint32)
        streams.append(a)
    out = dict(C=[int(x) for x in r.C], streams=streams, visits=[int(x) for x in r.visits],
               rounds=int(r.rounds), peak_frontier=int(r.peak_frontier))
    lib().bceo_cse_free(C.byref(r))
    return out


def encode_archive(Cvals, streams, n: int, offset: int, cfg: bytes | None = None) -> bytes:
    """AdaptiveCoder + header + concat (bce.cpp:1117-1167) over given count streams."""
    r = CseResult()
    keep = []
    for i in range(8):
        a = np.ascontiguousarray(streams[i], dtype=np.uint32)
        keep.append(a)
        r.tuples[i] = a.ctypes.data if a.size else None
        r.count[i] = a.shape[0]
        r.C[i] = Cvals[i]
    w = C.c_void_p()
    nw = C.c_size_t()
    cfgbuf = np.frombuffer(cfg, dtype=np.uint8) if cfg is not None else None
    rc = lib().bceo_encode_archive(C.byref(r), n, offset, cfgbuf.ctypes.data if cfgbuf is not None else None,
                                   C.byref(w), C.byref(nw))
    if rc != 0:
        raise RuntimeError(f"bceo_encode_archive failed: {rc}")
    out = C.string_at(w.value, nw.value * 2)
    lib().bceo_free(w)
    return out


def compress(data, cfg: bytes | None = None) -> bytes:
    T = _u8(data)
    w = C.c_void_p()
    nw = C.c_size_t()
    cfgbuf = np.frombuffer(cfg, dtype=np.uint8) if cfg is not None else None
    rc = lib().bceo_compress(T.ctypes.data, T.size, cfgbuf.ctypes.data if cfgbuf is not None else None,
                             C.byref(w), C.byref(nw))
    if rc != 0:
        raise RuntimeError(f"bceo_compress failed: {rc}")
    out = C.string_at(w.value, nw.value * 2)
    lib().bceo_free(w)
    return out


def unbwt_bitwise(ranks, offset: int, n: int) -> np.ndarray:
    out = np.empty(n, dtype=np.uint8)
    lib().bceo_unbwt_bitwise(_rank_ptrs(ranks), offset, n, out.ctypes.data)
    return out


def unbwt_bytewise(ranks, offset: int, n: int) -> np.ndarray:
    out = np.empty(n, dtype=np.uint8)
    rc = lib().bceo_unbwt_bytewise(_rank_ptrs(ranks), offset, n, out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"bceo_unbwt_bytewise failed: {rc}")
    return out


def default_config() -> bytes:
    return C.string_at(lib().bceo_default_config(), 288)


# ---- the unmodified reference -------------------------------------------------------------
def have_ref() -> bool:
    return TAP.exists() and REF_BIN.exists()


def tap():
    global _tap
    if _tap is None:
        _tap = C.CDLL(str(TAP))
        t = _tap
        t.bce_ref_front.argtypes = [C.c_char_p, C.c_int]
        t.bce_ref_n.restype = C.c_uint32
        t.bce_ref_offset.restype = C.c_uint32
        t.bce_ref_bwt.restype = C.c_void_p
        t.bce_ref_ranks.argtypes = [C.c_int]
        t.bce_ref_ranks.restype = C.c_void_p
        t.bce_ref_seconds_rankfile.restype = C.c_double
        t.bce_ref_seconds_encode.restype = C.c_double
        t.bce_ref_calls.argtypes = [C.c_int]
        t.bce_ref_calls.restype = C.c_uint64
        t.bce_ref_checksum.argtypes = [C.c_int, C.c_int]
        t.bce_ref_checksum.restype = C.c_uint64
        t.bce_ref_adaptive.argtypes = [C.c_int, C.POINTER(C.c_size_t)]
        t.bce_ref_adaptive.restype = C.c_void_p
        t.bce_ref_uniform.argtypes = [C.c_int, C.POINTER(C.c_size_t)]
        t.bce_ref_uniform.restype = C.c_void_p
    return _tap


A64 = 0x9E3779B97F4A7C15


def call_checksum(tuples, first_index: int = 0):
    """(sum, wsum) of ref_tap.cpp's per-stream call checksum over an (E, 5) uint32 array whose
    first row is call number `first_index` of its stream; both mod 2^64, so batches add up."""
    t = np.ascontiguousarray(tuples, dtype=np.uint32).reshape(-1, 5).astype(np.uint64)
    with np.errstate(over="ignore"):
        A = np.uint64(A64)
        h = t[:, 0]
        for c in range(1, 5):
            h = h * A + t[:, c]
        j = np.arange(first_index, first_index + t.shape[0], dtype=np.uint64)
        return int(h.sum(dtype=np.uint64)), int((h * (j * np.uint64(2) + np.uint64(1))).sum(dtype=np.uint64))


def call_checksum_fast(tuples, first_index: int = 0):
    """call_checksum through liboracle (C loop; the GIL is released, so streams can be summed in threads)."""
    t = np.ascontiguousarray(tuples, dtype=np.uint32)
    out = (C.c_uint64 * 2)()
    lib().bceo_call_checksum(t.ctypes.data, t.size // 5, first_index, out)
    return int(out[0]), int(out[1])


def word_checksum(words, first_index: int = 0):
    """(sum, wsum) of packed words as bce_gpu_resident_checksum defines them."""
    w = np.ascontiguousarray(words, dtype=np.uint32)
    out = (C.c_uint64 * 2)()
    lib().bceo_word_checksum(w.ctypes.data, w.size, first_index, out)
    return int(out[0]), int(out[1])


def ref_front(data, want_bwt=True, want_ranks=False, record=True, checksum=False):
    """Run the unmodified reference front end (RankFile + BCE<tap>::encode) on `data`."""
    T = _u8(data)
    with tempfile.NamedTemporaryFile(suffix=".in", delete=False) as f:
        f.write(T.tobytes())
        path = f.name
    try:
        flags = (1 if want_bwt else 0) | (2 if want_ranks else 0) | (0 if record else 4) | (8 if checksum else 0)
        # the reference prints progress to stdout; keep pytest output clean
        devnull = os.open(os.devnull, os.O_WRONLY)
        saved = os.dup(1)
        os.dup2(devnull, 1)
        try:
            rc = tap().bce_ref_front(path.encode(), flags)
        finally:
            os.dup2(saved, 1)
            os.close(saved)
            os.close(devnull)
        if rc != 0:
            raise RuntimeError("reference front end failed")
    finally:
        os.unlink(path)
    t = tap()
    n = int(t.bce_ref_n())
    out = dict(n=n, offset=int(t.bce_ref_offset()),
               seconds_rankfile=float(t.bce_ref_seconds_rankfile()),
               seconds_encode=float(t.bce_ref_seconds_encode()),
               calls=[int(t.bce_ref_calls(i)) for i in range(8)])
    if want_bwt:
        out["bwt"] = np.ctypeslib.as_array((C.c_uint8 * n).from_address(t.bce_ref_bwt())).copy()
    if want_ranks:
        words = n // 32 + 1
        out["ranks"] = [np.ctypeslib.as_array((C.c_uint64 * words).from_address(t.bce_ref_ranks(j))).copy()
                        for j in range(8)]
    if record or checksum:
        out["checksum"] = [(int(t.bce_ref_checksum(i, 0)), int(t.bce_ref_checksum(i, 1))) for i in range(8)]
    Cv = []
    for i in range(8):
        cnt = C.c_size_t()
        p = t.bce_ref_uniform(i, C.byref(cnt))
        u = np.ctypeslib.as_array((C.c_uint32 * (cnt.value * 2)).from_address(p)).reshape(-1, 2)
        Cv.append(int(u[0, 0]))        # first uniform call on stream i is set(C[i], n+1), bce.cpp:1129
    out["C"] = Cv
    if record:
        streams = []
        for i in range(8):
            cnt = C.c_size_t()
            p = t.bce_ref_adaptive(i, C.byref(cnt))
            a = (np.ctypeslib.as_array((C.c_uint32 * (cnt.value * 5)).from_address(p)).reshape(-1, 5).copy()
                 if cnt.value else np.zeros((0, 5), dtype=np.uint32))
            streams.append(a)
        out["streams"] = streams
    return out


def ref_compress(data, cfg_path: str | None = None, threads: int | None = None):
    """`bce_ref -c` on a temp file; returns the archive bytes."""
    T = _u8(data)
    env = dict(os.environ)
    if threads:
        env["OMP_NUM_THREADS"] = str(threads)
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "in")
        arc = os.path.join(d, "a.bce")
        with open(src, "wb") as f:
            f.write(T.tobytes())
        cmd = [str(REF_BIN), "-c", arc, src] + ([cfg_path] if cfg_path else [])
        subprocess.run(cmd, check=True, capture_output=True, env=env)
        with open(arc, "rb") as f:
            return f.read()


def ref_decompress(archive: bytes, low_mem: bool = False) -> bytes:
    with tempfile.TemporaryDirectory() as d:
        arc = os.path.join(d, "a.bce")
        dst = os.path.join(d, "out")
        with open(arc, "wb") as f:
            f.write(archive)
        subprocess.run([str(REF_BIN), "-ds" if low_mem else "-d", dst, arc], check=True, capture_output=True)
        with open(dst, "rb") as f:
            return f.read()
