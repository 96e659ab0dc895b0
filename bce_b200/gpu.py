"""ctypes binding of the C ABI in include/bce_gpu.h (libbce_gpu.so).

This is plumbing for tests, bench.py and the batch driver; the product boundary is the
C ABI itself (the `bce` tool in csrc/host links it directly).  There is no CPU fallback:
if the CUDA library is missing or no sm_100 device is present, construction raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
_LIB_PATH = _PKG / "libbce_gpu.so"

ERRORS = {
    0: "ok", -1: "bad argument", -2: "out of memory", -3: "CUDA failure",
    -4: "call sequence violated", -5: "CSE frontier exceeded its device memory",
    -6: "internal consistency check failed", -7: "no usable CUDA device",
}

# every symbol include/bce_gpu.h declares (tests check that the library exports them all)
ABI_SYMBOLS = [
    "bce_gpu_open", "bce_gpu_close", "bce_gpu_abi_version", "bce_gpu_error_string",
    "bce_gpu_last_error", "bce_gpu_get_stats", "bce_gpu_set_scratch_limit", "bce_gpu_bwt",
    "bce_gpu_wavelet", "bce_gpu_cse_begin", "bce_gpu_cse_next", "bce_gpu_compress_front",
    "bce_gpu_stage_input", "bce_gpu_front_resident", "bce_gpu_unbwt",
    "bce_gpu_set_emit_mode", "bce_gpu_cse_next_words", "bce_gpu_set_option",
    "bce_gpu_resident_checksum", "bce_gpu_cse_next_buckets", "bce_gpu_host_alloc", "bce_gpu_host_free",
    "bce_gpu_cse_next_words20", "bce_gpu_prefetch_input", "bce_gpu_compress_many", "bce_gpu_unbwt_many",
    "bce_gpu_compress_many_archives", "bce_gpu_decompress_many",
]
MANY_MAX_N = 65536            # BCE_GPU_MANY_MAX_N
OPT_EMIT_BATCH_BYTES, OPT_LOCAL_SORT_MIN, OPT_RESIDENT_CHECKSUM, OPT_SLOT_ENTER_NODES = 1, 2, 3, 4
OPT_MID_ENTER_NODES, OPT_NO_NARROW_KERNELS = 5, 6


class BceGpuError(RuntimeError):
    def __init__(self, code: int, detail: str = ""):
        self.code = code
        super().__init__(f"bce_gpu error {code} ({ERRORS.get(code, '?')}): {detail}")


class Tuple5(C.Structure):
    _fields_ = [("sym", C.c_uint32), ("k", C.c_uint32), ("c1", C.c_uint32), ("c2", C.c_uint32), ("cs", C.c_uint32)]


class CseBatch(C.Structure):
    _fields_ = [("tuples", C.POINTER(Tuple5) * 8), ("count", C.c_size_t * 8), ("done", C.c_int)]


class CseWords(C.Structure):
    _fields_ = [("words", C.POINTER(C.c_uint32) * 8), ("count", C.c_size_t * 8), ("done", C.c_int)]


class CseWords20(C.Structure):
    _fields_ = [("bytes", C.POINTER(C.c_uint8) * 8), ("count", C.c_size_t * 8), ("done", C.c_int)]


class ScanBucket(C.Structure):
    _fields_ = [("key", C.c_uint32), ("start", C.c_uint32), ("first", C.c_uint32), ("reserved", C.c_uint32)]


class ScanBuckets(C.Structure):
    _fields_ = [("syms", C.POINTER(C.c_uint8) * 8), ("count", C.c_size_t * 8),
                ("buckets", C.POINTER(ScanBucket) * 8), ("nbuckets", C.c_size_t * 8),
                ("halvings", C.c_uint64 * 8), ("done", C.c_int)]


class ManyResult(C.Structure):
    _fields_ = [("offset", C.c_uint32), ("C", C.c_uint32 * 8), ("done", C.c_int),
                ("words", C.POINTER(C.c_uint32) * 8), ("count", C.c_size_t * 8)]


class ManyArchive(C.Structure):
    _fields_ = [("words", C.POINTER(C.c_uint16)), ("nwords", C.c_size_t), ("done", C.c_int)]


EMIT_RAW, EMIT_CODER, EMIT_SCAN = 0, 1, 2


class Stats(C.Structure):
    _fields_ = [
        ("n", C.c_uint32), ("sort_rounds", C.c_uint32),
        ("sort_m", C.c_uint64 * 48), ("sort_passes", C.c_uint32 * 48),
        ("radix_launches", C.c_uint64), ("radix_elems", C.c_uint64),
        ("cse_visits", C.c_uint64), ("cse_tuples", C.c_uint64), ("cse_rounds", C.c_uint64),
        ("cse_launches", C.c_uint64), ("cse_peak_frontier", C.c_uint64), ("gpu_launches", C.c_uint64),
        ("ms_h2d", C.c_float), ("ms_d2h", C.c_float),
        ("ms_pack", C.c_float), ("ms_radix", C.c_float), ("ms_rerank", C.c_float),
        ("ms_rekey", C.c_float), ("ms_bwt_gather", C.c_float),
        ("ms_wavelet", C.c_float), ("ms_cse", C.c_float),
        ("ms_unbwt_bytes", C.c_float), ("ms_unbwt_chase", C.c_float),
        ("ms_bwt_total", C.c_float), ("ms_cse_total", C.c_float), ("ms_total", C.c_float),
        ("ms_cse_narrow", C.c_float), ("cse_rounds_narrow", C.c_uint32), ("ms_radix_kernel", C.c_float),
        ("cse_words", C.c_uint64), ("sort_local_elems", C.c_uint64), ("sort_fallback_elems", C.c_uint64),
        ("sort_radix_passes", C.c_uint32 * 48),
        ("unbwt_dicts", C.c_uint32), ("unbwt_serial", C.c_uint32), ("ms_coder", C.c_float),
        ("ms_decoder", C.c_float),
    ]

    def as_dict(self) -> dict:
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            if name in ("sort_m", "sort_passes", "sort_radix_passes"):
                v = [int(x) for x in v][: int(self.sort_rounds)]
            d[name] = v
        return d


_lib = None


def load_library() -> C.CDLL:
    """Load libbce_gpu.so; raise (never fall back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise BceGpuError(-7, f"{_LIB_PATH} not built: run `python -m bce_b200.build` (needs nvcc)")
    lib = C.CDLL(str(_LIB_PATH))
    vp, u32, u32p = C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)
    lib.bce_gpu_open.argtypes = [C.c_int, C.POINTER(vp)]
    lib.bce_gpu_close.argtypes = [vp]
    lib.bce_gpu_close.restype = None
    lib.bce_gpu_error_string.argtypes = [C.c_int]
    lib.bce_gpu_error_string.restype = C.c_char_p
    lib.bce_gpu_last_error.argtypes = [vp]
    lib.bce_gpu_last_error.restype = C.c_char_p
    lib.bce_gpu_get_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.bce_gpu_set_scratch_limit.argtypes = [vp, C.c_size_t]
    lib.bce_gpu_set_option.argtypes = [vp, C.c_int, C.c_uint64]
    lib.bce_gpu_cse_next_buckets.argtypes = [vp, C.POINTER(ScanBuckets)]
    lib.bce_gpu_cse_next_words20.argtypes = [vp, C.POINTER(CseWords20)]
    lib.bce_gpu_prefetch_input.argtypes = [vp, vp, u32]
    lib.bce_gpu_host_alloc.argtypes = [vp, C.c_size_t]
    lib.bce_gpu_host_alloc.restype = vp
    lib.bce_gpu_host_free.argtypes = [vp, vp]
    lib.bce_gpu_resident_checksum.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.bce_gpu_bwt.argtypes = [vp, vp, u32, vp, u32p, vp]
    lib.bce_gpu_wavelet.argtypes = [vp, vp, u32, C.POINTER(vp), u32p]
    lib.bce_gpu_cse_begin.argtypes = [vp, vp, u32, u32p]
    lib.bce_gpu_cse_next.argtypes = [vp, C.POINTER(CseBatch)]
    lib.bce_gpu_compress_front.argtypes = [vp, vp, u32, u32p, u32p]
    lib.bce_gpu_stage_input.argtypes = [vp, vp, u32]
    lib.bce_gpu_front_resident.argtypes = [vp, u32p, C.POINTER(C.c_uint64)]
    lib.bce_gpu_unbwt.argtypes = [vp, C.POINTER(vp), u32, u32, vp]
    lib.bce_gpu_set_emit_mode.argtypes = [vp, C.c_int, vp]
    lib.bce_gpu_cse_next_words.argtypes = [vp, C.POINTER(CseWords)]
    lib.bce_gpu_compress_many.argtypes = [vp, vp, C.POINTER(C.c_uint64), u32, C.POINTER(ManyResult)]
    lib.bce_gpu_unbwt_many.argtypes = [vp, vp, vp, vp, u32, vp]
    lib.bce_gpu_compress_many_archives.argtypes = [vp, vp, C.POINTER(C.c_uint64), u32, vp, C.POINTER(ManyArchive)]
    lib.bce_gpu_decompress_many.argtypes = [vp, vp, C.POINTER(C.c_uint64), vp, u32, vp, vp]
    _lib = lib
    return lib


def _as_u8(data) -> np.ndarray:
    if isinstance(data, (bytes, bytearray, memoryview)):
        return np.frombuffer(data, dtype=np.uint8)
    a = np.ascontiguousarray(data)
    if a.dtype != np.uint8:
        raise TypeError("expected bytes or a uint8 array")
    return a


def _pack(items, dtype, pad: bool = False):
    """The items (bytes or uint8 arrays) back to back as one array of dtype, and their k + 1 starts (uint64).  pad:
    one element more at the end, so that the buffer is never empty (the decompress calls take no null pointer)."""
    width = np.dtype(dtype).itemsize
    arrs = [_as_u8(d) for d in items]
    sizes = [a.size for a in arrs]
    if width > 1 and any(n % width for n in sizes):
        raise ValueError(f"every item must hold whole {np.dtype(dtype).name} elements")
    buf = np.concatenate(arrs + [np.zeros(width * int(pad), dtype=np.uint8)]).view(dtype)
    starts = np.zeros(len(arrs) + 1, dtype=np.uint64)
    np.cumsum(sizes, out=starts[1:])
    return buf, starts // np.uint64(width)


class Frontend:
    """One context per GPU (mirrors bce_gpu_open / bce_gpu_close)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.bce_gpu_open(device, C.byref(h))
        if rc != 0:
            raise BceGpuError(rc, "bce_gpu_open")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.bce_gpu_close(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise BceGpuError(rc, self.lib.bce_gpu_last_error(self.h).decode(errors="replace"))

    # -- stage A ------------------------------------------------------------------------
    def bwt(self, data, want_sa: bool = False):
        T = _as_u8(data)
        n = T.size
        L = np.empty(n, dtype=np.uint8)
        sa = np.empty(n, dtype=np.uint32) if want_sa else None
        off = C.c_uint32()
        self._check(self.lib.bce_gpu_bwt(self.h, T.ctypes.data, n, L.ctypes.data, C.byref(off),
                                         sa.ctypes.data if want_sa else None))
        return L, int(off.value), sa

    # -- stage B ------------------------------------------------------------------------
    def wavelet(self, L=None, n: int | None = None):
        if L is not None:
            L = _as_u8(L)
            n = L.size
        words = n // 32 + 1
        ranks = [np.empty(words, dtype=np.uint64) for _ in range(8)]
        ptrs = (C.c_void_p * 8)(*[r.ctypes.data for r in ranks])
        Cv = (C.c_uint32 * 8)()
        self._check(self.lib.bce_gpu_wavelet(self.h, L.ctypes.data if L is not None else None, n, ptrs, Cv))
        return ranks, [int(x) for x in Cv]

    def _drain(self):
        streams = [[] for _ in range(8)]
        batch = CseBatch()
        batches = 0
        while True:
            self._check(self.lib.bce_gpu_cse_next(self.h, C.byref(batch)))
            batches += 1
            for i in range(8):
                cnt = int(batch.count[i])
                if cnt:
                    addr = C.addressof(batch.tuples[i].contents)
                    arr = np.ctypeslib.as_array((C.c_uint32 * (cnt * 5)).from_address(addr)).reshape(cnt, 5)
                    streams[i].append(arr.copy())
            if batch.done:
                break
        out = [np.concatenate(s) if s else np.zeros((0, 5), dtype=np.uint32) for s in streams]
        self.last_batches = batches
        return out, batches

    def cse(self, L=None, n: int | None = None):
        """Returns (C[8], streams[8]); stream i is an (E_i, 5) uint32 array of set() arguments."""
        if L is not None:
            L = _as_u8(L)
            n = L.size
        Cv = (C.c_uint32 * 8)()
        self._check(self.lib.bce_gpu_cse_begin(self.h, L.ctypes.data if L is not None else None, n, Cv))
        streams, _ = self._drain()
        return [int(x) for x in Cv], streams

    def compress_front(self, data):
        """BWT + wavelet + CSE with the BWT staying on the device."""
        T = _as_u8(data)
        off = C.c_uint32()
        Cv = (C.c_uint32 * 8)()
        self._check(self.lib.bce_gpu_compress_front(self.h, T.ctypes.data, T.size, C.byref(off), Cv))
        streams, _ = self._drain()
        return int(off.value), [int(x) for x in Cv], streams

    def set_emit_mode(self, mode: int, cfg: bytes | None = None):
        """EMIT_RAW (20-byte counts), EMIT_CODER or EMIT_SCAN (packed words, include/bce_gpu.h)."""
        buf = np.frombuffer(cfg, dtype=np.uint8) if cfg is not None else None
        self._check(self.lib.bce_gpu_set_emit_mode(self.h, mode, buf.ctypes.data if buf is not None else None))

    def compress_front_words(self, data, mode: int = EMIT_CODER, cfg: bytes | None = None):
        """Fused front end with packed emission: (offset, C[8], 8 uint32 word arrays)."""
        T = _as_u8(data)
        self.set_emit_mode(mode, cfg)
        try:
            off = C.c_uint32()
            Cv = (C.c_uint32 * 8)()
            self._check(self.lib.bce_gpu_compress_front(self.h, T.ctypes.data, T.size, C.byref(off), Cv))
            streams = [[] for _ in range(8)]
            batch = CseWords()
            while True:
                self._check(self.lib.bce_gpu_cse_next_words(self.h, C.byref(batch)))
                for i in range(8):
                    cnt = int(batch.count[i])
                    if cnt:
                        addr = C.addressof(batch.words[i].contents)
                        streams[i].append(np.ctypeslib.as_array((C.c_uint32 * cnt).from_address(addr)).copy())
                if batch.done:
                    break
        finally:
            self.set_emit_mode(EMIT_RAW)
        out = [np.concatenate(s) if s else np.zeros(0, dtype=np.uint32) for s in streams]
        return int(off.value), [int(x) for x in Cv], out

    def iter_front_batches(self, data, mode: int = EMIT_RAW, cfg: bytes | None = None):
        """Fused front end, batch by batch, without keeping anything: yields ("head", offset, C[8]) first,
        then ("batch", [8 uint32 views into the context's pinned buffers]) until the loop is done.  A view
        is valid until the next batch is asked for (inputs whose counts do not fit in host memory)."""
        T = _as_u8(data)
        self.set_emit_mode(mode, cfg)
        try:
            off = C.c_uint32()
            Cv = (C.c_uint32 * 8)()
            self._check(self.lib.bce_gpu_compress_front(self.h, T.ctypes.data, T.size, C.byref(off), Cv))
            yield "head", int(off.value), [int(x) for x in Cv]
            batch = CseWords()
            while True:
                self._check(self.lib.bce_gpu_cse_next_words(self.h, C.byref(batch)))
                views = []
                for i in range(8):
                    cnt = int(batch.count[i])
                    if cnt:
                        addr = C.addressof(batch.words[i].contents)
                        views.append(np.ctypeslib.as_array((C.c_uint32 * cnt).from_address(addr)))
                    else:
                        views.append(np.zeros(0, dtype=np.uint32))
                yield "batch", views
                if batch.done:
                    break
        finally:
            self.set_emit_mode(EMIT_RAW)

    def compress_front_buckets(self, data):
        """`bce -s` front end: (offset, C[8], batches); a batch is a list of 8 tuples (syms uint8 array, buckets
        structured array with fields key / start / first, halvings) as bce_gpu_cse_next_buckets returns them."""
        T = _as_u8(data)
        self.set_emit_mode(EMIT_SCAN)
        try:
            off = C.c_uint32()
            Cv = (C.c_uint32 * 8)()
            self._check(self.lib.bce_gpu_compress_front(self.h, T.ctypes.data, T.size, C.byref(off), Cv))
            batches = []
            b = ScanBuckets()
            dt = np.dtype([("key", "<u4"), ("start", "<u4"), ("first", "<u4"), ("reserved", "<u4")])
            while True:
                self._check(self.lib.bce_gpu_cse_next_buckets(self.h, C.byref(b)))
                one = []
                for i in range(8):
                    cnt, nb = int(b.count[i]), int(b.nbuckets[i])
                    syms = (np.ctypeslib.as_array((C.c_uint8 * cnt).from_address(C.addressof(b.syms[i].contents))).copy()
                            if cnt else np.zeros(0, dtype=np.uint8))
                    bk = (np.frombuffer((C.c_uint8 * (16 * nb)).from_address(C.addressof(b.buckets[i].contents)), dtype=dt).copy()
                          if nb else np.zeros(0, dtype=dt))
                    one.append((syms, bk, int(b.halvings[i])))
                batches.append(one)
                if b.done:
                    break
        finally:
            self.set_emit_mode(EMIT_RAW)
        return int(off.value), [int(x) for x in Cv], batches

    def compress_many_call(self, inputs):
        """One bce_gpu_compress_many call in the context's emission mode: the ManyResult array (valid until the call
        after the next) for `inputs`, a list of bytes / uint8 arrays of 1 .. MANY_MAX_N bytes."""
        T, starts = _pack(inputs, np.uint8)
        out = (ManyResult * max(len(inputs), 1))()
        self._check(self.lib.bce_gpu_compress_many(self.h, T.ctypes.data if T.size else None,
                                                   starts.ctypes.data_as(C.POINTER(C.c_uint64)), len(inputs), out))
        return out

    def compress_front_many(self, inputs, mode: int = EMIT_RAW, cfg: bytes | None = None):
        """Front end of many small inputs (bce_gpu_compress_many), resubmitting the inputs that did not fit in a call's
        arena until all are done: [(offset, C[8], 8 streams)] per input; a stream is an (E, 5) uint32 array of set()
        arguments in EMIT_RAW mode, else the packed words.  self.last_many_calls = the calls it took."""
        self.set_emit_mode(mode, cfg)
        res = [None] * len(inputs)
        todo = list(range(len(inputs)))
        calls = 0
        try:
            while todo:
                out = self.compress_many_call([inputs[i] for i in todo])
                calls += 1
                left = []
                for j, i in enumerate(todo):
                    r = out[j]
                    if not r.done:
                        left.append(i)
                        continue
                    streams = []
                    for s in range(8):
                        cnt = int(r.count[s])
                        w = (np.ctypeslib.as_array((C.c_uint32 * cnt).from_address(C.addressof(r.words[s].contents))).copy()
                             if cnt else np.zeros(0, dtype=np.uint32))
                        streams.append(w.reshape(-1, 5) if mode == EMIT_RAW else w)
                    res[i] = (int(r.offset), [int(x) for x in r.C], streams)
                if len(left) == len(todo):
                    raise BceGpuError(-6, "compress_many: no input was done")
                todo = left
        finally:
            self.set_emit_mode(EMIT_RAW)
        self.last_many_calls = calls
        return res

    def compress_many_archives(self, inputs, cfg: bytes | None = None) -> list:
        """One bce_gpu_compress_many_archives call: per input of 1 .. MANY_MAX_N bytes its `bce -c` archive with the
        288-byte table cfg (None = the default), or None when it did not fit this call and has to be submitted again."""
        T, starts = _pack(inputs, np.uint8)
        buf = np.frombuffer(cfg, dtype=np.uint8) if cfg is not None else None
        out = (ManyArchive * max(len(inputs), 1))()
        self._check(self.lib.bce_gpu_compress_many_archives(self.h, T.ctypes.data if T.size else None,
                                                            starts.ctypes.data_as(C.POINTER(C.c_uint64)), len(inputs),
                                                            buf.ctypes.data if buf is not None else None, out))
        return [C.string_at(out[i].words, 2 * out[i].nwords) if out[i].done else None for i in range(len(inputs))]

    def prefetch_input(self, data):
        """bce_gpu_prefetch_input: upload the next input (page-locked memory) beside the current level loop."""
        T = _as_u8(data)
        self._check(self.lib.bce_gpu_prefetch_input(self.h, T.ctypes.data, T.size))

    def compress_front_discard(self, data, words20: bool = False, prefetch_next=None, on_batch=None):
        """Same call sequence a consumer makes (fused front end, then batches until done) in the
        context's current emission mode; the batches are left in pinned memory (bench e2e leg).
        on_batch(C, batch), if given, sees the input's C[8] and every CseWords20 / CseWords batch while
        its words are valid.  Returns (offset, total 32-bit words handed back)."""
        T = _as_u8(data)
        off = C.c_uint32()
        Cv = (C.c_uint32 * 8)()
        self._check(self.lib.bce_gpu_compress_front(self.h, T.ctypes.data, T.size, C.byref(off), Cv))
        if prefetch_next is not None:             # the next input's upload runs beside this input's level loop
            self.prefetch_input(prefetch_next)
        batch = CseWords20() if words20 else CseWords()
        nxt = self.lib.bce_gpu_cse_next_words20 if words20 else self.lib.bce_gpu_cse_next_words
        total = 0
        while True:
            self._check(nxt(self.h, C.byref(batch)))
            if on_batch is not None:
                on_batch(Cv, batch)
            total += sum(int(batch.count[i]) for i in range(8))
            if batch.done:
                break
        return int(off.value), total

    def compress_front_words20(self, data, cfg: bytes | None = None):
        """Fused front end, BCE_EMIT_CODER words as the 20-bit form of bce_gpu_cse_next_words20, unpacked to uint32
        arrays again: (offset, C[8], 8 word arrays)."""
        T = _as_u8(data)
        self.set_emit_mode(EMIT_CODER, cfg)
        try:
            off = C.c_uint32()
            Cv = (C.c_uint32 * 8)()
            self._check(self.lib.bce_gpu_compress_front(self.h, T.ctypes.data, T.size, C.byref(off), Cv))
            streams = [[] for _ in range(8)]
            batch = CseWords20()
            while True:
                self._check(self.lib.bce_gpu_cse_next_words20(self.h, C.byref(batch)))
                for i in range(8):
                    cnt = int(batch.count[i])
                    if cnt:
                        pairs = (cnt + 1) // 2
                        b = np.ctypeslib.as_array((C.c_uint8 * (5 * pairs)).from_address(C.addressof(batch.bytes[i].contents)))
                        b = b.reshape(pairs, 5).astype(np.uint32)
                        w = np.empty(2 * pairs, dtype=np.uint32)
                        w[0::2] = b[:, 0] | (b[:, 1] << np.uint32(8)) | ((b[:, 2] & np.uint32(15)) << np.uint32(16))
                        w[1::2] = (b[:, 2] >> np.uint32(4)) | (b[:, 3] << np.uint32(4)) | (b[:, 4] << np.uint32(12))
                        streams[i].append(w[:cnt].copy())
                if batch.done:
                    break
        finally:
            self.set_emit_mode(EMIT_RAW)
        return int(off.value), [int(x) for x in Cv], [np.concatenate(s) if s else np.zeros(0, dtype=np.uint32) for s in streams]

    # -- device-resident measurement -------------------------------------------------------
    def stage_input(self, data):
        T = _as_u8(data)
        self._check(self.lib.bce_gpu_stage_input(self.h, T.ctypes.data, T.size))

    def front_resident(self):
        off = C.c_uint32()
        tup = C.c_uint64()
        self._check(self.lib.bce_gpu_front_resident(self.h, C.byref(off), C.byref(tup)))
        return int(off.value), int(tup.value)

    # -- inverse --------------------------------------------------------------------------
    def unbwt(self, ranks, offset: int, n: int) -> np.ndarray:
        ranks = [np.ascontiguousarray(r, dtype=np.uint64) for r in ranks]
        ptrs = (C.c_void_p * 8)(*[r.ctypes.data for r in ranks])
        out = np.empty(n, dtype=np.uint8)
        self._check(self.lib.bce_gpu_unbwt(self.h, ptrs, offset, n, out.ctypes.data))
        return out

    def unbwt_many(self, dicts) -> list:
        """bce_gpu_unbwt_many: dicts = [(ranks8, offset, n), ...] with n <= MANY_MAX_N (ranks8: the 8 levels of n // 32
        + 1 words each) -> one uint8 array per dictionary, every inverse in one launch."""
        ns = np.array([int(n) for _, _, n in dicts], dtype=np.uint32)
        offs = np.array([int(o) for _, o, _ in dicts], dtype=np.uint32)
        levels = [np.ascontiguousarray(r, dtype=np.uint64) for ranks, _, _ in dicts for r in ranks]
        for i, (ranks, _, n) in enumerate(dicts):
            if len(ranks) != 8 or any(np.asarray(r).size != int(n) // 32 + 1 for r in ranks):
                raise ValueError(f"dictionary {i}: needs 8 levels of n // 32 + 1 = {int(n) // 32 + 1} words")
        words = np.concatenate(levels) if levels else np.zeros(0, dtype=np.uint64)
        out = np.empty(int(ns.sum(dtype=np.uint64)), dtype=np.uint8)
        self._check(self.lib.bce_gpu_unbwt_many(self.h, words.ctypes.data if words.size else None,
                                                ns.ctypes.data if ns.size else None,
                                                offs.ctypes.data if offs.size else None, len(dicts),
                                                out.ctypes.data if out.size else None))
        cuts = np.cumsum(ns, dtype=np.uint64)
        return [out[int(a):int(b)] for a, b in zip(np.concatenate([[0], cuts[:-1]]), cuts)]

    def decompress_many(self, archives, sizes) -> list:
        """bce_gpu_decompress_many: archives (bytes of uint16 words) whose headers claim sizes[i] bytes, 1 .. MANY_MAX_N
        each -> per archive its text, or BceGpuError(-1) where the host decoder rejects it; decode loops and inverses
        of all of them in two launches."""
        if len(archives) != len(sizes):
            raise ValueError("one size per archive")
        W, starts = _pack(archives, np.uint16, pad=True)
        ns = np.array([int(n) for n in sizes], dtype=np.uint32)
        out = np.empty(max(int(ns.sum(dtype=np.uint64)), 1), dtype=np.uint8)
        status = np.zeros(max(len(archives), 1), dtype=np.int32)
        self._check(self.lib.bce_gpu_decompress_many(self.h, W.ctypes.data, starts.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                     ns.ctypes.data if ns.size else None, len(archives), out.ctypes.data,
                                                     status.ctypes.data))
        res, at = [], 0
        for i, n in enumerate(ns.tolist()):
            res.append(BceGpuError(int(status[i]), f"archive {i}: damaged") if status[i] else out[at:at + n].tobytes())
            at += n
        return res

    def stats(self) -> dict:
        s = Stats()
        self._check(self.lib.bce_gpu_get_stats(self.h, C.byref(s)))
        return s.as_dict()

    def set_scratch_limit(self, nbytes: int):
        self._check(self.lib.bce_gpu_set_scratch_limit(self.h, nbytes))

    def resident_checksum(self):
        """Per-stream (sum, wsum) of the words the last front_resident run emitted (OPT_RESIDENT_CHECKSUM)."""
        a, b = (C.c_uint64 * 8)(), (C.c_uint64 * 8)()
        self._check(self.lib.bce_gpu_resident_checksum(self.h, a, b))
        return [(int(a[i]), int(b[i])) for i in range(8)]

    def set_option(self, option: int, value: int):
        """bce_gpu_set_option: OPT_EMIT_BATCH_BYTES / OPT_LOCAL_SORT_MIN (0 = default)."""
        self._check(self.lib.bce_gpu_set_option(self.h, option, value))
