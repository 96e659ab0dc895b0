"""ctypes binding of include/bce_host.h (libbce_host.so): host range coders + archive writer."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from .gpu import CseBatch, CseWords, ScanBucket, ScanBuckets, Tuple5, _pack

_LIB_PATH = Path(__file__).resolve().parent / "libbce_host.so"
_lib = None

HOST_SYMBOLS = [
    "bce_archive_begin", "bce_archive_feed", "bce_archive_finish", "bce_archive_abort",
    "bce_scan_begin", "bce_scan_feed", "bce_scan_finish", "bce_compress_buffer", "bce_scan_buffer",
    "bce_host_default_config", "bce_host_free",
    "bce_archive_feed_words", "bce_scan_feed_words", "bce_host_pack_counts", "bce_decode_buffer",
    "bce_archive_begin_words", "bce_archive_wait", "bce_scan_feed_buckets", "bce_archive_begin_words20",
    "bce_compress_many", "bce_decompress_many", "bce_archive_size",
]


def load_library() -> C.CDLL:
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise RuntimeError(f"{_LIB_PATH} not built: run `python -m bce_b200.build`")
        lib = C.CDLL(str(_LIB_PATH))
        vp = C.c_void_p
        lib.bce_archive_begin.argtypes = [C.c_uint32, C.POINTER(C.c_uint32), vp]
        lib.bce_archive_begin.restype = vp
        lib.bce_archive_feed.argtypes = [vp, C.POINTER(CseBatch), C.c_int]
        lib.bce_archive_finish.argtypes = [vp, C.c_uint32, C.POINTER(vp), C.POINTER(C.c_size_t)]
        lib.bce_archive_abort.argtypes = [vp]
        lib.bce_scan_begin.restype = vp
        lib.bce_scan_feed.argtypes = [vp, C.POINTER(CseBatch)]
        lib.bce_scan_finish.argtypes = [vp, vp]
        lib.bce_compress_buffer.argtypes = [vp, vp, C.c_uint32, vp, C.c_int, C.POINTER(vp), C.POINTER(C.c_size_t)]
        lib.bce_scan_buffer.argtypes = [vp, vp, C.c_uint32, vp]
        lib.bce_compress_many.argtypes = [vp, vp, C.POINTER(C.c_uint64), C.c_uint32, vp, C.c_int,
                                          C.POINTER(vp), C.POINTER(C.c_size_t)]
        lib.bce_decompress_many.argtypes = [vp, vp, C.POINTER(C.c_uint64), C.c_uint32, C.c_int,
                                            C.POINTER(vp), C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
        lib.bce_host_default_config.restype = vp
        lib.bce_host_free.argtypes = [vp]
        lib.bce_archive_feed_words.argtypes = [vp, C.POINTER(CseWords), C.c_int]
        lib.bce_scan_feed_words.argtypes = [vp, C.POINTER(CseWords)]
        lib.bce_scan_feed_buckets.argtypes = [vp, C.POINTER(ScanBuckets)]
        lib.bce_archive_begin_words.argtypes = [vp, C.POINTER(CseWords)]
        lib.bce_archive_wait.argtypes = [vp]
        lib.bce_host_pack_counts.argtypes = [C.c_int, vp, C.c_int, vp, C.c_size_t, vp]
        lib.bce_host_pack_counts.restype = C.c_size_t
        lib.bce_archive_size.argtypes = [vp, C.c_size_t, C.POINTER(C.c_uint32)]
        lib.bce_decode_buffer.argtypes = [vp, C.c_size_t, C.c_int, C.POINTER(vp), C.POINTER(C.c_size_t)]
        _lib = lib
    return _lib


def _batch_from(streams, done=True):
    keep = [np.ascontiguousarray(s, dtype=np.uint32) for s in streams]
    b = CseBatch()
    for i, a in enumerate(keep):
        b.count[i] = a.shape[0]
        if a.shape[0]:
            b.tuples[i] = C.cast(a.ctypes.data, C.POINTER(Tuple5))
    b.done = 1 if done else 0
    return b, keep


def encode_archive(Cvals, streams, n: int, offset: int, cfg: bytes | None = None, threads: int = 1,
                   pieces: int = 1) -> bytes:
    """Host archive writer over given count streams (optionally fed in `pieces` batches)."""
    lib = load_library()
    Cv = (C.c_uint32 * 8)(*Cvals)
    cfgbuf = np.frombuffer(cfg, dtype=np.uint8) if cfg is not None else None
    w = lib.bce_archive_begin(n, Cv, cfgbuf.ctypes.data if cfgbuf is not None else None)
    if not w:
        raise RuntimeError("bce_archive_begin failed")
    for p in range(pieces):
        part = [s[(s.shape[0] * p) // pieces:(s.shape[0] * (p + 1)) // pieces] for s in streams]
        b, keep = _batch_from(part, done=(p == pieces - 1))
        rc = lib.bce_archive_feed(w, C.byref(b), threads)
        assert rc == 0
    words = C.c_void_p()
    nw = C.c_size_t()
    rc = lib.bce_archive_finish(w, offset, C.byref(words), C.byref(nw))
    if rc != 0:
        raise RuntimeError(f"bce_archive_finish failed: {rc}")
    out = C.string_at(words.value, nw.value * 2)
    lib.bce_host_free(words)
    return out


def pack_counts(mode: int, streams, cfg: bytes | None = None):
    """Raw (E,5) count streams -> packed word streams with the device's formats (host packer)."""
    lib = load_library()
    cfgbuf = np.frombuffer(cfg, dtype=np.uint8) if cfg is not None else None
    out = []
    for i, s in enumerate(streams):
        a = np.ascontiguousarray(s, dtype=np.uint32)
        w = np.zeros(3 * a.shape[0] + 3, dtype=np.uint32)
        nw = lib.bce_host_pack_counts(mode, cfgbuf.ctypes.data if cfgbuf is not None else None, i,
                                      a.ctypes.data, a.shape[0], w.ctypes.data)
        out.append(w[:nw].copy())
    return out


def _words_batch(word_streams, done=True):
    keep = [np.ascontiguousarray(s, dtype=np.uint32) for s in word_streams]
    b = CseWords()
    for i, a in enumerate(keep):
        b.count[i] = a.shape[0]
        if a.shape[0]:
            b.words[i] = C.cast(a.ctypes.data, C.POINTER(C.c_uint32))
    b.done = 1 if done else 0
    return b, keep


def encode_archive_words(Cvals, word_streams, n: int, offset: int, cfg: bytes | None = None, threads: int = 1) -> bytes:
    """Archive writer over BCE_EMIT_CODER word streams."""
    lib = load_library()
    Cv = (C.c_uint32 * 8)(*Cvals)
    cfgbuf = np.frombuffer(cfg, dtype=np.uint8) if cfg is not None else None
    w = lib.bce_archive_begin(n, Cv, cfgbuf.ctypes.data if cfgbuf is not None else None)
    b, keep = _words_batch(word_streams)
    assert lib.bce_archive_feed_words(w, C.byref(b), threads) == 0
    words = C.c_void_p()
    nw = C.c_size_t()
    rc = lib.bce_archive_finish(w, offset, C.byref(words), C.byref(nw))
    if rc != 0:
        raise RuntimeError(f"bce_archive_finish failed: {rc}")
    out = C.string_at(words.value, nw.value * 2)
    lib.bce_host_free(words)
    return out


def pack20(words) -> np.ndarray:
    """uint32 words below 2^20 -> the byte string of bce_cse_words20 (word j at bit 20 j, 16 readable bytes of slack)."""
    w = np.ascontiguousarray(words, dtype=np.uint32)
    pairs = (w.shape[0] + 1) // 2
    a = np.zeros(2 * pairs, dtype=np.uint64)
    a[:w.shape[0]] = w
    v = a[0::2] | (a[1::2] << np.uint64(20))
    out = np.zeros(pairs * 5 + 16, dtype=np.uint8)
    for k in range(5):
        out[k:pairs * 5:5] = ((v >> np.uint64(8 * k)) & np.uint64(255)).astype(np.uint8)
    return out


def encode_archive_words20(Cvals, word_streams, n: int, offset: int, cfg: bytes | None = None, pieces: int = 1) -> bytes:
    """Archive writer over BCE_EMIT_CODER word streams handed over as 20-bit words (bce_archive_begin_words20 /
    bce_archive_wait), in `pieces` batches per stream cut at count boundaries."""
    from .gpu import CseWords20
    lib = load_library()
    lib.bce_archive_begin_words20.argtypes = [C.c_void_p, C.POINTER(CseWords20)]
    Cv = (C.c_uint32 * 8)(*Cvals)
    cfgbuf = np.frombuffer(cfg, dtype=np.uint8) if cfg is not None else None
    w = lib.bce_archive_begin(n, Cv, cfgbuf.ctypes.data if cfgbuf is not None else None)
    cuts = []
    for s in word_streams:                                   # a k > 31 count is three words: never cut inside one
        s = np.asarray(s, dtype=np.uint32)
        starts = []
        i = 0
        esc = ((s >> np.uint32(5)) & np.uint32(31)) == 0
        while i < s.shape[0]:
            starts.append(i)
            i += 3 if esc[i] else 1
        starts.append(s.shape[0])
        cuts.append([starts[(len(starts) - 1) * p // pieces] for p in range(pieces)] + [s.shape[0]])
    for p in range(pieces):
        b = CseWords20()
        keep = []
        for i, s in enumerate(word_streams):
            part = np.asarray(s, dtype=np.uint32)[cuts[i][p]:cuts[i][p + 1]]
            keep.append(pack20(part))
            b.count[i] = part.shape[0]
            if part.shape[0]:
                b.bytes[i] = C.cast(keep[-1].ctypes.data, C.POINTER(C.c_uint8))
        b.done = 1 if p == pieces - 1 else 0
        assert lib.bce_archive_begin_words20(w, C.byref(b)) == 0
        assert lib.bce_archive_wait(w) == 0
    words = C.c_void_p()
    nw = C.c_size_t()
    rc = lib.bce_archive_finish(w, offset, C.byref(words), C.byref(nw))
    if rc != 0:
        raise RuntimeError(f"bce_archive_finish failed: {rc}")
    out = C.string_at(words.value, nw.value * 2)
    lib.bce_host_free(words)
    return out


def scan_config_words(word_streams) -> bytes:
    lib = load_library()
    s = lib.bce_scan_begin()
    b, keep = _words_batch(word_streams)
    lib.bce_scan_feed_words(s, C.byref(b))
    out = np.zeros(288, dtype=np.uint8)
    rc = lib.bce_scan_finish(s, out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"bce_scan_finish failed: {rc}")
    return out.tobytes()


def bucket_scan_words(words):
    """What the device does to one stream's BCE_EMIT_SCAN words of a batch (csrc/cse.cu, cse_advance_buckets), in
    numpy: stable sort by the bucket bits 5..25 -> (syms, buckets[key, start, first], halvings)."""
    w = np.ascontiguousarray(words, dtype=np.uint32)
    key = (w >> np.uint32(5)) & np.uint32(0x1FFFFF)
    order = np.argsort(key, kind="stable")
    ks = key[order]
    heads = np.flatnonzero(np.concatenate([[True], ks[1:] != ks[:-1]])) if w.size else np.zeros(0, dtype=np.int64)
    dt = np.dtype([("key", "<u4"), ("start", "<u4"), ("first", "<u4"), ("reserved", "<u4")])
    bk = np.zeros(heads.size, dtype=dt)
    bk["key"], bk["start"], bk["first"] = ks[heads], heads, order[heads]
    esc = (w >> np.uint32(31)) != 0
    halvings = int(((w[esc] >> np.uint32(26)) & np.uint32(31)).sum())
    return (w[order] & np.uint32(31)).astype(np.uint8), bk, halvings


def scan_config_buckets(batches) -> bytes:
    """Scan config from batches bucketed as bce_gpu_cse_next_buckets does: batches[b][stream] = (syms, buckets, halvings)."""
    lib = load_library()
    s = lib.bce_scan_begin()
    for bi, one in enumerate(batches):
        b = ScanBuckets()
        keep = []
        for i, (syms, bk, halv) in enumerate(one):
            sy = np.ascontiguousarray(syms, dtype=np.uint8)
            bb = np.ascontiguousarray(bk)
            keep += [sy, bb]
            b.count[i], b.nbuckets[i], b.halvings[i] = sy.size, bb.size, halv
            if sy.size:
                b.syms[i] = C.cast(sy.ctypes.data, C.POINTER(C.c_uint8))
            if bb.size:
                b.buckets[i] = C.cast(bb.ctypes.data, C.POINTER(ScanBucket))
        b.done = 1 if bi == len(batches) - 1 else 0
        rc = lib.bce_scan_feed_buckets(s, C.byref(b))
        if rc != 0:
            raise RuntimeError(f"bce_scan_feed_buckets failed: {rc}")
    out = np.zeros(288, dtype=np.uint8)
    rc = lib.bce_scan_finish(s, out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"bce_scan_finish failed: {rc}")
    return out.tobytes()


def scan_config(streams) -> bytes:
    lib = load_library()
    s = lib.bce_scan_begin()
    b, keep = _batch_from(streams)
    lib.bce_scan_feed(s, C.byref(b))
    out = np.zeros(288, dtype=np.uint8)
    rc = lib.bce_scan_finish(s, out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"bce_scan_finish failed: {rc}")
    return out.tobytes()


def decompress(archive: bytes, low_memory: bool = False) -> bytes:
    """`bce -d` (GPU inverse BWT) / `bce -ds` (serial, host only) on an archive in memory."""
    lib = load_library()
    a = np.frombuffer(archive, dtype=np.uint16)
    out = C.c_void_p()
    n = C.c_size_t()
    rc = lib.bce_decode_buffer(a.ctypes.data, a.size, 1 if low_memory else 0, C.byref(out), C.byref(n))
    if rc != 0:
        raise RuntimeError(f"bce_decode_buffer failed: {rc}")
    data = C.string_at(out.value, n.value)
    lib.bce_host_free(out)
    return data


def default_config() -> bytes:
    return C.string_at(load_library().bce_host_default_config(), 288)


def compress(frontend, data, cfg: bytes | None = None, threads: int = 8) -> bytes:
    """Whole `bce -c` pipeline on a buffer: GPU front end + host coders."""
    lib = load_library()
    T = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else np.ascontiguousarray(data)
    cfgbuf = np.frombuffer(cfg, dtype=np.uint8) if cfg is not None else None
    words = C.c_void_p()
    nw = C.c_size_t()
    rc = lib.bce_compress_buffer(frontend.h, T.ctypes.data, T.size,
                                 cfgbuf.ctypes.data if cfgbuf is not None else None, threads,
                                 C.byref(words), C.byref(nw))
    frontend._check(rc)
    out = C.string_at(words.value, nw.value * 2)
    lib.bce_host_free(words)
    return out


def compress_many(frontend, inputs, cfg: bytes | None = None, threads: int = 8) -> list:
    """`bce -c` of many small inputs (1 .. gpu.MANY_MAX_N bytes each) through one front-end launch per arena's worth:
    one archive per input, the bytes compress() makes of it."""
    lib = load_library()
    T, starts = _pack(inputs, np.uint8)
    cfgbuf = np.frombuffer(cfg, dtype=np.uint8) if cfg is not None else None
    k = len(inputs)
    words = (C.c_void_p * max(k, 1))()
    nw = (C.c_size_t * max(k, 1))()
    rc = lib.bce_compress_many(frontend.h, T.ctypes.data if T.size else None, starts.ctypes.data_as(C.POINTER(C.c_uint64)),
                               k, cfgbuf.ctypes.data if cfgbuf is not None else None, threads, words, nw)
    frontend._check(rc)
    out = []
    for i in range(k):
        out.append(C.string_at(words[i], nw[i] * 2))
        lib.bce_host_free(words[i])
    return out


def archive_size(archive: bytes):
    """The text size an archive's header claims, or None when the header cannot be read."""
    if len(archive) % 2 or not archive:
        return None
    W = np.frombuffer(archive, dtype=np.uint16)
    n = C.c_uint32()
    return int(n.value) if load_library().bce_archive_size(W.ctypes.data, W.size, C.byref(n)) == 0 else None


def decompress_many(frontend, archives, threads: int = 8) -> list:
    """`bce -d` of many archives on the frontend's context (bce_decompress_many): per archive its bytes, or the
    BceGpuError of that archive alone (a damaged archive: code -1).  Archives of at most gpu.MANY_MAX_N bytes of text are
    decoded one per thread and inverted together on the GPU, larger ones as decompress() does."""
    from .gpu import BceGpuError
    lib = load_library()
    k = len(archives)
    res = [None] * k
    good = []
    for i, a in enumerate(archives):
        if len(a) % 2:                                # not a sequence of uint16 words
            res[i] = BceGpuError(-1, f"archive {i}: odd length {len(a)}")
        else:
            good.append(i)
    if not good:
        return res
    W, starts = _pack([archives[i] for i in good], np.uint16, pad=True)
    out = (C.c_void_p * len(good))()
    nout = (C.c_size_t * len(good))()
    status = (C.c_int * len(good))()
    rc = lib.bce_decompress_many(frontend.h, W.ctypes.data,
                                 starts.ctypes.data_as(C.POINTER(C.c_uint64)), len(good), threads, out, nout, status)
    frontend._check(rc)
    for j, i in enumerate(good):
        if status[j]:
            res[i] = BceGpuError(int(status[j]), f"archive {i}: damaged")
        else:
            res[i] = C.string_at(out[j], nout[j])
            lib.bce_host_free(out[j])
    return res


def scan(frontend, data) -> bytes:
    lib = load_library()
    T = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else np.ascontiguousarray(data)
    out = np.zeros(288, dtype=np.uint8)
    frontend._check(lib.bce_scan_buffer(frontend.h, T.ctypes.data, T.size, out.ctypes.data))
    return out.tobytes()
