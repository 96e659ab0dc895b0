"""Range coders of many small inputs on the host vs on the device (bce_gpu_compress_many_archives).

For each size (4, 16, 64 KiB) and generator (enwik-shaped, markov2-text, mixed-binary), FILES inputs (seeded), and for
calls of 1, 8, 64 and 256 of those inputs (the crossover that sets BCE_HOST_MANY_DEVICE_CODERS):
  host    one bce_gpu_compress_many call (front end, CODER words to pinned memory), then every input's archive written
          by the host coders (bce_archive_begin / feed_words / finish), one input per thread on THREADS threads -- what
          bce_compress_many does below its threshold
  device  one bce_gpu_compress_many_archives call: front end and coders on the device, the archives to pinned memory
Both are wall clock around calls that end in a device synchronise, archives in host memory, best of REPEAT.  Before
any time is taken the two must give the same archives.  Also reported: the coder kernel's device time (ms_coder), the
front end's (ms_cse_total) and the bytes copied to the host by each path.  Prints the card and its power limit.

    python tests/gpu_many_code_bench.py [--files 1000] [--out results.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from bce_b200 import Frontend, host, synth  # noqa: E402
from bce_b200.gpu import EMIT_CODER, EMIT_RAW, CseWords  # noqa: E402


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def host_path(fe, files, pool):
    """bce_gpu_compress_many + host coders, one input per thread: (archives, D2H bytes, front-end ms)."""
    lib = host.load_library()
    fe.set_emit_mode(EMIT_CODER)
    try:
        out = fe.compress_many_call(files)
    finally:
        fe.set_emit_mode(EMIT_RAW)
    st = fe.stats()
    assert all(out[j].done for j in range(len(files))), "the default arena holds every input"

    def code(j):
        r = out[j]
        w = lib.bce_archive_begin(len(files[j]), r.C, None)
        b = CseWords()
        for s in range(8):
            b.words[s], b.count[s] = r.words[s], r.count[s]
        b.done = 1
        assert lib.bce_archive_feed_words(w, C.byref(b), 1) == 0
        words, nw = C.c_void_p(), C.c_size_t()
        assert lib.bce_archive_finish(w, r.offset, C.byref(words), C.byref(nw)) == 0
        a = C.string_at(words.value, nw.value * 2)
        lib.bce_host_free(words)
        return a

    return list(pool.map(code, range(len(files)))), 4 * st["cse_words"], st["ms_cse_total"]


def device_path(fe, files):
    arcs = fe.compress_many_archives(files)
    assert all(a is not None for a in arcs), "the default arenas hold every input"
    st = fe.stats()
    return arcs, sum(len(a) for a in arcs), st["ms_cse_total"], st["ms_coder"]


def best(fn, repeat):
    t = []
    for _ in range(repeat):
        a = time.perf_counter()
        fn()
        t.append(time.perf_counter() - a)
    return min(t)


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=1000)
    ap.add_argument("--sizes", default="4096,16384,65536")
    ap.add_argument("--calls", default="1,8,64,256")
    ap.add_argument("--threads", type=int, default=16)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the rows to this JSON file")
    args = ap.parse_args()
    name = card()
    print("card, power limit:", name, flush=True)
    fe = Frontend(0)
    pool = ThreadPoolExecutor(args.threads)
    rows = []
    for size in (int(s) for s in args.sizes.split(",")):
        for gen in ("enwik-shaped", "markov2-text", "mixed-binary"):
            blob = synth.generate(gen, size * args.files, size).tobytes()
            files = [blob[i * size:(i + 1) * size] for i in range(args.files)]
            for k in [int(x) for x in args.calls.split(",")] + [args.files]:
                part = files[:k]
                ha, h_d2h, h_front = host_path(fe, part, pool)         # equal archives first (and a warm-up)
                da, d_d2h, d_front, d_coder = device_path(fe, part)
                assert ha == da, (size, gen, k)
                th = best(lambda: host_path(fe, part, pool), args.repeat)
                td = best(lambda: device_path(fe, part), args.repeat)
                _, _, _, d_coder = device_path(fe, part)
                row = dict(card=name, size=size, generator=gen, files=k, threads=args.threads,
                           host_s=th, device_s=td, speedup=th / td, front_kernel_ms=d_front, coder_kernel_ms=d_coder,
                           host_d2h_bytes=h_d2h, device_d2h_bytes=d_d2h)
                print(json.dumps(row), flush=True)
                rows.append(row)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(rows, indent=1))
    pool.shutdown()
    fe.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
