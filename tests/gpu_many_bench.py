"""Per-file cost of the front end on many small files, and what bce_gpu_compress_many saves.

For each size (4, 16, 64 KiB) and generator (enwik-shaped, markov2-text, mixed-binary), FILES inputs (seeded):
  (a) compress_front + its batches, file after file, on one context and on two (one thread each), coder words;
  (b) compress_front_many (one CTA per input), front end only: the kernel's device time, the call's device time
      with its copies, and the wall clock of the calls;
  (c) host.compress file after file vs host.compress_many, wall clock (archives included).
Before any time is reported, (a) and (b) must emit the same words for the first CHECK files, and (c) the same
archives.  Prints the card and its power limit, one JSON line per configuration.

    python tests/gpu_many_bench.py [--files 10000] [--out results.json]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from bce_b200 import Frontend, host, synth  # noqa: E402
from bce_b200.gpu import EMIT_CODER, EMIT_RAW  # noqa: E402

CHECK = 50


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def front_loop(fe, files):
    fe.set_emit_mode(EMIT_CODER)
    try:
        for d in files:
            fe.compress_front_discard(d)
    finally:
        fe.set_emit_mode(EMIT_RAW)


def many_front(fe, files):
    """compress_many_call until every file is done: (kernel ms, call ms incl. copies, calls)."""
    fe.set_emit_mode(EMIT_CODER)
    kern = total = 0.0
    calls = 0
    try:
        todo = list(range(len(files)))
        while todo:
            out = fe.compress_many_call([files[i] for i in todo])
            st = fe.stats()
            kern += st["ms_cse_total"]
            total += st["ms_total"]
            calls += 1
            todo = [i for j, i in enumerate(todo) if not out[j].done]
    finally:
        fe.set_emit_mode(EMIT_RAW)
    return kern, total, calls


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=10000)
    ap.add_argument("--sizes", default="4096,16384,65536")
    ap.add_argument("--out", default=None, help="also write the rows to this JSON file")
    args = ap.parse_args()
    name = card()
    print("card, power limit:", name, flush=True)
    fe, fe2 = Frontend(0), Frontend(0)
    rows = []
    for size in (int(s) for s in args.sizes.split(",")):
        for gen in ("enwik-shaped", "markov2-text", "mixed-binary"):
            blob = synth.generate(gen, size * args.files, size).tobytes()
            files = [blob[i * size:(i + 1) * size] for i in range(args.files)]
            # same words, same archives, before any timing
            got = fe.compress_front_many(files[:CHECK], EMIT_CODER)
            for d, (off, Cv, streams) in zip(files[:CHECK], got):
                off1, C1, s1 = fe.compress_front_words(d, EMIT_CODER)
                assert (off, Cv) == (off1, C1) and all(np.array_equal(streams[i], s1[i]) for i in range(8)), gen
            assert host.compress_many(fe, files[:CHECK]) == [host.compress(fe, d) for d in files[:CHECK]], gen
            # warm-up of every path; the full set once, so that the calls' buffers have their final size
            front_loop(fe, files[:20])
            front_loop(fe2, files[:20])
            many_front(fe, files)
            many_front(fe, files)
            host.compress_many(fe, files)

            t = time.perf_counter()
            front_loop(fe, files)
            a1 = time.perf_counter() - t
            t = time.perf_counter()
            th = [threading.Thread(target=front_loop, args=(f, files[w::2])) for w, f in enumerate((fe, fe2))]
            for x in th:
                x.start()
            for x in th:
                x.join()
            a2 = time.perf_counter() - t
            t = time.perf_counter()
            kern, call, calls = many_front(fe, files)
            b_wall = time.perf_counter() - t
            t = time.perf_counter()
            for d in files:
                host.compress(fe, d)
            c_loop = time.perf_counter() - t
            t = time.perf_counter()
            host.compress_many(fe, files)
            c_many = time.perf_counter() - t
            mb = size * args.files / 1e6
            row = dict(card=name, size=size, generator=gen, files=args.files,
                       a_front_loop_1ctx_s=a1, a_front_loop_2ctx_s=a2, a_us_per_file_1ctx=a1 / args.files * 1e6,
                       b_many_kernel_ms=kern, b_many_call_ms=call, b_many_wall_s=b_wall, b_calls=calls,
                       b_us_per_file=b_wall / args.files * 1e6,
                       c_compress_loop_s=c_loop, c_compress_many_s=c_many,
                       MBps=dict(a1=mb / a1, a2=mb / a2, b=mb / b_wall, c_loop=mb / c_loop, c_many=mb / c_many))
            print(json.dumps(row), flush=True)
            rows.append(row)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(rows, indent=1))
    fe.close()
    fe2.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
