"""Where decoding many small archives on the device (bce_gpu_decompress_many) beats the host decoders.

bce_decompress_many decodes a group of small archives either on the device (decode loops and inverses in two launches)
or with one host decoder per archive and thread, then the inverses in one bce_gpu_unbwt_many launch.  The
environment variable BCE_HOST_MANY_DEVICE_DECODERS moves the threshold between the two, so both paths run through the
same entry point (host.decompress_many) with the same grouping.  Two tables:
  corpus  FILES archives (300 and 1000) of 4, 16 and 64 KiB from each of three generators;
  calls   calls of 1, 8, 64 and 256 archives of the same sizes -- these set BCE_HOST_MANY_DEVICE_DECODERS.
Before any time is reported both paths must give identical bytes, and the inputs back.  Each time is the median of
REPS runs with a host clock around a call that ends in a device synchronise.  The device path also reports its last
call's kernel times (ms_decoder, ms_unbwt_chase) and its device time with copies (ms_total).  Prints the card and its
power limit, one JSON line per row.

    python tests/gpu_many_device_decode_bench.py [--threads 16] [--out results.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from bce_b200 import Frontend, host, synth  # noqa: E402

GENERATORS = ("enwik-shaped", "markov2-text", "mixed-binary")


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def timed(fe, arcs, threads, device, reps):
    os.environ["BCE_HOST_MANY_DEVICE_DECODERS"] = "1" if device else str(1 << 30)
    times, out = [], None
    for _ in range(reps):
        t = time.perf_counter()
        out = host.decompress_many(fe, arcs, threads=threads)
        times.append(time.perf_counter() - t)
    return statistics.median(times), out, fe.stats()


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="4096,16384,65536")
    ap.add_argument("--corpus", default="300,1000")
    ap.add_argument("--calls", default="1,8,64,256")
    ap.add_argument("--threads", type=int, default=16)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the rows to this JSON file")
    args = ap.parse_args()
    name = card()
    print("card, power limit:", name, "| host threads:", os.cpu_count(), "| decoder threads:", args.threads, flush=True)
    fe = Frontend(0)
    rows = []
    counts = sorted({int(x) for x in args.corpus.split(",")} | {int(x) for x in args.calls.split(",")})
    corpus_counts = {int(x) for x in args.corpus.split(",")}
    for size in (int(s) for s in args.sizes.split(",")):
        for gen in GENERATORS:
            most = max(counts)
            blob = synth.generate(gen, size * most, size).tobytes()
            files = [blob[i * size:(i + 1) * size] for i in range(most)]
            arcs_all = host.compress_many(fe, files, threads=args.threads)
            for k in counts:
                arcs, want = arcs_all[:k], files[:k]
                td, dev, st = timed(fe, arcs, args.threads, True, args.reps)
                th, hst, _ = timed(fe, arcs, args.threads, False, args.reps)
                assert dev == hst == want, (gen, size, k)
                row = dict(card=name, table="corpus" if k in corpus_counts else "calls", size=size, generator=gen,
                           archives=k, device_s=td, host_s=th, speedup=th / td,
                           device_last_call=dict(ms_decoder=st["ms_decoder"], ms_unbwt_chase=st["ms_unbwt_chase"],
                                                 ms_total=st["ms_total"], visits=st["cse_visits"]),
                           us_per_archive=dict(device=td / k * 1e6, host=th / k * 1e6))
                print(json.dumps(row), flush=True)
                rows.append(row)
    os.environ.pop("BCE_HOST_MANY_DEVICE_DECODERS", None)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(dict(card=name, threads=args.threads, rows=rows), indent=1))
    fe.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
