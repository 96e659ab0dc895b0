"""Per-archive cost of decompressing many small archives, and what bce_decompress_many saves.

For each size (4, 16, 64 KiB) and generator (enwik-shaped, markov2-text, mixed-binary), FILES seeded inputs are
compressed once (host.compress_many), then decompressed three ways, each timed with a host clock around calls that end
in a device synchronise:
  (a) host.decompress(a) per archive           -- `bce -d`: 8 level threads, a device opened per archive, bce_gpu_unbwt
  (b) host.decompress(a, low_memory=True)      -- `bce -ds`: 8 level threads, serial inverse on the host
  (c) host.decompress_many(fe, archives)       -- one archive per host thread, the inverses in bce_gpu_unbwt_many calls
Before any time is reported the three must give identical bytes (and the inputs back).  (c) also reports the kernel's
own time (ms_unbwt_chase of its last call) and the call's device time with its copies.  Prints the card and its power
limit, one JSON line per configuration.

    python tests/gpu_many_decompress_bench.py [--files 1000] [--out results.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from bce_b200 import Frontend, host, synth  # noqa: E402


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=1000)
    ap.add_argument("--sizes", default="4096,16384,65536")
    ap.add_argument("--threads", type=int, default=8)
    ap.add_argument("--out", default=None, help="also write the rows to this JSON file")
    args = ap.parse_args()
    name = card()
    print("card, power limit:", name, "| host threads:", os.cpu_count(), flush=True)
    fe = Frontend(0)
    rows = []
    for size in (int(s) for s in args.sizes.split(",")):
        for gen in ("enwik-shaped", "markov2-text", "mixed-binary"):
            blob = synth.generate(gen, size * args.files, size).tobytes()
            files = [blob[i * size:(i + 1) * size] for i in range(args.files)]
            arcs = host.compress_many(fe, files, threads=args.threads)
            # identical bytes from all three, before any timing (this also warms every path up)
            many = host.decompress_many(fe, arcs, threads=args.threads)
            assert many == files, gen
            assert [host.decompress(a) for a in arcs[:20]] == files[:20], gen
            assert [host.decompress(a, low_memory=True) for a in arcs[:20]] == files[:20], gen

            t = time.perf_counter()
            a_out = [host.decompress(a) for a in arcs]
            ta = time.perf_counter() - t
            t = time.perf_counter()
            b_out = [host.decompress(a, low_memory=True) for a in arcs]
            tb = time.perf_counter() - t
            t = time.perf_counter()
            c_out = host.decompress_many(fe, arcs, threads=args.threads)
            tc = time.perf_counter() - t
            st = fe.stats()
            assert a_out == b_out == c_out == files, gen
            mb = size * args.files / 1e6
            row = dict(card=name, size=size, generator=gen, files=args.files, archive_bytes=sum(map(len, arcs)),
                       a_decompress_s=ta, b_decompress_low_memory_s=tb, c_decompress_many_s=tc,
                       c_last_call_kernel_ms=st["ms_unbwt_chase"], c_last_call_device_ms=st["ms_total"],
                       c_last_call_dicts=st["unbwt_dicts"], c_last_call_serial=st["unbwt_serial"],
                       us_per_file=dict(a=ta / args.files * 1e6, b=tb / args.files * 1e6, c=tc / args.files * 1e6),
                       MBps=dict(a=mb / ta, b=mb / tb, c=mb / tc))
            print(json.dumps(row), flush=True)
            rows.append(row)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(rows, indent=1))
    fe.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
