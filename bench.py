#!/usr/bin/env python
"""bench.py -- BWT + CSE compression front end throughput on B200 (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one pass of the hot path (suffix sort/BWT + wavelet matrix + CSE level loop) over
one synthetic input per GPU.  At N = 1 the workload is the configuration BASELINE.json's target
is quoted on, configs[2]: 1 GB (10^9 bytes) of enwik-shaped synthetic text on a single B200
(`--workload enwik-100MB` runs configs[1]).  The working set (48 n bytes of keys, indices, SA
and ranks) exceeds the 126 MB L2 by far, so no L2 flush is needed between steps.
At N > 1 every rank compresses its own 1 GB input of the same generator (seed + rank): replicas
only, weak scaling with the per-GPU work of N = 1, no data-path collective; one small all_gather of
per-rank stats is the only traffic (SURVEY.md 8e).  `--workload batch-128MB` runs the 128 MiB
files of configs[4] instead.

Legs of the default arm:
  value  input resident in HBM when the timed region starts; counts written to HBM.
  e2e    the same through the C-ABI call a user makes, from pinned HOST memory, with the
         emitted counts copied back to pinned host memory inside the timed region.
  roofline     dominant kernel, algorithmic bytes / CUDA-event kernel time vs measured HBM peak.
  cpu_baseline rank 0, N = 1: the UNMODIFIED reference front end (oracle/_ref, built from
               /root/reference/bce.cpp with a recording coder) on a bounded sample.
`--impl reference` times that reference front end alone on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "compress_MBps_bwt_cse"
UNIT = "MB/s"
WORKLOADS = {
    # name: (generator, bytes, seed)
    "markov2-1MB": ("markov2-text", 10**6, 1),
    "enwik-100MB": ("enwik-shaped", 10**8, 2),
    "enwik-1GB": ("enwik-shaped", 10**9, 3),
    "mixed-256MB": ("mixed-binary", 268435456, 4),
    "batch-128MB": ("enwik-shaped", 134217728, 100),
}


def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path
# ---------------------------------------------------------------------------------------------
def reference_front_seconds(sample, threads: int):
    """Unmodified reference: RankFile ctor (rotate + BWT + wavelet) + BCE<tap>::encode (the CSE loop handing
    every count to a coder that only counts the calls: the reference is not charged for storing them), through
    oracle/_ref."""
    from oracle import oracle
    os.environ["OMP_NUM_THREADS"] = str(threads)
    r = oracle.ref_front(sample, want_bwt=False, want_ranks=False, record=False)
    return r["seconds_rankfile"] + r["seconds_encode"], r


def reference_rate(gen, seed, threads: int):
    """Bytes per second of the reference front end on a 4 MiB probe (it gets slower with size: an upper bound)."""
    from bce_b200 import synth
    probe = synth.generate(gen, 4 << 20, seed)
    t, _ = reference_front_seconds(probe, threads)
    return (4 << 20) / max(t, 1e-3)


def cpu_sample_bytes(gen, seed, nbytes: int, budget_s: float, threads: int) -> int:
    """The prefix of the workload the cpu_baseline leg times: about budget_s seconds of reference work."""
    return int(max(1 << 20, min(nbytes, 64 << 20, reference_rate(gen, seed, threads) * budget_s)))


NATIVE_NOTE = ("libbce_synth.so is the synthetic input generator only; the reference arm's compute is "
               "oracle/_ref/libbce_ref_tap.so = the unmodified /root/reference/bce.cpp")


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return 0
    from bce_b200 import synth
    from oracle import oracle
    gen, nbytes, seed = WORKLOADS[args.workload]
    if not oracle.have_ref():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built (needs /root/reference at build time)"}))
        return 0
    cores = os.cpu_count() or 1
    threads = min(8, cores)                              # the reference forks over 8 levels at most (bce.cpp:1250)
    # The reference gets slower per byte as the input grows (a 32 MB prefix of the 1 GB workload runs 15 % faster per
    # byte than a 64 MB one), so a prefix is not the configuration.  When one pass over the WHOLE workload fits the
    # budget it is timed exactly once (steps_run = 1, no warm-up pass: nothing to warm on the host); otherwise the
    # largest prefix that fits, and `config.sample_bytes` says so in both arms.
    est_full = 1.5 * nbytes / reference_rate(gen, seed, threads)      # the probe's rate is an upper bound: allow for the slow-down with size
    full = est_full <= args.ref_budget_s
    if full:
        sample_bytes, steps_run, warm_run = nbytes, 1, 0
    else:
        steps_run, warm_run = max(1, args.steps), min(1, args.warmup)
        sample_bytes = int(max(1 << 20, min(nbytes, nbytes * args.ref_budget_s / est_full / (steps_run + warm_run))))
    sample = synth.generate(gen, sample_bytes, seed)
    for _ in range(warm_run):
        reference_front_seconds(sample, threads)
    times = []
    r = None
    for _ in range(steps_run):
        t, r = reference_front_seconds(sample, threads)
        times.append(t)
    total = sum(times)
    value = sample_bytes * steps_run / total / 1e6
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "steps_run": steps_run, "warmup_run": warm_run,
        "ms_per_step": 1e3 * total / steps_run,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32",
        "data": "synthetic", "gpu_launches": 0,
        "config": {"workload": args.workload, "generator": gen, "bytes_per_gpu": nbytes, "seed": seed,
                   "sample_bytes": sample_bytes, "whole_workload": full},
        "stage_s": {"rankfile (rotate + BWT + wavelet)": r["seconds_rankfile"], "encode (CSE loop, counting coder)": r["seconds_encode"]},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "reference",
                         "sample": (f"the whole {args.workload} workload ({nbytes} bytes), one pass" if full else
                                    f"first {sample_bytes} bytes of {args.workload}") +
                                   f"; unmodified bce.cpp front end (rotate + BWT + wavelet + CSE loop, counts handed to a "
                                   f"coder that only counts them); BWT stage is the oracle's SA-IS stand-in for "
                                   f"libdivsufsort; OMP_NUM_THREADS={threads} of {cores} cores"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "native_note": NATIVE_NOTE,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def algorithmic_bytes(st: dict, executed: bool = False) -> dict:
    """SURVEY.md 8d.  P_r is the number of 8-bit digits the keys of round r have to be ordered by (what an LSD
    radix sort runs; sort_passes).  Rounds >= 1 are sorted tile by tile without radix passes over the working
    set (csrc/local_sort.cuh); `executed` prices those rounds at what was actually moved instead: one read and
    one write of the (key, idx) pairs (24 B per element) plus the radix passes of the fall-back elements."""
    n = st["n"]
    if executed:
        rp = st.get("sort_radix_passes") or st["sort_passes"]
        stage_a = 19 * n + sum((44 + 24 * (p if p else 1)) * m for m, p in zip(st["sort_m"], rp))
        stage_a += 24 * 8 * st.get("sort_fallback_elems", 0)
    else:
        stage_a = 19 * n + sum((44 + 24 * p) * m for m, p in zip(st["sort_m"], st["sort_passes"]))
    # emission counted at the bytes actually written: 4 B per packed word (SURVEY.md 8d assumes 20 B raw counts)
    stage_b = 19 * n + 48 * st["cse_visits"] + 4 * st["cse_words"]
    return {"stage_a": stage_a, "stage_b": stage_b, "total": stage_a + stage_b}


def run_batch_workload(args, rank: int, world: int, local_rank: int):
    """configs[4]: 64 files of 128 MiB (the enwik-shaped generator, seeds 100..163), one archive per file, on N GPUs.
    A step is the whole batch through bce_b200.batch.compress_files: workers pull files from a shared queue, read
    them, run the GPU front end + host range coders, write <file>.bce.  Untimed: generating the files.  `value` is
    the GPU-stage throughput (all bytes / the busiest rank's summed front-end time), `e2e` the true `bce -c` rate
    of the batch (wall clock of the slowest rank, file read and archive write included)."""
    import hashlib
    import shutil
    import tempfile

    import torch
    import torch.distributed as dist

    from bce_b200 import batch, synth
    torch.cuda.set_device(local_rank)
    gen, nbytes, seed0 = WORKLOADS["batch-128MB"]
    nfiles = args.files
    root = Path(os.environ.get("BCE_BENCH_TMP", "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir())) / "bce_batch_bench"
    if rank == 0:
        shutil.rmtree(root, ignore_errors=True)
        (root / "in").mkdir(parents=True)
    if world > 1:
        dist.barrier()
    for i in range(rank, nfiles, world):                       # untimed: synthetic inputs
        synth.generate(gen, nbytes, seed0 + i).tofile(root / "in" / f"file{i:02d}")
    if world > 1:
        dist.barrier()
    paths = [str(root / "in" / f"file{i:02d}") for i in range(nfiles)]
    # files in flight per GPU: a file's front end takes a tenth of the time its 8 coder threads do
    in_flight = args.in_flight or max(1, min(2, (os.cpu_count() or 8) // (8 * world)))
    fns = [batch.make_gpu_compressor(local_rank) for _ in range(in_flight)]
    for f in fns:
        f(synth.generate(gen, 1 << 22, 1), None)                # warm-up: context, buffers, kernels
    sampler = ClockSampler(local_rank)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler.start()
    t0 = time.perf_counter()
    res = batch.compress_files(paths, str(root / "out"), fns, device="cuda" if world > 1 else "cpu")
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    launches = sum(f.gpu_launches for f in fns)
    if world > 1:
        t = torch.tensor([wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall = float(t.item())
        t = torch.tensor([launches], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        launches = int(t.item())
    if rank == 0:
        tot = res.total
        golden = {}
        try:
            vec = json.loads((ROOT / "tests" / "golden" / "big_vectors.json").read_text())["vectors"]
            for name, idx in (("batch-128MB-seed100", 0), ("batch-128MB-seed163", 63)):
                f = root / "out" / f"file{idx:02d}.bce"
                if name in vec and f.exists():
                    golden[name] = hashlib.sha256(f.read_bytes()).hexdigest() == vec[name]["archive_sha256"]
        except Exception as e:                                   # noqa: BLE001
            golden = {"error": str(e)}
        gpu_s = tot.gpu_ms / 1e3
        line = {
            "metric": METRIC, "value": tot.bytes_in / gpu_s / 1e6 if gpu_s else None, "unit": UNIT, "n_gpus": world,
            "steps": 1, "warmup": 1, "ms_per_step": wall * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8/u32", "data": "synthetic",
            "config": {"workload": "batch-128MB", "generator": gen, "files": nfiles, "bytes_per_file": nbytes,
                       "seeds": [seed0, seed0 + nfiles - 1], "files_in_flight_per_gpu": in_flight,
                       "parallelism": f"replicas x{world}, shared file queue",
                       "l2": "every file's working set exceeds L2; no flush"},
            "e2e": {"value": tot.bytes_in / wall / 1e6, "unit": UNIT, "what": "files read, compressed (GPU front end + host "
                    "coders, 8 threads per in-flight file) and written as .bce; wall clock of the slowest rank",
                    "h2d_bytes_per_step": tot.bytes_in, "d2h_bytes_per_step": None, "archives_per_s": tot.inputs / wall},
            "batch": {"files_ok": tot.inputs, "files_failed": tot.failed, "bytes_in": tot.bytes_in, "bytes_out": tot.bytes_out,
                      "wall_s": wall, "gpu_s_busiest_rank": gpu_s,
                      "per_rank": [vars(r) for r in res.per_rank],
                      "files_per_rank": [sum(1 for f in res.files if f.rank == r) for r in range(world)],
                      "archives_equal_reference": golden, "host_cores": os.cpu_count()},
            "gpu_launches": launches, "clocks": clocks, "native_note": NATIVE_NOTE,
        }
        print(json.dumps(line))
        shutil.rmtree(root, ignore_errors=True)
    for f in fns:
        f.frontend.close()
    return 0


class WordSample:
    """A fixed sample of the coder words of all 8 streams of one input, taken batch by batch as the C ABI hands them
    back (20 bits each, bce_gpu_cse_next_words20): in every block of `stride` consecutive words of a stream the word
    at a seeded offset, at most BLOCKS words per stream (4 MiB in float32).  Streams differ in length by orders of
    magnitude (on text the top bit level emits nothing), so each stream's stride follows from its word count in
    `counts`, taken by a previous pass over the same input (WordSample() only counts); the same input therefore
    gives the same positions."""
    BLOCKS = 1 << 20

    def __init__(self, counts=(0,) * 8, seed: int = 1):
        import numpy as np
        rng = np.random.default_rng(seed)
        self.expect = list(counts)
        self.pos = []
        for c in self.expect:
            stride = max(1, -(-c // self.BLOCKS))
            blocks = -(-c // stride)
            p = np.arange(blocks, dtype=np.int64) * stride + rng.integers(0, stride, blocks)
            self.pos.append(p[p < c])
        self.count = [0] * 8
        self.parts = [[] for _ in range(8)]
        self.C = None

    def __call__(self, Cv, batch):
        import ctypes

        import numpy as np
        self.C = [int(x) for x in Cv]
        for i in range(8):
            cnt = int(batch.count[i])
            if not cnt:
                continue
            lo, hi = np.searchsorted(self.pos[i], [self.count[i], self.count[i] + cnt])
            j = self.pos[i][lo:hi] - self.count[i]
            if j.size:
                raw = (ctypes.c_uint8 * (5 * ((cnt + 1) // 2))).from_address(ctypes.addressof(batch.bytes[i].contents))
                o = 5 * (j // 2)
                b = [np.ctypeslib.as_array(raw)[o + k].astype(np.uint32) for k in range(5)]     # only the sampled words
                even = b[0] | (b[1] << 8) | ((b[2] & 15) << 16)
                odd = (b[2] >> 4) | (b[3] << 4) | (b[4] << 12)
                self.parts[i].append(np.where(j % 2 == 0, even, odd))
            self.count[i] += cnt

    def arrays(self) -> dict:
        """C[8], words per stream, sampled words per stream, and the samples of streams 0..7 in one array."""
        import numpy as np
        if self.count != self.expect:
            raise RuntimeError(f"words per stream {self.count} differ from the counting pass {self.expect}")
        parts = [np.concatenate(p) if p else np.zeros(0, dtype=np.uint32) for p in self.parts]
        return {"C": np.array(self.C, dtype=np.float64), "stream_words": np.array(self.count, dtype=np.float64),
                "stream_samples": np.array([p.size for p in parts], dtype=np.float64),
                "words_sample": np.concatenate(parts).astype(np.float32)}


def dump_outputs(dir_: str, arrays: dict):
    import numpy as np
    out = Path(dir_)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a)


def run_ours(args, rank: int, world: int, local_rank: int):
    import numpy as np
    import torch
    import torch.distributed as dist

    from bce_b200 import Frontend, batch, host, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    gen, nbytes, seed = WORKLOADS[args.workload]
    if args.bytes:
        nbytes = args.bytes
    my_seed = seed + rank                                  # one independent file per GPU
    data = synth.generate(gen, nbytes, my_seed)
    pinned = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    pinned.numpy()[:] = data
    host_in = pinned.numpy()

    fe = Frontend(local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def maxreduce(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- value leg: device resident ----------------------------------------------------------
    from bce_b200.gpu import EMIT_CODER
    fe.set_emit_mode(EMIT_CODER)          # what `bce -c` consumes: coder-ready 4-byte words
    fe.stage_input(host_in)
    for _ in range(args.warmup):
        fe.front_resident()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    dev_ms, stats_list = 0.0, []
    # the working set (48 n bytes of keys, indices, SA, ranks) exceeds the 126 MB L2 from n = 3 MB on; smaller
    # inputs get the L2 flushed between steps (a 512 MB buffer written on the device, outside the timed events)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda") if 48 * nbytes < (256 << 20) else None
    for _ in range(args.steps):
        if flush is not None:
            flush.fill_(1)
            torch.cuda.synchronize()
        resident = fe.front_resident()
        st = fe.stats()
        dev_ms += st["ms_total"]
        stats_list.append(st)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop()
    dev_ms = maxreduce(dev_ms)
    wall_ms = maxreduce(wall_ms)
    st = stats_list[-1]
    value = world * nbytes * args.steps / (dev_ms / 1e3) / 1e6

    # ---- e2e leg: host buffers through the C ABI -----------------------------------------------
    # Files in flight per GPU: as bce_b200.batch runs a GPU (several contexts, one file each), the copies of one
    # file cross PCIe while the kernels of the other run.  Every step is still one whole file: upload from pinned
    # memory, front end, all batches of words down to pinned memory.  The resident context is closed first: its
    # emission buffers hold all words of a file (~100 GB at 1 GB).
    in_flight = max(1, args.e2e_in_flight)
    ctx_limit = int(0.36 * torch.cuda.get_device_properties(local_rank).total_memory)
    if in_flight > 1 and 60 * nbytes > ctx_limit:
        in_flight = 1                                      # two working sets (48 n bytes of sort buffers each) would not fit
    fe.close()
    fes = [Frontend(local_rank) for _ in range(in_flight)]
    for f in fes:
        f.set_emit_mode(EMIT_CODER)
        if in_flight > 1:
            f.set_scratch_limit(ctx_limit)
        for _ in range(max(2, args.warmup // 2)):         # both pinned batch buffers get allocated here
            f.compress_front_discard(host_in, words20=True)
    fe = fes[0]
    shares = [args.steps // in_flight + (1 if i < args.steps % in_flight else 0) for i in range(in_flight)]
    counts_of = [0] * in_flight
    e2e_offset = None
    # --dump-outputs: an untimed pass counts the words of every stream; the last step of the first context then
    # hands its batches to a sampler (host work in that step)
    sample = None
    if args.dump_outputs and rank == 0:
        probe = WordSample()
        fes[0].compress_front_discard(host_in, words20=True, on_batch=probe)
        sample = WordSample(probe.count)

    def e2e_loop(i):
        nonlocal e2e_offset
        for k in range(shares[i]):
            last = k + 1 == shares[i]
            # a pipeline of inputs: the next step's upload (the same pinned buffer here) is started as soon as this step's
            # BWT exists and runs beside its level loop (bce_gpu_prefetch_input); the first step uploads in the open
            off, counts_of[i] = fes[i].compress_front_discard(host_in, words20=True,
                                                              prefetch_next=None if last else host_in,
                                                              on_batch=sample if i == 0 and last else None)
            if i == 0:
                e2e_offset = off

    barrier()
    t0 = time.perf_counter()
    if in_flight == 1:
        e2e_loop(0)
    else:
        import threading
        pool = [threading.Thread(target=e2e_loop, args=(i,)) for i in range(in_flight)]
        for t in pool:
            t.start()
        for t in pool:
            t.join()
    counts = counts_of[0]
    my_e2e_ms = (time.perf_counter() - t0) * 1e3            # this rank alone, before it waits for the others
    barrier()
    e2e_ms = maxreduce((time.perf_counter() - t0) * 1e3)
    e2e_value = world * nbytes * args.steps / (e2e_ms / 1e3) / 1e6
    st_e2e = fe.stats()
    for f in fes[1:]:
        f.close()
    fe.set_scratch_limit(0)
    # every rank's own e2e numbers (the job's e2e is the slowest rank's): where the time of a slow rank goes
    my_e2e = {"rank": rank, "e2e_ms_per_step": my_e2e_ms / args.steps, "ms_h2d": st_e2e["ms_h2d"], "ms_d2h": st_e2e["ms_d2h"],
              "ms_bwt_total": st_e2e["ms_bwt_total"], "ms_cse_total": st_e2e["ms_cse_total"],
              "d2h_GBps": (int(counts) * 2.5 / 1e9) / (st_e2e["ms_d2h"] / 1e3) if st_e2e["ms_d2h"] > 0 else None,
              "h2d_GBps": (nbytes / 1e9) / (st_e2e["ms_h2d"] / 1e3) if st_e2e["ms_h2d"] > 0 else None}
    if world > 1:
        e2e_ranks = [None] * world
        dist.all_gather_object(e2e_ranks, my_e2e)
    else:
        e2e_ranks = [my_e2e]

    if sample is not None:
        # what the last timed step of each leg handed its caller: the resident leg (offset, words emitted to HBM);
        # the host-buffer leg offset, C[8], words per stream and the sample of the words themselves
        dump_outputs(args.dump_outputs, {"resident_offset": np.array([resident[0]], dtype=np.float64),
                                         "resident_words": np.array([resident[1]], dtype=np.float64),
                                         "offset": np.array([e2e_offset], dtype=np.float64), **sample.arrays()})

    # ---- `bce -c` as a user runs it: front end + host range coders, archive in memory (rank 0) --------------
    fe.set_emit_mode(0)
    e2e_cli = None
    if rank == 0 and not args.no_cli:
        t0 = time.perf_counter()
        arc = host.compress(fe, host_in, threads=8)
        cli_s = time.perf_counter() - t0
        e2e_cli = {"seconds": cli_s, "MBps": nbytes / cli_s / 1e6, "archive_bytes": len(arc), "coder_threads": 8,
                   "host_cores": os.cpu_count(), "what": "bce_compress_buffer: H2D + front end + host range coders "
                   "(one thread per stream) + archive assembly, one pass, not in the timed region of `value`"}
        if args.workload == "mixed-256MB":                 # configs[3]: bce -s, then bce -c with the config it wrote
            t0 = time.perf_counter()
            cfg = host.scan(fe, host_in)
            scan_s = time.perf_counter() - t0
            t0 = time.perf_counter()
            arc2 = host.compress(fe, host_in, cfg=cfg, threads=8)
            e2e_cli.update(scan_seconds=scan_s, scan_MBps=nbytes / scan_s / 1e6,
                           compress_with_config_seconds=time.perf_counter() - t0, archive_with_config_bytes=len(arc2))
    fe.set_emit_mode(EMIT_CODER)

    # ---- roofline of the dominant kernel ---------------------------------------------------------
    peak, peak_src = measured_peak_gbs()
    ab = algorithmic_bytes(st)
    abx = algorithmic_bytes(st, executed=True)
    radix_ms = st["ms_radix_kernel"] or st["ms_radix"]
    cse_ms = st["ms_cse"]
    if radix_ms >= cse_ms:
        k_name = "radix_onesweep_kernel"
        k_launches = max(1, st["radix_launches"])
        k_bytes = 24.0 * st["radix_elems"] / k_launches
        k_ms = radix_ms / k_launches
        note = "sum of CUDA-event pairs around every radix_onesweep_kernel launch of the step"
    else:
        k_name = "cse_slots_kernel + cse_wide_kernel + cse_narrow_kernel (level loop)"
        k_launches = max(1, st["cse_launches"])
        k_bytes = (48.0 * st["cse_visits"] + 4.0 * st["cse_words"]) / k_launches
        k_ms = cse_ms / k_launches
        note = "one launch runs all rounds of the level loop"
    achieved = k_bytes / (k_ms / 1e3) / 1e9
    traffic, traffic_src = None, None
    try:                                   # measured DRAM bytes per algorithmic byte (ncu), see profiles/r2_traffic.json
        tj = json.loads((Path(__file__).resolve().parent / "profiles" / "r2_traffic.json").read_text())
        ent = tj["radix_onesweep_kernel" if radix_ms >= cse_ms else "cse_level_loop"]
        traffic, traffic_src = ent["ratio"] * k_bytes, f"{ent['ratio']} x algorithmic bytes of this launch; " + ent["source"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": k_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src, "launches_per_step": k_launches,
                "ms_per_launch": k_ms, "note": note,
                "whole_path": {"algorithmic_bytes": ab["total"], "GBps": ab["total"] / (st["ms_total"] / 1e3) / 1e9,
                               "frac": ab["total"] / (st["ms_total"] / 1e3) / 1e9 / peak,
                               "stage_a_bytes": ab["stage_a"], "stage_b_bytes": ab["stage_b"],
                               "note": "SURVEY.md 8d formula, P_r = 8-bit digits of the round's keys"},
                "whole_path_executed": {"algorithmic_bytes": abx["total"],
                                        "frac": abx["total"] / (st["ms_total"] / 1e3) / 1e9 / peak,
                                        "note": "rounds sorted tile by tile (no radix passes over the working set) priced "
                                                "at one read + one write of their pairs plus the fall-back radix passes"}}

    gathered = batch.gather_stats(batch.RankStats(args.steps, nbytes * args.steps, 0, st["cse_words"], dev_ms, wall_ms),
                                  device="cuda" if world > 1 else "cpu")

    # ---- cpu baseline (rank 0, N = 1 only) ---------------------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle
        if oracle.have_ref():
            cores = os.cpu_count() or 1
            threads = min(8, cores)
            sample_bytes = cpu_sample_bytes(gen, seed, nbytes, 12.0, threads)
            sample = synth.generate(gen, sample_bytes, seed)
            t, r = reference_front_seconds(sample, threads)
            cpu_baseline = {"value": sample_bytes / t / 1e6, "unit": UNIT, "cores": threads, "kind": "reference",
                            "sample": f"first {sample_bytes} bytes of {args.workload}: unmodified bce.cpp front end via "
                                      f"oracle/_ref (RankFile {r['seconds_rankfile']:.2f} s incl. SA-IS stand-in for "
                                      f"libdivsufsort, CSE loop {r['seconds_encode']:.2f} s), OMP_NUM_THREADS={threads}"}
        else:
            cpu_baseline = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "oracle/_ref not built"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32", "data": "synthetic",
            "config": {"workload": args.workload, "generator": gen, "bytes_per_gpu": nbytes, "seed": seed,
                       "sample_bytes": nbytes, "whole_workload": True,
                       "l2": "working set (48 n bytes of keys, indices, SA, ranks) exceeds L2; no flush" if flush is None
                             else "512 MB written on the device between timed steps (L2 flush)",
                       "parallelism": f"replicas x{world} (one input per GPU)"},
            "wall_ms_per_step": wall_ms / args.steps,
            "stage_ms": {k: st[k] for k in ("ms_pack", "ms_radix", "ms_rerank", "ms_rekey", "ms_bwt_gather",
                                            "ms_wavelet", "ms_cse", "ms_bwt_total", "ms_cse_total")},
            "counters": {"sort_rounds": st["sort_rounds"], "sort_m": st["sort_m"], "sort_passes": st["sort_passes"],
                         "sort_radix_passes": st.get("sort_radix_passes"), "sort_local_elems": st.get("sort_local_elems"),
                         "sort_fallback_elems": st.get("sort_fallback_elems"),
                         "visits": st["cse_visits"], "emitted_words": st["cse_words"], "cse_rounds": st["cse_rounds"],
                         "peak_frontier": st["cse_peak_frontier"]},
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": nbytes,
                    "d2h_bytes_per_step": (int(counts) * 5 + 1) // 2 + 64,
                    "emission": "BCE_EMIT_CODER words, 20 bits each (bce_gpu_cse_next_words20)",
                    "files_in_flight_per_gpu": in_flight,
                    "in_flight": "contexts per GPU, one whole file (upload, front end, all batches down) per step each, as "
                                 "bce_b200.batch runs a GPU: one file's copies cross PCIe under the other's kernels",
                    "h2d": "every step uploads its input from pinned host memory inside the timed region; from the second step "
                           "on the upload is started when the previous step's BWT exists and overlaps its level loop "
                           "(bce_gpu_prefetch_input)", "ms_per_step": e2e_ms / args.steps,
                    "ms_h2d": st_e2e["ms_h2d"], "ms_d2h": st_e2e["ms_d2h"],
                    "ms_bwt_total": st_e2e["ms_bwt_total"], "ms_cse_total": st_e2e["ms_cse_total"],
                    "cse_launches": st_e2e["cse_launches"],
                    "per_rank": e2e_ranks,
                    "aggregate_d2h_GBps_over_the_step": world * int(counts) * 2.5 / 1e9 / (e2e_ms / args.steps / 1e3),
                    "note": "ms_d2h is copy time on the copy stream; it runs under the level-loop kernels of the next "
                            "batch, so the step is max(kernels, copies) per batch, not their sum"},
            "e2e_cli": e2e_cli,
            "native_note": NATIVE_NOTE,
            "gpu_launches": int(sum(s["gpu_launches"] for s in stats_list)),
            "clocks": clocks,
            "per_rank": [vars(g) for g in gathered],
        }
        print(json.dumps(line))
    fe.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--bytes", type=int, default=0, help="override the input size (debugging)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--files", type=int, default=64, help="--workload batch-128MB: files in the batch (0 = time one "
                    "128 MiB input per GPU like the other workloads)")
    ap.add_argument("--in-flight", type=int, default=0, help="--workload batch-128MB: files in flight per GPU (0 = by host cores)")
    ap.add_argument("--e2e-in-flight", type=int, default=1,
                    help="e2e leg: files in flight per GPU (contexts). Measured with 2: 290 instead of 295 ms per 1 GB file on one GPU, "
                         "no change on eight (the copies are bound by the two PCIe switches' uplinks), hence 1")
    ap.add_argument("--no-cli", action="store_true", help="skip the `bce -c` wall-time leg (host coders)")
    ap.add_argument("--ref-budget-s", type=float, default=420.0,
                    help="--impl reference: seconds one run may take; the whole workload is timed once when it fits")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write what the last one returned as DIR/<name>.npy (float32 / float64, "
                         "under 64 MB; the coder words as a fixed sample, see WordSample), to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload is None:
        # weak scaling: every GPU compresses its own 1 GB input (seed + rank), the configuration the metric is
        # quoted on, at every N -- so that the per-N values are comparable.  BASELINE's batch configuration
        # (128 MiB files) is `--workload batch-128MB`.
        args.workload = "enwik-1GB"
    if args.dump_outputs and (args.impl == "reference" or (args.workload == "batch-128MB" and args.files > 0)):
        ap.error("--dump-outputs needs the single-input arm of --impl ours (with --workload batch-128MB: --files 0)")

    if args.impl == "reference":
        return run_reference(args, rank, world)

    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.workload == "batch-128MB" and args.files > 0:
            return run_batch_workload(args, rank, world, local_rank)
        return run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()


if __name__ == "__main__":
    sys.exit(main())
