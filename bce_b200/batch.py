"""Batch mode: independent files sharded over the GPUs of one node, one archive per file
(BASELINE configs[4]; the reference's per-file driver is main, bce.cpp:1403-1427).

The path does not shard inside an input (suffix order is global, SURVEY.md 8e), so multi-GPU
means replicas: one worker process per GPU (torchrun), every worker pulls the next file from a
shared queue -- an atomic counter in the process group's rendezvous store -- compresses it on its
GPU (front end + host range coders), writes `<out>/<name>.bce`, records a failure and goes on.
Nothing but a small stats vector and the per-file manifest crosses between ranks (one all_gather at
the end; NCCL on GPUs, gloo in the CPU tests).

    torchrun --nproc-per-node 8 -m bce_b200.batch --out DIR file1 file2 ...
    torchrun --nproc-per-node 8 -m bce_b200.batch --decompress --out DIR file1.bce file2.bce ...
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from dataclasses import asdict, dataclass, field
from pathlib import Path
from typing import Callable, Optional, Sequence

import torch
import torch.distributed as dist


@dataclass
class RankStats:
    inputs: int = 0
    bytes_in: int = 0
    bytes_out: int = 0
    counts: int = 0
    gpu_ms: float = 0.0
    wall_ms: float = 0.0
    failed: int = 0

    def as_tensor(self, device) -> torch.Tensor:
        return torch.tensor([self.inputs, self.bytes_in, self.bytes_out, self.counts, self.gpu_ms, self.wall_ms, self.failed],
                            dtype=torch.float64, device=device)

    @staticmethod
    def from_tensor(t: torch.Tensor) -> "RankStats":
        v = t.tolist()
        return RankStats(int(v[0]), int(v[1]), int(v[2]), int(v[3]), float(v[4]), float(v[5]), int(v[6]))


@dataclass
class FileResult:
    index: int
    path: str
    rank: int
    ok: bool
    bytes_in: int = 0
    bytes_out: int = 0
    archive: str = ""
    gpu_ms: float = 0.0
    wall_ms: float = 0.0
    error: str = ""


@dataclass
class BatchResult:
    per_rank: list = field(default_factory=list)
    outputs: dict = field(default_factory=dict)      # index -> whatever `work` returned (this rank only)
    files: list = field(default_factory=list)        # FileResult of every file, all ranks, by index (compress_files)

    @property
    def total(self) -> RankStats:
        t = RankStats()
        for r in self.per_rank:
            t.inputs += r.inputs
            t.bytes_in += r.bytes_in
            t.bytes_out += r.bytes_out
            t.counts += r.counts
            t.failed += r.failed
            t.gpu_ms = max(t.gpu_ms, r.gpu_ms)        # ranks run concurrently: the job takes the max
            t.wall_ms = max(t.wall_ms, r.wall_ms)
        return t


def _dist_on() -> bool:
    return dist.is_available() and dist.is_initialized()


def shard(num_inputs: int, rank: int, world: int) -> list:
    """Indices of the inputs rank `rank` processes under a static split (round robin: equal counts +-1)."""
    return list(range(rank, num_inputs, world))


class WorkQueue:
    """Shared queue of input indices: every pull is one atomic add on the process group's store, so a rank that
    finishes early takes the next file instead of idling (files differ in size and in coder time)."""

    def __init__(self, num_inputs: int, name: str = "bce_batch_next"):
        self.n = num_inputs
        self.key = name
        self.store = None
        self.local = 0
        if _dist_on():
            from torch.distributed import distributed_c10d as c10d
            self.store = c10d._get_default_store()

    def pull(self) -> Optional[int]:
        if self.store is not None:
            i = int(self.store.add(self.key, 1)) - 1
        else:
            i = self.local
            self.local += 1
        return i if i < self.n else None


def gather_stats(local: RankStats, device="cpu") -> list:
    """All ranks learn every rank's stats (the only collective on this path)."""
    if not _dist_on():
        return [local]
    world = dist.get_world_size()
    mine = local.as_tensor(device)
    out = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(out, mine)
    return [RankStats.from_tensor(t.cpu()) for t in out]


def run_batch(num_inputs: int, work: Callable[..., tuple], device="cpu", dynamic: bool = False,
              workers: int = 1) -> BatchResult:
    """`work(i)` processes input i on this rank's GPU and returns
    (bytes_in, bytes_out, counts, gpu_ms, wall_ms, output).  dynamic: pull indices from the shared queue
    instead of the static round-robin split.  An exception in `work` is that input's failure, not the batch's.
    workers > 1: that many threads of this rank pull from the queue, `work(i, w)` gets the worker's number (the GPU
    front end of a file takes a tenth of the time its eight host coder threads do: two files in flight per GPU keep
    sixteen cores busy instead of eight)."""
    import threading
    rank = dist.get_rank() if _dist_on() else 0
    world = dist.get_world_size() if _dist_on() else 1
    local = RankStats()
    res = BatchResult()
    queue = WorkQueue(num_inputs) if dynamic else None
    static = iter(shard(num_inputs, rank, world))
    lock = threading.Lock()

    def loop(w):
        while True:
            with lock:
                i = queue.pull() if queue else next(static, None)
            if i is None:
                break
            try:
                r = work(i, w) if workers > 1 else work(i)
            except Exception as e:                  # noqa: BLE001 -- recorded, the batch goes on
                with lock:
                    local.failed += 1
                    res.outputs[i] = e
                continue
            with lock:
                # a list: work item i was several inputs, one result or exception each
                for x in (r if isinstance(r, list) else [r]):
                    if isinstance(x, Exception):
                        local.failed += 1
                        continue
                    b_in, b_out, counts, gpu_ms, wall_ms, _ = x
                    local.inputs += 1
                    local.bytes_in += b_in
                    local.bytes_out += b_out
                    local.counts += counts
                    local.gpu_ms += gpu_ms
                    local.wall_ms += wall_ms
                res.outputs[i] = [x[5] if isinstance(x, tuple) else x for x in r] if isinstance(r, list) else r[5]

    if workers > 1:
        pool = [threading.Thread(target=loop, args=(w,)) for w in range(workers)]
        for t in pool:
            t.start()
        for t in pool:
            t.join()
    else:
        loop(0)
    res.per_rank = gather_stats(local, device)
    return res


MANY_RUN_BYTES = 64 << 20          # bytes of small files one queue pull claims


def small_file_runs(sizes: Sequence[int], max_n: int, budget: int = MANY_RUN_BYTES) -> list:
    """Work items of compress_files: runs of consecutive files of 1 .. max_n bytes (a size from stat; -1 = stat
    failed) up to `budget` bytes each, every other file alone.  Returns (file indices, is_run) pairs."""
    units, run, run_bytes = [], [], 0
    for i, sz in enumerate(sizes):
        small = 1 <= sz <= max_n
        if run and (not small or run_bytes + sz > budget):
            units.append((run, True))
            run, run_bytes = [], 0
        if small:
            run.append(i)
            run_bytes += sz
        else:
            units.append(([i], False))
    if run:
        units.append((run, True))
    return units


def _files_batch(paths: Sequence[str], out_dir: str, fns: list, read, single, many, dst_name, run_max: int,
                 device) -> BatchResult:
    """The file loop behind compress_files / decompress_files.  read(path) -> the file's contents (raises for a file
    that cannot be processed); single(fn, data) -> (bytes, gpu_ms); dst_name(path) -> the output's name.  If `many` is
    given -- many(fn, datas) -> (one result or exception per data, gpu_ms) -- one queue pull claims a run of consecutive
    files of 1 .. run_max bytes (sizes from stat, before the queue starts) and processes it with one `many` call; other
    files go alone through `single`."""
    rank = dist.get_rank() if _dist_on() else 0
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    mine = []
    if many is not None:
        def size(p):
            try:
                return os.stat(p).st_size
            except OSError:
                return -1
        units = small_file_runs([size(p) for p in paths], run_max)
    else:
        units = [([i], False) for i in range(len(paths))]

    def work(i, w=0):
        p = Path(paths[i])
        t0 = time.perf_counter()
        fr = FileResult(index=i, path=str(p), rank=rank, ok=False)
        mine.append(fr)
        try:
            data = read(p)
            res, gpu_ms = single(fns[w], data)
            dst = out / dst_name(p)
            dst.write_bytes(res)                                         # bce.cpp:1424-1427
        except Exception as e:                                           # noqa: BLE001
            fr.error = f"{type(e).__name__}: {e}"
            fr.wall_ms = (time.perf_counter() - t0) * 1e3
            raise
        fr.ok, fr.bytes_in, fr.bytes_out, fr.archive = True, len(data), len(res), str(dst)
        fr.gpu_ms, fr.wall_ms = float(gpu_ms), (time.perf_counter() - t0) * 1e3
        return fr.bytes_in, fr.bytes_out, 0, fr.gpu_ms, fr.wall_ms, str(dst)

    def work_run(idx, w):
        """A run of small files through one `many` call; a file that cannot be read or processed fails alone."""
        t0 = time.perf_counter()
        frs = [FileResult(index=i, path=str(Path(paths[i])), rank=rank, ok=False) for i in idx]
        mine.extend(frs)
        results, datas, live = [None] * len(idx), [], []
        for j, i in enumerate(idx):
            try:
                data = read(Path(paths[i]))
                if len(data) > run_max:
                    raise ValueError(f"file grew above {run_max} bytes while the batch ran")
                datas.append(data)
                live.append(j)
            except Exception as e:                                       # noqa: BLE001
                frs[j].error = f"{type(e).__name__}: {e}"
                results[j] = e
        if live:
            try:
                outs, gpu_ms = many(fns[w], datas)
                if len(outs) != len(live):
                    raise RuntimeError(f"{len(outs)} results for {len(live)} files")
                for j, data, res in zip(live, datas, outs):
                    fr = frs[j]
                    if isinstance(res, Exception):
                        fr.error = f"{type(res).__name__}: {res}"
                        results[j] = res
                        continue
                    dst = out / dst_name(Path(paths[idx[j]]))
                    dst.write_bytes(res)
                    fr.ok, fr.bytes_in, fr.bytes_out, fr.archive = True, len(data), len(res), str(dst)
                    fr.gpu_ms = float(gpu_ms) / len(live)
                    results[j] = (fr.bytes_in, fr.bytes_out, 0, fr.gpu_ms, 0.0, str(dst))
            except Exception as e:                                       # noqa: BLE001 -- every file of the call fails
                for j in live:
                    frs[j].ok = False
                    frs[j].error = f"{type(e).__name__}: {e}"
                    results[j] = e
        wall = (time.perf_counter() - t0) * 1e3
        for j, fr in enumerate(frs):
            fr.wall_ms = wall / len(frs)
            if isinstance(results[j], tuple):
                results[j] = results[j][:4] + (fr.wall_ms, results[j][5])
        return results

    def work_unit(u, w=0):
        idx, is_run = units[u]
        return work_run(idx, w) if is_run else work(idx[0], w)

    res = run_batch(len(units), work_unit, device=device, dynamic=True, workers=len(fns))
    records = [asdict(f) for f in mine]
    if _dist_on():
        everyone = [None] * dist.get_world_size()
        dist.all_gather_object(everyone, records)
        records = [r for part in everyone for r in part]
    res.files = sorted((FileResult(**r) for r in records), key=lambda f: f.index)
    return res


def _fn_list(fn) -> list:
    return list(fn) if isinstance(fn, (list, tuple)) else [fn]


def compress_files(paths: Sequence[str], out_dir: str, compress_fn, device="cpu",
                   cfg: Optional[bytes] = None) -> BatchResult:
    """One archive per file.  compress_fn(data: numpy uint8 array, cfg) -> (archive bytes, gpu_ms) runs the product
    path on this rank's GPU (see make_gpu_compressor); a list of such callables = that many files in flight on this
    rank, one worker thread each.  If the callables have `many(datas, cfg) -> (archives, gpu_ms)` (bce_gpu_compress_many),
    one queue pull claims a run of consecutive files of at most gpu.MANY_MAX_N bytes (sizes from stat, before the queue
    starts) and compresses it with one `many` call; larger files go alone through compress_fn.  Returns every rank's
    stats and the manifest of all files, one entry per file."""
    import numpy as np
    from .gpu import MANY_MAX_N
    fns = _fn_list(compress_fn)

    def read(p):
        data = np.fromfile(p, dtype=np.uint8)                            # File::File, bce.cpp:842-856
        if data.size == 0:
            raise ValueError("Error loading file")                       # bce.cpp:1412-1415
        if data.size > 0x7FFFFFFF:
            raise ValueError("file too large for the BCE v0.4 format (2^31 - 1 bytes)")
        return data

    many = None
    if all(callable(getattr(f, "many", None)) for f in fns):
        many = lambda f, datas: f.many(datas, cfg)                       # noqa: E731
    return _files_batch(paths, out_dir, fns, read, lambda f, data: f(data, cfg), many,
                        lambda p: p.name + ".bce", MANY_MAX_N, device)


def decompressed_name(p: Path) -> str:
    """`x.bce` -> `x`; an archive without the suffix gets `.out` appended (never the archive's own name)."""
    return p.name[:-4] if p.name.endswith(".bce") and len(p.name) > 4 else p.name + ".out"


def decompress_files(paths: Sequence[str], out_dir: str, decompress_fn, device="cpu") -> BatchResult:
    """One file per archive, named as the archive without `.bce`.  decompress_fn(archive bytes) -> (bytes, gpu_ms) runs
    `bce -d` on this rank's GPU (see make_gpu_decompressor); a list of such callables = that many archives in flight
    on this rank.  If the callables have `many(archives) -> (per archive its bytes or exception, gpu_ms)`
    (bce_decompress_many), one queue pull claims a run of consecutive archives of at most gpu.MANY_MAX_N bytes (the
    archives of small files) and decodes it with one `many` call; larger archives go alone.  A damaged or unreadable
    archive fails alone.  Returns every rank's stats and the manifest, one entry per archive."""
    from .gpu import MANY_MAX_N
    fns = _fn_list(decompress_fn)

    def read(p):
        data = Path(p).read_bytes()
        if not data:
            raise ValueError("Error loading file")
        return data

    many = None
    if all(callable(getattr(f, "many", None)) for f in fns):
        many = lambda f, archives: f.many(archives)                      # noqa: E731
    return _files_batch(paths, out_dir, fns, read, lambda f, data: f(data), many, decompressed_name, MANY_MAX_N,
                        device)


def make_gpu_compressor(device_index: int, threads: int = 8):
    """The product path for compress_files: GPU front end + host coders through the C ABI (no CPU fallback:
    Frontend raises without a usable device)."""
    from . import Frontend, host
    fe = Frontend(device_index)

    def compress(data, cfg):
        arc = host.compress(fe, data, cfg=cfg, threads=threads)
        st = fe.stats()
        compress.gpu_launches += int(st["gpu_launches"])
        return arc, st["ms_bwt_total"] + st["ms_cse_total"]

    def many(datas, cfg):
        arcs = host.compress_many(fe, datas, cfg=cfg, threads=threads)
        st = fe.stats()
        compress.gpu_launches += int(st["gpu_launches"])
        return arcs, st["ms_total"]

    compress.many = many
    compress.frontend = fe
    compress.gpu_launches = 0
    return compress


def make_gpu_decompressor(device_index: int, threads: int = 8):
    """The product path for decompress_files: host decoders + GPU inverse BWT through the C ABI; `many` decodes a run
    of archives with bce_decompress_many (one archive per host thread, the small inverses in one launch)."""
    from . import Frontend, host
    fe = Frontend(device_index)

    def decompress(archive):
        out = host.decompress_many(fe, [archive], threads=threads)[0]
        if isinstance(out, Exception):
            raise out
        return out, fe.stats()["ms_total"]

    def many(archives):
        outs = host.decompress_many(fe, archives, threads=threads)
        return outs, fe.stats()["ms_total"]

    decompress.many = many
    decompress.frontend = fe
    return decompress


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description="compress files, one .bce archive per file, on all GPUs of the node "
                                             "(--decompress: restore the files of .bce archives)")
    ap.add_argument("--out", required=True)
    ap.add_argument("--config", default=None, help="288-byte coder config written by bce -s")
    ap.add_argument("--decompress", action="store_true", help="the files are archives: write each one's file to --out")
    ap.add_argument("files", nargs="+")
    args = ap.parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cfg = Path(args.config).read_bytes() if args.config else None
    try:
        per_gpu = max(1, min(2, (os.cpu_count() or 8) // (8 * max(1, world))))     # files in flight per GPU: 8 coder threads each
        device = "cuda" if world > 1 else "cpu"
        t0 = time.perf_counter()
        if args.decompress:
            res = decompress_files(args.files, args.out, [make_gpu_decompressor(local_rank) for _ in range(per_gpu)],
                                   device=device)
        else:
            fn = [make_gpu_compressor(local_rank) for _ in range(per_gpu)]
            res = compress_files(args.files, args.out, fn, device=device, cfg=cfg)
        wall = time.perf_counter() - t0
        if (dist.get_rank() if _dist_on() else 0) == 0:
            t = res.total
            print(json.dumps({"files": t.inputs, "failed": t.failed, "bytes_in": t.bytes_in, "bytes_out": t.bytes_out,
                              "wall_s": wall, "MBps": t.bytes_in / wall / 1e6,
                              "failures": [asdict(f) for f in res.files if not f.ok]}))
        return 0 if res.total.failed == 0 else 1
    finally:
        if _dist_on():
            dist.destroy_process_group()


if __name__ == "__main__":
    sys.exit(main())
