"""CPU: compress_files with a compressor that has `many` (bce_gpu_compress_many): runs of consecutive small files go
through one `many` call per queue pull, larger files alone, and the manifest stays one entry per file -- over gloo
with two ranks, and in one process."""
import os
import socket
import sys
from pathlib import Path

import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parent.parent
MAX_N = 65536                     # gpu.MANY_MAX_N


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def fake_compressor():
    """Stands in for make_gpu_compressor: an archive says which path made it and, for `many`, how many files the call
    had and where the file was in it."""
    def single(data, cfg):
        return b"S" + bytes([int(data[0])]), 1.5

    def many(datas, cfg):
        return [b"M" + bytes([int(d[0]), len(datas), j]) for j, d in enumerate(datas)], 4.0

    single.many = many
    return single


def write_inputs(tmp):
    """16 files: 0..5 small, 6 large, 7..9 small, 10 missing, 11 small, 12 empty, 13..15 small."""
    sizes = {}
    for i in range(16):
        if i == 10:
            continue
        n = 0 if i == 12 else MAX_N + 1 if i == 6 else 1000 + 37 * i
        (Path(tmp) / f"in{i}").write_bytes(bytes([i]) * n)
        sizes[i] = n
    return [os.path.join(tmp, f"in{i}") for i in range(16)], sizes


def _worker(rank, world, port, q, tmp):
    sys.path.insert(0, str(ROOT))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from bce_b200 import batch
    paths = [os.path.join(tmp, f"in{i}") for i in range(16)]             # written by the test before the spawn
    res = batch.compress_files(paths, os.path.join(tmp, "out"), fake_compressor(), device="cpu")
    q.put((rank, [vars(f) for f in res.files], vars(res.total)))
    dist.barrier()
    dist.destroy_process_group()


def check_manifest(files, total, tmp, sizes):
    assert [f["index"] for f in files] == list(range(16))                    # every file exactly once
    bad = [f["index"] for f in files if not f["ok"]]
    assert bad == [10, 12]
    assert "Error loading file" in files[12]["error"]
    assert total["inputs"] == 14 and total["failed"] == 2
    assert total["bytes_in"] == sum(sizes.values())
    # runs are cut at the large file, the missing and the empty one
    runs = [range(0, 6), range(7, 10), range(11, 12), range(13, 16)]
    for run in runs:
        for j, i in enumerate(run):
            arc = (Path(tmp) / "out" / f"in{i}.bce").read_bytes()
            assert arc == b"M" + bytes([i, len(run), j]), i
            assert files[i]["bytes_in"] == sizes[i] and files[i]["bytes_out"] == len(arc)
    assert (Path(tmp) / "out" / "in6.bce").read_bytes() == b"S\x06"                 # above the limit: alone
    assert files[6]["gpu_ms"] == 1.5


def test_two_ranks_group_small_files(tmp_path):
    _, sizes = write_inputs(tmp_path)
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, str(tmp_path))) for r in range(world)]
    for p in procs:
        p.start()
    got = sorted(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert got[0][1] == got[1][1] and got[0][2] == got[1][2]
    check_manifest(got[0][1], got[0][2], tmp_path, {i: n for i, n in sizes.items() if n})


def test_one_process_and_run_budget(tmp_path):
    from bce_b200 import batch
    paths, sizes = write_inputs(tmp_path)
    res = batch.compress_files(paths, str(tmp_path / "out"), [fake_compressor(), fake_compressor()])
    check_manifest([vars(f) for f in res.files], vars(res.total), tmp_path, {i: n for i, n in sizes.items() if n})
    # a run never exceeds its byte budget; -1 (stat failed) and 0 go alone
    units = batch.small_file_runs([10, 10, 10, -1, 10, 0, 10, 10], 100, budget=20)
    assert units == [([0, 1], True), ([2], True), ([3], False), ([4], True), ([5], False), ([6, 7], True)]


def test_plain_compressor_keeps_one_file_per_pull(tmp_path):
    from bce_b200 import batch
    paths, sizes = write_inputs(tmp_path)
    res = batch.compress_files(paths, str(tmp_path / "o"), lambda d, cfg: (b"P" + bytes(d[:1]), 1.0))
    assert [f.index for f in res.files] == list(range(16))
    assert all((tmp_path / "o" / f"in{i}.bce").read_bytes() == b"P" + bytes([i]) for i in sizes if sizes[i])
