"""CPU: decompress_files with a decompressor that has `many` (bce_decompress_many): runs of consecutive small archives
go through one `many` call per queue pull, larger archives alone, a damaged archive fails alone inside its run, and the
output is the archive's name without `.bce` -- over gloo with two ranks, and in one process."""
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


def fake_decompressor():
    """Stands in for make_gpu_decompressor: the output says which path made it and, for `many`, how many archives the
    call had and where the archive was in it.  An archive starting with 0xEE is damaged."""
    def single(archive):
        return b"S" + archive[:1], 1.5

    def many(archives):
        return [ValueError("damaged") if a[0] == 0xEE else b"M" + bytes([a[0], len(archives), j])
                for j, a in enumerate(archives)], 4.0

    single.many = many
    return single


def archive_paths(tmp):
    return [os.path.join(tmp, f"in{i}.bin" if i == 15 else f"in{i}.bin.bce") for i in range(16)]


def write_archives(tmp):
    """16 archives: 0..5 small, 6 large, 7..9 small, 10 missing, 11 small, 12 empty, 13..15 small, 14 damaged;
    15 has no .bce suffix."""
    sizes = {}
    paths = archive_paths(tmp)
    for i, p in enumerate(paths):
        if i == 10:
            continue
        n = 0 if i == 12 else MAX_N + 1 if i == 6 else 1000 + 37 * i
        Path(p).write_bytes(bytes([0xEE if i == 14 else i]) * n)
        sizes[i] = n
    return paths, sizes


def _worker(rank, world, port, q, tmp):
    sys.path.insert(0, str(ROOT))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from bce_b200 import batch                                             # archives written by the test before the spawn
    res = batch.decompress_files(archive_paths(tmp), os.path.join(tmp, "out"), fake_decompressor(), device="cpu")
    q.put((rank, [vars(f) for f in res.files], vars(res.total)))
    dist.barrier()
    dist.destroy_process_group()


def check_manifest(files, total, tmp, sizes):
    assert [f["index"] for f in files] == list(range(16))                    # every archive exactly once
    bad = [f["index"] for f in files if not f["ok"]]
    assert bad == [10, 12, 14]
    assert "Error loading file" in files[12]["error"] and "damaged" in files[14]["error"]
    assert total["inputs"] == 13 and total["failed"] == 3
    runs = [range(0, 6), range(7, 10), range(11, 12), range(13, 16)]
    for run in runs:
        for j, i in enumerate(run):
            if i == 14:
                assert not (Path(tmp) / "out" / "in14.bin").exists()
                continue
            name = "in15.bin.out" if i == 15 else f"in{i}.bin"
            out = (Path(tmp) / "out" / name).read_bytes()
            assert out == b"M" + bytes([i, len(run), j]), i
            assert files[i]["bytes_in"] == sizes[i] and files[i]["bytes_out"] == len(out)
            assert files[i]["archive"] == str(Path(tmp) / "out" / name)
    assert (Path(tmp) / "out" / "in6.bin").read_bytes() == b"S\x06"                   # above the limit: alone
    assert files[6]["gpu_ms"] == 1.5


def test_two_ranks_group_small_archives(tmp_path):
    _, sizes = write_archives(tmp_path)
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


def test_one_process(tmp_path):
    from bce_b200 import batch
    paths, sizes = write_archives(tmp_path)
    res = batch.decompress_files(paths, str(tmp_path / "out"), [fake_decompressor(), fake_decompressor()])
    check_manifest([vars(f) for f in res.files], vars(res.total), tmp_path, {i: n for i, n in sizes.items() if n})


def test_output_names():
    from bce_b200 import batch
    assert batch.decompressed_name(Path("/a/x.txt.bce")) == "x.txt"
    assert batch.decompressed_name(Path("x.bin")) == "x.bin.out"
    assert batch.decompressed_name(Path(".bce")) == ".bce.out"
