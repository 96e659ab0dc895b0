"""bce_gpu_decompress_many: the whole decoder of many small archives on the device.

Its contract is the host decoder's (decode_to_ranks, then unbwt::bitwise): every text equals what `bce -ds`
(host.decompress(low_memory=True)) makes of the same archive, and an archive the host rejects has status -1."""
import ctypes as C
import random
import re
from pathlib import Path

import numpy as np
import pytest

from bce_b200 import host, synth
from bce_b200.gpu import MANY_MAX_N, BceGpuError
from oracle import oracle
from tests.inputs import rnd, small_cases
from tests.test_gpu_code_many import CASES, TABLES, archives
from tests.test_gpu_decompress_many import mutate, primitive

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
DEVICE_DECODERS = int(re.search(r"#define BCE_HOST_MANY_DEVICE_DECODERS (\d+)u",
                                (ROOT / "include" / "bce_host.h").read_text()).group(1))


def bce_ds(a):
    try:
        return host.decompress(a, low_memory=True)
    except (RuntimeError, ValueError):
        return None


def test_valid_archives_all_tables(frontend):
    """Every archive of the corpus under five tables (default, all 0, all 5, random, one from `bce -s`) in one call."""
    tables = dict(TABLES)
    tables["scan"] = host.scan(frontend, synth.generate("markov2-text", 60000, 5).tobytes())
    inputs = [d for _, d in CASES]
    arcs, names, data = [], [], []
    for tname, cfg in sorted(tables.items()):
        got, _ = archives(frontend, inputs, cfg)
        arcs += got
        names += [f"{name} ({tname})" for name, _ in CASES]
        data += inputs
    texts = frontend.decompress_many(arcs, [len(d) for d in data])
    st = frontend.stats()
    assert st["gpu_launches"] == 2 and st["ms_decoder"] > 0, st
    assert st["unbwt_dicts"] == len(arcs) and st["n"] == MANY_MAX_N
    assert st["cse_visits"] > 0 and st["cse_rounds"] > 0
    for a, d, t, name in zip(arcs, data, texts, names):
        assert not isinstance(t, BceGpuError), name
        if primitive(d):
            assert t == d, name
        assert t == bce_ds(a), name


def test_damaged_archives(frontend):
    """1000 seeded damages mixed with intact archives: status and text as `bce -ds`, archive by archive."""
    src = [d for _, d, _ in small_cases() if 2 <= len(d) <= 5000]
    src += [synth.generate("markov2-text", 300 + 97 * i, 60 + i).tobytes() for i in range(20)]
    src += [rnd(3000, 2, 7), rnd(3000, 256, 8)]
    arcs = [oracle.compress(d) for d in src]
    rng = random.Random(2026)
    batch, intact = [], []
    while len(batch) < 1100:
        a = mutate(rng.choice(arcs), rng)
        if len(batch) % 10 == 0:
            j = rng.randrange(len(arcs))
            a, ok = arcs[j], src[j]
        else:
            ok = None
        n = host.archive_size(a)
        if n is None or n > MANY_MAX_N:
            continue                                 # the caller refuses those before the device sees them
        batch.append(a)
        intact.append(ok)
    got = frontend.decompress_many(batch, [host.archive_size(a) for a in batch])
    rejected = accepted_damaged = 0
    for i, (a, g, ok) in enumerate(zip(batch, got, intact)):
        want = bce_ds(a)
        if want is None:
            assert isinstance(g, BceGpuError) and g.code == -1, i
            rejected += 1
        else:
            assert g == want, i
            if ok is None and want is not None:
                accepted_damaged += 1
        if ok is not None and primitive(ok):
            assert g == ok, i
    assert rejected > 100 and accepted_damaged > 50, (rejected, accepted_damaged)


def test_header_disagrees_with_n(frontend):
    data = [synth.generate("enwik-shaped", 1000 + 100 * i, i).tobytes() for i in range(5)]
    arcs = [oracle.compress(d) for d in data]
    sizes = [len(d) for d in data]
    sizes[2] += 1
    got = frontend.decompress_many(arcs, sizes)
    for i, (g, d) in enumerate(zip(got, data)):
        if i == 2:
            assert isinstance(g, BceGpuError) and g.code == -1
        else:
            assert g == d


@pytest.mark.parametrize("side", ["below", "at"])
def test_routing(frontend, side):
    """host.decompress_many on both sides of BCE_HOST_MANY_DEVICE_DECODERS, small and large archives in one call."""
    k = DEVICE_DECODERS - 1 if side == "below" else DEVICE_DECODERS
    small = [synth.generate(("enwik-shaped", "markov2-text", "mixed-binary")[i % 3], 200 + 131 * i, 900 + i).tobytes()
             for i in range(k)]
    arcs = host.compress_many(frontend, small, threads=8)
    assert host.decompress_many(frontend, arcs, threads=8) == small
    assert (frontend.stats()["ms_decoder"] > 0) == (side == "at")
    large = [synth.generate("enwik-shaped", MANY_MAX_N + 77, 3).tobytes()]
    mixed = arcs[: k // 2] + [oracle.compress(large[0])] + arcs[k // 2:] + [arcs[0][:8]]
    got = host.decompress_many(frontend, mixed, threads=8)
    assert got[: k // 2] + got[k // 2 + 1:-1] == small
    assert got[k // 2] == large[0]
    want = bce_ds(arcs[0][:8])
    assert got[-1] == want if want is not None else (isinstance(got[-1], BceGpuError) and got[-1].code == -1)


def test_host_max_n(frontend, monkeypatch):
    """Archives above the cap fail alone; the DEVICE_DECODERS + 4 below it still make a group for the device."""
    sizes = [500 + 40 * (i % 20) for i in range(DEVICE_DECODERS + 4)] + [1501, 1600, 2500, 9000, 40000]
    data = [synth.generate("markov2-text", n, i).tobytes() for i, n in enumerate(sizes)]
    arcs = host.compress_many(frontend, data, threads=8)
    monkeypatch.setenv("BCE_HOST_MAX_N", "1500")
    got = host.decompress_many(frontend, arcs, threads=8)
    assert frontend.stats()["ms_decoder"] > 0
    for d, g in zip(data, got):
        if len(d) > 1500:
            assert isinstance(g, BceGpuError) and g.code == -1
        else:
            assert g == d


def test_context_reuse(frontend):
    data = [synth.generate(("enwik-shaped", "markov2-text", "mixed-binary", "uniform")[i % 4], 700 + 811 * i, 70 + i).tobytes()
            for i in range(12)]
    for rep in range(2):
        arcs, _ = archives(frontend, data)
        assert frontend.decompress_many(arcs, [len(d) for d in data]) == data
        off, Cv, streams = frontend.compress_front(data[rep])
        want = oracle.cse(oracle.wavelet(oracle.bwt(data[rep])[0]), len(data[rep]))
        assert Cv == want["C"] and all(np.array_equal(streams[i], want["streams"][i]) for i in range(8))
        assert frontend.decompress_many(arcs[::-1], [len(d) for d in data[::-1]]) == data[::-1]
        ranks, off = oracle.wavelet(oracle.bwt(data[5])[0]), oracle.bwt(data[5])[1]
        assert frontend.unbwt(ranks, off, len(data[5])).tobytes() == data[5]
        dicts = []
        for d in data:
            L, o, _ = oracle.bwt(d)
            dicts.append((oracle.wavelet(L), o, len(d)))
        assert [g.tobytes() for g in frontend.unbwt_many(dicts)] == data
        assert frontend.decompress_many(arcs[:3], [len(d) for d in data[:3]]) == data[:3]
        assert frontend.stats()["gpu_launches"] == 2


@pytest.mark.parametrize("case", ["k0", "n0", "above-limit", "starts-decrease"])
def test_bad_arguments(frontend, case):
    a = oracle.compress(b"hello, world")
    W = np.frombuffer(a + a, dtype=np.uint16)
    h = len(a) // 2
    starts = {"k0": [0], "n0": [0, h], "above-limit": [0, h, 2 * h], "starts-decrease": [0, h, h - 1]}[case]
    n = {"k0": [], "n0": [0], "above-limit": [12, MANY_MAX_N + 1], "starts-decrease": [12, 12]}[case]
    k = len(starts) - 1
    st = np.zeros(max(k, 1) + 1, dtype=np.uint64)
    st[: len(starts)] = starts
    nn = np.array(n + [1], dtype=np.uint32)
    out = np.zeros(64, dtype=np.uint8)
    status = np.zeros(4, dtype=np.int32)
    rc = frontend.lib.bce_gpu_decompress_many(frontend.h, W.ctypes.data, st.ctypes.data_as(C.POINTER(C.c_uint64)),
                                              nn.ctypes.data, k, out.ctypes.data, status.ctypes.data)
    assert rc == -1
    assert frontend.decompress_many([a], [12]) == [b"hello, world"]    # the context is still usable
