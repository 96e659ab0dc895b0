"""bce_gpu_unbwt_many and bce_decompress_many: many small inverses in one launch, many archives in one call.

The kernel's contract is unbwt::bitwise with the host decoder's clamps (csrc/host/decode.cpp, unbwt_serial), for any
rank words: valid dictionaries are checked against the oracle and the inputs they came from, arbitrary words against
unbwt_ref below.  Archives are checked against `bce -ds` (host.decompress(low_memory=True)), damaged ones included."""
import json
import random
from pathlib import Path

import numpy as np
import pytest

from bce_b200 import host, synth
from bce_b200.gpu import MANY_MAX_N, BceGpuError
from oracle import oracle
from tests.inputs import rnd, small_cases

pytestmark = pytest.mark.gpu

GENERATORS = ("enwik-shaped", "markov2-text", "mixed-binary", "uniform")
GOLD = Path(__file__).resolve().parent / "golden"
M32 = 0xFFFFFFFF


def unbwt_ref(ranks, offset, n):
    """unbwt_serial (decode.cpp) restated: bit and ones_before read at min(pos, n), the row keeps its 32-bit value."""
    R = [[int(w) for w in r] for r in ranks]

    def ones(j, pos):
        p = min(pos, n)
        w = R[j][p >> 5]
        return ((w & M32) + bin((w >> 32) & ((1 << (p & 31)) - 1)).count("1")) & M32

    def bit(j, pos):
        p = min(pos, n)
        return (R[j][p >> 5] >> (32 + (p & 31))) & 1

    zeros = [(n - ones(j, n)) & M32 for j in range(8)]
    out = bytearray(n)
    s = 0
    for i in range(n - 1, -1, -1):
        c = 0
        for j in range(8):
            b = bit(j, s)
            c |= b << j
            s = (zeros[j] + ones(j, s)) & M32 if b else (s - ones(j, s)) & M32
        out[(i + offset) % n] = c
    return bytes(out)


def corpus():
    """(name, bytes, primitive or None = not known): the small cases, n = 1, 2, 7, 8, 9, 31-33, 300 seeded sizes up to
    the limit over the four generators, the limit itself and a long repeat near it."""
    cases = [(name, data, prim) for name, data, prim in small_cases()]
    cases += [(f"n{n}", rnd(n, 3, 100 + n), None) for n in (1, 2, 7, 8, 9, 31, 32, 33)]
    r = random.Random(2027)
    for i in range(300):
        n = r.choice((r.randint(1, 64), r.randint(1, 4096), r.randint(1, MANY_MAX_N)))
        cases.append((f"gen{i}-{n}", synth.generate(GENERATORS[i % 4], n, 500 + i).tobytes(), None))
    cases.append(("max", synth.generate("enwik-shaped", MANY_MAX_N, 78).tobytes(), True))
    rep = rnd(30000, 50, 12)
    cases.append(("long-repeat-62k", rep + rnd(2000, 50, 13) + rep + b"!", True))
    return cases


CASES = corpus()


def primitive(data):
    return data not in (data + data)[1:-1]


def dictionary(data):
    L, off, _ = oracle.bwt(data)
    return oracle.wavelet(L), off


def test_valid_dictionaries(frontend):
    """Every dictionary in one call, shuffled: each text is the oracle's unbwt::bitwise, and the input itself where
    the input is primitive.  The fast path took the primitive ones, the serial path the exact powers."""
    order = list(range(len(CASES)))
    random.Random(7).shuffle(order)
    cases = [CASES[i] for i in order]
    dicts = []
    for _, data, _ in cases:
        ranks, off = dictionary(data)
        dicts.append((ranks, off, len(data)))
    got = frontend.unbwt_many(dicts)
    st = frontend.stats()
    powers = 0
    for (name, data, prim), (ranks, off, n), g in zip(cases, dicts, got):
        assert g.tobytes() == oracle.unbwt_bitwise(ranks, off, n).tobytes(), name
        if primitive(data):
            assert g.tobytes() == data, name
        else:                                        # an exact power: LF has several cycles
            assert prim is not True, name
            powers += 1
    assert st["unbwt_dicts"] == len(cases)
    assert st["n"] == MANY_MAX_N
    assert powers >= 5 and st["unbwt_serial"] == powers
    assert st["gpu_launches"] == 1


def arbitrary_dicts():
    """Seeded rank words: random words (rows far beyond n), valid dictionaries with a few damaged words, and words
    whose base counts are small so that rows stay near n."""
    r = np.random.default_rng(99)
    out = []
    for i in range(60):
        n = int(r.integers(1, 300))
        w = n // 32 + 1
        kind = i % 3
        if kind == 0:
            ranks = [r.integers(0, 2**64, size=w, dtype=np.uint64) for _ in range(8)]
        elif kind == 1:
            ranks, _ = dictionary(rnd(n, 4, 1000 + i))
            ranks = [x.copy() for x in ranks]
            for _ in range(int(r.integers(1, 4))):
                j, k = int(r.integers(0, 8)), int(r.integers(0, w))
                ranks[j][k] ^= np.uint64(1) << np.uint64(int(r.integers(0, 64)))
        else:
            hi = r.integers(0, 2**32, size=(8, w), dtype=np.uint64) << np.uint64(32)
            lo = r.integers(0, n + 40, size=(8, w), dtype=np.uint64)
            ranks = [hi[j] | lo[j] for j in range(8)]
        out.append((ranks, int(r.integers(0, n + 1)), n))
    return out


def test_arbitrary_words(frontend):
    dicts = arbitrary_dicts()
    got = frontend.unbwt_many(dicts)
    for i, ((ranks, off, n), g) in enumerate(zip(dicts, got)):
        assert g.tobytes() == unbwt_ref(ranks, off, n), i
    st = frontend.stats()
    assert st["unbwt_dicts"] == len(dicts) and st["unbwt_serial"] > 0


def test_reference_restatement_matches_oracle():
    for name, data, _ in small_cases()[:12]:
        ranks, off = dictionary(data)
        assert unbwt_ref(ranks, off, len(data)) == oracle.unbwt_bitwise(ranks, off, len(data)).tobytes(), name


def powers():
    return [b"abab", b"z" * 257, rnd(64, 4, 7) * 16, b"\0" * 4096, b"\0" * MANY_MAX_N]


def test_archives_end_to_end(frontend):
    prim = [d for _, d, _ in CASES if primitive(d)][:120]
    large = [synth.generate("enwik-shaped", MANY_MAX_N + 5, 3).tobytes(), synth.generate("markov2-text", 300_000, 4).tobytes()]
    archives = host.compress_many(frontend, prim, threads=8)
    inputs = list(prim)
    for d in powers() + large + prim[:10]:
        archives.append(oracle.compress(d))
        inputs.append(d)
    kat = json.loads((GOLD / "kat.json").read_text())["vectors"]
    for v in kat:
        archives.append(bytes.fromhex(v["archive_hex"]))
        inputs.append(eval(v["input_py"]))
    got = host.decompress_many(frontend, archives, threads=8)
    for i, (a, d, g) in enumerate(zip(archives, inputs, got)):
        want = host.decompress(a, low_memory=True)
        assert g == want, i
        if want == d:
            continue
        assert d in [p for p in powers()], i                    # only exact powers do not come back
    for v, g in zip(kat, got[-len(kat):]):
        assert g == eval(v["input_py"])
    assert all(g == d for g, d in zip(got[:len(prim)], prim))


def mutate(a, rng):
    """One of the four damages of tests/fuzz_decoder.py."""
    a = bytearray(a)
    mode = rng.randrange(4)
    if mode == 0 and len(a) > 2:
        for _ in range(rng.randrange(1, 4)):
            a[rng.randrange(len(a))] ^= 1 << rng.randrange(8)
    elif mode == 1 and len(a) > 4:
        a = a[:rng.randrange(2, len(a)) // 2 * 2]
    elif mode == 2:
        a[rng.randrange(min(len(a), 12))] = rng.randrange(256)
    else:
        a += bytes(rng.randrange(256) for _ in range(2 * rng.randrange(1, 8)))
    return bytes(a)


def test_damaged_archives(frontend, monkeypatch):
    """Damaged archives fail alone or decode to what `bce -ds` makes of them; intact ones in the same call still
    decode.  A damaged header that claims more than the limit is refused before decoding (BCE_HOST_MAX_N), as both
    decoders read that cap."""
    monkeypatch.setenv("BCE_HOST_MAX_N", str(MANY_MAX_N))
    src = [d for _, d, _ in small_cases() if 2 <= len(d) <= 5000]
    arcs = [oracle.compress(d) for d in src]
    rng = random.Random(4242)
    batch, intact = [], []
    for i in range(200):
        batch.append(mutate(rng.choice(arcs), rng))
        intact.append(False)
        if i % 10 == 0:
            j = rng.randrange(len(arcs))
            batch.append(arcs[j])
            intact.append(src[j])
    got = host.decompress_many(frontend, batch, threads=8)
    errors = 0
    for i, (a, g, ok) in enumerate(zip(batch, got, intact)):
        try:
            want = host.decompress(a, low_memory=True)
        except (RuntimeError, ValueError):
            want = None
        if want is None:
            assert isinstance(g, BceGpuError) and g.code == -1, i
            errors += 1
        else:
            assert g == want, i
        if ok is not False and primitive(ok):        # an exact power comes back as `bce -ds` makes it, checked above
            assert g == ok, i
    assert errors > 20


def test_context_reuse(frontend):
    data = [synth.generate(GENERATORS[i % 4], 500 + 997 * i, 40 + i).tobytes() for i in range(12)]
    for rep in range(2):
        arcs = host.compress_many(frontend, data, threads=4)
        assert arcs == [oracle.compress(d) for d in data]
        assert host.decompress_many(frontend, arcs, threads=4) == data
        off, Cv, streams = frontend.compress_front(data[rep])
        want = oracle.cse(oracle.wavelet(oracle.bwt(data[rep])[0]), len(data[rep]))
        assert Cv == want["C"] and all(np.array_equal(streams[i], want["streams"][i]) for i in range(8))
        ranks, off = dictionary(data[5 + rep])
        assert frontend.unbwt(ranks, off, len(data[5 + rep])).tobytes() == data[5 + rep]
        assert [g.tobytes() for g in frontend.unbwt_many([dictionary(d) + (len(d),) for d in data])] == data
        assert host.decompress_many(frontend, [host.compress(frontend, data[7])]) == [data[7]]


def test_batch_round_trip(tmp_path):
    from bce_b200 import batch
    files = [(f"f{j}.txt", synth.generate(GENERATORS[j % 4], 100 + 1777 * j, j).tobytes()) for j in range(30)]
    files.append(("above-limit.bin", synth.generate("mixed-binary", MANY_MAX_N + 5, 3).tobytes()))
    paths = []
    for name, data in files:
        (tmp_path / name).write_bytes(data)
        paths.append(str(tmp_path / name))
    fn = batch.make_gpu_compressor(0, threads=4)
    try:
        res = batch.compress_files(paths, str(tmp_path / "arc"), fn)
    finally:
        fn.frontend.close()
    assert all(f.ok for f in res.files)
    arcs = [f.archive for f in res.files]
    trunc = tmp_path / "arc" / "truncated.bin.bce"
    trunc.write_bytes(Path(arcs[3]).read_bytes()[:7])
    arcs.append(str(trunc))
    dfn = batch.make_gpu_decompressor(0, threads=4)
    calls, many = [], dfn.many
    dfn.many = lambda archives: (calls.append(len(archives)), many(archives))[1]
    try:
        res = batch.decompress_files(arcs, str(tmp_path / "back"), dfn)
    finally:
        dfn.frontend.close()
    assert [f.ok for f in res.files] == [True] * len(files) + [False]
    assert res.total.failed == 1 and "truncated" in res.files[-1].path
    for (name, data), f in zip(files, res.files):
        assert Path(f.archive) == tmp_path / "back" / name
        assert Path(f.archive).read_bytes() == data, name
    assert max(calls) >= 30                                   # the small archives in one call


@pytest.mark.parametrize("case", ["k0", "n0", "above-limit", "offset-above-n"])
def test_bad_arguments(frontend, case):
    z = lambda n: [np.zeros(n // 32 + 1, dtype=np.uint64) for _ in range(8)]       # noqa: E731
    dicts = {"k0": [], "n0": [(z(0), 0, 0)], "above-limit": [(z(5), 0, 5), (z(MANY_MAX_N + 1), 0, MANY_MAX_N + 1)],
             "offset-above-n": [(z(9), 10, 9)]}[case]
    with pytest.raises(BceGpuError) as e:
        frontend.unbwt_many(dicts)
    assert e.value.code == -1
