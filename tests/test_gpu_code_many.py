"""bce_gpu_compress_many_archives: the range coders of many small inputs on the device.

Every archive must be byte-equal to oracle.compress(data, cfg) and to the archive the host coders make of the same
input's CODER words, for several context-bit tables; more than one call (a small arena), a context shared with the
other calls, bad arguments, and both sides of bce_compress_many's routing threshold give the same archives."""
import random
import re
from pathlib import Path

import numpy as np
import pytest

from bce_b200 import host, synth
from bce_b200.gpu import EMIT_CODER, EMIT_RAW, MANY_MAX_N, OPT_EMIT_BATCH_BYTES, BceGpuError
from oracle import oracle
from tests.inputs import rnd, small_cases

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
GENERATORS = ("enwik-shaped", "markov2-text", "mixed-binary", "uniform")
DEVICE_CODERS = int(re.search(r"#define BCE_HOST_MANY_DEVICE_CODERS (\d+)u",
                              (ROOT / "include" / "bce_host.h").read_text()).group(1))


def corpus():
    """(name, bytes): the small cases, n = 1, 2, 7 .. 9, exact powers, a long repeat near the limit, 256- and 2-symbol
    random data near the limit (k > 31 counts), the limit itself and 300 seeded sizes over the four generators."""
    cases = [(name, data) for name, data, _ in small_cases()]
    cases += [(f"n{n}", rnd(n, 3, 300 + n)) for n in (1, 2, 7, 8, 9)]
    cases += [("power-ab-32k", b"ab" * 16384), ("power-x-64k", b"x" * MANY_MAX_N),
              ("power-rnd-100x600", rnd(100, 26, 5) * 600)]
    rep = rnd(30000, 50, 12)
    cases += [("long-repeat-62k", rep + rnd(2000, 50, 13) + rep + b"!"),
              ("rnd256-64k", rnd(MANY_MAX_N, 256, 21)), ("rnd2-64k", rnd(MANY_MAX_N - 3, 2, 22)),
              ("max", synth.generate("enwik-shaped", MANY_MAX_N, 78).tobytes())]
    r = random.Random(4242)
    for i in range(300):
        n = r.choice((r.randint(1, 64), r.randint(1, 4096), r.randint(1, MANY_MAX_N)))
        cases.append((f"gen{i}-{n}", synth.generate(GENERATORS[i % 4], n, i).tobytes()))
    return cases


CASES = corpus()


def tables():
    r = np.random.default_rng(9)
    rand = r.integers(0, 6, size=288, dtype=np.uint8)
    rand[8 * 32 + 3] = 4                                   # a non-zero header row
    return {"default": None, "zeros": bytes(288), "fives": bytes([5]) * 288, "random": rand.tobytes()}


TABLES = tables()
_want = {}


def want(i, cfg_name, cfg):
    key = (i, cfg_name)
    if key not in _want:
        _want[key] = oracle.compress(CASES[i][1], cfg)
    return _want[key]


def archives(fe, inputs, cfg=None):
    """compress_many_archives until every input is done: (archives, calls)."""
    res, todo, calls = [None] * len(inputs), list(range(len(inputs))), 0
    while todo:
        out = fe.compress_many_archives([inputs[i] for i in todo], cfg)
        calls += 1
        assert any(a is not None for a in out), "no input was done"
        for i, a in zip(todo, out):
            res[i] = a
        todo = [i for i, a in zip(todo, out) if a is None]
    return res, calls


def host_coder_archives(fe, inputs, cfg):
    """The same inputs' CODER words from the front end, coded by the host coders."""
    got = fe.compress_front_many(inputs, EMIT_CODER, cfg)
    return [host.encode_archive_words(Cv, words, len(d), off, cfg) for d, (off, Cv, words) in zip(inputs, got)]


@pytest.mark.parametrize("cfg_name", sorted(TABLES))
def test_archives_match_oracle_and_host_coders(frontend, cfg_name):
    cfg = TABLES[cfg_name]
    inputs = [d for _, d in CASES]
    got, calls = archives(frontend, inputs, cfg)
    assert calls == 1
    st = frontend.stats()
    assert st["gpu_launches"] == 2 and st["ms_coder"] > 0, st
    hosted = host_coder_archives(frontend, inputs, cfg)
    for i, (name, _) in enumerate(CASES):
        assert got[i] == want(i, cfg_name, cfg), f"{name}: differs from the oracle ({cfg_name} table)"
        assert got[i] == hosted[i], f"{name}: differs from the host coders ({cfg_name} table)"


def test_table_from_scan(frontend):
    """A table `bce -s` derived from one of the inputs (non-zero header row included where it says so)."""
    cfg = host.scan(frontend, synth.generate("markov2-text", 60000, 5).tobytes())
    assert len(cfg) == 288
    pick = [i for i in range(len(CASES)) if i % 3 == 0]
    inputs = [CASES[i][1] for i in pick]
    got, _ = archives(frontend, inputs, cfg)
    for i, a in zip(pick, got):
        assert a == oracle.compress(CASES[i][1], cfg), CASES[i][0]


def test_resubmission(frontend):
    """A small arena: more than one call, the same archives."""
    inputs = [d for _, d in CASES]
    frontend.set_option(OPT_EMIT_BATCH_BYTES, 1 << 20)
    try:
        got, calls = archives(frontend, inputs, TABLES["random"])
    finally:
        frontend.set_option(OPT_EMIT_BATCH_BYTES, 0)
    assert calls > 1
    for i, (name, _) in enumerate(CASES):
        assert got[i] == want(i, "random", TABLES["random"]), name


def test_context_reuse_and_emission_state(frontend):
    """Interleaved with compress_front, compress_many and unbwt_many on one context: every result unchanged, and the
    context's emission mode and table are the ones set before the archive calls."""
    X, Y = TABLES["random"], TABLES["fives"]
    small = [CASES[i][1] for i in range(0, len(CASES), 7)]
    big = synth.generate("enwik-shaped", 300_000, 3).tobytes()
    L, off, _ = oracle.bwt(big)
    w = oracle.cse(oracle.wavelet(L), len(big))
    frontend.set_emit_mode(EMIT_CODER, X)
    try:
        for rep in range(2):
            got, _ = archives(frontend, small, Y)
            for d, a in zip(small, got):
                assert a == oracle.compress(d, Y), (rep, len(d))
            words = frontend.compress_many_call(small[:5])             # the context's mode: CODER with table X
            for j, d in enumerate(small[:5]):
                Ld, od, _ = oracle.bwt(d)
                wd = oracle.cse(oracle.wavelet(Ld), len(d))
                packed = host.pack_counts(EMIT_CODER, wd["streams"], X)
                r = words[j]
                assert r.done and r.offset == od
                for s in range(8):
                    cnt = int(r.count[s])
                    v = np.ctypeslib.as_array(r.words[s], shape=(cnt,)) if cnt else np.zeros(0, np.uint32)
                    assert np.array_equal(v, packed[s]), (rep, j, s)
            frontend.set_emit_mode(EMIT_RAW)
            o, Cv, streams = frontend.compress_front(big)
            assert (o, Cv) == (off, w["C"])
            assert all(np.array_equal(streams[s], w["streams"][s]) for s in range(8))
            texts = [CASES[i][1] for i in range(1, 40, 4)]
            dicts = []
            for t in texts:
                Lt, ot, _ = oracle.bwt(t)
                dicts.append((oracle.wavelet(Lt), ot, len(t)))
            assert [g.tobytes() for g in frontend.unbwt_many(dicts)] == texts
            frontend.set_emit_mode(EMIT_CODER, X)
    finally:
        frontend.set_emit_mode(EMIT_RAW)


@pytest.mark.parametrize("case", ["k0", "empty", "too-long", "cell6"])
def test_bad_arguments(frontend, case):
    inputs, cfg = [b"abc", b"hello"], None
    if case == "k0":
        inputs = []
    elif case == "empty":
        inputs = [b"abc", b""]
    elif case == "too-long":
        inputs = [b"abc", bytes(MANY_MAX_N + 1)]
    else:
        cfg = bytes([5] * 287 + [6])
    with pytest.raises(BceGpuError) as e:
        frontend.compress_many_archives(inputs, cfg)
    assert e.value.code == -1
    assert frontend.compress_many_archives([b"abc", b"hello"]) == [oracle.compress(b"abc"), oracle.compress(b"hello")]


@pytest.mark.parametrize("side", ["host", "device"])
def test_routing_threshold(frontend, side):
    """bce_compress_many codes calls of fewer than BCE_HOST_MANY_DEVICE_CODERS inputs on the host (one front-end launch)
    and larger ones on the device (front end + coders): the same archives either way."""
    k = DEVICE_CODERS - 1 if side == "host" else DEVICE_CODERS
    pick = [(7 * j) % len(CASES) for j in range(k)]
    inputs = [CASES[i][1] for i in pick]
    got = host.compress_many(frontend, inputs, TABLES["random"], threads=4)
    st = frontend.stats()
    assert st["gpu_launches"] == (1 if side == "host" else 2) and (st["ms_coder"] > 0) == (side == "device"), st
    for i, a in zip(pick, got):
        assert a == want(i, "random", TABLES["random"]), CASES[i][0]
