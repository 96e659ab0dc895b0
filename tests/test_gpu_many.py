"""bce_gpu_compress_many: the one-CTA-per-input front end, input by input against the oracle.

Raw counts are compared count by count with oracle.cse, offset and C with the oracle's BWT and wavelet, and coder-mode
archives byte for byte with oracle.compress.  The same inputs in another call order, and with an arena too small for
one call, must give the same per-input results."""
import random
from pathlib import Path

import numpy as np
import pytest

from bce_b200 import host, synth
from bce_b200.gpu import EMIT_CODER, EMIT_RAW, EMIT_SCAN, MANY_MAX_N, OPT_EMIT_BATCH_BYTES, BceGpuError
from oracle import oracle
from tests.inputs import rnd, small_cases

pytestmark = pytest.mark.gpu

GENERATORS = ("enwik-shaped", "markov2-text", "mixed-binary", "uniform")


def corpus():
    """(name, bytes): every small case, n = 1, 2, 7, 8, 9, 500 random sizes up to the limit, the limit itself and a
    long repeat near it (about 8 x 30000 rounds of the level loop)."""
    cases = [(name, data) for name, data, _ in small_cases()]
    cases += [(f"n{n}", rnd(n, 3, 100 + n)) for n in (1, 2, 7, 8, 9)]
    r = random.Random(2026)
    for i in range(500):
        n = r.choice((r.randint(1, 64), r.randint(1, 4096), r.randint(1, MANY_MAX_N)))
        if i % 3 == 0:
            cases.append((f"rnd{i}-{n}", rnd(n, r.choice((2, 4, 26, 256)), i)))
        else:
            cases.append((f"gen{i}-{n}", synth.generate(GENERATORS[i % 4], n, i).tobytes()))
    cases.append(("max", synth.generate("enwik-shaped", MANY_MAX_N, 77).tobytes()))
    rep = rnd(30000, 50, 12)
    cases.append(("long-repeat-62k", rep + rnd(2000, 50, 13) + rep + b"!"))
    return cases


CASES = corpus()
_want = {}


def want(name, data):
    if name not in _want:
        L, off, _ = oracle.bwt(data)
        w = oracle.cse(oracle.wavelet(L), len(data))
        _want[name] = (off, w["C"], w["streams"], sum(w["visits"]), w["rounds"])
    return _want[name]


def check_raw(results, cases):
    for (name, data), (off, Cv, streams) in zip(cases, results):
        woff, wC, wstreams, _, _ = want(name, data)
        assert off == woff and Cv == wC, name
        for i in range(8):
            assert np.array_equal(streams[i], wstreams[i]), (name, i)


def test_raw_counts_offset_and_C(frontend):
    res = frontend.compress_front_many([d for _, d in CASES], EMIT_RAW)
    check_raw(res, CASES)
    st = frontend.stats()
    assert frontend.last_many_calls == 1
    assert st["cse_visits"] == sum(want(n, d)[3] for n, d in CASES)
    assert st["cse_rounds"] == sum(want(n, d)[4] for n, d in CASES)


def test_shuffled_order(frontend):
    order = list(range(len(CASES)))
    random.Random(5).shuffle(order)
    cases = [CASES[i] for i in order]
    check_raw(frontend.compress_front_many([d for _, d in cases], EMIT_RAW), cases)


def test_coder_archives(frontend):
    cases = CASES[:40] + CASES[-2:] + CASES[40::12]
    archives = host.compress_many(frontend, [d for _, d in cases], threads=8)
    for (name, data), arc in zip(cases, archives):
        assert arc == oracle.compress(data), name
    # the same words as the per-input front end emits
    words = frontend.compress_front_many([d for _, d in cases[-3:]], EMIT_CODER)
    for (name, data), (off, Cv, streams) in zip(cases[-3:], words):
        off1, C1, streams1 = frontend.compress_front_words(data, EMIT_CODER)
        assert (off, Cv) == (off1, C1), name
        for i in range(8):
            assert np.array_equal(streams[i], streams1[i]), (name, i)


def test_resubmission(frontend):
    """An arena of one input's worst case: most calls finish a few inputs, the rest are submitted again."""
    cases = CASES[:30] + CASES[-12:]
    frontend.set_option(OPT_EMIT_BATCH_BYTES, 4096)
    try:
        res = frontend.compress_front_many([d for _, d in cases], EMIT_RAW)
        assert frontend.last_many_calls > 1
        check_raw(res, cases)
        archives = host.compress_many(frontend, [d for _, d in cases], threads=4)
        for (name, data), arc in zip(cases, archives):
            assert arc == oracle.compress(data), name
    finally:
        frontend.set_option(OPT_EMIT_BATCH_BYTES, 0)


def test_batch_routes_small_files(tmp_path):
    """bce_b200.batch with the product compressor: the small files go through one compress_many call, the file above
    the limit through compress_front; every archive is the oracle's."""
    from bce_b200 import batch
    cases = CASES[:20] + [("above-limit", synth.generate("enwik-shaped", MANY_MAX_N + 5, 3).tobytes())]
    paths = []
    for j, (_, data) in enumerate(cases):
        (tmp_path / f"f{j}").write_bytes(data)
        paths.append(str(tmp_path / f"f{j}"))
    fn = batch.make_gpu_compressor(0, threads=4)
    calls, many = [], fn.many
    fn.many = lambda datas, cfg: (calls.append(len(datas)), many(datas, cfg))[1]
    try:
        res = batch.compress_files(paths, str(tmp_path / "out"), fn)
    finally:
        fn.frontend.close()
    assert calls == [20] and all(f.ok for f in res.files)
    for (name, data), f in zip(cases, res.files):
        assert Path(f.archive).read_bytes() == oracle.compress(data), name


@pytest.mark.parametrize("inputs", [[b"a" * (MANY_MAX_N + 1)], [], [b"abc", b"", b"x"]],
                         ids=["above-limit", "k0", "empty-input"])
def test_bad_arguments(frontend, inputs):
    with pytest.raises(BceGpuError) as e:
        frontend.compress_many_call(inputs)
    assert e.value.code == -1


def test_scan_mode_refused(frontend):
    with pytest.raises(BceGpuError) as e:
        frontend.compress_front_many([b"hello"], EMIT_SCAN)
    assert e.value.code == -1
