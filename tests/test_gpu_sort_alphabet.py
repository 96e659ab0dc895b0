"""The suffix sort's round 0 on small alphabets and its re-rank at tile edges, against the oracle's SA and BWT.

Round 0 sorts windows of 7-bit symbol codes (7 radix digits) when 2 .. 128 byte values occur and windows of bytes
(8 digits) otherwise; the digit histograms of the coded keys come from the text's code-pair histogram.  The cases
sit on both sides of that choice, with the byte values 0x00 and 0xFF among the symbols (their codes are the two ends
of the code range), and check from the trace and the stats which keys round 0 used.

The re-rank reads one head mask per row of 32 slots and per-tile carries scanned before it runs (4096 slots per
tile): working sets below one tile, one slot either side of whole tiles, and groups that span many tiles."""
import os
import re

import numpy as np
import pytest

from bce_b200 import synth
from oracle import oracle
from tests.test_gpu_parity import first_diff

pytestmark = pytest.mark.gpu

RR_TILE = 4096
P23 = 1 << 23


def alphabet(n, sigma, seed):
    """n bytes drawn from sigma byte values that include 0x00 and 0xFF (sigma >= 2)."""
    rng = np.random.default_rng(seed)
    values = np.concatenate([[0, 255], rng.choice(np.arange(1, 255), size=sigma - 2, replace=False)]).astype(np.uint8)
    T = values[rng.integers(0, sigma, size=n)]
    T[:sigma] = values                     # every value occurs
    return T


def power3(seed):
    """An exact power over three byte values: a primitive word of 10007 bytes, 37 times."""
    w = alphabet(10_007, 3, seed)
    return np.tile(w, 37)


def run_then(n, run_byte, last_byte):
    T = np.full(n, run_byte, dtype=np.uint8)
    T[-1] = last_byte
    return T


def uniform(n, seed):
    return np.random.default_rng(seed).integers(0, 256, size=n, dtype=np.uint8)


# name: (make, keys of round 0: "codes" or "bytes")
CASES = {
    "sigma-2": (lambda: alphabet(300_001, 2, 1), "codes"),
    "sigma-64": (lambda: alphabet(300_002, 64, 2), "codes"),
    "sigma-65": (lambda: alphabet(300_003, 65, 3), "codes"),
    "sigma-127": (lambda: alphabet(300_004, 127, 4), "codes"),
    "sigma-128": (lambda: alphabet(300_005, 128, 5), "codes"),
    "sigma-129": (lambda: alphabet(300_006, 129, 6), "bytes"),
    "power3": (lambda: power3(7), "codes"),
    "enwik-2^24+5": (lambda: synth.generate("enwik-shaped", (1 << 24) + 5, 8), "codes"),
    "uniform-2^23+1": (lambda: uniform(P23 + 1, 9), "bytes"),
    # re-rank tile edges (round 0's working set is the whole text)
    "m-1000": (lambda: alphabet(1000, 5, 10), "codes"),
    "m-4095": (lambda: uniform(RR_TILE - 1, 11), "bytes"),
    "m-4097": (lambda: alphabet(RR_TILE + 1, 100, 12), "codes"),
    "m-3x4096-1": (lambda: uniform(3 * RR_TILE - 1, 13), "bytes"),
    "m-5x4096+1": (lambda: alphabet(5 * RR_TILE + 1, 3, 14), "codes"),
    "run-200k-then-b": (lambda: run_then(200_000, ord("a"), ord("b")), "codes"),
    "run-20x4096-then-00": (lambda: run_then(20 * RR_TILE, 0xFF, 0x00), "codes"),
}


def traced(capfd, fn):
    capfd.readouterr()
    os.environ["BCE_GPU_TRACE"] = "1"
    try:
        out = fn()
    finally:
        os.environ["BCE_GPU_TRACE"] = "0"
    return out, capfd.readouterr().err


@pytest.mark.parametrize("name", list(CASES))
def test_sort_alphabet(frontend, capfd, name):
    make, keys = CASES[name]
    T = make()
    (L, off, sa), err = traced(capfd, lambda: frontend.bwt(T, want_sa=True))
    Lo, offo, sao = oracle.bwt(T, want_sa=True)
    assert off == offo
    assert first_diff(sa, sao) is None, first_diff(sa, sao)
    assert first_diff(L, Lo) is None, first_diff(L, Lo)

    sigma = int(np.count_nonzero(np.bincount(T, minlength=256)))
    chosen = re.findall(r"\] round 0: (\d+) byte values, keys from (7-bit codes|bytes)", err)
    assert chosen == [(str(sigma), "7-bit codes" if keys == "codes" else "bytes")], chosen
    st = frontend.stats()
    assert st["sort_m"][0] == T.size
    # constant digits are skipped; the rest of the 7 (codes) or 8 (bytes) digits run
    assert 1 <= st["sort_passes"][0] <= (7 if keys == "codes" else 8)
    if name in ("sigma-64", "sigma-65", "sigma-127", "sigma-128", "enwik-2^24+5"):
        assert st["sort_passes"][0] == 7
    if name in ("sigma-129", "uniform-2^23+1"):
        assert st["sort_passes"][0] == 8
