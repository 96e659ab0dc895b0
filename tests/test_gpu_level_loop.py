"""Every kernel instance of the CSE level loop (csrc/cse.cu, CseKernel) on inputs the oracle can check.

The host picks the instance from the frontier size, so most of them run only at sizes the oracle cannot check.  Each
configuration below moves the thresholds (public options only) so that the instances it names run on a small input,
in both emission widths: raw counts, compared count by count with the oracle, and coder words, compared as the
archive they make.  The BCE_GPU_TRACE line of every launch names the instance, which proves it ran."""
import os
import re

import numpy as np
import pytest

from bce_b200 import host, synth
from bce_b200.gpu import OPT_MID_ENTER_NODES, OPT_NO_NARROW_KERNELS, OPT_SLOT_ENTER_NODES
from oracle import oracle

pytestmark = pytest.mark.gpu

TEXT = synth.generate("markov2-text", 200_000, 1).tobytes()


def traced(capfd, fn):
    """Runs fn with launch tracing on; returns its result and the instances that were launched."""
    capfd.readouterr()
    os.environ["BCE_GPU_TRACE"] = "1"
    try:
        out = fn()
    finally:
        os.environ["BCE_GPU_TRACE"] = "0"
    return out, set(re.findall(r"\] cse (\w+) kernel: rounds", capfd.readouterr().err))


def check_both_widths(frontend, capfd, data, options, expect):
    for opt, value in options.items():
        frontend.set_option(opt, value)
    try:
        Lo, offo, _ = oracle.bwt(data)
        want = oracle.cse(oracle.wavelet(Lo), len(data))
        (off, Cv, streams), ran = traced(capfd, lambda: frontend.compress_front(data))
        assert off == offo and Cv == want["C"]
        for i in range(8):
            assert np.array_equal(streams[i], want["streams"][i]), ("raw", i)
        st = frontend.stats()
        assert st["cse_visits"] == sum(want["visits"]) and st["cse_rounds"] == want["rounds"]
        assert expect <= ran, ("raw", sorted(expect - ran))
        archive, ran = traced(capfd, lambda: host.compress(frontend, data, threads=1))
        assert archive == oracle.compress(data)
        assert expect <= ran, ("coder", sorted(expect - ran))
    finally:
        for opt in options:
            frontend.set_option(opt, 0)


def test_narrow_instances(frontend, capfd):
    """Default thresholds: the roots go to the one-CTA kernel, growing frontiers to both cluster kernels."""
    check_both_widths(frontend, capfd, TEXT, {}, {"tiny", "cluster1", "cluster8"})


def test_mid_instances_and_512_node_tiles(frontend, capfd):
    """Cluster kernels off and an early hand-over from cse_mid_kernel: its three instances (32 / 64 / 128 nodes per
    chunk) and the wide kernel's 512-node tiles above 3000 nodes."""
    check_both_widths(frontend, capfd, TEXT, {OPT_NO_NARROW_KERNELS: 1, OPT_MID_ENTER_NODES: 3000},
                      {"mid1", "mid2", "mid4", "wide2"})


def test_slot_layout(frontend, capfd):
    check_both_widths(frontend, capfd, TEXT, {OPT_SLOT_ENTER_NODES: 2048}, {"slots"})


def test_1024_node_tiles(frontend, capfd):
    """The wide kernel's 1024-node tiles take frontiers of at least SLOT_ENTER_NODES = S when the slot layout is off,
    which it is for inputs below 8 S bytes.  Cluster and medium kernels off; the 512-node tiles hand over above 1.5 S,
    so the input's peak frontier must exceed that with S > n / 8."""
    for data in (synth.generate("uniform", 100_000, 9).tobytes(), TEXT):
        frontend.compress_front(data)
        peak = frontend.stats()["cse_peak_frontier"]
        S = len(data) // 8 + 1
        if peak > S + S // 2:
            break
    else:
        pytest.fail("no input with a peak frontier above 1.5 x n / 8")
    check_both_widths(frontend, capfd, data, {OPT_NO_NARROW_KERNELS: 1, OPT_MID_ENTER_NODES: 1, OPT_SLOT_ENTER_NODES: S},
                      {"wide4"})
