"""The front end's large-input paths, count by count against the oracle, at the sizes that switch them on.

Several branches of the suffix sort and of the level loop take over only above a size threshold, so no input the other
parity tests use reaches them:

  * suffix_sort.cu: (idx, rank) pairs binned by the top 8 bits of idx and scattered from there (m >= 2^23 and
    4n > 64 MiB), round 0's arithmetic bin sizes, the partition histogram from the tile-local sort or from
    rekey_kernel, the index tie-break round with a working set of millions, round 0 without any radix pass (one
    repeated byte), and the BWT through the inverse suffix array (binned) instead of the gather (n >= 2^23, no
    tie-break);
  * cse.cu: the slot layout at the default SLOT_ENTER_NODES, the flat layout capped at 16 Mi nodes beside it, the
    hosted two-set emission with the batch cut where the frontier collapses, millions of rounds in cse_tiny_kernel,
    and the wide kernel alone when the scratch limit leaves no room for the slots.

Each case runs at a size (or with a shape) that reaches the paths it names, checks everything the oracle can check
(BWT, SA, rank words, every count of every stream or per-stream checksums, the archive, the device-resident
emission, the inverse) and asserts from the stats and the BCE_GPU_TRACE lines that those paths ran: a threshold that
moves must make a case fail, not pass without reaching its path.

Inputs are made inside the tests, never at import.  The oracle's results are computed in a thread pool (its C calls
release the GIL) while the GPU works on the cases before, and each case drops them when it is done."""
import os
import re
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass

import numpy as np
import pytest

from bce_b200 import host, synth
from bce_b200.gpu import EMIT_CODER, EMIT_RAW, OPT_EMIT_BATCH_BYTES, OPT_RESIDENT_CHECKSUM
from oracle import oracle
from tests.test_gpu_parity import first_diff

pytestmark = pytest.mark.gpu

P23, P24 = 1 << 23, 1 << 24
SLOT_ENTER_NODES = 2_000_000       # default of BCE_GPU_OPT_SLOT_ENTER_NODES (ctx.h)
M64 = (1 << 64) - 1


def seeded(n, sigma, seed):
    return np.random.default_rng(seed).integers(0, sigma, size=n, dtype=np.uint8)


def power_17():
    return np.tile(seeded(1_000_003, 4, 17), 17)


def near_power_17():
    T = power_17()
    T[T.size // 2] ^= 1            # primitive now, but every rotation stays tied with a shifted copy for ~15 periods
    return T


def run_then_b(n):
    T = np.full(n, ord("a"), dtype=np.uint8)
    T[-1] = ord("b")
    return T


def tail_repeat():
    block = seeded(1 << 20, 256, 23)
    T = np.concatenate([block, block])
    T[(1 << 20) + (1 << 19)] ^= 0x40
    return T


@dataclass
class Case:
    make: object                 # () -> uint8 array
    primitive: bool
    counts: str = ""             # "" (no level loop), "full" (count by count) or "sums" (per-stream checksums)
    batched: bool = False        # counts again with small emission batches
    resident: bool = False       # EMIT_CODER device-resident run against the oracle's packed words
    scratch: bool = False        # counts again under a scratch limit that leaves no room for the slot layout


CASES = {
    "uniform-2^23-1": Case(lambda: synth.generate("uniform", P23 - 1, 31), True),
    "uniform-2^23": Case(lambda: synth.generate("uniform", P23, 32), True),
    "uniform-2^24": Case(lambda: synth.generate("uniform", P24, 33), True),
    "uniform-2^24+1": Case(lambda: synth.generate("uniform", P24 + 1, 34), True, counts="sums"),
    "binary-2^24+1": Case(lambda: seeded(P24 + 1, 2, 35), True),
    "markov-20M": Case(lambda: synth.generate("markov2-text", 20_000_000, 1), True, counts="full", batched=True, scratch=True),
    "markov-2^25+17": Case(lambda: synth.generate("markov2-text", (1 << 25) + 17, 2), True, counts="sums"),
    "mixed-24M": Case(lambda: synth.generate("mixed-binary", 24_000_005, 4), True, counts="full", resident=True),
    "power-17": Case(power_17, False, counts="full", resident=True),
    "one-byte": Case(lambda: np.full(P24 + 3, ord("z"), dtype=np.uint8), False, counts="full", resident=True),
    "near-power-17": Case(near_power_17, True),
    "run-then-b": Case(lambda: run_then_b(P24 + 1), True),
    "tail-1M": Case(lambda: run_then_b((1 << 20) + 3), True, counts="full", resident=True),
    "tail-repeat": Case(tail_repeat, True, counts="full", batched=True),
}


# ---- the oracle's side ------------------------------------------------------------------------------------------------

def oracle_case(name):
    """Everything the oracle has to say about one case: BWT, SA, rank words, and for level-loop cases the counts (or
    their per-stream call counts and checksums), visits, rounds, the packed words' checksums and the archive."""
    case = CASES[name]
    T = case.make()
    L, off, sa = oracle.bwt(T, want_sa=True)
    out = dict(L=L, off=off, sa=sa, ranks=oracle.wavelet(L))
    if case.counts:
        want = oracle.cse(out["ranks"], T.size)
        out.update(C=want["C"], visits=sum(want["visits"]), rounds=want["rounds"], peak=want["peak_frontier"])
        streams = want.pop("streams")
        if case.counts == "full":
            out["streams"] = streams
        else:
            out["calls"] = [s.shape[0] for s in streams]
            out["sums"] = [oracle.call_checksum_fast(s) for s in streams]
        if case.resident:
            words = host.pack_counts(EMIT_CODER, streams)
            out["resident"] = ([oracle.word_checksum(w) for w in words], sum(w.size for w in words))
        del streams
        out["archive"] = oracle.compress(T)
    return out


class OracleResults:
    """The oracle runs ahead of the GPU by at most AHEAD cases, so that at most that many cases' results are held."""
    AHEAD = 4

    def __init__(self, names):
        self.names = names
        self.pool = ThreadPoolExecutor(min(self.AHEAD, os.cpu_count() or 1))
        self.futures = {}

    def take(self, name):
        """The case's results; the cache forgets them (large arrays are freed once the case is done)."""
        at = self.names.index(name) if name in self.names else len(self.names)
        for nxt in [name] + self.names[at + 1:at + 1 + self.AHEAD]:
            if nxt not in self.futures:
                self.futures[nxt] = self.pool.submit(oracle_case, nxt)
        return self.futures.pop(name).result()


@pytest.fixture(scope="module")
def oracle_results(request):
    """The oracle's results of the cases selected in this module, computed in the order the cases run."""
    names = [it.callspec.params["name"] for it in request.session.items
             if it.module is request.module and hasattr(it, "callspec") and "name" in it.callspec.params]
    res = OracleResults(list(dict.fromkeys(names)))
    yield res
    for f in res.futures.values():
        f.cancel()
    res.pool.shutdown(wait=True)


# ---- the GPU's side -----------------------------------------------------------------------------------------------------

def traced(capfd, fn):
    """Runs fn with launch tracing on; returns its result and the trace (stderr)."""
    capfd.readouterr()
    os.environ["BCE_GPU_TRACE"] = "1"
    try:
        out = fn()
    finally:
        os.environ["BCE_GPU_TRACE"] = "0"
    return out, capfd.readouterr().err


@dataclass
class SortPath:
    rounds: list        # per round: (m, tiebreak, partitioned)
    scatters: int       # binned rank scatters
    bwt: str            # "binned" or "gather"
    shift: int          # binned BWT: bin of position i is i >> shift


def sort_path(err):
    tb = {int(r): (int(m), int(t)) for r, m, t in re.findall(r"\] sort round (\d+) m=(\d+) h=\d+ tiebreak=(\d)", err)}
    part = {int(r): int(p) for r, p in re.findall(r"\] rerank round (\d+) m=\d+: .* partitioned=(\d)\)", err)}
    bwt = re.findall(r"\] bwt (binned|gather)(?: shift=(\d+))?", err)
    assert len(bwt) == 1 and sorted(tb) == sorted(part) == list(range(len(tb))), "suffix sort trace incomplete"
    return SortPath([(tb[r][0], tb[r][1], part[r]) for r in range(len(tb))], err.count("] rank scatter:"),
                    bwt[0][0], int(bwt[0][1] or -1))


def loop_kernels(err):
    """{kernel instance: rounds it ran} from the level loop's trace."""
    ran = {}
    for k, a, b in re.findall(r"\] cse (\w+) kernel: rounds (\d+)\.\.(\d+)", err):
        ran[k] = ran.get(k, 0) + int(b) - int(a)
    return ran


def cse_begin(err):
    m = re.findall(r"\] cse_begin n=\d+ cap=(\d+) ecap_words=\d+ sets=(\d)", err)
    assert len(m) == 1
    return int(m[0][0]), int(m[0][1])


def drain_and_compare(frontend, T, want):
    """Fused front end with RAW emission, batch by batch: every count of every stream against the oracle's as the
    batch arrives (or, for inputs whose counts are too many to hold twice, the per-stream call counts and checksums).
    Returns the number of batches."""
    full = "streams" in want
    count = [0] * 8
    acc = [(0, 0)] * 8
    batches = 0
    with ThreadPoolExecutor(8) as pool:
        for item in frontend.iter_front_batches(T, EMIT_RAW):
            if item[0] == "head":
                assert item[1] == want["off"] and item[2] == want["C"], (item[1:], want["off"], want["C"])
                continue
            views = [v.reshape(-1, 5) for v in item[1]]
            batches += 1
            if full:
                for i in range(8):
                    k = views[i].shape[0]
                    ref = want["streams"][i][count[i]:count[i] + k]
                    d = first_diff(views[i], ref)
                    assert d is None, f"stream {i}, batch {batches}, counts from {count[i]}: {d}"
            else:
                parts = list(pool.map(lambda i: oracle.call_checksum_fast(views[i], count[i]), range(8)))
                acc = [((a + p) & M64, (b + q) & M64) for (a, b), (p, q) in zip(acc, parts)]
            for i in range(8):
                count[i] += views[i].shape[0]
    if full:
        assert count == [s.shape[0] for s in want["streams"]], (count, [s.shape[0] for s in want["streams"]])
    else:
        assert count == want["calls"], (count, want["calls"])
        assert acc == want["sums"], "per-stream checksums of the counts differ from the oracle's"
    st = frontend.stats()
    assert st["cse_visits"] == want["visits"] and st["cse_rounds"] == want["rounds"], \
        (st["cse_visits"], want["visits"], st["cse_rounds"], want["rounds"])
    return batches


def flat_only_scratch_limit(n, peak):
    """A scratch budget under which cse_begin (cse.cu) keeps a flat frontier that holds every level of this input but
    sets aside no slot layout, for RAW and CODER emission alike (n between 16 M and 32 M bytes).

    cse_begin sizes the flat frontier first: cap = n/2 + 4 nodes per level (rounded up to 4; below the 16 Mi cap that
    applies beside the slots), 48 arrays of cap words (three per node, two parities, eight levels), halved while they
    take more than budget / 2.  The slot layout then needs arena_cap >= 8 x SLOT_ENTER_NODES places, at per_place bytes
    each (24 for the two arenas, wmax x 2 for the E-slots: 5 words for RAW counts, 3 for CODER words, 1 for the
    directories), out of half of what the frontier and the tile descriptors leave.

    With the full cap the frontier alone needs budget >= 96 x need(cap), which leaves at least 48 x need(cap) > 16 M x
    35 bytes for the slots: they always fit.  So the budget is twice the frontier at cap / 2 -- halved exactly once,
    the frontier at cap / 2 fills half of it -- and the other half, less the descriptors, is too small for the
    slots."""
    def need(count, elem):                  # Carver::need
        return (count * elem + 255) & ~255

    def frontier_bytes(cap):
        return 48 * need(cap, 4)

    cap_full = (n // 2 + 4 + 3) & ~3
    assert cap_full <= 16 << 20
    cap = (cap_full // 2 + 3) & ~3
    limit = 2 * frontier_bytes(cap)
    assert frontier_bytes(cap_full) > limit // 2 and frontier_bytes(cap) <= limit // 2
    left = limit - frontier_bytes(cap) - need(3 * 8 * (cap // 256 + 2), 8)      # desc_tiles for CS_THREADS = 256
    for wmax in (5, 3):
        per_place = 2 * 12 + (wmax * 4) // 2 + 1
        assert (left // 2) // per_place < 8 * SLOT_ENTER_NODES, wmax
    assert peak <= cap, "the flat frontier at cap / 2 would not hold the widest round"
    return limit, cap


# ---- the paths each case must reach ------------------------------------------------------------------------------------

def check_sort_path(name, n, sp, st):
    m = st["sort_m"]
    assert [r[0] for r in sp.rounds] == m and st["sort_rounds"] == len(m)
    part = [r for r, (_, _, p) in enumerate(sp.rounds) if p]
    tie = [r for r, (_, t, _) in enumerate(sp.rounds) if t]
    big = n * 4 > 64 << 20
    # the partitioned re-rank follows the sizes exactly, and every partitioned round scatters from the bins
    assert part == [r for r in range(len(m)) if big and m[r] >= P23], (part, m)
    assert sp.scatters == len(part)
    want_bwt = "binned" if n >= P23 and not tie else "gather"
    assert sp.bwt == want_bwt, (sp.bwt, tie)
    if sp.bwt == "binned":
        assert sp.shift == max(0, (n - 1).bit_length() - 8)

    if name == "uniform-2^23-1":
        assert sp.bwt == "gather" and not part
    elif name in ("uniform-2^23", "uniform-2^24"):
        assert sp.bwt == "binned" and sp.shift == {"uniform-2^23": 15, "uniform-2^24": 16}[name] and not part
    elif name == "uniform-2^24+1":
        assert 0 in part and sp.shift == 17 and (n - 1) >> 17 == 128      # 129 bins, the last with one index
    elif name == "binary-2^24+1":
        local = [r for r in range(1, len(m)) if m[r] >= P23 and st["sort_radix_passes"][r] == 0]
        rekey = [r for r in range(1, len(m)) if m[r] >= P23 and st["sort_radix_passes"][r] > 0]
        assert local and rekey, (m, st["sort_radix_passes"])
        assert set(local + rekey) <= set(part)
    elif name in ("power-17", "one-byte"):
        assert tie and m[tie[0]] == n and tie[0] in part and sp.bwt == "gather", (tie, m)
        if name == "one-byte":
            assert st["sort_passes"][0] == 0, st["sort_passes"]     # every window equal: round 0 runs no radix pass
    elif name in ("near-power-17", "run-then-b"):
        assert not tie and sp.bwt == "binned" and sp.shift == 17
        assert sum(x >= P23 for x in m) >= 20, m                   # ties survive until h is near n


def check_loop_path(name, n, ran, begin, st, want):
    cap, sets = begin
    assert sets == 2                                   # hosted emission: two emission sets alternate
    peak = st["cse_peak_frontier"]
    if name in ("uniform-2^24+1", "markov-20M", "markov-2^25+17", "mixed-24M"):
        assert n >= 8 * SLOT_ENTER_NODES and peak >= SLOT_ENTER_NODES and "slots" in ran, (peak, ran)
        assert want["peak"] >= SLOT_ENTER_NODES
    if name == "markov-2^25+17":
        assert n // 2 + 4 > 16 << 20 and cap == 16 << 20, cap       # flat layout capped beside the slots
    if name == "uniform-2^24+1":
        assert peak >= 20_000_000, peak
    if name == "mixed-24M":
        assert peak >= 10_000_000 and want["rounds"] >= 24_000, (peak, want["rounds"])
    if name == "power-17":
        assert want["visits"] != 8 * (n - 1)
    if name == "one-byte":
        assert all(s.shape[0] == 0 for s in want["streams"])
    if name in ("tail-1M", "tail-repeat"):
        assert ran.get("tiny", 0) >= 7_000_000, ran                 # millions of rounds of one or two nodes
    if name == "tail-1M":
        assert want["visits"] == 8 * (n - 1) and want["rounds"] >= 8 * (n - 1) - 1, (want["visits"], want["rounds"])


@pytest.mark.parametrize("name", list(CASES))
def test_scale_path(frontend, capfd, oracle_results, name):
    case = CASES[name]
    T = case.make()
    n = T.size
    want = oracle_results.take(name)

    # BWT, offset and suffix array; the sort's path
    (L, off, sa), err = traced(capfd, lambda: frontend.bwt(T, want_sa=True))
    st = frontend.stats()
    assert off == want["off"]
    assert first_diff(L, want["L"]) is None, ("L", first_diff(L, want["L"]))
    assert first_diff(sa, want["sa"]) is None, ("SA", first_diff(sa, want["sa"]))
    del L, sa, want["sa"]
    check_sort_path(name, n, sort_path(err), st)

    # rank words of the wavelet matrix, and C
    ranks, Cv = frontend.wavelet(want["L"])
    for j in range(8):
        assert first_diff(ranks[j], want["ranks"][j]) is None, (j, first_diff(ranks[j], want["ranks"][j]))
    if case.counts:
        assert Cv == want["C"]
    del ranks

    if case.primitive:
        out = frontend.unbwt(want["ranks"], want["off"], n)
        assert first_diff(out, T) is None, ("unbwt", first_diff(out, T))
        del out
    del want["ranks"], want["L"]

    if not case.counts:
        return
    _, err = traced(capfd, lambda: drain_and_compare(frontend, T, want))
    check_loop_path(name, n, loop_kernels(err), cse_begin(err), frontend.stats(), want)
    if name == "markov-20M":
        assert re.search(r"\] cse: batch cut at round \d+", err), "no batch cut where the frontier collapsed"

    if case.batched:
        frontend.set_option(OPT_EMIT_BATCH_BYTES, 1 << 20)
        try:
            batches, err = traced(capfd, lambda: drain_and_compare(frontend, T, want))
        finally:
            frontend.set_option(OPT_EMIT_BATCH_BYTES, 0)
        # the batch size grows to what one round needs, so count the drains where they happen: the kernel that
        # returns kCseDrain (status 2) stopped to hand a full batch over and is entered again from where it stopped
        drained = set(re.findall(r"\] cse (\w+) kernel: rounds \d+\.\.\d+ status=2 ", err))
        assert batches >= 8, batches
        if name == "markov-20M":
            assert "slots" in drained, (batches, drained)
        else:       # the tail's single-node rounds emit too little to fill a batch; cse_mid_kernel drains before it
            assert drained & {"mid1", "mid2", "mid4"}, (batches, drained)

    if case.scratch:
        limit, cap = flat_only_scratch_limit(n, want["peak"])
        frontend.set_scratch_limit(limit)
        try:
            _, err = traced(capfd, lambda: drain_and_compare(frontend, T, want))
        finally:
            frontend.set_scratch_limit(0)
        ran = loop_kernels(err)
        assert "wide4" in ran and "slots" not in ran, ran
        assert cse_begin(err)[0] == cap

    if case.resident:
        frontend.set_option(OPT_RESIDENT_CHECKSUM, 1)
        frontend.set_emit_mode(EMIT_CODER)
        try:
            frontend.stage_input(T)
            off2, total = frontend.front_resident()
            got = frontend.resident_checksum()
        finally:
            frontend.set_emit_mode(EMIT_RAW)
            frontend.set_option(OPT_RESIDENT_CHECKSUM, 0)
        sums, words = want["resident"]
        assert off2 == want["off"] and total == words, (off2, total, words)
        assert got == sums, "resident emission differs from the oracle's packed words"

    assert host.compress(frontend, T, threads=8) == want["archive"], "archive differs from the oracle's"
