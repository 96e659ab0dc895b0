"""One long-lived context against the oracle across interleaved calls, sizes, options and context-bit tables.

The batch driver (bce_b200/batch.py) keeps one context per worker for a whole corpus: compress_many runs of small
files between compress_front runs of large ones, sizes jumping both ways, the emission mode and the context-bit table
switched on every call.  What a context carries from one call to the next is what the other GPU tests never vary on
purpose:

  * grow-only device buffers (DevBuf::ensure clears a buffer once, when it is allocated): after a larger input, text,
    bwt, ranks, scratch and the tile descriptors hold that input's bytes past n, so every kernel that reads past n
    relies on its masking and padding;
  * host-side run state (CseHost, the pinned flips, the prefetch, the resident flags, the emission mode and table);
  * non-default context-bit tables on every path that packs CODER words (compress_many, the 20-bit words, the
    resident checksum, every level-loop kernel instance);
  * the validity windows the header promises for batches and compress_many results.

A seeded random schedule runs every public operation on a pool of inputs (sizes at the word, tile and buffer-rounding
edges; the compress_many limit), with five context-bit tables and the tuning options changing as it goes; poison steps
fill every buffer with other bytes in between.  Directed sequences cover the seams a random schedule rarely hits, and
two contexts run their own schedules at once from two threads, as two batch workers do.  Every result is compared
with the oracle; the BCE_GPU_TRACE lines prove that the schedule reached every kernel instance under a non-default
table, compress_many, and both outcomes of a prefetch."""
import ctypes as C
import os
import random
import re
import threading
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass, field

import numpy as np
import pytest

from bce_b200 import Frontend, host, synth
from bce_b200.gpu import (EMIT_CODER, EMIT_RAW, EMIT_SCAN, MANY_MAX_N, OPT_EMIT_BATCH_BYTES, OPT_LOCAL_SORT_MIN,
                          OPT_MID_ENTER_NODES, OPT_NO_NARROW_KERNELS, OPT_RESIDENT_CHECKSUM, OPT_SLOT_ENTER_NODES,
                          BceGpuError, CseBatch, CseWords)
from oracle import oracle
from tests.inputs import rnd
from tests.test_gpu_parity import first_diff

pytestmark = pytest.mark.gpu

SEEDS = (1, 2, 3)
STEPS = 200
THREAD_SEEDS = (11, 12)
THREAD_STEPS = 80
M64 = (1 << 64) - 1
KERNELS = {"tiny", "cluster1", "cluster8", "mid1", "mid2", "mid4", "slots", "wide2", "wide4"}   # CseKernel (cse.cu)
OPTION_NAMES = {OPT_EMIT_BATCH_BYTES: "EMIT_BATCH_BYTES", OPT_LOCAL_SORT_MIN: "LOCAL_SORT_MIN",
                OPT_SLOT_ENTER_NODES: "SLOT_ENTER_NODES", OPT_MID_ENTER_NODES: "MID_ENTER_NODES",
                OPT_NO_NARROW_KERNELS: "NO_NARROW_KERNELS", OPT_RESIDENT_CHECKSUM: "RESIDENT_CHECKSUM"}
EMIT_BATCH_VALUES = (0, 4096, 1 << 18, 1 << 20, 8 * 20 * 210_000)


# ---- the input pool ---------------------------------------------------------------------------------------------------

def u8(b):
    return np.frombuffer(bytes(b), dtype=np.uint8).copy()


def run_then_b(n):
    T = np.full(n, ord("a"), dtype=np.uint8)
    T[-1] = ord("b")
    return T


def all_256():
    T = np.repeat(np.arange(256, dtype=np.uint8), 256)
    return T[np.random.default_rng(20).permutation(T.size)]


def high_half(n, seed):
    return (u8(rnd(n, 128, seed)) + 0x80).astype(np.uint8)


POOL = {   # name -> maker; the primitive flag is computed (is_primitive), the oracle's results in the fixture
    "n1": lambda: u8(b"\x9c"),
    "n2": lambda: u8(b"ba"),
    "n31": lambda: u8(rnd(31, 3, 1)),
    "n32": lambda: u8(rnd(32, 256, 2)),
    "n33": lambda: u8(rnd(33, 2, 3)),
    "n63": lambda: u8(rnd(63, 26, 4)),
    "n64-power": lambda: u8(rnd(8, 3, 5) * 8),
    "n65": lambda: u8(rnd(65, 4, 6)),
    "power-63": lambda: u8(rnd(7, 4, 7) * 9),
    "all-same-257": lambda: u8(b"z" * 257),
    "n16383": lambda: synth.generate("markov2-text", 16383, 11),
    "n16384": lambda: u8(rnd(16384, 4, 12)),
    "n16385": lambda: synth.generate("uniform", 16385, 13),
    "enwik-40k": lambda: synth.generate("enwik-shaped", 40000, 23),
    "high-40k": lambda: high_half(40000, 18),
    "uniform-100k": lambda: synth.generate("uniform", 100_000, 9),
    "text-200k": lambda: synth.generate("markov2-text", 200_000, 1),
    "many-a-b": lambda: run_then_b(MANY_MAX_N),             # the deepest level loop of the many path
    "many-power-64": lambda: u8(rnd(64, 256, 19) * 1024),
    "many-all-256": all_256,
    "many-2sym": lambda: u8(rnd(MANY_MAX_N, 2, 21)),
    "many-uniform": lambda: synth.generate("uniform", MANY_MAX_N, 22),   # ranks of the sort need all 16 bits
    "enwik-1MiB-5": lambda: synth.generate("enwik-shaped", (1 << 20) - 5, 14),
    "mixed-1MiB+5": lambda: synth.generate("mixed-binary", (1 << 20) + 5, 15),
    "binary-2.5MiB": lambda: u8(rnd(5 << 19, 2, 16)),     # round 1 keeps all 2.5 M rotations: tile-local sort by default
    "high-3MiB": lambda: high_half((3 << 20) + 7, 17),     # the largest: poison steps only
}
NAMES = list(POOL)
IDX = {name: i for i, name in enumerate(NAMES)}
POISON = IDX["high-3MiB"]
TEXT = IDX["text-200k"]
LOWENT = IDX["binary-2.5MiB"]
DEEP = IDX["many-a-b"]
MANY_64K = [IDX[k] for k in ("many-uniform", "many-all-256", "many-2sym", "many-power-64")]


def is_primitive(T):
    """Not an exact power: T differs from its rotation by n / q for every prime q dividing n."""
    n, m, q = T.size, T.size, 2
    primes = []
    while q * q <= m:
        if m % q == 0:
            primes.append(q)
            while m % q == 0:
                m //= q
        q += 1
    if m > 1:
        primes.append(m)
    return not any(np.array_equal(T[:n - n // p], T[n // p:]) for p in primes if p > 1 and n > 1)


def tables():
    """None (the default), all 0, all 5 (words up to 2^20 - 1), seeded random 0..5, and one whose 8 used rows all differ
    over k = 2..31 (the default's rows 0 and 1 are equal, which would hide a level / row mix-up)."""
    rng = np.random.default_rng(288)
    rows = rng.integers(0, 6, size=(9, 32), dtype=np.uint8)
    for a in range(8):
        for b in range(a):
            assert not np.array_equal(rows[a, 2:], rows[b, 2:])
    return [None, bytes(288), bytes([5] * 288), rng.integers(0, 6, size=288, dtype=np.uint8).tobytes(), rows.tobytes()]


TABLES = tables()
TABLE_NAMES = ["default", "zeros", "fives", "random", "distinct-rows"]


# ---- the oracle's side ------------------------------------------------------------------------------------------------

def oracle_base(i):
    T = POOL[NAMES[i]]()
    L, off, sa = oracle.bwt(T, want_sa=True)
    ranks = oracle.wavelet(L)
    w = oracle.cse(ranks, T.size)
    out = dict(T=T, n=T.size, primitive=is_primitive(T), off=off, C=w["C"], visits=sum(w["visits"]),
               rounds=w["rounds"], peak=w["peak_frontier"])
    if i == POISON:           # held as per-stream call counts and checksums only
        out.update(calls=[s.shape[0] for s in w["streams"]], sums=[oracle.call_checksum_fast(s) for s in w["streams"]])
    else:
        out.update(L=L, sa=sa, ranks=ranks, streams=w["streams"])
    return out


class Want:
    """The oracle's results for the pool: the base results of every input (computed once), and memoised packed words,
    archives and scan tables per (input, table)."""

    def __init__(self):
        with ThreadPoolExecutor(min(8, os.cpu_count() or 1)) as pool:
            self.base = list(pool.map(oracle_base, range(len(NAMES))))
        self.lock = threading.Lock()
        self.memo = {}
        w = self.base[DEEP]
        assert w["rounds"] <= 8 * w["n"] + 64 and w["rounds"] >= 8 * (w["n"] - 1) - 1, w["rounds"]
        assert not self.base[IDX["n64-power"]]["primitive"] and not self.base[IDX["many-power-64"]]["primitive"]
        assert all(self.base[i]["primitive"] for i in MANY_64K[:3] + [DEEP, TEXT, LOWENT])
        # the wide kernel's 1024-node tiles: an input whose peak frontier exceeds 1.5 S with S = n / 8 + 1 (see
        # test_gpu_level_loop.test_1024_node_tiles)
        for name in ("uniform-100k", "text-200k"):
            b = self.base[IDX[name]]
            S = b["n"] // 8 + 1
            if b["peak"] > S + S // 2:
                self.wide4 = (IDX[name], S)
                break
        else:
            raise AssertionError("no input with a peak frontier above 1.5 x n / 8")

    def _get(self, key, make):
        with self.lock:
            if key in self.memo:
                return self.memo[key]
        v = make()
        with self.lock:
            self.memo[key] = v
        return v

    def packed(self, i, mode, t=0):
        return self._get(("packed", i, mode, t), lambda: host.pack_counts(mode, self.base[i]["streams"], TABLES[t]))

    def archive(self, i, t=0):
        return self._get(("archive", i, t), lambda: oracle.compress(self.base[i]["T"], TABLES[t]))

    def scan_config(self, i):
        return self._get(("scan", i), lambda: host.scan_config(self.base[i]["streams"]))


# ---- the schedule -----------------------------------------------------------------------------------------------------

SINGLE_OPS = ("bwt", "wavelet", "cse", "front", "words", "words20", "scan_words", "scan", "compress", "resident",
              "unbwt", "front_prefetch")
MANY_OPS = ("many_raw", "many_coder", "many_archives")
UPLOADS = {"bwt", "front", "words", "words20", "scan_words", "scan", "compress", "resident", "front_prefetch"}
LOOP_OPS = UPLOADS - {"bwt"} | {"cse"}
TABLE_OPS = {"words", "words20", "compress", "resident", "front_prefetch", "many_coder", "many_archives"}
ARCHIVE_OPS = {"compress", "many_archives"}

# the four configurations of test_gpu_level_loop.py: options and the kernel instances they make run on their input
KERNEL_CONFIGS = ["narrow", "mid", "slots", "wide4"]
KERNEL_EXPECT = {"narrow": {"tiny", "cluster1", "cluster8"}, "mid": {"mid1", "mid2", "mid4", "wide2"},
                 "slots": {"slots"}, "wide4": {"wide4"}}


def config_options(name, wide4_S):
    o = {"narrow": {}, "mid": {OPT_NO_NARROW_KERNELS: 1, OPT_MID_ENTER_NODES: 3000},
         "slots": {OPT_SLOT_ENTER_NODES: 2048},
         "wide4": {OPT_NO_NARROW_KERNELS: 1, OPT_MID_ENTER_NODES: 1, OPT_SLOT_ENTER_NODES: wide4_S}}[name]
    return {k: o.get(k, 0) for k in (OPT_SLOT_ENTER_NODES, OPT_MID_ENTER_NODES, OPT_NO_NARROW_KERNELS)}


@dataclass
class Step:
    op: str
    inp: object = None           # pool index, or a tuple of them (many ops)
    table: int = 0
    opts: dict = field(default_factory=dict)    # option changes applied before the operation (they persist)
    prefetch: int = None         # front_prefetch: the input uploaded beside the level loop
    config: str = ""             # kernel configuration in force (for the coverage assertion)

    def describe(self):
        inp = ",".join(NAMES[i] for i in self.inp) if isinstance(self.inp, tuple) else NAMES[self.inp] if self.inp is not None else "-"
        opts = " ".join(f"{OPTION_NAMES[k]}={v}" for k, v in self.opts.items())
        pre = f" prefetch={NAMES[self.prefetch]}" if self.prefetch is not None else ""
        return f"{self.op}({inp}) table={TABLE_NAMES[self.table]}{pre}{' set ' + opts if opts else ''}"


def schedule(seed, want, steps, poison, max_n=1 << 30):
    """A deterministic sequence of steps.  Every 10th step is a poison step (if asked for); every 8th step runs a table-
    dependent level-loop operation with a non-default table under the next of the four kernel configurations on its
    input, so that across a seed every kernel instance runs under a non-default table; the others draw an operation,
    an input, a table and option changes.  A prefetch is followed by a step on the prefetched input (adopted) or on
    another one (discarded)."""
    r = random.Random(seed)
    wide4_i, wide4_S = want.wide4
    ids = [i for i in range(len(NAMES)) if i != POISON and want.base[i]["n"] <= max_n]
    weight = [1 if want.base[i]["n"] > (1 << 19) else 4 for i in ids]
    small = [i for i in ids if want.base[i]["n"] <= MANY_MAX_N]
    small_w = [4 if want.base[i]["n"] == MANY_MAX_N else 1 for i in small]
    cur = {"config": "narrow", OPT_NO_NARROW_KERNELS: 0}
    out, kstep, forced = [], 0, None
    for s in range(steps):
        if poison and s % 10 == 0:
            out.append(Step("poison", config=cur["config"]))
            continue
        changes = {}
        if s % 8 == 4 and forced is None:
            name = KERNEL_CONFIGS[kstep % 4]
            kstep += 1
            changes.update(config_options(name, wide4_S))
            cur["config"] = name
            step = Step(r.choice(("words", "words20", "compress", "resident")), wide4_i if name == "wide4" else TEXT,
                        r.randrange(1, len(TABLES)))
        elif s % 25 == 7 and forced is None and LOWENT in ids:
            changes[OPT_LOCAL_SORT_MIN] = 0     # the tile-local sort at its default threshold
            step = Step("bwt", LOWENT)
        else:
            if forced is not None:
                op, inp = forced
                forced = None
            else:
                op = r.choice(SINGLE_OPS + MANY_OPS)
                inp = r.choices(ids, weight)[0]
            if r.random() < 0.3:
                name = r.choice(KERNEL_CONFIGS[:3])
                if inp == wide4_i and op in LOOP_OPS and r.random() < 0.5:
                    name = "wide4"
                changes.update(config_options(name, wide4_S))
                cur["config"] = name
            if r.random() < 0.3:
                changes[OPT_EMIT_BATCH_BYTES] = r.choice(EMIT_BATCH_VALUES)
            if r.random() < 0.2:
                changes[OPT_LOCAL_SORT_MIN] = r.choice((0, 1))
            no_narrow = changes.get(OPT_NO_NARROW_KERNELS, cur[OPT_NO_NARROW_KERNELS])
            if op in MANY_OPS:
                k = r.randint(1, 6)
                inp = tuple(r.choices(small, small_w, k=k))
            elif inp == DEEP and no_narrow and op in LOOP_OPS:
                inp = TEXT                      # half a million one-node rounds are for the one-CTA kernels
            if op == "unbwt" and not want.base[inp]["primitive"]:
                op = "bwt"
            step = Step(op, inp, r.randrange(len(TABLES)) if op in TABLE_OPS else 0)
            if op == "front_prefetch":
                step.prefetch = r.choices(ids, weight)[0]
                if r.random() < 0.5:
                    forced = (r.choice(sorted(UPLOADS)), step.prefetch)
                else:
                    forced = (r.choice(sorted(UPLOADS)), r.choice([i for i in ids if i != step.prefetch]))
        cur[OPT_NO_NARROW_KERNELS] = changes.get(OPT_NO_NARROW_KERNELS, cur[OPT_NO_NARROW_KERNELS])
        step.opts = changes
        step.config = cur["config"]
        out.append(step)
    return out


# ---- the GPU's side ---------------------------------------------------------------------------------------------------

class Pinned:
    """Page-locked copies of the pool's inputs (bce_gpu_host_alloc), so that a prefetch can be adopted."""

    def __init__(self, fe, want):
        self.fe, self.ptrs, self.views = fe, [], []
        for b in want.base:
            p = fe.lib.bce_gpu_host_alloc(fe.h, b["n"])
            assert p, "bce_gpu_host_alloc failed"
            v = np.ctypeslib.as_array((C.c_uint8 * b["n"]).from_address(p))
            v[:] = b["T"]
            self.ptrs.append(p)
            self.views.append(v)

    def free(self):
        self.views = []
        for p in self.ptrs:
            self.fe.lib.bce_gpu_host_free(self.fe.h, p)
        self.ptrs = []


def same(got, want, what):
    d = first_diff(got, want)
    assert d is None, f"{what}: {d}"


def same_streams(got, want, what):
    for s in range(8):
        same(got[s], want[s], f"{what}, stream {s}")


def words_of(ptr, cnt):
    return np.ctypeslib.as_array((C.c_uint32 * cnt).from_address(C.addressof(ptr.contents))) if cnt else np.zeros(0, np.uint32)


@dataclass
class Coverage:
    kernels: set = field(default_factory=set)          # instances launched by a table-dependent op, non-default table
    config_kernels: dict = field(default_factory=dict)  # kernel configuration -> instances launched under it
    many: int = 0                                       # compress_many launches with a non-default table
    prefetch: set = field(default_factory=set)
    local_sorted: int = 0
    poison: int = 0


class Runner:
    """Runs steps on one context and checks each against the oracle.  trace(fn) runs fn and returns (result, the
    BCE_GPU_TRACE lines it printed) -- or no lines where tracing is not captured."""

    def __init__(self, fe, want, seed, trace=None):
        self.fe, self.want, self.seed = fe, want, seed
        self.trace = trace or (lambda fn: (fn(), ""))
        self.pinned = Pinned(fe, want)
        self.opts = {k: 0 for k in OPTION_NAMES}
        self.cov = Coverage()

    def close(self):
        for k in OPTION_NAMES:
            self.fe.set_option(k, 0)
        self.fe.set_emit_mode(EMIT_RAW)
        self.pinned.free()

    def set_options(self, changes):
        for k, v in changes.items():
            self.fe.set_option(k, v)
            self.opts[k] = v

    def stats(self, n, visits=0, rounds=0):
        st = self.fe.stats()
        got = (st["n"], st["cse_visits"], st["cse_rounds"])
        assert got == (n, visits, rounds), f"stats (n, cse_visits, cse_rounds) {got}, oracle {(n, visits, rounds)}"
        return st

    def run(self, steps):
        for j, step in enumerate(steps):
            try:
                self.set_options(step.opts)
                _, err = self.trace(lambda: self.do(step))
                self.account(step, err)
            except Exception as e:
                last = "\n".join(f"  step {k}: {steps[k].describe()}" for k in range(max(0, j - 10), j))
                opts = " ".join(f"{OPTION_NAMES[k]}={v}" for k, v in self.opts.items())
                raise AssertionError(f"seed {self.seed}, step {j}: {step.describe()} (options in force: {opts}) failed: "
                                     f"{type(e).__name__}: {e}\nthe steps before it:\n{last}") from e

    def account(self, step, err):
        ran = set(re.findall(r"\] cse (\w+) kernel: rounds", err))
        self.cov.config_kernels.setdefault(step.config, set()).update(ran)
        if step.op in TABLE_OPS and step.table:
            self.cov.kernels |= ran
            self.cov.many += len(re.findall(r"\] compress_many k=", err))
        for outcome in re.findall(r"\] prefetched input: [^,]+, (adopted|another input: discarded)", err):
            self.cov.prefetch.add(outcome.split()[-1])

    # -- operations ---------------------------------------------------------------------------------------------------
    def do(self, step):
        getattr(self, "op_" + step.op)(step)

    def op_poison(self, step):
        """The largest high-entropy input through compress_front in small batches, then compress_many calls over 64 KiB
        inputs: text, bwt, ranks, scratch, both emission sets and pinned flips, the many slots and arena and both many
        flips hold other bytes afterwards."""
        w = self.want.base[POISON]
        self.fe.set_option(OPT_EMIT_BATCH_BYTES, 1 << 20)
        count, acc = [0] * 8, [(0, 0)] * 8
        try:
            for item in self.fe.iter_front_batches(self.pinned.views[POISON], EMIT_RAW):
                if item[0] == "head":
                    assert (item[1], item[2]) == (w["off"], w["C"]), "poison: offset / C"
                    continue
                for s, v in enumerate(item[1]):
                    p, q = oracle.call_checksum_fast(v, count[s])
                    acc[s] = ((acc[s][0] + p) & M64, (acc[s][1] + q) & M64)
                    count[s] += v.size // 5
        finally:
            self.fe.set_option(OPT_EMIT_BATCH_BYTES, self.opts[OPT_EMIT_BATCH_BYTES])
        assert count == w["calls"] and acc == w["sums"], "poison: counts differ from the oracle's"
        self.stats(w["n"], w["visits"], w["rounds"])
        for order in (MANY_64K, MANY_64K[::-1]):
            res = self.fe.compress_front_many([self.pinned.views[i] for i in order], EMIT_RAW)
            for i, (off, Cv, streams) in zip(order, res):
                b = self.want.base[i]
                assert (off, Cv) == (b["off"], b["C"]), ("poison many", NAMES[i])
                same_streams(streams, b["streams"], f"poison many {NAMES[i]}")
        self.cov.poison += 1

    def op_bwt(self, step):
        i, b = step.inp, self.want.base[step.inp]
        L, off, sa = self.fe.bwt(self.pinned.views[i], want_sa=True)
        assert off == b["off"], ("offset", off, b["off"])
        same(L, b["L"], "BWT")
        same(sa, b["sa"], "SA")
        st = self.stats(b["n"])
        if i == LOWENT and self.opts[OPT_LOCAL_SORT_MIN] == 0:
            assert st["sort_local_elems"] > 0, "the tile-local sort did not run by default"
            self.cov.local_sorted += 1
        ranks, Cv = self.fe.wavelet(None, b["n"])          # from the BWT left on the device
        for j in range(8):
            same(ranks[j], b["ranks"][j], f"rank words of level {j} (resident BWT)")
        assert Cv == b["C"], ("C (resident BWT)", Cv, b["C"])

    def op_wavelet(self, step):
        b = self.want.base[step.inp]
        ranks, Cv = self.fe.wavelet(b["L"])
        for j in range(8):
            same(ranks[j], b["ranks"][j], f"rank words of level {j}")
        assert Cv == b["C"], ("C", Cv, b["C"])
        self.stats(b["n"])

    def op_cse(self, step):
        b = self.want.base[step.inp]
        Cv, streams = self.fe.cse(b["L"])
        assert Cv == b["C"], ("C", Cv, b["C"])
        same_streams(streams, b["streams"], "counts")
        self.stats(b["n"], b["visits"], b["rounds"])

    def op_front(self, step):
        b = self.want.base[step.inp]
        off, Cv, streams = self.fe.compress_front(self.pinned.views[step.inp])
        assert (off, Cv) == (b["off"], b["C"]), ("offset / C", off, Cv)
        same_streams(streams, b["streams"], "counts")
        self.stats(b["n"], b["visits"], b["rounds"])

    def _words(self, step, got, mode):
        b = self.want.base[step.inp]
        off, Cv, words = got
        assert (off, Cv) == (b["off"], b["C"]), ("offset / C", off, Cv)
        same_streams(words, self.want.packed(step.inp, mode, step.table if mode == EMIT_CODER else 0), "words")
        self.stats(b["n"], b["visits"], b["rounds"])

    def op_words(self, step):
        self._words(step, self.fe.compress_front_words(self.pinned.views[step.inp], EMIT_CODER, TABLES[step.table]), EMIT_CODER)

    def op_words20(self, step):
        self._words(step, self.fe.compress_front_words20(self.pinned.views[step.inp], TABLES[step.table]), EMIT_CODER)

    def op_scan_words(self, step):
        self._words(step, self.fe.compress_front_words(self.pinned.views[step.inp], EMIT_SCAN), EMIT_SCAN)

    def op_scan(self, step):
        b = self.want.base[step.inp]
        assert host.scan(self.fe, self.pinned.views[step.inp]) == self.want.scan_config(step.inp), "scan table"
        self.stats(b["n"], b["visits"], b["rounds"])

    def op_compress(self, step):
        b = self.want.base[step.inp]
        arc = host.compress(self.fe, self.pinned.views[step.inp], TABLES[step.table], threads=4)
        assert arc == self.want.archive(step.inp, step.table), "archive differs from the oracle's"
        self.stats(b["n"], b["visits"], b["rounds"])
        if b["primitive"]:
            assert host.decompress(arc) == b["T"].tobytes(), "decompressed archive differs from the input"

    def op_resident(self, step):
        b = self.want.base[step.inp]
        self.fe.set_option(OPT_RESIDENT_CHECKSUM, 1)
        self.fe.set_emit_mode(EMIT_CODER, TABLES[step.table])
        try:
            self.fe.stage_input(self.pinned.views[step.inp])
            off, total = self.fe.front_resident()
            sums = self.fe.resident_checksum()
        finally:
            self.fe.set_emit_mode(EMIT_RAW)
            self.fe.set_option(OPT_RESIDENT_CHECKSUM, self.opts[OPT_RESIDENT_CHECKSUM])
        words = self.want.packed(step.inp, EMIT_CODER, step.table)
        assert off == b["off"] and total == sum(w.size for w in words), ("offset / words", off, total)
        assert sums == [oracle.word_checksum(w) for w in words], "resident checksums differ from the oracle's words"
        self.stats(b["n"], b["visits"], b["rounds"])

    def op_unbwt(self, step):
        b = self.want.base[step.inp]
        same(self.fe.unbwt(b["ranks"], b["off"], b["n"]), b["T"], "unbwt")
        self.stats(b["n"])

    def op_front_prefetch(self, step):
        """compress_front in CODER mode with the next input's upload started beside the level loop."""
        b = self.want.base[step.inp]
        got = [[] for _ in range(8)]
        head = []

        def take(Cv, batch):
            if not head:
                head.append([int(x) for x in Cv])
            for s in range(8):
                got[s].append(words_of(batch.words[s], int(batch.count[s])).copy())

        self.fe.set_emit_mode(EMIT_CODER, TABLES[step.table])
        try:
            off, _ = self.fe.compress_front_discard(self.pinned.views[step.inp], prefetch_next=self.pinned.views[step.prefetch],
                                                    on_batch=take)
        finally:
            self.fe.set_emit_mode(EMIT_RAW)
        words = [np.concatenate(g) for g in got]
        self._words(step, (off, head[0], words), EMIT_CODER)

    def _many_stats(self, inps):
        bs = [self.want.base[i] for i in inps]
        self.stats(max(b["n"] for b in bs), sum(b["visits"] for b in bs), sum(b["rounds"] for b in bs))

    def op_many_raw(self, step):
        res = self.fe.compress_front_many([self.pinned.views[i] for i in step.inp], EMIT_RAW)
        for i, (off, Cv, streams) in zip(step.inp, res):
            b = self.want.base[i]
            assert (off, Cv) == (b["off"], b["C"]), ("offset / C", NAMES[i])
            same_streams(streams, b["streams"], f"counts of {NAMES[i]}")
        if self.fe.last_many_calls == 1:
            self._many_stats(step.inp)

    def op_many_coder(self, step):
        res = self.fe.compress_front_many([self.pinned.views[i] for i in step.inp], EMIT_CODER, TABLES[step.table])
        for i, (off, Cv, words) in zip(step.inp, res):
            b = self.want.base[i]
            assert (off, Cv) == (b["off"], b["C"]), ("offset / C", NAMES[i])
            same_streams(words, self.want.packed(i, EMIT_CODER, step.table), f"words of {NAMES[i]}")
        if self.fe.last_many_calls == 1:
            self._many_stats(step.inp)

    def op_many_archives(self, step):
        arcs = host.compress_many(self.fe, [self.pinned.views[i] for i in step.inp], TABLES[step.table], threads=4)
        for i, arc in zip(step.inp, arcs):
            assert arc == self.want.archive(i, step.table), f"archive of {NAMES[i]} differs from the oracle's"
        batch = self.opts[OPT_EMIT_BATCH_BYTES] or (1 << 30)
        if batch // 4 >= sum(24 * self.want.base[i]["n"] for i in step.inp):   # the arena holds every worst case: one call
            self._many_stats(step.inp)


# ---- fixtures ---------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def want():
    """The oracle's results of the pool, and the archives the schedules will ask for (computed in a thread pool)."""
    w = Want()
    need = set()
    for seed in SEEDS:
        for s in schedule(seed, w, STEPS, poison=True):
            if s.op in ARCHIVE_OPS:
                need |= {(i, s.table) for i in (s.inp if isinstance(s.inp, tuple) else (s.inp,))}
    for seed in THREAD_SEEDS:
        for s in schedule(seed, w, THREAD_STEPS, poison=False, max_n=1 << 18):
            if s.op in ARCHIVE_OPS:
                need |= {(i, s.table) for i in (s.inp if isinstance(s.inp, tuple) else (s.inp,))}
    with ThreadPoolExecutor(min(8, os.cpu_count() or 1)) as pool:
        list(pool.map(lambda it: w.archive(*it), sorted(need)))
    return w


def tracer(capfd):
    def run(fn):
        capfd.readouterr()
        os.environ["BCE_GPU_TRACE"] = "1"
        try:
            out = fn()
        finally:
            os.environ["BCE_GPU_TRACE"] = "0"
        return out, capfd.readouterr().err
    return run


# ---- 4. the seeded random schedule ------------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", SEEDS)
def test_random_schedule(want, capfd, seed):
    steps = schedule(seed, want, STEPS, poison=True)
    with Frontend(0) as fe:
        r = Runner(fe, want, seed, tracer(capfd))
        try:
            r.run(steps)
        finally:
            r.close()
    cov = r.cov
    # without these the schedule could stop reaching a path and still pass
    assert KERNELS <= cov.kernels, f"instances that never ran under a non-default table: {sorted(KERNELS - cov.kernels)}"
    for name, expect in KERNEL_EXPECT.items():
        assert expect <= cov.config_kernels.get(name, set()), (name, sorted(expect - cov.config_kernels.get(name, set())))
    assert cov.many > 0, "no compress_many launch with a non-default table"
    assert cov.prefetch == {"adopted", "discarded"}, f"prefetch outcomes seen: {sorted(cov.prefetch)}"
    assert cov.local_sorted > 0, "no BWT of the low-entropy input under the default LOCAL_SORT_MIN"
    assert cov.poison >= STEPS // 10


# ---- 5. directed sequences --------------------------------------------------------------------------------------------

def check_front(r, i, t=4):
    """Input i completely: raw counts, CODER words with table t, and the stats of each run."""
    r.op_front(Step("front", i))
    r.op_words(Step("words", i, t))


def test_prefetch_around_many(want, capfd):
    trace = tracer(capfd)
    B = IDX["mixed-1MiB+5"]
    with Frontend(0) as fe:
        r = Runner(fe, want, 0, trace)
        try:
            # prefetch, then compress_many: the many call overwrites the text buffer, so the prefetch is dropped
            fe.prefetch_input(r.pinned.views[B])
            r.op_many_raw(Step("many_raw", tuple(MANY_64K)))
            _, err = trace(lambda: r.op_front(Step("front", B)))
            assert "adopted" not in err, "compress_front adopted a prefetch that compress_many overwrote"
            # prefetch, then unbwt (never reads the text): the prefetch is adopted
            fe.prefetch_input(r.pinned.views[B])
            r.op_unbwt(Step("unbwt", IDX["enwik-40k"]))
            _, err = trace(lambda: r.op_front(Step("front", B)))
            assert "adopted" in err, err[-2000:]
            # prefetch while another input's counts are drained, then bwt of the prefetched input
            A = TEXT
            fe.set_option(OPT_EMIT_BATCH_BYTES, 1 << 18)
            a = want.base[A]
            count = [0] * 8
            for item in fe.iter_front_batches(r.pinned.views[A], EMIT_RAW):
                if item[0] == "head":
                    assert (item[1], item[2]) == (a["off"], a["C"])
                    fe.prefetch_input(r.pinned.views[B])
                    continue
                for s, v in enumerate(item[1]):
                    v = v.reshape(-1, 5)
                    same(v, a["streams"][s][count[s]:count[s] + v.shape[0]], f"stream {s}")
                    count[s] += v.shape[0]
            assert count == [s.shape[0] for s in a["streams"]]
            fe.set_option(OPT_EMIT_BATCH_BYTES, 0)
            _, err = trace(lambda: r.op_bwt(Step("bwt", B)))
            assert "adopted" in err, err[-2000:]
        finally:
            r.close()


def multi_run(runs=40, m=30000):
    """Runs of 40 different bytes, each ended by its own separator: about 40 nodes per level for 8 m rounds (the
    cluster kernels' range), each emitting a count."""
    return np.concatenate([np.concatenate([np.full(m, 65 + j, np.uint8), np.array([200 + j], np.uint8)]) for j in range(runs)])


def test_abandoned_runs(want, capfd):
    """A run abandoned after one batch -- its frontier in the slot layout, in cse_mid_kernel, in the cluster kernels --
    must leave nothing behind that the next runs see: a smaller input, then a larger one, checked completely."""
    trace = tracer(capfd)
    text = want.base[TEXT]["T"]
    cases = [("slots", {OPT_SLOT_ENTER_NODES: 2048, OPT_EMIT_BATCH_BYTES: 1 << 18}, text, {"slots"}),
             ("mid", {OPT_NO_NARROW_KERNELS: 1, OPT_MID_ENTER_NODES: 3000, OPT_EMIT_BATCH_BYTES: 1 << 18}, text,
              {"mid1", "mid2", "mid4"}),
             ("cluster", {OPT_EMIT_BATCH_BYTES: 4096}, multi_run(), {"cluster1", "cluster8"})]
    with Frontend(0) as fe:
        r = Runner(fe, want, 0, trace)
        try:
            for name, opts, T, target in cases:
                r.set_options(opts)
                off, Cv = C.c_uint32(), (C.c_uint32 * 8)()
                _, err = trace(lambda: fe._check(fe.lib.bce_gpu_compress_front(fe.h, T.ctypes.data, T.size, C.byref(off), Cv)))
                seen = []
                while True:
                    b = CseBatch()
                    _, err = trace(lambda: fe._check(fe.lib.bce_gpu_cse_next(fe.h, C.byref(b))))
                    seen += re.findall(r"\] cse (\w+) kernel: rounds", err)
                    assert not b.done, f"{name}: the run ended before a batch was cut in {sorted(target)} (kernels {seen[-20:]})"
                    if seen and seen[-1] in target:
                        break                    # abandoned here
                check_front(r, IDX["n16385"])
                check_front(r, IDX["mixed-1MiB+5"], t=3)
                r.set_options({k: 0 for k in opts})
        finally:
            r.close()


def test_options_changed_mid_run(want):
    """Every option, and the emission table, changed between two cse_next_words calls of one run: that run's words
    follow the settings it started with, and the next runs are right under the new ones."""
    with Frontend(0) as fe:
        r = Runner(fe, want, 0)
        try:
            r.set_options({OPT_EMIT_BATCH_BYTES: 1 << 18})
            T = r.pinned.views[TEXT]
            fe.set_emit_mode(EMIT_CODER, TABLES[4])
            off, Cv = C.c_uint32(), (C.c_uint32 * 8)()
            fe._check(fe.lib.bce_gpu_compress_front(fe.h, T.ctypes.data, T.size, C.byref(off), Cv))
            got, batches = [[] for _ in range(8)], 0
            while True:
                b = CseWords()
                fe._check(fe.lib.bce_gpu_cse_next_words(fe.h, C.byref(b)))
                batches += 1
                for s in range(8):
                    got[s].append(words_of(b.words[s], int(b.count[s])).copy())
                if b.done:
                    break
                if batches == 1:
                    r.set_options({OPT_EMIT_BATCH_BYTES: 4096, OPT_LOCAL_SORT_MIN: 1, OPT_SLOT_ENTER_NODES: 2048,
                                   OPT_MID_ENTER_NODES: 3000, OPT_NO_NARROW_KERNELS: 1, OPT_RESIDENT_CHECKSUM: 1})
                    fe.set_emit_mode(EMIT_CODER, TABLES[2])
            fe.set_emit_mode(EMIT_RAW)
            assert batches > 1
            r._words(Step("words", TEXT, 4), (int(off.value), [int(x) for x in Cv], [np.concatenate(g) for g in got]), EMIT_CODER)
            for i in (IDX["enwik-40k"], IDX["uniform-100k"]):
                check_front(r, i, t=3)
                r.op_bwt(Step("bwt", i))
                r.op_resident(Step("resident", i, 1))
            r.op_many_coder(Step("many_coder", (IDX["n65"], IDX["many-2sym"]), 4))
        finally:
            r.close()


def test_validity_windows(want):
    """A batch of cse_next_words, and the ManyResult words of a compress_many call, stay valid until the call after the
    next: the views of call j (not copies) still hold what they held once call j + 1 has returned."""
    with Frontend(0) as fe:
        r = Runner(fe, want, 0)
        try:
            r.set_options({OPT_EMIT_BATCH_BYTES: 4096})
            big = IDX["enwik-1MiB-5"]
            T = r.pinned.views[big]
            fe.set_emit_mode(EMIT_CODER, TABLES[3])
            off, Cv = C.c_uint32(), (C.c_uint32 * 8)()
            fe._check(fe.lib.bce_gpu_compress_front(fe.h, T.ctypes.data, T.size, C.byref(off), Cv))
            got, prev, batches = [[] for _ in range(8)], None, 0
            while True:
                b = CseWords()
                fe._check(fe.lib.bce_gpu_cse_next_words(fe.h, C.byref(b)))
                batches += 1
                views = [words_of(b.words[s], int(b.count[s])) for s in range(8)]
                copies = [v.copy() for v in views]
                if prev is not None:
                    for s in range(8):
                        same(prev[0][s], prev[1][s], f"batch {batches - 1}, stream {s}, after batch {batches} arrived")
                prev = (views, copies)
                for s in range(8):
                    got[s].append(copies[s])
                if b.done:
                    break
            fe.set_emit_mode(EMIT_RAW)
            assert batches >= 3, batches
            r._words(Step("words", big, 3), (int(off.value), [int(x) for x in Cv], [np.concatenate(g) for g in got]), EMIT_CODER)

            r.set_options({OPT_EMIT_BATCH_BYTES: 0})
            calls = [tuple(MANY_64K[:2]) + (IDX["n33"],), (IDX["many-a-b"], IDX["n1"]), tuple(MANY_64K[2:])]
            fe.set_emit_mode(EMIT_CODER, TABLES[4])
            prev = None
            for inps in calls:
                out = fe.compress_many_call([r.pinned.views[i] for i in inps])
                res = []
                for j, i in enumerate(inps):
                    assert out[j].done, NAMES[i]
                    views = [words_of(out[j].words[s], int(out[j].count[s])) for s in range(8)]
                    same_streams([v.copy() for v in views], want.packed(i, EMIT_CODER, 4), f"many words of {NAMES[i]}")
                    res.append((i, views, [v.copy() for v in views]))
                if prev is not None:
                    for i, views, copies in prev:
                        same_streams(views, copies, f"many words of {NAMES[i]} after the next call")
                prev = res
            fe.set_emit_mode(EMIT_RAW)
        finally:
            r.close()


def test_emission_state_after_every_kind_of_call(want):
    """After any call that ran with a non-default table, set_emit_mode(CODER, None) means the default table again."""
    X = TABLES[4]
    with Frontend(0) as fe:
        r = Runner(fe, want, 0)
        v = r.pinned.views
        small = (IDX["n65"], IDX["many-uniform"])

        def with_table(fn):
            fe.set_emit_mode(EMIT_CODER, X)
            try:
                fn()
            finally:
                fe.set_emit_mode(EMIT_RAW)

        kinds = {
            "front words": lambda: fe.compress_front_words(v[IDX["enwik-40k"]], EMIT_CODER, X),
            "20-bit words": lambda: fe.compress_front_words20(v[IDX["enwik-40k"]], X),
            "compress_many": lambda: fe.compress_front_many([v[i] for i in small], EMIT_CODER, X),
            "host.compress": lambda: host.compress(fe, v[IDX["enwik-40k"]], X, threads=2),
            "host.compress_many": lambda: host.compress_many(fe, [v[i] for i in small], X, threads=2),
            "host.scan": lambda: with_table(lambda: host.scan(fe, v[IDX["enwik-40k"]])),
            "front_resident": lambda: with_table(lambda: (fe.stage_input(v[IDX["n16384"]]), fe.front_resident())),
        }
        try:
            for kind, fn in kinds.items():
                fn()
                try:
                    r.op_words(Step("words", IDX["n16383"], 0))
                    r.op_many_coder(Step("many_coder", (IDX["many-all-256"], IDX["n31"]), 0))
                    r.op_compress(Step("compress", IDX["n16385"], 0))
                except AssertionError as e:
                    raise AssertionError(f"after {kind} with a non-default table: {e}") from e
        finally:
            r.close()


def test_calls_after_error_codes(want):
    """An error code leaves the context usable: each failed call is followed by a correct one."""
    with Frontend(0) as fe:
        r = Runner(fe, want, 0)
        try:
            r.op_front(Step("front", IDX["enwik-40k"]))
            with pytest.raises(BceGpuError) as e:
                fe.compress_many_call([r.pinned.views[IDX["n33"]], np.zeros(MANY_MAX_N + 1, np.uint8)])
            assert e.value.code == -1
            r.op_many_raw(Step("many_raw", (IDX["n33"], IDX["many-2sym"])))

            with pytest.raises(BceGpuError) as e:             # the many call left no BWT on the device, not even enwik-40k's
                fe.wavelet(None, want.base[IDX["enwik-40k"]]["n"])
            assert e.value.code == -4
            r.op_wavelet(Step("wavelet", IDX["many-2sym"]))
            r.op_cse(Step("cse", IDX["n16383"]))
            r.op_front(Step("front", IDX["n16384"]))

            b = want.base[IDX["enwik-1MiB-5"]]                # a scratch limit that leaves the frontier no room
            r.op_bwt(Step("bwt", IDX["enwik-1MiB-5"]))
            fe.set_scratch_limit(3 << 20)
            Cv = (C.c_uint32 * 8)()
            rc = fe.lib.bce_gpu_cse_begin(fe.h, None, b["n"], Cv)
            batch = CseBatch()
            while rc == 0 and not batch.done:
                rc = fe.lib.bce_gpu_cse_next(fe.h, C.byref(batch))
            assert rc in (-2, -5), rc
            fe.set_scratch_limit(0)
            r.op_cse(Step("cse", IDX["enwik-1MiB-5"]))
            check_front(r, IDX["enwik-1MiB-5"])
            check_front(r, IDX["n2"])
            r.op_compress(Step("compress", IDX["enwik-40k"], 3))
        finally:
            fe.set_scratch_limit(0)
            r.close()


def test_many_inputs_per_cta(want, capfd):
    """More inputs than the grid has CTAs, so that each CTA takes input after input (largest first) and reads rank words
    an earlier input of its own left behind: every input against the oracle, raw counts and CODER words."""
    rr = random.Random(7)
    pool = [i for i in range(len(NAMES)) if want.base[i]["n"] <= MANY_MAX_N]
    extra = [u8(rnd(rr.randint(1, 300), rr.choice((2, 4, 26, 256)), 1000 + j)) for j in range(60)]
    items = [want.base[rr.choice(pool)]["T"] if rr.random() < 0.3 else extra[rr.randrange(len(extra))] for _ in range(3000)]
    ref = {}
    for T in items:
        key = T.tobytes()
        if key not in ref:
            L, off, _ = oracle.bwt(T)
            w = oracle.cse(oracle.wavelet(L), T.size)
            ref[key] = (off, w["C"], w["streams"])
    trace = tracer(capfd)
    with Frontend(0) as fe:
        res, err = trace(lambda: fe.compress_front_many(items, EMIT_RAW))
        k, ctas = map(int, re.findall(r"\] compress_many k=(\d+) largest=\d+ ctas=(\d+)", err)[0])
        assert k > ctas, (k, ctas)
        for j, (T, (off, Cv, streams)) in enumerate(zip(items, res)):
            woff, wC, wstreams = ref[T.tobytes()]
            assert (off, Cv) == (woff, wC), j
            same_streams(streams, wstreams, f"input {j} (n = {T.size})")
        res = fe.compress_front_many(items, EMIT_CODER, TABLES[4])
        packed = {}
        for j, (T, (off, Cv, words)) in enumerate(zip(items, res)):
            key = T.tobytes()
            if key not in packed:
                packed[key] = host.pack_counts(EMIT_CODER, ref[key][2], TABLES[4])
            same_streams(words, packed[key], f"input {j} (n = {T.size}), CODER")


# ---- 6. two contexts in two threads -----------------------------------------------------------------------------------

def test_two_contexts_in_two_threads(want):
    """Two contexts on one GPU, each running its own schedule from its own thread, as two batch workers do.  Contention
    may slow the grid barriers and chained scans down, never change a result; BCE_GPU_E_INTERNAL would be a finding."""
    errors = []

    def worker(seed):
        try:
            with Frontend(0) as fe:
                r = Runner(fe, want, seed)
                try:
                    r.run(schedule(seed, want, THREAD_STEPS, poison=False, max_n=1 << 18))
                finally:
                    r.close()
        except BaseException as e:           # reported from the main thread
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(s,)) for s in THREAD_SEEDS]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, "\n\n".join(str(e) for e in errors)
