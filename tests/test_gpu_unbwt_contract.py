"""bce_gpu_unbwt -- the inverse BWT of one dictionary of any size, which `bce -d`, host.decompress and every archive
above BCE_GPU_MANY_MAX_N in bce_decompress_many run -- against its contract (include/bce_gpu.h): the text is what the
host decoder's unbwt_serial (`bce -ds`, csrc/host/decode.cpp) makes of the same words, for any words,

    out[(n - 1 - k + offset) mod n] = byte of row s_k,   s_0 = 0,   s_{k+1} = clamped descent from s_k

with every bit and ones_before read at min(pos, n) and the row kept as a 32-bit value.

  * valid dictionaries (exact powers included: their LF has several cycles) against oracle.unbwt_bitwise, and the
    input where it is primitive;
  * consistent words that no BWT produced (a true rank directory over random bits: LF is a random permutation, so
    row 0's cycle has any length) and inconsistent words (what damaged archives decode to) against unbwt_clamped;
  * archives, damaged ones included, through host.decompress_many, host.decompress and the CLI against `bce -ds`.

Before every case the context inverts a different primitive text of the same size, so the scratch the text is
assembled in holds other bytes at every position: a position the kernels never write fails the case instead of
passing by luck.  stats.unbwt_serial tells which path ran: 0 for words that are a rank directory (device), 1 for the
others (the host walk)."""
import functools
import random
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from bce_b200 import build, host, synth
from bce_b200.gpu import MANY_MAX_N, BceGpuError
from oracle import oracle
from tests.inputs import rnd, small_cases

M32 = 0xFFFFFFFF
GENERATORS = ("enwik-shaped", "markov2-text", "mixed-binary", "uniform")


# ---- the clamped reference ------------------------------------------------------------------------------------------

def levels(ranks):
    return [np.ascontiguousarray(r, dtype=np.uint64) for r in ranks]


def ones_before(r, n, pos):
    p = min(pos, n)
    w = int(r[p >> 5])
    return ((w & M32) + bin((w >> 32) & ((1 << (p & 31)) - 1)).count("1")) & M32


def descend(R, zeros, n, s):
    """The clamped descent from the rows s (uint64 array of 32-bit values): (byte, next row) of every row."""
    s = s.astype(np.uint64)
    chr_ = np.zeros(s.shape, dtype=np.uint8)
    for j in range(8):
        p = np.minimum(s, np.uint64(n))
        w = R[j][p >> np.uint64(5)]
        sh = p & np.uint64(31)
        bit = (w >> (np.uint64(32) + sh)) & np.uint64(1)
        ones = ((w & np.uint64(M32)) + np.bitwise_count((w >> np.uint64(32)) & ((np.uint64(1) << sh) - np.uint64(1)))) \
            & np.uint64(M32)
        chr_ |= bit.astype(np.uint8) << np.uint8(j)
        s = np.where(bit == 1, (np.uint64(zeros[j]) + ones) & np.uint64(M32), (s - ones) & np.uint64(M32))
    return chr_, s


def walk(ranks, n):
    """The bytes of steps 0 .. p-1 and p: the walk returns to row 0 after p steps (then repeats), or p = n."""
    R = levels(ranks)
    zeros = [(n - ones_before(R[j], n, n)) & M32 for j in range(8)]
    L = np.empty(n, dtype=np.uint8)
    LF = np.empty(n, dtype=np.uint64)
    for a in range(0, n, 1 << 22):
        L[a:a + (1 << 22)], LF[a:a + (1 << 22)] = descend(R, zeros, n, np.arange(a, min(n, a + (1 << 22)), dtype=np.uint64))
    far = {}                                      # rows >= n: every read of their descent hits word n / 32
    steps = bytearray(n)
    s, p = 0, n
    for k in range(n):
        if s < n:
            c, s = int(L[s]), int(LF[s])
        else:
            if s not in far:
                c1, t1 = descend(R, zeros, n, np.array([s], dtype=np.uint64))
                far[s] = (int(c1[0]), int(t1[0]))
            c, s = far[s]
        steps[k] = c
        if s == 0:
            p = k + 1
            break
    return np.frombuffer(bytes(steps[:p]), dtype=np.uint8), p


def unbwt_clamped(ranks, offset, n):
    """The contract restated: LF and the byte of every row < n vectorised, the walk in Python."""
    seq, _ = walk(ranks, n)
    out = np.empty(n, dtype=np.uint8)
    out[(n - 1 - np.arange(n, dtype=np.int64) + offset) % n] = np.resize(seq, n)
    return out.tobytes()


def consistent(ranks, n):
    """The words are a rank directory: base(W[0]) = 0, base(W[i+1]) = base(W[i]) + popc(data(W[i])) for i < n/32."""
    m = n // 32
    for r in levels(ranks):
        base = r & np.uint64(M32)
        pc = np.bitwise_count(r[:m] >> np.uint64(32)).astype(np.uint64)
        if base[0] != 0 or not np.array_equal(base[1:m + 1], (base[:m] + pc) & np.uint64(M32)):
            return False
    return True


def rank_words(data):
    """uint32 data words of one level (n // 32 + 1) -> rank words with a true directory."""
    d = data.astype(np.uint64)
    base = np.concatenate([[0], np.cumsum(np.bitwise_count(d[:-1]).astype(np.uint64))]).astype(np.uint64)
    return (d << np.uint64(32)) | base


def random_consistent(n, ands, rng):
    """Random data bits (each set with probability 2^-ands) under a correct rank directory, bits at and beyond n
    included: LF is a random permutation of [0, n)."""
    w = n // 32 + 1
    out = []
    for _ in range(8):
        d = np.full(w, M32, dtype=np.uint64)
        for _ in range(ands):
            d &= rng.integers(0, 2**32, size=w, dtype=np.uint64)
        out.append(rank_words(d))
    return out


def period(ranks, n):
    return walk(ranks, n)[1]


def primitive(data):
    return data not in (data + data)[1:-1]


def dictionary(data):
    L, off, _ = oracle.bwt(data)
    return oracle.wavelet(L), off


def inconsistent_dicts(sizes, seed):
    """The generators of test_gpu_decompress_many.arbitrary_dicts at the given sizes, and one more: random base counts
    with every data bit at and beyond n set, so that rows >= n read bit 1 on every level."""
    r = np.random.default_rng(seed)
    out = []
    for i, n in enumerate(sizes):
        w = n // 32 + 1
        kind = i % 4
        if kind == 0:                                           # random words: rows far beyond n
            ranks = [r.integers(0, 2**64, size=w, dtype=np.uint64) for _ in range(8)]
        elif kind == 1:                                         # a valid dictionary with a few flipped bits
            ranks = [x.copy() for x in dictionary(rnd(n, 4, 1000 + i))[0]]
            for _ in range(int(r.integers(1, 4))):
                j, k = int(r.integers(0, 8)), int(r.integers(0, w))
                ranks[j][k] ^= np.uint64(1) << np.uint64(int(r.integers(0, 64)))
        elif kind == 2:                                         # small base counts: rows stay near n
            hi = r.integers(0, 2**32, size=(8, w), dtype=np.uint64) << np.uint64(32)
            lo = r.integers(0, n + 40, size=(8, w), dtype=np.uint64)
            ranks = [hi[j] | lo[j] for j in range(8)]
        else:                                                   # data bits at and beyond n set
            ranks = [r.integers(0, 2**64, size=w, dtype=np.uint64) for _ in range(8)]
            for x in ranks:
                x[-1] |= np.uint64(M32 & ~((1 << (n & 31)) - 1)) << np.uint64(32)
        out.append((ranks, int(r.integers(0, n)), n))
    return out


# ---- CPU: the reference against the restatement and the oracle ----------------------------------------------------

def test_clamped_reference_matches_restatement():
    from tests.test_gpu_decompress_many import arbitrary_dicts, unbwt_ref
    cases = [(ranks, min(off, n - 1), n) for ranks, off, n in arbitrary_dicts()]
    cases += inconsistent_dicts([int(x) for x in np.random.default_rng(5).integers(1, 300, 24)], 6)
    rng = np.random.default_rng(7)
    cases += [(random_consistent(n, a, rng), int(rng.integers(0, n)), n)
              for n in (1, 2, 3, 31, 32, 33, 64, 65, 200, 299) for a in (1, 4)]
    for i, (ranks, off, n) in enumerate(cases):
        assert unbwt_clamped(ranks, off, n) == unbwt_ref(ranks, off, n), i


def test_clamped_reference_matches_oracle():
    datas = [d for _, d, _ in small_cases()]
    datas += [rnd(q, 256, q) * k for q, k in ((1, 300), (2, 101), (3, 70), (31, 9), (32, 5), (33, 33), (1000, 3))]
    for i, data in enumerate(datas):
        ranks, off = dictionary(data)
        n = len(data)
        assert consistent(ranks, n), i
        got = unbwt_clamped(ranks, off, n)
        assert got == oracle.unbwt_bitwise(ranks, off, n).tobytes(), i
        if primitive(data):
            assert got == data and period(ranks, n) == n, i


def test_generators_make_what_they_claim():
    rng = np.random.default_rng(8)
    for n in (1, 2, 31, 32, 33, 1000, 4097):
        ranks = random_consistent(n, 2, rng)
        assert consistent(ranks, n)
        R = levels(ranks)
        zeros = [(n - ones_before(R[j], n, n)) & M32 for j in range(8)]
        _, LF = descend(R, zeros, n, np.arange(n, dtype=np.uint64))
        assert np.array_equal(np.sort(LF), np.arange(n, dtype=np.uint64)), n          # a permutation of [0, n)
    bad = inconsistent_dicts([int(x) for x in rng.integers(65537, 70000, 8)], 9)
    assert not any(consistent(r, n) for r, _, n in bad)


# ---- GPU ----------------------------------------------------------------------------------------------------------

def first_diff(got, want):
    a, b = np.frombuffer(got, dtype=np.uint8), np.frombuffer(want, dtype=np.uint8)
    d = np.nonzero(a != b)[0]
    return None if d.size == 0 else f"{d.size} of {a.size} bytes differ, first at {int(d[0])}: got {a[d[0]]} want {b[d[0]]}"


def gpu_dictionary(fe, data):
    L, off, _ = fe.bwt(data)
    return fe.wavelet(L)[0], off


def prime(fe, n, want, seed):
    """Invert a primitive text of n bytes that differs from `want` at every position: the output scratch of the next
    inversion of n rows then holds other bytes everywhere."""
    w = np.frombuffer(want, dtype=np.uint8)
    for s in range(seed, seed + 100):
        P = ((w.astype(np.int64) + 1 + np.random.default_rng(s).integers(0, 255, size=n)) % 256).astype(np.uint8)
        if n == 1 or primitive(P.tobytes()):
            break
    P = P.tobytes()
    ranks, off = dictionary(P) if n <= 1 << 22 else gpu_dictionary(fe, P)
    assert fe.unbwt(ranks, off, n).tobytes() == P
    assert fe.stats()["unbwt_serial"] == 0


def check(fe, ranks, off, n, want, serial, seed=0):
    prime(fe, n, want, seed)
    got = fe.unbwt(ranks, off, n).tobytes()
    assert first_diff(got, want) is None, (n, off, first_diff(got, want))
    assert fe.stats()["unbwt_serial"] == serial


def power_size(q, t):
    """A multiple of q, at least 2q, near t and congruent to t mod 32 where q allows it."""
    k0 = max(2, -(-t // q))
    for k in range(k0, k0 + 64):
        if (q * k - t) % 32 == 0:
            return q * k
    return q * k0


PERIODS = (1, 2, 3, 31, 32, 33, 1000, 4097)
TARGETS = (5, 30, 32 * 37 - 1, 32 * 37 + 1, 65535, 65537, 1 << 20)


def power_cases():
    cases = {}
    for q in PERIODS:
        for t in TARGETS:
            n = power_size(q, t)
            cases.setdefault((q, n), None)
    return sorted(cases)


def power_block(q):
    if q == 1:
        return b"\0"                                   # a zero-filled file
    for s in range(q, q + 50):
        b = rnd(q, 3 if q % 2 else 256, s)
        if primitive(b):
            return b


@pytest.mark.gpu
@pytest.mark.parametrize("q,n", power_cases(), ids=[f"q{q}-n{n}" for q, n in power_cases()])
def test_valid_power(frontend, q, n):
    """An exact power w^(n/q): LF has several cycles, row 0's of length q; the text is unbwt::bitwise's."""
    data = power_block(q) * (n // q)
    assert len(data) == n and not (n > q and primitive(data))
    ranks, off = dictionary(data)
    want = oracle.unbwt_bitwise(ranks, off, n).tobytes()
    check(frontend, ranks, off, n, want, 0, seed=n)
    assert period(ranks, n) == q


def primitive_cases():
    out = [b"x", b"ab", b"ba", b"a" + b"b" * 40, b"b" * 40 + b"a"]
    for n in (3, 31, 32, 33, 32 * 37 - 1, 32 * 37 + 1, 65535, 65536, 65537, (1 << 20) + 3):
        out.append(synth.generate(GENERATORS[n % 4], n, n).tobytes())
    out.append(b"b" * 70000 + b"a")                     # least rotation at n - 1
    out.append(b"a" + b"b" * 70000)                     # ... at 0
    return out


@pytest.mark.gpu
def test_valid_primitive(frontend):
    for i, data in enumerate(primitive_cases()):
        n = len(data)
        assert primitive(data)
        ranks, off = dictionary(data)
        if data.startswith(b"b" * 40):
            assert off == n - 1
        for o in sorted({off, 0, n - 1}):
            want = oracle.unbwt_bitwise(ranks, o, n).tobytes()
            if o == off:
                assert want == data
            check(frontend, ranks, o, n, want, 0, seed=i)


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["power-17", "one-byte", "power-above-chain-64"])
def test_large_power(frontend, name):
    """The exact powers of test_gpu_scale_paths, and one above the size where unbwt_run makes its chains 64 rows
    long (shiftB = 6: n / (SMs * 2048 * 4) > 32)."""
    if name == "power-17":
        data = np.tile(np.random.default_rng(17).integers(0, 4, size=1_000_003, dtype=np.uint8), 17).tobytes()
        q = 1_000_003
    elif name == "one-byte":
        data, q = b"z" * ((1 << 24) + 3), 1
    else:
        threshold = 33 * sm_count() * 8192
        q = 4097
        data = power_block(q) * (threshold // q + 2)
        assert len(data) >= threshold and (len(data) // (sm_count() * 2048 * 4)) > 32
    n = len(data)
    ranks, off = gpu_dictionary(frontend, data)
    want = oracle.unbwt_bitwise(ranks, off, n).tobytes()
    if name == "one-byte":
        assert want == data
    check(frontend, ranks, off, n, want, 0, seed=3)
    assert period(ranks, n) == q


@pytest.mark.gpu
def test_consistent_random_words(frontend):
    """LF a random permutation: row 0's cycle of every length, shorter than a chain, and not dividing n.  The device
    path takes these words, and the fill of steps p .. n-1 from steps k mod p is checked hardest here."""
    rng = np.random.default_rng(2031)
    sizes = [1, 2, 3, 31, 32, 33, 63, 64, 65, 1000, 4097, 65535, 65537, 100_003, 262_145, 300_000]
    sizes += [int(x) for x in rng.integers(1, 300_000, 16)]
    seen = []
    for i, n in enumerate(sizes):
        ranks = random_consistent(n, (1, 3, 6, 9)[i % 4], rng)
        off = int(rng.integers(0, n))
        p = period(ranks, n)
        seen.append((n, p))
        check(frontend, ranks, off, n, unbwt_clamped(ranks, off, n), 0, seed=i)
    assert any(p < 32 and p < n for n, p in seen), seen
    assert sum(p < n and n % p for n, p in seen) >= 5, seen
    assert any(p >= 32 and p < n for n, p in seen), seen


@pytest.mark.gpu
def test_inconsistent_words(frontend):
    """Words that are no rank directory (only damaged archives decode to them) take the host walk: rows reach n and
    beyond, and the text is still the clamped walk's."""
    rng = np.random.default_rng(77)
    sizes = [65537, 65568, 100_003, 131_071, 299_999] + [int(x) for x in rng.integers(65537, 300_000, 11)] + [1, 5, 33]
    cases = inconsistent_dicts(sizes, 78)
    inconsistent = 0
    for i, (ranks, off, n) in enumerate(cases):
        bad = not consistent(ranks, n)
        inconsistent += bad
        check(frontend, ranks, off, n, unbwt_clamped(ranks, off, n), int(bad), seed=i)
    assert inconsistent >= len(cases) - 2, inconsistent


def ds(a):
    """`bce -ds` of an archive, None where it rejects it."""
    try:
        return host.decompress(a, low_memory=True)
    except (RuntimeError, ValueError):
        return None


def mutate(a, rng):
    from tests.test_gpu_decompress_many import mutate as m
    return m(a, rng)


@functools.lru_cache(maxsize=1)
def archive_cases():
    r = random.Random(151)
    inputs = [synth.generate(GENERATORS[i % 4], r.randint(70_000, 150_000), 60 + i).tobytes() for i in range(8)]
    arcs = [oracle.compress(d) for d in inputs]
    rng = random.Random(2026)
    batch = []
    for _ in range(150):
        j = rng.randrange(len(arcs))
        batch.append((mutate(arcs[j], rng), inputs[j], True))
    powers = [b"\0" * 70_000, rnd(1000, 256, 5) * 80, rnd(33, 3, 6) * 3000, rnd(4097, 2, 7) * 20]
    for d in powers + inputs:
        batch.append((oracle.compress(d), d, False))
    return batch


@pytest.mark.gpu
def test_archives(frontend, monkeypatch):
    """Damaged archives of 70-150 KB inputs, exact powers and intact archives, all above BCE_GPU_MANY_MAX_N, through
    host.decompress_many (its large path is bce_gpu_unbwt on the frontend's context): every text is `bce -ds`'s."""
    monkeypatch.setenv("BCE_HOST_MAX_N", str(1 << 20))
    batch = archive_cases()
    got = host.decompress_many(frontend, [a for a, _, _ in batch], threads=8)
    with ThreadPoolExecutor(8) as pool:
        wants = list(pool.map(ds, [a for a, _, _ in batch]))
    wrong = errors = 0
    for i, ((a, d, damaged), g, want) in enumerate(zip(batch, got, wants)):
        if want is None:
            assert isinstance(g, BceGpuError) and g.code == -1, i
            errors += 1
            continue
        assert isinstance(g, bytes) and first_diff(g, want) is None, (i, first_diff(g, want) if isinstance(g, bytes) else g)
        if damaged:
            wrong += want != d
        else:
            assert len(d) > MANY_MAX_N and (g == d or not primitive(d)), i   # a power comes back as `bce -ds` makes it
    assert wrong > 30 and errors > 10, (wrong, errors)


@pytest.mark.gpu
def test_decompress_and_cli(monkeypatch, tmp_path):
    """host.decompress (a device opened per call) and `bce -d` against `bce -ds`: a large power, damaged archives
    that decode to something else, an intact archive."""
    monkeypatch.setenv("BCE_HOST_MAX_N", str(1 << 20))
    batch = archive_cases()
    picks = [batch[-9], batch[-12]]                                  # the power of 4097 bytes, the zero-filled file
    for a, d, damaged in batch[:150]:
        try:
            w = host.decompress(a, low_memory=True)
        except RuntimeError:
            continue
        if w != d and len(w) > MANY_MAX_N:
            picks.append((a, d, damaged))
            if len(picks) == 5:
                break
    picks.append(batch[-1])
    assert len(picks) == 6
    assert build.BIN_BCE.exists(), "the bce tool was not built"
    for i, (a, d, _) in enumerate(picks):
        want = host.decompress(a, low_memory=True)
        assert first_diff(host.decompress(a), want) is None, i
        arc = tmp_path / f"a{i}.bce"
        arc.write_bytes(a)
        for flag in ("-d", "-ds"):
            r = subprocess.run([str(build.BIN_BCE), flag, str(tmp_path / f"out{i}{flag}"), str(arc)],
                               capture_output=True, timeout=600)
            assert r.returncode == 0, (i, flag, r.stdout)
        assert (tmp_path / f"out{i}-d").read_bytes() == (tmp_path / f"out{i}-ds").read_bytes() == want, i


@pytest.mark.gpu
def test_context_reuse(frontend):
    """unbwt of a power, a damaged dictionary and a primitive input, interleaved with compress_front and unbwt_many
    on one context: every result unchanged."""
    pw = rnd(31, 3, 40) * 4000
    pr = synth.generate("enwik-shaped", 200_001, 41).tobytes()
    bad_ranks, bad_off, bad_n = inconsistent_dicts([150_000], 42)[0]
    assert not consistent(bad_ranks, bad_n)
    pw_ranks, pw_off = dictionary(pw)
    pr_ranks, pr_off = dictionary(pr)
    want_pw = oracle.unbwt_bitwise(pw_ranks, pw_off, len(pw)).tobytes()
    want_bad = unbwt_clamped(bad_ranks, bad_off, bad_n)
    small = [synth.generate(GENERATORS[i % 4], 300 + 5000 * i, 50 + i).tobytes() for i in range(6)]
    small_dicts = [dictionary(d) + (len(d),) for d in small]
    front = small[4]
    fw = oracle.cse(oracle.wavelet(oracle.bwt(front)[0]), len(front))
    for _ in range(2):
        assert frontend.unbwt(pw_ranks, pw_off, len(pw)).tobytes() == want_pw
        off, Cv, streams = frontend.compress_front(front)
        assert Cv == fw["C"] and all(np.array_equal(streams[i], fw["streams"][i]) for i in range(8))
        assert frontend.unbwt(bad_ranks, bad_off, bad_n).tobytes() == want_bad
        assert frontend.stats()["unbwt_serial"] == 1
        assert [g.tobytes() for g in frontend.unbwt_many(small_dicts)] == small
        assert frontend.unbwt(pr_ranks, pr_off, len(pr)).tobytes() == pr
        assert frontend.stats()["unbwt_serial"] == 0
