// format.h -- the BCE v0.4 archive format, defined once for the host coders (g++: csrc/host, libbce_host and `bce`)
// and the device coders (nvcc: code_many.cu, decode_many.cu, cse_rule.cuh).  Archives must be bit-exact drop-ins for
// the reference's, and a damaged archive must be rejected -- or decoded -- the same way on both sides, so every format
// decision lives here: the default config table and its check, the model layout and context index, the packed count
// words, the range coder's scalar steps, the archive header, the rank dictionary's words and the decode node rule.
// What stays with each side is how it runs them: the host's serial loops and the device's warp-parallel adaptive steps
// (reductions in the encoder, a scan in the decoder), and the model update.
//
// No CUDA runtime, no STL.  Where the two sides differ it is in the instruction only: the bit operations below, and
// the 64-bit division (`/` on the host, div64 on the device).
#pragma once

#include <stddef.h>
#include <stdint.h>

#ifdef __CUDACC__
#define BCE_HD __host__ __device__ __forceinline__
#else
#define BCE_HD inline
#endif

namespace bcefmt {

constexpr int kMaxAdaptive = 31;               // AdaptiveCoder<31>::max, bce.cpp:1381
constexpr int kConfigRows = 9;                 // streams 0..7 + header row 8
constexpr int kConfigCols = kMaxAdaptive + 1;

// ---- bit operations ---------------------------------------------------------------------------------------------
BCE_HD uint32_t popc32(uint32_t v) {
#ifdef __CUDA_ARCH__
  return uint32_t(__popc(v));
#else
  return uint32_t(__builtin_popcount(v));
#endif
}
BCE_HD uint32_t popc64(uint64_t v) {
#ifdef __CUDA_ARCH__
  return uint32_t(__popcll(v));
#else
  return uint32_t(__builtin_popcountll(v));
#endif
}
BCE_HD uint32_t ctz64(uint64_t v) {            // v != 0
#ifdef __CUDA_ARCH__
  return uint32_t(__ffsll((long long)v) - 1);
#else
  return uint32_t(__builtin_ctzll(v));
#endif
}
BCE_HD uint32_t clz64(uint64_t v) {            // clz64(0) = 64 on both sides
#ifdef __CUDA_ARCH__
  return uint32_t(__clzll((long long)v));
#else
  return v ? uint32_t(__builtin_clzll(v)) : 64u;
#endif
}

#ifdef __CUDA_ARCH__
// 1 / v for a normal v >= 1 with a relative error of a few 2^-53 and no call: __drcp_rn's path for special operands
// is a call, whose convention makes a kernel with much live state spill.  The hardware estimate, then two Newton steps.
__device__ __forceinline__ double rcp_nocall(double v) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(v));
  r = fma(r, fma(-v, r, 1.0), r);
  return fma(r, fma(-v, r, 1.0), r);
}

// floor(x / d) for d >= 1 without the 64-bit division routine (a call, whose convention spills): the high half by a
// 32-bit division, the low quotient (below 2^32) estimated in double precision -- relative error a few 2^-53, so off
// by at most 1 -- and corrected.
__device__ __forceinline__ uint64_t div64(uint64_t x, uint32_t d) {
  const uint32_t xh = uint32_t(x >> 32), qh = xh / d;
  const uint64_t y = (uint64_t(xh - qh * d) << 32) | uint32_t(x);            // < d 2^32
  uint64_t ql = uint64_t(__dmul_rn(__ull2double_rn(y), rcp_nocall(double(d))));
  int64_t r = int64_t(y - ql * d);                                          // |r| < 3 d
  for (int t = 0; t < 3 && r < 0; ++t) { --ql; r += d; }
  for (int t = 0; t < 3 && r >= int64_t(d); ++t) { ++ql; r -= d; }
  return (uint64_t(qh) << 32) + ql;
}
#endif

BCE_HD uint64_t div_step(uint64_t x, uint32_t d) {   // floor(x / d), d >= 1: a coding step's width
#ifdef __CUDA_ARCH__
  return div64(x, d);
#else
  return x / d;
#endif
}

// floor(d / step) for a d below step * range, range <= 2^31: the decoder's symbol of a uniform step.  The device
// estimates it in double precision (off by at most one) and corrects it.
BCE_HD uint64_t uniform_quotient(uint64_t d, uint64_t step, uint32_t range) {
#ifdef __CUDA_ARCH__
  uint64_t q = uint64_t(__dmul_rn(__ull2double_rn(d), rcp_nocall(__ull2double_rn(step))));
  if (q > range - 1) q = range - 1;
  for (int t = 0; t < 3 && q * step > d; ++t) --q;
  for (int t = 0; t < 3 && (q + 1) * step <= d; ++t) ++q;
  return q;
#else
  (void)range;
  return d / step;
#endif
}

// x86 SHL: the count is taken mod 64.  The reference shifts 64-bit values by amounts that can reach or exceed 64
// (bce.cpp:175-176, undefined behaviour in C++, SURVEY.md Q6); archives only decode identically if those shifts
// behave like the instruction the reference was compiled to.
BCE_HD uint64_t shl_x86(uint64_t v, uint64_t count) { return v << (count & 63u); }

// ---- config table -----------------------------------------------------------------------------------------------
// context bits per (stream, k), bce.cpp:713-724; row 8 (the header coder) is all 0
constexpr uint8_t kDefaultConfig[kConfigRows][kConfigCols] = {
  {0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,0},
  {0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,0},
  {0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,3,3,3,3,0},
  {0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,0},
  {0,0,5,5,4,4,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,0},
  {0,0,5,5,4,4,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,0},
  {0,0,5,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,0},
  {0,0,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,2,2,2,2,2,2,0},
  {0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0}};

// Context bits are coded in 0..5 (bce.cpp:686): a table with more cannot have come from `bce -s`.  Checks cfg[0 ..
// count); on failure *bad (when given) is the first value out of range.
inline bool config_ok(const uint8_t* cfg, int count, uint32_t* bad = nullptr) {
  for (int i = 0; i < count; ++i)
    if (cfg[i] > 5) {
      if (bad) *bad = cfg[i];
      return false;
    }
  return true;
}

// ---- adaptive model layout (ContextModel, bce.cpp:671-677, :700-705) --------------------------------------------
// One table per k = 2..31 of 4^bits rows, a row being k one-byte counters and two more bytes (the host keeps the
// row's sum there).  layout_row adds k's table at *start: off[k] = its first byte | bits << 24 (off may be null).
BCE_HD void layout_row(uint32_t* off, uint32_t k, uint32_t bits, uint32_t& start) {
  if (off) off[k] = start | (bits << 24);
  start += (k + 2) << (bits * 2);
}
// a whole config row; returns the table's bytes
BCE_HD uint32_t model_layout(const uint8_t* bits, uint32_t* off) {
  uint32_t start = 0;
  for (uint32_t k = 2; k < uint32_t(kConfigCols); ++k) layout_row(off, k, bits[k], start);
  return start;
}
// context index of (c1, c2) out of cs at b context bits each (bce.cpp:674, uint32 wrap-around as there)
BCE_HD uint32_t context_index(uint32_t b, uint32_t c1, uint32_t c2, uint32_t cs) {
  return (((c1 << b) / cs) << b) | ((c2 << b) / cs);
}
// the row of context ctx in k's table (off_k from layout_row)
BCE_HD size_t row_offset(uint32_t off_k, uint32_t k, uint32_t ctx) {
  return (off_k & 0x00FFFFFFu) + size_t(ctx) * (k + 2);
}

// ---- packed count words (include/bce_gpu.h) ---------------------------------------------------------------------
// One count -> BCE_EMIT_CODER (coder = true) or BCE_EMIT_SCAN words in e0..e2; returns their number (1 or 3).
//   CODER  [ctx:10 @10 | k:5 @5 | sym:5]; k > 31 halves first (bce.cpp:507-510) and writes k field 0, then
//          [low bits:10 @10 | nb:5 @5 | k:5] and [low bits >> 10]
//   SCAN   [esc:1 | nb:5 @26 | q2:8 @18 | q1:8 @10 | k:5 @5 | sym:5] (bce.cpp:737-744: a different halving)
BCE_HD uint32_t pack_count(bool coder, const uint8_t* bits_row, uint32_t sym, uint32_t k, uint32_t c1, uint32_t c2,
                           uint32_t cs, uint32_t& e0, uint32_t& e1, uint32_t& e2) {
  uint32_t nb = 0, s = sym;
  if (coder) {
    while (k > 31u) { k = (k + (~s & 1u)) >> 1; s >>= 1; ++nb; }                 // bce.cpp:507-510
    const uint32_t ctx = context_index(bits_row[k], c1, c2, cs);
    const uint32_t w = (ctx << 10) | (k << 5) | s;
    if (nb == 0) { e0 = w; e1 = e2 = 0; return 1u; }
    const uint32_t low = sym & ((1u << nb) - 1u);                                  // nb <= 27
    e0 = (ctx << 10) | s;                                                         // k field 0: two more words
    e1 = k | (nb << 5) | ((low & 0x3FFu) << 10);
    e2 = low >> 10;
    return 3u;
  }
  while (k > 31u) { k = (k >> 1) + (~s & 1u); s >>= 1; ++nb; }                   // bce.cpp:738-741
  const uint32_t q1 = (c1 << 8) / cs, q2 = (c2 << 8) / cs;                        // bce.cpp:743
  e0 = (nb ? 0x80000000u | (nb << 26) : 0u) | (q2 << 18) | (q1 << 10) | (k << 5) | s;
  e1 = e2 = 0;
  return 1u;
}
// CODER word -> symbol, k and context; k == 0 is the escape: two more words follow (coder_escape)
BCE_HD void coder_fields(uint32_t w, uint32_t& sym, uint32_t& k, uint32_t& ctx) {
  sym = w & 31u;
  ctx = (w >> 10) & 1023u;
  k = (w >> 5) & 31u;
}
// the two escape words -> k after the halvings, their number nb and the nb uniform bits (low bit first)
BCE_HD void coder_escape(uint32_t w1, uint32_t w2, uint32_t& k, uint32_t& nb, uint32_t& low) {
  nb = (w1 >> 5) & 31u;
  low = (w1 >> 10) | (w2 << 10);
  k = w1 & 31u;
}
// SCAN word -> its bucket (k, q1, q2) = bits 5..25; bucket -> k and the collector's key (q2 << 16) | q1
BCE_HD uint32_t scan_bucket(uint32_t w) { return (w >> 5) & 0x1FFFFFu; }
BCE_HD uint32_t bucket_k(uint32_t b) { return b & 31u; }
BCE_HD uint32_t bucket_key(uint32_t b) { return (((b >> 13) & 255u) << 16) | ((b >> 5) & 255u); }

// ---- range encoder (bce.cpp:520-553, :610-615, :655-661; VCoder :364-370) ----------------------------------------
// 64-bit carry-less range coder with 16-bit output words, written to out(word).  Renormalisation is bounded at 4
// shifts, which is exact: each shift leaves 0xFFFF in the low 16 bits of hi ^ lo, so after 4 its top 16 are not 0.
template <class Sink>
struct RangeEncoder {
  uint64_t lo = 0, hi = ~0ull;
  Sink out;

  BCE_HD void renormalise() {
    for (int t = 0; t < 4 && ((hi ^ lo) >> 48) == 0; ++t) {
      out(uint32_t(hi >> 48));
      lo <<= 16;
      hi = (hi << 16) | 0xFFFFu;
    }
  }
  BCE_HD void restart_if_narrow(uint64_t total) {
    if (hi - lo < total) {
      for (int shift = 48; shift >= 0; shift -= 16) out(uint32_t(lo >> shift));
      lo = 0;
      hi = ~0ull;
    }
  }
  BCE_HD void put_uniform(uint32_t sym, uint32_t range) {     // set(s, k)
    restart_if_narrow(range);
    const uint64_t step = div_step(hi - lo, range);
    lo += step * sym;
    hi = lo + step - 1;
    renormalise();
  }
  BCE_HD void put(uint32_t cum, uint32_t freq, uint32_t total) {   // the coding step of set(s, k, c1, c2, cs)
    restart_if_narrow(total);
    const uint64_t step = div_step(hi - lo, total);
    lo += step * cum;
    hi = lo + step * freq - 1;
    renormalise();
  }
  BCE_HD void finish() {                                      // after a renormalise hi ^ lo >= 2^48: bits <= 16
    renormalise();
    const uint32_t bits = clz64(lo ^ hi) + 1;
    out(uint32_t((hi >> (64 - bits)) << (16 - bits)));
  }
  BCE_HD void put_config(const uint8_t* bits) {               // a stream's config row, bce.cpp:685-691
    uint32_t last = 0;
    for (int j = 0; j < kConfigCols; ++j) {
      const uint32_t b = bits[j];
      put_uniform(b != last, 2);
      if (b != last) put_uniform(b, 6);
      last = b;
    }
  }
  BCE_HD void varint(uint32_t v) {
    for (int j = 0; j < 32 && v; ++j, v >>= 1) put_uniform(v & 1u, 3);
    put_uniform(2, 3);
  }
};

// ---- range decoder (bce.cpp:495-501, :566-608, :663-669; VCoder :372-377) ----------------------------------------
// The scalar half of the decoder; the adaptive step (a serial walk on the host, a warp scan on the device) stays with
// each side and uses restart_if_narrow / renormalise.  A read past the end of the words gives 0.
struct RangeDecoder {
  const uint16_t* words;
  uint32_t count, pos;
  uint64_t lo, hi, code;

  BCE_HD uint32_t next() { return pos < count ? uint32_t(words[pos++]) : 0u; }
  BCE_HD void init(const uint16_t* w, uint32_t cnt) {          // preloads four words
    words = w; count = cnt; pos = 0; lo = 0; hi = ~0ull; code = 0;
    for (int i = 0; i < 4; ++i) code = (code << 16) | next();
  }
  BCE_HD void renormalise() {                                  // at most 4 shifts, as in the encoder
    for (int t = 0; t < 4 && ((hi ^ lo) >> 48) == 0; ++t) {
      code = (code << 16) + next();
      lo <<= 16;
      hi = (hi << 16) | 0xFFFFu;
    }
  }
  BCE_HD void restart_if_narrow(uint64_t total) {
    if (hi - lo < total) {
      for (int i = 0; i < 4; ++i) code = (code << 16) + next();
      lo = 0;
      hi = ~0ull;
    }
  }
  BCE_HD uint32_t get_uniform(uint32_t range) {
    restart_if_narrow(range);
    const uint64_t step = div_step(hi - lo, range), d = code - lo;
    // code - lo >= step range only in a damaged stream: the reference's quotient is clamped to range - 1
    const uint64_t q = d >= step * range ? range - 1 : uniform_quotient(d, step, range);
    lo += step * q;
    hi = lo + step - 1;
    renormalise();
    return uint32_t(q);
  }
  BCE_HD uint32_t varint() {                                   // at most 31 bits
    uint32_t v = 0;
    for (int i = 0; i < 31; ++i) {
      const uint32_t d = get_uniform(3);
      if (d == 2) break;
      v |= d << i;
    }
    return v;
  }
  // a stream's config row (bce.cpp:693-697) -> the model layout (layout_row; off may be null); returns table bytes
  BCE_HD uint32_t config(uint32_t* off) {
    uint32_t last = 0, start = 0;
    for (uint32_t j = 0; j < uint32_t(kConfigCols); ++j) {
      const uint32_t b = get_uniform(2) ? get_uniform(6) : last;
      last = b;
      if (j >= 2) layout_row(off, j, b, start);
    }
    return start;
  }
};

// ---- archive header (BCE::encode / BCE::decode, bce.cpp:1141-1157, :1178-1190) ------------------------------------
// An archive is [header words][header][stream 0] .. [stream 7]; the header codes config row 8, n, the BWT offset, the
// total stream words and the sizes of streams 0..6.  enc has coded its config row already.
template <class Sink>
BCE_HD void write_header(RangeEncoder<Sink>& enc, uint32_t n, uint32_t offset, const uint32_t sizes[8]) {
  enc.varint(n);
  enc.put_uniform(offset, n + 1);
  uint32_t total = 0;
  for (int s = 0; s < 8; ++s) total += sizes[s];
  enc.varint(total);
  uint32_t left = total;
  for (int s = 0; s < 7; ++s) {
    enc.put_uniform(sizes[s], left + 1);
    left -= sizes[s];
  }
  enc.finish();
}
// Reads the header of archive words a[0 .. len): n, offset and the start of each stream, at(i, start) for i = 0..8
// (start 8 = len).  n_ok(n) is the caller's own check of n, made before anything after n is read.  Returns false for
// anything that is not a header of an archive of len words.
template <class NOk, class At>
BCE_HD bool read_header(const uint16_t* a, uint64_t len, NOk n_ok, uint32_t& n, uint32_t& offset, At at) {
  if (len == 0) return false;
  const uint32_t hw = a[0];
  if (1 + uint64_t(hw) > len) return false;
  RangeDecoder h;
  h.init(a + 1, hw);
  h.config(nullptr);
  n = h.varint();
  if (n == 0 || !n_ok(n)) return false;
  offset = h.get_uniform(n + 1);
  if (offset > n) return false;
  uint32_t size = h.varint();
  uint64_t start = 1 + uint64_t(hw);
  at(0, start);
  for (int i = 0; i < 7; ++i) {
    const uint32_t l = h.get_uniform(size + 1);
    if (l > size) return false;
    start += l;
    size -= l;
    if (start > len) return false;
    at(i + 1, start);
  }
  at(8, len);
  return true;
}

// ---- rank dictionary of the decoder (class Rank, bce.cpp:130-219) -------------------------------------------------
// Word = [32 data bits | 32-bit count of ones before the word], R[0 .. n / 32].  Positions are clamped to [0, n]: a
// damaged archive must not read outside the dictionary.
BCE_HD uint32_t ones_before(const uint64_t* R, uint32_t n, uint32_t pos) {      // Rank::get<1>, :147-151
  if (pos > n) pos = n;
  const uint64_t w = R[pos / 32];
  const uint32_t below = uint32_t(w >> 32) & uint32_t((1ull << (pos % 32)) - 1);
  return uint32_t(w) + popc32(below);
}
// Rank::set, :153-185: makes ones_before(pos) = ones.  Returns false when nothing changes, else the new value of word
// pos / 32 in *b (the caller writes it).
BCE_HD bool pin_word(const uint64_t* R, uint32_t n, uint32_t pos, uint32_t ones, uint64_t& b) {
  if (pos > n) return false;
  uint64_t need = uint32_t(ones - ones_before(R, n, pos));   // ones that still have to move in front of pos
  if (need == 0) return false;
  const uint64_t o = pos % 32;
  b = R[pos / 32];
  const uint32_t base = uint32_t(b);
  if (uint64_t(base) + o + 32 < need) {                      // more than this word can ever show: the
    b += need - o - base;                                    // surplus lives in the base count only (:166-169)
    need = o;
  }
  const uint64_t above = ~0ull << (32 + o);                  // data bits at and after pos
  const uint64_t take_at = ctz64(((b & above) >> 32) | (1ull << 31));                  // :172
  // :173.  ~(b | above) is 0 only in a damaged archive (a base count of 0xFFFFFFFF while need > 0): clz64(0) = 64
  const uint64_t put_end = 64 - uint64_t(clz64(~(b | above)));
  const uint64_t take = (shl_x86(1, take_at + need) - shl_x86(1, take_at)) << 32;      // :175
  const uint64_t put = shl_x86(1, put_end) - shl_x86(1, put_end - need);               // :176
  b += uint64_t(popc32(uint32_t(put)));                      // what falls below data bit 0 goes to the base count
  b &= ~take;
  b |= (put >> 32) << 32;
  return true;
}
// Rank::finalize, :187-194: word w followed by a word with base count next gets its last data bit from the difference
BCE_HD uint64_t finish_word(uint64_t w, uint32_t next) {
  const uint32_t here = uint32_t(w) + popc64(w >> 32);
  return w | (uint64_t(uint32_t(next - here)) << 63);
}

// ---- decode node rule (BCE::code with mode = 0, bce.cpp:1259-1352) -------------------------------------------------
// One node (s, x0, x1) of a level with rank dictionary R (ones_before(pos), pin(pos, ones)).  count(k, c0, x1, x)
// decodes a count below k from the level's stream; zero(s, a, b) / one(s, a, b) take the children and return false
// when they cannot.  Returns false when a count falls outside the interval the dictionary allows (damaged archive).
template <class Rank, class Count, class Zero, class One>
BCE_HD bool decode_node(uint32_t s, uint32_t x0, uint32_t x1, uint32_t n, uint32_t one_base, Rank& R, Count count,
                        Zero zero, One one) {
  const uint32_t x = x0 + x1;
  if (!x0 || !x1 || uint64_t(s) + x0 + x1 > n) return false;       // every node is an interval inside [0, n)
  const uint32_t s1 = R.ones_before(s);                              // :1265
  const uint32_t c1 = R.ones_before(s + x) - s1;                     // _1x :1271
  if (s1 > s || c1 > x) return false;
  const uint32_t s0 = s - s1;
  if (c1 == 0) {                                                     // :1274-1279
    if (!zero(s0, x0, x1)) return false;
    R.pin(s + x0, s1);
    return true;
  }
  const uint32_t c0 = x - c1;
  if (c0 == 0) {                                                     // :1282-1287
    if (!one(one_base + s1, x0, x1)) return false;
    R.pin(s + x0, s1 + x0);
    return true;
  }
  const uint32_t lo = x0 > c1 ? x0 - c1 : 0u;                        // :1290-1294
  const uint32_t hi = x0 - (c1 > x1 ? c1 - x1 : 0u);
  if (hi < lo) return false;
  uint32_t z0 = lo;                                                  // _0x0
  if (hi != lo) z0 = lo + count(hi - lo + 1, c0, x1, x);             // :1304
  if (z0 > hi || z0 > c0) return false;
  const uint32_t z1 = c0 - z0;                                       // :1337
  if (z0 && z1 && !zero(s0, z0, z1)) return false;
  if (z1 > x1 || x1 - z1 > c1) return false;
  const uint32_t o1 = x1 - z1, o0 = c1 - o1;                         // :1343-1344
  if (o0 && o1 && !one(one_base + s1, o0, o1)) return false;
  R.pin(s + x0, s1 + o0);                                            // :1350
  return true;
}

}  // namespace bcefmt
