// cse_rule.cuh -- the level loop's node rule and the words it emits, shared by every kernel that runs it
// (cse.cu and its headers, many.cu).
#pragma once

#include "ctx.h"

namespace bce {

enum : uint32_t { kEmitRaw = 0, kEmitCoder = 1, kEmitScan = 2 };

struct CseArgs {
  const uint64_t* ranks[8];
  uint32_t C[8];                         // first position of the one-half of level i (bce.cpp:1259)
  uint32_t* fs[2][8];                    // frontier, structure of arrays: position
  uint32_t* fa[2][8];                    //   x0
  uint32_t* fb[2][8];                    //   x1
  uint32_t cap;                          // nodes per frontier buffer, multiple of 4
  uint32_t* emit[8];                     // emission buffers (words)
  unsigned long long ecap[8];            // their capacity in words (no round may start that could overflow it)
  unsigned long long esoft[8];           // batch target: once a stream holds this many words the batch ends with the round
  uint64_t* desc;                        // 3 x desc_tiles
  uint32_t desc_tiles;
  uint32_t round_limit;                  // no input needs more than 8 n rounds: beyond it something is broken
  uint32_t use_narrow;                   // 1 = hand narrow frontiers to the cluster kernels
  uint32_t narrow_enter;                 // ... once every level holds at most this many nodes
  uint32_t use_tiny, tiny_enter;         // 1 = the one-CTA kernel takes frontiers of <= tiny_enter nodes per level
  uint32_t emit_mode;                    // kEmitRaw / kEmitCoder / kEmitScan
  unsigned long long min_nodes, max_nodes;   // wide kernel: leave (kCseGoWide) when the frontier is outside
  uint8_t cfgbits[8][32];                // kEmitCoder: context bits per (stream, k), bce.cpp:713-724
  CseDeviceState* st;
};

__device__ __forceinline__ uint32_t rank1_word(uint64_t w, uint32_t pos) {      // Rank::get<1>, bce.cpp:147-151
  return uint32_t(w) + __popc(uint32_t(w >> 32) & ((1u << (pos & 31u)) - 1u));
}

// One emitted count -> words.  Returns the number of words (5 raw, 1 or 3 packed); e0..e2 hold
// them (raw: sym, k, c1 -- the caller appends c2 = x1 and cs = x).
__device__ __forceinline__ uint32_t count_words(const CseArgs& a, int level, uint32_t sym, uint32_t k,
                                                uint32_t c1, uint32_t c2, uint32_t cs,
                                                uint32_t& e0, uint32_t& e1, uint32_t& e2) {
  if (a.emit_mode == kEmitRaw) { e0 = sym; e1 = k; e2 = c1; return 5u; }
  return bcefmt::pack_count(a.emit_mode == kEmitCoder, a.cfgbits[level], sym, k, c1, c2, cs, e0, e1, e2);
}
__device__ __forceinline__ void put_words(uint32_t* dst, uint32_t nw, uint32_t e0, uint32_t e1, uint32_t e2,
                                          uint32_t x1, uint32_t x) {
  dst[0] = e0;
  if (nw == 5u) { dst[1] = e1; dst[2] = e2; dst[3] = x1; dst[4] = x; }
  else if (nw == 3u) { dst[1] = e1; dst[2] = e2; }
}
__device__ __forceinline__ uint32_t max_words(const CseArgs& a) {
  return a.emit_mode == kEmitRaw ? 5u : a.emit_mode == kEmitCoder ? 3u : 1u;
}

// The three rank words a node needs, bce.cpp:1265, 1271, 1301: at s, s + x and s + x0.
__device__ __forceinline__ void rank_words(const uint64_t* __restrict__ R, uint32_t s, uint32_t x0, uint32_t x1,
                                           uint64_t& wa, uint64_t& wb, uint64_t& wc) {
  wa = __ldg(R + (s >> 5));
  wb = __ldg(R + ((s + x0 + x1) >> 5));
  wc = __ldg(R + ((s + x0) >> 5));
}

// One node of level l, bce.cpp:1265-1345: from its three rank words, its zero-child (z: it exists), its one-child (o)
// and the count it hands to coder_[l].set (:1302) as words (count_words; nw = 0: no count).  Fields of a child that
// does not exist are 0.
struct CseStep {
  bool z, o;
  uint32_t zs, za, zb, os, oa, ob;
  uint32_t nw, e0, e1, e2;
};
__device__ __forceinline__ CseStep cse_step(const CseArgs& a, int l, uint32_t one_base, uint32_t s, uint32_t x0,
                                            uint32_t x1, uint64_t wa, uint64_t wb, uint64_t wc) {
  CseStep r{false, false, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
  const uint32_t x = x0 + x1;
  const uint32_t s1 = rank1_word(wa, s);
  const uint32_t c1 = rank1_word(wb, s + x) - s1;               // _1x
  const uint32_t s0 = s - s1;
  const uint32_t z0 = (s + x0 - rank1_word(wc, s + x0)) - s0;   // _0x0 (:1301)
  r.zs = s0;
  r.os = one_base + s1;
  if (c1 == 0) { r.z = true; r.za = x0; r.zb = x1; }            // :1274
  else if (c1 == x) { r.o = true; r.oa = x0; r.ob = x1; }       // :1282
  else {
    const uint32_t c0 = x - c1;
    const uint32_t lo = x0 > c1 ? x0 - c1 : 0u;                 // :1290-1294
    const uint32_t hi = x0 - (c1 > x1 ? c1 - x1 : 0u);
    const uint32_t z1 = c0 - z0, o1 = x1 - z1, o0c = c1 - o1;   // _0x1, _1x1, _1x0
    if (hi != lo) r.nw = count_words(a, l, z0 - lo, hi - lo + 1, c0, x1, x, r.e0, r.e1, r.e2);   // :1302
    if (z0 && z1) { r.z = true; r.za = z0; r.zb = z1; }         // :1338
    if (o0c && o1) { r.o = true; r.oa = o0c; r.ob = o1; }       // :1345
  }
  return r;
}

// Position t of a level's ordered frontier in the flat layout: the zero-half (cz nodes) from the front of the buffer,
// the one-half from its back.
__device__ __forceinline__ uint32_t flat_at(uint32_t cap, uint32_t cz, uint32_t t) { return t < cz ? t : cap - 1u - (t - cz); }

}  // namespace bce
