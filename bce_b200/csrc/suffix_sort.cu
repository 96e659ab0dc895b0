// suffix_sort.cu -- stage A: cyclic suffix sort and BWT on the device.
//
// Replaces File::rotate (bce.cpp:858-894) and File::bwt / divbwt (bce.cpp:896-910).
// The reference rotates the text to its least rotation and suffix-sorts it with
// libdivsufsort; the net effect (SURVEY.md 4-2) is the BWT of the *cyclic rotations*
// of T with row 0 = least rotation and offset = its start index.  Here all n rotations
// are sorted directly by prefix doubling over packed rank keys:
//
//   round 0   key(i) = 8 bytes T[i..i+8) (cyclic, big-endian), or their 7-bit codes packed into 56 bits when at
//             most 128 byte values occur; LSD radix sort of (key, i); the first pass makes the keys from the
//             text and is unordered (radix_sort.cu)
//   re-rank   rank[i] = SA position of the head of i's group; rotations alone in their
//             group are final and leave the working set
//   round r   key = (dense group id << 32) | rank[(i + h) mod n], h = 8 * 2^(r-1); the groups are
//             short, so the working set is sorted tile by tile (local_sort.cuh; the tile sort makes
//             its keys itself) and only groups that cross a tile boundary are radix-sorted;
//             groups stay where they are, so the list slot of an element fixes its SA position
//   end       working set empty, or h >= n (T is a power w^k: remaining ties are identical
//             rotations, ordered by index so that offset is the smallest one)
//
// Kernels here: K0b text codes + code-pair histogram (round 0 on at most 128 byte values), K1 pack (only when round 0 runs no radix pass), K3h head masks + tile totals, K3c their scan into
// carries, K3 re-rank + stable compaction + binned rank pairs, K3b rank scatter, K4 key rebuild with digit histograms (radix path
// of small or declined rounds), K5 BWT gather.
#include <algorithm>
#include <utility>

#include "ctx.h"
#include "local_sort.cuh"

namespace bce {

// ---------------------------------------------------------------------------------
// K0: make T cyclic for 64 bytes past the end so that window reads need no modulo
// ---------------------------------------------------------------------------------
__global__ void pad_cyclic_kernel(uint8_t* T, uint32_t n) {
  uint32_t k = threadIdx.x;
  if (k < 64) T[size_t(n) + k] = T[k % n];
}

// ---------------------------------------------------------------------------------
// K0b: round 0's text as 7-bit symbol codes, and the cyclic histogram of its code pairs
// ---------------------------------------------------------------------------------
// When at most 128 byte values occur, round 0 sorts windows of 8 codes packed into 56 bits (pack_codes7): 7 radix
// digits instead of 8.  The code of a byte is its rank among the values that occur, so the order of windows, their
// equality and everything after round 0 are unchanged.  Every 8-bit digit of such a key is made of two adjacent codes
// (digit p, at bit 8p: the low p + 1 bits of code 6 - p and the high 7 - p bits of code 7 - p), and over all rotations
// the pairs (C[i + j], C[i + j + 1]) are the same multiset for every j: the histogram of the n cyclic code pairs gives
// every digit's histogram (digit_hist_kernel) -- one read of the text, as the byte histogram is for byte windows.
struct CodeTable { uint8_t v[256]; };
constexpr int kCodeBits = 7, kCodes = 1 << kCodeBits;
constexpr size_t kPairHistSmem = size_t(kCodes) * kCodes * 4;

__global__ void __launch_bounds__(256) code_text_kernel(const uint8_t* __restrict__ T, uint32_t n, CodeTable tab,
                                                        uint8_t* __restrict__ C, uint32_t* __restrict__ pair_hist) {
  extern __shared__ uint32_t s_pair[];                       // [kCodes * kCodes]: (earlier code << 7) | later code
  __shared__ uint8_t s_tab[256];
  for (int i = threadIdx.x; i < kCodes * kCodes; i += blockDim.x) s_pair[i] = 0;
  s_tab[threadIdx.x] = tab.v[threadIdx.x];
  __syncthreads();
  // codes of bytes [0, n + 16): every word a window of a rotation below n reads (T is cyclic for 64 bytes past n)
  const uint32_t words = (n + 16 + 3) / 4;
  const uint32_t* T32 = reinterpret_cast<const uint32_t*>(T);
  uint32_t* C32 = reinterpret_cast<uint32_t*>(C);
  for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < words; w += gridDim.x * blockDim.x) {
    const uint32_t t = T32[w];
    uint32_t c[5];
#pragma unroll
    for (int j = 0; j < 4; ++j) c[j] = s_tab[(t >> (8 * j)) & 255u];
    c[4] = s_tab[T[size_t(w) * 4 + 4]];
    C32[w] = c[0] | (c[1] << 8) | (c[2] << 16) | (c[3] << 24);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (w * 4 + j < n) atomicAdd(&s_pair[(c[j] << kCodeBits) | c[j + 1]], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kCodes * kCodes; i += blockDim.x)
    if (s_pair[i]) atomicAdd(&pair_hist[i], s_pair[i]);
}

// block p: histogram of digit p (shift 8p) of the packed keys from the code-pair histogram
__global__ void __launch_bounds__(256) digit_hist_kernel(const uint32_t* __restrict__ pair_hist, uint32_t* __restrict__ hist) {
  __shared__ uint32_t s_h[256];
  const int p = blockIdx.x;
  s_h[threadIdx.x] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < kCodes * kCodes; i += blockDim.x) {
    const uint32_t v = pair_hist[i];
    if (!v) continue;
    const uint32_t x = uint32_t(i) >> kCodeBits, y = uint32_t(i) & (kCodes - 1);   // x is the earlier code of the pair
    atomicAdd(&s_h[((x & ((2u << p) - 1u)) << (kCodeBits - p)) | (y >> p)], v);
  }
  __syncthreads();
  hist[p * 256 + threadIdx.x] = s_h[threadIdx.x];
}

// ---------------------------------------------------------------------------------
// K1: pack the window keys of the text with their indices
// ---------------------------------------------------------------------------------
// Thread t of a CTA makes keys tile + 256 r + t (r = 0 .. 7): the 12 bytes a key and its index take are
// written as coalesced rows (the first version wrote 64 bytes per thread: 32 sectors per store request).
constexpr int PK_ROWS = 8;

__global__ void __launch_bounds__(256) pack_keys_kernel(const uint8_t* __restrict__ T, uint32_t n, bool codes7,
                                                        uint64_t* __restrict__ keys,
                                                        uint32_t* __restrict__ idx) {
  const uint64_t* T64 = reinterpret_cast<const uint64_t*>(T);
  const uint32_t tile = blockIdx.x * (256 * PK_ROWS);
#pragma unroll
  for (int r = 0; r < PK_ROWS; ++r) {
    const uint32_t i = tile + r * 256 + threadIdx.x;
    if (i < n) {
      keys[i] = window_key_bits(T64, i, codes7);
      idx[i] = i;
    }
  }
}

// ---------------------------------------------------------------------------------
// K3: re-rank + stable compaction of the rotations that are still tied
// ---------------------------------------------------------------------------------
// Three launches.  K3h (rerank_heads_kernel) reads the sorted keys and writes one 32-bit head mask per row of 32 slots
// and three totals per tile; K3c (rerank_carry_kernel) scans the tile totals into the carries every tile needs (the
// last head before it, the survivors and the surviving heads before it); K3 (rerank_kernel) reads the head masks
// instead of the keys, so no tile waits for another.  (A single pass with three chained scans over the tiles in flight
// spent a quarter of its stall samples waiting for predecessors that had not yet published: profiles/r2_cse_experiments.md.)
constexpr int RR_THREADS = 256;
constexpr int RR_WARPS = RR_THREADS / 32;
constexpr int RR_ROWS = 16;                         // rows of 32 consecutive slots per warp
constexpr int RR_WCHUNK = 32 * RR_ROWS;             // slots per warp
constexpr int RR_TILE = RR_WARPS * RR_WCHUNK;       // 4096 slots per tile
constexpr int RR_CARRY_THREADS = 1024;

// The rule of a row of 32 slots from its head mask H (bit l: slot rowbase + l is the first of its group; slot 0 of the
// working set always is) and next_first (the slot behind the row is a head, or does not exist):
//   L lone slots (a group of one: a head whose successor is a head or the end), S survivors (tied slots),
//   SH surviving heads.  H is the same in all lanes, so these are a handful of bit operations.
__device__ __forceinline__ void rerank_row_masks(uint32_t H, uint32_t next_first, uint32_t rowbase, uint32_t m,
                                                 uint32_t& S, uint32_t& SH, uint32_t& L) {
  const uint32_t valid = rowbase >= m ? 0u : m - rowbase;                        // slots of the row below m
  const uint32_t in_mask = valid >= 32u ? 0xFFFFFFFFu : (1u << valid) - 1u;
  uint32_t nh = (H >> 1) | (next_first << 31);                                   // the slot behind is a head ...
  if (valid <= 32u) nh |= valid ? ~((1u << (valid - 1u)) - 1u) : 0xFFFFFFFFu;    // ... or does not exist
  L = H & nh & in_mask;
  S = in_mask & ~L;
  SH = H & ~L;
}

// A warp's survivors, surviving heads and (slot + 1) of its last head (0: none) from the head masks of its rows;
// after_is_head: the slot after the warp's last one is a head or the end of the working set.
__device__ __forceinline__ void rerank_warp_totals(const uint32_t (&H)[RR_ROWS], bool after_is_head, uint32_t wbase,
                                                   uint32_t m, uint32_t& wsurv, uint32_t& wshead, uint32_t& whead) {
  wsurv = wshead = whead = 0;
#pragma unroll
  for (int k = 0; k < RR_ROWS; ++k) {
    uint32_t S, SH, L;
    const uint32_t next_first = k + 1 < RR_ROWS ? (H[k + 1 < RR_ROWS ? k + 1 : k] & 1u) : (after_is_head ? 1u : 0u);
    rerank_row_masks(H[k], next_first, wbase + k * 32, m, S, SH, L);
    wsurv += __popc(S);
    wshead += __popc(SH);
    if (H[k]) whead = wbase + k * 32 + (31 - __clz(H[k])) + 1;
  }
}

// K3h: head masks of the rows (lane l of a warp holds slots wbase + 32 k + l, as in K3) and the tile's totals:
// tsum[t] = (slot + 1) of its last head, tsum[tiles + t] survivors, tsum[2 tiles + t] surviving heads
__global__ void __launch_bounds__(RR_THREADS) rerank_heads_kernel(const uint64_t* __restrict__ key, uint32_t m,
                                                                  uint32_t* __restrict__ heads,
                                                                  uint32_t* __restrict__ tsum, uint32_t tiles) {
  __shared__ uint32_t s_w[3][RR_WARPS];
  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t tile = blockIdx.x;
  const uint32_t wbase = tile * RR_TILE + warp * RR_WCHUNK;      // < 2^32: m < 2^31
  uint64_t k64[RR_ROWS];
#pragma unroll
  for (int k = 0; k < RR_ROWS; ++k) {
    const uint32_t q = wbase + k * 32 + lane;
    k64[k] = q < m ? key[q] : 0;
  }
  // the keys just outside the warp's chunk (uniform loads)
  const uint64_t key_before = (wbase > 0 && wbase - 1 < m) ? key[wbase - 1] : 0;
  const uint64_t key_after = (wbase + RR_WCHUNK < m) ? key[wbase + RR_WCHUNK] : 0;
  // head = first slot of a (new) group
  uint32_t H[RR_ROWS], mine = 0;
#pragma unroll
  for (int k = 0; k < RR_ROWS; ++k) {
    const uint32_t q = wbase + k * 32 + lane;
    const uint64_t up = __shfl_up_sync(0xffffffffu, k64[k], 1);
    const uint64_t wrap = k ? __shfl_sync(0xffffffffu, k64[k ? k - 1 : 0], 31) : key_before;
    const uint64_t prev = lane ? up : wrap;
    H[k] = __ballot_sync(0xffffffffu, q < m && (q == 0 || k64[k] != prev));
    if (lane == unsigned(k)) mine = H[k];
  }
  const uint32_t row = wbase / 32 + lane;                            // lane k < RR_ROWS stores row k's mask
  if (lane < unsigned(RR_ROWS) && row * 32 < m) heads[row] = mine;
  const bool after_is_head = (wbase + RR_WCHUNK >= m) || (key_after != __shfl_sync(0xffffffffu, k64[RR_ROWS - 1], 31));
  uint32_t wsurv, wshead, whead;
  rerank_warp_totals(H, after_is_head, wbase, m, wsurv, wshead, whead);
  if (lane == 0) { s_w[0][warp] = whead; s_w[1][warp] = wsurv; s_w[2][warp] = wshead; }
  __syncthreads();
  if (tid < 3) {
    uint32_t v = 0;
#pragma unroll
    for (int w = 0; w < RR_WARPS; ++w) v = tid ? v + s_w[tid][w] : max(v, s_w[0][w]);
    tsum[size_t(tid) * tiles + tile] = v;
  }
}

// K3c: the tile totals become, in place, exclusive carries (a max-scan for the last head -- it only grows along the
// tiles -- and sum-scans for survivors and surviving heads); totals[0] = all survivors, totals[1] = all surviving
// heads.  One CTA: warp w owns a contiguous run of tiles, reduces it, the 32 run totals are scanned, then every warp
// scans its run 32 tiles at a time (at most 2^31 / 4096 = 512 K tiles: a few tens of microseconds).
__global__ void __launch_bounds__(RR_CARRY_THREADS) rerank_carry_kernel(uint32_t* __restrict__ tsum, uint32_t tiles,
                                                                        uint32_t* __restrict__ totals) {
  constexpr int NW = RR_CARRY_THREADS / 32;
  __shared__ uint32_t s_w[3][NW];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t* th = tsum;
  uint32_t* ts = tsum + tiles;
  uint32_t* tg = tsum + 2 * size_t(tiles);
  const uint32_t run = ((tiles + NW - 1) / NW + 31) & ~31u;
  const uint32_t lo = min(tiles, warp * run), hi = min(tiles, lo + run);
  uint32_t h = 0, s = 0, g = 0;
  for (uint32_t j = lo + lane; j < hi; j += 32) { h = max(h, th[j]); s += ts[j]; g += tg[j]; }
  h = __reduce_max_sync(0xffffffffu, h);
  s = __reduce_add_sync(0xffffffffu, s);
  g = __reduce_add_sync(0xffffffffu, g);
  if (lane == 0) { s_w[0][warp] = h; s_w[1][warp] = s; s_w[2][warp] = g; }
  __syncthreads();
  uint32_t ch = 0, cs = 0, cg = 0;               // carries into the warp's run
  for (unsigned w = 0; w < warp; ++w) { ch = max(ch, s_w[0][w]); cs += s_w[1][w]; cg += s_w[2][w]; }
  if (threadIdx.x == RR_CARRY_THREADS - 1) { totals[0] = cs + s; totals[1] = cg + g; }
  for (uint32_t base = lo; base < hi; base += 32) {
    const uint32_t j = base + lane;
    const bool in = j < hi;
    const uint32_t vh = in ? th[j] : 0u, vs = in ? ts[j] : 0u, vg = in ? tg[j] : 0u;
    uint32_t ih = vh, is = vs, ig = vg;          // inclusive scans inside the 32 tiles
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t oh = __shfl_up_sync(0xffffffffu, ih, d), os = __shfl_up_sync(0xffffffffu, is, d),
                     og = __shfl_up_sync(0xffffffffu, ig, d);
      if (lane >= unsigned(d)) { ih = max(ih, oh); is += os; ig += og; }
    }
    const uint32_t eh = __shfl_up_sync(0xffffffffu, ih, 1);
    if (in) {
      th[j] = max(ch, lane ? eh : 0u);
      ts[j] = cs + is - vs;
      tg[j] = cg + ig - vg;
    }
    ch = max(ch, __shfl_sync(0xffffffffu, ih, 31));
    cs += __shfl_sync(0xffffffffu, is, 31);
    cg += __shfl_sync(0xffffffffu, ig, 31);
  }
}

struct RerankArgs {
  const uint32_t* heads;    // head mask of every row of 32 slots (K3h)
  const uint32_t* carry;    // per tile: (slot + 1) of the last head before it, survivors before it, surviving heads
                            //   before it, at carry[0 / tiles / 2 tiles + tile] (K3c)
  const uint32_t* idx;      // rotation start of every slot (sorted along with the keys)
  const uint32_t* sapos;    // SA position of every slot (NULL in round 0: slot == SA position)
  uint32_t m;
  uint32_t* sa;
  uint32_t* rnk;
  uint64_t* pairs;          // when set: (idx << 32 | rank) per slot instead of the random rank scatter, binned by
  uint32_t* part_cursor;    //   idx >> part_shift through [256] write cursors (order inside a bin is irrelevant:
  int part_shift;           //   every pair is a store to its own address)
  uint32_t* idx_out;        // compacted working set of the next round
  uint32_t* sapos_out;
  uint32_t* gd_out;         // dense group id of every survivor
  uint32_t tiles;
};

// Lane l of a warp holds slots wbase + 32 k + l (k = 0 .. RR_ROWS-1): every load and store of a row is
// one coalesced access, a slot's neighbours sit in the neighbouring lanes, and everything positional --
// the governing group head of a slot, how many survivors and surviving heads precede it -- comes from
// the head masks of the rows (one 32-bit word per row, the same in all lanes) with popc / clz.
// (A first version gave every thread 8-16 consecutive slots: ncu showed 22 sectors per store request
// and the L1 as the busiest unit.)
__global__ void __launch_bounds__(RR_THREADS) rerank_kernel(RerankArgs a) {
  __shared__ uint32_t s_whead[RR_WARPS], s_wsurv[RR_WARPS], s_wshead[RR_WARPS];
  __shared__ uint32_t s_bcnt[256], s_bstart[256], s_gbase[256];   // binned pairs: per-bin count, tile-local start, global start
  __shared__ uint32_t s_bscan[RR_WARPS];
  __shared__ uint64_t s_stage[RR_TILE];

  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  s_bcnt[tid] = 0;
  __syncthreads();
  const uint32_t tile = blockIdx.x;
  const uint32_t wbase = tile * RR_TILE + warp * RR_WCHUNK;      // < 2^32: m < 2^31
  const bool binned = a.pairs != nullptr;

  uint32_t idx[RR_ROWS], sap[RR_ROWS];
#pragma unroll
  for (int k = 0; k < RR_ROWS; ++k) {
    const uint32_t q = wbase + k * 32 + lane;
    const bool in = q < a.m;
    idx[k] = in ? a.idx[q] : 0;
    sap[k] = in ? (a.sapos ? a.sapos[q] : q) : 0;
  }
  // the warp's 16 head masks (64 aligned bytes, the same in every lane) and the first bit of the next warp's
  uint32_t H[RR_ROWS];
  const uint32_t rows = (a.m + 31) / 32, row0 = wbase / 32;
#pragma unroll
  for (int k = 0; k < RR_ROWS; k += 4) {
    uint4 v = make_uint4(0, 0, 0, 0);
    if (row0 + k + 3 < rows) v = *reinterpret_cast<const uint4*>(a.heads + row0 + k);
    else if (row0 + k < rows) {
      v.x = a.heads[row0 + k];
      v.y = row0 + k + 1 < rows ? a.heads[row0 + k + 1] : 0u;
      v.z = row0 + k + 2 < rows ? a.heads[row0 + k + 2] : 0u;
    }
    H[k] = v.x; H[k + 1] = v.y; H[k + 2] = v.z; H[k + 3] = v.w;
  }
  const bool after_is_head = (wbase + RR_WCHUNK >= a.m) || (a.heads[row0 + RR_ROWS] & 1u);
  // binned pairs, step 1: every slot takes a place in its bin (any order), bins get their sizes
  uint32_t bpos[RR_ROWS / 2];                       // two 16-bit places per register
  if (binned) {
#pragma unroll
    for (int k = 0; k < RR_ROWS; ++k) {
      const uint32_t q = wbase + k * 32 + lane;
      const uint32_t at = q < a.m ? atomicAdd(&s_bcnt[(idx[k] >> a.part_shift) & 255u], 1u) : 0u;
      bpos[k / 2] = (k & 1) ? (bpos[k / 2] | (at << 16)) : at;
    }
  }
  uint32_t wsurv, wshead, whead;
  rerank_warp_totals(H, after_is_head, wbase, a.m, wsurv, wshead, whead);
  if (lane == 0) { s_whead[warp] = whead; s_wsurv[warp] = wsurv; s_wshead[warp] = wshead; }
  __syncthreads();
  if (binned) {   // step 2: thread d owns bin d: room in the bin's global run, start inside the staging buffer
    const uint32_t c = s_bcnt[tid];
    uint32_t tot;
    s_bstart[tid] = block_exclusive_scan<uint32_t, RR_THREADS>(c, s_bscan, tot);
    s_gbase[tid] = c ? atomicAdd(&a.part_cursor[tid], c) : 0u;
  }
  uint32_t run_head = a.carry[tile];                           // (slot + 1) of the last head before the current row
  uint32_t out_at = a.carry[a.tiles + tile];                   // survivors before the current row
  uint32_t gd_run = a.carry[2 * size_t(a.tiles) + tile];       // surviving heads before the current row
#pragma unroll
  for (int w = 0; w < RR_WARPS; ++w) {
    if (unsigned(w) < warp) { run_head = max(run_head, s_whead[w]); out_at += s_wsurv[w]; gd_run += s_wshead[w]; }
  }

#pragma unroll
  for (int k = 0; k < RR_ROWS; ++k) {
    const uint32_t q = wbase + k * 32 + lane;
    uint32_t S, SH, L;
    const uint32_t next_first = k + 1 < RR_ROWS ? (H[k + 1 < RR_ROWS ? k + 1 : k] & 1u) : (after_is_head ? 1u : 0u);
    rerank_row_masks(H[k], next_first, wbase + k * 32, a.m, S, SH, L);
    const uint32_t le = lanemask_lt() | (1u << lane);
    const uint32_t hm = H[k] & le;
    const uint32_t my_head = hm ? wbase + k * 32 + (31 - __clz(hm)) + 1 : run_head;
    if (q < a.m) {
      // slots of one group are consecutive in SA, so the head's SA position is sap - distance
      const uint32_t rank = sap[k] - (q - (my_head - 1));
      // SA is final for a slot once its group is a single rotation; tied slots come back next round
      if ((L >> lane) & 1u) a.sa[sap[k]] = idx[k];
      if (binned) s_stage[s_bstart[(idx[k] >> a.part_shift) & 255u] + ((bpos[k / 2] >> ((k & 1) * 16)) & 0xFFFFu)] = (uint64_t(idx[k]) << 32) | rank;
      else a.rnk[idx[k]] = rank;
      if ((S >> lane) & 1u) {
        const uint32_t at = out_at + __popc(S & lanemask_lt());
        a.idx_out[at] = idx[k];
        a.sapos_out[at] = sap[k];
        a.gd_out[at] = gd_run + __popc(SH & le) - 1;
      }
    }
    if (H[k]) run_head = wbase + k * 32 + (31 - __clz(H[k])) + 1;
    out_at += __popc(S);
    gd_run += __popc(SH);
  }
  if (binned) {   // step 3: the staged pairs leave as one run per bin
    __syncthreads();
    const uint32_t tile_valid = min(uint32_t(RR_TILE), a.m - tile * RR_TILE);
    for (uint32_t j = tid; j < tile_valid; j += RR_THREADS) {
      const uint64_t pr = s_stage[j];
      const uint32_t d = (uint32_t(pr >> 32) >> a.part_shift) & 255u;
      a.pairs[s_gbase[d] + (j - s_bstart[d])] = pr;
    }
  }
}

// bin starts of the binned pairs: exclusive scan of the bin sizes
__global__ void __launch_bounds__(256) partition_cursor_kernel(const uint32_t* __restrict__ hist, uint32_t* __restrict__ cursor) {
  __shared__ uint32_t s_scan[8];
  uint32_t tot;
  cursor[threadIdx.x] = block_exclusive_scan<uint32_t, 256>(hist[threadIdx.x], s_scan, tot);
}

// K3b: ranks from (idx, rank) pairs that were partitioned by the top bits of idx
__global__ void __launch_bounds__(256) scatter_ranks_kernel(const uint64_t* __restrict__ pairs, uint32_t m,
                                                            uint32_t* __restrict__ rnk) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= m) return;
  const uint64_t p = pairs[q];
  rnk[uint32_t(p >> 32)] = uint32_t(p);
}

// ---------------------------------------------------------------------------------
// K4: key rebuild for the next doubling step (gather-bound) + the histograms of what it wrote
// ---------------------------------------------------------------------------------
// The kernel waits on random 4-byte gathers, so counting the digits of the keys it has in registers
// is free: the sort that follows needs no histogram pass over the keys, and the re-rank gets the
// bin sizes of its rank pairs (binned by the top bits of idx) without one over the indices.
struct RekeyHist {
  RadixShifts sh;
  int npass;
  uint32_t* hist;       // [npass][256]
  uint32_t* phist;      // [256]: digit (idx >> pshift), or NULL
  int pshift;
};
constexpr int RK_THREADS = 256;
constexpr int RK_ITEMS = 4;

__device__ __forceinline__ void hist_add(uint32_t* set, uint32_t d, bool full_warp, unsigned lane) {
  if (full_warp) {                       // one add of 32 where the whole warp agrees (sorted group ids, high rank bytes)
    const uint32_t d0 = __shfl_sync(0xffffffffu, d, 0);
    if (__all_sync(0xffffffffu, d == d0)) {
      if (lane == 0) atomicAdd(&set[d0], 32u);
      return;
    }
  }
  atomicAdd(&set[d], 1u);
}

__global__ void __launch_bounds__(RK_THREADS) rekey_kernel(const uint32_t* __restrict__ idx,
                                                           const uint32_t* __restrict__ gd,
                                                           const uint32_t* __restrict__ rnk, uint32_t m,
                                                           uint32_t n, uint32_t h, int tiebreak,
                                                           uint64_t* __restrict__ key, RekeyHist rh) {
  __shared__ uint32_t s_hist[2][kRadixMaxPasses + 1][256];        // two sets: even and odd warps
  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < 2 * (kRadixMaxPasses + 1) * 256; i += RK_THREADS) (&s_hist[0][0][0])[i] = 0;
  __syncthreads();
  uint32_t (*set)[256] = s_hist[warp & 1];
  const uint32_t chunk = RK_THREADS * RK_ITEMS;
  for (uint64_t base = uint64_t(blockIdx.x) * chunk; base < m; base += uint64_t(gridDim.x) * chunk) {
    uint32_t i[RK_ITEMS], second[RK_ITEMS], g[RK_ITEMS];
    bool in[RK_ITEMS];
#pragma unroll
    for (int u = 0; u < RK_ITEMS; ++u) {
      const uint64_t q = base + uint64_t(u) * RK_THREADS + tid;
      in[u] = q < m;
      i[u] = in[u] ? idx[q] : 0u;
    }
#pragma unroll
    for (int u = 0; u < RK_ITEMS; ++u) {
      if (tiebreak) {
        second[u] = i[u];                 // identical rotations: order by start index
      } else {
        uint64_t j = uint64_t(i[u]) + h;
        if (j >= n) j -= n;
        second[u] = in[u] ? rnk[j] : 0u;
      }
    }
#pragma unroll
    for (int u = 0; u < RK_ITEMS; ++u) {
      const uint64_t q = base + uint64_t(u) * RK_THREADS + tid;
      g[u] = in[u] ? gd[q] : 0u;
    }
#pragma unroll
    for (int u = 0; u < RK_ITEMS; ++u) {
      const uint64_t q = base + uint64_t(u) * RK_THREADS + tid;
      const uint64_t k = (uint64_t(g[u]) << 32) | second[u];
      if (in[u]) key[q] = k;
      const bool full_warp = __ballot_sync(0xffffffffu, in[u]) == 0xffffffffu;
      if (in[u] || full_warp) {
        for (int p = 0; p < rh.npass; ++p) hist_add(set[p], uint32_t(k >> rh.sh.s[p]) & 255u, full_warp, lane);
        if (rh.phist) hist_add(set[kRadixMaxPasses], (i[u] >> rh.pshift) & 255u, full_warp, lane);
      }
    }
  }
  __syncthreads();
  for (int j = tid; j < rh.npass * 256; j += RK_THREADS) {
    const uint32_t v = s_hist[0][j >> 8][j & 255] + s_hist[1][j >> 8][j & 255];
    if (v) atomicAdd(&rh.hist[j], v);
  }
  if (rh.phist) {
    const uint32_t v = s_hist[0][kRadixMaxPasses][tid] + s_hist[1][kRadixMaxPasses][tid];
    if (v) atomicAdd(&rh.phist[tid], v);
  }
}

// ---------------------------------------------------------------------------------
// K5: BWT gather  L[r] = T[(SA[r] - 1) mod n]   (bce.cpp:901-902 net effect)
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bwt_gather_kernel(const uint8_t* __restrict__ T,
                                                         const uint32_t* __restrict__ sa, uint32_t n,
                                                         uint8_t* __restrict__ L) {
  uint32_t r4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (r4 >= n) return;
  uint32_t out = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint32_t r = r4 + j;
    if (r < n) {
      uint32_t s = sa[r];
      uint32_t c = T[s ? s - 1 : n - 1];
      out |= c << (8 * j);
    }
  }
  if (r4 + 4 <= n) *reinterpret_cast<uint32_t*>(L + r4) = out;
  else for (int j = 0; r4 + j < n; ++j) L[r4 + j] = uint8_t(out >> (8 * j));
}

// The same through the inverse: after the last round rnk[i] is the SA row of rotation i, so L[rnk[i]] = T[i - 1].
// A one-byte store per row to a random address costs a DRAM sector each way (ncu, round 1: 39 B per row, 69 % DRAM
// busy, 19 ms at 1 GB).  Here the rows are binned first: K5a reads rnk and T as streams and writes (row inside its bin
// << 8 | byte) grouped by the row's top bits -- a counting sort of the tile in shared memory, one atomicAdd per
// (tile, bin) on the bin's cursor, one run per bin; the order inside a bin is irrelevant, every word is a store to its
// own address, and the bin sizes are arithmetic because rnk is a permutation -- and K5b stores from that order, so a
// bin's slice of L (n / 256 bytes) is filled while it sits in L2.  5 + 4 + 4 + 1 = 14 B per row of streams.
constexpr int BG_THREADS = 256, BG_ITEMS = 16, BG_TILE = BG_THREADS * BG_ITEMS;
__global__ void bwt_cursor_kernel(uint32_t* cursor, int shift) { cursor[threadIdx.x] = threadIdx.x << shift; }

__global__ void __launch_bounds__(BG_THREADS) bwt_bin_kernel(const uint8_t* __restrict__ T, const uint32_t* __restrict__ rnk,
                                                             uint32_t n, int shift, uint32_t* __restrict__ cursor,
                                                             uint32_t* __restrict__ pairs) {
  __shared__ uint32_t s_cnt[256], s_start[256], s_gbase[256];
  __shared__ uint32_t s_scan[BG_THREADS / 32];
  __shared__ uint32_t s_stage[BG_TILE];
  __shared__ uint8_t s_bin[BG_TILE];
  const unsigned tid = threadIdx.x;
  const uint32_t base = blockIdx.x * BG_TILE;
  s_cnt[tid] = 0;
  __syncthreads();
  uint32_t word[BG_ITEMS], pos[BG_ITEMS];
  const uint32_t mask = (1u << shift) - 1u;
#pragma unroll
  for (int k = 0; k < BG_ITEMS; ++k) {
    const uint32_t i = base + k * BG_THREADS + tid;
    word[k] = pos[k] = 0;
    if (i < n) {
      const uint32_t r = rnk[i];
      const uint32_t byte = T[i ? i - 1 : n - 1];
      const uint32_t bin = r >> shift;
      pos[k] = atomicAdd(&s_cnt[bin], 1u) | (bin << 16);         // place inside the tile's bin (any order will do); BG_TILE <= 65536
      word[k] = ((r & mask) << 8) | byte;
    }
  }
  __syncthreads();
  uint32_t tot;
  const uint32_t mine = s_cnt[tid];
  s_start[tid] = block_exclusive_scan<uint32_t, BG_THREADS>(mine, s_scan, tot);
  if (mine) s_gbase[tid] = atomicAdd(&cursor[tid], mine);
  __syncthreads();
#pragma unroll
  for (int k = 0; k < BG_ITEMS; ++k)
    if (base + k * BG_THREADS + tid < n) {
      const uint32_t at = s_start[pos[k] >> 16] + (pos[k] & 0xFFFFu);
      s_stage[at] = word[k];
      s_bin[at] = uint8_t(pos[k] >> 16);
    }
  __syncthreads();
  const uint32_t valid = min(uint32_t(BG_TILE), n - base);
  for (uint32_t j = tid; j < valid; j += BG_THREADS) {          // one run per bin
    const uint32_t bin = s_bin[j];
    pairs[s_gbase[bin] + (j - s_start[bin])] = s_stage[j];
  }
}

// rnk is a permutation of the rows, so bin b holds exactly the rows [b << shift, (b + 1) << shift) and its words sit
// at those positions of `pairs`
__global__ void __launch_bounds__(256) bwt_scatter_kernel(const uint32_t* __restrict__ pairs, uint32_t n, int shift,
                                                          uint8_t* __restrict__ L) {
  for (uint32_t j = blockIdx.x * 256u + threadIdx.x; j < n; j += gridDim.x * 256u) {
    const uint32_t p = pairs[j];
    L[((j >> shift) << shift) + (p >> 8)] = uint8_t(p);
  }
}

static inline int bits_for(uint32_t values) {   // bits needed for 0 .. values-1
  int b = 0;
  while (b < 32 && (uint64_t(1) << b) < values) ++b;
  return b ? b : 1;
}

// i >> top_byte_shift(n) is below 256 for every i < n: the bin of an index or an SA row in the binned rank update and BWT
static inline int top_byte_shift(uint32_t n) { return std::max(0, bits_for(n) - 8); }

// ---------------------------------------------------------------------------------
// The driver: setup, one doubling round after another, the BWT
// ---------------------------------------------------------------------------------
// Large working sets update the rank array through (idx, rank) pairs binned by the top 8 bits of idx: a random 4-byte
// store per slot into a 4n-byte array costs more than everything else in the re-rank together (each one a
// read-modify-write of a 32-byte sector); from the bins every 1/256 slice of the array stays in L2 while it is filled.
constexpr uint32_t kBinnedRanksMinSlots = 8u << 20;        // working sets of at least this many slots ...
constexpr size_t kBinnedRanksMinBytes = size_t(64) << 20;  // ... when the rank array is larger than this
// Texts of at least this many bytes (T does not fit L2 anyway) get their BWT through the inverse suffix array, binned
constexpr uint32_t kBinnedBwtMinN = 8u << 20;
// A round >= 1 keeps the tile-local sort while at most 1 / kLocalFallbackDiv of its slots lie in groups that cross a
// tile boundary (those go through the radix sort); the fall-back list is sized for that many
constexpr uint32_t kLocalFallbackDiv = 4;

// What a round does, known before its keys are made
struct RoundPlan {
  int shifts[kRadixMaxPasses];   // digits of an LSD sort of the round's keys, least significant first
  int np = 0;
  bool tiebreak = false;         // h >= n: the ties left are identical rotations, ordered by start index
  bool binned = false;           // ranks updated through pairs binned by idx >> part_shift (the key rebuild counts the bins)
  int part_shift = 0;
};

static RoundPlan plan_round(int round, uint32_t m, uint32_t n, uint64_t h, uint32_t groups, bool codes7) {
  RoundPlan p;
  p.binned = m >= kBinnedRanksMinSlots && size_t(n) * 4 > kBinnedRanksMinBytes;
  p.part_shift = top_byte_shift(n);
  if (round == 0) {                                    // key = the window of 8 bytes, or of 8 codes of 7 bits
    for (int s = 0; s < (codes7 ? 8 * kCodeBits : 64); s += 8) p.shifts[p.np++] = s;
    return p;
  }
  p.tiebreak = h >= n;
  const int nbits = bits_for(n), gbits = bits_for(groups);
  for (int s = 0; s < nbits; s += 8) p.shifts[p.np++] = s;                                       // rank (or index)
  for (int s = 0; s < gbits && p.np < kRadixMaxPasses; s += 8) p.shifts[p.np++] = 32 + s;      // dense group id
  return p;
}

// The sort's read-backs, in pinned host memory past the radix sort's histograms and digit starts
struct SortReadback {
  uint32_t totals[2];   // re-rank: survivors, surviving groups
  uint32_t err;         // chained-scan watchdog of the radix passes
  uint32_t fb_total;    // slots the tile-local sort hands to the radix sort
  uint32_t offset;      // SA[0]
  uint32_t bins[256];   // round 0: sizes of the rank-pair bins
};
constexpr size_t kPinnedSortReadback = 32 * 1024;

// Device buffers of the sort, carved once.  Of a pair, [0] is what the round works on; a round leaves the next round's
// working set in idx / sapos / gd [1], and next_round() exchanges them.
struct SortBuffers {
  uint64_t* key[2];      // the round's keys are made in [0]; a sort into [1] swaps the key and idx pairs; [1] then holds
                         // the binned rank pairs
  uint32_t* idx[2];      // rotation start of every slot
  uint32_t* sapos[2];    // SA position of every slot (round 0: the slot itself, [0] not read)
  uint32_t* gd[2];       // dense group id of every slot
  uint32_t* sa;
  uint32_t* rnk;
  uint64_t* fb_key[2];   // fall-back list of the tile-local sort (local_sort.cuh), ping-ponged by its radix sort
  uint32_t* fb_idx[2];
  uint32_t* fb_slot;
  uint32_t *lt_pre, *lt_suf, *lt_cnt, *lt_off;                          // per tile of the tile-local sort
  uint32_t* rr_heads;    // re-rank: head mask of every row of 32 slots
  uint32_t* rr_tsum;     // re-rank: 3 x tiles totals, then carries
  uint32_t* pair_hist;   // round 0 on 7-bit codes: [128 x 128] code pairs (the coded text itself lives in rnk, which
                         //   round 0 first writes in its re-rank)
  uint32_t *err, *totals, *fb_total, *hist, *part_hist, *part_cursor;   // in Ctx::small
  SortReadback* rb;

  void next_round() {
    std::swap(idx[0], idx[1]);
    std::swap(sapos[0], sapos[1]);
    std::swap(gd[0], gd[1]);
  }
};

static int carve(Ctx* c, uint32_t n, SortBuffers& b) {
  const size_t N = n, FB = N / kLocalFallbackDiv + 1, LT = N / LS_TILE + 2;
  const size_t RH = (N + 31) / 32, RT = 3 * ((N + RR_TILE - 1) / RR_TILE);
  const size_t need = 2 * Carver::need(N, 8) + 8 * Carver::need(N, 4) + 2 * Carver::need(FB, 8) +
                      3 * Carver::need(FB, 4) + 4 * Carver::need(LT, 4) + Carver::need(RH, 4) + Carver::need(RT, 4) +
                      Carver::need(kCodes * kCodes, 4) + 4096;
  BCE_TRY(c->scratch.ensure(c, need));
  Carver cv(c->scratch.p, c->scratch.cap);
  for (auto& k : b.key) k = cv.take<uint64_t>(N);
  for (auto& v : b.idx) v = cv.take<uint32_t>(N);
  b.sa = cv.take<uint32_t>(N);
  b.rnk = cv.take<uint32_t>(N);
  for (auto& v : b.sapos) v = cv.take<uint32_t>(N);
  for (auto& v : b.gd) v = cv.take<uint32_t>(N);
  for (auto& k : b.fb_key) k = cv.take<uint64_t>(FB);
  for (auto& v : b.fb_idx) v = cv.take<uint32_t>(FB);
  b.fb_slot = cv.take<uint32_t>(FB);
  b.lt_pre = cv.take<uint32_t>(LT);
  b.lt_suf = cv.take<uint32_t>(LT);
  b.lt_cnt = cv.take<uint32_t>(LT);
  b.lt_off = cv.take<uint32_t>(LT);
  b.rr_heads = cv.take<uint32_t>(RH);
  b.rr_tsum = cv.take<uint32_t>(RT);
  b.pair_hist = cv.take<uint32_t>(kCodes * kCodes);
  if (!cv.ok()) { set_error(c, "suffix sort: scratch carve failed"); return BCE_GPU_E_NOMEM; }

  char* small = c->small.as<char>();
  b.err = reinterpret_cast<uint32_t*>(small + kSmallErr);
  b.totals = reinterpret_cast<uint32_t*>(small + kSmallRerankTotals);
  b.fb_total = b.totals + 3;
  b.hist = reinterpret_cast<uint32_t*>(small + kSmallHist);
  b.part_hist = reinterpret_cast<uint32_t*>(small + kSmallPartHist);
  b.part_cursor = reinterpret_cast<uint32_t*>(small + kSmallPartCursor);
  b.rb = reinterpret_cast<SortReadback*>(c->pinned_small.as<char>() + kPinnedSortReadback);
  return BCE_GPU_OK;
}

// Adds the stream's time since the last lap to acc (synchronises).
static int lap(Ctx* c, float& acc) {
  BCE_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  BCE_CUDA(c, cudaEventSynchronize(c->ev[1]));
  float ms = 0;
  BCE_CUDA(c, cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
  acc += ms;
  BCE_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  return BCE_GPU_OK;
}

// Round 0's keys are the 8-symbol windows of T or, when 2 .. 128 byte values occur, of its 7-bit codes (written to
// b.rnk); *text receives the one the keys are made from.  Either way the digit histograms of every pass of the round
// end in the host mirror of the radix sort's histograms, from one read of T for the byte histogram and, with codes,
// one more that codes it and counts its code pairs.
static int round0_text(Ctx* c, SortBuffers& b, uint32_t n, const uint8_t** text, bool* codes7) {
  cudaStream_t st = c->stream;
  const uint8_t* T = c->text.as<uint8_t>();
  uint32_t* h_hist = c->pinned_small.as<uint32_t>();
  BCE_CUDA(c, cudaMemsetAsync(b.hist, 0, 256 * 4, st));
  byte_hist_launch(c, T, n, b.hist);
  c->stats.gpu_launches++;
  BCE_CUDA(c, cudaGetLastError());
  BCE_CUDA(c, cudaMemcpyAsync(h_hist, b.hist, 256 * 4, cudaMemcpyDeviceToHost, st));
  BCE_CUDA(c, cudaStreamSynchronize(st));
  CodeTable tab;
  uint32_t sigma = 0;
  for (int v = 0; v < 256; ++v) tab.v[v] = uint8_t(h_hist[v] ? sigma++ : 0);
  *codes7 = sigma >= 2 && sigma <= uint32_t(kCodes);
  BCE_TRACE("round 0: %u byte values, keys from %s", sigma, *codes7 ? "7-bit codes" : "bytes");
  if (!*codes7) {               // byte p of key i is T[(i + 7 - p) mod n]: every digit has the byte histogram
    *text = T;
    for (int p = 7; p >= 0; --p)
      for (int d = 0; d < 256; ++d) h_hist[p * 256 + d] = h_hist[d];
    return BCE_GPU_OK;
  }
  uint8_t* C = reinterpret_cast<uint8_t*>(b.rnk);
  BCE_CUDA(c, cudaMemsetAsync(b.pair_hist, 0, kPairHistSmem, st));
  const uint32_t words = (n + 16 + 3) / 4, want = (words + 255) / 256, most = uint32_t(c->sm_count) * 3;
  code_text_kernel<<<want < most ? want : most, 256, kPairHistSmem, st>>>(T, n, tab, C, b.pair_hist);
  digit_hist_kernel<<<kCodeBits, 256, 0, st>>>(b.pair_hist, b.hist);
  c->stats.gpu_launches += 2;
  BCE_CUDA(c, cudaGetLastError());
  BCE_CUDA(c, cudaMemcpyAsync(h_hist, b.hist, kCodeBits * 256 * 4, cudaMemcpyDeviceToHost, st));
  BCE_CUDA(c, cudaStreamSynchronize(st));
  *text = C;
  return BCE_GPU_OK;
}

int sort_init_device(Ctx* c) {
  BCE_CUDA(c, cudaFuncSetAttribute(code_text_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kPairHistSmem)));
  return BCE_GPU_OK;
}

// Orders the working set by the round's keys; they and the indices end sorted in b.key[0] / b.idx[0].  Round 0: radix
// passes whose first makes the keys from the text.  Later rounds: tile by tile (local_sort.cuh, the keys made on the
// way) plus a radix sort of the slots in groups that cross a tile boundary, or, where those are too many or the
// working set is small, rekey_kernel and radix passes.
static int sort_round(Ctx* c, SortBuffers& b, const RoundPlan& p, int round, uint32_t m, uint32_t n, uint64_t h,
                      const uint8_t* text0, bool codes7) {
  cudaStream_t st = c->stream;
  bce_gpu_stats& S = c->stats;
  const uint32_t second_h = uint32_t(p.tiebreak ? 0 : h);
  const uint32_t ltiles = (m + LS_TILE - 1) / LS_TILE;
  bool local = false;
  if (round > 0 && m >= c->local_sort_min) {
    ls_classify_kernel<<<(ltiles + 255) / 256, 256, 0, st>>>(b.gd[0], m, ltiles, b.lt_pre, b.lt_suf, b.lt_cnt);
    ls_scan_kernel<<<1, 1024, 0, st>>>(b.lt_cnt, ltiles, b.lt_off, b.fb_total);
    S.gpu_launches += 2;
    BCE_CUDA(c, cudaGetLastError());
    BCE_CUDA(c, cudaMemcpyAsync(&b.rb->fb_total, b.fb_total, 4, cudaMemcpyDeviceToHost, st));
    BCE_CUDA(c, cudaStreamSynchronize(st));
    BCE_TRACE("local sort round %d: %u of %u slots in groups that cross a tile boundary", round, b.rb->fb_total, m);
    local = b.rb->fb_total <= m / kLocalFallbackDiv;
  }
  const uint32_t m_fb = local ? b.rb->fb_total : 0;
  if (local) {
    if (p.binned) {        // bin sizes of the rank pairs (rekey_kernel counts them on the other path)
      BCE_CUDA(c, cudaMemsetAsync(b.part_hist, 0, 256 * 4, st));
      const uint32_t want = (m + 255) / 256, most = uint32_t(c->sm_count) * 8;
      ls_idx_hist_kernel<<<want < most ? want : most, 256, 0, st>>>(b.idx[0], m, p.part_shift, b.part_hist);
      S.gpu_launches++;
    }
    BCE_TRY(lap(c, S.ms_rekey));
  } else if (round > 0) {  // working-set slot -> key of the next doubling step, digit histograms counted on the way
    RekeyHist rh;
    for (int i = 0; i < kRadixMaxPasses; ++i) rh.sh.s[i] = i < p.np ? p.shifts[i] : 0;
    rh.npass = p.np;
    rh.hist = b.hist;
    rh.phist = p.binned ? b.part_hist : nullptr;
    rh.pshift = p.part_shift;
    BCE_CUDA(c, cudaMemsetAsync(b.hist, 0, kRadixMaxPasses * 256 * 4, st));
    BCE_CUDA(c, cudaMemsetAsync(b.part_hist, 0, 256 * 4, st));
    const uint32_t chunk = RK_THREADS * RK_ITEMS;
    const uint32_t want = (m + chunk - 1) / chunk, most = uint32_t(c->sm_count) * 8;
    rekey_kernel<<<want < most ? want : most, RK_THREADS, 0, st>>>(b.idx[0], b.gd[0], b.rnk, m, n, second_h,
                                                                   p.tiebreak ? 1 : 0, b.key[0], rh);
    S.gpu_launches++;
    BCE_CUDA(c, cudaGetLastError());
    BCE_TRY(lap(c, S.ms_rekey));
  }
  BCE_TRACE("sort round %d m=%u h=%llu tiebreak=%d passes<=%d", round, m, (unsigned long long)h, int(p.tiebreak), p.np);
  int ran = 0;
  if (local) {
    LocalSortArgs la;
    la.vin = b.idx[0]; la.gd = b.gd[0]; la.rnk = b.rnk;
    la.n = n; la.h = second_h; la.tiebreak = p.tiebreak ? 1 : 0;
    la.kout = b.key[1]; la.vout = b.idx[1]; la.m = m;
    la.pre = b.lt_pre; la.suf = b.lt_suf; la.off = b.lt_off;
    la.fb_key = b.fb_key[0]; la.fb_idx = b.fb_idx[0]; la.fb_slot = b.fb_slot;
    ls_sort_kernel<<<ltiles, LS_THREADS, 0, st>>>(la);
    S.gpu_launches++;
    BCE_CUDA(c, cudaGetLastError());
    if (m_fb) {
      uint64_t* sk; uint32_t* sv; int fran = 0;
      BCE_TRY(radix_sort_pairs(c, b.fb_key[0], b.fb_key[1], b.fb_idx[0], b.fb_idx[1], m_fb, p.shifts, p.np, &sk, &sv,
                               &fran, nullptr));
      ls_place_kernel<<<(m_fb + 255) / 256, 256, 0, st>>>(sk, sv, b.fb_slot, m_fb, b.key[1], b.idx[1]);
      S.gpu_launches++;
      BCE_CUDA(c, cudaGetLastError());
    }
    std::swap(b.key[0], b.key[1]);
    std::swap(b.idx[0], b.idx[1]);
    ran = p.np;                          // reported as the passes an LSD sort of these keys would take
    S.sort_local_elems += m;
    S.sort_fallback_elems += m_fb;
  } else {
    RadixHistSource src;
    if (round == 0) { src.window_text = text0; src.codes7 = codes7; src.host_hist = true; }
    else src.dev_hist = b.hist;
    uint64_t* ks; uint32_t* vs;
    BCE_TRY(radix_sort_pairs(c, b.key[0], b.key[1], b.idx[0], b.idx[1], m, p.shifts, p.np, &ks, &vs, &ran, &src));
    if (ks != b.key[0]) {
      std::swap(b.key[0], b.key[1]);
      std::swap(b.idx[0], b.idx[1]);
    }
    if (round == 0 && ran == 0) {        // every window is the same byte repeated: no pass ran, nothing made the keys
      pack_keys_kernel<<<(n + 256 * PK_ROWS - 1) / (256 * PK_ROWS), 256, 0, st>>>(text0, n, codes7, b.key[0], b.idx[0]);
      S.gpu_launches++;
    }
  }
  BCE_TRY(lap(c, S.ms_radix));
  S.sort_m[round] = m;
  S.sort_passes[round] = uint32_t(ran);
  S.sort_radix_passes[round] = local ? 0u : uint32_t(ran);
  S.sort_rounds = uint32_t(round + 1);
  return BCE_GPU_OK;
}

// Re-rank: SA and rank for every slot; the still-tied slots go, compacted, to idx / sapos / gd [1].  Returns the next
// round's working-set size and group count.
static int rerank_round(Ctx* c, SortBuffers& b, const RoundPlan& p, int round, uint32_t m, uint32_t n,
                        uint32_t* m_next, uint32_t* groups) {
  cudaStream_t st = c->stream;
  bce_gpu_stats& S = c->stats;
  RerankArgs a;
  a.tiles = (m + RR_TILE - 1) / RR_TILE;
  rerank_heads_kernel<<<a.tiles, RR_THREADS, 0, st>>>(b.key[0], m, b.rr_heads, b.rr_tsum, a.tiles);
  rerank_carry_kernel<<<1, RR_CARRY_THREADS, 0, st>>>(b.rr_tsum, a.tiles, b.totals);
  S.gpu_launches += 2;
  BCE_CUDA(c, cudaGetLastError());
  a.heads = b.rr_heads; a.carry = b.rr_tsum; a.idx = b.idx[0]; a.sapos = round ? b.sapos[0] : nullptr; a.m = m;
  a.sa = b.sa; a.rnk = b.rnk;
  a.pairs = nullptr; a.part_cursor = nullptr; a.part_shift = p.part_shift;
  if (p.binned) {
    if (round == 0) {                  // every idx in [0, n) is present: the bin sizes are arithmetic
      for (uint32_t d = 0; d < 256; ++d) {
        const uint64_t lo = uint64_t(d) << p.part_shift, hi = uint64_t(d + 1) << p.part_shift;
        b.rb->bins[d] = uint32_t(lo >= n ? 0 : (hi < n ? hi : n) - lo);
      }
      BCE_CUDA(c, cudaMemcpyAsync(b.part_hist, b.rb->bins, 256 * 4, cudaMemcpyHostToDevice, st));
    }                                  // later rounds: counted over the working set by sort_round
    partition_cursor_kernel<<<1, 256, 0, st>>>(b.part_hist, b.part_cursor);
    S.gpu_launches++;
    a.pairs = b.key[1];
    a.part_cursor = b.part_cursor;
  }
  a.idx_out = b.idx[1]; a.sapos_out = b.sapos[1]; a.gd_out = b.gd[1];
  rerank_kernel<<<a.tiles, RR_THREADS, 0, st>>>(a);
  S.gpu_launches++;
  BCE_CUDA(c, cudaGetLastError());
  BCE_CUDA(c, cudaMemcpyAsync(b.rb->totals, b.totals, 8, cudaMemcpyDeviceToHost, st));
  BCE_CUDA(c, cudaMemcpyAsync(&b.rb->err, b.err, 4, cudaMemcpyDeviceToHost, st));   // the round's radix passes
  float before = S.ms_rerank;
  BCE_TRY(lap(c, S.ms_rerank));
  BCE_TRACE("rerank round %d m=%u: %.3f ms (rank pairs partitioned=%d)", round, m, S.ms_rerank - before, int(p.binned));
  if (p.binned) {
    scatter_ranks_kernel<<<(m + 255) / 256, 256, 0, st>>>(b.key[1], m, b.rnk);
    S.gpu_launches++;
    BCE_CUDA(c, cudaGetLastError());
    before = S.ms_rerank;
    BCE_TRY(lap(c, S.ms_rerank));
    BCE_TRACE("rank scatter: %.3f ms", S.ms_rerank - before);
  }
  if (b.rb->err) { set_error(c, "suffix sort: chained-scan watchdog fired"); return BCE_GPU_E_INTERNAL; }
  *m_next = b.rb->totals[0];
  *groups = b.rb->totals[1];
  if (p.tiebreak && *m_next) { set_error(c, "suffix sort: ties left after index tie-break"); return BCE_GPU_E_INTERNAL; }
  return BCE_GPU_OK;
}

// L[r] = T[(SA[r] - 1) mod n] and offset = SA[0].  Texts that do not fit L2 go through the inverse (binned rows); that
// needs rnk to be the inverse suffix array, which it is unless identical rotations were told apart by index (then
// equal rotations share a rank).
static int bwt_step(Ctx* c, const SortBuffers& b, uint32_t n, bool had_tiebreak) {
  cudaStream_t st = c->stream;
  const uint8_t* T = c->text.as<uint8_t>();
  uint8_t* L = c->bwt.as<uint8_t>();
  if (!had_tiebreak && n >= kBinnedBwtMinN) {
    const int shift = top_byte_shift(n);
    uint32_t* rows = reinterpret_cast<uint32_t*>(b.key[0]);          // the sort's buffers are dead
    BCE_TRACE("bwt binned shift=%d: positions binned through the inverse suffix array", shift);
    bwt_cursor_kernel<<<1, 256, 0, st>>>(b.part_cursor, shift);
    bwt_bin_kernel<<<(n + BG_TILE - 1) / BG_TILE, BG_THREADS, 0, st>>>(T, b.rnk, n, shift, b.part_cursor, rows);
    bwt_scatter_kernel<<<(n + 255) / 256, 256, 0, st>>>(rows, n, shift, L);
    c->stats.gpu_launches += 3;
  } else {
    BCE_TRACE("bwt gather: bytes gathered through the suffix array (tie-break ran: %d)", int(had_tiebreak));
    bwt_gather_kernel<<<((n + 3) / 4 + 255) / 256, 256, 0, st>>>(T, b.sa, n, L);
    c->stats.gpu_launches++;
  }
  BCE_CUDA(c, cudaGetLastError());
  BCE_CUDA(c, cudaMemcpyAsync(&b.rb->offset, b.sa, 4, cudaMemcpyDeviceToHost, st));
  BCE_TRY(lap(c, c->stats.ms_bwt_gather));
  c->offset = b.rb->offset;
  return BCE_GPU_OK;
}

int suffix_sort_bwt(Ctx* c, uint32_t n, uint32_t* sa_host) {
  BCE_TRY(c->bwt.ensure(c, size_t(n) + 64));
  SortBuffers b;
  BCE_TRY(carve(c, n, b));
  BCE_CUDA(c, cudaMemsetAsync(b.err, 0, 64, c->stream));
  bce_gpu_stats& S = c->stats;
  S.sort_rounds = 0;
  c->pass_ev_n = 0;

  BCE_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  pad_cyclic_kernel<<<1, 64, 0, c->stream>>>(c->text.as<uint8_t>(), n);
  S.gpu_launches++;
  BCE_CUDA(c, cudaGetLastError());
  BCE_TRY(lap(c, S.ms_pack));

  const uint8_t* text0 = nullptr;
  bool codes7 = false;
  BCE_TRY(round0_text(c, b, n, &text0, &codes7));
  BCE_TRY(lap(c, S.ms_radix));

  uint32_t m = n, groups = 0;
  uint64_t h = 8;                 // rounds >= 1: the groups agree on h bytes, the key's second half starts h bytes on
  bool had_tiebreak = false;      // identical rotations were ordered by index: rnk is then not a permutation
  for (int round = 0; m > 0; ++round) {
    if (round >= kMaxSortRounds) { set_error(c, "suffix sort: too many rounds"); return BCE_GPU_E_INTERNAL; }
    const RoundPlan p = plan_round(round, m, n, h, groups, codes7);
    had_tiebreak |= p.tiebreak;
    BCE_TRY(sort_round(c, b, p, round, m, n, h, text0, codes7));
    BCE_TRY(rerank_round(c, b, p, round, m, n, &m, &groups));
    b.next_round();
    if (round > 0) h *= 2;
  }
  BCE_TRY(bwt_step(c, b, n, had_tiebreak));

  for (int i = 0; i + 1 < c->pass_ev_n; i += 2) {      // the stream is idle here (lap synchronised)
    float pms = 0;
    if (cudaEventElapsedTime(&pms, c->pass_ev[i], c->pass_ev[i + 1]) == cudaSuccess) S.ms_radix_kernel += pms;
  }
  c->pass_ev_n = 0;
  c->bwt_resident = true;
  if (sa_host) BCE_TRY(d2h(c, sa_host, b.sa, size_t(n) * 4));
  return BCE_GPU_OK;
}

}  // namespace bce
