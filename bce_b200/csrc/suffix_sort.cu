// suffix_sort.cu -- stage A: cyclic suffix sort and BWT on the device.
//
// Replaces File::rotate (bce.cpp:858-894) and File::bwt / divbwt (bce.cpp:896-910).
// The reference rotates the text to its least rotation and suffix-sorts it with
// libdivsufsort; the net effect (SURVEY.md 4-2) is the BWT of the *cyclic rotations*
// of T with row 0 = least rotation and offset = its start index.  Here all n rotations
// are sorted directly by prefix doubling over packed rank keys:
//
//   round 0   key(i) = 8 bytes T[i..i+8) (cyclic, big-endian); LSD radix sort of (key, i); the first
//             pass makes the keys from the text and is unordered (radix_sort.cu)
//   re-rank   rank[i] = SA position of the head of i's group; rotations alone in their
//             group are final and leave the working set
//   round r   key = (dense group id << 32) | rank[(i + h) mod n], h = 8 * 2^(r-1); the groups are
//             short, so the working set is sorted tile by tile (local_sort.cuh; the tile sort makes
//             its keys itself) and only groups that cross a tile boundary are radix-sorted;
//             groups stay where they are, so the list slot of an element fixes its SA position
//   end       working set empty, or h >= n (T is a power w^k: remaining ties are identical
//             rotations, ordered by index so that offset is the smallest one)
//
// Kernels here: K1 pack (only without the fused first pass), K3 re-rank + stable compaction + binned rank
// pairs (single pass, chained scans), K3b rank scatter, K4 key rebuild with digit histograms (radix path
// of small or declined rounds), K5 BWT gather.
#include <stdlib.h>

#include <algorithm>

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
// K1: pack 8-byte big-endian keys; one thread makes the 8 keys of an aligned octet
// ---------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t bswap64(uint64_t v) {
  uint32_t lo = uint32_t(v), hi = uint32_t(v >> 32);
  return (uint64_t(__byte_perm(lo, 0, 0x0123)) << 32) | __byte_perm(hi, 0, 0x0123);
}

// Thread t of a CTA makes keys tile + 256 r + t (r = 0 .. 7): the 12 bytes a key and its index take are
// written as coalesced rows (the first version wrote 64 bytes per thread: 32 sectors per store request).
constexpr int PK_ROWS = 8;

__global__ void __launch_bounds__(256) pack_keys_kernel(const uint8_t* __restrict__ T, uint32_t n,
                                                        uint64_t* __restrict__ keys,
                                                        uint32_t* __restrict__ idx) {
  const uint64_t* T64 = reinterpret_cast<const uint64_t*>(T);
  const uint32_t tile = blockIdx.x * (256 * PK_ROWS);
#pragma unroll
  for (int r = 0; r < PK_ROWS; ++r) {
    const uint32_t i = tile + r * 256 + threadIdx.x;
    if (i < n) {
      // the text is cyclic for 64 bytes past n (pad_cyclic_kernel), so both words exist
      const uint64_t a = bswap64(T64[i >> 3]), b = bswap64(T64[(i >> 3) + 1]);
      const uint32_t sh = (i & 7u) * 8;
      keys[i] = sh ? (a << sh) | (b >> (64 - sh)) : a;
      idx[i] = i;
    }
  }
}

// ---------------------------------------------------------------------------------
// K3: re-rank + stable compaction of the rotations that are still tied
// ---------------------------------------------------------------------------------
constexpr int RR_THREADS = 256;
constexpr int RR_WARPS = RR_THREADS / 32;
#ifndef BCE_RR_ROWS
#define BCE_RR_ROWS 16
#endif
constexpr int RR_ROWS = BCE_RR_ROWS;                // rows of 32 consecutive slots per warp
constexpr int RR_WCHUNK = 32 * RR_ROWS;             // slots per warp
constexpr int RR_TILE = RR_WARPS * RR_WCHUNK;       // 4096 slots per tile
#ifndef BCE_RR_LOOKBACK
#define BCE_RR_LOOKBACK 4
#endif
constexpr int RR_LOOKBACK = BCE_RR_LOOKBACK;        // descriptors x 32 fetched per step of the two sum scans

struct RerankArgs {
  const uint64_t* key;      // sorted keys of the working set
  const uint32_t* idx;      // rotation start of every slot (sorted along with the keys)
  const uint32_t* sapos;    // SA position of every slot (NULL in round 0: slot == SA position)
  uint32_t m;
  uint32_t* sa;
  uint32_t* rnk;
  uint64_t* pairs;          // when set: (idx << 32 | rank) per slot instead of the random rank scatter
  uint32_t* part_cursor;    // when set: [256] write cursors; the pairs go out binned by idx >> part_shift
  int part_shift;           //   (order inside a bin is irrelevant: every pair is a store to its own address)
  uint32_t* idx_out;        // compacted working set of the next round
  uint32_t* sapos_out;
  uint32_t* gd_out;         // dense group id of every survivor
  uint32_t* totals;         // [0] survivors, [1] surviving groups
  uint64_t* desc;           // 3 x tiles tagged descriptors
  uint32_t tiles;
  uint32_t* ticket;
  uint32_t tag;
  uint32_t* err;
  uint32_t dbg;             // timing experiments only: 1 no rank scatter, 2 no SA write, 4 no compaction writes
};

// Lane l of a warp holds slots wbase + 32 k + l (k = 0 .. RR_ROWS-1): every load and store of a row is
// one coalesced access, a slot's neighbours sit in the neighbouring lanes, and everything positional --
// the governing group head of a slot, how many survivors and surviving heads precede it -- comes from
// ballot masks of the rows (one 32-bit word per row, the same in all lanes) with popc / clz.
// (A first version gave every thread 8-16 consecutive slots: ncu showed 22 sectors per store request
// and the L1 as the busiest unit.)
// timing experiments (parts of the kernel switched off, results wrong) exist in experiment builds only
#ifdef BCE_GPU_EXPERIMENTS
#define RR_DBG(a) ((a).dbg)
#else
#define RR_DBG(a) 0u
#endif

__global__ void __launch_bounds__(RR_THREADS) rerank_kernel(RerankArgs a) {
  __shared__ uint32_t s_whead[RR_WARPS], s_wsurv[RR_WARPS], s_wshead[RR_WARPS];
  __shared__ uint32_t s_tile;
  __shared__ uint32_t s_carry[3];
  __shared__ uint32_t s_bcnt[256], s_bstart[256], s_gbase[256];   // binned pairs: per-bin count, tile-local start, global start
  __shared__ uint32_t s_bscan[RR_WARPS];
  __shared__ uint64_t s_stage[RR_TILE];

  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(a.ticket, 1u);
  s_bcnt[tid] = 0;
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint32_t wbase = tile * RR_TILE + warp * RR_WCHUNK;      // < 2^32: m < 2^31
  const bool binned = a.pairs && a.part_cursor;

  uint64_t key[RR_ROWS];
  uint32_t idx[RR_ROWS], sap[RR_ROWS];
#pragma unroll
  for (int k = 0; k < RR_ROWS; ++k) {
    const uint32_t q = wbase + k * 32 + lane;
    const bool in = q < a.m;
    key[k] = in ? a.key[q] : 0;
    idx[k] = in ? a.idx[q] : 0;
    sap[k] = in ? (a.sapos ? a.sapos[q] : q) : 0;
  }
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
  // the keys just outside the warp's chunk (uniform loads)
  const uint64_t key_before = (wbase > 0 && wbase - 1 < a.m) ? a.key[wbase - 1] : 0;
  const uint64_t key_after = (wbase + RR_WCHUNK < a.m) ? a.key[wbase + RR_WCHUNK] : 0;

  // head = first slot of a (new) group
  uint32_t H[RR_ROWS];
#pragma unroll
  for (int k = 0; k < RR_ROWS; ++k) {
    const uint32_t q = wbase + k * 32 + lane;
    const uint64_t up = __shfl_up_sync(0xffffffffu, key[k], 1);
    const uint64_t wrap = k ? __shfl_sync(0xffffffffu, key[k ? k - 1 : 0], 31) : key_before;
    const uint64_t prev = lane ? up : wrap;
    H[k] = __ballot_sync(0xffffffffu, q < a.m && (q == 0 || key[k] != prev));
  }
  // is the slot after the warp's last one a head (or the end)?
  const bool after_is_head = (wbase + RR_WCHUNK >= a.m) ||
                             (key_after != __shfl_sync(0xffffffffu, key[RR_ROWS - 1], 31));
  // lone = a group of one: head whose successor is a head (or the end of the working set).  H[k] is the same in all
  // lanes, so the three masks of a row are a handful of bit operations, no further ballots:
  //   L lone slots, S survivors (tied slots), SH surviving heads
  auto masks = [&](int k, uint32_t& S, uint32_t& SH, uint32_t& L) {
    const uint32_t rowbase = wbase + k * 32;
    const uint32_t valid = rowbase >= a.m ? 0u : a.m - rowbase;                   // slots of the row below m
    const uint32_t in_mask = valid >= 32u ? 0xFFFFFFFFu : (1u << valid) - 1u;
    const uint32_t next_first = k + 1 < RR_ROWS ? (H[k + 1 < RR_ROWS ? k + 1 : k] & 1u) : (after_is_head ? 1u : 0u);
    uint32_t nh = (H[k] >> 1) | (next_first << 31);                               // the slot behind is a head ...
    if (valid <= 32u) nh |= valid ? ~((1u << (valid - 1u)) - 1u) : 0xFFFFFFFFu;   // ... or does not exist
    L = H[k] & nh & in_mask;
    S = in_mask & ~L;
    SH = H[k] & ~L;
  };
  uint32_t wsurv = 0, wshead = 0, whead = 0;          // this warp's survivors, surviving heads, (slot + 1) of its last head
#pragma unroll
  for (int k = 0; k < RR_ROWS; ++k) {
    uint32_t S, SH, L;
    masks(k, S, SH, L);
    wsurv += __popc(S);
    wshead += __popc(SH);
    if (H[k]) whead = wbase + k * 32 + (31 - __clz(H[k])) + 1;
  }
  if (lane == 0) { s_whead[warp] = whead; s_wsurv[warp] = wsurv; s_wshead[warp] = wshead; }
  __syncthreads();
  if (binned) {   // step 2: thread d owns bin d: room in the bin's global run, start inside the staging buffer
    const uint32_t c = s_bcnt[tid];
    uint32_t tot;
    s_bstart[tid] = block_exclusive_scan<uint32_t, RR_THREADS>(c, s_bscan, tot);
    s_gbase[tid] = c ? atomicAdd(&a.part_cursor[tid], c) : 0u;
  }
  uint32_t head_before = 0, surv_before = 0, shead_before = 0, tile_head = 0, tile_surv = 0, tile_shead = 0;
#pragma unroll
  for (int w = 0; w < RR_WARPS; ++w) {
    const uint32_t hv = s_whead[w], sv = s_wsurv[w], shv = s_wshead[w];
    if (unsigned(w) < warp) { head_before = max(head_before, hv); surv_before += sv; shead_before += shv; }
    tile_head = max(tile_head, hv);
    tile_surv += sv;
    tile_shead += shv;
  }
  // carries across tiles: three independent chained scans, one warp each
  if (warp < 3) {
    uint64_t* d = a.desc + size_t(warp) * a.tiles;
    uint32_t v;
    if (warp == 0) v = lookback_warp_max(d, tile, 0u, a.tag, tile_head, a.err);
    else if (warp == 1) v = lookback_warp_wide<RR_LOOKBACK>(d, tile, 0u, a.tag, tile_surv, a.err);
    else v = lookback_warp_wide<RR_LOOKBACK>(d, tile, 0u, a.tag, tile_shead, a.err);
    if (lane == 0) s_carry[warp] = v;
  }
  __syncthreads();
  uint32_t run_head = max(head_before, s_carry[0]);     // (slot + 1) of the last head before the current row
  uint32_t out_at = s_carry[1] + surv_before;           // survivors before the current row
  uint32_t gd_run = s_carry[2] + shead_before;          // surviving heads before the current row

#pragma unroll
  for (int k = 0; k < RR_ROWS; ++k) {
    const uint32_t q = wbase + k * 32 + lane;
    uint32_t S, SH, L;
    masks(k, S, SH, L);
    const uint32_t le = lanemask_lt() | (1u << lane);
    const uint32_t hm = H[k] & le;
    const uint32_t my_head = hm ? wbase + k * 32 + (31 - __clz(hm)) + 1 : run_head;
    if (q < a.m) {
      // slots of one group are consecutive in SA, so the head's SA position is sap - distance
      const uint32_t rank = sap[k] - (q - (my_head - 1));
      // SA is final for a slot once its group is a single rotation; tied slots come back next round
      if (((L >> lane) & 1u) && !(RR_DBG(a) & 2u)) a.sa[sap[k]] = idx[k];
      if (binned) s_stage[s_bstart[(idx[k] >> a.part_shift) & 255u] + ((bpos[k / 2] >> ((k & 1) * 16)) & 0xFFFFu)] = (uint64_t(idx[k]) << 32) | rank;
      else if (a.pairs) a.pairs[q] = (uint64_t(idx[k]) << 32) | rank;
      else if (!(RR_DBG(a) & 1u)) a.rnk[idx[k]] = rank;
      if (((S >> lane) & 1u) && !(RR_DBG(a) & 4u)) {
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
  if (tile == a.tiles - 1 && tid == RR_THREADS - 1) {
    a.totals[0] = s_carry[1] + tile_surv;
    a.totals[1] = s_carry[2] + tile_shead;
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
// is free: the sort that follows needs no histogram pass over the keys, and neither does the pass
// that partitions the rank scatter by the top bits of idx.
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

int suffix_sort_bwt(Ctx* c, uint32_t n, uint32_t* sa_host) {
  cudaStream_t st = c->stream;
  uint8_t* T = c->text.as<uint8_t>();
  BCE_TRY(c->bwt.ensure(c, size_t(n) + 64));
  uint8_t* L = c->bwt.as<uint8_t>();

  // scratch: two key buffers, two index buffers, SA, rank, and the positional side arrays
  const size_t N = n;
  // fall-back list of the tile-local sort (local_sort.cuh): at most a quarter of the working set
  const size_t FB = N / 4 + 1;
  const size_t LT = N / LS_TILE + 2;
  size_t need = 2 * Carver::need(N, 8) + 8 * Carver::need(N, 4) + 2 * Carver::need(FB, 8) + 3 * Carver::need(FB, 4) +
                4 * Carver::need(LT, 4) + 4096;
  BCE_TRY(c->scratch.ensure(c, need));
  Carver cv(c->scratch.p, c->scratch.cap);
  uint64_t* keyA = cv.take<uint64_t>(N);
  uint64_t* keyB = cv.take<uint64_t>(N);
  uint32_t* idxA = cv.take<uint32_t>(N);
  uint32_t* idxB = cv.take<uint32_t>(N);
  uint32_t* sa = cv.take<uint32_t>(N);
  uint32_t* rnk = cv.take<uint32_t>(N);
  uint32_t* saposA = cv.take<uint32_t>(N);
  uint32_t* saposB = cv.take<uint32_t>(N);
  uint32_t* gdA = cv.take<uint32_t>(N);
  uint32_t* gdB = cv.take<uint32_t>(N);
  uint64_t* fbkA = cv.take<uint64_t>(FB);
  uint64_t* fbkB = cv.take<uint64_t>(FB);
  uint32_t* fbvA = cv.take<uint32_t>(FB);
  uint32_t* fbvB = cv.take<uint32_t>(FB);
  uint32_t* fb_slot = cv.take<uint32_t>(FB);
  uint32_t* lt_pre = cv.take<uint32_t>(LT);
  uint32_t* lt_suf = cv.take<uint32_t>(LT);
  uint32_t* lt_cnt = cv.take<uint32_t>(LT);
  uint32_t* lt_off = cv.take<uint32_t>(LT);
  if (!cv.ok()) { set_error(c, "suffix sort: scratch carve failed"); return BCE_GPU_E_NOMEM; }

  char* small = c->small.as<char>();
  uint32_t* d_err = reinterpret_cast<uint32_t*>(small + kSmallErr);
  uint32_t* d_ticket = reinterpret_cast<uint32_t*>(small + kSmallRerankTicket);
  uint32_t* d_totals = reinterpret_cast<uint32_t*>(small + kSmallRerankTotals);
  uint32_t* d_hist = reinterpret_cast<uint32_t*>(small + kSmallHist);
  uint32_t* d_phist = reinterpret_cast<uint32_t*>(small + kSmallPartHist);
  uint32_t* d_pcursor = d_phist + 256;
  uint32_t* h_small = c->pinned_small.as<uint32_t>() + 8192;   // past the sort's host mirror
  BCE_CUDA(c, cudaMemsetAsync(d_err, 0, 64, st));

  bce_gpu_stats& S = c->stats;
  S.sort_rounds = 0;
  c->pass_ev_n = 0;

  cudaEvent_t e0 = c->ev[0], e1 = c->ev[1];
  auto lap = [&](float& acc) -> int {
    BCE_CUDA(c, cudaEventRecord(e1, st));
    BCE_CUDA(c, cudaEventSynchronize(e1));
    float ms = 0;
    BCE_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
    acc += ms;
    BCE_CUDA(c, cudaEventRecord(e0, st));
    return BCE_GPU_OK;
  };
  BCE_CUDA(c, cudaEventRecord(e0, st));

  pad_cyclic_kernel<<<1, 64, 0, st>>>(T, n);
  S.gpu_launches++;
  // the first radix pass of round 0 makes keys and indices from the text itself (BCE_GPU_PACK=1: a
  // separate pack kernel writes them first)
  const bool use_local = exp_env("BCE_GPU_NO_LOCAL_SORT", 0) == 0;
  const uint32_t local_min = c->local_sort_min;   // smaller working sets take the plain radix path (BCE_GPU_OPT_LOCAL_SORT_MIN)
  const bool fused_pack = exp_env("BCE_GPU_PACK", 0) == 0 && exp_env("BCE_GPU_RADIX_STABLE_FIRST", 0) == 0;
  if (!fused_pack) {
    pack_keys_kernel<<<(n + 256 * PK_ROWS - 1) / (256 * PK_ROWS), 256, 0, st>>>(T, n, keyA, idxA);
    S.gpu_launches++;
  }
  BCE_CUDA(c, cudaGetLastError());
  BCE_TRY(lap(S.ms_pack));

  uint64_t* kcur = keyA; uint64_t* kalt = keyB;
  uint32_t* vcur = idxA; uint32_t* valt = idxB;
  uint32_t* sap_cur = nullptr;            // round 0: slot == SA position
  uint32_t* sap_next = saposA;
  uint32_t* gd_next = gdA;
  uint32_t m = n, groups = 0;
  uint64_t h = 8;
  const int nbits = bits_for(n);
  bool had_tiebreak = false;              // identical rotations were ordered by index: rnk is then not a permutation

  for (int round = 0;; ++round) {
    if (round >= kMaxSortRounds) { set_error(c, "suffix sort: too many rounds"); return BCE_GPU_E_INTERNAL; }
    int shifts[8], np = 0;
    bool tiebreak = false;
    // Large working sets update the rank array through pairs partitioned by the top 8 bits of idx
    // (see the re-rank step below); decided here because the key rebuild counts that digit too.
    const bool partitioned = exp_env("BCE_GPU_NO_PARTITION", 0) == 0 && m >= (8u << 20) && size_t(n) * 4 > (size_t(64) << 20);
    const int pshift = 32 + std::max(0, nbits - 8);
    bool local_plan = false;               // this round's sort is done tile by tile (local_sort.cuh)
    uint32_t m_fb = 0;                     // ... except for this many slots, which go through the radix sort
    if (round == 0) {
      for (int s = 0; s < 64; s += 8) shifts[np++] = s;
    } else {
      tiebreak = h >= n;
      if (tiebreak) had_tiebreak = true;
      for (int s = 0; s < nbits; s += 8) shifts[np++] = s;
      int gbits = bits_for(groups);
      for (int s = 0; s < gbits && np < 8; s += 8) shifts[np++] = 32 + s;
      // Rounds >= 1: the groups are short, so tiles are sorted where they are (keys made on the way) and
      // only the groups that cross a tile boundary go through the radix sort (local_sort.cuh)
      uint32_t* gd_cur = gd_next == gdA ? gdB : gdA;
      if (use_local && m >= local_min) {
        const uint32_t ltiles = (m + LS_TILE - 1) / LS_TILE;
        ls_classify_kernel<<<(ltiles + 255) / 256, 256, 0, st>>>(gd_cur, m, ltiles, lt_pre, lt_suf, lt_cnt);
        ls_scan_kernel<<<1, 1024, 0, st>>>(lt_cnt, ltiles, lt_off, d_totals + 3);
        S.gpu_launches += 2;
        BCE_CUDA(c, cudaGetLastError());
        BCE_CUDA(c, cudaMemcpyAsync(h_small + 4, d_totals + 3, 4, cudaMemcpyDeviceToHost, st));
        BCE_CUDA(c, cudaStreamSynchronize(st));
        m_fb = h_small[4];
        BCE_TRACE("local sort round %d: %u of %u slots in groups that cross a tile boundary", round, m_fb, m);
        local_plan = m_fb <= FB - 1 && m_fb <= m / 4;
      }
      if (local_plan) {
        if (partitioned) {
          BCE_CUDA(c, cudaMemsetAsync(d_phist, 0, 256 * 4, st));
          const uint32_t want = (m + 255) / 256, most = uint32_t(c->sm_count) * 8;
          ls_idx_hist_kernel<<<want < most ? want : most, 256, 0, st>>>(vcur, m, pshift - 32, d_phist);
          S.gpu_launches++;
        }
        BCE_TRY(lap(S.ms_rekey));
      } else {
        // working-set slot -> key of the next doubling step, digit histograms counted on the way
        RekeyHist rh;
        for (int i = 0; i < kRadixMaxPasses; ++i) rh.sh.s[i] = i < np ? shifts[i] : 0;
        rh.npass = np;
        rh.hist = d_hist;
        rh.phist = partitioned ? d_phist : nullptr;
        rh.pshift = pshift - 32;
        BCE_CUDA(c, cudaMemsetAsync(d_hist, 0, kRadixMaxPasses * 256 * 4, st));
        BCE_CUDA(c, cudaMemsetAsync(d_phist, 0, 256 * 4, st));
        const uint32_t chunk = RK_THREADS * RK_ITEMS;
        const uint32_t want = (m + chunk - 1) / chunk, most = uint32_t(c->sm_count) * 8;
        rekey_kernel<<<want < most ? want : most, RK_THREADS, 0, st>>>(vcur, gd_next == gdA ? gdB : gdA, rnk, m, n,
                                                                       uint32_t(tiebreak ? 0 : h), tiebreak ? 1 : 0, kcur, rh);
        S.gpu_launches++;
        BCE_CUDA(c, cudaGetLastError());
        BCE_TRY(lap(S.ms_rekey));
      }
    }
    BCE_TRACE("sort round %d m=%u h=%llu tiebreak=%d passes<=%d", round, m, (unsigned long long)h, int(tiebreak), np);
    uint64_t* ks; uint32_t* vs; int ran = 0;
    bool local_done = false;
    if (local_plan) {
      const uint32_t ltiles = (m + LS_TILE - 1) / LS_TILE;
      LocalSortArgs la;
      la.vin = vcur; la.gd = gd_next == gdA ? gdB : gdA; la.rnk = rnk;
      la.n = n; la.h = uint32_t(tiebreak ? 0 : h); la.tiebreak = tiebreak ? 1 : 0;
      la.kout = kalt; la.vout = valt; la.m = m;
      la.pre = lt_pre; la.suf = lt_suf; la.off = lt_off;
      la.fb_key = fbkA; la.fb_idx = fbvA; la.fb_slot = fb_slot;
      ls_sort_kernel<<<ltiles, LS_THREADS, 0, st>>>(la);
      S.gpu_launches++;
      BCE_CUDA(c, cudaGetLastError());
      if (m_fb) {
        uint64_t* sk; uint32_t* sv; int fran = 0;
        BCE_TRY(radix_sort_pairs(c, fbkA, fbkB, fbvA, fbvB, m_fb, shifts, np, &sk, &sv, &fran, nullptr));
        ls_place_kernel<<<(m_fb + 255) / 256, 256, 0, st>>>(sk, sv, fb_slot, m_fb, kalt, valt);
        S.gpu_launches++;
        BCE_CUDA(c, cudaGetLastError());
      }
      ks = kalt; vs = valt;
      ran = np;                          // reported as the passes an LSD sort of these keys would take
      S.sort_local_elems += m;
      S.sort_fallback_elems += m_fb;
      local_done = true;
    }
    RadixHistSource hsrc;
    if (round == 0) { hsrc.window_text = T; hsrc.keys_from_text = fused_pack; } else hsrc.dev_hist = d_hist;
    if (!local_done) BCE_TRY(radix_sort_pairs(c, kcur, kalt, vcur, valt, m, shifts, np, &ks, &vs, &ran, &hsrc));
    if (round == 0 && fused_pack && ran == 0) {      // every window is the same byte repeated: no pass ran, nothing made the keys
      pack_keys_kernel<<<(n + 256 * PK_ROWS - 1) / (256 * PK_ROWS), 256, 0, st>>>(T, n, ks, vs);
      S.gpu_launches++;
    }
    BCE_TRY(lap(S.ms_radix));
    S.sort_m[round] = m;
    S.sort_passes[round] = uint32_t(ran);
    S.sort_radix_passes[round] = local_done ? 0u : uint32_t(ran);
    S.sort_rounds = uint32_t(round + 1);

    // re-rank: writes SA and rank for every slot, compacts the still-tied slots
    uint32_t* v_other = (vs == idxA) ? idxB : idxA;
    RerankArgs a;
    a.key = ks; a.idx = vs; a.sapos = sap_cur; a.m = m;
    a.sa = sa; a.rnk = rnk;
    // Large working sets: a billion random 4-byte stores into a 4n-byte array cost more than
    // everything else in this kernel together (each one a read-modify-write of a 32-byte
    // sector).  Write (idx, rank) pairs in slot order instead, partition them by the top 8 bits
    // of idx with one keys-only radix pass, and scatter from that order: every 1/256 slice of
    // the rank array then stays in L2 while it is being filled.
    uint64_t* pair_buf = (ks == keyA) ? keyB : keyA;
    a.pairs = partitioned ? pair_buf : nullptr;
    // the pairs leave the kernel already binned by the top bits of idx (BCE_GPU_PARTITION=radix: in slot
    // order, binned afterwards by one keys-only radix pass)
    const bool binned = partitioned && exp_env("BCE_GPU_PARTITION", 0) == 0;
    a.part_cursor = nullptr;
    a.part_shift = pshift - 32;
    if (binned) {
      if (round == 0) {                  // every idx in [0, n) is present: the bin sizes are arithmetic
        uint32_t* all_idx = h_small + 16;
        const int sft = pshift - 32;
        for (uint32_t d = 0; d < 256; ++d) {
          const uint64_t lo = uint64_t(d) << sft, hi = uint64_t(d + 1) << sft;
          all_idx[d] = uint32_t(lo >= n ? 0 : (hi < n ? hi : n) - lo);
        }
        BCE_CUDA(c, cudaMemcpyAsync(d_phist, all_idx, 256 * 4, cudaMemcpyHostToDevice, st));
      }                                  // later rounds: counted by rekey_kernel over this round's working set
      partition_cursor_kernel<<<1, 256, 0, st>>>(d_phist, d_pcursor);
      S.gpu_launches++;
      a.part_cursor = d_pcursor;
    }
    a.idx_out = v_other; a.sapos_out = sap_next; a.gd_out = gd_next;
    a.totals = d_totals;
    a.tiles = (m + RR_TILE - 1) / RR_TILE;
    BCE_TRY(c->desc.ensure(c, size_t(a.tiles) * 3 * sizeof(uint64_t)));
    a.desc = c->desc.as<uint64_t>();
    a.ticket = d_ticket;
    a.tag = uint32_t(next_tag(c));
    a.err = d_err;
    a.dbg = uint32_t(exp_env("BCE_GPU_RERANK_DBG", 0));      // experiment builds only: timing with parts switched off
    BCE_CUDA(c, cudaMemsetAsync(d_ticket, 0, 4, st));
    rerank_kernel<<<a.tiles, RR_THREADS, 0, st>>>(a);
    S.gpu_launches++;
    BCE_CUDA(c, cudaGetLastError());
    BCE_CUDA(c, cudaMemcpyAsync(h_small, d_totals, 8, cudaMemcpyDeviceToHost, st));
    BCE_CUDA(c, cudaMemcpyAsync(h_small + 2, d_err, 4, cudaMemcpyDeviceToHost, st));
    { const float before = S.ms_rerank;
      BCE_TRY(lap(S.ms_rerank));      // synchronises
      BCE_TRACE("rerank round %d m=%u: %.3f ms (dbg=%u, partitioned=%d)", round, m, S.ms_rerank - before, a.dbg, int(partitioned));
      if (a.dbg) { set_error(c, "rerank timing experiment"); return BCE_GPU_E_INTERNAL; } }
    if (binned) {
      scatter_ranks_kernel<<<(m + 255) / 256, 256, 0, st>>>(pair_buf, m, rnk);
      S.gpu_launches++;
      BCE_CUDA(c, cudaGetLastError());
      const float before = S.ms_rerank;
      BCE_TRY(lap(S.ms_rerank));
      BCE_TRACE("rank scatter: %.3f ms", S.ms_rerank - before);
    } else if (partitioned) {
      uint64_t* pk; uint32_t* pv; int pran = 0;
      RadixHistSource psrc;
      uint32_t all_idx[256];
      if (round == 0) {                  // every idx in [0, n) is present: the digit counts are arithmetic
        const int sft = pshift - 32;
        for (uint32_t d = 0; d < 256; ++d) {
          const uint64_t lo = uint64_t(d) << sft, hi = uint64_t(d + 1) << sft;
          all_idx[d] = uint32_t(lo >= n ? 0 : (hi < n ? hi : n) - lo);
        }
        psrc.host_hist = all_idx;
      } else {
        psrc.dev_hist = d_phist;          // counted by rekey_kernel over this round's working set
      }
      BCE_TRY(radix_sort_pairs(c, pair_buf, ks, nullptr, nullptr, m, &pshift, 1, &pk, &pv, &pran, &psrc));
      scatter_ranks_kernel<<<(m + 255) / 256, 256, 0, st>>>(pk, m, rnk);
      S.gpu_launches++;
      BCE_CUDA(c, cudaGetLastError());
      const float before = S.ms_rerank;
      BCE_TRY(lap(S.ms_rerank));
      BCE_TRACE("rank partition + scatter: %.3f ms", S.ms_rerank - before);
    }
    if (h_small[2]) { set_error(c, "suffix sort: chained-scan watchdog fired"); return BCE_GPU_E_INTERNAL; }
    uint32_t m_next = h_small[0];
    groups = h_small[1];
    if (tiebreak && m_next) { set_error(c, "suffix sort: ties left after index tie-break"); return BCE_GPU_E_INTERNAL; }

    // next round: survivors live in v_other / sap_next / gd_next
    vcur = v_other; valt = (v_other == idxA) ? idxB : idxA;
    kcur = keyA; kalt = keyB;
    sap_cur = sap_next;
    sap_next = (sap_next == saposA) ? saposB : saposA;
    gd_next = (gd_next == gdA) ? gdB : gdA;
    m = m_next;
    if (m == 0) break;
    if (round > 0) h *= 2;
    if (round == 0) h = 8;
  }

  // binned inverse form for inputs whose T does not fit L2 anyway; needs rnk to be the inverse suffix array, which it
  // is unless identical rotations were told apart by index (then equal rotations share a rank)
  if (!had_tiebreak && n >= (8u << 20) && exp_env("BCE_GPU_BWT_GATHER", 0) == 0) {
    const int shift = std::max(0, bits_for(n) - 8);
    uint32_t* pairs = reinterpret_cast<uint32_t*>(keyA);             // the sort's buffers are dead
    BCE_TRACE("bwt binned shift=%d: positions binned through the inverse suffix array", shift);
    bwt_cursor_kernel<<<1, 256, 0, st>>>(d_pcursor, shift);
    bwt_bin_kernel<<<(n + BG_TILE - 1) / BG_TILE, BG_THREADS, 0, st>>>(T, rnk, n, shift, d_pcursor, pairs);
    bwt_scatter_kernel<<<(n + 255) / 256, 256, 0, st>>>(pairs, n, shift, L);
    S.gpu_launches += 3;
  } else {
    BCE_TRACE("bwt gather: bytes gathered through the suffix array (tie-break ran: %d)", int(had_tiebreak));
    bwt_gather_kernel<<<((n + 3) / 4 + 255) / 256, 256, 0, st>>>(T, sa, n, L);
    S.gpu_launches++;
  }
  BCE_CUDA(c, cudaGetLastError());
  BCE_CUDA(c, cudaMemcpyAsync(h_small, sa, 4, cudaMemcpyDeviceToHost, st));
  BCE_TRY(lap(S.ms_bwt_gather));
  c->offset = h_small[0];
  for (int i = 0; i + 1 < c->pass_ev_n; i += 2) {      // the stream is idle here (lap synchronised)
    float pms = 0;
    if (cudaEventElapsedTime(&pms, c->pass_ev[i], c->pass_ev[i + 1]) == cudaSuccess) S.ms_radix_kernel += pms;
  }
  c->pass_ev_n = 0;
  c->bwt_resident = true;
  if (sa_host) BCE_TRY(d2h(c, sa_host, sa, N * 4));
  return BCE_GPU_OK;
}

}  // namespace bce
