// radix_sort.cu -- LSD radix sort of (u64 key, u32 value) pairs, 8-bit digits.
//
// This is the sort core that replaces libdivsufsort's suffix sorter (call site
// bce.cpp:901) in the prefix-doubling suffix sort (suffix_sort.cu).  One pass is a
// single kernel ("onesweep"): every tile ranks its elements by digit in shared memory,
// learns where its digit runs start in the output through a chained scan over tiles
// (decoupled look-back on tagged descriptors, common.cuh), and writes keys and values
// out of a shared-memory staging buffer so that every digit run is a coalesced burst.
// The first pass of a sort needs no stability and runs without chained scan and stable ranking
// (radix_unordered_kernel); in round 0 of the suffix sort it also makes the keys from the text.
// Digit histograms come from a RadixHistSource where the caller has one (the text's byte histogram,
// counts taken by the kernel that wrote the keys), else from one extra read of the keys.
//
// HBM traffic per pass: read 12 B + write 12 B per element  (SURVEY.md 8d: 24 m P_r).
#include <math.h>

#include "ctx.h"

namespace bce {

constexpr int RS_MIN_TILE = 2048;       // smallest tile of any kernel configuration (descriptor sizing)
constexpr int RS_MAX_PASSES = kRadixMaxPasses;
constexpr int kRadixThreads = 256, kRadixItems = 24;                       // tile of the stable and the unordered pass
constexpr size_t kRadixSmem = size_t(kRadixThreads) * kRadixItems * 12 + size_t(kRadixThreads / 32) * 1024;
constexpr size_t kRadixUnorderedSmem = size_t(256) * kRadixItems * 12;

size_t radix_desc_words(uint32_t m) { return (size_t(m) / RS_MIN_TILE + 1) * 256; }

// ---- histograms of every digit position in one read ------------------------------
// One histogram set per warp (shared-memory atomics of different warps never meet), and a digit
// on which the whole warp agrees -- the sorted group ids and the high bytes of ranks -- costs one
// add of 32 instead of 32 serialised adds on one address.
constexpr int RH_THREADS = 256;
constexpr int RH_WARPS = RH_THREADS / 32;

__global__ void __launch_bounds__(RH_THREADS) radix_hist_kernel(const uint64_t* __restrict__ keys, uint32_t m,
                                                                int npass, RadixShifts sh,
                                                                uint32_t* __restrict__ hist) {
  extern __shared__ uint32_t rh_smem[];                     // [RH_WARPS][npass][256]
  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < RH_WARPS * npass * 256; i += RH_THREADS) rh_smem[i] = 0;
  __syncthreads();
  uint32_t* h = rh_smem + size_t(warp) * npass * 256;
  const uint32_t stride = gridDim.x * RH_THREADS;
  const uint32_t rounds = (m + stride - 1) / stride;       // the same for every thread: whole warps stay converged
  uint32_t i = blockIdx.x * RH_THREADS + tid;
  for (uint32_t r = 0; r < rounds; ++r, i += stride) {
    const bool in = i < m;
    const uint64_t k = in ? keys[i] : 0;
    const unsigned active = __ballot_sync(0xffffffffu, in);
    if (active == 0xffffffffu) {
      for (int p = 0; p < npass; ++p) {
        const uint32_t d = uint32_t(k >> sh.s[p]) & 255u;
        int same;
        __match_all_sync(0xffffffffu, d, &same);
        if (same) { if (lane == 0) h[p * 256 + d] += 32; }
        else atomicAdd(&h[p * 256 + d], 1u);
        __syncwarp();
      }
    } else if (in) {
      for (int p = 0; p < npass; ++p) atomicAdd(&h[p * 256 + (uint32_t(k >> sh.s[p]) & 255u)], 1u);
    }
  }
  __syncthreads();
  for (int j = tid; j < npass * 256; j += RH_THREADS) {
    uint32_t v = 0;
#pragma unroll
    for (int w = 0; w < RH_WARPS; ++w) v += rh_smem[size_t(w) * npass * 256 + j];
    if (v) atomicAdd(&hist[j], v);
  }
}

// ---- one pass ------------------------------------------------------------------------
struct RadixPass {
  const uint64_t* kin;
  const uint32_t* vin;
  uint64_t* kout;
  uint32_t* vout;
  uint32_t m;
  int shift;
  bool codes7;            // FROM_TEXT: the text holds 7-bit symbol codes (window_key_bits)
  const uint32_t* base;   // [256] exclusive start of every digit in the output
  uint64_t* desc;         // [tiles][256] tagged descriptors
  uint32_t* ticket;       // tile dispenser (zero at launch)
  uint32_t tag;
  uint32_t* err;
};

// BALLOT picks how a warp finds the lanes that hold the same digit: MATCH.ANY costs time in proportion to the
// number of different digits in the warp, eight ballots cost the same whatever the digits are.  The host
// chooses per pass from the digit histogram (see radix_sort_pairs).
template <int RS_THREADS, int RS_ITEMS, int MIN_CTAS, bool BALLOT = false>
__global__ void __launch_bounds__(RS_THREADS, MIN_CTAS) radix_onesweep_kernel(RadixPass p) {
  constexpr int RS_TILE = RS_THREADS * RS_ITEMS;
  constexpr int RS_WARPS = RS_THREADS / 32;
  extern __shared__ __align__(16) unsigned char rs_smem[];
  uint64_t* s_keys = reinterpret_cast<uint64_t*>(rs_smem);                         // [RS_TILE]
  uint32_t* s_vals = reinterpret_cast<uint32_t*>(rs_smem + size_t(RS_TILE) * 8);    // [RS_TILE]
  uint32_t (*s_whist)[256] = reinterpret_cast<uint32_t (*)[256]>(rs_smem + size_t(RS_TILE) * 12);   // [RS_WARPS][256]
  __shared__ uint32_t s_goff[256];
  __shared__ uint32_t s_dstart[256];
  __shared__ uint32_t s_scan[RS_WARPS];
  __shared__ uint32_t s_tile;

  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // tiles are handed out in launch order so that every predecessor is already running
  if (tid == 0) s_tile = atomicAdd(p.ticket, 1u);
  for (int i = tid; i < RS_WARPS * 256; i += RS_THREADS) (&s_whist[0][0])[i] = 0;
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint32_t tile_base = tile * uint32_t(RS_TILE);
  const uint32_t valid = min(uint32_t(RS_TILE), p.m - tile_base);
  const uint32_t wbase = tile_base + warp * (32 * RS_ITEMS);

  uint64_t key[RS_ITEMS];
  uint32_t val[RS_ITEMS];
  uint32_t pos[RS_ITEMS];
#pragma unroll
  for (int k = 0; k < RS_ITEMS; ++k) {
    uint32_t idx = wbase + k * 32 + lane;
    bool in = idx < p.m;
    key[k] = in ? p.kin[idx] : ~0ull;      // padding sorts to the very end of the tile
    val[k] = (in && p.vin) ? p.vin[idx] : 0u;     // vin == NULL: keys only
  }
  // rank inside the warp's chunk, in index order (stable)
#pragma unroll
  for (int k = 0; k < RS_ITEMS; ++k) {
    uint32_t d = uint32_t(key[k] >> p.shift) & 255u;
unsigned peers;
    if (BALLOT) {
      peers = 0xffffffffu;
#pragma unroll
      for (int b = 0; b < 8; ++b) {
        const unsigned v = __ballot_sync(0xffffffffu, (d >> b) & 1u);
        peers &= ((d >> b) & 1u) ? v : ~v;
      }
    } else {
      peers = __match_any_sync(0xffffffffu, d);
    }
    unsigned leader = __ffs(peers) - 1;
    uint32_t before = 0;
    if (lane == leader) {
      before = s_whist[warp][d];
      s_whist[warp][d] = before + __popc(peers);
    }
    before = __shfl_sync(0xffffffffu, before, leader);
    pos[k] = before + __popc(peers & lanemask_lt());
    __syncwarp();
  }
  __syncthreads();

  // thread d owns digit d: turn per-warp counts into per-warp offsets, get the tile count
  {
    const uint32_t d = tid;
    uint32_t sum = 0;
    if (d < 256u) {
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) {
      uint32_t c = s_whist[w][d];
      s_whist[w][d] = sum;
      sum += c;
    }
    }
    uint32_t tot;
    uint32_t dstart = block_exclusive_scan<uint32_t, RS_THREADS>(sum, s_scan, tot);
    if (d < 256u) {
      s_dstart[d] = dstart;
      uint32_t publish = (d == 255u) ? sum - (uint32_t(RS_TILE) - valid) : sum;
      uint32_t excl = lookback_serial(p.desc + d, 256u, tile, p.tag, publish, p.err);
      s_goff[d] = p.base[d] + excl - dstart;     // global index = s_goff[digit] + local index
    }
  }
  __syncthreads();

#pragma unroll
  for (int k = 0; k < RS_ITEMS; ++k) {
    uint32_t d = uint32_t(key[k] >> p.shift) & 255u;
    pos[k] += s_dstart[d] + s_whist[warp][d];
    s_keys[pos[k]] = key[k];
    s_vals[pos[k]] = val[k];
  }
  __syncthreads();
  for (uint32_t j = tid; j < valid; j += RS_THREADS) {
    uint64_t k64 = s_keys[j];
    uint32_t d = uint32_t(k64 >> p.shift) & 255u;
    uint32_t g = s_goff[d] + j;
    p.kout[g] = k64;
    if (p.vout) p.vout[g] = s_vals[j];
  }
}


// ---- the first pass of a sort --------------------------------------------------------------
// An LSD pass has to be stable only to keep what earlier passes established; the first pass has
// nothing to keep (equal keys may come out in any order -- they are told apart, if at all, by later
// rounds of the suffix sort).  So it needs neither the chained scan nor a stable ranking: a key
// takes the next free place in its digit's bin of the tile (shared-memory atomic), the tile takes
// room in the digit's global run with one atomicAdd per digit, and the staged keys leave as runs.
// FROM_TEXT: the keys are the 8-symbol cyclic windows of `text` (window_key_bits) and the values their start
// indices; they are made here instead of being read (no pack kernel, 1 byte read per key instead of 12).
template <int RS_ITEMS, int MIN_CTAS, bool FROM_TEXT>
__global__ void __launch_bounds__(256, MIN_CTAS) radix_unordered_kernel(RadixPass p, uint32_t* __restrict__ cursor,
                                                                        const uint8_t* __restrict__ text) {
  constexpr int RS_THREADS = 256;
  constexpr int RS_TILE = RS_THREADS * RS_ITEMS;
  extern __shared__ __align__(16) unsigned char ru_smem[];
  uint64_t* s_keys = reinterpret_cast<uint64_t*>(ru_smem);                         // [RS_TILE]
  uint32_t* s_vals = reinterpret_cast<uint32_t*>(ru_smem + size_t(RS_TILE) * 8);    // [RS_TILE]
  __shared__ uint32_t s_cnt[256], s_start[256], s_goff[256];
  __shared__ uint32_t s_scan[RS_THREADS / 32];

  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  s_cnt[tid] = 0;
  __syncthreads();
  const uint32_t tile_base = blockIdx.x * uint32_t(RS_TILE);
  const uint32_t valid = min(uint32_t(RS_TILE), p.m - tile_base);
  const uint32_t wbase = tile_base + warp * (32 * RS_ITEMS);
  const bool has_vals = FROM_TEXT || p.vin != nullptr;

  uint64_t key[RS_ITEMS];
  uint32_t val[RS_ITEMS];
  uint32_t pos[RS_ITEMS / 2];                       // two 16-bit places per register
#pragma unroll
  for (int k = 0; k < RS_ITEMS; ++k) {
    const uint32_t idx = wbase + k * 32 + lane;
    const bool in = idx < p.m;
    if (FROM_TEXT) {
      key[k] = in ? window_key_bits(reinterpret_cast<const uint64_t*>(text), idx, p.codes7) : 0ull;
      val[k] = idx;
    } else {
      key[k] = in ? p.kin[idx] : 0ull;
      val[k] = (in && has_vals) ? p.vin[idx] : 0u;
    }
  }
#pragma unroll
  for (int k = 0; k < RS_ITEMS; ++k) {
    const bool in = wbase + k * 32 + lane < p.m;
    const uint32_t at = in ? atomicAdd(&s_cnt[uint32_t(key[k] >> p.shift) & 255u], 1u) : 0u;
    pos[k / 2] = (k & 1) ? (pos[k / 2] | (at << 16)) : at;
  }
  __syncthreads();
  {
    const uint32_t c = s_cnt[tid];
    uint32_t tot;
    const uint32_t st = block_exclusive_scan<uint32_t, RS_THREADS>(c, s_scan, tot);
    s_start[tid] = st;
    s_goff[tid] = p.base[tid] + (c ? atomicAdd(&cursor[tid], c) : 0u) - st;    // global index = s_goff[digit] + staged index
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < RS_ITEMS; ++k) {
    if (wbase + k * 32 + lane < p.m) {
      const uint32_t at = s_start[uint32_t(key[k] >> p.shift) & 255u] + ((pos[k / 2] >> ((k & 1) * 16)) & 0xFFFFu);
      s_keys[at] = key[k];
      s_vals[at] = val[k];
    }
  }
  __syncthreads();
  for (uint32_t j = tid; j < valid; j += RS_THREADS) {
    const uint64_t k64 = s_keys[j];
    const uint32_t g = s_goff[uint32_t(k64 >> p.shift) & 255u] + j;
    p.kout[g] = k64;
    if (has_vals) p.vout[g] = s_vals[j];
  }
}

// A pass ranks with eight ballots instead of MATCH.ANY when more than this many different digits are expected among
// a warp's 32 keys.
constexpr double kBallotAboveDistinct = 24;

int radix_sort_pairs(Ctx* c, uint64_t* keyA, uint64_t* keyB, uint32_t* valA, uint32_t* valB,
                     uint32_t m, const int* shifts, int npass, uint64_t** out_k, uint32_t** out_v,
                     int* passes_run, const RadixHistSource* src) {
  *out_k = keyA;
  *out_v = valA;
  if (passes_run) *passes_run = 0;
  if (m <= 1 || npass <= 0) return BCE_GPU_OK;
  if (npass > RS_MAX_PASSES) return BCE_GPU_E_ARG;

  char* small = c->small.as<char>();
  uint32_t* d_hist = reinterpret_cast<uint32_t*>(small + kSmallHist);
  uint32_t* d_base = reinterpret_cast<uint32_t*>(small + kSmallBase);
  uint32_t* d_ticket = reinterpret_cast<uint32_t*>(small + kSmallTicket);
  uint32_t* d_err = reinterpret_cast<uint32_t*>(small + kSmallErr);
  uint32_t* h_hist = c->pinned_small.as<uint32_t>();

  BCE_TRY(c->desc.ensure(c, radix_desc_words(m) * sizeof(uint64_t)));

  RadixShifts sh;
  for (int i = 0; i < RS_MAX_PASSES; ++i) sh.s[i] = i < npass ? shifts[i] : 0;
  const uint8_t* window_text = src ? src->window_text : nullptr;
  const uint32_t* dev_hist = src ? src->dev_hist : nullptr;
  // hist, base, tickets (err is the caller's); a histogram that already sits in d_hist stays
  if (dev_hist == d_hist) BCE_CUDA(c, cudaMemsetAsync(d_base, 0, kSmallErr - kSmallBase, c->stream));
  else BCE_CUDA(c, cudaMemsetAsync(d_hist, 0, kSmallErr, c->stream));
  if (src && src->host_hist) {
    // the caller derived them (the suffix sort's round 0: from the text's byte or symbol-pair histogram)
  } else if (dev_hist) {
    BCE_CUDA(c, cudaMemcpyAsync(h_hist, dev_hist, npass * 256 * 4, cudaMemcpyDeviceToHost, c->stream));
    BCE_CUDA(c, cudaStreamSynchronize(c->stream));
  } else {
    const size_t hsmem = size_t(RH_WARPS) * npass * 256 * 4;
    uint64_t hb64 = (uint64_t(m) + 255) / 256, hbmax = uint64_t(c->sm_count) * 3;
    int hb = int(hb64 < hbmax ? hb64 : hbmax);
    radix_hist_kernel<<<hb, RH_THREADS, hsmem, c->stream>>>(keyA, m, npass, sh, d_hist);
    c->stats.gpu_launches++;
    BCE_CUDA(c, cudaGetLastError());
    BCE_CUDA(c, cudaMemcpyAsync(h_hist, d_hist, npass * 256 * 4, cudaMemcpyDeviceToHost, c->stream));
    BCE_CUDA(c, cudaStreamSynchronize(c->stream));
  }

  // exclusive scans on the host (8 x 256 values); passes whose digit is constant are skipped
  bool run[RS_MAX_PASSES];
  uint32_t* h_base = h_hist + RS_MAX_PASSES * 256;
  for (int p = 0; p < npass; ++p) {
    run[p] = true;
    uint32_t acc = 0;
    for (int d = 0; d < 256; ++d) {
      uint32_t cnt = h_hist[p * 256 + d];
      if (cnt == m) run[p] = false;
      h_base[p * 256 + d] = acc;
      acc += cnt;
    }
  }
  BCE_CUDA(c, cudaMemcpyAsync(d_base, h_base, npass * 256 * 4, cudaMemcpyHostToDevice, c->stream));

  uint64_t* kin = keyA; uint64_t* kout = keyB;
  uint32_t* vin = valA; uint32_t* vout = valB;
  // 256 threads x 24 keys, 2 CTAs/SM: fastest tile shape on B200 on real keys (1 GB text, radix stage 125 ms; 256 x 16 x 3 CTAs:
  // 140; 256 x 20 x 3: 134; 256 x 28 x 2: 129; 384 x 16 x 2: 149; 512 x 16 x 1: 166 -- profiles/r1_radix_experiments.md)
  constexpr int RS_THREADS = kRadixThreads, RS_TILE = kRadixThreads * kRadixItems;
  constexpr size_t rs_smem = kRadixSmem;
  const uint32_t tiles = (m + RS_TILE - 1) / RS_TILE;
  const bool unordered_first = !(src && src->stable_first);
  int ran = 0;
  for (int p = 0; p < npass; ++p) {
    if (!run[p]) continue;
    RadixPass a;
    a.kin = kin; a.vin = vin; a.kout = kout; a.vout = vout;
    a.m = m; a.shift = shifts[p];
    a.codes7 = src && src->codes7;
    a.base = d_base + p * 256;
    a.desc = c->desc.as<uint64_t>();
    a.ticket = d_ticket + p;
    a.tag = uint32_t(next_tag(c));
    a.err = d_err;
    const bool timed = c->pass_ev_n + 2 <= 256;
    if (timed) cudaEventRecord(c->pass_ev[c->pass_ev_n], c->stream);
    if (ran == 0 && unordered_first) {
      uint32_t* d_cursor = reinterpret_cast<uint32_t*>(small + kSmallRadixCursor);
      BCE_CUDA(c, cudaMemsetAsync(d_cursor, 0, 256 * 4, c->stream));
      constexpr int UI = kRadixItems;
      constexpr size_t usmem = kRadixUnorderedSmem;
      const uint32_t ugrid = (m + 256 * UI - 1) / (256 * UI);
      if (window_text) radix_unordered_kernel<UI, 2, true><<<ugrid, 256, usmem, c->stream>>>(a, d_cursor, window_text);
      else radix_unordered_kernel<UI, 2, false><<<ugrid, 256, usmem, c->stream>>>(a, d_cursor, nullptr);
    } else {
      // expected number of different digits among 32 keys drawn from this pass's histogram
      double distinct = 0;
      for (int d = 0; d < 256; ++d) {
        const double q = double(h_hist[p * 256 + d]) / double(m);
        if (q > 0) distinct += 1.0 - pow(1.0 - q, 32.0);
      }
      // keys that are text windows arrive sorted by the bytes that follow: after the first passes a
      // warp's keys share their context and with it, mostly, the digit
      const bool context_sorted = window_text && ran >= 2;
      const bool ballot = distinct > kBallotAboveDistinct && !context_sorted;
      if (ballot) radix_onesweep_kernel<kRadixThreads, kRadixItems, 2, true><<<tiles, RS_THREADS, rs_smem, c->stream>>>(a);
      else radix_onesweep_kernel<kRadixThreads, kRadixItems, 2, false><<<tiles, RS_THREADS, rs_smem, c->stream>>>(a);
    }
    if (timed) { cudaEventRecord(c->pass_ev[c->pass_ev_n + 1], c->stream); c->pass_ev_n += 2; }
    c->stats.gpu_launches++;
    c->stats.radix_launches++;
    c->stats.radix_elems += m;
    BCE_CUDA(c, cudaGetLastError());
    uint64_t* tk = kin; kin = kout; kout = tk;
    uint32_t* tv = vin; vin = vout; vout = tv;
    ++ran;
  }
  *out_k = kin;
  *out_v = vin;
  if (passes_run) *passes_run = ran;
  return BCE_GPU_OK;
}


// Function attributes are per device: bce_gpu_open sets them for the context's device.
int radix_init_device(Ctx* c) {
  BCE_CUDA(c, cudaFuncSetAttribute(radix_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, RH_WARPS * RS_MAX_PASSES * 1024));
  BCE_CUDA(c, cudaFuncSetAttribute(radix_onesweep_kernel<kRadixThreads, kRadixItems, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kRadixSmem)));
  BCE_CUDA(c, cudaFuncSetAttribute(radix_onesweep_kernel<kRadixThreads, kRadixItems, 2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kRadixSmem)));
  BCE_CUDA(c, cudaFuncSetAttribute(radix_unordered_kernel<kRadixItems, 2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kRadixUnorderedSmem)));
  BCE_CUDA(c, cudaFuncSetAttribute(radix_unordered_kernel<kRadixItems, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kRadixUnorderedSmem)));
  return BCE_GPU_OK;
}

}  // namespace bce
