// unbwt_many.cu -- the inverse BWT of many small rank dictionaries in one launch (bce_gpu_unbwt_many).
//
// For a dictionary of a few kilobytes the multi-launch inverse (unbwt.cu) is a dozen launches, a synchronisation and
// a read-back.  Here one CTA inverts one dictionary, and a persistent grid of such CTAs takes dictionaries, largest
// first, from an atomic work counter.  A dictionary of n <= BCE_GPU_MANY_MAX_N rows lives in shared memory:
//   LF pass     one thread per row p < n descends the 8 levels (the rank words are read from global memory) and keeps
//               the byte of the row, L[p], and the row it leads to, LF[p] (u16: every row below n fits).  Positions are
//               clamped to [0, n] as the host decoder's DecodeRank does (bit and ones_before read at min(pos, n); the
//               row itself keeps its 32-bit value), so every read stays inside the dictionary whatever the words are.
//               A row whose LF is >= n is marked in a bitmap.
//   fast path   no LF >= n: rows that are multiples of B start chains; every chain is walked to the next such row (its
//               length bounded by n) and one thread follows the chains from chain 0.  If they add up to n steps
//               without meeting a chain twice, every chain on the walk knows its first step and writes its bytes; a
//               last chain that overruns n is cut there.  The valid archive of a primitive input always takes it: its
//               LF is one n-cycle.
//   serial path everything else (exact powers, whose LF has several cycles, and damaged dictionaries): one thread
//               walks the n steps, rows < n through the shared tables, rows >= n (and rows marked in the bitmap) by
//               the clamped descent, whose reads of a row >= n all hit word n / 32.
// Either way text i is what unbwt::bitwise (the host's unbwt_serial, `bce -ds`) makes of the same words:
//      out[(n - 1 - k + offset) mod n] = byte of row LF^k(0),   k = 0 .. n - 1.
#include <algorithm>
#include <numeric>
#include <vector>

#include "ctx.h"

namespace bce {

constexpr uint32_t kUmMaxN = BCE_GPU_MANY_MAX_N;
static_assert(kUmMaxN <= (1u << 16), "LF of a row below n is kept as u16");
constexpr int UM_THREADS = 512;
constexpr uint32_t kUmMaxChains = 512;         // B = the least power of two >= 32 that gives at most this many chains
constexpr uint32_t kUmNone = 0xFFFFFFFFu;

struct UmArgs {
  const uint64_t* ranks;
  const UmDict* dict;
  const uint32_t* order;                       // dictionary taken by job j (largest first)
  uint32_t k;
  uint32_t* next_job;
  uint32_t* serial;                            // dictionaries that took the serial path
  uint8_t* out;
  const int* status;                           // null, or per dictionary: non-zero = skip it (a rejected archive)
};

struct UmShared {
  uint32_t nxt[kUmMaxChains], len[kUmMaxChains], first[kUmMaxChains];
  uint32_t zeros[8];
  uint32_t job;
  uint32_t fast;
};

// Dynamic shared memory for dictionaries of up to N rows: LF (u16), L (u8), the bitmap of rows whose LF is >= n.
struct UmLayout {
  size_t lf, l, big, total;
};
static UmLayout um_layout(uint32_t N) {
  auto al = [](size_t b) { return (b + 15) & ~size_t(15); };
  UmLayout s;
  size_t at = 0;
  s.lf = at; at += al(size_t(N) * 2);
  s.l = at; at += al(N);
  s.big = at; at += al((size_t(N) / 32 + 1) * 4);
  s.total = at;
  return s;
}

// unbwt::bitwise's step from row s (bce.cpp:1020-1027) with DecodeRank's clamps: the byte of row s, returns LF(s)
__device__ __forceinline__ uint32_t um_descend(const uint64_t* __restrict__ R, uint32_t wpl, uint32_t n,
                                               const uint32_t* zeros, uint32_t s, uint32_t& chr) {
  chr = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t p = min(s, n);
    const uint64_t w = __ldg(R + size_t(j) * wpl + (p >> 5));
    const uint32_t bit = uint32_t(w >> (32 + (p & 31u))) & 1u;
    const uint32_t ones = uint32_t(w) + __popc(uint32_t(w >> 32) & ((1u << (p & 31u)) - 1u));
    chr |= bit << j;
    s = bit ? zeros[j] + ones : s - ones;
  }
  return s;
}

__global__ void __launch_bounds__(UM_THREADS) unbwt_many_kernel(UmArgs a, UmLayout lay) {
  extern __shared__ __align__(16) char dyn[];
  __shared__ UmShared sh;
  uint16_t* const LF = reinterpret_cast<uint16_t*>(dyn + lay.lf);
  uint8_t* const L = reinterpret_cast<uint8_t*>(dyn + lay.l);
  uint32_t* const big = reinterpret_cast<uint32_t*>(dyn + lay.big);
  const unsigned tid = threadIdx.x;

  for (;;) {
    if (tid == 0) sh.job = atomicAdd(a.next_job, 1u);
    __syncthreads();
    const uint32_t job = sh.job;
    if (job >= a.k) break;
    const uint32_t id = a.order[job];
    if (a.status && a.status[id]) { __syncthreads(); continue; }
    const UmDict d = a.dict[id];
    const uint32_t n = d.n, wpl = n / 32 + 1;
    const uint64_t* __restrict__ R = a.ranks + d.words;
    uint8_t* const out = a.out + d.out;
    if (tid < 8) {                                                   // zeros_before(n) of level tid
      const uint64_t w = __ldg(R + size_t(tid) * wpl + (n >> 5));
      sh.zeros[tid] = n - (uint32_t(w) + __popc(uint32_t(w >> 32) & ((1u << (n & 31u)) - 1u)));
    }
    for (uint32_t i = tid; i < wpl; i += UM_THREADS) big[i] = 0;
    __syncthreads();

    // ---- LF pass ------------------------------------------------------------------------------------------------
    bool mine_big = false;
    for (uint32_t p = tid; p < n; p += UM_THREADS) {
      uint32_t chr;
      const uint32_t s = um_descend(R, wpl, n, sh.zeros, p, chr);
      L[p] = uint8_t(chr);
      LF[p] = uint16_t(s);
      if (s >= n) { atomicOr(&big[p >> 5], 1u << (p & 31u)); mine_big = true; }
    }
    const bool any_big = __syncthreads_or(mine_big);

    // ---- fast path: chains from the rows that are multiples of B --------------------------------------------------
    uint32_t shiftB = 5;
    while (((n - 1) >> shiftB) + 1 > kUmMaxChains) ++shiftB;
    const uint32_t chains = ((n - 1) >> shiftB) + 1, mask = (1u << shiftB) - 1u;
    if (!any_big) {
      for (uint32_t c = tid; c < chains; c += UM_THREADS) {
        uint32_t r = c << shiftB, steps = 0;
        do {
          r = LF[r];
          ++steps;
        } while ((r & mask) != 0 && steps < n);
        sh.nxt[c] = r >> shiftB;                                     // r < n: a chain index (of no use once len = n)
        sh.len[c] = steps;
        sh.first[c] = kUmNone;
      }
      __syncthreads();
      if (tid == 0) {
        uint32_t c = 0, k = 0, ok = 1;
        while (k < n) {
          if (sh.first[c] != kUmNone) { ok = 0; break; }             // a cycle shorter than n: not one walk of n steps
          sh.first[c] = k;
          k += sh.len[c];
          c = sh.nxt[c];
        }
        sh.fast = ok;
      }
    } else if (tid == 0) {
      sh.fast = 0;
    }
    __syncthreads();

    if (sh.fast) {
      for (uint32_t c = tid; c < chains; c += UM_THREADS) {
        const uint32_t k0 = sh.first[c];
        if (k0 == kUmNone) continue;                                 // not on the walk from row 0
        const uint32_t steps = min(sh.len[c], n - k0);
        uint32_t r = c << shiftB, at = (n - 1 - k0 + d.offset) % n;
        for (uint32_t t = 0; t < steps; ++t) {
          out[at] = L[r];
          r = LF[r];
          at = at ? at - 1 : n - 1;
        }
      }
    } else if (tid == 0) {
      // ---- serial path: unbwt::bitwise's walk itself --------------------------------------------------------------
      atomicAdd(a.serial, 1u);
      uint32_t s = 0, at = (n - 1 + d.offset) % n;
      for (uint32_t i = 0; i < n; ++i) {
        uint32_t chr, to;
        if (s < n && !(any_big && ((big[s >> 5] >> (s & 31u)) & 1u))) {
          chr = L[s];
          to = LF[s];
        } else {
          to = um_descend(R, wpl, n, sh.zeros, s, chr);
        }
        out[at] = uint8_t(chr);
        at = at ? at - 1 : n - 1;
        s = to;
      }
    }
    __syncthreads();                                                 // shared tables free for the next dictionary
  }
}

int unbwt_many_launch(Ctx* c, const uint64_t* d_ranks, const UmDict* d_dict, const uint32_t* d_order,
                      const int* d_status, uint32_t k, uint32_t N, uint32_t* d_ctr, uint8_t* d_out) {
  const UmLayout lay = um_layout(N);
  BCE_CUDA(c, cudaFuncSetAttribute(unbwt_many_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(lay.total)));
  int occ = 0;
  BCE_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, unbwt_many_kernel, UM_THREADS, lay.total));
  if (occ < 1) { set_error(c, "unbwt_many: %zu bytes of shared memory per CTA do not fit an SM", lay.total); return BCE_GPU_E_INTERNAL; }
  const unsigned ctas = unsigned(std::min<size_t>(k, size_t(c->sm_count) * occ));
  UmArgs a;
  a.ranks = d_ranks;
  a.dict = d_dict;
  a.order = d_order;
  a.k = k;
  a.next_job = d_ctr;
  a.serial = d_ctr + 1;
  a.out = d_out;
  a.status = d_status;
  BCE_TRACE("unbwt_many k=%u largest=%u ctas=%u (%d per SM) smem=%zu B", k, N, ctas, occ, lay.total);
  unbwt_many_kernel<<<ctas, UM_THREADS, lay.total, c->stream>>>(a, lay);
  c->stats.gpu_launches++;
  BCE_CUDA(c, cudaGetLastError());
  return BCE_GPU_OK;
}

int unbwt_many_run(Ctx* c, const uint64_t* ranks, const uint32_t* n, const uint32_t* offset, uint32_t k,
                   uint8_t* out_host) {
  cudaStream_t st = c->stream;
  std::vector<UmDict> dict(k);
  std::vector<uint32_t> order(k);
  uint32_t N = 0;
  unsigned long long words = 0, bytes = 0;
  for (uint32_t i = 0; i < k; ++i) {
    dict[i] = UmDict{words, bytes, n[i], offset[i]};
    words += 8ull * (n[i] / 32 + 1);
    bytes += n[i];
    N = std::max(N, n[i]);
  }
  std::iota(order.begin(), order.end(), 0u);
  std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return n[x] > n[y]; });

  auto al = [](size_t b) { return (b + 255) & ~size_t(255); };
  const size_t need = al(words * 8) + al(size_t(k) * sizeof(UmDict)) + al(size_t(k) * 4) + 256 + al(bytes);
  if (need > scratch_budget(c)) { set_error(c, "unbwt_many: %zu bytes of scratch needed", need); return BCE_GPU_E_NOMEM; }
  BCE_TRY(c->scratch.ensure(c, need));
  char* base = c->scratch.as<char>();
  auto* d_ranks = reinterpret_cast<uint64_t*>(base);
  auto* d_dict = reinterpret_cast<UmDict*>(base + al(words * 8));
  auto* d_order = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(d_dict) + al(size_t(k) * sizeof(UmDict)));
  auto* d_ctr = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(d_order) + al(size_t(k) * 4));
  auto* d_out = reinterpret_cast<uint8_t*>(d_ctr) + 256;

  cudaEvent_t e0 = c->ev[4], e1 = c->ev[5];
  float ms = 0;
  BCE_CUDA(c, cudaEventRecord(e0, st));
  BCE_TRY(h2d(c, d_ranks, ranks, words * 8));
  BCE_TRY(h2d(c, d_dict, dict.data(), size_t(k) * sizeof(UmDict)));
  BCE_TRY(h2d(c, d_order, order.data(), size_t(k) * 4));
  BCE_CUDA(c, cudaEventRecord(e1, st));
  BCE_CUDA(c, cudaEventSynchronize(e1));
  BCE_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
  c->stats.ms_h2d += ms;

  BCE_CUDA(c, cudaMemsetAsync(d_ctr, 0, 256, st));
  BCE_CUDA(c, cudaEventRecord(e0, st));
  BCE_TRY(unbwt_many_launch(c, d_ranks, d_dict, d_order, nullptr, k, N, d_ctr, d_out));
  BCE_CUDA(c, cudaEventRecord(e1, st));
  BCE_CUDA(c, cudaEventSynchronize(e1));
  BCE_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
  c->stats.ms_unbwt_chase += ms;

  uint32_t ctr[2] = {0, 0};
  BCE_CUDA(c, cudaEventRecord(e0, st));
  BCE_TRY(d2h(c, ctr, d_ctr, sizeof ctr));
  BCE_TRY(d2h(c, out_host, d_out, bytes));
  BCE_CUDA(c, cudaEventRecord(e1, st));
  BCE_CUDA(c, cudaEventSynchronize(e1));
  BCE_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
  c->stats.ms_d2h += ms;
  c->stats.unbwt_dicts = k;
  c->stats.unbwt_serial = ctr[1];
  c->stats.ms_total = c->stats.ms_h2d + c->stats.ms_unbwt_chase + c->stats.ms_d2h;
  return BCE_GPU_OK;
}

}  // namespace bce
