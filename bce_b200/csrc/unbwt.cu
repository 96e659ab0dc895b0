// unbwt.cu -- inverse path for `bce -d`: wavelet matrix -> text.
//
// Replaces unbwt::bytewise::unbwt (bce.cpp:1043-1103): the chunked wavelet -> bytes loop
// (:1050-1085), libdivsufsort's inverse_bw_transform(..., idx = 1) (:1091) and the final
// rotate by `offset` (:1093).  unbwt::bitwise (:999-1038) states the same mapping serially:
// descending the 8 levels from row s yields the byte of row s AND the row of the preceding
// character (after 8 stable bit partitions the rows are in F-column order), i.e. the LF
// mapping.  The text is the walk
//      out[(n-1-k + offset) mod n] = byte of row LF^k(0),   k = 0 .. n-1        (:1018-1029)
// with DecodeRank's clamps for words no archive writer made (see bce_gpu.h).  Three paths:
//   check       one streaming pass over the 8 levels confirms that the words are a true rank
//               directory (the base count of every word is the base of the one before plus its
//               data bits, the first is 0).  Then every level is a stable partition of [0, n)
//               onto itself, LF is a permutation of [0, n) and no row ever reaches n.
//   device      K11 gives L and LF for all rows.  K12 breaks the cycles at the rows that are
//               multiples of B: pass 1 walks every chain to the next marked row (length +
//               successor), pointer jumping ranks the chains on the list from chain 0, pass 2
//               walks those chains again and writes bytes at their final positions.  Chain 0's
//               list closes after p steps, the length of row 0's cycle; p = n for the archive of
//               a primitive input.  When p < n (an exact power, or words no BWT produced) the
//               rest of the walk repeats the first p steps and one more kernel copies them.
//   host        words that fail the check (only damaged archives make them) take unbwt_serial's
//               clamped walk on the caller's host words: what `bce -ds` costs, and no device
//               thread walks n steps alone.
// The byte of a row is recovered from its LF value by a search in the 256-entry F-column
// table, so a step costs one 4-byte gather.  Gather-bound by nature.
#include <algorithm>

#include "ctx.h"

namespace bce {

__device__ __forceinline__ uint32_t rank1_w(uint64_t w, uint32_t pos) {
  return uint32_t(w) + __popc(uint32_t(w >> 32) & ((1u << (pos & 31u)) - 1u));
}

// The words are a rank directory: base(W[0]) = 0 and base(W[i+1]) = base(W[i]) + popc(data(W[i])) for i < n/32, on
// every level (blockIdx.y; levels back to back, `words` each).  Sets *bad otherwise.
__global__ void __launch_bounds__(256) rank_check_kernel(const uint64_t* __restrict__ R, uint32_t words,
                                                         uint32_t* __restrict__ bad) {
  const uint64_t* __restrict__ W = R + size_t(blockIdx.y) * words;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < words; i += gridDim.x * blockDim.x) {
    uint32_t want = 0;
    if (i) {
      const uint64_t w = __ldg(W + i - 1);
      want = uint32_t(w) + __popc(uint32_t(w >> 32));
    }
    if (uint32_t(__ldg(W + i)) != want) *bad = 1;
  }
}

struct UnbwtLevels {
  const uint64_t* rank[8];
  uint32_t zeros[8];
};

// K11: LF[p] for every row p (the byte falls out of LF through the F table)
__global__ void __launch_bounds__(256) lf_from_wavelet_kernel(UnbwtLevels lv, uint32_t n,
                                                              uint32_t* __restrict__ LF,
                                                              uint8_t* __restrict__ L) {
  uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  uint32_t s = p, chr = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    uint64_t w = __ldg(lv.rank[j] + (s >> 5));
    uint32_t bit = uint32_t(w >> (32 + (s & 31u))) & 1u;      // Rank::bit, bce.cpp:196-198
    uint32_t r1 = rank1_w(w, s);
    chr |= bit << j;
    s = bit ? lv.zeros[j] + r1 : s - r1;                      // :1026
  }
  LF[p] = s;
  L[p] = uint8_t(chr);
}

__global__ void fstart_kernel(const uint32_t* __restrict__ hist, uint32_t* __restrict__ fstart) {
  // exclusive prefix of the byte histogram: first row of every byte in the F column
  if (threadIdx.x == 0) {
    uint32_t run = 0;
    for (int v = 0; v < 256; ++v) { fstart[v] = run; run += hist[v]; }
    fstart[256] = run;
  }
}

__global__ void __launch_bounds__(256) chase_measure_kernel(const uint32_t* __restrict__ LF, uint32_t n,
                                                            uint32_t shiftB, uint32_t chains,
                                                            uint32_t* __restrict__ nxt,
                                                            uint32_t* __restrict__ len) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= chains) return;
  const uint32_t mask = (1u << shiftB) - 1u;
  uint32_t r = j << shiftB, steps = 0;
  do {
    r = __ldg(LF + r);
    ++steps;
  } while ((r & mask) != 0 && steps < n);
  nxt[j] = r >> shiftB;
  len[j] = steps;
}

// pointer jumping: dist[j] = steps from the start of chain j to the end of the list that
// starts at chain 0 (the list ends when a chain leads back to row 0)
__global__ void __launch_bounds__(256) jump_init_kernel(const uint32_t* __restrict__ nxt,
                                                        const uint32_t* __restrict__ len, uint32_t chains,
                                                        uint32_t* __restrict__ link,
                                                        unsigned long long* __restrict__ dist) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= chains) return;
  link[j] = nxt[j] == 0 ? 0xFFFFFFFFu : nxt[j];
  dist[j] = len[j];
}
__global__ void __launch_bounds__(256) jump_step_kernel(const uint32_t* __restrict__ link_in,
                                                        const unsigned long long* __restrict__ dist_in,
                                                        uint32_t chains, uint32_t* __restrict__ link_out,
                                                        unsigned long long* __restrict__ dist_out) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= chains) return;
  uint32_t l = link_in[j];
  unsigned long long d = dist_in[j];
  if (l != 0xFFFFFFFFu) { d += dist_in[l]; l = link_in[l]; }
  link_out[j] = l;
  dist_out[j] = d;
}

__global__ void __launch_bounds__(256) chase_write_kernel(const uint32_t* __restrict__ LF,
                                                          const uint32_t* __restrict__ fstart, uint32_t n,
                                                          uint32_t shiftB, uint32_t chains,
                                                          const uint32_t* __restrict__ len,
                                                          const uint32_t* __restrict__ link,
                                                          const unsigned long long* __restrict__ dist,
                                                          uint32_t offset, uint8_t* __restrict__ out) {
  __shared__ uint32_t s_f[257];
  for (int v = threadIdx.x; v < 257; v += blockDim.x) s_f[v] = fstart[v];
  __syncthreads();
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= chains || link[j] != 0xFFFFFFFFu) return;       // not on row 0's cycle: the list from it never ends
  const unsigned long long total = dist[0];                 // p, the length of row 0's cycle
  // k = steps from row 0 to this chain's first row (< p); out index of step k is n-1-k+offset (mod n)
  const unsigned long long k0 = total - dist[j];
  uint64_t at = (uint64_t(n) - 1 - (k0 % n) + offset) % n;
  uint32_t r = j << shiftB;
  const uint32_t steps = len[j];
  for (uint32_t t = 0; t < steps; ++t) {
    uint32_t to = __ldg(LF + r);
    // byte of row r = the byte whose F-column range contains LF[r]
    uint32_t lo = 0, hi = 256;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      uint32_t mid = (lo + hi) >> 1;
      if (s_f[mid] <= to) lo = mid; else hi = mid;
    }
    out[at] = uint8_t(lo);
    at = at ? at - 1 : uint64_t(n) - 1;
    r = to;
  }
}

// steps k = p .. n-1 of the walk repeat step k mod p (row LF^p(0) is row 0 again); they read only steps < p
__global__ void __launch_bounds__(256) period_fill_kernel(const unsigned long long* __restrict__ dist, uint32_t n,
                                                          uint32_t offset, uint8_t* __restrict__ out) {
  const uint32_t p = uint32_t(dist[0]);
  for (uint32_t k = p + blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x)
    out[(n - 1 - k + offset) % n] = out[(n - 1 - k % p + offset) % n];
}

// unbwt_serial (host/decode.cpp) on the caller's words: bit and ones_before read at min(pos, n), the row keeps its
// 32-bit value
static void unbwt_host_walk(const uint64_t* const ranks[8], uint32_t offset, uint32_t n, uint8_t* out) {
  auto ones = [&](int j, uint32_t pos) {
    const uint32_t p = std::min(pos, n);
    const uint64_t w = ranks[j][p >> 5];
    return uint32_t(w) + uint32_t(__builtin_popcount(uint32_t(w >> 32) & ((1u << (p & 31u)) - 1u)));
  };
  uint32_t zeros[8];
  for (int j = 0; j < 8; ++j) zeros[j] = n - ones(j, n);
  uint32_t s = 0;
  for (uint64_t i = n; i-- > 0;) {
    uint32_t chr = 0;
    for (int j = 0; j < 8; ++j) {
      const uint32_t p = std::min(s, n);
      const uint32_t b = uint32_t(ranks[j][p >> 5] >> (32 + (p & 31u))) & 1u;
      chr |= b << j;
      s = b ? zeros[j] + ones(j, s) : s - ones(j, s);
    }
    out[(i + offset) % n] = uint8_t(chr);
  }
}

// ranks must already be in Ctx::ranks (8 x words); host_ranks are the same words on the host.  zeros[j] = rank0_j(n).
int unbwt_run(Ctx* c, const uint64_t* const host_ranks[8], uint32_t offset, uint32_t n, uint8_t* out_host) {
  cudaStream_t st = c->stream;
  const size_t words = size_t(n) / 32 + 1;
  uint32_t shiftB = 5;
  {
    uint64_t want = uint64_t(n) / (uint64_t(c->sm_count) * 2048 * 4);
    while (shiftB < 10 && (1ull << shiftB) < want) ++shiftB;
  }
  const uint32_t chains = uint32_t((uint64_t(n) + (1u << shiftB) - 1) >> shiftB);

  size_t need = Carver::need(n, 4) + 2 * Carver::need(size_t(n) + 64, 1) + 4 * Carver::need(chains, 4) +
                2 * Carver::need(chains, 8) + 4096;
  BCE_TRY(c->scratch.ensure(c, need));
  Carver cv(c->scratch.p, c->scratch.cap);
  uint32_t* LF = cv.take<uint32_t>(n);
  uint8_t* L = cv.take<uint8_t>(size_t(n) + 64);
  uint8_t* out = cv.take<uint8_t>(size_t(n) + 64);
  uint32_t* nxt = cv.take<uint32_t>(chains);
  uint32_t* len = cv.take<uint32_t>(chains);
  uint32_t* linkA = cv.take<uint32_t>(chains);
  uint32_t* linkB = cv.take<uint32_t>(chains);
  unsigned long long* distA = cv.take<unsigned long long>(chains);
  unsigned long long* distB = cv.take<unsigned long long>(chains);
  if (!cv.ok()) { set_error(c, "unbwt: scratch carve failed"); return BCE_GPU_E_NOMEM; }

  UnbwtLevels lv;
  for (int j = 0; j < 8; ++j) {
    lv.rank[j] = c->ranks.as<uint64_t>() + size_t(j) * words;
    lv.zeros[j] = c->C[(j + 1) & 7];          // C[i] = zeros of level (i+7)%8
  }
  char* small = c->small.as<char>();
  uint32_t* d_hist = reinterpret_cast<uint32_t*>(small + kSmallUnbwt);
  uint32_t* d_fstart = d_hist + 256;
  uint32_t* d_bad = d_fstart + 257;

  BCE_CUDA(c, cudaEventRecord(c->ev[0], st));
  BCE_CUDA(c, cudaMemsetAsync(d_bad, 0, 4, st));
  const dim3 check_grid(std::min<uint32_t>(uint32_t((words + 255) / 256), c->sm_count * 4), 8);
  rank_check_kernel<<<check_grid, 256, 0, st>>>(c->ranks.as<uint64_t>(), uint32_t(words), d_bad);
  c->stats.gpu_launches++;
  BCE_CUDA(c, cudaGetLastError());
  uint32_t bad = 0;
  BCE_TRY(d2h(c, &bad, d_bad, 4));
  c->stats.unbwt_dicts = 1;
  if (bad) {
    c->stats.unbwt_serial = 1;
    unbwt_host_walk(host_ranks, offset, n, out_host);
    return BCE_GPU_OK;
  }
  lf_from_wavelet_kernel<<<(n + 255) / 256, 256, 0, st>>>(lv, n, LF, L);
  BCE_CUDA(c, cudaMemsetAsync(d_hist, 0, 256 * 4, st));
  byte_hist_launch(c, L, n, d_hist);
  fstart_kernel<<<1, 32, 0, st>>>(d_hist, d_fstart);
  c->stats.gpu_launches += 3;
  BCE_CUDA(c, cudaGetLastError());
  BCE_CUDA(c, cudaEventRecord(c->ev[1], st));

  const uint32_t cb = (chains + 255) / 256;
  chase_measure_kernel<<<cb, 256, 0, st>>>(LF, n, shiftB, chains, nxt, len);
  jump_init_kernel<<<cb, 256, 0, st>>>(nxt, len, chains, linkA, distA);
  c->stats.gpu_launches += 2;
  uint32_t* li = linkA; uint32_t* lo = linkB;
  unsigned long long* di = distA; unsigned long long* dout = distB;
  for (uint64_t span = 1; span < chains; span <<= 1) {
    jump_step_kernel<<<cb, 256, 0, st>>>(li, di, chains, lo, dout);
    c->stats.gpu_launches++;
    uint32_t* tl = li; li = lo; lo = tl;
    unsigned long long* td = di; di = dout; dout = td;
  }
  chase_write_kernel<<<cb, 256, 0, st>>>(LF, d_fstart, n, shiftB, chains, len, li, di, offset, out);
  period_fill_kernel<<<std::min<uint32_t>((n + 255) / 256, c->sm_count * 8), 256, 0, st>>>(di, n, offset, out);
  c->stats.gpu_launches += 2;
  BCE_CUDA(c, cudaGetLastError());
  BCE_CUDA(c, cudaEventRecord(c->ev[2], st));
  BCE_CUDA(c, cudaEventSynchronize(c->ev[2]));
  float a = 0, b = 0;
  BCE_CUDA(c, cudaEventElapsedTime(&a, c->ev[0], c->ev[1]));
  BCE_CUDA(c, cudaEventElapsedTime(&b, c->ev[1], c->ev[2]));
  c->stats.ms_unbwt_bytes += a;
  c->stats.ms_unbwt_chase += b;
  return d2h(c, out_host, out, n);
}

}  // namespace bce
