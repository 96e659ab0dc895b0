// many.cu -- the whole front end for many small inputs in one launch (bce_gpu_compress_many).
//
// For an input of a few kilobytes the multi-launch front end (suffix_sort.cu, wavelet.cu, cse.cu) is nothing but
// launches, read-backs and synchronisations on one SM.  Here one CTA runs every stage of one input, without the host
// and without a grid barrier, and a persistent grid of such CTAs takes inputs from an atomic work counter:
//   suffix sort   prefix doubling; a round is a stable LSD sort (8-bit digits) of the rank pairs
//                 (rank[i], rank[(i + h) mod n]) in index order -- ranks are dense and below n <= 2^16, so a pair is
//                 one 32-bit key -- then a re-rank by a block scan.  Equal rotations (exact powers) stay in ascending
//                 index order because every sort is stable and starts from index order.
//   BWT           L[r] = T[(SA[r] - 1) mod n], offset = SA[0]
//   wavelet       8 stable bit partitions, rank words [bits << 32 | ones before], n / 32 + 1 per level (wavelet.cu's
//                 layout), C[i] = zeros of level (i + 7) % 8
//   level loop    warp w runs level w: it walks its frontier (flat layout, flat_at) 32 nodes at a time with the shared
//                 node rule (cse_rule.cuh), ballots and a warp scan place the children and the emitted words; one
//                 __syncthreads per round.  Emission goes to the CTA's staging area
//   output        the input's words are reserved in the call's arena with one atomicAdd and copied there; the per-input
//                 directory says where.  An input that does not fit is left "not done" and no CTA takes another
//                 input: the host resubmits those.  Where an input lands in the arena depends on timing, what it
//                 contains does not.
#include <algorithm>
#include <numeric>
#include <vector>

#include "ctx.h"
#include "cse_rule.cuh"

namespace bce {

constexpr uint32_t kManyMaxN = BCE_GPU_MANY_MAX_N;   // ranks < 2^16: a rank pair is one 32-bit key
static_assert(kManyMaxN <= (1u << 16), "rank pairs must fit 32 bits");
constexpr int MN_THREADS = 256;                      // 256 threads = one per digit of a sort pass, 8 warps = 8 levels
constexpr int MN_WARPS = MN_THREADS / 32;

struct ManySlot {                   // one CTA's scratch, sized for the call's largest input N
  size_t rank, key0, key1, val0, val1, bytes, bstride, ranks, front, stage, total;
  uint32_t words_per_level, fcap, scap;
};
static ManySlot many_slot(uint32_t N, uint32_t maxw) {
  ManySlot s;
  auto al = [](size_t b) { return (b + 255) & ~size_t(255); };
  s.words_per_level = N / 32 + 1;
  s.fcap = N / 2 + 2;                                   // a level's nodes are disjoint intervals of >= 2 positions
  s.scap = std::max(N, 2u) * maxw;                      // a level visits at most n - 1 nodes, one count each
  size_t at = 0;
  s.rank = at; at += al(size_t(N) * 4);
  s.key0 = at; at += al(size_t(N) * 4);
  s.key1 = at; at += al(size_t(N) * 4);
  s.val0 = at; at += al(size_t(N) * 4);
  s.val1 = at; at += al(size_t(N) * 4);
  s.bstride = al(size_t(N) + 64);
  s.bytes = at; at += 3 * s.bstride;                    // L and the two wavelet buffers
  s.ranks = at; at += al(size_t(8) * s.words_per_level * 8);
  s.front = at; at += al(size_t(2) * 8 * 3 * s.fcap * 4);
  s.stage = at; at += al(size_t(8) * s.scap * 4);
  s.total = at;
  return s;
}

struct ManyArgs {
  const uint8_t* text;                   // the inputs back to back
  const unsigned long long* starts;      // k + 1 offsets into text
  const uint32_t* order;                 // input taken by job j (largest first)
  uint32_t k;
  char* slots;
  ManySlot slot;
  uint32_t* arena;
  unsigned long long arena_cap;          // words
  unsigned long long* arena_used;
  uint32_t* next_job;
  uint32_t* stop;                        // 1 = the arena is full: no CTA takes another input
  ManyEntry* dir;
  CseArgs rule;                          // emit_mode and cfgbits for cse_step; nothing else of it is read
};

struct ManyShared {
  uint32_t hist[256], base[256];
  uint32_t wcnt[MN_WARPS][256], pfx[MN_WARPS][256];
  uint32_t wtot[2][MN_WARPS];
  uint32_t cz[2][8], co[2][8];
  uint32_t zeros[8];
  uint32_t words[8];
  uint32_t job;
  uint32_t err;
  unsigned long long at;
  uint32_t fits;
};

template <typename P> __device__ __forceinline__ void swap(P& x, P& y) { P t = x; x = y; y = t; }
__device__ __forceinline__ uint32_t lane_lt() { uint32_t m; asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m)); return m; }

// Exclusive block scan of one value per thread; `total` = the sum over the block.
__device__ __forceinline__ uint32_t many_scan(ManyShared& sh, uint32_t v, uint32_t& total) {
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= unsigned(d)) inc += o;
  }
  if (lane == 31) sh.wtot[0][warp] = inc;
  __syncthreads();
  uint32_t pre = 0;
  total = 0;
#pragma unroll
  for (int w = 0; w < MN_WARPS; ++w) {
    const uint32_t t = sh.wtot[0][w];
    if (unsigned(w) < warp) pre += t;
    total += t;
  }
  __syncthreads();
  return pre + inc - v;
}

// One stable counting-sort pass on the digit (key >> shift) & 255.  Returns false (and moves nothing) when every key
// has the same digit.
__device__ bool many_sort_pass(ManyShared& sh, const uint32_t* kin, const uint32_t* vin, uint32_t* kout, uint32_t* vout,
                               uint32_t n, int shift) {
  const unsigned tid = threadIdx.x, warp = tid >> 5;
  sh.hist[tid] = 0;
  __syncthreads();
  for (uint32_t i = tid; i < n; i += MN_THREADS) atomicAdd(&sh.hist[(kin[i] >> shift) & 255u], 1u);
  __syncthreads();
  const uint32_t h = sh.hist[tid];
  if (__syncthreads_or(h == n)) return false;
  uint32_t total;
  sh.base[tid] = many_scan(sh, h, total);
  __syncthreads();
  for (uint32_t t0 = 0; t0 < n; t0 += MN_THREADS) {
    const uint32_t i = t0 + tid;
    const bool live = i < n;
    const uint32_t key = live ? kin[i] : 0u, d = (key >> shift) & 255u;
    const uint32_t peers = __match_any_sync(0xffffffffu, live ? d : 256u);
    const uint32_t rank = __popc(peers & lane_lt());
    if (live && rank == 0) sh.wcnt[warp][d] = __popc(peers);
    __syncthreads();
    {   // thread tid owns digit tid: where each warp's run of it starts (warps in order: stable)
      uint32_t acc = sh.base[tid];
#pragma unroll
      for (int w = 0; w < MN_WARPS; ++w) { sh.pfx[w][tid] = acc; acc += sh.wcnt[w][tid]; sh.wcnt[w][tid] = 0; }
      sh.base[tid] = acc;
    }
    __syncthreads();
    if (live) {
      const uint32_t at = sh.pfx[warp][d] + rank;
      kout[at] = key;
      vout[at] = vin[i];
    }
  }
  __syncthreads();
  return true;
}

// Dense ranks from keys in sorted order: rank[val[r]] = number of distinct keys before r.  Returns the group count.
__device__ uint32_t many_rerank(ManyShared& sh, const uint32_t* key, const uint32_t* val, uint32_t* rank, uint32_t n) {
  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t carry = 0;
  int par = 0;
  for (uint32_t t0 = 0; t0 < n; t0 += MN_THREADS, par ^= 1) {
    const uint32_t r = t0 + tid;
    const bool live = r < n;
    const bool head = live && (r == 0 || key[r - 1] != key[r]);
    const uint32_t bal = __ballot_sync(0xffffffffu, head);
    if (lane == 0) sh.wtot[par][warp] = __popc(bal);
    __syncthreads();
    uint32_t pre = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < MN_WARPS; ++w) {
      const uint32_t t = sh.wtot[par][w];
      if (unsigned(w) < warp) pre += t;
      tot += t;
    }
    if (live) rank[val[r]] = carry + pre + __popc(bal & lane_lt()) + uint32_t(head) - 1u;
    carry += tot;
  }
  __syncthreads();
  return carry;
}

__global__ void __launch_bounds__(MN_THREADS) many_kernel(ManyArgs a) {
  __shared__ ManyShared sh;
  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  char* slot = a.slots + size_t(blockIdx.x) * a.slot.total;
  uint32_t* rank = reinterpret_cast<uint32_t*>(slot + a.slot.rank);
  uint32_t* const key0 = reinterpret_cast<uint32_t*>(slot + a.slot.key0);
  uint32_t* const val0 = reinterpret_cast<uint32_t*>(slot + a.slot.val0);
  uint32_t* const key1 = reinterpret_cast<uint32_t*>(slot + a.slot.key1);
  uint32_t* const val1 = reinterpret_cast<uint32_t*>(slot + a.slot.val1);
  uint8_t* L = reinterpret_cast<uint8_t*>(slot + a.slot.bytes);
  uint8_t* const wbuf0 = L + a.slot.bstride;
  uint8_t* const wbuf1 = L + 2 * a.slot.bstride;
  uint64_t* R = reinterpret_cast<uint64_t*>(slot + a.slot.ranks);
  uint32_t* front = reinterpret_cast<uint32_t*>(slot + a.slot.front);
  uint32_t* stage = reinterpret_cast<uint32_t*>(slot + a.slot.stage);
  const uint32_t fcap = a.slot.fcap, scap = a.slot.scap;
  const uint32_t maxw = max_words(a.rule);
  for (int w = 0; w < MN_WARPS; ++w) sh.wcnt[w][tid] = 0;

  for (;;) {
    if (tid == 0) sh.job = *reinterpret_cast<volatile uint32_t*>(a.stop) ? a.k : atomicAdd(a.next_job, 1u);
    __syncthreads();
    const uint32_t job = sh.job;
    if (job >= a.k) break;
    const uint32_t in = a.order[job];
    const uint8_t* T = a.text + a.starts[in];
    const uint32_t n = uint32_t(a.starts[in + 1] - a.starts[in]);

    // ---- suffix sort: round 0 sorts by the first byte, round h by (rank[i], rank[i + h]) -------------------------
    // (kc, vc) hold the current order, (ko, vo) receive the next pass
    uint32_t *kc = key0, *vc = val0, *ko = key1, *vo = val1;
    for (uint32_t i = tid; i < n; i += MN_THREADS) { kc[i] = T[i]; vc[i] = i; }
    __syncthreads();
    if (many_sort_pass(sh, kc, vc, ko, vo, n, 0)) { swap(kc, ko); swap(vc, vo); }
    uint32_t groups = many_rerank(sh, kc, vc, rank, n);
    for (uint32_t len = 1; groups < n && len < n; len *= 2) {
      const uint32_t h = len;
      const int b = 32 - __clz(groups - 1u);                     // bits of the largest rank (0: all ranks are 0)
      for (uint32_t i = tid; i < n; i += MN_THREADS) {
        const uint32_t j = i + h < n ? i + h : i + h - n;
        kc[i] = (rank[i] << b) | rank[j];
        vc[i] = i;
      }
      __syncthreads();
      for (int shift = 0; shift < 2 * b; shift += 8)
        if (many_sort_pass(sh, kc, vc, ko, vo, n, shift)) { swap(kc, ko); swap(vc, vo); }
      groups = many_rerank(sh, kc, vc, rank, n);
    }
    const uint32_t* SA = vc;
    const uint32_t offset = SA[0];
    for (uint32_t r = tid; r < n; r += MN_THREADS) { const uint32_t s = SA[r]; L[r] = T[s ? s - 1 : n - 1]; }
    if (tid < 8) sh.zeros[tid] = 0;
    __syncthreads();

    // ---- wavelet matrix -------------------------------------------------------------------------------------------
    {
      uint32_t z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      for (uint32_t r = tid; r < n; r += MN_THREADS) {
        const uint32_t c = L[r];
#pragma unroll
        for (int j = 0; j < 8; ++j) z[j] += ((c >> j) & 1u) ^ 1u;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) z[j] += __shfl_xor_sync(0xffffffffu, z[j], d);
        if (lane == 0) atomicAdd(&sh.zeros[j], z[j]);
      }
    }
    __syncthreads();
    const uint32_t wpl = n / 32 + 1;
    for (int j = 0; j < 8; ++j) {
      const uint8_t* src = j == 0 ? L : (j & 1) ? wbuf0 : wbuf1;
      uint8_t* dst = (j & 1) ? wbuf1 : wbuf0;
      uint64_t* Rj = R + size_t(j) * wpl;
      const uint32_t zj = sh.zeros[j];
      uint32_t carry = 0;                                        // ones before the tile
      int par = 0;
      for (uint32_t t0 = 0; t0 <= n; t0 += MN_THREADS, par ^= 1) {   // position n's word exists too
        const uint32_t pos = t0 + tid;
        const bool live = pos < n;
        const uint32_t c = live ? src[pos] : 0u;
        const bool one = live && ((c >> j) & 1u);
        const uint32_t bal = __ballot_sync(0xffffffffu, one);
        if (lane == 0) sh.wtot[par][warp] = __popc(bal);
        __syncthreads();
        uint32_t pre = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < MN_WARPS; ++w) {
          const uint32_t t = sh.wtot[par][w];
          if (unsigned(w) < warp) pre += t;
          tot += t;
        }
        const uint32_t ones_warp = carry + pre;                  // ones before this warp's 32 positions
        if (lane == 0 && pos / 32 < wpl) Rj[pos / 32] = (uint64_t(bal) << 32) | ones_warp;
        if (live && j < 7) {
          const uint32_t ones_before = ones_warp + __popc(bal & lane_lt());
          dst[one ? zj + ones_before : pos - ones_before] = uint8_t(c);
        }
        carry += tot;
      }
      __syncthreads();
    }

    // ---- level loop ---------------------------------------------------------------------------------------------
    auto C = [&](int i) { return sh.zeros[(i + 7) & 7]; };     // bce.cpp:1128
    // frontier of (parity p, level l): arrays s, x0, x1 of fcap nodes each
    auto fr = [&](int p, int l, int f) { return front + (size_t((p * 8 + l) * 3 + f)) * fcap; };
    if (tid < 8) {                                               // roots (bce.cpp:1238-1240)
      const uint32_t zr = C(tid), orr = n - C(tid);
      const bool root = zr && orr;
      if (root) { fr(0, tid, 0)[0] = 0; fr(0, tid, 1)[0] = zr; fr(0, tid, 2)[0] = orr; }
      sh.cz[0][tid] = root ? 1u : 0u;
      sh.co[0][tid] = 0;
    }
    if (tid == 0) sh.err = 0;
    __syncthreads();
    const uint32_t round_limit = 8u * n + 64u;
    const int l = int(warp), ln = (l + 1) & 7;
    const uint64_t* __restrict__ Rl = R + size_t(l) * wpl;
    uint32_t* st = stage + size_t(l) * scap;
    const uint32_t one_base = C(ln);
    uint32_t cursor = 0, round = 0;
    unsigned long long visits = 0;
    int p = 0;
    for (;;) {
      uint32_t total = 0;
#pragma unroll
      for (int k = 0; k < 8; ++k) total += sh.cz[p][k] + sh.co[p][k];
      if (total == 0) break;
      if (round >= round_limit) { if (tid == 0) sh.err |= kManyErrRunaway; break; }
      visits += total;
      const int q = p ^ 1;
      const uint32_t cz = sh.cz[p][l], cnt = cz + sh.co[p][l];
      const uint32_t *fs = fr(p, l, 0), *fa = fr(p, l, 1), *fb = fr(p, l, 2);
      uint32_t *ns = fr(q, ln, 0), *na = fr(q, ln, 1), *nb = fr(q, ln, 2);
      uint32_t zc = 0, oc = 0;
      bool overflow = false;
      for (uint32_t t0 = 0; t0 < cnt; t0 += 32) {
        const uint32_t t = t0 + lane;
        const bool live = t < cnt;
        uint32_t s = 0, x0 = 0, x1 = 0;
        CseStep r{false, false, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
        if (live) {
          const uint32_t idx = flat_at(fcap, cz, t);
          s = fs[idx]; x0 = fa[idx]; x1 = fb[idx];
          // rank_words reads through the non-coherent cache, which may still hold the previous input's rank words
          // (this kernel wrote them): the same three words, from L2
          const uint64_t wa = __ldcg(Rl + (s >> 5)), wb = __ldcg(Rl + ((s + x0 + x1) >> 5)), wc = __ldcg(Rl + ((s + x0) >> 5));
          r = cse_step(a.rule, l, one_base, s, x0, x1, wa, wb, wc);
        }
        const uint32_t zb = __ballot_sync(0xffffffffu, r.z), ob = __ballot_sync(0xffffffffu, r.o);
        uint32_t inc = r.nw;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
          if (lane >= unsigned(d)) inc += o;
        }
        if (r.z) { const uint32_t at = zc + __popc(zb & lane_lt()); ns[at] = r.zs; na[at] = r.za; nb[at] = r.zb; }
        if (r.o) { const uint32_t at = fcap - 1u - (oc + __popc(ob & lane_lt())); ns[at] = r.os; na[at] = r.oa; nb[at] = r.ob; }
        if (r.nw) {
          const uint32_t pe = cursor + inc - r.nw;
          if (pe + r.nw <= scap) put_words(st + pe, r.nw, r.e0, r.e1, r.e2, x1, x0 + x1);
          else overflow = true;
        }
        zc += __popc(zb);
        oc += __popc(ob);
        cursor += __shfl_sync(0xffffffffu, inc, 31);
      }
      if (__any_sync(0xffffffffu, overflow) && lane == 0) atomicOr(&sh.err, kManyErrStage);
      if (lane == 0) { sh.cz[q][ln] = zc; sh.co[q][ln] = oc; }
      __syncthreads();
      p = q;
      ++round;
    }

    // ---- reserve the input's words in the arena, copy them, fill the directory ------------------------------------
    if (lane == 0) sh.words[l] = cursor;
    __syncthreads();
    if (tid == 0) {
      unsigned long long w = 0;
      for (int k = 0; k < 8; ++k) w += sh.words[k];
      const unsigned long long at = atomicAdd(a.arena_used, w);
      sh.at = at;
      sh.fits = at + w <= a.arena_cap;
      if (!sh.fits) atomicExch(a.stop, 1u);
    }
    __syncthreads();
    ManyEntry& e = a.dir[in];
    if (sh.fits) {
      unsigned long long at = sh.at;
      for (int k = 0; k < 8; ++k) {
        const uint32_t* sk = stage + size_t(k) * scap;
        const uint32_t cntk = min(sh.words[k], scap);
        for (uint32_t i = tid; i < cntk; i += MN_THREADS) a.arena[at + i] = sk[i];
        at += sh.words[k];
      }
      if (tid < 8) { e.C[tid] = C(tid); e.count[tid] = sh.words[tid]; }
      if (tid == 0) {
        e.offset = offset;
        e.rounds = max(round, 1u);                  // the reference's do..while (bce.cpp:1246) runs at least once
        e.visits = visits;
        e.start = sh.at;
        e.err = sh.err;
        e.done = 1;
      }
    }
    __syncthreads();
  }
}

unsigned long long many_arena_cap(const Ctx* c, const uint64_t* starts, uint32_t k, uint32_t maxw) {
  uint32_t N = 0;
  unsigned long long worst_sum = 0;
  for (uint32_t i = 0; i < k; ++i) {
    const uint32_t n = uint32_t(starts[i + 1] - starts[i]);
    N = std::max(N, n);
    worst_sum += 8ull * n * maxw;
  }
  const unsigned long long cap = std::max<unsigned long long>(c->emit_batch_bytes / 4, 8ull * N * maxw);
  return std::min(cap, std::max(worst_sum, 8ull * N * maxw));
}

int many_launch(Ctx* c, const uint8_t* T, const uint64_t* starts, uint32_t k, uint32_t mode, const uint8_t (*cfg)[32],
                size_t tail_min, size_t tail_want, ManyDevice* d) {
  cudaStream_t st = c->stream;
  const uint32_t maxw = mode == BCE_EMIT_RAW ? 5u : 3u;
  uint32_t N = 0;
  std::vector<uint32_t> order(k);
  std::vector<unsigned long long> rel(size_t(k) + 1);
  for (uint32_t i = 0; i < k; ++i) {
    N = std::max(N, uint32_t(starts[i + 1] - starts[i]));
    rel[i] = starts[i] - starts[0];
  }
  rel[k] = starts[k] - starts[0];
  std::iota(order.begin(), order.end(), 0u);
  std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) {
    return starts[x + 1] - starts[x] > starts[y + 1] - starts[y];
  });
  const ManySlot slot = many_slot(N, maxw);
  const unsigned long long arena_cap = many_arena_cap(c, starts, k, maxw);

  int occ = 0;
  BCE_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, many_kernel, MN_THREADS, 0));
  auto al = [](size_t b) { return (b + 255) & ~size_t(255); };
  const size_t fixed = al(rel.size() * 8) + al(size_t(k) * 4) + al(size_t(k) * sizeof(ManyEntry)) + 256 + al(arena_cap * 4);
  size_t ctas = std::min<size_t>(k, size_t(c->sm_count) * std::max(occ, 1));
  const size_t budget = scratch_budget(c);
  if (fixed + std::max(slot.total, tail_min) > budget) {
    set_error(c, "compress_many: %zu bytes of scratch needed", fixed + std::max(slot.total, tail_min));
    return BCE_GPU_E_NOMEM;
  }
  ctas = std::min(ctas, (budget - fixed) / slot.total);
  const size_t tail = std::max(std::min(std::max(ctas * slot.total, tail_want), budget - fixed), tail_min);
  BCE_TRY(c->scratch.ensure(c, fixed + std::max(ctas * slot.total, tail)));
  char* base = c->scratch.as<char>();
  auto* d_starts = reinterpret_cast<unsigned long long*>(base);
  auto* d_order = reinterpret_cast<uint32_t*>(base + al(rel.size() * 8));
  auto* d_dir = reinterpret_cast<ManyEntry*>(reinterpret_cast<char*>(d_order) + al(size_t(k) * 4));
  auto* d_ctr = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(d_dir) + al(size_t(k) * sizeof(ManyEntry)));
  auto* d_arena = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(d_ctr) + 256);
  char* d_slots = reinterpret_cast<char*>(d_arena) + al(arena_cap * 4);

  cudaEvent_t e0 = c->ev[4], e1 = c->ev[5];
  BCE_CUDA(c, cudaEventRecord(e0, st));
  const size_t bytes = size_t(rel[k]);
  BCE_TRY(c->text.ensure(c, bytes + 64));
  BCE_TRY(h2d(c, c->text.p, T + starts[0], bytes));
  BCE_TRY(h2d(c, d_starts, rel.data(), rel.size() * 8));
  BCE_TRY(h2d(c, d_order, order.data(), size_t(k) * 4));
  BCE_CUDA(c, cudaEventRecord(e1, st));
  BCE_CUDA(c, cudaEventSynchronize(e1));
  float ms = 0;
  BCE_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
  c->stats.ms_h2d += ms;

  BCE_CUDA(c, cudaMemsetAsync(d_dir, 0, size_t(k) * sizeof(ManyEntry) + 256, st));   // directory and counters
  ManyArgs a;
  memset(&a, 0, sizeof a);
  a.text = c->text.as<uint8_t>();
  a.starts = d_starts;
  a.order = d_order;
  a.k = k;
  a.slots = d_slots;
  a.slot = slot;
  a.arena = d_arena;
  a.arena_cap = arena_cap;
  a.arena_used = d_ctr;
  a.next_job = reinterpret_cast<uint32_t*>(d_ctr + 1);
  a.stop = reinterpret_cast<uint32_t*>(d_ctr + 2);
  a.dir = d_dir;
  a.rule.emit_mode = mode;
  memcpy(a.rule.cfgbits, cfg, sizeof a.rule.cfgbits);
  BCE_TRACE("compress_many k=%u largest=%u ctas=%zu (%d per SM) slot=%zu B arena=%llu words", k, N, ctas, occ,
            slot.total, arena_cap);
  BCE_CUDA(c, cudaEventRecord(e0, st));
  many_kernel<<<unsigned(ctas), MN_THREADS, 0, st>>>(a);
  c->stats.gpu_launches++;
  BCE_CUDA(c, cudaGetLastError());
  BCE_CUDA(c, cudaEventRecord(e1, st));
  d->dir = d_dir;
  d->starts = d_starts;
  d->arena = d_arena;
  d->used = d_ctr;
  d->order = d_order;
  d->arena_cap = arena_cap;
  d->tail = d_slots;
  d->tail_bytes = tail;
  return BCE_GPU_OK;
}

int many_run(Ctx* c, const uint8_t* T, const uint64_t* starts, uint32_t k, bce_many_result* out) {
  if (c->emit_mode == BCE_EMIT_SCAN) {
    set_error(c, "compress_many: BCE_EMIT_SCAN is not supported (bce -s collects its counts per input)");
    return BCE_GPU_E_ARG;
  }
  ManyDevice dev;
  BCE_TRY(many_launch(c, T, starts, k, c->emit_mode, c->emit_cfg, 0, 0, &dev));
  const unsigned long long arena_cap = dev.arena_cap;
  const ManyEntry* d_dir = dev.dir;
  const uint32_t* d_arena = dev.arena;
  const unsigned long long* d_ctr = dev.used;
  cudaEvent_t e0 = c->ev[4], e1 = c->ev[5];
  float ms = 0;

  // read-back on the copy stream: the directory, then the arena's used part
  cudaStream_t cs = c->copy_stream;
  const size_t dir_bytes = size_t(k) * sizeof(ManyEntry);
  std::vector<ManyEntry> dir(k);
  unsigned long long used = 0;
  BCE_CUDA(c, cudaStreamWaitEvent(cs, e1, 0));
  BCE_CUDA(c, cudaMemcpyAsync(&used, d_ctr, 8, cudaMemcpyDeviceToHost, cs));
  BCE_CUDA(c, cudaMemcpyAsync(dir.data(), d_dir, dir_bytes, cudaMemcpyDeviceToHost, cs));
  BCE_CUDA(c, cudaStreamSynchronize(cs));
  BCE_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
  c->stats.ms_cse_total += ms;
  used = std::min(used, arena_cap);
  PinnedBuf& pin = c->many_flip ? c->pinned_many2 : c->pinned_many;
  c->many_flip ^= 1;
  BCE_TRY(pin.ensure(c, std::max<size_t>(used * 4, 4)));
  BCE_CUDA(c, cudaEventRecord(e0, cs));
  if (used) BCE_CUDA(c, cudaMemcpyAsync(pin.p, d_arena, used * 4, cudaMemcpyDeviceToHost, cs));
  BCE_CUDA(c, cudaEventRecord(e1, cs));
  BCE_CUDA(c, cudaEventSynchronize(e1));
  BCE_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
  c->stats.ms_d2h += ms;

  const uint32_t* words = pin.as<uint32_t>();
  int rc = BCE_GPU_OK;
  for (uint32_t i = 0; i < k; ++i) {
    const ManyEntry& e = dir[i];
    bce_many_result& o = out[i];
    memset(&o, 0, sizeof o);
    o.done = int(e.done);
    if (!e.done) continue;
    if (e.err && rc == BCE_GPU_OK) {
      set_error(c, "compress_many: input %u: %s", i,
                (e.err & kManyErrRunaway) ? "level loop ran past its round limit" : "staging area overflowed");
      rc = BCE_GPU_E_INTERNAL;
    }
    o.offset = e.offset;
    size_t at = size_t(e.start);
    for (int s = 0; s < 8; ++s) {
      o.C[s] = e.C[s];
      o.words[s] = words + at;
      o.count[s] = e.count[s];
      at += e.count[s];
    }
    c->stats.cse_visits += e.visits;
    c->stats.cse_rounds += e.rounds;
    for (int s = 0; s < 8; ++s) c->stats.cse_words += e.count[s];
  }
  if (c->emit_mode == BCE_EMIT_RAW) c->stats.cse_tuples = c->stats.cse_words / 5;
  c->stats.cse_launches = 1;
  c->stats.ms_total = c->stats.ms_h2d + c->stats.ms_cse_total + c->stats.ms_d2h;
  return rc;
}

}  // namespace bce
