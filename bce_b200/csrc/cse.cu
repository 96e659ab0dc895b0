// cse.cu -- stage B2: the CSE level loop (Compression by Substring Enumeration).
//
// Replaces BCE::code(mode = 1) (bce.cpp:1236-1373), its pArray queues (:226-356) and the
// root set-up (:1124-1130, :1238-1240).  A node (level i, position s, x0, x1) is the interval
// [s, s + x0 + x1) of level i's bit vector; per node the reference does three rank queries,
// hands one bounded count to coder_[i].set (:1302) and pushes up to two children to level
// (i+1)%8.  Nodes are independent; what the archive depends on is only the ORDER of the
// emitted counts per stream: ascending round, ascending position (SURVEY.md 4-4).
//
// Device design.  The frontier of a level is a flat structure-of-arrays list sorted by position
// (zero-half from the front, one-half from the back of one buffer, flat_at).  Per round and level
// three prefix sums -- zero-children, one-children, emitted words -- fix every output position, so
// the stable partition into the next level's halves and the emission order need no atomics.
//   huge frontiers    cse_slots_kernel (cse_slots.cuh): per-chunk output slots, warps that never wait
//   wide frontiers    cse_wide_kernel (cse_wide.cuh): persistent cooperative kernel, all SMs,
//                     software pipelined tiles, grid barrier between rounds
//   medium frontiers  cse_mid_kernel (cse_mid.cuh): slot layout, one grid barrier per round
//   narrow frontiers  cse_narrow_kernel (below): ONE cluster of 8 CTAs, one per level, frontiers
//                     in shared memory, children handed over through distributed shared memory,
//                     hardware cluster barrier between rounds; cse_tiny_kernel: one CTA
// All of them apply one node rule (cse_step, cse_rule.cuh) and one round verdict (must_drain, round_status).  A
// kernel runs rounds until its verdict says otherwise; the host then picks the next one
// (pick_kernel) and drains the emission buffers.
//
// Emission is word based.  Raw mode writes the five arguments of set() (20 B, bce_tuple);
// the packed modes write what the host coder actually consumes (one word; three when k > 31):
//   coder  [ctx:10 @10|k:5 @5|sym:5]   ctx = get_context index, bce.cpp:671-677, for the stream's configured
//          context bits.  k > 31 was halved nb times (bce.cpp:507-510): the word's k field is 0 then (a count's k
//          is at least 2) and two more words follow, [low[0..10) @10|nb:5 @5|k:5] and [low >> 10], with k, nb and
//          the nb low bits of the symbol.  Every word is below 2^20, so a batch crosses PCIe as 2.5 bytes per word
//          (cse_pack20_kernel)
//   scan   [esc:1|nb:5 @26|q2:8 @18|q1:8 @10|k:5 @5|sym:5]   ScanCoder::set, bce.cpp:737-744
//
// Algorithmic HBM bytes (SURVEY.md 8d): 48 B per node visit + 20 B per emitted count.
#include <cooperative_groups.h>

#include <algorithm>

#include "ctx.h"
#include "cse_rule.cuh"

namespace cg = cooperative_groups;

namespace bce {

#ifndef BCE_CS_THREADS
#define BCE_CS_THREADS 256
#endif
constexpr int CS_THREADS = BCE_CS_THREADS;   // threads of a wide-kernel CTA
constexpr int CS_MAX_TILE = CS_THREADS * 4;

enum : uint32_t { kCseRunning = 0, kCseDone = 1, kCseDrain = 2, kCseOverflow = 3, kCseRunaway = 4,
                  kCseGoWide = 5, kCseGoNarrow = 6 };

constexpr uint32_t kNarrowEnter = 256;     // every level at most this: the one-node-per-thread cluster kernel (leaves above 512)
constexpr int NM_THREADS = 512, NM_K = 8;  // the 8-nodes-per-thread instance: 4096 nodes per level
constexpr uint32_t kMediumEnter = NM_THREADS * NM_K / 4;   // entered at <= 1024 per level, left above 2048

struct CseDeviceState {
  uint32_t cnt[2][8][2];                 // [round parity][level][half] frontier sizes
  unsigned long long emitted[2][8];      // [round parity][level] words in the emission buffer
  unsigned long long visits;
  unsigned long long peak_frontier;
  uint32_t round;
  uint32_t status;
  uint32_t err;                          // 1 = chained-scan watchdog, 2 = grid-barrier watchdog
  uint32_t barrier_fail;                 // round at which the grid barrier timed out (+1), 0 = never
  unsigned long long arrivals;           // grid barrier: total CTA arrivals since cse_begin
  unsigned long long barriers;           // grid barriers completed since cse_begin
#ifdef BCE_GPU_EXPERIMENTS
  unsigned long long prof[8];            // cse_mid_kernel: SM cycles of CTA 0 per phase of a round, summed
#endif
};

__device__ __forceinline__ uint32_t vol_load(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long vol_load64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}


// The round verdict.  A stream must be drained once it holds a batch's worth of words or before a round that could
// overflow its buffer (a round emits at most one count, max_words words, per node).
__device__ __forceinline__ bool must_drain(unsigned long long emitted, unsigned long long nodes, uint32_t maxw,
                                           unsigned long long ecap, unsigned long long esoft) {
  return emitted >= esoft || emitted + nodes * maxw > ecap;
}
// What a kernel does with the round it is about to run, by priority: the loop is done, it has run away, the frontier
// does not fit, a narrower kernel takes over, the kernel must leave (its host picks another), the batch is full, run.
__device__ __forceinline__ uint32_t round_status(unsigned long long nodes, uint32_t round, uint32_t round_limit,
                                                 bool overflow, bool go_narrow, bool leave, bool drain) {
  return nodes == 0 ? kCseDone
       : round >= round_limit ? kCseRunaway
       : overflow ? kCseOverflow
       : go_narrow ? kCseGoNarrow
       : leave ? kCseGoWide
       : drain ? kCseDrain : kCseRunning;
}

// Grid-wide barrier.  Every CTA adds one arrival; barrier number b (0-based, counted since
// cse_begin) is passed when the counter reaches (b + 1) * gridDim.x.  The counter only grows,
// so there is no reset race.  The spin is bounded: a logic error becomes BCE_GPU_E_INTERNAL.
__device__ __forceinline__ bool grid_barrier(CseDeviceState* S, unsigned long long index, uint32_t round) {
  __syncthreads();
  bool ok = true;
  if (threadIdx.x == 0) {
    const unsigned long long target = (index + 1) * gridDim.x;
    // release on the arrival, acquire on the poll: what the CTA wrote before is visible to every CTA that sees the
    // count complete (cumulative through the block barrier above), without the two sequentially-consistent fences
    // (MEMBAR.SC.GPU) the first version paid per round -- rounds of small frontiers are nothing but latency
    asm volatile("red.release.gpu.global.add.u64 [%0], %1;" ::"l"(&S->arrivals), "l"(1ull) : "memory");
    uint32_t spins = 0;
    for (;;) {
      unsigned long long seen;
      asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(seen) : "l"(&S->arrivals) : "memory");
      if (seen >= target) break;
      if (++spins > (1u << 22)) {
        atomicExch(&S->barrier_fail, round + 1);
        atomicExch(&S->err, 2u);
        ok = false;
        break;
      }
      if (spins > 32) __nanosleep(20);
    }
  }
  __syncthreads();
  return ok;
}

// The barrier's targets are multiples of gridDim.x: a launch with another grid size starts a new count.
__global__ void cse_reset_barrier_kernel(CseDeviceState* S) {
  S->arrivals = 0;
  S->barriers = 0;
}

__global__ void cse_init_kernel(CseArgs a, uint32_t n) {
  // roots: node (0, C[i], n - C[i]) in the zero-half of level i when both are non-zero
  // (bce.cpp:1238-1240)
  const int i = threadIdx.x;
  CseDeviceState* S = a.st;
  if (i < 8) {
    uint32_t z = a.C[i], o = n - a.C[i];
    bool root = z && o;
    if (root) { a.fs[0][i][0] = 0; a.fa[0][i][0] = z; a.fb[0][i][0] = o; }
    S->cnt[0][i][0] = root ? 1u : 0u;
    S->cnt[0][i][1] = 0;
    S->cnt[1][i][0] = S->cnt[1][i][1] = 0;
    S->emitted[0][i] = S->emitted[1][i] = 0;
  }
  if (i == 0) { S->visits = 0; S->peak_frontier = 0; S->round = 0; S->status = kCseRunning; S->err = 0;
                S->barrier_fail = 0; S->arrivals = 0; S->barriers = 0;
#ifdef BCE_GPU_EXPERIMENTS
                for (int k = 0; k < 8; ++k) S->prof[k] = 0;
#endif
  }
}

__global__ void cse_reset_emitted_kernel(CseDeviceState* S) {
  if (threadIdx.x < 8) S->emitted[0][threadIdx.x] = S->emitted[1][threadIdx.x] = 0;
  if (threadIdx.x == 0 && S->status == kCseDrain) S->status = kCseRunning;
}

// Order-sensitive checksum of a run of emitted words (bce_gpu_resident_checksum): acc[0] += SUM w,
// acc[1] += SUM w * (2 (first + j) + 1), mod 2^64 -- sums commute, so the atomics do not make it nondeterministic.
__global__ void __launch_bounds__(256) cse_checksum_kernel(const uint32_t* __restrict__ words, unsigned long long count,
                                                           unsigned long long first, unsigned long long* acc) {
  unsigned long long s = 0, ws = 0;
  for (unsigned long long j = blockIdx.x * 256ull + threadIdx.x; j < count; j += gridDim.x * 256ull) {
    const unsigned long long w = words[j];
    s += w;
    ws += w * (2ull * (first + j) + 1ull);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, d);
    ws += __shfl_xor_sync(0xffffffffu, ws, d);
  }
  if ((threadIdx.x & 31) == 0) { atomicAdd(&acc[0], s); atomicAdd(&acc[1], ws); }
}

// Words below 2^20 leave as 20 bits each: a thread turns 8 words into 20 bytes (five aligned 32-bit stores).
__global__ void __launch_bounds__(256) cse_pack20_kernel(const uint32_t* __restrict__ words, unsigned long long count,
                                                         uint32_t* __restrict__ out) {
  const unsigned long long groups = (count + 7) / 8;
  for (unsigned long long q = blockIdx.x * 256ull + threadIdx.x; q < groups; q += gridDim.x * 256ull) {
    const unsigned long long j = 8 * q;
    uint32_t a[8];
    if (j + 8 <= count) {
      const uint4 v0 = *reinterpret_cast<const uint4*>(words + j);         // emission buffers are 256-byte aligned
      const uint4 v1 = *reinterpret_cast<const uint4*>(words + j + 4);
      a[0] = v0.x; a[1] = v0.y; a[2] = v0.z; a[3] = v0.w; a[4] = v1.x; a[5] = v1.y; a[6] = v1.z; a[7] = v1.w;
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) a[k] = j + k < count ? words[j + k] : 0u;
    }
    uint32_t* o = out + 5 * q;                                             // word k of the group sits at bit 20 k
    o[0] = a[0] | (a[1] << 20);
    o[1] = (a[1] >> 12) | (a[2] << 8) | (a[3] << 28);
    o[2] = (a[3] >> 4) | (a[4] << 16);
    o[3] = (a[4] >> 16) | (a[5] << 4) | (a[6] << 24);
    o[4] = (a[6] >> 8) | (a[7] << 12);
  }
}

// ---- bce -s: bucketing of a batch of BCE_EMIT_SCAN words (ScanCoder::set, bce.cpp:737-744) ---------------
// word = [esc:1|nb:5 @26|q2:8 @18|q1:8 @10|k:5 @5|sym:5]: bits 5..25 are the bucket (k, q1, q2).  The word rides in
// the upper half of a 64-bit sort key whose low 21 bits are the bucket; the value is the word's position.
__global__ void __launch_bounds__(256) scan_keys_kernel(const uint32_t* __restrict__ words, uint32_t cnt,
                                                        uint64_t* __restrict__ key, uint32_t* __restrict__ val,
                                                        unsigned long long* halvings) {
  unsigned long long nb = 0;
  for (uint32_t i = blockIdx.x * 256u + threadIdx.x; i < cnt; i += gridDim.x * 256u) {
    const uint32_t w = words[i];
    key[i] = (uint64_t(w) << 32) | bcefmt::scan_bucket(w);
    val[i] = i;
    if (w >> 31) nb += (w >> 26) & 31u;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) nb += __shfl_xor_sync(0xffffffffu, nb, d);
  if ((threadIdx.x & 31) == 0 && nb) atomicAdd(halvings, nb);
}

// After the stable sort: symbols as bytes in bucket order; one record per bucket (written where an atomic
// counter says: the host orders them by `start`, so the order the atomics resolve in does not matter).
__global__ void __launch_bounds__(256) scan_compact_kernel(const uint64_t* __restrict__ key, const uint32_t* __restrict__ val,
                                                           uint32_t cnt, uint8_t* __restrict__ syms,
                                                           bce_scan_bucket* __restrict__ buckets, uint32_t cap, uint32_t* nbuckets) {
  for (uint32_t i = blockIdx.x * 256u + threadIdx.x; i < cnt; i += gridDim.x * 256u) {
    const uint64_t k = key[i];
    syms[i] = uint8_t(uint32_t(k >> 32) & 31u);
    const uint32_t b = uint32_t(k) & 0x1FFFFFu;
    if (i == 0 || (uint32_t(key[i - 1]) & 0x1FFFFFu) != b) {
      const uint32_t slot = atomicAdd(nbuckets, 1u);
      if (slot < cap) buckets[slot] = bce_scan_bucket{b, i, val[i], 0u};
    }
  }
}

// vector load of ITEMS consecutive frontier entries; `rev` = stored back to front
template <int ITEMS>
__device__ __forceinline__ void load_items(const uint32_t* base, uint32_t first, bool rev, uint32_t cap, uint32_t (&out)[ITEMS]) {
  if constexpr (ITEMS == 4) {
    uint4 v = __ldcg(reinterpret_cast<const uint4*>(base + (rev ? cap - 4 - first : first)));
    if (rev) { out[0] = v.w; out[1] = v.z; out[2] = v.y; out[3] = v.x; }
    else { out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w; }
  } else if constexpr (ITEMS == 2) {
    uint2 v = __ldcg(reinterpret_cast<const uint2*>(base + (rev ? cap - 2 - first : first)));
    if (rev) { out[0] = v.y; out[1] = v.x; } else { out[0] = v.x; out[1] = v.y; }
  } else {
    out[0] = __ldcg(base + (rev ? cap - 1 - first : first));
  }
}

}  // namespace bce

#include "cse_wide.cuh"   // cse_wide_kernel<ITEMS>: the software-pipelined wide kernel
#include "cse_slots.cuh"  // cse_slots_kernel: huge frontiers, per-chunk output slots, warps that never wait
#include "cse_mid.cuh"    // cse_mid_kernel: thousands to half a million nodes per round, one grid barrier per round

namespace bce {

// ---------------------------------------------------------------------------------
// narrow mode: one cluster, one CTA per level
// ---------------------------------------------------------------------------------
// THREADS x K nodes per level fit: <1024, 1> for the long tail of tiny frontiers, <512, 8> (8 nodes
// per thread, 24 rank words in flight) for frontiers of a few thousand nodes per level, where a
// round of the wide kernel is five dependent trips to global memory plus a grid barrier.
template <int THREADS, int K>
struct NarrowShared {
  static constexpr int CAP = THREADS * K;
  uint32_t s[2][CAP], a[2][CAP], b[2][CAP];             // this level's frontier, double buffered
  uint32_t cz[2], co[2];                                // zero-/one-half sizes of buffer p
  uint32_t all_cnt[2][8];                               // every level's frontier size (all-gathered)
  unsigned long long all_emitted[2][8];                 // every level's emission cursor (all-gathered)
  uint64_t scan[THREADS / 32];
  uint32_t decision;
};

template <int THREADS, int K>
__global__ void __cluster_dims__(8, 1, 1) __launch_bounds__(THREADS, 1) cse_narrow_kernel(CseArgs a) {
  using Shared = NarrowShared<THREADS, K>;
  constexpr uint32_t CAP = Shared::CAP;
  cg::cluster_group cluster = cg::this_cluster();
  extern __shared__ __align__(16) unsigned char narrow_smem[];
  Shared& sh = *reinterpret_cast<Shared*>(narrow_smem);
  const unsigned tid = threadIdx.x;
  const int l = int(cluster.block_rank());          // level handled by this CTA
  const int ln = (l + 1) & 7;
  CseDeviceState* S = a.st;
  const uint64_t* __restrict__ R = a.ranks[l];
  const uint32_t maxw = max_words(a);

  uint32_t round = S->round;
  const int gpar = round & 1;
  // frontier of this level from the wide layout (zero-half ascending, one-half from the back)
  {
    const uint32_t cz = S->cnt[gpar][l][0], co = S->cnt[gpar][l][1];
    if (tid == 0) { sh.cz[0] = cz; sh.co[0] = co; }
    for (uint32_t t = tid; t < cz + co && t < CAP; t += THREADS) {
      const uint32_t idx = flat_at(a.cap, cz, t);
      sh.s[0][t] = a.fs[gpar][l][idx];
      sh.a[0][t] = a.fa[gpar][l][idx];
      sh.b[0][t] = a.fb[gpar][l][idx];
    }
    if (tid < 8) {
      sh.all_cnt[0][tid] = S->cnt[gpar][tid][0] + S->cnt[gpar][tid][1];
      sh.all_emitted[0][tid] = S->emitted[gpar][tid];
    }
  }
  unsigned long long visits = 0, peak = 0;
  int p = 0;
  cluster.sync();                                    // nobody writes into a CTA that is still loading
#ifdef BCE_GPU_EXPERIMENTS
  long long stamp_ = clock64();
  unsigned long long prof_[5] = {0, 0, 0, 0, 0};     // (registers: a stamp costs two instructions, not a trip to memory)
#define NARROW_STAMP(i) do { const long long now_ = clock64(); prof_[i] += (unsigned long long)(now_ - stamp_); stamp_ = now_; } while (0)
#else
#define NARROW_STAMP(i) do { } while (0)
#endif

  uint32_t status;
  for (;;) {
    const uint32_t cnt = min(sh.cz[p] + sh.co[p], CAP);
    const unsigned long long cursor = sh.all_emitted[p][l];      // this level's words so far (every CTA holds all eight)
    const unsigned warp_of_tid = tid >> 5;
    uint32_t s[K], x0[K], x1[K];
    uint64_t wa[K], wb[K], wc[K];
#pragma unroll
    for (int j = 0; j < K; ++j) {
      const uint32_t t = tid * K + j;
      const bool live = t < cnt;
      s[j] = live ? sh.s[p][t] : 0u;
      x0[j] = live ? sh.a[p][t] : 0u;
      x1[j] = live ? sh.b[p][t] : 0u;
    }
#pragma unroll
    for (int j = 0; j < K; ++j) {
      if (tid * K + j < cnt) rank_words(R, s[j], x0[j], x1[j], wa[j], wb[j], wc[j]);
      else { wa[j] = wb[j] = wc[j] = 0; }
    }
    // the decision about this round is taken while its rank words are on their way (a round that is not run has
    // loaded them for nothing: cnt <= CAP nodes of the shared frontier are always valid)
    if (tid < 32) {                                  // lanes 0..7 look at a level each (the same in every CTA of the cluster)
      const int k = tid & 7;
      const uint32_t cntk = sh.all_cnt[p][k];
      unsigned long long ecap_k = 0, esoft_k = 0;     // (selected, not indexed: the arguments stay in the constant bank)
#pragma unroll
      for (int j = 0; j < 8; ++j) if (k == j) { ecap_k = a.ecap[j]; esoft_k = a.esoft[j]; }
      const unsigned long long em_k = sh.all_emitted[p][k];
      const bool drain = (__ballot_sync(0xffffffffu, must_drain(em_k, cntk, maxw, ecap_k, esoft_k)) & 0xFFu) != 0;
      uint32_t total = cntk, widest = cntk;
#pragma unroll
      for (int d = 1; d < 8; d <<= 1) {
        total += __shfl_xor_sync(0xffffffffu, total, d);
        widest = max(widest, __shfl_xor_sync(0xffffffffu, widest, d));
      }
      if (tid == 0) {
        // the one-node-per-thread instance is quicker for <= kNarrowEnter nodes, the one-CTA kernel for a handful;
        // a node has <= 2 children: with at most CAP / 2 nodes per level the next round always fits
        const bool narrower = K > 1 ? widest <= kNarrowEnter : a.use_tiny && widest <= a.tiny_enter;
        sh.decision = round_status(total, round, a.round_limit, false, narrower, widest > CAP / 2, drain);
        if (sh.decision == kCseRunning) { visits += total; peak = max(peak, (unsigned long long)total); }
      }
    }
    __syncthreads();
    status = sh.decision;
    if (status != kCseRunning) break;
    NARROW_STAMP(0);

    uint32_t fz = 0, fo = 0, nwsum = 0;
    uint32_t cs0[K], ca[K], cb[K], cs1[K], oa[K], ob[K];       // zero-child and one-child of every node
    uint32_t e0[K], e1[K], e2[K], nw[K];
#pragma unroll
    for (int j = 0; j < K; ++j) {
      cs0[j] = ca[j] = cb[j] = cs1[j] = oa[j] = ob[j] = e0[j] = e1[j] = e2[j] = nw[j] = 0;
      if (tid * K + j < cnt) {
        const CseStep r = cse_step(a, l, a.C[ln], s[j], x0[j], x1[j], wa[j], wb[j], wc[j]);
        cs0[j] = r.zs; cs1[j] = r.os;
        fz |= uint32_t(r.z) << j; ca[j] = r.za; cb[j] = r.zb;
        fo |= uint32_t(r.o) << j; oa[j] = r.oa; ob[j] = r.ob;
        nw[j] = r.nw; e0[j] = r.e0; e1[j] = r.e1; e2[j] = r.e2;
        nwsum += nw[j];
      }
    }
    NARROW_STAMP(1);
    const uint64_t mine = uint64_t(__popc(fz)) | (uint64_t(__popc(fo)) << 21) | (uint64_t(nwsum) << 42);
    uint64_t tot;
    const bool scan_active = warp_of_tid == 0 || warp_of_tid * 32u * K < cnt;      // other warps hold no node: zeros
    const uint64_t excl = block_exclusive_scan_sparse<uint64_t, THREADS>(mine, sh.scan, tot, scan_active);
    NARROW_STAMP(2);
    const uint32_t tz = uint32_t(tot) & 0x1FFFFFu, to = uint32_t(tot >> 21) & 0x1FFFFFu, te = uint32_t(tot >> 42) & 0x1FFFFFu;
    const int q = p ^ 1;
    // the next level's CTA receives its frontier directly in its shared memory
    uint32_t* rs = cluster.map_shared_rank(&sh.s[q][0], ln);
    uint32_t* ra = cluster.map_shared_rank(&sh.a[q][0], ln);
    uint32_t* rb = cluster.map_shared_rank(&sh.b[q][0], ln);
    {
      uint32_t zat = uint32_t(excl) & 0x1FFFFFu;
      uint32_t oat = tz + (uint32_t(excl >> 21) & 0x1FFFFFu);
      unsigned long long pe = cursor + (uint32_t(excl >> 42) & 0x1FFFFFu);
#pragma unroll
      for (int j = 0; j < K; ++j) {
        if (nw[j]) {
          if (pe + nw[j] <= a.ecap[l]) put_words(a.emit[l] + pe, nw[j], e0[j], e1[j], e2[j], x1[j], x0[j] + x1[j]);
          pe += nw[j];
        }
        if (fz >> j & 1u) { rs[zat] = cs0[j]; ra[zat] = ca[j]; rb[zat] = cb[j]; ++zat; }
        if (fo >> j & 1u) { rs[oat] = cs1[j]; ra[oat] = oa[j]; rb[oat] = ob[j]; ++oat; }
      }
    }
    if (tid == 0) {
      *cluster.map_shared_rank(&sh.cz[q], ln) = tz;
      *cluster.map_shared_rank(&sh.co[q], ln) = to;
    }
    if (tid < 8) {            // all-gather: level ln's next size and this level's cursor, to every CTA
      cluster.map_shared_rank(&sh.all_cnt[q][0], tid)[ln] = tz + to;
      cluster.map_shared_rank(&sh.all_emitted[q][0], tid)[l] = cursor + te;
    }
    NARROW_STAMP(3);
    cluster.sync();
    NARROW_STAMP(4);
    p = q;
    ++round;
  }

  // hand the state back in the wide layout
  {
    const int opar = round & 1;
    const uint32_t cz = sh.cz[p], co = sh.co[p];
    for (uint32_t t = tid; t < cz + co; t += THREADS) {
      const uint32_t idx = flat_at(a.cap, cz, t);
      a.fs[opar][l][idx] = sh.s[p][t];
      a.fa[opar][l][idx] = sh.a[p][t];
      a.fb[opar][l][idx] = sh.b[p][t];
    }
    if (tid == 0) {
      S->cnt[opar][l][0] = cz;
      S->cnt[opar][l][1] = co;
      S->emitted[opar][l] = sh.all_emitted[p][l];
      if (l == 0) {
        S->round = round;
        S->status = status;
        S->visits += visits;
        if (peak > S->peak_frontier) S->peak_frontier = peak;
#ifdef BCE_GPU_EXPERIMENTS
        for (int k = 0; k < 5; ++k) S->prof[k] += prof_[k];
#endif
      }
    }
  }
  cluster.sync();     // no CTA may leave while its shared memory can still be a target
}

// ---------------------------------------------------------------------------------
// tiny mode: the last thousands of rounds carry a handful of nodes per level (one per long
// repeat that is still being told apart).  ONE CTA, warp w = level w, at most 32 nodes per level:
// ballots instead of block scans, __syncthreads instead of a cluster barrier -- a round costs
// little more than the latency of its three rank-word loads.
// ---------------------------------------------------------------------------------
constexpr int TN_ITEMS = 1;                       // nodes per lane (4 was measured: 1.25 us per round instead of 0.84, no net gain)
constexpr int TN_CAP = 32 * TN_ITEMS;             // nodes per level
constexpr uint32_t kTinyEnter = TN_CAP / 4, kTinyLeave = TN_CAP / 2;    // <= 2 children per node: the next round fits

struct TinyShared {
  uint32_t s[2][8][TN_CAP], a[2][8][TN_CAP], b[2][8][TN_CAP];
  uint32_t cz[2][8], co[2][8];
  unsigned long long emitted[2][8];
};

__global__ void __launch_bounds__(256, 1) cse_tiny_kernel(CseArgs a) {
  __shared__ TinyShared sh;
  const unsigned tid = threadIdx.x, lane = tid & 31;
  const int l = int(tid >> 5);                       // level handled by this warp
  const int ln = (l + 1) & 7;
  CseDeviceState* S = a.st;
  const uint64_t* __restrict__ R = a.ranks[l];
  const uint32_t maxw = max_words(a);
  const uint32_t one_base = a.C[ln];

  uint32_t round = S->round;
  {
    const int gpar = round & 1;
    const uint32_t cz = S->cnt[gpar][l][0], co = S->cnt[gpar][l][1];
    if (lane == 0) { sh.cz[0][l] = cz; sh.co[0][l] = co; sh.emitted[0][l] = S->emitted[gpar][l]; }
    for (uint32_t t = lane; t < cz + co && t < uint32_t(TN_CAP); t += 32) {
      const uint32_t idx = flat_at(a.cap, cz, t);
      sh.s[0][l][t] = a.fs[gpar][l][idx];
      sh.a[0][l][t] = a.fa[gpar][l][idx];
      sh.b[0][l][t] = a.fb[gpar][l][idx];
    }
  }
  unsigned long long cursor = S->emitted[round & 1][l];
  unsigned long long visits = 0, peak = 0;
  int p = 0;
  __syncthreads();

  uint32_t status;
  for (;;) {
    {   // every thread takes the same decision from the same shared values
      uint32_t total = 0, widest = 0, drain = 0;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const uint32_t cnt = sh.cz[p][k] + sh.co[p][k];
        total += cnt;
        widest = max(widest, cnt);
        if (must_drain(sh.emitted[p][k], cnt, maxw, a.ecap[k], a.esoft[k])) drain = 1;
      }
      status = round_status(total, round, a.round_limit, false, false, widest > kTinyLeave, drain);
      if (status != kCseRunning) break;
      visits += total;
      peak = max(peak, (unsigned long long)total);
    }
    const uint32_t cnt = sh.cz[p][l] + sh.co[p][l];
    // lane owns nodes lane * TN_ITEMS + j: consecutive nodes, so offsets are one warp scan of per-lane sums
    uint32_t s[TN_ITEMS], x0[TN_ITEMS], x1[TN_ITEMS];
    uint64_t wa[TN_ITEMS], wb[TN_ITEMS], wc[TN_ITEMS];
#pragma unroll
    for (int j = 0; j < TN_ITEMS; ++j) {
      const uint32_t t = lane * TN_ITEMS + j;
      const bool live = t < cnt;
      s[j] = live ? sh.s[p][l][t] : 0u;
      x0[j] = live ? sh.a[p][l][t] : 0u;
      x1[j] = live ? sh.b[p][l][t] : 0u;
      if (live) rank_words(R, s[j], x0[j], x1[j], wa[j], wb[j], wc[j]);
      else { wa[j] = wb[j] = wc[j] = 0; }
    }
    uint32_t fz = 0, fo = 0, nwsum = 0;
    uint32_t cs0[TN_ITEMS], ca[TN_ITEMS], cb[TN_ITEMS], cs1[TN_ITEMS], oa[TN_ITEMS], ob[TN_ITEMS];
    uint32_t e0[TN_ITEMS], e1[TN_ITEMS], e2[TN_ITEMS], nw[TN_ITEMS];
#pragma unroll
    for (int j = 0; j < TN_ITEMS; ++j) {
      cs0[j] = ca[j] = cb[j] = cs1[j] = oa[j] = ob[j] = e0[j] = e1[j] = e2[j] = nw[j] = 0;
      if (lane * TN_ITEMS + j < cnt) {
        const CseStep r = cse_step(a, l, one_base, s[j], x0[j], x1[j], wa[j], wb[j], wc[j]);
        cs0[j] = r.zs; cs1[j] = r.os;
        fz |= uint32_t(r.z) << j; ca[j] = r.za; cb[j] = r.zb;
        fo |= uint32_t(r.o) << j; oa[j] = r.oa; ob[j] = r.ob;
        nw[j] = r.nw; e0[j] = r.e0; e1[j] = r.e1; e2[j] = r.e2;
        nwsum += nw[j];
      }
    }
    // packed inclusive warp scan: zero-children | one-children << 8 | emitted words << 16
    const uint32_t mine = uint32_t(__popc(fz)) | (uint32_t(__popc(fo)) << 8) | (nwsum << 16);
    uint32_t inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= unsigned(d)) inc += o;
    }
    const uint32_t tot = __shfl_sync(0xffffffffu, inc, 31);
    const uint32_t tz = tot & 255u, to = (tot >> 8) & 255u, te = tot >> 16;
    const uint32_t excl = inc - mine;
    const int q = p ^ 1;
    {
      uint32_t zat = excl & 255u, oat = tz + ((excl >> 8) & 255u);
      unsigned long long pe = cursor + (excl >> 16);
#pragma unroll
      for (int j = 0; j < TN_ITEMS; ++j) {
        if (nw[j]) {
          if (pe + nw[j] <= a.ecap[l]) put_words(a.emit[l] + pe, nw[j], e0[j], e1[j], e2[j], x1[j], x0[j] + x1[j]);
          pe += nw[j];
        }
        if (fz >> j & 1u) { sh.s[q][ln][zat] = cs0[j]; sh.a[q][ln][zat] = ca[j]; sh.b[q][ln][zat] = cb[j]; ++zat; }
        if (fo >> j & 1u) { sh.s[q][ln][oat] = cs1[j]; sh.a[q][ln][oat] = oa[j]; sh.b[q][ln][oat] = ob[j]; ++oat; }
      }
    }
    cursor += te;
    if (lane == 0) { sh.cz[q][ln] = tz; sh.co[q][ln] = to; sh.emitted[q][l] = cursor; }
    __syncthreads();
    p = q;
    ++round;
  }

  {   // hand the state back in the wide layout
    const int opar = round & 1;
    const uint32_t cz = sh.cz[p][l], co = sh.co[p][l];
    for (uint32_t t = lane; t < cz + co; t += 32) {
      const uint32_t idx = flat_at(a.cap, cz, t);
      a.fs[opar][l][idx] = sh.s[p][l][t];
      a.fa[opar][l][idx] = sh.a[p][l][t];
      a.fb[opar][l][idx] = sh.b[p][l][t];
    }
    if (lane == 0) {
      S->cnt[opar][l][0] = cz;
      S->cnt[opar][l][1] = co;
      S->emitted[opar][l] = cursor;
      if (l == 0) {
        S->round = round;
        S->status = status;
        S->visits += visits;
        if (peak > S->peak_frontier) S->peak_frontier = peak;
      }
    }
  }
}

// ---------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------
// Every instance of the level loop's kernels the host can launch.
enum class CseKernel { Tiny, Cluster1, Cluster8, Mid1, Mid2, Mid4, Slots, Wide2, Wide4 };
static const char* const kCseKernelName[] = {"tiny", "cluster1", "cluster8", "mid1", "mid2", "mid4", "slots", "wide2", "wide4"};
static bool is_narrow(CseKernel k) { return k <= CseKernel::Cluster8; }

struct CseHost {
  CseArgs args;
  uint32_t n = 0;
  uint32_t pick_widest = 0;              // widest level when a kernel last asked for a narrower or wider one (pick_kernel)
  uint32_t last_round = 0;
  // wide kernel variants: [0] = 2 nodes per thread (512-node tiles), [1] = 4 (1024-node tiles)
  const void* var_fn[2] = {nullptr, nullptr};
  size_t var_smem[2] = {0, 0};
  int var_grid[2] = {0, 0};
  unsigned long long slot_enter = 0;     // frontiers of this many nodes go to the slot layout and the 1024-node tiles
  unsigned long long known_nodes = 0;    // frontier size after the last launch
  // emission: one or two sets of device buffers (two = copy of batch k overlaps compute of k+1)
  int sets = 1;
  uint32_t* emit_dev[2][8] = {};
  size_t ecap_words = 0;                 // allocated per stream and set
  size_t batch_words = 0;                // capacity the kernels are told (<= ecap_words); grows if a round does not fit
  int fill_set = 0;                      // set the kernels write next
  // a computed batch waiting to be copied out / returned
  bool pending = false, pending_done = false;
  int pending_set = 0;
  size_t pending_cnt[8] = {};
  int pinned_flip = 0;
  bool use_medium = false;               // the <512, 8> cluster kernel is available
  int last_grid = 0;                     // grid size of the previous wide launch (0 = none since cse_begin)
  bool tail_cut = false;                 // hosted emission: the batch was already cut where the frontier collapsed
  bool finished = false;                 // the level loop terminated
  uint32_t desc_epoch = 0;               // round >> 29 at which the descriptors were last cleared
  unsigned long long sum_words[8] = {};  // resident checksum: words of every stream summed so far
  // huge frontiers: slot layout (cse_slots.cuh)
  SlotArgs slot = {};
  bool slots_ok = false;                 // memory for the slot layout was set aside
  bool in_slots = false;                 // the frontier currently lives in slots (else flat layout)
  const void* slot_fn = nullptr;
  int slot_grid = 0;
  // frontiers between the cluster kernels' and the wide kernel's: slot layout with redundant scans (cse_mid.cuh)
  MidArgs mid = {};
  bool mid_ok = false;
  const void* mid_fn[3] = {nullptr, nullptr, nullptr};   // 1, 2, 4 nodes per lane
  int mid_grid = 0;
  unsigned long long mid_enter = 0;      // frontiers of at most this many nodes go to cse_mid_kernel
  unsigned long long mid_e0 = 0, mid_e1 = 0;   // ... at most e0: 1 node per lane, at most e1: 2, else 4
};

static size_t env_size(const char* name, size_t dflt) { return exp_env(name, dflt); }   // experiment builds only

void cse_destroy(Ctx* c) {
  delete c->cse;
  c->cse = nullptr;
  c->cse_active = false;
}

int cse_begin(Ctx* c, uint32_t n) {
  if (!c->ranks_resident) { set_error(c, "cse_begin: wavelet matrix not built"); return BCE_GPU_E_STATE; }
  if (!c->cse) c->cse = new CseHost();
  CseHost* H = c->cse;
  H->n = n;
  cudaStream_t st = c->stream;
  CseArgs& a = H->args;
  a.emit_mode = c->emit_mode;
  memcpy(a.cfgbits, c->emit_cfg, sizeof a.cfgbits);
  const size_t wmax = a.emit_mode == kEmitRaw ? 5 : 3;      // words one count can take (scan: 1, sized like coder)

  // ---- sizing: frontier first (correctness), emission with what is left ------------
  const size_t budget = scratch_budget(c);
  const size_t cap_full = ((size_t(n) / 2 + 4) + 3) & ~size_t(3);
  size_t cap = cap_full;
  auto frontier_bytes = [](size_t cp) { return 48 * Carver::need(cp, 4); };
  // Inputs whose frontier can reach millions of nodes keep it in the slot layout while it is that large
  // (cse_slots.cuh); the flat layout then only has to hold what the other kernels see: at most kSlotLeave nodes
  // coming back plus one doubling before the host switches over again.
  const size_t kFlatCapWithSlots = std::max<size_t>(size_t(16) << 20, size_t(4) * c->slot_enter_nodes);
  H->slot_enter = c->slot_enter_nodes;
  const bool want_slots = uint64_t(n) >= 8 * c->slot_enter_nodes && env_size("BCE_GPU_NO_SLOTS", 0) == 0;
  if (want_slots && cap > kFlatCapWithSlots) cap = kFlatCapWithSlots;
  while (cap > 4096 && frontier_bytes(cap) > budget / 2) cap = (cap / 2 + 3) & ~size_t(3);
  const size_t desc_tiles = 8 * (cap / CS_THREADS + 2);      // sized for the smallest tile of any variant
  const size_t desc_bytes = Carver::need(3 * desc_tiles, 8);
  size_t left = budget > frontier_bytes(cap) + desc_bytes ? budget - frontier_bytes(cap) - desc_bytes : 0;
  // slot layout: two node arenas (3 x 4 B per place), E-slots, directories -- from half of what is left
  size_t arena_cap = 0, chunk_cap = 0, dir_cap = 0, slot_bytes = 0;
  int slot_grid = 0;
  if (want_slots) {
    const void* fn = a.emit_mode == kEmitRaw ? (const void*)cse_slots_kernel<5> : (const void*)cse_slots_kernel<3>;
    int per_sm = 0;
    BCE_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, SL_THREADS, 0));
    slot_grid = per_sm * c->sm_count;
    H->slot_fn = fn;
    const size_t per_place = 2 * 12 + (wmax * 4) / 2 + 1;   // arenas + E-slot share (one E-slot per 2 places) + directories
    arena_cap = std::min<size_t>(size_t(4) * n + 4096, (left / 2) / per_place);
    arena_cap = std::min<size_t>(arena_cap, 0xFFFF0000ull) & ~size_t(SL_CH - 1);
    chunk_cap = arena_cap / (2 * SL_CH) + 16;
    dir_cap = 2 * chunk_cap + 64;
    slot_bytes = 6 * Carver::need(arena_cap, 4) + Carver::need(chunk_cap * SL_CH * wmax, 4) + Carver::need(chunk_cap, 2) +
                 2 * Carver::need(dir_cap, 1) + 4 * Carver::need(dir_cap, 4) + Carver::need(size_t(16) * slot_grid, 4) +
                 Carver::need(1, sizeof(SlotState)) + 4096;
    if (slot_grid < 1 || arena_cap < 8 * c->slot_enter_nodes || slot_bytes > left) { slot_bytes = 0; }
    else left -= slot_bytes;
  }
  H->slots_ok = slot_bytes != 0;
  H->in_slots = false;
  // medium frontiers: two arenas of MD_SLOTS slots, double-buffered E-slots and the two directories
  size_t mid_bytes = 0;
  H->mid_ok = false;
  H->mid_enter = std::min<unsigned long long>(c->mid_enter_nodes, mid_max_nodes(4));
  // (a small MID_ENTER_NODES -- tests -- scales the instance thresholds down with it, so that all three instances run)
  H->mid_e0 = std::min<unsigned long long>({env_size("BCE_GPU_MID_E0", 96 << 10), mid_max_nodes(1) * 3 / 4, H->mid_enter / 4});
  H->mid_e1 = std::min<unsigned long long>({env_size("BCE_GPU_MID_E1", 192 << 10), mid_max_nodes(2) * 3 / 4, H->mid_enter / 2});
  if (n >= 8192 && H->mid_enter > 1) {
    const bool raw = a.emit_mode == kEmitRaw;
    H->mid_fn[0] = raw ? (const void*)cse_mid_kernel<5, 1> : (const void*)cse_mid_kernel<3, 1>;
    H->mid_fn[1] = raw ? (const void*)cse_mid_kernel<5, 2> : (const void*)cse_mid_kernel<3, 2>;
    H->mid_fn[2] = raw ? (const void*)cse_mid_kernel<5, 4> : (const void*)cse_mid_kernel<3, 4>;
    int per_sm = 1;
    for (const void* fn : H->mid_fn) {
      int p1 = 0;
      BCE_CUDA(c, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(MidShared))));
      BCE_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p1, fn, MD_THREADS, sizeof(MidShared)));
      per_sm = std::min(per_sm, p1);
    }
    mid_bytes = Carver::need(6 * MD_PLACES, 4) + Carver::need(2 * size_t(MD_SLOTS), 1) +
                Carver::need(2 * size_t(MD_TCAP) * 32 * MD_MAX_ITEMS * wmax, 4) + Carver::need(2 * size_t(MD_TCAP), 2) + 4096;
    if (per_sm < 1 || mid_bytes > left / 2) mid_bytes = 0;
    else { left -= mid_bytes; H->mid_grid = c->sm_count; }
  }
  H->sets = (c->cse_resident || env_size("BCE_GPU_NO_OVERLAP", 0)) ? 1 : 2;
  // words handed back per batch and stream: small batches let the copy of batch k overlap the
  // kernels of batch k+1 (two pinned buffers of this size alternate)
  const size_t batch_bytes = c->emit_batch_bytes;          // BCE_GPU_OPT_EMIT_BATCH_BYTES
  size_t ew = size_t(n) * wmax;                              // a level emits at most n-1 counts in total
  const size_t per_level_min = (cap + CS_MAX_TILE) * wmax;   // one round must always fit
  if (ew * 8 * 4 * H->sets > left) ew = left / (8 * 4 * H->sets);
  if (ew < per_level_min) ew = per_level_min;
  const size_t need = frontier_bytes(cap) + desc_bytes + size_t(H->sets) * 8 * Carver::need(ew, 4) + slot_bytes + mid_bytes + 4096;
  BCE_TRY(c->scratch.ensure(c, need));
  Carver cv(c->scratch.p, c->scratch.cap);
  for (int p = 0; p < 2; ++p)
    for (int l = 0; l < 8; ++l) {
      a.fs[p][l] = cv.take<uint32_t>(cap);
      a.fa[p][l] = cv.take<uint32_t>(cap);
      a.fb[p][l] = cv.take<uint32_t>(cap);
    }
  a.desc = cv.take<uint64_t>(3 * desc_tiles);
  for (int s = 0; s < H->sets; ++s)
    for (int l = 0; l < 8; ++l) H->emit_dev[s][l] = cv.take<uint32_t>(ew);
  if (H->slots_ok) {
    SlotArgs& sl = H->slot;
    for (int p = 0; p < 2; ++p) {
      sl.ns[p] = cv.take<uint32_t>(arena_cap);
      sl.na[p] = cv.take<uint32_t>(arena_cap);
      sl.nb[p] = cv.take<uint32_t>(arena_cap);
      sl.cnt[p] = cv.take<uint8_t>(dir_cap);
      sl.P[p] = cv.take<uint32_t>(dir_cap);
      sl.start[p] = cv.take<uint32_t>(dir_cap);
    }
    sl.eslot = cv.take<uint32_t>(chunk_cap * SL_CH * wmax);
    sl.ecnt = cv.take<uint16_t>(chunk_cap);
    sl.partial = cv.take<uint32_t>(size_t(16) * slot_grid);
    sl.ss = cv.take<SlotState>(1);
    sl.arena_cap = uint32_t(arena_cap);
    sl.chunk_cap = uint32_t(chunk_cap);
    sl.dir_cap = uint32_t(dir_cap);
    H->slot_grid = slot_grid;
  }
  if (mid_bytes) {
    MidArgs& m = H->mid;
    m.arena = cv.take<uint32_t>(6 * MD_PLACES);
    m.cnt = cv.take<uint8_t>(2 * size_t(MD_SLOTS));
    m.eslot = cv.take<uint32_t>(2 * size_t(MD_TCAP) * 32 * MD_MAX_ITEMS * wmax);
    m.ecnt = cv.take<uint16_t>(2 * size_t(MD_TCAP));
    H->mid_ok = true;
  }
  if (!cv.ok()) { set_error(c, "cse_begin: scratch carve failed (need %zu)", need); return BCE_GPU_E_NOMEM; }
  H->ecap_words = ew;
  // per-stream target: the streams are uneven (the largest carries about a third of the words), so a third of the
  // batch's words per stream makes batches of about batch_bytes in all
  // ... and never more than a third of a word per input byte, so that a smaller input still leaves in a
  // handful of batches whose copies overlap the kernels (the whole emission is ~1.6 words per byte)
  H->batch_words = c->cse_resident ? ew : std::min(ew, std::max(std::min(batch_bytes / 12, size_t(n) / env_size("BCE_GPU_BATCH_DIV", 3)), size_t(1) << 16));
  H->fill_set = 0;
  // the worst case (every node emits its widest count) is checked against the whole device buffer; the batch
  // size is a target that the words actually emitted are compared with (a round emits ~0.2 words per node)
  for (int l = 0; l < 8; ++l) { a.emit[l] = H->emit_dev[0][l]; a.ecap[l] = ew; a.esoft[l] = H->batch_words; }
  const size_t words = size_t(n) / 32 + 1;
  for (int l = 0; l < 8; ++l) { a.ranks[l] = c->ranks.as<uint64_t>() + size_t(l) * words; a.C[l] = c->C[l]; }
  a.cap = uint32_t(cap);
  a.desc_tiles = uint32_t(desc_tiles);
  a.round_limit = uint32_t(std::min<uint64_t>(uint64_t(n) * 8 + 64, 0xFFFFFFF0ull));
  a.use_narrow = c->no_narrow_kernels ? 0u : 1u;
  a.min_nodes = 0;
  a.max_nodes = ~0ull;
  a.st = reinterpret_cast<CseDeviceState*>(c->small.as<char>() + kSmallCse);
  static_assert(sizeof(CseDeviceState) <= 1024, "state must fit its slot in Ctx::small");
  H->use_medium = a.use_narrow && !env_size("BCE_GPU_NO_MEDIUM", 0);
  a.use_tiny = (a.use_narrow && !env_size("BCE_GPU_NO_TINY", 0)) ? 1u : 0u;
  a.tiny_enter = kTinyEnter;
  H->pick_widest = 1;                    // the roots are one node per level
  a.narrow_enter = H->use_medium ? kMediumEnter : kNarrowEnter;
  // function attributes are per device: set for this context's device on every run (a process may hold
  // contexts on several GPUs)
  BCE_CUDA(c, cudaFuncSetAttribute(cse_narrow_kernel<1024, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   int(sizeof(NarrowShared<1024, 1>))));
  BCE_CUDA(c, cudaFuncSetAttribute(cse_narrow_kernel<NM_THREADS, NM_K>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   int(sizeof(NarrowShared<NM_THREADS, NM_K>))));
  H->last_round = 0;
  H->known_nodes = 0;
  H->pending = H->pending_done = H->finished = false;
  H->tail_cut = false;
  H->last_grid = 0;
  H->pinned_flip = 0;                        // single-batch runs always land in the same pinned buffer

  BCE_CUDA(c, cudaMemsetAsync(a.desc, 0, 3 * desc_tiles * sizeof(uint64_t), st));
  H->desc_epoch = 0;
  if (c->cse_resident && c->resident_checksum) {
    BCE_CUDA(c, cudaMemsetAsync(c->small.as<char>() + kSmallChecksum, 0, 16 * sizeof(unsigned long long), st));
    for (auto& w : H->sum_words) w = 0;
  }
  cse_init_kernel<<<1, 32, 0, st>>>(a, n);
  c->stats.gpu_launches++;
  BCE_CUDA(c, cudaGetLastError());

  {   // wide kernel instances: raw counts need 5 staging words per node, packed ones 3
    const bool packed = a.emit_mode != kEmitRaw;
    const void* f2 = packed ? (const void*)cse_wide_kernel<2, 3> : (const void*)cse_wide_kernel<2, 5>;
    const void* f4 = packed ? (const void*)cse_wide_kernel<4, 3> : (const void*)cse_wide_kernel<4, 5>;
    const size_t s2 = packed ? 2 * sizeof(WideStage<2, 3>) : 2 * sizeof(WideStage<2, 5>);
    const size_t s4 = packed ? 2 * sizeof(WideStage<4, 3>) : 2 * sizeof(WideStage<4, 5>);
    {
      int p2 = 0, p4 = 0;
      BCE_CUDA(c, cudaFuncSetAttribute(f2, cudaFuncAttributeMaxDynamicSharedMemorySize, int(s2)));
      BCE_CUDA(c, cudaFuncSetAttribute(f4, cudaFuncAttributeMaxDynamicSharedMemorySize, int(s4)));
      BCE_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p2, f2, CS_THREADS, s2));
      BCE_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p4, f4, CS_THREADS, s4));
      if (p2 < 1 || p4 < 1) { H->var_fn[0] = nullptr; set_error(c, "cse kernel does not fit on an SM"); return BCE_GPU_E_CUDA; }
      H->var_fn[0] = f2; H->var_smem[0] = s2; H->var_grid[0] = p2 * c->sm_count;
      H->var_fn[1] = f4; H->var_smem[1] = s4; H->var_grid[1] = p4 * c->sm_count;
    }
  }
  c->cse_active = true;
  c->cse_done = false;
  BCE_TRACE("cse_begin n=%u cap=%zu ecap_words=%zu sets=%d mode=%u grids=%d/%d", n, cap, ew, H->sets, a.emit_mode,
            H->var_grid[0], H->var_grid[1]);
  return BCE_GPU_OK;
}

// The kernel that takes the next rounds, and the frontier sizes (min_nodes, max_nodes) at which a wide kernel hands
// back (kCseGoWide): the gaps between the thresholds that enter and leave a kernel keep the host from switching back
// and forth.  Narrow or not follows the widest level; the kernels for wider frontiers follow the frontier size.
struct CsePick {
  CseKernel k;
  unsigned long long min_nodes, max_nodes;
};
static CsePick pick_kernel(const CseHost* H, uint32_t widest, unsigned long long nodes) {
  if (H->args.use_narrow) {
    if (H->args.use_tiny && widest <= kTinyEnter) return {CseKernel::Tiny, 0, ~0ull};
    if (widest <= kNarrowEnter) return {CseKernel::Cluster1, 0, ~0ull};
    if (H->use_medium && widest <= kMediumEnter) return {CseKernel::Cluster8, 0, ~0ull};
  }
  // huge frontiers: the slot layout while the frontier holds at least half of slot_enter nodes
  const unsigned long long big = H->slot_enter;
  if (H->slots_ok && (H->in_slots || nodes >= big)) return {CseKernel::Slots, big / 2, ~0ull};
  // some thousand to half a million nodes per round: the thinner a round, the fewer nodes per lane (a warp alone on its
  // scheduler is bound by its own latencies)
  if (H->mid_ok && nodes <= H->mid_enter) {
    if (nodes <= H->mid_e0) return {CseKernel::Mid1, 0, mid_max_nodes(1)};
    if (nodes <= H->mid_e1) return {CseKernel::Mid2, H->mid_e0 * 3 / 4, mid_max_nodes(2)};
    return {CseKernel::Mid4, H->mid_e1 * 3 / 4, mid_max_nodes(4)};
  }
  // 1024-node tiles while the frontier is huge, 512-node tiles below (more CTAs per round); from those back to
  // cse_mid_kernel once the frontier has shrunk
  if (nodes >= big) return {CseKernel::Wide4, big / 2, ~0ull};
  return {CseKernel::Wide2, H->mid_ok ? H->mid_enter : 0, big + big / 2};
}

// Runs kernels until the level loop ends or an emission buffer of set `set` may overflow.
// On return cnt[l] = words emitted into that set, *done = loop finished.
static int run_batch(Ctx* c, int set, size_t cnt[8], bool* done) {
  CseHost* H = c->cse;
  cudaStream_t st = c->stream;
  CseDeviceState* h_state = reinterpret_cast<CseDeviceState*>(c->pinned_small.as<char>() + 40 * 1024);
  for (int l = 0; l < 8; ++l) H->args.emit[l] = H->emit_dev[set][l];
  BCE_CUDA(c, cudaEventRecord(c->ev[2], st));
  bool cut = false;                      // batch ended by the host between two kernels
  for (int hops = 0;; ++hops) {
    if (hops > 100000) { set_error(c, "cse: wide/narrow ping-pong"); return BCE_GPU_E_INTERNAL; }
    const CsePick pick = pick_kernel(H, H->pick_widest, H->known_nodes);
    const CseKernel k = pick.k;
    H->args.min_nodes = pick.min_nodes;
    H->args.max_nodes = pick.max_nodes;
    BCE_CUDA(c, cudaEventRecord(c->ev[0], st));
    // the grid barrier's targets are multiples of the grid size: another grid starts a new count
    const int grid = k == CseKernel::Slots ? H->slot_grid
                   : k == CseKernel::Wide2 ? H->var_grid[0] : k == CseKernel::Wide4 ? H->var_grid[1]
                   : is_narrow(k) ? 0 : H->mid_grid;
    if (grid && grid != H->last_grid) {
      if (H->last_grid) { cse_reset_barrier_kernel<<<1, 1, 0, st>>>(H->args.st); c->stats.gpu_launches++; }
      H->last_grid = grid;
    }
    switch (k) {
      case CseKernel::Tiny:
        cse_tiny_kernel<<<1, 256, 0, st>>>(H->args);
        BCE_CUDA(c, cudaGetLastError());
        break;
      case CseKernel::Cluster1:
        cse_narrow_kernel<1024, 1><<<8, 1024, sizeof(NarrowShared<1024, 1>), st>>>(H->args);
        BCE_CUDA(c, cudaGetLastError());
        break;
      case CseKernel::Cluster8:
        cse_narrow_kernel<NM_THREADS, NM_K><<<8, NM_THREADS, sizeof(NarrowShared<NM_THREADS, NM_K>), st>>>(H->args);
        BCE_CUDA(c, cudaGetLastError());
        break;
      case CseKernel::Mid1:
      case CseKernel::Mid2:
      case CseKernel::Mid4: {
        // slot layout with one grid barrier per round.  The kernel reads the flat layout in its first round and writes
        // it back when it leaves (kCseGoWide outside [min_nodes, max_nodes], kCseGoNarrow, batch full, done).
        void* kargs[] = {&H->args, &H->mid};
        BCE_CUDA(c, cudaLaunchCooperativeKernel(H->mid_fn[int(k) - int(CseKernel::Mid1)], dim3(grid), dim3(MD_THREADS),
                                                kargs, sizeof(MidShared), st));
        break;
      }
      case CseKernel::Slots: {
        // coming from the flat layout the frontier is converted first and the kernel starts with its scan phase; it
        // comes back (kCseGoWide) when fewer than min_nodes are left
        uint32_t first_scan = 0;
        if (!H->in_slots) {
          cse_flat_to_slots_kernel<<<c->sm_count * 4, 256, 0, st>>>(H->args, H->slot);
          c->stats.gpu_launches++;
          BCE_CUDA(c, cudaGetLastError());
          first_scan = 1;
          H->in_slots = true;
        }
        void* kargs[] = {&H->args, &H->slot, &first_scan};
        BCE_CUDA(c, cudaLaunchCooperativeKernel(H->slot_fn, dim3(grid), dim3(SL_THREADS), kargs, 0, st));
        break;
      }
      case CseKernel::Wide2:
      case CseKernel::Wide4: {
        if ((H->last_round >> 29) != H->desc_epoch) {   // 30-bit tags: no descriptor older than 2^29 rounds may survive
          BCE_CUDA(c, cudaMemsetAsync(H->args.desc, 0, 3 * size_t(H->args.desc_tiles) * sizeof(uint64_t), st));
          H->desc_epoch = H->last_round >> 29;
        }
        const int v = k == CseKernel::Wide4 ? 1 : 0;
        void* kargs[] = {&H->args};
        BCE_CUDA(c, cudaLaunchCooperativeKernel(H->var_fn[v], dim3(grid), dim3(CS_THREADS), kargs, H->var_smem[v], st));
        break;
      }
    }
    c->stats.gpu_launches++;
    c->stats.cse_launches++;
    BCE_CUDA(c, cudaMemcpyAsync(h_state, H->args.st, sizeof(CseDeviceState), cudaMemcpyDeviceToHost, st));
    BCE_CUDA(c, cudaEventRecord(c->ev[1], st));
    BCE_CUDA(c, cudaStreamSynchronize(st));
    {
      float lms = 0;
      BCE_CUDA(c, cudaEventElapsedTime(&lms, c->ev[0], c->ev[1]));
      if (is_narrow(k)) { c->stats.ms_cse_narrow += lms; c->stats.cse_rounds_narrow += h_state->round - H->last_round; }
      BCE_TRACE("cse %s kernel: rounds %u..%u status=%u err=%u visits=%llu %.3f ms", kCseKernelName[int(k)],
                H->last_round, h_state->round, h_state->status, h_state->err, h_state->visits, lms);
#ifdef BCE_GPU_EXPERIMENTS
      {
        static unsigned long long prev[8] = {};
        if (h_state->prof[0] < prev[0]) for (auto& v : prev) v = 0;     // a new run started the sums again
        const uint32_t nr = std::max(1u, h_state->round - H->last_round);
        BCE_TRACE("   phases (CTA 0, cycles per round): %.0f %.0f %.0f %.0f %.0f %.0f", double(h_state->prof[0] - prev[0]) / nr,
                  double(h_state->prof[1] - prev[1]) / nr, double(h_state->prof[2] - prev[2]) / nr, double(h_state->prof[3] - prev[3]) / nr,
                  double(h_state->prof[4] - prev[4]) / nr, double(h_state->prof[5] - prev[5]) / nr);
        for (int i = 0; i < 8; ++i) prev[i] = h_state->prof[i];
      }
#endif
      H->last_round = h_state->round;
      if (H->in_slots && h_state->status == kCseGoWide && !h_state->err) {
        // the frontier has shrunk: back to the flat layout (exact half sizes come with it)
        cse_slots_to_flat_kernel<<<c->sm_count * 4, 256, 0, st>>>(H->args, H->slot);
        c->stats.gpu_launches++;
        BCE_CUDA(c, cudaGetLastError());
        BCE_CUDA(c, cudaMemcpyAsync(h_state, H->args.st, sizeof(CseDeviceState), cudaMemcpyDeviceToHost, st));
        BCE_CUDA(c, cudaStreamSynchronize(st));
        H->in_slots = false;
      }
      const int par = h_state->round & 1;
      H->known_nodes = 0;
      for (int l = 0; l < 8; ++l) H->known_nodes += h_state->cnt[par][l][0] + h_state->cnt[par][l][1];
    }
    if (h_state->err) break;
    if (h_state->status == kCseGoWide || h_state->status == kCseGoNarrow) {
      {   // the widest level decides whether a narrow kernel takes the next rounds
        const int par = h_state->round & 1;
        uint32_t widest = 0;
        for (int l = 0; l < 8; ++l) widest = std::max(widest, h_state->cnt[par][l][0] + h_state->cnt[par][l][1]);
        H->pick_widest = widest;
        // the one-node-per-thread kernel asked to leave (> 512) or the wide one asked to hand over (<= narrow_enter):
        // both are consistent with pick_kernel, so no kernel is relaunched just to bounce back
      }
      // Hosted emission: when the frontier has collapsed, what follows is thousands of short rounds
      // that emit little.  End the batch here so that its copy to the host runs under that tail
      // instead of after it.
      if (H->sets == 2 && !H->tail_cut && H->known_nodes < 2000000ull) {
        const int par = h_state->round & 1;
        size_t have = 0;
        for (int l = 0; l < 8; ++l) have += size_t(h_state->emitted[par][l]);
        if (have >= (size_t(4) << 20)) {
          BCE_TRACE("cse: batch cut at round %u: frontier down to %llu nodes, %zu words pending", h_state->round,
                    H->known_nodes, have);
          H->tail_cut = true;
          cut = true;
          break;
        }
      }
      continue;
    }
    break;
  }
  BCE_CUDA(c, cudaEventRecord(c->ev[3], st));
  BCE_CUDA(c, cudaEventSynchronize(c->ev[3]));
  float ms = 0;
  BCE_CUDA(c, cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]));
  c->stats.ms_cse += ms;

  if (h_state->err) {
    set_error(c, "cse: %s watchdog fired (round %u, barrier_fail %u, arrivals %llu, barriers %llu)",
              h_state->err == 2 ? "grid-barrier" : "chained-scan", h_state->round, h_state->barrier_fail,
              h_state->arrivals, h_state->barriers);
    return BCE_GPU_E_INTERNAL;
  }
  if (h_state->status == kCseRunaway) {
    set_error(c, "cse: level loop still running after %u rounds (n = %u)", h_state->round, H->n);
    return BCE_GPU_E_INTERNAL;
  }
  if (h_state->status == kCseOverflow) {
    set_error(c, "cse: node frontier exceeded %u nodes per level at round %u", H->args.cap, h_state->round);
    return BCE_GPU_E_FRONTIER;
  }
  if (h_state->status != kCseDone && h_state->status != kCseDrain && !cut) {
    set_error(c, "cse: unexpected kernel status %u", h_state->status);
    return BCE_GPU_E_INTERNAL;
  }
  const int par = h_state->round & 1;
  size_t total = 0;
  for (int l = 0; l < 8; ++l) { cnt[l] = size_t(h_state->emitted[par][l]); total += cnt[l]; }
  if (h_state->status == kCseDrain && total == 0) {
    // the coming round alone does not fit the batch size: enlarge it (the buffers are big enough
    // for any round) and go on -- nothing was processed, no state is lost
    if (H->batch_words < H->ecap_words) {
      H->batch_words = std::min(H->ecap_words, H->batch_words * 2);
      for (int l = 0; l < 8; ++l) H->args.esoft[l] = H->batch_words;
      BCE_TRACE("cse: batch size raised to %zu words per stream", H->batch_words);
      cse_reset_emitted_kernel<<<1, 32, 0, st>>>(H->args.st);
      c->stats.gpu_launches++;
      BCE_CUDA(c, cudaGetLastError());
      return run_batch(c, set, cnt, done);
    }
    set_error(c, "cse: kernel asked to drain empty emission buffers at round %u", h_state->round);
    return BCE_GPU_E_INTERNAL;
  }
  c->stats.cse_words += total;
  if (H->args.emit_mode == kEmitRaw) c->stats.cse_tuples += total / 5;
  c->stats.cse_visits = h_state->visits;
  c->stats.cse_rounds = h_state->round ? h_state->round : 1;   // the reference's do..while runs at least once
  c->stats.cse_peak_frontier = h_state->peak_frontier;
  if (c->cse_resident && c->resident_checksum) {
    unsigned long long* acc = reinterpret_cast<unsigned long long*>(c->small.as<char>() + kSmallChecksum);
    for (int l = 0; l < 8; ++l) {
      if (!cnt[l]) continue;
      const int grid = int(std::min<size_t>((cnt[l] + 255) / 256, size_t(c->sm_count) * 8));
      cse_checksum_kernel<<<grid, 256, 0, st>>>(H->emit_dev[set][l], cnt[l], H->sum_words[l], acc + 2 * l);
      c->stats.gpu_launches++;
      H->sum_words[l] += cnt[l];
    }
    BCE_CUDA(c, cudaGetLastError());
  }
  *done = h_state->status == kCseDone;
  if (*done) {
    H->finished = true;
  } else {
    cse_reset_emitted_kernel<<<1, 32, 0, st>>>(H->args.st);
    c->stats.gpu_launches++;
    BCE_CUDA(c, cudaGetLastError());
  }
  return BCE_GPU_OK;
}

// One batch of emitted words.  resident: counts stay in device memory (measurement), the
// whole loop runs here.  Otherwise a batch is copied to pinned host memory on the copy stream
// while the kernels already fill the other buffer set with the next batch.
int cse_advance(Ctx* c, bool resident, CseWordBatch* out, bool pack20) {
  if (!c->cse_active || !c->cse) { set_error(c, "cse_next without cse_begin"); return BCE_GPU_E_STATE; }
  CseHost* H = c->cse;
  if (out) memset(out, 0, sizeof *out);
  if (c->cse_done) { if (out) out->done = 1; return BCE_GPU_OK; }

  if (resident) {
    size_t cnt[8];
    bool done = false;
    BCE_TRY(run_batch(c, 0, cnt, &done));
    if (done) c->cse_done = true;
    return BCE_GPU_OK;
  }
  if (!out) return BCE_GPU_E_ARG;

  if (!H->pending) {                                    // first call: nothing computed yet
    BCE_TRY(run_batch(c, H->fill_set, H->pending_cnt, &H->pending_done));
    H->pending = true;
    H->pending_set = H->fill_set;
    if (H->sets == 2) H->fill_set ^= 1;
  }
  // copy the pending batch out on the copy stream ...
  if (pack20 && H->args.emit_mode != kEmitCoder) { set_error(c, "20-bit words need BCE_EMIT_CODER"); return BCE_GPU_E_STATE; }
  size_t bytes = 64, at_b[8];
  for (int l = 0; l < 8; ++l) {                           // the pack kernel writes whole groups of 8 words = 20 bytes
    at_b[l] = bytes;                                      // (+ 16: the host reads 8 bytes at a time)
    bytes += ((pack20 ? (H->pending_cnt[l] + 7) / 8 * 20 + 16 : H->pending_cnt[l] * 4) + 15) & ~size_t(15);
  }
  PinnedBuf& pin = H->pinned_flip ? c->pinned_emit2 : c->pinned_emit;
  H->pinned_flip ^= 1;
  BCE_TRY(pin.ensure(c, bytes));
  char* hp = pin.as<char>();
  if (pack20) BCE_TRY(c->pack_tmp.ensure(c, bytes));
  cudaStream_t cs = c->copy_stream;
  if (pack20) {
    // Packed on the compute stream, before the next batch's kernels: those are persistent and hold every SM, a pack
    // kernel on the copy stream would wait for them and the copy with it (measured: e2e 326 -> 360 ms).  ~0.5 ms per GB.
    for (int l = 0; l < 8; ++l) {
      if (!H->pending_cnt[l]) continue;
      uint32_t* pk = reinterpret_cast<uint32_t*>(c->pack_tmp.as<char>() + at_b[l]);
      const size_t groups = (H->pending_cnt[l] + 7) / 8;
      const int grid = int(std::min<size_t>((groups + 255) / 256, size_t(c->sm_count) * 8));
      cse_pack20_kernel<<<grid, 256, 0, c->stream>>>(H->emit_dev[H->pending_set][l], H->pending_cnt[l], pk);
      c->stats.gpu_launches++;
    }
    BCE_CUDA(c, cudaGetLastError());
  }
  BCE_CUDA(c, cudaEventRecord(c->ev[6], c->stream));            // everything computed so far ...
  BCE_CUDA(c, cudaStreamWaitEvent(cs, c->ev[6], 0));            // ... is visible to the copies
  BCE_CUDA(c, cudaEventRecord(c->ev[4], cs));
  for (int l = 0; l < 8; ++l) {
    out->words[l] = reinterpret_cast<const uint32_t*>(hp + at_b[l]);
    out->count[l] = H->pending_cnt[l];
    if (!H->pending_cnt[l]) continue;
    if (pack20)
      BCE_CUDA(c, cudaMemcpyAsync(hp + at_b[l], c->pack_tmp.as<char>() + at_b[l], (H->pending_cnt[l] * 5 + 1) / 2, cudaMemcpyDeviceToHost, cs));
    else
      BCE_CUDA(c, cudaMemcpyAsync(hp + at_b[l], H->emit_dev[H->pending_set][l], H->pending_cnt[l] * sizeof(uint32_t),
                                  cudaMemcpyDeviceToHost, cs));
  }
  BCE_CUDA(c, cudaEventRecord(c->ev[5], cs));
  const bool this_done = H->pending_done;
  H->pending = false;
  // ... and meanwhile compute the next one into the other set
  if (!this_done && H->sets == 2) {
    BCE_TRY(run_batch(c, H->fill_set, H->pending_cnt, &H->pending_done));
    H->pending = true;
    H->pending_set = H->fill_set;
    H->fill_set ^= 1;
  }
  BCE_CUDA(c, cudaEventSynchronize(c->ev[5]));
  float ms = 0;
  BCE_CUDA(c, cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]));
  c->stats.ms_d2h += ms;
  out->done = this_done ? 1 : 0;
  if (this_done) c->cse_done = true;
  return BCE_GPU_OK;
}

// `bce -s`: one batch of counts, bucketed on the device (include/bce_gpu.h, bce_gpu_cse_next_buckets).  The batch is
// computed, every stream's words are sorted stably by bucket with the suffix sorter's radix passes, symbols and the
// bucket table go to pinned memory.  No overlap with the next batch's kernels: the host's flush (bce.cpp:751-800,
// six simulated coders per symbol) is what `bce -s` waits for.
int cse_advance_buckets(Ctx* c, bce_scan_buckets* out) {
  if (!c->cse_active || !c->cse) { set_error(c, "cse_next_buckets without cse_begin"); return BCE_GPU_E_STATE; }
  CseHost* H = c->cse;
  memset(out, 0, sizeof *out);
  if (c->cse_done) { out->done = 1; return BCE_GPU_OK; }
  size_t cnt[8];
  bool done = false;
  BCE_TRY(run_batch(c, 0, cnt, &done));
  cudaStream_t st = c->stream;
  size_t maxcnt = 0, total = 0, bucket_cap[8], bucket_total = 0;
  for (int l = 0; l < 8; ++l) {
    if (cnt[l] > 0xFFFFFFF0ull) { set_error(c, "scan batch of %zu words", cnt[l]); return BCE_GPU_E_INTERNAL; }
    maxcnt = std::max(maxcnt, cnt[l]);
    total += (cnt[l] + 15) & ~size_t(15);
    bucket_cap[l] = std::min<size_t>(cnt[l], size_t(1) << 21);
    bucket_total += bucket_cap[l];
  }
  const size_t need = 2 * Carver::need(maxcnt, 8) + 2 * Carver::need(maxcnt, 4) + Carver::need(total, 1) +
                      Carver::need(bucket_total, sizeof(bce_scan_bucket)) + 4096;
  BCE_TRY(c->scan_tmp.ensure(c, need));
  Carver cv(c->scan_tmp.p, c->scan_tmp.cap);
  uint64_t* kA = cv.take<uint64_t>(maxcnt);
  uint64_t* kB = cv.take<uint64_t>(maxcnt);
  uint32_t* vA = cv.take<uint32_t>(maxcnt);
  uint32_t* vB = cv.take<uint32_t>(maxcnt);
  uint8_t* syms = cv.take<uint8_t>(total);
  bce_scan_bucket* buckets = cv.take<bce_scan_bucket>(bucket_total);
  struct Counters { unsigned long long halvings[8]; uint32_t nbuckets[8]; };
  Counters* d_cnt = reinterpret_cast<Counters*>(cv.take<unsigned char>(sizeof(Counters)));
  if (!cv.ok()) { set_error(c, "scan bucketing: scratch carve failed"); return BCE_GPU_E_NOMEM; }
  BCE_CUDA(c, cudaMemsetAsync(d_cnt, 0, sizeof(Counters), st));
  const int shifts[3] = {0, 8, 16};
  size_t sym_at[8], bucket_at[8], sa = 0, ba = 0;
  for (int l = 0; l < 8; ++l) {
    sym_at[l] = sa;
    bucket_at[l] = ba;
    sa += (cnt[l] + 15) & ~size_t(15);
    ba += bucket_cap[l];
    if (!cnt[l]) continue;
    const uint32_t m = uint32_t(cnt[l]);
    const int grid = int(std::min<size_t>((m + 255) / 256, size_t(c->sm_count) * 8));
    scan_keys_kernel<<<grid, 256, 0, st>>>(H->emit_dev[0][l], m, kA, vA, &d_cnt->halvings[l]);
    c->stats.gpu_launches++;
    BCE_CUDA(c, cudaGetLastError());
    uint64_t* ok = kA;
    uint32_t* ov = vA;
    int ran = 0;
    RadixHistSource stable;
    stable.stable_first = true;                          // insertion order inside a bucket is what flush() depends on
    BCE_TRY(radix_sort_pairs(c, kA, kB, vA, vB, m, shifts, 3, &ok, &ov, &ran, &stable));
    scan_compact_kernel<<<grid, 256, 0, st>>>(ok, ov, m, syms + sym_at[l], buckets + bucket_at[l], uint32_t(bucket_cap[l]),
                                              &d_cnt->nbuckets[l]);
    c->stats.gpu_launches++;
    BCE_CUDA(c, cudaGetLastError());
  }
  Counters* h_cnt = reinterpret_cast<Counters*>(c->pinned_small.as<char>() + 44 * 1024);
  BCE_CUDA(c, cudaMemcpyAsync(h_cnt, d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, st));
  BCE_CUDA(c, cudaStreamSynchronize(st));
  size_t pin_bytes = 64;
  for (int l = 0; l < 8; ++l) {
    if (h_cnt->nbuckets[l] > bucket_cap[l]) { set_error(c, "scan bucketing: %u buckets in stream %d", h_cnt->nbuckets[l], l); return BCE_GPU_E_INTERNAL; }
    pin_bytes += ((cnt[l] + 15) & ~size_t(15)) + size_t(h_cnt->nbuckets[l]) * sizeof(bce_scan_bucket);
  }
  PinnedBuf& pin = H->pinned_flip ? c->pinned_emit2 : c->pinned_emit;
  H->pinned_flip ^= 1;
  BCE_TRY(pin.ensure(c, pin_bytes));
  char* hp = pin.as<char>();
  size_t at = 0;
  BCE_CUDA(c, cudaEventRecord(c->ev[4], st));
  for (int l = 0; l < 8; ++l) {
    out->count[l] = cnt[l];
    out->nbuckets[l] = h_cnt->nbuckets[l];
    out->halvings[l] = h_cnt->halvings[l];
    out->syms[l] = reinterpret_cast<const uint8_t*>(hp + at);
    if (cnt[l]) BCE_CUDA(c, cudaMemcpyAsync(hp + at, syms + sym_at[l], cnt[l], cudaMemcpyDeviceToHost, st));
    at += (cnt[l] + 15) & ~size_t(15);
    out->buckets[l] = reinterpret_cast<const bce_scan_bucket*>(hp + at);
    const size_t bb = size_t(h_cnt->nbuckets[l]) * sizeof(bce_scan_bucket);
    if (bb) BCE_CUDA(c, cudaMemcpyAsync(hp + at, buckets + bucket_at[l], bb, cudaMemcpyDeviceToHost, st));
    at += bb;
  }
  BCE_CUDA(c, cudaEventRecord(c->ev[5], st));
  BCE_CUDA(c, cudaEventSynchronize(c->ev[5]));
  float ms = 0;
  BCE_CUDA(c, cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]));
  c->stats.ms_d2h += ms;
  out->done = done ? 1 : 0;
  if (done) c->cse_done = true;
  return BCE_GPU_OK;
}

}  // namespace bce
