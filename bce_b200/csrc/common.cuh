// common.cuh -- shared device/host helpers for libbce_gpu (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/bce_gpu.h"

namespace bce {

constexpr int kSMsB200 = 148;

// ---------------------------------------------------------------------------------
// host side: error plumbing and a grow-only device buffer
// ---------------------------------------------------------------------------------
struct Ctx;
void set_error(Ctx* c, const char* fmt, ...);
bool trace_on();
#define BCE_TRACE(...) do { if (bce::trace_on()) { fprintf(stderr, "[bce_gpu] " __VA_ARGS__); fputc('\n', stderr); fflush(stderr); } } while (0)

#define BCE_CUDA(ctx, call)                                                         \
  do {                                                                              \
    cudaError_t e__ = (call);                                                       \
    if (e__ != cudaSuccess) {                                                       \
      bce::set_error((ctx), "%s:%d %s -> %s", __FILE__, __LINE__, #call,            \
                     cudaGetErrorString(e__));                                      \
      return (e__ == cudaErrorMemoryAllocation) ? BCE_GPU_E_NOMEM : BCE_GPU_E_CUDA; \
    }                                                                               \
  } while (0)

#define BCE_TRY(expr)            \
  do {                           \
    int rc__ = (expr);           \
    if (rc__ != BCE_GPU_OK) return rc__; \
  } while (0)

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(Ctx* c, size_t bytes);   // grow-only; contents are not preserved on growth
  void release();
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinnedBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(Ctx* c, size_t bytes);
  void release();
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// carve aligned pieces out of one scratch allocation
struct Carver {
  char* base;
  size_t off = 0, cap;
  Carver(void* b, size_t c) : base(reinterpret_cast<char*>(b)), cap(c) {}
  template <class T> T* take(size_t count) {
    size_t bytes = (count * sizeof(T) + 255) & ~size_t(255);
    if (off + bytes > cap) { off = cap + 1; return nullptr; }
    T* r = reinterpret_cast<T*>(base + off);
    off += bytes;
    return r;
  }
  bool ok() const { return off <= cap; }
  static size_t need(size_t count, size_t elem) { return (count * elem + 255) & ~size_t(255); }
};

// ---------------------------------------------------------------------------------
// device side
// ---------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

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
// by at most 1 -- and corrected.  The range coders of code_many.cu and decode_many.cu share it.
__device__ __forceinline__ uint64_t div64(uint64_t x, uint32_t d) {
  const uint32_t xh = uint32_t(x >> 32), qh = xh / d;
  const uint64_t y = (uint64_t(xh - qh * d) << 32) | uint32_t(x);            // < d 2^32
  uint64_t ql = uint64_t(__dmul_rn(__ull2double_rn(y), rcp_nocall(double(d))));
  int64_t r = int64_t(y - ql * d);                                          // |r| < 3 d
  for (int t = 0; t < 3 && r < 0; ++t) { --ql; r += d; }
  for (int t = 0; t < 3 && r >= int64_t(d); ++t) { ++ql; r -= d; }
  return (uint64_t(qh) << 32) + ql;
}

__device__ __forceinline__ uint64_t bswap64(uint64_t v) {
  const uint32_t lo = uint32_t(v), hi = uint32_t(v >> 32);
  return (uint64_t(__byte_perm(lo, 0, 0x0123)) << 32) | __byte_perm(hi, 0, 0x0123);
}

// The suffix sort's round-0 key of rotation i: the 8 bytes T[i..i+8) big-endian, from two word loads and a funnel
// shift.  T64 is the text as words; it must be cyclic for 8 bytes past its end so that both words exist (the suffix
// sort pads 64, pad_cyclic_kernel).
__device__ __forceinline__ uint64_t window_key(const uint64_t* T64, uint32_t i) {
  const uint64_t a = bswap64(T64[i >> 3]), b = bswap64(T64[(i >> 3) + 1]);
  const uint32_t sh = (i & 7u) * 8;
  return sh ? (a << sh) | (b >> (64 - sh)) : a;
}

// The same window over a text of 7-bit symbol codes (the suffix sort's round 0 when at most 128 byte values occur):
// the low 7 bits of the 8 bytes packed into 56 bits in three steps -- byte pairs, then 16-bit halves of 32-bit
// words, then the two words -- so the key has 7 digits of 8 bits instead of 8 and keeps the order of the window.
__device__ __forceinline__ uint64_t pack_codes7(uint64_t w) {
  w = (((w >> 8) & 0x007F007F007F007Full) << 7) | (w & 0x007F007F007F007Full);
  w = (((w >> 16) & 0x00003FFF00003FFFull) << 14) | (w & 0x00003FFF00003FFFull);
  return ((w >> 32) << 28) | (w & 0x0FFFFFFFull);
}
__device__ __forceinline__ uint64_t window_key_bits(const uint64_t* T64, uint32_t i, bool codes7) {
  const uint64_t w = window_key(T64, i);
  return codes7 ? pack_codes7(w) : w;
}

// Tagged tile descriptors for single-pass chained scans (decoupled look-back).
// word = [ tag:30 | status:2 | value:32 ]; a word whose tag differs from the current
// pass/round tag is "not written yet", so the arrays never need clearing between passes.
constexpr uint32_t kDescAgg = 1, kDescPrefix = 2;
__device__ __forceinline__ uint64_t desc_pack(uint32_t tag, uint32_t status, uint32_t value) {
  return (uint64_t(tag & 0x3FFFFFFFu) << 34) | (uint64_t(status) << 32) | value;
}
__device__ __forceinline__ uint32_t desc_tag(uint64_t w) { return uint32_t(w >> 34); }
__device__ __forceinline__ uint32_t desc_status(uint64_t w) { return uint32_t(w >> 32) & 3u; }
__device__ __forceinline__ void desc_store(uint64_t* p, uint64_t v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t desc_load(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// Spin until the descriptor carries `tag`.  The budget bounds the wait so that a logic
// error surfaces as BCE_GPU_E_INTERNAL instead of a hung GPU.
constexpr uint32_t kSpinBudget = 1u << 18;
#ifndef BCE_SPIN_HOT
#define BCE_SPIN_HOT 64
#define BCE_SPIN_SLEEP 20
#endif
__device__ __forceinline__ uint64_t desc_wait(const uint64_t* p, uint32_t tag, uint32_t* err) {
  uint64_t w = desc_load(p);
  uint32_t spins = 0;
  while (desc_tag(w) != (tag & 0x3FFFFFFFu)) {
    if (++spins > kSpinBudget) {
      atomicExch(err, 1u);
      return desc_pack(tag, kDescPrefix, 0);
    }
    if (spins > BCE_SPIN_HOT) __nanosleep(BCE_SPIN_SLEEP);      // poll hot at first: the usual wait is one L2 round trip
    w = desc_load(p);
  }
  return w;
}

// Look-back by one thread (used where 256 threads each chase their own digit).  Descriptors
// of 8 predecessors are fetched per step so that a walk of depth d costs d/8 L2 round trips.
// Returns the exclusive prefix of `agg` over tiles [0, tile) and publishes the inclusive one.
__device__ __forceinline__ uint32_t lookback_serial(uint64_t* desc, uint32_t stride, uint32_t tile,
                                                    uint32_t tag, uint32_t agg, uint32_t* err) {
  if (tile == 0) {
    desc_store(desc, desc_pack(tag, kDescPrefix, agg));
    return 0;
  }
  desc_store(desc + size_t(tile) * stride, desc_pack(tag, kDescAgg, agg));
  #ifndef BCE_LB_BATCH
#define BCE_LB_BATCH 2
#endif
  constexpr int kBatch = BCE_LB_BATCH;
  uint32_t excl = 0;
  uint32_t t = tile;                      // next predecessor to look at is t - 1
  bool done = false;
  while (!done && t > 0) {
    uint64_t w[kBatch];
    const uint32_t nb = t < uint32_t(kBatch) ? t : uint32_t(kBatch);
#pragma unroll
    for (int k = 0; k < kBatch; ++k)
      if (uint32_t(k) < nb) w[k] = desc_load(desc + size_t(t - 1 - k) * stride);
#pragma unroll
    for (int k = 0; k < kBatch; ++k) {
      if (!done && uint32_t(k) < nb) {
        uint64_t v = w[k];
        if (desc_tag(v) != (tag & 0x3FFFFFFFu)) v = desc_wait(desc + size_t(t - 1 - k) * stride, tag, err);
        excl += uint32_t(v);
        if (desc_status(v) == kDescPrefix) done = true;
      }
    }
    t -= nb;
  }
  desc_store(desc + size_t(tile) * stride, desc_pack(tag, kDescPrefix, excl + agg));
  return excl;
}

// Warp-wide look-back over a chain of tiles [first, tile): all 32 lanes must call it.
// Returns (to every lane) the exclusive prefix and publishes the inclusive one.
__device__ __forceinline__ uint32_t lookback_warp(uint64_t* desc, uint32_t tile, uint32_t first,
                                                  uint32_t tag, uint32_t agg, uint32_t* err) {
  const unsigned lane = lane_id();
  if (tile == first) {
    if (lane == 0) desc_store(desc + tile, desc_pack(tag, kDescPrefix, agg));
    return 0;
  }
  if (lane == 0) desc_store(desc + tile, desc_pack(tag, kDescAgg, agg));
  uint32_t excl = 0;
  int64_t base = int64_t(tile) - 1;
  for (;;) {
    int64_t t = base - lane;
    bool inside = t >= int64_t(first);
    uint64_t w = inside ? desc_wait(desc + t, tag, err) : desc_pack(tag, kDescPrefix, 0);
    unsigned pm = __ballot_sync(0xffffffffu, desc_status(w) == kDescPrefix);
    uint32_t v = uint32_t(w);
    if (pm) {
      unsigned stop = __ffs(pm) - 1;           // nearest predecessor with a full prefix
      if (lane > stop) v = 0;
      excl += __reduce_add_sync(0xffffffffu, v);
      break;
    }
    excl += __reduce_add_sync(0xffffffffu, v);
    base -= 32;
  }
  if (lane == 0) desc_store(desc + tile, desc_pack(tag, kDescPrefix, excl + agg));
  return excl;
}

// Wide-window look-back, second half: the caller has published its aggregate (tile != first); walk
// the predecessors, return the exclusive prefix, publish the inclusive one.  Every lane fetches B
// predecessor descriptors per step (B independent loads in flight), so one step covers 32*B tiles.
// A persistent kernel runs gridDim tiles of the same phase at once; none of them has an inclusive
// prefix yet, so the walk has to get past all of them -- the window is what bounds the number of
// serial L2 round trips.
template <int B>
__device__ __forceinline__ uint32_t lookback_resolve_wide(uint64_t* desc, uint32_t tile, uint32_t first,
                                                          uint32_t tag, uint32_t agg, uint32_t* err) {
  const unsigned lane = lane_id();
  uint32_t excl = 0;
  int64_t base = int64_t(tile) - 1;
  for (;;) {
    uint64_t w[B];
#pragma unroll
    for (int k = 0; k < B; ++k) {
      const int64_t t = base - (k * 32 + int(lane));
      w[k] = t >= int64_t(first) ? desc_load(desc + t) : desc_pack(tag, kDescPrefix, 0);
    }
#pragma unroll
    for (int k = 0; k < B; ++k) {
      const int64_t t = base - (k * 32 + int(lane));
      if (t >= int64_t(first) && desc_tag(w[k]) != (tag & 0x3FFFFFFFu)) w[k] = desc_wait(desc + t, tag, err);
    }
    bool done = false;
#pragma unroll
    for (int k = 0; k < B; ++k) {
      if (!done) {
        const unsigned pm = __ballot_sync(0xffffffffu, desc_status(w[k]) == kDescPrefix);
        uint32_t v = uint32_t(w[k]);
        if (pm) {
          const unsigned stop = __ffs(pm) - 1;
          if (lane > stop) v = 0;
          done = true;
        }
        excl += __reduce_add_sync(0xffffffffu, v);
      }
    }
    if (done) break;
    base -= 32 * B;
  }
  if (lane == 0) desc_store(desc + tile, desc_pack(tag, kDescPrefix, excl + agg));
  return excl;
}

// Publish the aggregate, then resolve: the whole chained-scan step of one tile.
template <int B>
__device__ __forceinline__ uint32_t lookback_warp_wide(uint64_t* desc, uint32_t tile, uint32_t first,
                                                       uint32_t tag, uint32_t agg, uint32_t* err) {
  if (tile == first) {
    if (lane_id() == 0) desc_store(desc + tile, desc_pack(tag, kDescPrefix, agg));
    return 0;
  }
  if (lane_id() == 0) desc_store(desc + tile, desc_pack(tag, kDescAgg, agg));
  return lookback_resolve_wide<B>(desc, tile, first, tag, agg, err);
}

// The same for blocks of many warps in latency-bound kernels: the warp totals are scanned by shuffles in every warp
// (one shared load per lane instead of a walk over all of them), and a warp whose threads all hold zero -- `active`
// false, not the first warp -- only keeps the barriers company (its return value and `total` are then undefined).
template <class T, int THREADS>
__device__ __forceinline__ T block_exclusive_scan_sparse(T v, T* scratch, T& total, bool active) {
  constexpr int NW = THREADS / 32;
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  T inc = v;
  if (active) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      T o = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= unsigned(d)) inc += o;
    }
  }
  if (lane == 31) scratch[warp] = active ? inc : T(0);
  __syncthreads();
  T woff = 0;
  if (active) {
    T winc = lane < unsigned(NW) ? scratch[lane] : T(0);
#pragma unroll
    for (int d = 1; d < NW; d <<= 1) {
      T o = __shfl_up_sync(0xffffffffu, winc, d);
      if (lane >= unsigned(d)) winc += o;
    }
    total = __shfl_sync(0xffffffffu, winc, NW - 1);
    const T before = __shfl_sync(0xffffffffu, winc, warp ? warp - 1 : 0);
    woff = warp ? before : T(0);
  }
  __syncthreads();          // scratch may be reused right after
  return woff + inc - v;
}

// Block-wide exclusive scan of one value per thread (THREADS multiple of 32, <= 1024).
// `total` receives the block sum.  Uses (THREADS/32) words of shared scratch.
template <class T, int THREADS>
__device__ __forceinline__ T block_exclusive_scan(T v, T* scratch, T& total) {
  constexpr int NW = THREADS / 32;
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  T inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    T o = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= unsigned(d)) inc += o;
  }
  if (lane == 31) scratch[warp] = inc;
  __syncthreads();
  T woff = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < NW; ++w) {
    T s = scratch[w];
    if (unsigned(w) < warp) woff += s;
    tot += s;
  }
  __syncthreads();          // scratch may be reused right after
  total = tot;
  return woff + inc - v;
}

#endif  // __CUDACC__

}  // namespace bce
