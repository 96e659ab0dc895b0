// decode_many.cu -- the whole decoder of many small archives on the device (bce_gpu_decompress_many).
//
// The host decoder (csrc/host/decode.cpp: decode_to_ranks, decode_levels, decode_node, DecodeRank; coders.cpp:
// StreamDecoder, RangeDecoder, ContextModel) restated, check for check, so that an archive decodes -- or is rejected --
// exactly as `bce -ds` decodes it, damaged archives included:
//   shape      a persistent grid; one CTA of 8 warps per archive, taken largest first from an atomic counter.  Warp w
//              owns level w: stream w's range decoder, its model and its rank dictionary; warp 0 first reads the header.
//   decoder    warp-uniform lo / hi / code; a read past the end of a stream gives 0.  The adaptive step needs no serial
//              search: lane j holds counter j of the row, and with step = (hi - lo) / total and c_j = sum_{i <= j}
//              (row[i] + 1) (a warp scan), top_j = lo - 1 + step c_j is what the host's loop holds after j iterations;
//              the symbol is the first j < k with !(top_j < code), else k - 1.  A uniform step divides by a 64-bit step:
//              code - lo >= step range gives the host's clamp to range - 1, else the quotient (< range) is estimated in
//              double precision and corrected.  A count with k > 31 is the host's recursion unrolled.
//   model      one table per warp in global memory, the host's layout (the two sum bytes of a row are not used: the sum
//              is a warp reduction), sized by the stream's own config row and zeroed per archive.
//   dictionary the 8 levels' DecodeRank words in dynamic shared memory (2n + 64 bytes per level set), written to the
//              inverse's layout after DecodeRank::finish.
//   rounds     decode_levels: per round, warp w runs level w's zero-half, then its one-half, in order; children go to
//              level (w + 1) % 8's lists for the next round; one __syncthreads ends a round.
//   frontier   lists of chunks of 32 nodes in global memory, one pool per CTA.  The host rejects an archive once its
//              visits exceed 8n (checked per round), so a round that would exceed what is left is refused before it runs,
//              and the nodes of one round and of the next never exceed 8n together.  The pool holds 8n nodes plus one
//              partial chunk per list and side: round r takes chunks from one end of the pool and round r + 1 from the
//              other, and running out of chunks proves the next round over budget.  Damaged archives can hold
//              overlapping nodes, so no bound from disjoint intervals is used.
// Every loop is bounded (the visit budget, at most 4 shifts per renormalisation, at most 32 halvings) and no CTA waits
// for another, so a logic error shows as a status, never as a hang.  The inverse (unbwt_many_kernel) then runs on the
// dictionaries where they are and skips the rejected archives.
#include <algorithm>
#include <numeric>
#include <vector>

#include "ctx.h"

namespace bce {

constexpr int DM_THREADS = 256;
constexpr uint32_t kFullMask = 0xffffffffu;
constexpr uint32_t kChunk = 32;                      // nodes per frontier chunk: one per lane
constexpr uint32_t kNoChunk = 0xffffffffu;
// largest model table of a stream: every k of 2 .. 31 at 5 context bits, (k + 2) << 10 bytes each
constexpr size_t kDmTableMax = 555u << 10;
// slots (tables and frontier pools) of one call, beyond one CTA per SM
constexpr size_t kDmSlotBudget = size_t(1) << 30;

struct DmArgs {
  const uint16_t* words;                             // every archive back to back
  const unsigned long long* starts;                  // k + 1
  const uint32_t* n;                                 // what each header must claim
  const uint32_t* order;                             // archive taken by job j (largest first)
  uint32_t k;
  UmDict* dict;                                      // words / out / n filled by the host; offset by the decoder
  uint64_t* ranks;                                   // the dictionaries, unbwt_many's layout
  int* status;
  uint32_t* next_job;
  unsigned long long* visits;                        // of accepted archives
  unsigned long long* rounds;
  char* slots;
  size_t slot_bytes, pool_offset;                    // per CTA: 8 tables of kDmTableMax, then the pool
  uint32_t pool_chunks;                              // chunks per pool
};

// RangeDecoder (coders.cpp) with warp-uniform state
struct WarpDecoder {
  const uint16_t* w;
  uint32_t count, pos;
  uint64_t lo, hi, code;

  __device__ __forceinline__ uint32_t next() { return pos < count ? uint32_t(w[pos++]) : 0u; }
  __device__ __forceinline__ void init(const uint16_t* words, uint32_t cnt) {
    w = words; count = cnt; pos = 0; lo = 0; hi = ~0ull; code = 0;
    for (int i = 0; i < 4; ++i) code = (code << 16) | next();
  }
  __device__ __forceinline__ void renormalise() {    // at most 4 shifts, as in the encoder
    for (int t = 0; t < 4 && ((hi ^ lo) >> 48) == 0; ++t) {
      code = (code << 16) + next();
      lo <<= 16;
      hi = (hi << 16) | 0xFFFFu;
    }
  }
  __device__ __forceinline__ void restart_if_narrow(uint64_t total) {
    if (hi - lo < total) {
      for (int i = 0; i < 4; ++i) code = (code << 16) + next();
      lo = 0;
      hi = ~0ull;
    }
  }
  __device__ __forceinline__ uint32_t get_uniform(uint32_t range) {
    restart_if_narrow(range);
    const uint64_t step = div64(hi - lo, range), d = code - lo;
    uint64_t q;
    if (d >= step * range) {                         // the host's clamp (only a damaged stream gets here)
      q = range - 1;
    } else {                                         // q < range <= 2^31: off by at most one after the estimate
      q = uint64_t(__dmul_rn(__ull2double_rn(d), rcp_nocall(__ull2double_rn(step))));
      if (q > range - 1) q = range - 1;
      for (int t = 0; t < 3 && q * step > d; ++t) --q;
      for (int t = 0; t < 3 && (q + 1) * step <= d; ++t) ++q;
    }
    lo += step * q;
    hi = lo + step - 1;
    renormalise();
    return uint32_t(q);
  }
  // RangeDecoder::get with lane j holding row[j] (0 at and beyond k)
  __device__ __forceinline__ uint32_t get(uint32_t c, uint32_t k, uint32_t total, uint32_t lane) {
    restart_if_narrow(total);
    const uint64_t step = div64(hi - lo, total);
    uint32_t cj = lane < k ? c + 1 : 0u;             // inclusive scan of row[i] + 1
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t v = __shfl_up_sync(kFullMask, cj, d);
      if (lane >= uint32_t(d)) cj += v;
    }
    const uint64_t top = lo - 1 + step * cj;
    const uint32_t hit = __ballot_sync(kFullMask, lane < k && !(top < code));
    const uint32_t sym = hit ? uint32_t(__ffs(hit)) - 1 : k - 1;
    const uint64_t top_s = __shfl_sync(kFullMask, top, sym);
    const uint64_t below = __shfl_sync(kFullMask, top, sym ? sym - 1 : 0);
    lo = sym ? below + 1 : lo;
    hi = top_s;
    renormalise();
    return sym;
  }
  __device__ __forceinline__ uint32_t varint() {     // StreamDecoder::varint
    uint32_t v = 0;
    for (int i = 0; i < 31; ++i) {
      const uint32_t d = get_uniform(3);
      if (d == 2) break;
      v |= d << i;
    }
    return v;
  }
  // StreamDecoder's constructor: the config row -> ContextModel::configure's offsets (off[k] | bits << 24), table bytes
  __device__ __forceinline__ uint32_t config(uint32_t* off) {
    uint32_t last = 0, start = 0;
    for (uint32_t j = 0; j < 32; ++j) {
      const uint32_t b = get_uniform(2) ? get_uniform(6) : last;
      last = b;
      if (j >= 2) {
        if (off) off[j] = start | (b << 24);
        start += (j + 2) << (b * 2);
      }
    }
    return start;
  }
};

// x86 SHL: the count is taken mod 64 (decode.cpp, shl_x86)
__device__ __forceinline__ uint64_t shl_x86(uint64_t v, uint64_t count) { return v << (count & 63u); }

// DecodeRank over shared words R[0 .. n / 32]
__device__ __forceinline__ uint32_t ones_before(const uint64_t* R, uint32_t n, uint32_t pos) {
  if (pos > n) pos = n;
  const uint64_t w = R[pos / 32];
  const uint32_t below = uint32_t(w >> 32) & uint32_t((1ull << (pos % 32)) - 1);
  return uint32_t(w) + uint32_t(__popc(below));
}
__device__ __forceinline__ void pin(uint64_t* R, uint32_t n, uint32_t pos, uint32_t ones, bool writer) {
  if (pos > n) return;
  uint64_t need = uint32_t(ones - ones_before(R, n, pos));
  if (need == 0) return;
  const uint64_t word = pos / 32, o = pos % 32;
  uint64_t b = R[word];
  const uint32_t base = uint32_t(b);
  if (uint64_t(base) + o + 32 < need) {
    b += need - o - base;
    need = o;
  }
  const uint64_t above = ~0ull << (32 + o);
  const uint64_t take_at = uint64_t(__ffsll((long long)(((b & above) >> 32) | (1ull << 31))) - 1);
  const uint64_t put_end = 64 - uint64_t(__clzll((long long)~(b | above)));     // __clzll(0) = 64
  const uint64_t take = (shl_x86(1, take_at + need) - shl_x86(1, take_at)) << 32;
  const uint64_t put = shl_x86(1, put_end) - shl_x86(1, put_end - need);
  b += uint64_t(__popc(uint32_t(put)));
  b &= ~take;
  b |= (put >> 32) << 32;
  __syncwarp();                                      // every lane has read the word before lane 0 rewrites it
  if (writer) R[word] = b;
  __syncwarp();
}

struct DmShared {
  uint32_t job, bad, hdr_ok, offset;
  unsigned long long at[9];
  uint32_t C[8];
  uint32_t used[3];                                  // chunks taken by round r in used[r % 3], from end r % 2
  uint32_t head[2][8][2], count[2][8][2];            // [round parity][level][half]
};

// node = s (24 bits) | x0 (20 bits) | x1 (20 bits): s <= 2n, x0 and x1 <= n
__device__ __forceinline__ uint64_t pack_node(uint32_t s, uint32_t x0, uint32_t x1) {
  return uint64_t(s) | (uint64_t(x0) << 24) | (uint64_t(x1) << 44);
}

// One list being written (warp-uniform): its chunks are linked through link[].
struct ListOut {
  uint32_t head, tail, count;
};

__global__ void __launch_bounds__(DM_THREADS, 3) decode_many_kernel(DmArgs a) {
  extern __shared__ __align__(16) uint64_t dict_sh[];
  __shared__ DmShared sh;
  __shared__ uint32_t s_off[8][32];
  const uint32_t tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const bool writer = lane == 0;
  char* slot = a.slots + size_t(blockIdx.x) * a.slot_bytes;
  uint8_t* const table = reinterpret_cast<uint8_t*>(slot + size_t(w) * kDmTableMax);
  uint64_t* const pool = reinterpret_cast<uint64_t*>(slot + a.pool_offset);
  uint32_t* const link = reinterpret_cast<uint32_t*>(pool + size_t(a.pool_chunks) * kChunk);
  const uint32_t P = a.pool_chunks;

  for (;;) {
    if (tid == 0) sh.job = atomicAdd(a.next_job, 1u);
    __syncthreads();
    const uint32_t job = sh.job;
    if (job >= a.k) break;
    const uint32_t id = a.order[job];
    const uint32_t n = a.n[id], wpl = n / 32 + 1;
    const uint16_t* const A = a.words + a.starts[id];
    const uint64_t len = a.starts[id + 1] - a.starts[id];
    for (uint32_t i = tid; i < 8 * wpl; i += DM_THREADS) dict_sh[i] = 0;
    if (tid == 0) { sh.bad = 0; sh.hdr_ok = 0; sh.used[0] = sh.used[1] = sh.used[2] = 0; }

    // ---- header (decode_to_ranks), warp 0 ---------------------------------------------------------------------
    if (w == 0) {
      bool ok = len != 0;
      uint32_t hw = 0;
      if (ok) { hw = A[0]; ok = 1 + uint64_t(hw) <= len; }
      if (ok) {
        WarpDecoder h;
        h.init(A + 1, hw);
        h.config(nullptr);
        const uint32_t nh = h.varint();
        ok = nh != 0 && nh == n;
        uint32_t offset = 0, size = 0;
        if (ok) { offset = h.get_uniform(n + 1); ok = offset <= n; }
        if (ok) size = h.varint();
        uint64_t at = 1 + uint64_t(hw);
        if (writer) sh.at[0] = at;
        for (int i = 0; i < 7 && ok; ++i) {
          const uint32_t l = h.get_uniform(size + 1);
          if (l > size) { ok = false; break; }
          at += l;
          size -= l;
          if (at > len) ok = false;                  // at[i + 1] > len (it never decreases)
          if (writer) sh.at[i + 1] = at;
        }
        if (ok && len < at) ok = false;              // at[8] = len < at[7]
        if (writer) { sh.at[8] = len; sh.offset = offset; sh.hdr_ok = ok; }
      }
    }
    __syncthreads();
    if (!sh.hdr_ok) {
      if (tid == 0) a.status[id] = BCE_GPU_E_ARG;
      __syncthreads();
      continue;
    }

    // ---- stream w: config row, table, C[w] --------------------------------------------------------------------
    WarpDecoder dec;
    dec.init(A + sh.at[w], uint32_t(sh.at[w + 1] - sh.at[w]));
    const uint32_t tbytes = dec.config(s_off[w]);
    {
      uint4* t4 = reinterpret_cast<uint4*>(table);
#pragma unroll 1
      for (uint32_t i = lane; i < (tbytes + 15) / 16; i += 32) t4[i] = make_uint4(0, 0, 0, 0);
    }
    {
      const uint32_t c = dec.get_uniform(n + 1);
      if (writer) { sh.C[w] = c; if (c > n) atomicOr(&sh.bad, 1u); }
    }
    __syncthreads();
    if (sh.bad) {
      if (tid == 0) a.status[id] = BCE_GPU_E_ARG;
      __syncthreads();
      continue;
    }
    uint64_t* const R = dict_sh + size_t(w) * wpl;
    pin(R, n, n, n - sh.C[(w + 1) & 7], writer);    // ranks[(i + 7) % 8].pin(n, n - C[i])
    const uint32_t one_base = sh.C[(w + 1) & 7];
    // round 0's lists are "written by round -1": parity 1, counter used[2], the high end of the pool
    if (writer) {
      const uint32_t c = sh.C[w];
      sh.count[1][w][1] = 0;
      sh.head[1][w][1] = kNoChunk;
      if (c && n - c) {
        const uint32_t ch = P - 1 - atomicAdd(&sh.used[2], 1u);
        pool[size_t(ch) * kChunk] = pack_node(0, c, n - c);
        sh.head[1][w][0] = ch;
        sh.count[1][w][0] = 1;
      } else {
        sh.head[1][w][0] = kNoChunk;
        sh.count[1][w][0] = 0;
      }
    }
    __syncthreads();

    // ---- decode_levels ------------------------------------------------------------------------------------------
    const uint64_t budget = 8ull * n;
    uint64_t visits = 0;
    uint32_t rounds = 0;
    bool accepted = false;
    const uint32_t d = (w + 1) & 7;                  // where this level's children go
    for (uint32_t r = 0, r3 = 0;; ++r, r3 = r3 == 2 ? 0 : r3 + 1) {   // every round visits >= 1 node of the budget
      const uint32_t cp = (r + 1) & 1, np = r & 1;   // lists read / written this round; chunks taken from end np
      uint64_t total = 0;
      for (int i = 0; i < 16; ++i) total += sh.count[cp][i >> 1][i & 1];
      if (total == 0) { accepted = true; break; }
      if (visits + total > budget) break;            // the host would reject after this round
      visits += total;
      ++rounds;
      const uint32_t other = sh.used[r3 ? r3 - 1 : 2];   // chunks the lists being read hold (round r - 1's)
      if (tid == 0) sh.used[r3 == 2 ? 0 : r3 + 1] = 0;  // round r + 1's counter: round r - 2's, read by nobody now
      ListOut out0{kNoChunk, kNoChunk, 0}, out1{kNoChunk, kNoChunk, 0};   // the zero-half and one-half children
      bool fail = false;
      auto push = [&](ListOut& L, uint64_t node) -> bool {
        const uint32_t at = L.count % kChunk;
        if (at == 0) {                               // a new chunk from end np
          uint32_t got = 0;
          if (writer) got = atomicAdd(&sh.used[r3], 1u);
          got = __shfl_sync(kFullMask, got, 0);
          if (uint64_t(got) + 1 + other > P) return false;   // the next round exceeds the budget: see the header
          const uint32_t ch = np ? P - 1 - got : got;
          if (L.tail == kNoChunk) L.head = ch;
          else if (writer) link[L.tail] = ch;
          L.tail = ch;
        }
        if (writer) pool[size_t(L.tail) * kChunk + at] = node;
        ++L.count;
        return true;
      };
      for (int half = 0; half < 2 && !fail; ++half) {
        const uint32_t cnt = sh.count[cp][w][half];
        uint32_t chunk = sh.head[cp][w][half];
        uint64_t mine = 0;
#pragma unroll 1
        for (uint32_t j = 0; j < cnt; ++j) {
          const uint32_t at = j % kChunk;
          if (at == 0) {
            if (j) chunk = link[chunk];
            mine = j + lane < cnt ? pool[size_t(chunk) * kChunk + lane] : 0ull;
          }
          const uint64_t nd = __shfl_sync(kFullMask, mine, at);
          const uint32_t s = uint32_t(nd) & 0xFFFFFFu, x0 = uint32_t(nd >> 24) & 0xFFFFFu, x1 = uint32_t(nd >> 44);
          // ---- decode_node ----
          const uint32_t x = x0 + x1;
          if (!x0 || !x1 || uint64_t(s) + x0 + x1 > n) { fail = true; break; }
          const uint32_t s1 = ones_before(R, n, s);
          const uint32_t c1 = ones_before(R, n, s + x) - s1;
          if (s1 > s || c1 > x) { fail = true; break; }
          const uint32_t s0 = s - s1;
          if (c1 == 0) {
            if (!push(out0, pack_node(s0, x0, x1))) { fail = true; break; }
            pin(R, n, s + x0, s1, writer);
            continue;
          }
          const uint32_t c0 = x - c1;
          if (c0 == 0) {
            if (!push(out1, pack_node(one_base + s1, x0, x1))) { fail = true; break; }
            pin(R, n, s + x0, s1 + x0, writer);
            continue;
          }
          const uint32_t zlo = x0 > c1 ? x0 - c1 : 0u;
          const uint32_t zhi = x0 - (c1 > x1 ? c1 - x1 : 0u);
          if (zhi < zlo) { fail = true; break; }
          uint32_t z0 = zlo;
          if (zhi != zlo) {                          // StreamDecoder::count(zhi - zlo + 1, c0, x1, x)
            uint32_t k = zhi - zlo + 1, lows = 0, nb = 0;
            for (; k > 31u && nb < 32; ++nb) {
              const uint32_t low = dec.get_uniform(2);
              lows |= low << nb;
              k = (k + (~low & 1u)) >> 1;
            }
            const uint32_t o = s_off[w][k], b = o >> 24;
            const uint32_t ctx = (((c0 << b) / x) << b) | ((x1 << b) / x);
            uint8_t* row = table + (o & 0x00FFFFFFu) + size_t(ctx) * (k + 2);
            const uint32_t c = lane < k ? uint32_t(row[lane]) : 0u;
            const uint32_t tot = k + __reduce_add_sync(kFullMask, c);
            const uint32_t sym = dec.get(c, k, tot, lane);
            const uint32_t freq = __shfl_sync(kFullMask, c, sym) + 1;
            if (freq == 0xFF) {                      // ContextModel::bump: every counter halves
              if (lane < k) row[lane] = uint8_t((c + (lane == sym)) >> 1);
            } else if (lane == sym) {
              row[lane] = uint8_t(freq);
            }
            __syncwarp();
            z0 = zlo + ((sym << nb) | lows);
          }
          if (z0 > zhi || z0 > c0) { fail = true; break; }
          const uint32_t z1 = c0 - z0;
          if (z0 && z1 && !push(out0, pack_node(s0, z0, z1))) { fail = true; break; }
          if (z1 > x1 || x1 - z1 > c1) { fail = true; break; }
          const uint32_t o1 = x1 - z1, o0 = c1 - o1;
          if (o0 && o1 && !push(out1, pack_node(one_base + s1, o0, o1))) { fail = true; break; }
          pin(R, n, s + x0, s1 + o0, writer);
        }
      }
      if (writer) {
        if (fail) atomicOr(&sh.bad, 1u);
        sh.head[np][d][0] = out0.head;
        sh.count[np][d][0] = out0.count;
        sh.head[np][d][1] = out1.head;
        sh.count[np][d][1] = out1.count;
      }
      __syncthreads();                               // the round's end: every level's lists and words are written
      if (sh.bad) break;
    }

    // ---- DecodeRank::finish, the dictionary to device memory -------------------------------------------------------
    const UmDict& dd = a.dict[id];
    if (accepted) {
      uint64_t* const G = a.ranks + dd.words;
      for (uint32_t i = tid; i < 8 * wpl; i += DM_THREADS) {
        const uint32_t l = i / wpl, j = i - l * wpl;
        uint64_t v = dict_sh[i];
        if (j + 1 < wpl) {
          const uint32_t here = uint32_t(v) + uint32_t(__popcll(v >> 32));
          const uint32_t nxt = uint32_t(dict_sh[size_t(l) * wpl + j + 1]);
          v |= uint64_t(uint32_t(nxt - here)) << 63;
        }
        G[i] = v;
      }
    }
    if (tid == 0) {
      if (accepted) {
        a.dict[id].offset = sh.offset;
        atomicAdd(a.visits, (unsigned long long)visits);
        atomicAdd(a.rounds, (unsigned long long)rounds);
      } else {
        a.status[id] = BCE_GPU_E_ARG;
      }
    }
    __syncthreads();                                 // shared words and lists free for the next archive
  }
}

int decode_many_run(Ctx* c, const uint16_t* words, const uint64_t* starts, const uint32_t* n, uint32_t k,
                    uint8_t* out, int* status) {
  cudaStream_t st = c->stream;
  const uint64_t w0 = starts[0], nw = starts[k] - starts[0];
  std::vector<unsigned long long> rel(k + 1);
  std::vector<UmDict> dict(k);
  std::vector<uint32_t> order(k);
  uint32_t N = 0;
  unsigned long long rwords = 0, bytes = 0;
  for (uint32_t i = 0; i < k; ++i) {
    rel[i] = starts[i] - w0;
    dict[i] = UmDict{rwords, bytes, n[i], 0};
    rwords += 8ull * (n[i] / 32 + 1);
    bytes += n[i];
    N = std::max(N, n[i]);
  }
  rel[k] = nw;
  std::iota(order.begin(), order.end(), 0u);
  std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return n[x] > n[y]; });

  const size_t smem = size_t(8) * (N / 32 + 1) * 8;
  BCE_CUDA(c, cudaFuncSetAttribute(decode_many_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  int occ = 0;
  BCE_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, decode_many_kernel, DM_THREADS, smem));
  if (occ < 1) { set_error(c, "decompress_many: %zu bytes of shared memory per CTA do not fit an SM", smem); return BCE_GPU_E_INTERNAL; }

  auto al = [](size_t b) { return (b + 255) & ~size_t(255); };
  DmArgs a;
  memset(&a, 0, sizeof a);
  a.pool_chunks = uint32_t((8ull * N + kChunk - 1) / kChunk + 40);   // 8N nodes + one partial chunk per list and end
  a.pool_offset = 8 * kDmTableMax;
  a.slot_bytes = al(a.pool_offset + size_t(a.pool_chunks) * (kChunk * 8 + 4));
  const size_t fixed = al(nw * 2) + al(size_t(k + 1) * 8) + 2 * al(size_t(k) * 4) + al(size_t(k) * sizeof(UmDict)) +
                       al(size_t(k) * 4) + 256 + al(rwords * 8) + al(bytes);
  size_t ctas = std::min<size_t>(k, size_t(c->sm_count) * occ);
  ctas = std::min(ctas, std::max<size_t>(c->sm_count, kDmSlotBudget / a.slot_bytes));
  ctas = std::max<size_t>(1, std::min(ctas, (scratch_budget(c) > fixed ? scratch_budget(c) - fixed : 0) / a.slot_bytes));
  const size_t need = fixed + ctas * a.slot_bytes;
  if (need > scratch_budget(c)) { set_error(c, "decompress_many: %zu bytes of scratch needed", need); return BCE_GPU_E_NOMEM; }
  BCE_TRY(c->scratch.ensure(c, need));
  char* p = c->scratch.as<char>();
  auto take = [&](size_t b) { char* q = p; p += al(b); return q; };
  auto* d_words = reinterpret_cast<uint16_t*>(take(nw * 2));
  auto* d_starts = reinterpret_cast<unsigned long long*>(take(size_t(k + 1) * 8));
  auto* d_n = reinterpret_cast<uint32_t*>(take(size_t(k) * 4));
  auto* d_order = reinterpret_cast<uint32_t*>(take(size_t(k) * 4));
  auto* d_dict = reinterpret_cast<UmDict*>(take(size_t(k) * sizeof(UmDict)));
  auto* d_status = reinterpret_cast<int*>(take(size_t(k) * 4));
  auto* d_ctr = reinterpret_cast<unsigned long long*>(take(256));   // [0] decode jobs | [1] unbwt jobs, serial | visits | rounds
  auto* d_ranks = reinterpret_cast<uint64_t*>(take(rwords * 8));
  auto* d_out = reinterpret_cast<uint8_t*>(take(bytes));
  char* d_slots = p;

  cudaEvent_t e0 = c->ev[4], e1 = c->ev[5], e2 = c->ev[6], e3 = c->ev[7];
  float ms = 0;
  BCE_CUDA(c, cudaEventRecord(e0, st));
  if (nw) BCE_TRY(h2d(c, d_words, words + w0, nw * 2));
  BCE_TRY(h2d(c, d_starts, rel.data(), size_t(k + 1) * 8));
  BCE_TRY(h2d(c, d_n, n, size_t(k) * 4));
  BCE_TRY(h2d(c, d_order, order.data(), size_t(k) * 4));
  BCE_TRY(h2d(c, d_dict, dict.data(), size_t(k) * sizeof(UmDict)));
  BCE_CUDA(c, cudaEventRecord(e1, st));
  BCE_CUDA(c, cudaMemsetAsync(d_status, 0, size_t(k) * 4, st));
  BCE_CUDA(c, cudaMemsetAsync(d_ctr, 0, 256, st));

  a.words = d_words;
  a.starts = d_starts;
  a.n = d_n;
  a.order = d_order;
  a.k = k;
  a.dict = d_dict;
  a.ranks = d_ranks;
  a.status = d_status;
  a.next_job = reinterpret_cast<uint32_t*>(d_ctr);
  a.visits = d_ctr + 2;
  a.rounds = d_ctr + 3;
  a.slots = d_slots;
  BCE_TRACE("decompress_many k=%u largest=%u ctas=%zu (%d per SM) smem=%zu B slot=%zu B", k, N, ctas, occ, smem,
            a.slot_bytes);
  BCE_CUDA(c, cudaEventRecord(e2, st));
  decode_many_kernel<<<unsigned(ctas), DM_THREADS, smem, st>>>(a);
  c->stats.gpu_launches++;
  BCE_CUDA(c, cudaGetLastError());
  BCE_CUDA(c, cudaEventRecord(e3, st));
  BCE_CUDA(c, cudaEventSynchronize(e3));
  BCE_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
  c->stats.ms_h2d += ms;
  BCE_CUDA(c, cudaEventElapsedTime(&ms, e2, e3));
  c->stats.ms_decoder += ms;

  auto* u_ctr = reinterpret_cast<uint32_t*>(d_ctr + 1);
  BCE_CUDA(c, cudaEventRecord(e0, st));
  BCE_TRY(unbwt_many_launch(c, d_ranks, d_dict, d_order, d_status, k, N, u_ctr, d_out));
  BCE_CUDA(c, cudaEventRecord(e1, st));
  BCE_CUDA(c, cudaEventSynchronize(e1));
  BCE_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
  c->stats.ms_unbwt_chase += ms;

  unsigned long long ctr[4] = {0, 0, 0, 0};
  BCE_CUDA(c, cudaEventRecord(e0, st));
  BCE_TRY(d2h(c, ctr, d_ctr, sizeof ctr));
  BCE_TRY(d2h(c, status, d_status, size_t(k) * 4));
  BCE_TRY(d2h(c, out, d_out, bytes));
  BCE_CUDA(c, cudaEventRecord(e1, st));
  BCE_CUDA(c, cudaEventSynchronize(e1));
  BCE_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
  c->stats.ms_d2h += ms;
  uint32_t accepted = 0;
  for (uint32_t i = 0; i < k; ++i) {
    if (status[i]) memset(out + dict[i].out, 0, n[i]);        // a rejected archive's text is left zero
    else ++accepted;
  }
  c->stats.unbwt_dicts = accepted;
  c->stats.unbwt_serial = uint32_t(ctr[1] >> 32);
  c->stats.cse_visits = ctr[2];
  c->stats.cse_rounds = ctr[3];
  c->stats.ms_total = c->stats.ms_h2d + c->stats.ms_decoder + c->stats.ms_unbwt_chase + c->stats.ms_d2h;
  return BCE_GPU_OK;
}

}  // namespace bce
