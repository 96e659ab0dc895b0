// code_many.cu -- the range coders of many small inputs on the device (bce_gpu_compress_many_archives).
//
// many_kernel (many.cu) leaves every input's CODER words in its arena and a directory of where they are.  A second
// launch turns them into finished archives, so that only the archives cross PCIe:
//   shape     a persistent grid; one CTA of 8 warps per input, taken largest first from an atomic counter; warp w codes
//             stream w (the level many_kernel's warp w ran), then warp 0 codes the header
//   coder     the range encoder, word fields and model layout of format.h, which the host's StreamEncoder
//             (csrc/host/coders.cpp) codes with too: all 32 lanes keep the same 64-bit range and lane 0 writes the
//             output words; lane j holds counter j of the current row, so the cumulative frequency and the total are
//             two warp reductions and the halving is one store per lane
//   model     one table per warp in global memory, format.h's layout (a row: k byte counters, then two bytes the host
//             keeps the row's sum in -- here the sum comes from the reduction and those bytes are not used), zeroed
//             before each input
//   output    the input's archive -- [header length][header][stream 0 .. 7], ArchiveWriter::finish -- is reserved in the
//             call's archive arena with one atomicAdd and copied there.  An archive that does not fit is left "not
//             done" and no CTA takes another input, as in many_kernel.
//
// Staging bound.  Let phi = log2(hi - lo + 1) <= 64.  A coding step of frequency f out of total t lowers phi by at most
// log2(t / f) + 2 (step = floor((hi - lo) / t) >= (hi - lo) / 2t once hi - lo >= t); a renormalised word raises it by 16;
// a restart (4 words) happens only at phi <= log2 t, t <= 65537, and raises phi to 64, by more than 47.  So a stream
// writes at most 4/47 of the phi it loses, plus the finish word.  Per stream that loss is at most 32 x 3 + 32 x 4.59
// (config prefix) + 18.01 (C) < 261, plus per count 15 (adaptive step: t <= 31 + 31 x 254) and 3 per uniform bit of
// a k > 31 count; a stream has at most n counts.  The header (row 8 prefix, varints and uniforms of totals below 2^23)
// needs fewer than 60 words.  Staging beyond these bounds sets an error and is never written.
#include <algorithm>
#include <vector>

#include "ctx.h"

namespace bce {

constexpr int CM_THREADS = 256;
constexpr uint32_t kHeaderCap = 96;
constexpr uint32_t kFull = 0xffffffffu;
enum : uint32_t { kCodeErrStage = 4, kCodeErrWord = 8 };

// staging words one stream of an input of n bytes can need (bound above)
static uint32_t stream_bound(uint32_t n) {
  uint32_t nb = 0;                                                  // uniform bits of a k > 31 count: k <= n halves
  for (uint32_t k = n; k > 31; k = (k + 1) / 2) ++nb;               // to at most (k + 1) / 2 each time
  return uint32_t((4ull * (261 + (15ull + 3 * nb) * n) + 46) / 47) + 1;
}

struct CodeEntry {                  // per-input result directory (device; copied to the host after the launch)
  uint32_t done, err, nwords, rounds;
  unsigned long long start;         // first uint16 of the archive in the arena
  unsigned long long visits, words;
};

struct CodeArgs {
  const ManyEntry* dir;
  const unsigned long long* starts;
  const uint32_t* order;
  const uint32_t* arena;            // many_kernel's words
  uint32_t k;
  uint8_t cfg[9][32];
  uint32_t off[8][32];              // model_layout's offsets per (stream, k), context bits masked off
  uint32_t tbytes[8];               // table bytes per stream
  char* slots;
  size_t slot_bytes, table_stride;
  uint32_t stage_cap;               // uint16 words per stream
  uint16_t* out;
  unsigned long long out_cap;       // uint16 words
  unsigned long long* out_used;
  uint32_t* next_job;
  uint32_t* stop;
  CodeEntry* res;
};

// The encoder's words: all 32 lanes keep the same range and count the words; lane 0 writes those within the cap.
struct LaneSink {
  uint32_t pos, cap;
  uint16_t* out;
  bool writer;
  __device__ __forceinline__ void operator()(uint32_t w) {
    if (writer && pos < cap) out[pos] = uint16_t(w);
    ++pos;
  }
};
using WarpRange = bcefmt::RangeEncoder<LaneSink>;

__global__ void __launch_bounds__(CM_THREADS) code_many_kernel(CodeArgs a) {
  __shared__ uint32_t s_off[8][32];
  __shared__ uint8_t s_bits[9][32];
  __shared__ uint16_t hdr[kHeaderCap];
  __shared__ uint32_t words[8];
  __shared__ uint32_t s_job, err, hlen;
  __shared__ unsigned long long at;
  __shared__ uint32_t fits;
  const unsigned tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  s_off[w][lane] = a.off[w][lane];
  for (uint32_t i = tid; i < 9 * 32; i += CM_THREADS) s_bits[i / 32][i % 32] = a.cfg[i / 32][i % 32];
  char* slot = a.slots + size_t(blockIdx.x) * a.slot_bytes;
  uint8_t* table = reinterpret_cast<uint8_t*>(slot + w * a.table_stride);
  uint16_t* stage = reinterpret_cast<uint16_t*>(slot + 8 * a.table_stride) + size_t(w) * a.stage_cap;

  for (;;) {
    if (tid == 0) err = 0;
    const uint32_t job = next_job(a.next_job, a.stop, a.k, s_job);
    if (job >= a.k) break;
    const uint32_t in = a.order[job];
    const ManyEntry& e = a.dir[in];
    if (!e.done) { __syncthreads(); continue; }                   // its words did not fit the front end's arena
    CodeEntry& r = a.res[in];
    if (e.err) {
      if (tid == 0) { r.err = e.err; r.done = 1; }
      __syncthreads();
      continue;
    }
    const uint32_t n = uint32_t(a.starts[in + 1] - a.starts[in]);

    // ---- stream w ---------------------------------------------------------------------------------------------------
    {
      uint4* t4 = reinterpret_cast<uint4*>(table);
#pragma unroll 1
      for (uint32_t i = lane; i < (a.tbytes[w] + 15) / 16; i += 32) t4[i] = make_uint4(0, 0, 0, 0);
      __syncwarp();
      WarpRange rc{0, ~0ull, {0, a.stage_cap, stage, lane == 0}};
      const uint8_t* bits = s_bits[w];
      rc.put_config(bits);
      rc.put_uniform(e.C[w], n + 1);
      uint32_t first = 0;
      for (int s = 0; s < int(w); ++s) first += e.count[s];
      const uint32_t* src = a.arena + e.start + first;
      const uint32_t W = e.count[w];
      uint32_t base = 0, win = lane < W ? __ldg(src + lane) : 0u;
      auto word = [&](uint32_t i) {                                // i is the same on every lane and never decreases
        if (i >= base + 32) {
          base = i;
          win = base + lane < W ? __ldg(src + base + lane) : 0u;
        }
        return __shfl_sync(kFull, win, i - base);
      };
      bool bad = false;
      for (uint32_t i = 0; i < W; ++i) {                           // code_packed, coders.cpp
        const uint32_t w0 = word(i);
        uint32_t sym, k, ctx;
        bcefmt::coder_fields(w0, sym, k, ctx);
        if (k == 0) {                                              // k > 31: nb uniform bits first
          const uint32_t w1 = word(i + 1), w2 = word(i + 2);
          i += 2;
          uint32_t nb, low;
          bcefmt::coder_escape(w1, w2, k, nb, low);
          for (uint32_t j = 0; j < nb; ++j) rc.put_uniform((low >> j) & 1u, 2);
        }
        if (k < 2 || sym >= k || ctx >= (1u << (2 * bits[k]))) { bad = true; break; }
        uint8_t* row = table + s_off[w][k] + ctx * (k + 2);          // row_offset without its mask (see CodeArgs)
        const uint32_t c = lane < k ? uint32_t(row[lane]) : 0u;
        const uint32_t below = sym + __reduce_add_sync(kFull, lane < sym ? c : 0u);
        const uint32_t total = k + __reduce_add_sync(kFull, c);
        const uint32_t freq = __shfl_sync(kFull, c, sym) + 1;
        rc.put(below, freq, total);
        if (freq == 0xFF) {                                        // ContextModel::bump: every counter halves
          if (lane < k) row[lane] = uint8_t((c + (lane == sym)) >> 1);
        } else if (lane == sym) {
          row[lane] = uint8_t(freq);
        }
      }
      rc.finish();
      if (lane == 0) {
        words[w] = rc.out.pos;
        if (bad) atomicOr(&err, kCodeErrWord);
        if (rc.out.pos > rc.out.cap) atomicOr(&err, kCodeErrStage);
      }
    }
    __syncthreads();

    // ---- header (ArchiveWriter::finish), warp 0 ------------------------------------------------------------------
    if (w == 0) {
      WarpRange rc{0, ~0ull, {0, kHeaderCap, hdr, lane == 0}};
      rc.put_config(s_bits[8]);
      // bcefmt::write_header restated, like row_offset above: calling the two changed this kernel's code (same
      // registers) and timed it about 1 % slower on a B200 at 1000 W
      rc.varint(n);
      rc.put_uniform(e.offset, n + 1);
      uint32_t total = 0;
      for (int s = 0; s < 8; ++s) total += words[s];
      rc.varint(total);
      uint32_t left = total;
      for (int s = 0; s < 7; ++s) {
        rc.put_uniform(words[s], left + 1);
        left -= words[s];
      }
      rc.finish();
      if (lane == 0) {
        hlen = rc.out.pos;
        if (rc.out.pos > rc.out.cap) atomicOr(&err, kCodeErrStage);
      }
    }
    __syncthreads();

    // ---- reserve the archive in the arena, copy it, fill the directory ------------------------------------------
    if (tid == 0) {
      fits = 0;
      if (err) {
        r.err = err;
        r.done = 1;
      } else {
        unsigned long long total = 1ull + hlen;
        for (int s = 0; s < 8; ++s) total += words[s];
        fits = arena_reserve(a.out_used, a.out_cap, a.stop, total, at);
      }
    }
    __syncthreads();
    if (fits) {
      uint16_t* o = a.out + at;
      for (uint32_t i = tid; i <= hlen; i += CM_THREADS) o[i] = i ? hdr[i - 1] : uint16_t(hlen);
      o += 1 + hlen;
      unsigned long long nw = 1ull + hlen, nwords = 0;
      for (int s = 0; s < 8; ++s) {
        const uint16_t* st = reinterpret_cast<const uint16_t*>(slot + 8 * a.table_stride) + size_t(s) * a.stage_cap;
        for (uint32_t i = tid; i < words[s]; i += CM_THREADS) o[i] = st[i];
        o += words[s];
        nw += words[s];
        nwords += e.count[s];
      }
      if (tid == 0) {
        r.start = at;
        r.nwords = uint32_t(nw);
        r.rounds = e.rounds;
        r.visits = e.visits;
        r.words = nwords;
        r.done = 1;
      }
    }
    __syncthreads();
  }
}

int code_many_run(Ctx* c, const uint8_t* T, const uint64_t* starts, uint32_t k, const uint8_t (*cfg)[32],
                  bce_many_archive* out) {
  CodeArgs a;
  memset(&a, 0, sizeof a);
  memcpy(a.cfg, cfg, sizeof a.cfg);
  size_t tmax = 16;
  for (int s = 0; s < 8; ++s) {
    a.tbytes[s] = bcefmt::model_layout(cfg[s], a.off[s]);
    for (int kk = 2; kk < 32; ++kk) a.off[s][kk] &= 0x00FFFFFFu;   // the kernel takes the bits from its config rows
    tmax = std::max<size_t>(tmax, a.tbytes[s]);
  }
  uint32_t N = 0;
  unsigned long long bound_sum = 0;                                 // every input's archive at its largest
  for (uint32_t i = 0; i < k; ++i) {
    const uint32_t n = uint32_t(starts[i + 1] - starts[i]);
    N = std::max(N, n);
    bound_sum += 8ull * stream_bound(n) + 1 + kHeaderCap;
  }
  a.table_stride = Carver::need(tmax, 1);
  a.stage_cap = stream_bound(N);
  a.slot_bytes = 8 * a.table_stride + Carver::need(size_t(8) * a.stage_cap, 2);
  // The archive arena holds the archives of every input whose words fit the front end's arena: a stream of W words
  // costs at most 3 W + 24 uint16 (32 bits of phi per word at most, bound above), so a call's archives need at most
  // 3 x (arena words) + 289 per input -- and never more than all inputs' bounds.
  const unsigned long long arena_cap = many_arena_cap(c, starts, k, 3);
  a.out_cap = std::min(3 * arena_cap + 289ull * k, bound_sum);
  const size_t fixed = 256 + Carver::need(k, sizeof(CodeEntry)) + Carver::need(a.out_cap, 2);
  size_t want = 0;
  BCE_TRY(many_grid(c, "compress_many_archives", reinterpret_cast<const void*>(code_many_kernel), CM_THREADS, 0, k, &want));

  ManyDevice dev;
  BCE_TRY(many_launch(c, T, starts, k, BCE_EMIT_CODER, cfg, fixed + a.slot_bytes, fixed + want * a.slot_bytes, &dev));
  const size_t ctas = std::min(want, (dev.tail_bytes - fixed) / a.slot_bytes);
  Carver cv(dev.tail, dev.tail_bytes);
  auto* d_ctr = cv.take<unsigned long long>(32);        // used uint16, next job, stop; zeroed with the directory
  auto* d_res = cv.take<CodeEntry>(k);
  a.out = cv.take<uint16_t>(a.out_cap);
  a.slots = cv.take<char>(ctas * a.slot_bytes);
  a.dir = dev.dir;
  a.starts = dev.starts;
  a.order = dev.order;
  a.arena = dev.arena;
  a.k = k;
  a.out_used = d_ctr;
  a.next_job = reinterpret_cast<uint32_t*>(d_ctr + 1);
  a.stop = reinterpret_cast<uint32_t*>(d_ctr + 2);
  a.res = d_res;

  cudaStream_t st = c->stream;
  const cudaEvent_t ev[2] = {c->ev[6], c->ev[7]};
  BCE_CUDA(c, cudaMemsetAsync(d_ctr, 0, 256 + size_t(k) * sizeof(CodeEntry), st));
  BCE_TRACE("compress_many_archives k=%u largest=%u ctas=%zu slot=%zu B archive arena=%llu words", k, N, ctas,
            a.slot_bytes, a.out_cap);
  BCE_CUDA(c, cudaEventRecord(ev[0], st));
  code_many_kernel<<<unsigned(ctas), CM_THREADS, 0, st>>>(a);
  c->stats.gpu_launches++;
  BCE_CUDA(c, cudaGetLastError());
  BCE_CUDA(c, cudaEventRecord(ev[1], st));

  std::vector<CodeEntry> res(k);
  const void* arena = nullptr;
  BCE_TRY(read_arena(c, ev, c->stats.ms_coder, d_ctr, d_res, res.data(), size_t(k) * sizeof(CodeEntry), a.out,
                     a.out_cap, 2, &arena));
  BCE_TRY(add_ms(c, dev.ev[0], dev.ev[1], c->stats.ms_cse_total));
  const uint16_t* words = static_cast<const uint16_t*>(arena);
  int rc = BCE_GPU_OK;
  for (uint32_t i = 0; i < k; ++i) {
    const CodeEntry& e = res[i];
    bce_many_archive& o = out[i];
    o.words = nullptr;
    o.nwords = 0;
    o.done = int(e.done);
    if (!e.done) continue;
    if (e.err) {
      if (rc == BCE_GPU_OK)
        set_error(c, "compress_many_archives: input %u: %s", i,
                  (e.err & kManyErrRunaway) ? "level loop ran past its round limit"
                  : (e.err & kManyErrStage) ? "staging area overflowed"
                  : (e.err & kCodeErrStage) ? "coder staging overflowed" : "malformed coder word");
      rc = BCE_GPU_E_INTERNAL;
      continue;
    }
    o.words = words + e.start;
    o.nwords = e.nwords;
    c->stats.cse_visits += e.visits;
    c->stats.cse_rounds += e.rounds;
    c->stats.cse_words += e.words;
  }
  c->stats.cse_launches = 1;
  c->stats.ms_total = c->stats.ms_h2d + c->stats.ms_cse_total + c->stats.ms_coder + c->stats.ms_d2h;
  return rc;
}

}  // namespace bce
