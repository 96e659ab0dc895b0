// ctx.h -- the context behind bce_gpu_ctx and the internal stage entry points.
#pragma once

#include <stdlib.h>

#include <algorithm>
#include <numeric>
#include <vector>

#include "common.cuh"

struct bce_gpu_ctx {};   // opaque to callers; bce::Ctx derives from it

namespace bce {

constexpr int kMaxSortRounds = 48;

// Knobs read from the environment exist only in experiment builds (-DBCE_GPU_EXPERIMENTS, see
// bce_b200/build.py); the shipped library takes every such decision from the defaults measured in
// profiles/ and never calls getenv on a launch path.
inline size_t exp_env(const char* name, size_t dflt) {
#ifdef BCE_GPU_EXPERIMENTS
  const char* v = getenv(name);
  if (v && *v) return size_t(strtoull(v, nullptr, 10));
#else
  (void)name;
#endif
  return dflt;
}

struct CseDeviceState;   // cse.cu

struct Ctx : bce_gpu_ctx {
  int device = 0;
  int sm_count = 0;
  size_t total_mem = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;
  cudaStream_t h2d_stream = nullptr;        // bce_gpu_prefetch_input: the next input's upload, beside the level loop
  cudaEvent_t ev_prefetch[2] = {};
  const uint8_t* prefetch_src = nullptr;    // what the pending prefetch copies (compared by address and size)
  uint32_t prefetch_n = 0;
  bool prefetch_pending = false;
  cudaEvent_t ev[8] = {};
  cudaEvent_t pass_ev[256] = {};     // start/stop pairs around individual radix passes (resolved lazily)
  int pass_ev_n = 0;
  char err[512] = {0};
  size_t scratch_limit = 0;

  // persistent device data
  DevBuf text;        // T, padded (n + 64)
  DevBuf bwt;         // L, padded
  DevBuf ranks;       // 8 x rank_words u64
  DevBuf scratch;     // carved per stage
  DevBuf small;       // counters, histograms, descriptors' tickets, state structs
  DevBuf desc;        // tile descriptors (tagged, never cleared between passes)
  PinnedBuf pinned_small;   // host mirror for small read-backs
  PinnedBuf pinned_emit;    // emitted counts handed to the caller (two buffers alternate)
  PinnedBuf pinned_emit2;
  PinnedBuf pinned_io;      // staging for pageable caller buffers
  DevBuf scan_tmp;          // bce -s: sort buffers, bucketed symbols and bucket tables of one batch
  DevBuf pack_tmp;          // a batch's words as 20 bits each, on their way to the host (bce_gpu_cse_next_words20)
  PinnedBuf pinned_many;    // words of a bce_gpu_compress_many call (two buffers alternate)
  PinnedBuf pinned_many2;
  int many_flip = 0;

  uint32_t desc_tag = 0;    // monotonically increasing pass tag (30 bits used)

  // options (bce_gpu_set_option)
  size_t emit_batch_bytes = size_t(1) << 30;   // BCE_GPU_OPT_EMIT_BATCH_BYTES
  uint32_t local_sort_min = 1u << 20;          // BCE_GPU_OPT_LOCAL_SORT_MIN
  bool resident_checksum = false;              // BCE_GPU_OPT_RESIDENT_CHECKSUM
  uint64_t slot_enter_nodes = 2000000;         // BCE_GPU_OPT_SLOT_ENTER_NODES
  uint64_t mid_enter_nodes = 400000;           // BCE_GPU_OPT_MID_ENTER_NODES
  bool no_narrow_kernels = false;              // BCE_GPU_OPT_NO_NARROW_KERNELS

  // state of the current input
  uint32_t n = 0;
  bool text_resident = false;
  bool bwt_resident = false;
  bool ranks_resident = false;
  uint32_t offset = 0;
  uint32_t C[8] = {};

  // emission format for the next cse_begin (bce_gpu_set_emit_mode)
  uint32_t emit_mode = 0;
  uint8_t emit_cfg[8][32] = {};
  bool cse_resident = false;   // counts stay in device memory (front_resident)
  int cse_emit_mode_active = 0; // mode the current run was started with

  // CSE run state (host side)
  bool cse_active = false;
  bool cse_done = false;
  struct CseHost* cse = nullptr;

  bce_gpu_stats stats = {};
};

// layout of Ctx::small (device) in bytes; Ctx::pinned_small mirrors it on the host
constexpr size_t kSmallHist = 0;                              // 8 x 256 u32  digit histograms
constexpr size_t kSmallBase = kSmallHist + 8 * 256 * 4;       // 8 x 256 u32  digit starts
constexpr size_t kSmallTicket = kSmallBase + 8 * 256 * 4;     // 16 u32       radix tile dispensers
constexpr size_t kSmallErr = kSmallTicket + 64;               // 1 u32        chained-scan watchdog flag
constexpr size_t kSmallRerankTotals = kSmallErr + 64;         // 2 u32 re-rank totals; [3] the tile-local sort's fall-back count
constexpr size_t kSmallWavelet = kSmallRerankTotals + 64;     // 256 u32 hist + 8 u32 zeros + 8 tickets
constexpr size_t kSmallCse = kSmallWavelet + 2048;            // CseDeviceState
constexpr size_t kSmallUnbwt = kSmallCse + 1024;              // inverse BWT: 256 u32 hist, 257 u32 F starts, 1 u32 check flag
constexpr size_t kSmallChecksum = 44 * 1024;                  // 8 x 2 u64    per-stream checksums of the resident emission
constexpr size_t kSmallRadixCursor = 52 * 1024;               // 256 u32      write cursors of a sort's first (unordered) pass
constexpr size_t kSmallPartHist = 48 * 1024;                  // 256 u32      histogram of the rank-scatter partition digit
constexpr size_t kSmallPartCursor = kSmallPartHist + 1024;    // 256 u32      write cursors of the binned rank pairs / BWT rows
constexpr size_t kSmallBytes = 64 * 1024;

// ---- stage entry points (each launches kernels on ctx->stream) --------------------
// radix_sort.cu: LSD radix sort of (u64 key, u32 value) pairs on digit shifts[0..npass).
// Buffers are ping-ponged; *out_k / *out_v receive the pointers that hold the result.
// Where the digit histograms of a sort come from (default: one extra read of the keys).
struct RadixHistSource {
  const uint8_t* window_text = nullptr;   // keys are the 8-symbol cyclic windows of this text (window_key_bits) and the values
                                          // their start indices; the first pass makes them, so keyA / valA are not read.  If no
                                          // pass runs (one repeated byte), nothing makes them: the caller has to pack them itself.
  bool codes7 = false;                    // window_text holds 7-bit symbol codes: the key packs 8 of them into 56 bits
  bool host_hist = false;                 // [npass][256] already in the host mirror of the histograms (Ctx::pinned_small)
  const uint32_t* dev_hist = nullptr;     // [npass][256] already counted on the device (e.g. by the kernel that wrote the keys);
                                          // may be Ctx::small + kSmallHist itself
  bool stable_first = false;              // every pass stable, the first included: equal keys keep their input order
                                          // (the suffix sorter does not need that: ties are told apart by later rounds)
};
int radix_sort_pairs(Ctx* c, uint64_t* keyA, uint64_t* keyB, uint32_t* valA, uint32_t* valB,
                     uint32_t m, const int* shifts, int npass, uint64_t** out_k, uint32_t** out_v,
                     int* passes_run, const RadixHistSource* src = nullptr);
constexpr int kRadixMaxPasses = 8;
struct RadixShifts { int s[kRadixMaxPasses]; };
size_t radix_desc_words(uint32_t m);

// suffix_sort.cu
int suffix_sort_bwt(Ctx* c, uint32_t n, uint32_t* sa_host_or_null);
// wavelet.cu
int wavelet_build(Ctx* c, uint32_t n);
void byte_hist_launch(Ctx* c, const uint8_t* L, uint32_t n, uint32_t* d_hist);   // adds L[0..n)'s byte histogram to d_hist[256]
// cse.cu
int cse_begin(Ctx* c, uint32_t n);
struct CseWordBatch { const uint32_t* words[8]; size_t count[8]; int done; };
// pack20: out->words[i] points at 20-bit words, two in 5 bytes (BCE_EMIT_CODER: every word is below 2^20)
int cse_advance(Ctx* c, bool resident, CseWordBatch* out, bool pack20 = false);
int cse_advance_buckets(Ctx* c, bce_scan_buckets* out);
void cse_destroy(Ctx* c);
// unbwt.cu
// host_ranks: the same 8 levels as Ctx::ranks, on the host (words that are no rank directory are walked there)
int unbwt_run(Ctx* c, const uint64_t* const host_ranks[8], uint32_t offset, uint32_t n, uint8_t* out_host);
// ---- the many calls: k items of 1 .. BCE_GPU_MANY_MAX_N bytes, one CTA per item on a persistent grid -------------
// Job j takes item order[j]: the largest first, so the longest CTAs start first; equal sizes keep their index order.
template <class Size> std::vector<uint32_t> largest_first(uint32_t k, Size size_of) {
  std::vector<uint32_t> order(k);
  std::iota(order.begin(), order.end(), 0u);
  std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return size_of(x) > size_of(y); });
  return order;
}
// CTAs of a persistent grid of `kernel`: as many as are resident at once, at most k (BCE_GPU_E_INTERNAL when not even
// one fits an SM).  Sets the kernel's dynamic shared memory limit to smem when it is not 0.
int many_grid(Ctx* c, const char* call, const void* kernel, int threads, size_t smem, uint32_t k, size_t* ctas);
// starts - starts[0], the k + 1 offsets of the items in a buffer that holds only them
std::vector<unsigned long long> rebase_starts(const uint64_t* starts, uint32_t k);
// Adds the milliseconds from `start` to `end` to stat once `end` has happened.
int add_ms(Ctx* c, cudaEvent_t start, cudaEvent_t end, float& stat);

// The job of a persistent CTA: thread 0 takes the next from *next (k once *stop is set; stop may be null), and every
// thread returns it.  Job k and above: none left.
__device__ __forceinline__ uint32_t next_job(uint32_t* next, const uint32_t* stop, uint32_t k, uint32_t& shared_job) {
  if (threadIdx.x == 0) shared_job = stop && *reinterpret_cast<const volatile uint32_t*>(stop) ? k : atomicAdd(next, 1u);
  __syncthreads();
  return shared_job;
}
// One thread reserves len elements of an arena of cap: at = the first of them.  When they do not fit it sets *stop, so
// that no CTA takes another job, and returns false; the host submits the items left again.
__device__ __forceinline__ bool arena_reserve(unsigned long long* used, unsigned long long cap, uint32_t* stop,
                                              unsigned long long len, unsigned long long& at) {
  at = atomicAdd(used, len);
  const bool fits = at + len <= cap;
  if (!fits) atomicExch(stop, 1u);
  return fits;
}

// unbwt_many.cu: k dictionaries of 1 .. BCE_GPU_MANY_MAX_N rows in one launch (arguments checked)
int unbwt_many_run(Ctx* c, const uint64_t* ranks, const uint32_t* n, const uint32_t* offset, uint32_t k,
                   uint8_t* out_host);
struct UmDict {                     // one dictionary of unbwt_many_kernel (device)
  unsigned long long words;         // its first rank word
  unsigned long long out;           // its first output byte
  uint32_t n, offset;
};
struct UmTable {                    // k dictionaries back to back: rank words and texts
  std::vector<UmDict> dict;
  uint32_t N;                       // the largest n
  unsigned long long words, bytes;  // in all
};
UmTable um_table(const uint32_t* n, const uint32_t* offset, uint32_t k);   // offset null: 0 (the decoder fills it in)
// Queues unbwt_many_kernel on c->stream over dictionaries already on the device: order = dictionary taken by job j
// (largest first), N = the largest n, d_ctr = 2 zeroed counters (work, serial), d_status = null or per dictionary
// non-zero to skip it.
int unbwt_many_launch(Ctx* c, const uint64_t* d_ranks, const UmDict* d_dict, const uint32_t* d_order,
                      const int* d_status, uint32_t k, uint32_t N, uint32_t* d_ctr, uint8_t* d_out);
// decode_many.cu: k archives whose headers must claim n[i] (1 .. BCE_GPU_MANY_MAX_N, arguments checked) -> their
// texts back to back in out, status[i] = 0 or BCE_GPU_E_ARG; the decode loop and the inverse in two launches.
int decode_many_run(Ctx* c, const uint16_t* words, const uint64_t* starts, const uint32_t* n, uint32_t k,
                    uint8_t* out, int* status);
// many.cu: the whole front end of k inputs of 1 .. BCE_GPU_MANY_MAX_N bytes in one launch (arguments checked)
int many_run(Ctx* c, const uint8_t* T, const uint64_t* starts, uint32_t k, bce_many_result* out);
struct ManyEntry {                  // per-input directory many_kernel fills on the device
  uint32_t done, err, offset, rounds;
  uint32_t C[8];
  uint32_t count[8];                // words per stream
  unsigned long long start;         // first word in the arena
  unsigned long long visits;
};
enum : uint32_t { kManyErrRunaway = 1, kManyErrStage = 2 };
struct ManyDevice {                 // what many_launch leaves on the device once its kernel is queued
  ManyEntry* dir;                   // k entries
  const unsigned long long* starts; // k + 1 offsets of the inputs in c->text
  const uint32_t* arena;
  const unsigned long long* used;   // words of the arena taken
  const uint32_t* order;            // input taken by job j (largest first)
  unsigned long long arena_cap;     // words
  char* tail;                       // tail_bytes of scratch that the caller's next launch on c->stream may use (it
  size_t tail_bytes;                // overlaps the kernel's CTA slots, which are dead once the kernel has ended)
  cudaEvent_t ev[2];                // recorded on c->stream before and after many_kernel: its time is ms_cse_total's
};
// The read-back of an arena a launch on c->stream filled, on the copy stream: once launch[1] (recorded after the
// launch) has happened, the used count and dir_bytes of directory, and launch[0] .. launch[1] added to launch_ms; then
// the used part of the arena (at most cap elements of elem bytes) into the next of the two pinned buffers, *host, with
// the copy's time (timed by the same event pair) added to ms_d2h.
int read_arena(Ctx* c, const cudaEvent_t launch[2], float& launch_ms, const unsigned long long* d_used,
               const void* d_dir, void* dir, size_t dir_bytes, const void* d_arena, unsigned long long cap, size_t elem,
               const void** host);
// The arena of one call in words: a batch of BCE_GPU_OPT_EMIT_BATCH_BYTES, never less than the largest input's worst
// case (else that input could never be done) and never more than every input's.
unsigned long long many_arena_cap(const Ctx* c, const uint64_t* starts, uint32_t k, uint32_t maxw);
// Uploads the inputs and queues many_kernel with emission `mode` (kEmitRaw / kEmitCoder) and context bits cfg;
// tail_min / tail_want: bytes the caller needs after the kernel (BCE_GPU_E_NOMEM when tail_min does not fit).
int many_launch(Ctx* c, const uint8_t* T, const uint64_t* starts, uint32_t k, uint32_t mode, const uint8_t (*cfg)[32],
                size_t tail_min, size_t tail_want, ManyDevice* d);
// code_many.cu: the archives of k inputs -- many_launch in CODER mode, then every range coder on the device.  cfg: the
// 9 x 32 table (row 8: the header coder), cells checked.
int code_many_run(Ctx* c, const uint8_t* T, const uint64_t* starts, uint32_t k, const uint8_t (*cfg)[32],
                  bce_many_archive* out);

// api.cu helpers
int next_tag(Ctx* c);
bool is_pinned(const void* p);
int h2d(Ctx* c, void* dst, const void* src, size_t bytes);
int d2h(Ctx* c, void* dst, const void* src, size_t bytes);
int radix_init_device(Ctx* c);   // radix_sort.cu: per-device function attributes
int sort_init_device(Ctx* c);    // suffix_sort.cu: the same
size_t scratch_budget(Ctx* c);

}  // namespace bce
