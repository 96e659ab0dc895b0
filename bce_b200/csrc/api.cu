// api.cu -- the extern "C" boundary declared in include/bce_gpu.h.
#include <stdarg.h>
#include <stdlib.h>

#include <algorithm>
#include <chrono>
#include <new>

#include "ctx.h"

namespace bce {

// BCE_GPU_TRACE=1: launch-by-launch timing on stderr (diagnostics only; read once per API call, never
// on a launch path)
static bool g_trace = false;
bool trace_on() { return g_trace; }
static void refresh_trace() {
  const char* v = getenv("BCE_GPU_TRACE");
  g_trace = v && *v && *v != '0';
}

void set_error(Ctx* c, const char* fmt, ...) {
  if (!c) return;
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(c->err, sizeof c->err, fmt, ap);
  va_end(ap);
}

int DevBuf::ensure(Ctx* c, size_t bytes) {
  if (bytes <= cap && p) return BCE_GPU_OK;
  if (p) { cudaFree(p); p = nullptr; cap = 0; }
  size_t want = (bytes + (size_t(1) << 20) - 1) & ~((size_t(1) << 20) - 1);
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    p = nullptr;
    cudaGetLastError();
    set_error(c, "cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
    return BCE_GPU_E_NOMEM;
  }
  // descriptor words rely on "tag 0 = never written": fresh memory is cleared once
  e = cudaMemsetAsync(p, 0, want, c->stream);
  if (e != cudaSuccess) { set_error(c, "cudaMemset failed: %s", cudaGetErrorString(e)); return BCE_GPU_E_CUDA; }
  cap = want;
  return BCE_GPU_OK;
}
void DevBuf::release() {
  if (p) cudaFree(p);
  p = nullptr; cap = 0;
}
int PinnedBuf::ensure(Ctx* c, size_t bytes) {
  if (bytes <= cap && p) return BCE_GPU_OK;
  if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
  size_t want = (bytes + (size_t(1) << 20) - 1) & ~((size_t(1) << 20) - 1);
  cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
  if (e != cudaSuccess) {
    p = nullptr;
    cudaGetLastError();
    set_error(c, "cudaHostAlloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
    return BCE_GPU_E_NOMEM;
  }
  cap = want;
  return BCE_GPU_OK;
}
void PinnedBuf::release() {
  if (p) cudaFreeHost(p);
  p = nullptr; cap = 0;
}

int next_tag(Ctx* c) {
  // tags are unique per pass; 0 means "never written".  On wrap the descriptors are cleared.
  if (++c->desc_tag >= 0x3FFFFFFFu) {
    c->desc_tag = 1;
    if (c->desc.p) cudaMemsetAsync(c->desc.p, 0, c->desc.cap, c->stream);
  }
  return int(c->desc_tag);
}

// Host <-> device copies of caller memory.  Pageable memory is legal for cudaMemcpyAsync
// (the runtime stages it); large pageable copies go through our own pinned staging buffer
// in chunks so that the copy engine runs at pinned speed.
constexpr size_t kStageChunk = size_t(64) << 20;
bool is_pinned(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeHost;
}
int h2d(Ctx* c, void* dst, const void* src, size_t bytes) {
  if (!bytes) return BCE_GPU_OK;
  if (is_pinned(src) || bytes <= (size_t(1) << 20)) {
    BCE_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
    BCE_CUDA(c, cudaStreamSynchronize(c->stream));
    return BCE_GPU_OK;
  }
  BCE_TRY(c->pinned_io.ensure(c, 2 * kStageChunk));
  char* stage = c->pinned_io.as<char>();
  cudaEvent_t done[2] = {c->ev[6], c->ev[7]};
  bool used[2] = {false, false};
  size_t at = 0;
  for (int b = 0; at < bytes; b ^= 1) {
    size_t len = bytes - at < kStageChunk ? bytes - at : kStageChunk;
    if (used[b]) BCE_CUDA(c, cudaEventSynchronize(done[b]));
    memcpy(stage + b * kStageChunk, static_cast<const char*>(src) + at, len);
    BCE_CUDA(c, cudaMemcpyAsync(static_cast<char*>(dst) + at, stage + b * kStageChunk, len,
                                cudaMemcpyHostToDevice, c->stream));
    BCE_CUDA(c, cudaEventRecord(done[b], c->stream));
    used[b] = true;
    at += len;
  }
  BCE_CUDA(c, cudaStreamSynchronize(c->stream));
  return BCE_GPU_OK;
}
int d2h(Ctx* c, void* dst, const void* src, size_t bytes) {
  if (!bytes) return BCE_GPU_OK;
  if (is_pinned(dst) || bytes <= (size_t(1) << 20)) {
    BCE_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    BCE_CUDA(c, cudaStreamSynchronize(c->stream));
    return BCE_GPU_OK;
  }
  BCE_TRY(c->pinned_io.ensure(c, 2 * kStageChunk));
  char* stage = c->pinned_io.as<char>();
  cudaEvent_t done[2] = {c->ev[6], c->ev[7]};
  size_t at = 0, pending_at[2] = {0, 0}, pending_len[2] = {0, 0};
  bool used[2] = {false, false};
  for (int b = 0; at < bytes; b ^= 1) {
    size_t len = bytes - at < kStageChunk ? bytes - at : kStageChunk;
    if (used[b]) {
      BCE_CUDA(c, cudaEventSynchronize(done[b]));
      memcpy(static_cast<char*>(dst) + pending_at[b], stage + b * kStageChunk, pending_len[b]);
    }
    BCE_CUDA(c, cudaMemcpyAsync(stage + b * kStageChunk, static_cast<const char*>(src) + at, len,
                                cudaMemcpyDeviceToHost, c->stream));
    BCE_CUDA(c, cudaEventRecord(done[b], c->stream));
    used[b] = true; pending_at[b] = at; pending_len[b] = len;
    at += len;
  }
  BCE_CUDA(c, cudaStreamSynchronize(c->stream));
  // drain in issue order: the older of the two pending chunks first
  int order[2] = {0, 1};
  if (used[0] && used[1] && pending_at[1] < pending_at[0]) { order[0] = 1; order[1] = 0; }
  for (int k = 0; k < 2; ++k) {
    int b = order[k];
    if (used[b]) memcpy(static_cast<char*>(dst) + pending_at[b], stage + b * kStageChunk, pending_len[b]);
  }
  return BCE_GPU_OK;
}

size_t scratch_budget(Ctx* c) {
  size_t b = size_t(double(c->total_mem) * 0.70);
  if (c->scratch_limit && c->scratch_limit < b) b = c->scratch_limit;
  return b;
}

static int check_n(Ctx* c, uint32_t n) {
  if (n == 0 || n >= 0x80000000u) { set_error(c, "n = %u outside 1 .. 2^31-1", n); return BCE_GPU_E_ARG; }
  return BCE_GPU_OK;
}

static void begin_call(Ctx* c) {
  refresh_trace();
  c->err[0] = 0;
  cudaSetDevice(c->device);
}

static int upload_text(Ctx* c, const uint8_t* T, uint32_t n) {
  if (c->prefetch_pending) {                           // bce_gpu_prefetch_input: the copy may already be there
    c->prefetch_pending = false;
    const bool arrived = cudaEventQuery(c->ev_prefetch[1]) == cudaSuccess;
    BCE_CUDA(c, cudaEventSynchronize(c->ev_prefetch[1]));
    BCE_TRACE("prefetched input: %s, %s", arrived ? "already on the device" : "still in flight",
              (c->prefetch_src == T && c->prefetch_n == n) ? "adopted" : "another input: discarded");
    if (c->prefetch_src == T && c->prefetch_n == n) {
      float ms = 0;
      BCE_CUDA(c, cudaEventElapsedTime(&ms, c->ev_prefetch[0], c->ev_prefetch[1]));
      c->stats.ms_h2d += ms;                           // the copy's own duration; it ran beside the previous level loop
      c->n = n;
      c->text_resident = true;
      c->bwt_resident = false;
      c->ranks_resident = false;
      return BCE_GPU_OK;
    }
  }
  BCE_TRY(c->text.ensure(c, size_t(n) + 128));
  cudaEvent_t a = c->ev[4], b = c->ev[5];
  BCE_CUDA(c, cudaEventRecord(a, c->stream));
  BCE_TRY(h2d(c, c->text.p, T, n));
  BCE_CUDA(c, cudaEventRecord(b, c->stream));
  BCE_CUDA(c, cudaEventSynchronize(b));
  float ms = 0;
  BCE_CUDA(c, cudaEventElapsedTime(&ms, a, b));
  c->stats.ms_h2d += ms;
  c->n = n;
  c->text_resident = true;
  c->bwt_resident = false;
  c->ranks_resident = false;
  return BCE_GPU_OK;
}

static int run_bwt(Ctx* c, uint32_t n, uint32_t* sa_host) {
  cudaEvent_t a = c->ev[4], b = c->ev[5];
  BCE_CUDA(c, cudaEventRecord(a, c->stream));
  BCE_TRY(suffix_sort_bwt(c, n, sa_host));
  BCE_CUDA(c, cudaEventRecord(b, c->stream));
  BCE_CUDA(c, cudaEventSynchronize(b));
  float ms = 0;
  BCE_CUDA(c, cudaEventElapsedTime(&ms, a, b));
  c->stats.ms_bwt_total += ms;
  return BCE_GPU_OK;
}

static int run_cse_begin(Ctx* c, uint32_t n) {
  c->cse_emit_mode_active = int(c->emit_mode);
  cudaEvent_t a = c->ev[4], b = c->ev[5];
  BCE_CUDA(c, cudaEventRecord(a, c->stream));
  BCE_TRY(wavelet_build(c, n));
  BCE_TRY(cse_begin(c, n));
  BCE_CUDA(c, cudaEventRecord(b, c->stream));
  BCE_CUDA(c, cudaEventSynchronize(b));
  float ms = 0;
  BCE_CUDA(c, cudaEventElapsedTime(&ms, a, b));
  c->stats.ms_cse_total += ms;
  return BCE_GPU_OK;
}

static const uint8_t kDefaultCfg[8][32] = {                              // bce.cpp:713-724, rows 0..7
  {0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,0},
  {0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,0},
  {0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,3,3,3,3,0},
  {0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,0},
  {0,0,5,5,4,4,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,0},
  {0,0,5,5,4,4,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,0},
  {0,0,5,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,0},
  {0,0,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,2,2,2,2,2,2,0}};

static void reset_stats(Ctx* c, uint32_t n) {
  memset(&c->stats, 0, sizeof c->stats);
  c->stats.n = n;
}

// Checks of the compress_many calls' inputs, then the context state they leave: no text, BWT or level loop resident.
static int begin_many(Ctx* c, const uint64_t* starts, uint32_t k) {
  if (k == 0) { set_error(c, "compress_many: no inputs"); return BCE_GPU_E_ARG; }
  uint32_t largest = 0;
  for (uint32_t i = 0; i < k; ++i) {
    if (starts[i + 1] <= starts[i] || starts[i + 1] - starts[i] > BCE_GPU_MANY_MAX_N) {
      set_error(c, "compress_many: input %u: size outside 1 .. %u", i, unsigned(BCE_GPU_MANY_MAX_N));
      return BCE_GPU_E_ARG;
    }
    largest = std::max(largest, uint32_t(starts[i + 1] - starts[i]));
  }
  reset_stats(c, largest);
  if (c->prefetch_pending) {                           // the text buffer is about to be overwritten
    BCE_CUDA(c, cudaEventSynchronize(c->ev_prefetch[1]));
    c->prefetch_pending = false;
  }
  c->cse_active = false;
  c->cse_resident = false;
  c->text_resident = c->bwt_resident = c->ranks_resident = false;
  return BCE_GPU_OK;
}

}  // namespace bce

using bce::Ctx;

extern "C" {

int bce_gpu_abi_version(void) { return BCE_GPU_ABI_VERSION; }

const char* bce_gpu_error_string(int code) {
  switch (code) {
    case BCE_GPU_OK: return "ok";
    case BCE_GPU_E_ARG: return "bad argument";
    case BCE_GPU_E_NOMEM: return "out of memory";
    case BCE_GPU_E_CUDA: return "CUDA failure";
    case BCE_GPU_E_STATE: return "call sequence violated";
    case BCE_GPU_E_FRONTIER: return "CSE frontier exceeded its device memory";
    case BCE_GPU_E_INTERNAL: return "internal consistency check failed";
    case BCE_GPU_E_NODEVICE: return "no usable CUDA device";
    default: return "unknown error";
  }
}

int bce_gpu_open(int device, bce_gpu_ctx** out) {
  if (!out) return BCE_GPU_E_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) { cudaGetLastError(); return BCE_GPU_E_NODEVICE; }
  if (device < 0 || device >= count) return BCE_GPU_E_ARG;
  if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return BCE_GPU_E_NODEVICE; }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { cudaGetLastError(); return BCE_GPU_E_CUDA; }
  if (prop.major < 10 || !prop.cooperativeLaunch) return BCE_GPU_E_NODEVICE;   // built for sm_100a only
  Ctx* c = new (std::nothrow) Ctx();
  if (!c) return BCE_GPU_E_NOMEM;
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->total_mem = prop.totalGlobalMem;
  bool ok = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&c->h2d_stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreate(&c->ev_prefetch[0]) == cudaSuccess && cudaEventCreate(&c->ev_prefetch[1]) == cudaSuccess;
  for (int i = 0; ok && i < 8; ++i) ok = cudaEventCreate(&c->ev[i]) == cudaSuccess;
  for (int i = 0; ok && i < 256; ++i) ok = cudaEventCreate(&c->pass_ev[i]) == cudaSuccess;
  if (ok) ok = bce::radix_init_device(c) == BCE_GPU_OK;      // per-device function attributes
  if (ok) ok = bce::sort_init_device(c) == BCE_GPU_OK;
  if (ok) ok = c->small.ensure(c, bce::kSmallBytes) == BCE_GPU_OK;
  if (ok) ok = c->pinned_small.ensure(c, bce::kSmallBytes) == BCE_GPU_OK;
  if (ok) ok = cudaStreamSynchronize(c->stream) == cudaSuccess;
  if (!ok) { bce_gpu_close(c); return BCE_GPU_E_CUDA; }
  *out = c;
  return BCE_GPU_OK;
}

void bce_gpu_close(bce_gpu_ctx* h) {
  if (!h) return;
  Ctx* c = static_cast<Ctx*>(h);
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  bce::cse_destroy(c);
  c->text.release(); c->bwt.release(); c->ranks.release(); c->scratch.release();
  c->small.release(); c->desc.release();
  c->scan_tmp.release(); c->pack_tmp.release();
  c->pinned_small.release(); c->pinned_emit.release(); c->pinned_emit2.release(); c->pinned_io.release();
  c->pinned_many.release(); c->pinned_many2.release();
  for (auto& e : c->ev) if (e) cudaEventDestroy(e);
  for (auto& e : c->pass_ev) if (e) cudaEventDestroy(e);
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->h2d_stream) { cudaStreamSynchronize(c->h2d_stream); cudaStreamDestroy(c->h2d_stream); }
  for (auto& e : c->ev_prefetch) if (e) cudaEventDestroy(e);
  delete c;
}

const char* bce_gpu_last_error(const bce_gpu_ctx* h) {
  return h ? static_cast<const Ctx*>(h)->err : "null context";
}

int bce_gpu_get_stats(const bce_gpu_ctx* h, bce_gpu_stats* out) {
  if (!h || !out) return BCE_GPU_E_ARG;
  *out = static_cast<const Ctx*>(h)->stats;
  return BCE_GPU_OK;
}

int bce_gpu_set_scratch_limit(bce_gpu_ctx* h, size_t bytes) {
  if (!h) return BCE_GPU_E_ARG;
  static_cast<Ctx*>(h)->scratch_limit = bytes;
  return BCE_GPU_OK;
}

void* bce_gpu_host_alloc(bce_gpu_ctx* h, size_t bytes) {
  if (!h || !bytes) return nullptr;
  Ctx* c = static_cast<Ctx*>(h);
  cudaSetDevice(c->device);
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    bce::set_error(c, "cudaHostAlloc(%zu bytes) failed", bytes);
    return nullptr;
  }
  return p;
}

void bce_gpu_host_free(bce_gpu_ctx* h, void* p) {
  if (!h || !p) return;
  cudaSetDevice(static_cast<Ctx*>(h)->device);
  cudaFreeHost(p);
}

int bce_gpu_set_option(bce_gpu_ctx* h, int option, uint64_t value) {
  if (!h) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  switch (option) {
    case BCE_GPU_OPT_EMIT_BATCH_BYTES:
      c->emit_batch_bytes = value ? size_t(value) : size_t(1) << 30;
      return BCE_GPU_OK;
    case BCE_GPU_OPT_LOCAL_SORT_MIN:
      c->local_sort_min = value ? uint32_t(value > 0xFFFFFFFFull ? 0xFFFFFFFFull : value) : 1u << 20;
      return BCE_GPU_OK;
    case BCE_GPU_OPT_SLOT_ENTER_NODES:
      c->slot_enter_nodes = value ? value : 2000000;
      return BCE_GPU_OK;
    case BCE_GPU_OPT_MID_ENTER_NODES:
      c->mid_enter_nodes = value ? value : 400000;
      return BCE_GPU_OK;
    case BCE_GPU_OPT_NO_NARROW_KERNELS:
      c->no_narrow_kernels = value != 0;
      return BCE_GPU_OK;
    case BCE_GPU_OPT_RESIDENT_CHECKSUM:
      c->resident_checksum = value != 0;
      return BCE_GPU_OK;
    default:
      set_error(c, "bce_gpu_set_option: unknown option %d", option);
      return BCE_GPU_E_ARG;
  }
}

int bce_gpu_bwt(bce_gpu_ctx* h, const uint8_t* T, uint32_t n, uint8_t* L_out, uint32_t* offset_out,
                uint32_t* SA_out) {
  if (!h || !T) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  BCE_TRY(bce::check_n(c, n));
  bce::reset_stats(c, n);
  c->cse_active = false;
  BCE_TRY(bce::upload_text(c, T, n));
  BCE_TRY(bce::run_bwt(c, n, SA_out));
  if (offset_out) *offset_out = c->offset;
  if (L_out) BCE_TRY(bce::d2h(c, L_out, c->bwt.p, n));
  return BCE_GPU_OK;
}

static int load_bwt(Ctx* c, const uint8_t* L, uint32_t n) {
  if (L) {
    BCE_TRY(c->bwt.ensure(c, size_t(n) + 64));
    BCE_TRY(bce::h2d(c, c->bwt.p, L, n));
    c->n = n;
    c->bwt_resident = true;
    c->ranks_resident = false;
  } else if (!c->bwt_resident || c->n != n) {
    bce::set_error(c, "no BWT of length %u resident on the device", n);
    return BCE_GPU_E_STATE;
  }
  return BCE_GPU_OK;
}

int bce_gpu_wavelet(bce_gpu_ctx* h, const uint8_t* L, uint32_t n, uint64_t* const ranks_out[8],
                    uint32_t C_out[8]) {
  if (!h) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  BCE_TRY(bce::check_n(c, n));
  if (L) bce::reset_stats(c, n);
  c->cse_active = false;
  BCE_TRY(load_bwt(c, L, n));
  BCE_TRY(bce::wavelet_build(c, n));
  if (C_out) for (int i = 0; i < 8; ++i) C_out[i] = c->C[i];
  if (ranks_out) {
    const size_t words = size_t(n) / 32 + 1;
    for (int j = 0; j < 8; ++j)
      if (ranks_out[j])
        BCE_TRY(bce::d2h(c, ranks_out[j], c->ranks.as<uint64_t>() + size_t(j) * words, words * 8));
  }
  return BCE_GPU_OK;
}

int bce_gpu_cse_begin(bce_gpu_ctx* h, const uint8_t* L, uint32_t n, uint32_t C_out[8]) {
  if (!h) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  BCE_TRY(bce::check_n(c, n));
  if (L) bce::reset_stats(c, n);
  c->cse_resident = false;
  BCE_TRY(load_bwt(c, L, n));
  BCE_TRY(bce::run_cse_begin(c, n));
  if (C_out) for (int i = 0; i < 8; ++i) C_out[i] = c->C[i];
  return BCE_GPU_OK;
}

static int next_words(Ctx* c, bce::CseWordBatch* wb, bool pack20 = false) {
  const auto t0 = std::chrono::steady_clock::now();
  BCE_TRY(bce::cse_advance(c, false, wb, pack20));
  c->stats.ms_cse_total += std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return BCE_GPU_OK;
}

int bce_gpu_cse_next(bce_gpu_ctx* h, bce_cse_batch* out) {
  if (!h || !out) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  if (c->cse_active && c->cse_emit_mode_active != BCE_EMIT_RAW) {
    bce::set_error(c, "cse_next: the run emits packed words, use bce_gpu_cse_next_words");
    return BCE_GPU_E_STATE;
  }
  bce::CseWordBatch wb;
  BCE_TRY(next_words(c, &wb));
  for (int i = 0; i < 8; ++i) {
    out->tuples[i] = reinterpret_cast<const bce_tuple*>(wb.words[i]);
    out->count[i] = wb.count[i] / 5;
  }
  out->done = wb.done;
  return BCE_GPU_OK;
}

int bce_gpu_cse_next_words(bce_gpu_ctx* h, bce_cse_words* out) {
  if (!h || !out) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  bce::CseWordBatch wb;
  BCE_TRY(next_words(c, &wb));
  for (int i = 0; i < 8; ++i) { out->words[i] = wb.words[i]; out->count[i] = wb.count[i]; }
  out->done = wb.done;
  return BCE_GPU_OK;
}

int bce_gpu_cse_next_words20(bce_gpu_ctx* h, bce_cse_words20* out) {
  if (!h || !out) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  if (!c->cse_active || c->cse_emit_mode_active != BCE_EMIT_CODER) {
    bce::set_error(c, "cse_next_words20: needs a run started in BCE_EMIT_CODER mode");
    return BCE_GPU_E_STATE;
  }
  bce::CseWordBatch wb;
  BCE_TRY(next_words(c, &wb, true));
  for (int i = 0; i < 8; ++i) { out->bytes[i] = reinterpret_cast<const uint8_t*>(wb.words[i]); out->count[i] = wb.count[i]; }
  out->done = wb.done;
  return BCE_GPU_OK;
}

int bce_gpu_cse_next_buckets(bce_gpu_ctx* h, bce_scan_buckets* out) {
  if (!h || !out) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  if (!c->cse_active || c->cse_emit_mode_active != BCE_EMIT_SCAN) {
    bce::set_error(c, "cse_next_buckets: needs a run started in BCE_EMIT_SCAN mode");
    return BCE_GPU_E_STATE;
  }
  const auto t0 = std::chrono::steady_clock::now();
  BCE_TRY(bce::cse_advance_buckets(c, out));
  c->stats.ms_cse_total += std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return BCE_GPU_OK;
}

int bce_gpu_set_emit_mode(bce_gpu_ctx* h, int mode, const uint8_t* cfg288) {
  if (!h || mode < BCE_EMIT_RAW || mode > BCE_EMIT_SCAN) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  c->emit_mode = uint32_t(mode);
  if (cfg288) {
    for (int i = 0; i < 8; ++i)
      for (int k = 0; k < 32; ++k) {
        if (cfg288[i * 32 + k] > 5) { bce::set_error(c, "config: context bits %u > 5", cfg288[i * 32 + k]); return BCE_GPU_E_ARG; }
        c->emit_cfg[i][k] = cfg288[i * 32 + k];
      }
  } else {
    memcpy(c->emit_cfg, bce::kDefaultCfg, sizeof bce::kDefaultCfg);
  }
  return BCE_GPU_OK;
}

int bce_gpu_compress_front(bce_gpu_ctx* h, const uint8_t* T, uint32_t n, uint32_t* offset_out,
                           uint32_t C_out[8]) {
  if (!h || !T) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  BCE_TRY(bce::check_n(c, n));
  bce::reset_stats(c, n);
  c->cse_active = false;
  c->cse_resident = false;
  BCE_TRY(bce::upload_text(c, T, n));
  BCE_TRY(bce::run_bwt(c, n, nullptr));
  BCE_TRY(bce::run_cse_begin(c, n));
  if (offset_out) *offset_out = c->offset;
  if (C_out) for (int i = 0; i < 8; ++i) C_out[i] = c->C[i];
  return BCE_GPU_OK;
}

int bce_gpu_compress_many(bce_gpu_ctx* h, const uint8_t* T, const uint64_t* starts, uint32_t k, bce_many_result* out) {
  if (!h || !T || !starts || !out) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  BCE_TRY(bce::begin_many(c, starts, k));
  return bce::many_run(c, T, starts, k, out);
}

int bce_gpu_compress_many_archives(bce_gpu_ctx* h, const uint8_t* T, const uint64_t* starts, uint32_t k,
                                   const uint8_t* cfg288, bce_many_archive* out) {
  if (!h || !T || !starts || !out) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  uint8_t cfg[9][32] = {};
  if (cfg288) {
    for (int i = 0; i < 288; ++i)
      if (cfg288[i] > 5) { bce::set_error(c, "config: context bits %u > 5", cfg288[i]); return BCE_GPU_E_ARG; }
    memcpy(cfg, cfg288, sizeof cfg);
  } else {
    memcpy(cfg, bce::kDefaultCfg, sizeof bce::kDefaultCfg);   // row 8 (the header coder) stays 0
  }
  BCE_TRY(bce::begin_many(c, starts, k));
  return bce::code_many_run(c, T, starts, k, cfg, out);
}

int bce_gpu_prefetch_input(bce_gpu_ctx* h, const uint8_t* T, uint32_t n) {
  if (!h || !T) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  BCE_TRY(bce::check_n(c, n));
  if (!bce::is_pinned(T)) return BCE_GPU_OK;           // pageable memory cannot be copied asynchronously: the next call uploads it
  if (c->prefetch_pending) { BCE_CUDA(c, cudaEventSynchronize(c->ev_prefetch[1])); c->prefetch_pending = false; }
  // the text buffer is free once the BWT exists (the wavelet matrix and the level loop never read it)
  BCE_TRY(c->text.ensure(c, size_t(n) + 128));
  BCE_CUDA(c, cudaStreamSynchronize(c->stream));       // idle between calls; orders a fresh buffer's clearing before the copy
  BCE_CUDA(c, cudaEventRecord(c->ev_prefetch[0], c->h2d_stream));
  BCE_CUDA(c, cudaMemcpyAsync(c->text.p, T, n, cudaMemcpyHostToDevice, c->h2d_stream));
  BCE_CUDA(c, cudaEventRecord(c->ev_prefetch[1], c->h2d_stream));
  c->text_resident = false;
  c->prefetch_src = T;
  c->prefetch_n = n;
  c->prefetch_pending = true;
  return BCE_GPU_OK;
}

int bce_gpu_stage_input(bce_gpu_ctx* h, const uint8_t* T, uint32_t n) {
  if (!h || !T) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  BCE_TRY(bce::check_n(c, n));
  bce::reset_stats(c, n);
  c->cse_active = false;
  return bce::upload_text(c, T, n);
}

int bce_gpu_front_resident(bce_gpu_ctx* h, uint32_t* offset_out, uint64_t* tuples_out) {
  if (!h) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  if (!c->text_resident) { bce::set_error(c, "front_resident: no staged input"); return BCE_GPU_E_STATE; }
  const uint32_t n = c->n;
  const float h2d_ms = c->stats.ms_h2d;
  bce::reset_stats(c, n);
  c->stats.ms_h2d = h2d_ms;
  c->cse_active = false;
  c->cse_resident = true;
  BCE_TRY(bce::run_bwt(c, n, nullptr));
  BCE_TRY(bce::run_cse_begin(c, n));
  while (!c->cse_done) {
    cudaEvent_t e0 = c->ev[4], e1 = c->ev[5];
    BCE_CUDA(c, cudaEventRecord(e0, c->stream));
    BCE_TRY(bce::cse_advance(c, true, nullptr));
    BCE_CUDA(c, cudaEventRecord(e1, c->stream));
    BCE_CUDA(c, cudaEventSynchronize(e1));
    float ms = 0;
    BCE_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
    c->stats.ms_cse_total += ms;
  }
  c->stats.ms_total = c->stats.ms_bwt_total + c->stats.ms_cse_total;
  if (offset_out) *offset_out = c->offset;
  if (tuples_out) *tuples_out = c->emit_mode == BCE_EMIT_RAW ? c->stats.cse_tuples : c->stats.cse_words;
  return BCE_GPU_OK;
}

int bce_gpu_resident_checksum(bce_gpu_ctx* h, uint64_t sum[8], uint64_t wsum[8]) {
  if (!h || !sum || !wsum) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  if (!c->cse_resident || !c->cse_done || !c->resident_checksum) {
    bce::set_error(c, "resident_checksum: no finished front_resident run with BCE_GPU_OPT_RESIDENT_CHECKSUM set");
    return BCE_GPU_E_STATE;
  }
  uint64_t acc[16];
  BCE_TRY(bce::d2h(c, acc, c->small.as<char>() + bce::kSmallChecksum, sizeof acc));
  for (int i = 0; i < 8; ++i) { sum[i] = acc[2 * i]; wsum[i] = acc[2 * i + 1]; }
  return BCE_GPU_OK;
}

int bce_gpu_unbwt(bce_gpu_ctx* h, const uint64_t* const ranks[8], uint32_t offset, uint32_t n, uint8_t* out) {
  if (!h || !ranks || !out) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  BCE_TRY(bce::check_n(c, n));
  if (offset >= n) { bce::set_error(c, "offset %u >= n %u", offset, n); return BCE_GPU_E_ARG; }
  bce::reset_stats(c, n);
  c->cse_active = false;
  const size_t words = size_t(n) / 32 + 1;
  BCE_TRY(c->ranks.ensure(c, 8 * words * 8));
  for (int j = 0; j < 8; ++j) {
    if (!ranks[j]) return BCE_GPU_E_ARG;
    BCE_TRY(bce::h2d(c, c->ranks.as<uint64_t>() + size_t(j) * words, ranks[j], words * 8));
    // zeros of level j = n - rank1(n), read off the last word (Rank::get<0>(n), bce.cpp:1052-1061)
    uint64_t w = ranks[j][n / 32];
    uint32_t ones = uint32_t(w) + uint32_t(__builtin_popcount(uint32_t(w >> 32) & ((1u << (n % 32)) - 1u)));
    c->C[(j + 1) & 7] = n - ones;
  }
  c->n = n;
  c->ranks_resident = true;
  c->bwt_resident = false;
  c->text_resident = false;
  return bce::unbwt_run(c, ranks, offset, n, out);
}

int bce_gpu_unbwt_many(bce_gpu_ctx* h, const uint64_t* ranks, const uint32_t* n, const uint32_t* offset, uint32_t k,
                       uint8_t* out) {
  if (!h || !ranks || !n || !offset || !out) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  if (k == 0) { bce::set_error(c, "unbwt_many: no dictionaries"); return BCE_GPU_E_ARG; }
  uint32_t largest = 0;
  for (uint32_t i = 0; i < k; ++i) {
    if (n[i] == 0 || n[i] > BCE_GPU_MANY_MAX_N) {
      bce::set_error(c, "unbwt_many: dictionary %u: n = %u outside 1 .. %u", i, n[i], unsigned(BCE_GPU_MANY_MAX_N));
      return BCE_GPU_E_ARG;
    }
    if (offset[i] > n[i]) { bce::set_error(c, "unbwt_many: dictionary %u: offset %u > n %u", i, offset[i], n[i]); return BCE_GPU_E_ARG; }
    largest = std::max(largest, n[i]);
  }
  bce::reset_stats(c, largest);
  c->cse_active = false;                 // the scratch a level loop in progress keeps its state in is about to be reused
  c->cse_resident = false;
  return bce::unbwt_many_run(c, ranks, n, offset, k, out);
}

int bce_gpu_decompress_many(bce_gpu_ctx* h, const uint16_t* words, const uint64_t* starts, const uint32_t* n,
                            uint32_t k, uint8_t* out, int* status) {
  if (!h || !words || !starts || !n || !out || !status) return BCE_GPU_E_ARG;
  Ctx* c = static_cast<Ctx*>(h);
  bce::begin_call(c);
  if (k == 0) { bce::set_error(c, "decompress_many: no archives"); return BCE_GPU_E_ARG; }
  uint32_t largest = 0;
  for (uint32_t i = 0; i < k; ++i) {
    if (n[i] == 0 || n[i] > BCE_GPU_MANY_MAX_N) {
      bce::set_error(c, "decompress_many: archive %u: n = %u outside 1 .. %u", i, n[i], unsigned(BCE_GPU_MANY_MAX_N));
      return BCE_GPU_E_ARG;
    }
    if (starts[i + 1] < starts[i]) { bce::set_error(c, "decompress_many: archive %u: starts decrease", i); return BCE_GPU_E_ARG; }
    largest = std::max(largest, n[i]);
  }
  bce::reset_stats(c, largest);
  c->cse_active = false;                 // the scratch a level loop in progress keeps its state in is about to be reused
  c->cse_resident = false;
  return bce::decode_many_run(c, words, starts, n, k, out, status);
}

}  // extern "C"
