// host_api.cpp -- extern "C" surface of libbce_host (include/bce_host.h).
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <new>
#include <thread>
#include <vector>

#include "../../../include/bce_host.h"
#include "archive.hpp"
#include "decode.hpp"

using namespace bcehost;

struct bce_archive_writer { ArchiveWriter* w; };
struct bce_scan { ScanSession* s; };

static ConfigTable table_from(const uint8_t* cfg288) {
  ConfigTable t = default_config();
  if (cfg288) std::memcpy(t.data(), cfg288, 288);
  return t;
}

// The C ABI never lets an exception out: allocation failures become BCE_GPU_E_NOMEM.
#define BCE_HOST_GUARD(body)                                   \
  try { body }                                                 \
  catch (const std::bad_alloc&) { return BCE_GPU_E_NOMEM; }    \
  catch (...) { return BCE_GPU_E_INTERNAL; }

static bool table_ok(const uint8_t* cfg288) { return !cfg288 || bcefmt::config_ok(cfg288, 288); }   // null: the default

#ifndef BCE_HOST_NO_GPU
// The inputs todo of a bce_compress_many call as one submission: T itself when todo is every input, else the inputs
// copied back to back into packed.  sub receives the submission's k + 1 offsets.
static const uint8_t* gather(const uint8_t* T, const uint64_t* starts, uint32_t k, const std::vector<uint32_t>& todo,
                             std::vector<uint8_t>& packed, std::vector<uint64_t>& sub) {
  if (todo.size() == k) {
    sub.assign(starts, starts + k + 1);
    return T;
  }
  packed.clear();
  sub.assign(1, 0);
  for (uint32_t i : todo) {
    packed.insert(packed.end(), T + starts[i], T + starts[i + 1]);
    sub.push_back(packed.size());
  }
  return packed.data();
}

// The rounds of bce_compress_many: call(base, sub, m, res) submits the m inputs still to do (gathered), and finish(res,
// todo, done) handles those the call finished, done being their positions in todo; the rest go again.  A call that
// finishes none is BCE_GPU_E_INTERNAL.
template <class Result, class Call, class Finish>
static int resubmit(const uint8_t* T, const uint64_t* starts, uint32_t k, Call call, Finish finish) {
  std::vector<uint32_t> todo(k);
  for (uint32_t i = 0; i < k; ++i) todo[i] = i;
  std::vector<uint8_t> packed;
  std::vector<uint64_t> sub;
  std::vector<Result> res;
  while (!todo.empty()) {
    const uint8_t* base = gather(T, starts, k, todo, packed, sub);
    res.assign(todo.size(), Result{});
    int rc = call(base, sub.data(), uint32_t(todo.size()), res.data());
    if (rc) return rc;
    std::vector<uint32_t> done, left;
    for (size_t j = 0; j < todo.size(); ++j) (res[j].done ? done : left).push_back(uint32_t(j));
    if (done.empty()) return BCE_GPU_E_INTERNAL;
    rc = finish(res.data(), todo, done);
    if (rc) return rc;
    for (uint32_t& j : left) j = todo[j];
    todo.swap(left);
  }
  return BCE_GPU_OK;
}

#endif

extern "C" {

const uint8_t* bce_host_default_config(void) {
  return reinterpret_cast<const uint8_t*>(default_config().data());
}
void bce_host_free(void* p) { std::free(p); }

bce_archive_writer* bce_archive_begin(uint32_t n, const uint32_t C[8], const uint8_t* cfg288) {
  if (!C || n == 0 || n >= 0x80000000u || !table_ok(cfg288)) return nullptr;
  auto* h = new (std::nothrow) bce_archive_writer{nullptr};
  if (!h) return nullptr;
  try { h->w = new ArchiveWriter(n, C, table_from(cfg288)); }
  catch (...) { h->w = nullptr; }
  if (!h->w) { delete h; return nullptr; }
  return h;
}
int bce_archive_feed(bce_archive_writer* h, const bce_cse_batch* batch, int threads) {
  if (!h || !batch) return BCE_GPU_E_ARG;
  BCE_HOST_GUARD(h->w->feed(*batch, threads);)
  return BCE_GPU_OK;
}
int bce_archive_feed_words(bce_archive_writer* h, const bce_cse_words* batch, int threads) {
  if (!h || !batch) return BCE_GPU_E_ARG;
  BCE_HOST_GUARD(h->w->feed_words(*batch, threads);)
  return BCE_GPU_OK;
}
int bce_archive_begin_words(bce_archive_writer* h, const bce_cse_words* batch) {
  if (!h || !batch) return BCE_GPU_E_ARG;
  BCE_HOST_GUARD(h->w->begin_words(*batch);)
  return BCE_GPU_OK;
}
int bce_archive_begin_words20(bce_archive_writer* h, const bce_cse_words20* batch) {
  if (!h || !batch) return BCE_GPU_E_ARG;
  BCE_HOST_GUARD(h->w->begin_words20(*batch);)
  return BCE_GPU_OK;
}
int bce_archive_wait(bce_archive_writer* h) {
  if (!h) return BCE_GPU_E_ARG;
  h->w->wait_words();
  return BCE_GPU_OK;
}
int bce_scan_feed_words(bce_scan* h, const bce_cse_words* batch) {
  if (!h || !batch) return BCE_GPU_E_ARG;
  BCE_HOST_GUARD(h->s->feed_words(*batch);)
  return BCE_GPU_OK;
}
int bce_scan_feed_buckets(bce_scan* h, const bce_scan_buckets* batch) {
  if (!h || !batch) return BCE_GPU_E_ARG;
  BCE_HOST_GUARD(h->s->feed_buckets(*batch);)
  return BCE_GPU_OK;
}
size_t bce_host_pack_counts(int mode, const uint8_t* cfg288, int stream, const bce_tuple* t, size_t count, uint32_t* words) {
  if (!table_ok(cfg288) || stream < 0 || stream > 7) return 0;
  ConfigTable tab = table_from(cfg288);
  size_t at = 0;
  for (size_t i = 0; i < count; ++i) {
    uint32_t e[3];
    const uint32_t nw = bcefmt::pack_count(mode == BCE_EMIT_CODER, tab[stream].data(), t[i].sym, t[i].k, t[i].c1, t[i].c2,
                                           t[i].cs, e[0], e[1], e[2]);
    for (uint32_t j = 0; j < nw; ++j) words[at++] = e[j];
  }
  return at;
}
int bce_archive_finish(bce_archive_writer* h, uint32_t offset, uint16_t** words, size_t* nwords) {
  if (!h || !words || !nwords) return BCE_GPU_E_ARG;
  std::vector<uint16_t> out;
  try { out = h->w->finish(offset); }
  catch (...) { delete h->w; delete h; return BCE_GPU_E_NOMEM; }
  delete h->w;
  delete h;
  uint16_t* mem = static_cast<uint16_t*>(std::malloc(out.size() * sizeof(uint16_t) + 2));
  if (!mem) return BCE_GPU_E_NOMEM;
  std::memcpy(mem, out.data(), out.size() * sizeof(uint16_t));
  *words = mem;
  *nwords = out.size();
  return BCE_GPU_OK;
}
void bce_archive_abort(bce_archive_writer* h) {
  if (!h) return;
  delete h->w;
  delete h;
}

bce_scan* bce_scan_begin(void) {
  auto* h = new (std::nothrow) bce_scan{nullptr};
  if (!h) return nullptr;
  try { h->s = new ScanSession(); }
  catch (...) { h->s = nullptr; }
  if (!h->s) { delete h; return nullptr; }
  return h;
}
int bce_scan_feed(bce_scan* h, const bce_cse_batch* batch) {
  if (!h || !batch) return BCE_GPU_E_ARG;
  BCE_HOST_GUARD(h->s->feed(*batch);)
  return BCE_GPU_OK;
}
int bce_scan_finish(bce_scan* h, uint8_t cfg288_out[288]) {
  if (!h || !cfg288_out) return BCE_GPU_E_ARG;
  int rc = BCE_GPU_OK;
  try {
    ConfigTable t = h->s->finish();
    std::memcpy(cfg288_out, t.data(), 288);
  } catch (const std::bad_alloc&) { rc = BCE_GPU_E_NOMEM; }
  catch (...) { rc = BCE_GPU_E_INTERNAL; }
  delete h->s;
  delete h;
  return rc;
}

int bce_decode_buffer(const uint16_t* words, size_t nwords, int low_memory, uint8_t** out, size_t* nout) {
  if (!words || !out || !nout) return BCE_GPU_E_ARG;
  std::vector<uint8_t> text;
  int rc = BCE_GPU_OK;
  BCE_HOST_GUARD(
    std::vector<uint16_t> archive(words, words + nwords);
    rc = decode_archive(archive, low_memory != 0, text);                         // BCE::decode, bce.cpp:1169-1233
  )
  if (rc) return rc;
  uint8_t* mem = static_cast<uint8_t*>(std::malloc(text.size() + 1));
  if (!mem) return BCE_GPU_E_NOMEM;
  std::memcpy(mem, text.data(), text.size());
  *out = mem;
  *nout = text.size();
  return BCE_GPU_OK;
}

#ifndef BCE_HOST_NO_GPU
int bce_compress_buffer(bce_gpu_ctx* ctx, const uint8_t* T, uint32_t n, const uint8_t* cfg288, int threads,
                        uint16_t** words, size_t* nwords) {
  using clk = std::chrono::steady_clock;
  auto secs = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double>(b - a).count(); };
  const bool timing = std::getenv("BCE_TIME") != nullptr;           // the reference's -DM_TIME lines, per phase
  const auto t0 = clk::now();
  uint32_t offset = 0, C[8];
  // the device emits coder-ready words: context index and k > 31 halving are done there
  int rc = bce_gpu_set_emit_mode(ctx, BCE_EMIT_CODER, cfg288);
  if (rc) return rc;
  rc = bce_gpu_compress_front(ctx, T, n, &offset, C);               // RankFile ctor, bce.cpp:1411
  if (rc) { bce_gpu_set_emit_mode(ctx, BCE_EMIT_RAW, nullptr); return rc; }
  const auto t1 = clk::now();
  bce_archive_writer* w = bce_archive_begin(n, C, cfg288);          // BCE::encode, bce.cpp:1417
  if (!w) { bce_gpu_set_emit_mode(ctx, BCE_EMIT_RAW, nullptr); return BCE_GPU_E_NOMEM; }
  // Double buffering over the context's two pinned batch buffers: while the coder threads work on batch j, the
  // next call copies batch j+1 out and runs the kernels of batch j+2 (a batch stays valid until the call after
  // the next one, include/bce_gpu.h).  threads <= 1 keeps the serial form.
  bce_cse_words20 cur, nxt;                             // 20 bits per word over PCIe
  double gpu_s = 0, wait_s = 0;
  size_t nbatch = 0, nw = 0;
  auto fail = [&](int code) { bce_archive_abort(w); bce_gpu_set_emit_mode(ctx, BCE_EMIT_RAW, nullptr); return code; };
  {
    const auto a = clk::now();
    rc = bce_gpu_cse_next_words20(ctx, &cur);
    gpu_s += secs(a, clk::now());
    if (rc) return fail(rc);
  }
  for (;;) {
    ++nbatch;
    for (int i = 0; i < 8; ++i) nw += cur.count[i];
    if (threads <= 1) {
      const auto a = clk::now();
      try { w->w->begin_words20(cur); w->w->wait_words(); } catch (...) { return fail(BCE_GPU_E_NOMEM); }
      wait_s += secs(a, clk::now());
      if (cur.done) break;
      const auto b = clk::now();
      rc = bce_gpu_cse_next_words20(ctx, &nxt);
      gpu_s += secs(b, clk::now());
      if (rc) return fail(rc);
    } else {
      try { w->w->begin_words20(cur); } catch (...) { return fail(BCE_GPU_E_NOMEM); }
      const bool last = cur.done != 0;
      if (!last) {
        const auto a = clk::now();
        rc = bce_gpu_cse_next_words20(ctx, &nxt);                  // coders of batch j run under this call
        gpu_s += secs(a, clk::now());
      }
      const auto b = clk::now();
      w->w->wait_words();
      wait_s += secs(b, clk::now());
      if (last) break;
      if (rc) return fail(rc);
    }
    cur = nxt;
  }
  bce_gpu_set_emit_mode(ctx, BCE_EMIT_RAW, nullptr);
  const auto t2 = clk::now();
  double busiest = 0;
  for (int i = 0; i < 8; ++i) busiest = std::max(busiest, w->w->busy_seconds(i));
  rc = bce_archive_finish(w, offset, words, nwords);
  if (timing)
    std::fprintf(stderr, "[bce] front (H2D + BWT + wavelet) %.3f s | in cse_next_words %.3f s (%s the coders) | waiting for "
                 "the coders after it %.3f s | busiest coder %.3f s (%d threads, %zu words in %zu batches) | finish %.3f s\n",
                 secs(t0, t1), gpu_s, threads > 1 ? "under" : "not overlapped with", wait_s, busiest, threads, nw, nbatch,
                 secs(t2, clk::now()));
  return rc;
}

int bce_compress_many(bce_gpu_ctx* ctx, const uint8_t* T, const uint64_t* starts, uint32_t k, const uint8_t* cfg288,
                      int threads, uint16_t* words[], size_t nwords[]) {
  if (!ctx || !T || !starts || !words || !nwords || k == 0 || !table_ok(cfg288)) return BCE_GPU_E_ARG;
  for (uint32_t i = 0; i < k; ++i) { words[i] = nullptr; nwords[i] = 0; }
  int rc;
  if (k >= BCE_HOST_MANY_DEVICE_CODERS) {        // the range coders on the device too
    auto call = [&](const uint8_t* base, const uint64_t* sub, uint32_t m, bce_many_archive* res) {
      return bce_gpu_compress_many_archives(ctx, base, sub, m, cfg288, res);
    };
    auto finish = [&](const bce_many_archive* res, const std::vector<uint32_t>& todo, const std::vector<uint32_t>& done) {
      for (uint32_t j : done) {
        uint16_t* mem = static_cast<uint16_t*>(std::malloc(res[j].nwords * sizeof(uint16_t) + 2));
        if (!mem) return BCE_GPU_E_NOMEM;
        std::memcpy(mem, res[j].words, res[j].nwords * sizeof(uint16_t));
        words[todo[j]] = mem;
        nwords[todo[j]] = res[j].nwords;
      }
      return BCE_GPU_OK;
    };
    try { rc = resubmit<bce_many_archive>(T, starts, k, call, finish); }
    catch (const std::bad_alloc&) { rc = BCE_GPU_E_NOMEM; }
  } else {
    rc = bce_gpu_set_emit_mode(ctx, BCE_EMIT_CODER, cfg288);
    if (rc) return rc;
    auto call = [&](const uint8_t* base, const uint64_t* sub, uint32_t m, bce_many_result* res) {
      return bce_gpu_compress_many(ctx, base, sub, m, res);
    };
    // every done input becomes an archive (BCE::encode, bce.cpp:1117-1167), one input per thread
    auto finish = [&](const bce_many_result* res, const std::vector<uint32_t>& todo, const std::vector<uint32_t>& done) {
      std::atomic<size_t> next{0};
      std::atomic<int> err{BCE_GPU_OK};
      auto code = [&]() {
        for (size_t d; (d = next.fetch_add(1)) < done.size();) {
          const bce_many_result& r = res[done[d]];
          const uint32_t i = todo[done[d]];
          bce_archive_writer* w = bce_archive_begin(uint32_t(starts[i + 1] - starts[i]), r.C, cfg288);
          if (!w) { err = BCE_GPU_E_NOMEM; continue; }
          bce_cse_words b;
          for (int s = 0; s < 8; ++s) { b.words[s] = r.words[s]; b.count[s] = r.count[s]; }
          b.done = 1;
          int e = bce_archive_feed_words(w, &b, 1);
          if (e) { bce_archive_abort(w); err = e; continue; }
          e = bce_archive_finish(w, r.offset, &words[i], &nwords[i]);
          if (e) err = e;
        }
      };
      const size_t nt = std::min<size_t>(std::max(threads, 1), done.size());
      try {
        std::vector<std::thread> pool;
        for (size_t t = 1; t < nt; ++t) pool.emplace_back(code);
        code();
        for (auto& t : pool) t.join();
      } catch (...) { return int(BCE_GPU_E_NOMEM); }
      return int(err);
    };
    try { rc = resubmit<bce_many_result>(T, starts, k, call, finish); }
    catch (const std::bad_alloc&) { rc = BCE_GPU_E_NOMEM; }
    bce_gpu_set_emit_mode(ctx, BCE_EMIT_RAW, nullptr);
  }
  if (rc)
    for (uint32_t i = 0; i < k; ++i) { std::free(words[i]); words[i] = nullptr; nwords[i] = 0; }
  return rc;
}

// Text bytes of the small archives one bce_gpu_unbwt_many call inverts: bounds its device memory (about three bytes
// per text byte: rank words and output) and the host memory of the decoded dictionaries waiting for it.
static constexpr uint64_t kUnbwtManyBytes = uint64_t(64) << 20;

int bce_archive_size(const uint16_t* words, size_t nwords, uint32_t* n) {
  if (!words || !n) return BCE_GPU_E_ARG;
  return archive_size(words, nwords, *n);
}

int bce_decompress_many(bce_gpu_ctx* ctx, const uint16_t* words, const uint64_t* starts, uint32_t k, int threads,
                        uint8_t* out[], size_t nout[], int status[]) {
  if (!ctx || !words || !starts || !out || !nout || !status || k == 0) return BCE_GPU_E_ARG;
  for (uint32_t i = 0; i < k; ++i) {
    out[i] = nullptr; nout[i] = 0; status[i] = BCE_GPU_OK;
    if (starts[i + 1] < starts[i]) return BCE_GPU_E_ARG;
  }
  int rc = BCE_GPU_OK;
  auto give = [&](uint32_t i, const uint8_t* text, size_t len) {     // malloc'd copy for the caller
    uint8_t* mem = static_cast<uint8_t*>(std::malloc(len + 1));
    if (!mem) return false;
    std::memcpy(mem, text, len);
    out[i] = mem;
    nout[i] = len;
    return true;
  };
  try {
    // small archives (n from the header) go in groups through one level-serial decoder per thread and one
    // bce_gpu_unbwt_many call per group; a header that cannot be read is that archive's error
    std::vector<uint32_t> small, large;
    std::vector<uint32_t> size(k, 0);
    const char* cap = std::getenv("BCE_HOST_MAX_N");                 // as decode_to_ranks: refused before decoding
    const uint64_t max_n = cap ? std::strtoull(cap, nullptr, 10) : ~0ull;
    const char* dd = std::getenv("BCE_HOST_MANY_DEVICE_DECODERS");    // measurements: move the threshold
    const uint64_t device_min = dd ? std::strtoull(dd, nullptr, 10) : BCE_HOST_MANY_DEVICE_DECODERS;
    for (uint32_t i = 0; i < k; ++i) {
      const int e = archive_size(words + starts[i], size_t(starts[i + 1] - starts[i]), size[i]);
      if (e) status[i] = e;
      else if (size[i] > max_n) status[i] = BCE_GPU_E_ARG;
      else (size[i] <= BCE_GPU_MANY_MAX_N ? small : large).push_back(i);
    }
    struct Decoded { std::vector<DecodeRank> ranks; uint32_t n = 0, offset = 0; };
    for (size_t g0 = 0; g0 < small.size() && rc == BCE_GPU_OK;) {
      size_t g1 = g0;
      for (uint64_t b = 0; g1 < small.size() && (g1 == g0 || b + size[small[g1]] <= kUnbwtManyBytes); ++g1)
        b += size[small[g1]];
      if (g1 - g0 >= device_min) {                 // the whole decoder on the device
        std::vector<uint16_t> w;
        std::vector<uint64_t> sub{0};
        std::vector<uint32_t> n;
        uint64_t bytes = 0;
        for (size_t j = g0; j < g1; ++j) {
          const uint32_t i = small[j];
          w.insert(w.end(), words + starts[i], words + starts[i + 1]);
          sub.push_back(w.size());
          n.push_back(size[i]);
          bytes += size[i];
        }
        if (w.empty()) w.push_back(0);                                 // never a null pointer
        std::vector<uint8_t> text(bytes);
        std::vector<int> st(g1 - g0);
        rc = bce_gpu_decompress_many(ctx, w.data(), sub.data(), n.data(), uint32_t(g1 - g0), text.data(), st.data());
        if (rc) break;
        uint64_t at = 0;
        for (size_t j = g0; j < g1; at += n[j - g0], ++j) {
          if (st[j - g0]) status[small[j]] = st[j - g0];
          else if (!give(small[j], text.data() + at, n[j - g0])) { rc = BCE_GPU_E_NOMEM; break; }
        }
        g0 = g1;
        continue;
      }
      std::vector<Decoded> dec(g1 - g0);
      std::atomic<size_t> next{g0};
      std::atomic<int> err{BCE_GPU_OK};
      auto work = [&]() {                                             // BCE::decode, bce.cpp:1169-1233, one archive per thread
        for (size_t j; (j = next.fetch_add(1)) < g1;) {
          const uint32_t i = small[j];
          Decoded& d = dec[j - g0];
          int e;
          try {
            e = decode_to_ranks(words + starts[i], size_t(starts[i + 1] - starts[i]), d.ranks, d.n, d.offset, 1);
          } catch (const std::bad_alloc&) { e = BCE_GPU_E_NOMEM; }
          catch (...) { e = BCE_GPU_E_INTERNAL; }                   // nothing may leave a worker thread
          if (e == BCE_GPU_E_ARG) { status[i] = e; d.ranks.clear(); }
          else if (e) err = e;
        }
      };
      const size_t nt = std::min<size_t>(std::max(threads, 1), g1 - g0);
      {
        std::vector<std::thread> pool;
        try {
          for (size_t t = 1; t < nt; ++t) pool.emplace_back(work);
        } catch (...) {}                                               // fewer threads: the running ones take the rest
        work();
        for (auto& t : pool) t.join();
      }
      rc = err;
      if (rc) break;
      // the intact ones' dictionaries back to back, then one launch for all their inverses
      std::vector<uint32_t> ids, n, offset;
      std::vector<uint64_t> rw;
      uint64_t bytes = 0;
      for (size_t j = g0; j < g1; ++j) {
        Decoded& d = dec[j - g0];
        if (d.ranks.empty()) continue;
        ids.push_back(small[j]);
        n.push_back(d.n);
        offset.push_back(d.offset);
        bytes += d.n;
        for (const DecodeRank& r : d.ranks) rw.insert(rw.end(), r.words().begin(), r.words().end());
        std::vector<DecodeRank>().swap(d.ranks);
      }
      if (!ids.empty()) {
        std::vector<uint8_t> text(bytes);
        rc = bce_gpu_unbwt_many(ctx, rw.data(), n.data(), offset.data(), uint32_t(ids.size()), text.data());
        if (rc) break;
        uint64_t at = 0;
        for (size_t j = 0; j < ids.size(); at += n[j], ++j)
          if (!give(ids[j], text.data() + at, n[j])) { rc = BCE_GPU_E_NOMEM; break; }
      }
      g0 = g1;
    }
    // larger archives one at a time: the 8-level-thread decoder and bce_gpu_unbwt on the caller's context
    for (size_t j = 0; j < large.size() && rc == BCE_GPU_OK; ++j) {
      const uint32_t i = large[j];
      std::vector<DecodeRank> ranks;
      uint32_t n = 0, offset = 0;
      const int e = decode_to_ranks(words + starts[i], size_t(starts[i + 1] - starts[i]), ranks, n, offset,
                                    default_level_threads());
      if (e == BCE_GPU_E_ARG) { status[i] = e; continue; }
      if (e) { rc = e; break; }
      const uint64_t* lv[8];
      for (int l = 0; l < 8; ++l) lv[l] = ranks[l].words().data();
      std::vector<uint8_t> text(n);
      rc = bce_gpu_unbwt(ctx, lv, offset % n, n, text.data());      // unbwt::bytewise, bce.cpp:1043-1103
      if (!rc && !give(i, text.data(), n)) rc = BCE_GPU_E_NOMEM;
    }
  } catch (const std::bad_alloc&) { rc = BCE_GPU_E_NOMEM; }
  catch (...) { rc = BCE_GPU_E_INTERNAL; }                            // e.g. std::system_error from a thread
  if (rc)
    for (uint32_t i = 0; i < k; ++i) { std::free(out[i]); out[i] = nullptr; nout[i] = 0; }
  return rc;
}

int bce_scan_buffer(bce_gpu_ctx* ctx, const uint8_t* T, uint32_t n, uint8_t cfg288_out[288]) {
  uint32_t offset = 0, C[8];
  int rc = bce_gpu_set_emit_mode(ctx, BCE_EMIT_SCAN, nullptr);
  if (rc) return rc;
  rc = bce_gpu_compress_front(ctx, T, n, &offset, C);
  if (rc) { bce_gpu_set_emit_mode(ctx, BCE_EMIT_RAW, nullptr); return rc; }
  bce_scan* s = bce_scan_begin();
  if (!s) { bce_gpu_set_emit_mode(ctx, BCE_EMIT_RAW, nullptr); return BCE_GPU_E_NOMEM; }
  // the counts arrive bucketed by (k, context key) from the device; the host appends runs of symbol bytes and
  // runs ScanCoder's flush unchanged (bce.cpp:751-800)
  bce_scan_buckets batch;
  do {
    rc = bce_gpu_cse_next_buckets(ctx, &batch);
    if (!rc) rc = bce_scan_feed_buckets(s, &batch);
    if (rc) { delete s->s; delete s; bce_gpu_set_emit_mode(ctx, BCE_EMIT_RAW, nullptr); return rc; }
  } while (!batch.done);
  bce_gpu_set_emit_mode(ctx, BCE_EMIT_RAW, nullptr);
  return bce_scan_finish(s, cfg288_out);
}
#endif

}  // extern "C"
