// decode.cpp -- see decode.hpp.
#include "decode.hpp"

#include <array>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <cstdio>
#include <thread>
#include <cstdlib>
#include <memory>
#include <new>

#include "../../../include/bce_gpu.h"
#include "coders.hpp"

namespace bcehost {

// The reference shifts 64-bit values by amounts that can reach or exceed 64 (bce.cpp:175-176,
// undefined behaviour in C++, SURVEY.md Q6).  Archives only decode identically if those shifts
// behave like the x86 SHL instruction the reference was compiled to: the count is taken mod 64.
static inline uint64_t shl_x86(uint64_t v, uint64_t count) { return v << (count & 63u); }

uint32_t DecodeRank::ones_before(uint32_t pos) const {
  if (pos > n_) pos = n_;
  const uint64_t w = w_[pos / 32];
  const uint32_t below = uint32_t(w >> 32) & uint32_t((1ull << (pos % 32)) - 1);
  return uint32_t(w) + uint32_t(__builtin_popcount(below));
}

void DecodeRank::pin(uint32_t pos, uint32_t ones) {
  if (pos > n_) return;
  uint64_t need = uint32_t(ones - ones_before(pos));      // ones that still have to move in front of pos
  if (need == 0) return;
  const uint64_t word = pos / 32, o = pos % 32;
  uint64_t b = w_[word];
  const uint32_t base = uint32_t(b);
  if (uint64_t(base) + o + 32 < need) {                    // more than this word can ever show: the
    b += need - o - base;                                  // surplus lives in the base count only (:166-169)
    need = o;
  }
  const uint64_t above = ~0ull << (32 + o);                // data bits at and after pos
  const uint64_t take_at = uint64_t(__builtin_ctzll(((b & above) >> 32) | (1ull << 31)));   // :172
  // :173.  ~(b | above) is 0 only in a damaged archive (a base count of 0xFFFFFFFF while need > 0), where
  // __builtin_clzll is undefined: define it as 64, as the device decoder (decode_many.cu) does
  const uint64_t hole = ~(b | above);
  const uint64_t put_end = 64 - uint64_t(hole ? __builtin_clzll(hole) : 64);
  const uint64_t take = (shl_x86(1, take_at + need) - shl_x86(1, take_at)) << 32;           // :175
  const uint64_t put = shl_x86(1, put_end) - shl_x86(1, put_end - need);                    // :176
  b += uint64_t(__builtin_popcount(uint32_t(put)));        // what falls below data bit 0 goes to the base count
  b &= ~take;
  b |= (put >> 32) << 32;
  w_[word] = b;
}

void DecodeRank::finish() {
  for (size_t i = 0; i + 1 < w_.size(); ++i) {
    const uint32_t here = uint32_t(w_[i]) + uint32_t(__builtin_popcountll(w_[i] >> 32));
    const uint32_t next = uint32_t(w_[i + 1]);
    w_[i] |= uint64_t(uint32_t(next - here)) << 63;
  }
}

namespace {

struct Node { uint32_t s, x0, x1; };

// One node of the decode loop (the body of BCE::code with mode = 0, bce.cpp:1259-1352).
// Returns false when a count falls outside the interval the dictionary allows (damaged archive).
inline bool decode_node(const Node& nd, StreamDecoder& dec, DecodeRank& R, uint32_t one_base, uint32_t n,
                        std::array<std::vector<Node>, 2>& out) {
  const uint32_t s = nd.s, x0 = nd.x0, x1 = nd.x1, x = x0 + x1;
  if (!x0 || !x1 || uint64_t(s) + x0 + x1 > n) return false;       // every node is an interval inside [0, n)
  const uint32_t s1 = R.ones_before(s);                               // :1265
  const uint32_t c1 = R.ones_before(s + x) - s1;                      // _1x :1271
  if (s1 > s || c1 > x) return false;
  const uint32_t s0 = s - s1;
  if (c1 == 0) {                                                      // :1274-1279
    out[0].push_back({s0, x0, x1});
    R.pin(s + x0, s1);
    return true;
  }
  const uint32_t c0 = x - c1;
  if (c0 == 0) {                                                      // :1282-1287
    out[1].push_back({one_base + s1, x0, x1});
    R.pin(s + x0, s1 + x0);
    return true;
  }
  const uint32_t lo = x0 > c1 ? x0 - c1 : 0u;                         // :1290-1294
  const uint32_t hi = x0 - (c1 > x1 ? c1 - x1 : 0u);
  if (hi < lo) return false;
  uint32_t z0 = lo;                                                   // _0x0
  if (hi != lo) z0 = lo + dec.count(hi - lo + 1, c0, x1, x);          // :1304
  if (z0 > hi || z0 > c0) return false;
  const uint32_t z1 = c0 - z0;                                        // :1337
  if (z0 && z1) out[0].push_back({s0, z0, z1});
  if (z1 > x1 || x1 - z1 > c1) return false;
  const uint32_t o1 = x1 - z1, o0 = c1 - o1;                          // :1343-1344
  if (o0 && o1) out[1].push_back({one_base + s1, o0, o1});
  R.pin(s + x0, s1 + o0);                                             // :1350
  return true;
}

// barrier for the 8 level threads: spins for the common short wait, then sleeps on a condition
// variable so that a box with fewer free cores than levels is not burnt by polling
class LevelBarrier {
 public:
  explicit LevelBarrier(int parties) : parties_(parties) {}
  void wait() {
    const uint32_t gen = gen_.load(std::memory_order_acquire);
    if (count_.fetch_add(1, std::memory_order_acq_rel) + 1 == parties_) {
      count_.store(0, std::memory_order_relaxed);
      {
        std::lock_guard<std::mutex> g(m_);
        gen_.store(gen + 1, std::memory_order_release);
      }
      cv_.notify_all();
      return;
    }
    for (int spins = 0; spins < 4000; ++spins)
      if (gen_.load(std::memory_order_acquire) != gen) return;
    std::unique_lock<std::mutex> lk(m_);
    cv_.wait(lk, [&] { return gen_.load(std::memory_order_acquire) != gen; });
  }

 private:
  const int parties_;
  std::atomic<int> count_{0};
  std::atomic<uint32_t> gen_{0};
  std::mutex m_;
  std::condition_variable cv_;
};

// BCE::code with mode = 0, bce.cpp:1236-1373: per round, per level, zero-half then one-half,
// ascending position; every count comes from the level's own decoder.  A level only touches its
// own decoder, its own dictionary and its own output lists, so -- like the reference's
// `omp parallel for` over the levels (:1250) -- the 8 levels of a round run on 8 threads.
bool decode_levels(std::array<std::unique_ptr<StreamDecoder>, 8>& dec, const std::array<uint32_t, 8>& C,
                   std::vector<DecodeRank>& ranks, uint32_t n, int threads) {
  std::array<std::array<std::vector<Node>, 2>, 8> cur, nxt;
  for (int i = 0; i < 8; ++i)
    if (C[i] && n - C[i]) cur[i][0].push_back({0, C[i], n - C[i]});          // :1238-1240
  std::atomic<uint64_t> visits{0};
  std::atomic<bool> bad{false};

  auto run_level = [&](int i) {                       // one level of one round
    uint64_t mine = 0;
    for (int half = 0; half < 2; ++half) {
      const std::vector<Node>& list = cur[i][half];
      const size_t count = list.size();
      for (size_t j = 0; j < count; ++j) {
        if (j + 12 < count) {                         // the three words node j+12 will read and rewrite
          const Node& f = list[j + 12];
          ranks[i].prefetch(f.s);
          ranks[i].prefetch(f.s + f.x0);
          ranks[i].prefetch(f.s + f.x0 + f.x1);
        }
        ++mine;
        if (!decode_node(list[j], *dec[i], ranks[i], C[(i + 1) % 8], n, nxt[i])) { bad.store(true); return; }
      }
    }
    // a well-formed archive visits 8(n-1) nodes in total
    if (visits.fetch_add(mine) + mine > 8ull * n) bad.store(true);
  };

  if (threads < 2) {
    bool again = true;
    while (again && !bad.load()) {
      again = false;
      for (int i = 0; i < 8; ++i) run_level(i);
      for (int i = 0; i < 8; ++i) { cur[i][0].clear(); cur[i][1].clear(); }
      for (int i = 0; i < 8; ++i) {                                           // :1361-1370
        const int d = (i + 1) % 8;
        for (int half = 0; half < 2; ++half) {
          cur[d][half].swap(nxt[i][half]);
          nxt[i][half].clear();
          if (!cur[d][half].empty()) again = true;
        }
      }
    }
    return !bad.load();
  }

  LevelBarrier barrier(8);
  std::atomic<int> live{1};                           // some level has nodes for the coming round
  auto worker = [&](int i) {
    for (;;) {
      run_level(i);
      barrier.wait();                                 // every level of this round is done
      const bool damaged = bad.load();                // nobody writes it until the next run_level
      if (i == 0) live.store(0);
      cur[i][0].clear();
      cur[i][1].clear();
      barrier.wait();                                 // old lists cleared before anybody refills them
      const int d = (i + 1) % 8;
      for (int half = 0; half < 2; ++half) {          // :1361-1370
        cur[d][half].swap(nxt[i][half]);
        if (!cur[d][half].empty()) live.store(1);
      }
      barrier.wait();
      if (!live.load() || damaged) return;
    }
  };
  std::vector<std::thread> pool;
  for (int i = 1; i < 8; ++i) pool.emplace_back(worker, i);
  worker(0);
  for (auto& t : pool) t.join();
  return !bad.load();
}

}  // namespace

int default_level_threads() {
  int threads = std::thread::hardware_concurrency() >= 4 ? 8 : 1;
  if (const char* v = std::getenv("BCE_HOST_THREADS")) threads = std::atoi(v);
  return threads;
}

int archive_size(const uint16_t* a, size_t len, uint32_t& n) {
  if (len == 0) return BCE_GPU_E_ARG;
  const size_t header_words = a[0];                                           // :1178
  if (1 + header_words > len) return BCE_GPU_E_ARG;
  StreamDecoder header(-1, a + 1, header_words);                              // :1179
  n = header.varint();                                                        // :1181
  return n == 0 ? BCE_GPU_E_ARG : BCE_GPU_OK;
}

int decode_to_ranks(const uint16_t* a, size_t len, std::vector<DecodeRank>& ranks, uint32_t& n, uint32_t& offset,
                    int threads) {
  if (len == 0) return BCE_GPU_E_ARG;
  const size_t header_words = a[0];                                           // :1178
  if (1 + header_words > len) return BCE_GPU_E_ARG;
  StreamDecoder header(-1, a + 1, header_words);                              // :1179
  n = header.varint();                                                        // :1181
  if (n == 0) return BCE_GPU_E_ARG;
  if (const char* cap = std::getenv("BCE_HOST_MAX_N"))                        // refuse absurd sizes early (tests, services)
    if (uint64_t(n) > std::strtoull(cap, nullptr, 10)) return BCE_GPU_E_ARG;
  offset = header.uniform(n + 1);
  if (offset > n) return BCE_GPU_E_ARG;
  uint32_t size = header.varint();
  std::array<size_t, 9> at{};
  at[0] = 1 + header_words;
  for (int i = 0; i < 7; ++i) {                                               // :1187-1190
    const uint32_t len = header.uniform(size + 1);
    if (len > size) return BCE_GPU_E_ARG;
    at[i + 1] = at[i] + len;
    size -= len;
  }
  at[8] = len;
  for (int i = 0; i < 8; ++i)
    if (at[i + 1] < at[i] || at[i + 1] > len) return BCE_GPU_E_ARG;
  std::array<std::unique_ptr<StreamDecoder>, 8> dec;
  for (int i = 0; i < 8; ++i) dec[i].reset(new StreamDecoder(i, a + at[i], at[i + 1] - at[i]));   // :1193-1202

  ranks.clear();
  for (int i = 0; i < 8; ++i) ranks.emplace_back(n);                          // :1205
  std::array<uint32_t, 8> C;
  for (int i = 0; i < 8; ++i) {                                               // :1208-1211
    C[i] = dec[i]->uniform(n + 1);
    if (C[i] > n) return BCE_GPU_E_ARG;
    ranks[(i + 7) % 8].pin(n, n - C[i]);
  }
  if (!decode_levels(dec, C, ranks, n, threads)) return BCE_GPU_E_ARG;        // :1218
  for (auto& r : ranks) r.finish();                                           // :1220-1223
  return BCE_GPU_OK;
}

std::vector<uint8_t> unbwt_serial(const std::vector<DecodeRank>& ranks, uint32_t offset, uint32_t n) {
  std::vector<uint8_t> out(n);
  uint32_t zeros[8];
  for (int j = 0; j < 8; ++j) zeros[j] = ranks[j].zeros_before(n);            // :1006-1015
  uint64_t s = 0;
  for (uint64_t i = n; i-- > 0;) {                                            // :1019-1029
    uint32_t chr = 0;
    for (int j = 0; j < 8; ++j) {
      const uint32_t b = ranks[j].bit(uint32_t(s));
      chr |= b << j;
      s = b ? zeros[j] + ranks[j].ones_before(uint32_t(s)) : ranks[j].zeros_before(uint32_t(s));
    }
    out[(i + offset) % n] = uint8_t(chr);
  }
  return out;
}

int decode_archive(std::vector<uint16_t>& archive, bool low_memory, std::vector<uint8_t>& out) {
  std::vector<DecodeRank> ranks;
  uint32_t n = 0, offset = 0;
  using clk = std::chrono::steady_clock;
  const bool timing = std::getenv("BCE_TIME") != nullptr;
  const auto t0 = clk::now();
  int rc;
  try {
    rc = decode_to_ranks(archive.data(), archive.size(), ranks, n, offset, default_level_threads());
  } catch (const std::bad_alloc&) {
    return BCE_GPU_E_NOMEM;
  } catch (...) {                                                             // e.g. std::system_error from a level worker thread
    return BCE_GPU_E_INTERNAL;
  }
  if (rc) return rc;
  const auto t1 = clk::now();
  if (timing) std::fprintf(stderr, "[bce] decode loop %.3f s (n = %u)\n", std::chrono::duration<double>(t1 - t0).count(), n);
  std::vector<uint16_t>().swap(archive);                                      // :1203
  if (low_memory) {
    try { out = unbwt_serial(ranks, offset, n); }
    catch (const std::bad_alloc&) { return BCE_GPU_E_NOMEM; }
    return BCE_GPU_OK;
  }
  bce_gpu_ctx* ctx = nullptr;
  rc = bce_gpu_open(0, &ctx);
  if (rc) return rc;
  const uint64_t* lv[8];
  for (int j = 0; j < 8; ++j) lv[j] = ranks[j].words().data();
  try { out.resize(n); }
  catch (const std::bad_alloc&) { bce_gpu_close(ctx); return BCE_GPU_E_NOMEM; }
  const auto t2 = clk::now();
  rc = bce_gpu_unbwt(ctx, lv, offset % n, n, out.data());                     // unbwt::bytewise, :1043-1103
  const auto t3 = clk::now();
  bce_gpu_close(ctx);
  if (timing)
    std::fprintf(stderr, "[bce] open device %.3f s | inverse BWT %.3f s | close device %.3f s\n",
                 std::chrono::duration<double>(t2 - t1).count(), std::chrono::duration<double>(t3 - t2).count(),
                 std::chrono::duration<double>(clk::now() - t3).count());
  return rc;
}

}  // namespace bcehost
