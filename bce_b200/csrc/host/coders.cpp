// coders.cpp -- see coders.hpp.  Every routine names the reference lines whose behaviour it
// reproduces (bce.cpp:line); the arithmetic must match bit for bit.
#include "coders.hpp"

#include <algorithm>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>

namespace bcehost {

// ---- configuration table ---------------------------------------------------------------------------------------
const ConfigTable& default_config() {
  static const ConfigTable t = [] {
    ConfigTable c;
    std::memcpy(c.data(), bcefmt::kDefaultConfig, sizeof bcefmt::kDefaultConfig);
    return c;
  }();
  return t;
}

bool load_config_file(const std::string& path, ConfigTable& table) {
  std::ifstream f(path, std::ios::binary | std::ios::ate);
  const std::streamoff size = f ? std::streamoff(f.tellg()) : -1;
  if (size != std::streamoff(kConfigRows * kConfigCols)) {          // bce.cpp:629-632
    std::printf("Config not found or wrong size.\n");
    return false;
  }
  f.seekg(0, std::ios::beg);
  ConfigTable tmp;
  if (!f.read(reinterpret_cast<char*>(tmp.data()), size)) {         // bce.cpp:636-639
    std::printf("Could not read Config.\n");
    return false;
  }
  if (!bcefmt::config_ok(tmp[0].data(), kConfigRows * kConfigCols)) {
    std::printf("Config holds context bits above 5; ignored.\n");
    return false;
  }
  table = tmp;
  return true;
}

bool save_config_file(const std::string& path, const ConfigTable& table) {
  std::ofstream f(path, std::ios::binary | std::ios::trunc);
  f.write(reinterpret_cast<const char*>(table.data()), kConfigRows * kConfigCols);
  return bool(f);
}

// ---- range coder -----------------------------------------------------------------------------------------------
uint32_t RangeDecoder::get(const uint8_t* row, uint32_t k, uint32_t total) {   // bce.cpp:573-581
  restart_if_narrow(total);
  const uint64_t step = (hi - lo) / total;
  uint64_t top = lo - 1;                        // wraps exactly like the reference when lo == 0
  uint64_t bottom = lo;
  uint32_t sym = 0;
  for (;; ++sym) {
    bottom = top + 1;
    top += step * (uint64_t(row[sym]) + 1);
    if (!(top < code) || sym + 1 >= k) break;  // the bound only matters for corrupt archives
  }
  lo = bottom;
  hi = top;
  // the reference bumps the counter before shift_in (:583-587); the two do not interact
  renormalise();
  return sym;
}

// ---- adaptive model --------------------------------------------------------------------------------------------
StreamEncoder::StreamEncoder(int id, const ConfigTable& cfg) {
  const auto& bits = cfg[(id < 0 || id > 7) ? 8 : id];              // bce.cpp:683-684
  rc_.put_config(bits.data());
  model_.configure(bits.data());
}

void StreamEncoder::count(uint32_t sym, uint32_t k, uint32_t c1, uint32_t c2, uint32_t cs) {
  while (k > uint32_t(kMaxAdaptive)) {                              // bce.cpp:507-510
    rc_.put_uniform(sym & 1u, 2);
    k = (k + (~sym & 1u)) >> 1;
    sym >>= 1;
  }
  uint8_t* row = model_.row(k, c1, c2, cs);
  uint32_t below = sym, total = k;                                  // bce.cpp:514-518
  for (uint32_t i = 0; i < sym; ++i) below += row[i];
  total += ContextModel::sum(row, k);
  rc_.put(below, uint32_t(row[sym]) + 1, total);
  ContextModel::bump(row, k, sym);
}

// Packed counts (include/bce_gpu.h, BCE_EMIT_CODER): W(j) reads word j; codes the counts that START in [first, count)
// and returns the index behind the last word used (a k > 31 count at the end reaches up to two words past `count`).
template <class W>
static inline size_t code_packed(RangeEncoder& rc, ContextModel& model, size_t first, size_t count, W word) {
  size_t i = first;
  for (; i < count; ++i) {
    uint32_t sym, k, ctx;
    bcefmt::coder_fields(word(i), sym, k, ctx);
    if (k == 0) {                                                   // k > 31: nb uniform bits first (bce.cpp:507-510)
      const uint32_t w1 = word(i + 1), w2 = word(i + 2);
      i += 2;
      uint32_t nb, low;
      bcefmt::coder_escape(w1, w2, k, nb, low);
      for (uint32_t j = 0; j < nb; ++j) rc.put_uniform((low >> j) & 1u, 2);
    }
    uint8_t* row = model.row_at(k, ctx);
    uint32_t below = sym, total = k;                                // bce.cpp:514-518
    for (uint32_t j = 0; j < sym; ++j) below += row[j];
    total += ContextModel::sum(row, k);
    rc.put(below, uint32_t(row[sym]) + 1, total);
    ContextModel::bump(row, k, sym);
  }
  return i;
}

void StreamEncoder::packed(const uint32_t* words, size_t count) {
  code_packed(rc_, model_, 0, count, [words](size_t j) { return words[j]; });
}

// 20-bit words (bce_cse_words20): unpacked a block at a time into aligned words -- one 8-byte load per pair in a
// loop of its own -- so that the coder's loop reads what it reads in the 32-bit form.
void StreamEncoder::packed20(const uint8_t* b, size_t count) {
  constexpr size_t BLK = 4096;                                      // even: a block starts on a 5-byte group
  uint32_t buf[BLK + 4];
  size_t skip = 0;                                                  // words of this block already used by the last count of the previous one
  for (size_t base = 0; base < count; base += BLK) {
    const size_t n = std::min(BLK, count - base), m = std::min(n + 2, count - base);
    const uint8_t* p = b + 5 * (base >> 1);
    for (size_t t = 0; t < m; t += 2, p += 5) {                     // (8 bytes past the last word are readable)
      uint64_t v;
      memcpy(&v, p, 8);
      buf[t] = uint32_t(v) & 0xFFFFFu;
      buf[t + 1] = uint32_t(v >> 20) & 0xFFFFFu;
    }
    const uint32_t* w = buf;
    const size_t end = code_packed(rc_, model_, skip, n, [w](size_t j) { return w[j]; });
    skip = end - n;
  }
}

StreamDecoder::StreamDecoder(const uint16_t* words, uint32_t count) : rd_(words, count) {
  model_.configure(rd_);                                            // bce.cpp:693-697
}

uint32_t StreamDecoder::count(uint32_t k, uint32_t c1, uint32_t c2, uint32_t cs) {   // bce.cpp:555-590
  if (k > uint32_t(kMaxAdaptive)) {
    const uint32_t low = rd_.get_uniform(2);
    return (count((k + (~low & 1u)) >> 1, c1, c2, cs) << 1) | low;
  }
  uint8_t* row = model_.row(k, c1, c2, cs);
  uint32_t total = k;
  total += ContextModel::sum(row, k);
  const uint32_t sym = rd_.get(row, k, total);
  ContextModel::bump(row, k, sym);
  return sym;
}

// ---- scan policy -----------------------------------------------------------------------
void ScanCollector::count(uint32_t sym, uint32_t k, uint32_t c1, uint32_t c2, uint32_t cs) {
  while (k > uint32_t(kMaxAdaptive)) {                              // bce.cpp:738-741 (note: not :509's halving)
    nats_ += std::log(2);
    k = (k >> 1) + (~sym & 1u);
    sym >>= 1;
  }
  stat_[k][(((c2 << 8) / cs) << 16) | ((c1 << 8) / cs)].push_back(uint8_t(sym));   // bce.cpp:743
}

void ScanCollector::packed(const uint32_t* words, size_t count) {
  for (size_t i = 0; i < count; ++i) {
    const uint32_t w = words[i], b = bcefmt::scan_bucket(w);
    if (w >> 31)
      for (uint32_t nb = (w >> 26) & 31u; nb; --nb) nats_ += std::log(2);         // one addition per halving, as :739
    stat_[bcefmt::bucket_k(b)][bcefmt::bucket_key(b)].push_back(uint8_t(w & 31u));
  }
}

// The same state the calls of count() in stream order would leave.  What flush() (below) reads is, per (k, key), the
// symbols in insertion order -- the runs arrive in that order, the device sort is stable and batches are fed in
// order -- and, because it walks an unordered_map, the ORDER IN WHICH THE KEYS OF ONE k WERE FIRST INSERTED
// (libstdc++ links a new node at the head of its bucket; later insertions into an existing key change nothing):
// new keys are inserted by ascending position of their first count.  nats_ only ever receives log 2 before flush
// (:739), so `halvings` equal additions reproduce it exactly.
void ScanCollector::bucketed(const uint8_t* syms, size_t count, const bce_scan_bucket* buckets, size_t nbuckets,
                             uint64_t halvings) {
  for (uint64_t i = 0; i < halvings; ++i) nats_ += std::log(2);
  if (!nbuckets) return;
  std::vector<bce_scan_bucket> by_first(buckets, buckets + nbuckets), by_start(buckets, buckets + nbuckets);
  std::sort(by_first.begin(), by_first.end(), [](const bce_scan_bucket& a, const bce_scan_bucket& b) { return a.first < b.first; });
  std::sort(by_start.begin(), by_start.end(), [](const bce_scan_bucket& a, const bce_scan_bucket& b) { return a.start < b.start; });
  for (const bce_scan_bucket& b : by_first)                                    // first appearances, in stream order
    stat_[bcefmt::bucket_k(b.key)][bcefmt::bucket_key(b.key)];
  for (size_t j = 0; j < by_start.size(); ++j) {
    const uint32_t key = by_start[j].key;
    const size_t a = by_start[j].start, e = j + 1 < by_start.size() ? by_start[j + 1].start : count;
    std::vector<uint8_t>& v = stat_[bcefmt::bucket_k(key)][bcefmt::bucket_key(key)];
    v.insert(v.end(), syms + a, syms + e);
  }
}

void ScanCollector::finish(ConfigTable& table) {                    // bce.cpp:751-800
  std::vector<uint16_t> sim;
  for (uint32_t k = 2; k < uint32_t(kMaxAdaptive); ++k) {
    double best = 0;
    for (auto& kv : stat_[k]) best += std::log(k) * kv.second.size();
    for (uint32_t bits = 0; bits <= 5; ++bits) {
      sim.assign(size_t(k) << (2 * bits), 0);
      double z = 0;
      for (auto& kv : stat_[k]) {
        uint32_t key = kv.first;
        uint16_t q1 = uint16_t(key), q2 = uint16_t(key >> 16);
        q1 >>= 8 - bits;
        q2 >>= 8 - bits;
        uint16_t* ctx = &sim[size_t((uint32_t(q1) << bits) | q2) * k];
        for (uint8_t s : kv.second) {
          uint32_t total = k;
          for (uint32_t i = 0; i < k; ++i) total += ctx[i];
          z += std::log(static_cast<double>(total) / (1 + ctx[s]));
          if (++ctx[s] == 0xFF)
            for (uint32_t i = 0; i < k; ++i) ctx[i] >>= 1;
        }
      }
      if (z < best) {
        best = z;
        table[row_][k] = uint8_t(bits);
      }
    }
    nats_ += best;
  }
  std::printf("Result size: %.1f B\n", nats_ / std::log(256));
}

}  // namespace bcehost
