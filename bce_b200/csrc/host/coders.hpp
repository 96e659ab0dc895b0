// coders.hpp -- host-side entropy coders of BCE v0.4, behaviourally identical to the
// reference (archives must be bit-exact drop-ins) but written from the behavioural spec in
// SURVEY.md Appendix A rather than transcribed:
//
//   RangeEncoder / RangeDecoder   64-bit carry-less range coder with 16-bit output words
//                                 (bce.cpp:538-553, :592-615, :655-669)
//   ContextModel                  adaptive byte counters per (k, quantised c1/cs, c2/cs)
//                                 (bce.cpp:671-677, :700-705, :531-533)
//   StreamEncoder / StreamDecoder the AdaptiveCoder<31> policy: config prefix, uniform and
//                                 adaptive symbols, k > 31 binary decomposition, varints
//                                 (bce.cpp:484-724, VCoder :362-378)
//   ScanCollector                 the ScanCoder<31> policy for `bce -s` (bce.cpp:726-834)
//
// They are serial per stream, so one file's eight streams stay on the host.  Many small inputs have eight streams
// each, enough to fill a GPU with one coder per warp: csrc/code_many.cu restates the encoders for the device
// (bce_gpu_compress_many_archives), and the arithmetic of both must stay the same.
#pragma once

#include "../../../include/bce_gpu.h"

#include <array>
#include <cstdint>
#include <string>
#include <unordered_map>
#include <vector>

namespace bcehost {

constexpr int kMaxAdaptive = 31;               // AdaptiveCoder<31>::max, bce.cpp:1381
constexpr int kConfigRows = 9;                 // streams 0..7 + header row 8
constexpr int kConfigCols = kMaxAdaptive + 1;
using ConfigTable = std::array<std::array<uint8_t, kConfigCols>, kConfigRows>;

const ConfigTable& default_config();            // bce.cpp:713-724
// bce -c ... cfg: 288 bytes; wrong size / unreadable is non-fatal and prints the reference's
// message (bce.cpp:626-641).  Returns true when the table was replaced.
bool load_config_file(const std::string& path, ConfigTable& table);
bool save_config_file(const std::string& path, const ConfigTable& table);   // bce.cpp:810-813

class RangeEncoder {
 public:
  void put_uniform(uint32_t sym, uint32_t range);                 // set(s, k)
  void put(uint32_t cum, uint32_t freq, uint32_t total);          // coding step of set(s,k,c1,c2,cs)
  void finish();                                                  // flush()
  const std::vector<uint16_t>& words() const { return out_; }
  std::vector<uint16_t>& words() { return out_; }

 private:
  void renormalise();
  void restart_if_narrow(uint64_t total);
  uint64_t lo_ = 0, hi_ = ~0ull;
  std::vector<uint16_t> out_;
};

class RangeDecoder {
 public:
  RangeDecoder() = default;
  RangeDecoder(const uint16_t* words, size_t count);
  uint32_t get_uniform(uint32_t range);
  // adaptive step: walks the cumulative frequencies of row[0..k) like bce.cpp:573-581
  uint32_t get(const uint8_t* row, uint32_t k, uint32_t total);

 private:
  uint16_t next() { return pos_ < count_ ? words_[pos_++] : 0; }
  void renormalise();
  void restart_if_narrow(uint64_t total);
  const uint16_t* words_ = nullptr;
  size_t count_ = 0, pos_ = 0;
  uint64_t lo_ = 0, hi_ = ~0ull, code_ = 0;
};

class ContextModel {
 public:
  void configure(const std::array<uint8_t, kConfigCols>& bits);   // bce.cpp:700-705
  // counters of the context (k, c1, c2, cs); uint32 wrap-around as in bce.cpp:674.
  // A row is k one-byte counters followed by their sum as a uint16 (kept up to date by bump), so that a
  // symbol costs one load for the total instead of k adds; the layout is internal, the counters and every
  // coded interval are the reference's.
  uint8_t* row(uint32_t k, uint32_t c1, uint32_t c2, uint32_t cs) {
    const uint32_t o = off_[k], b = o >> 24;
    const uint32_t ctx = (((c1 << b) / cs) << b) | ((c2 << b) / cs);
    return stat_.data() + (o & 0x00FFFFFFu) + size_t(ctx) * (k + 2);
  }
  // same counters addressed by a context index computed elsewhere (packed device words)
  uint8_t* row_at(uint32_t k, uint32_t ctx) { return stat_.data() + (off_[k] & 0x00FFFFFFu) + size_t(ctx) * (k + 2); }
  static uint32_t sum(const uint8_t* row, uint32_t k) { return uint32_t(row[k]) | (uint32_t(row[k + 1]) << 8); }
  static void bump(uint8_t* row, uint32_t k, uint32_t sym) {      // bce.cpp:531-533
    uint32_t s = sum(row, k) + 1;
    if (++row[sym] == 0xFF) {
      s = 0;
      for (uint32_t i = 0; i < k; ++i) { row[i] >>= 1; s += row[i]; }
    }
    row[k] = uint8_t(s);
    row[k + 1] = uint8_t(s >> 8);
  }
  size_t table_bytes() const { return stat_.size(); }

 private:
  std::array<uint32_t, kConfigCols> off_{};
  std::vector<uint8_t> stat_;
};

class StreamEncoder {
 public:
  StreamEncoder(int id, const ConfigTable& cfg);                  // AdaptiveCoder(int), init(1, i)
  void uniform(uint32_t sym, uint32_t range) { rc_.put_uniform(sym, range); }
  void count(uint32_t sym, uint32_t k, uint32_t c1, uint32_t c2, uint32_t cs);
  void varint(uint32_t v);                                        // VCoder::setv
  // BCE_EMIT_CODER words (include/bce_gpu.h): context index and k > 31 halving done on the device
  void packed(const uint32_t* words, size_t count);
  void packed20(const uint8_t* bytes, size_t count);              // the same words, 20 bits each (bce_cse_words20)
  void finish() { rc_.finish(); }
  const std::vector<uint16_t>& words() const { return rc_.words(); }

 private:
  RangeEncoder rc_;
  ContextModel model_;
};

class StreamDecoder {
 public:
  StreamDecoder(int id, const uint16_t* words, size_t count);     // reads its config row back
  uint32_t uniform(uint32_t range) { return rd_.get_uniform(range); }
  uint32_t count(uint32_t k, uint32_t c1, uint32_t c2, uint32_t cs);
  uint32_t varint();                                              // VCoder::getv (at most 31 bits)

 private:
  RangeDecoder rd_;
  ContextModel model_;
};

// `bce -s`: records every adaptive symbol per context, then picks for every k the number of
// context bits (0..5) that minimises the simulated adaptive code length.
// host-side packer with the device's word formats (tests, and callers that hold raw counts)
size_t pack_count(int mode, const uint8_t* bits_row, uint32_t sym, uint32_t k, uint32_t c1, uint32_t c2,
                  uint32_t cs, uint32_t out[3]);

class ScanCollector {
 public:
  explicit ScanCollector(int id) : row_(id < 0 || id > 7 ? 8 : id) {}
  void count(uint32_t sym, uint32_t k, uint32_t c1, uint32_t c2, uint32_t cs);   // bce.cpp:737-744
  void packed(const uint32_t* words, size_t count);                              // BCE_EMIT_SCAN words
  // a batch bucketed on the device (bce_gpu_cse_next_buckets): runs of symbol bytes per (k, key)
  void bucketed(const uint8_t* syms, size_t count, const bce_scan_bucket* buckets, size_t nbuckets, uint64_t halvings);
  // bce.cpp:751-800: fills table[row] and prints "Result size: %.1f B"
  void finish(ConfigTable& table);

 private:
  std::array<std::unordered_map<uint32_t, std::vector<uint8_t>>, kMaxAdaptive + 1> stat_;
  double nats_ = 0;
  int row_;
};

}  // namespace bcehost
