// decode.hpp -- host side of `bce -d` / `bce -ds`: archive -> rank dictionaries -> text.
//
// BCE::decode (bce.cpp:1169-1233) stays host code by nature: the CSE loop in decode mode
// (bce.cpp:1236-1373 with mode = 0) asks the arithmetic decoder for every count and feeds it
// back into the rank dictionary it is walking, one stream after the other.  What follows the
// loop -- unbwt::bytewise (bce.cpp:1043-1103) -- is the data-parallel part and runs on the GPU
// (bce_gpu_unbwt); `-ds` keeps the serial unbwt::bitwise (bce.cpp:999-1038) on the host.
#pragma once

#include <cstdint>
#include <vector>

#include "../format.h"

namespace bcehost {

// The decoder's rank dictionary (class Rank, bce.cpp:130-219, write side :153-194).
// Word = [32 data bits | 32-bit count of ones before the word].  While decoding, only the
// positions that were pinned with pin() answer ones_before() exactly; the ones of a known
// interval sit right-aligned against its upper boundary, and what does not fit into the word of
// that boundary is only accounted for in the word's base count.  finish() derives the last bit
// of every word from the next word's base count.
class DecodeRank {
 public:
  explicit DecodeRank(uint32_t n) : w_(size_t(n) / 32 + 1, 0), n_(n) {}
  // positions are clamped to [0, n]: a corrupt archive must not read outside the dictionary
  uint32_t ones_before(uint32_t pos) const { return bcefmt::ones_before(w_.data(), n_, pos); }   // Rank::get<1>
  uint32_t zeros_before(uint32_t pos) const { return pos - ones_before(pos); }
  uint32_t bit(uint32_t pos) const {
    if (pos > n_) pos = n_;
    return uint32_t(w_[pos / 32] >> (pos % 32 + 32)) & 1u;
  }
  void prefetch(uint32_t pos) const { __builtin_prefetch(&w_[(pos > n_ ? n_ : pos) / 32], 1); }
  void pin(uint32_t pos, uint32_t ones) {              // Rank::set, :153-185
    uint64_t b;
    if (bcefmt::pin_word(w_.data(), n_, pos, ones, b)) w_[pos / 32] = b;
  }
  void finish() {                                      // Rank::finalize, :187-194
    for (size_t i = 0; i + 1 < w_.size(); ++i) w_[i] = bcefmt::finish_word(w_[i], uint32_t(w_[i + 1]));
  }
  const std::vector<uint64_t>& words() const { return w_; }

 private:
  std::vector<uint64_t> w_;
  uint32_t n_;
};

// Decodes a whole archive (uint16 words as read from the file).  low_memory = `-ds`: serial
// inverse on the host; otherwise the inverse BWT runs on the GPU through bce_gpu_unbwt.
// Returns 0, or a negative bce_gpu error code (BCE_GPU_E_ARG for an archive that is not one:
// every count that comes out of the decoders is checked against the interval it must lie in, so a
// damaged archive ends in an error, never in an out-of-bounds access or an endless loop).
int decode_archive(std::vector<uint16_t>& archive, bool low_memory, std::vector<uint8_t>& out);

// Only the host half: header + 8 streams (archive words a[0 .. len)) -> the 8 rank dictionaries (after finish()),
// n, offset.  threads >= 2 decodes the 8 levels of a round on 8 threads, else on the calling thread.
int decode_to_ranks(const uint16_t* a, size_t len, std::vector<DecodeRank>& ranks, uint32_t& n, uint32_t& offset,
                    int threads);
// The level-thread count `bce -d` uses: 8 on a machine with at least 4 hardware threads, else 1 (BCE_HOST_THREADS
// overrides it).
int default_level_threads();
// n from an archive's header alone (0 or BCE_GPU_E_ARG), to pick a decoder before decoding.
int archive_size(const uint16_t* a, size_t len, uint32_t& n);

// unbwt::bitwise, bce.cpp:999-1038
std::vector<uint8_t> unbwt_serial(const std::vector<DecodeRank>& ranks, uint32_t offset, uint32_t n);

}  // namespace bcehost
