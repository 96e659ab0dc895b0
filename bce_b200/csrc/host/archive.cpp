// archive.cpp -- see archive.hpp.
#include "archive.hpp"

#include <chrono>
#include <thread>

namespace bcehost {

ArchiveWriter::ArchiveWriter(uint32_t n, const uint32_t C[8], const ConfigTable& cfg) : n_(n), cfg_(cfg) {
  for (int i = 0; i < 8; ++i) {
    streams_.emplace_back(new StreamEncoder(i, cfg_));              // bce.cpp:1124
    streams_[i]->uniform(C[i], n + 1);                              // bce.cpp:1129
  }
}

static void code_stream(StreamEncoder* enc, const bce_tuple* t, size_t count) {
  for (size_t j = 0; j < count; ++j) enc->count(t[j].sym, t[j].k, t[j].c1, t[j].c2, t[j].cs);   // bce.cpp:1302
}

void ArchiveWriter::feed(const bce_cse_batch& batch, int threads) {
  if (threads <= 1) {
    for (int i = 0; i < 8; ++i) code_stream(streams_[i].get(), batch.tuples[i], batch.count[i]);
    return;
  }
  // the streams are independent coders; the reference forks over them the same way (bce.cpp:1250)
  std::vector<std::thread> pool;
  for (int i = 0; i < 8; ++i)
    if (batch.count[i]) pool.emplace_back(code_stream, streams_[i].get(), batch.tuples[i], batch.count[i]);
  for (auto& t : pool) t.join();
}

void ArchiveWriter::feed_words(const bce_cse_words& batch, int threads) {
  if (threads <= 1) {
    for (int i = 0; i < 8; ++i) streams_[i]->packed(batch.words[i], batch.count[i]);
    return;
  }
  std::vector<std::thread> pool;
  for (int i = 0; i < 8; ++i)
    if (batch.count[i]) pool.emplace_back([this, &batch, i] { streams_[i]->packed(batch.words[i], batch.count[i]); });
  for (auto& t : pool) t.join();
}

void ArchiveWriter::worker(int i) {
  for (;;) {
    const void* words;
    size_t count;
    bool b20;
    {
      std::unique_lock<std::mutex> lk(mu_);
      cv_work_.wait(lk, [&] { return stop_ || job_ready_[i]; });
      if (stop_ && !job_ready_[i]) return;
      words = job_words_[i];
      count = job_count_[i];
      b20 = job_20_[i];
      job_ready_[i] = false;
    }
    const auto t0 = std::chrono::steady_clock::now();
    if (b20) streams_[i]->packed20(static_cast<const uint8_t*>(words), count);
    else streams_[i]->packed(static_cast<const uint32_t*>(words), count);
    const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    {
      std::lock_guard<std::mutex> lk(mu_);
      busy_[i] += dt;
      if (--jobs_open_ == 0) cv_done_.notify_all();
    }
  }
}

void ArchiveWriter::begin_words(const bce_cse_words& batch) {
  if (pool_.empty())
    for (int i = 0; i < 8; ++i) pool_.emplace_back(&ArchiveWriter::worker, this, i);
  std::lock_guard<std::mutex> lk(mu_);
  for (int i = 0; i < 8; ++i) {
    if (!batch.count[i]) continue;
    job_words_[i] = batch.words[i];
    job_count_[i] = batch.count[i];
    job_20_[i] = false;
    job_ready_[i] = true;
    ++jobs_open_;
  }
  cv_work_.notify_all();
}

void ArchiveWriter::begin_words20(const bce_cse_words20& batch) {
  if (pool_.empty())
    for (int i = 0; i < 8; ++i) pool_.emplace_back(&ArchiveWriter::worker, this, i);
  std::lock_guard<std::mutex> lk(mu_);
  for (int i = 0; i < 8; ++i) {
    if (!batch.count[i]) continue;
    job_words_[i] = batch.bytes[i];
    job_count_[i] = batch.count[i];
    job_20_[i] = true;
    job_ready_[i] = true;
    ++jobs_open_;
  }
  cv_work_.notify_all();
}

void ArchiveWriter::wait_words() {
  std::unique_lock<std::mutex> lk(mu_);
  cv_done_.wait(lk, [&] { return jobs_open_ == 0; });
}

ArchiveWriter::~ArchiveWriter() {
  {
    std::lock_guard<std::mutex> lk(mu_);
    stop_ = true;
  }
  cv_work_.notify_all();
  for (auto& t : pool_) t.join();
}

std::vector<uint16_t> ArchiveWriter::finish(uint32_t offset) {
  wait_words();
  uint32_t sizes[8], total = 0;
  for (int i = 0; i < 8; ++i) {                                     // bce.cpp:1134-1138
    streams_[i]->finish();
    sizes[i] = uint32_t(streams_[i]->words().size());
    total += sizes[i];
  }
  StreamEncoder header(-1, cfg_);                                   // bce.cpp:1141-1148
  bcefmt::write_header(header.coder(), n_, offset, sizes);

  std::vector<uint16_t> out;                                        // bce.cpp:1152-1157
  out.reserve(1 + header.words().size() + total);
  out.push_back(uint16_t(header.words().size()));
  out.insert(out.end(), header.words().begin(), header.words().end());
  for (auto& s : streams_) out.insert(out.end(), s->words().begin(), s->words().end());
  return out;
}

ScanSession::ScanSession() {
  for (int i = 0; i < 8; ++i) streams_.emplace_back(new ScanCollector(i));
}

void ScanSession::feed(const bce_cse_batch& batch) {
  for (int i = 0; i < 8; ++i) {
    const bce_tuple* t = batch.tuples[i];
    for (size_t j = 0; j < batch.count[i]; ++j) streams_[i]->count(t[j].sym, t[j].k, t[j].c1, t[j].c2, t[j].cs);
  }
}

void ScanSession::feed_words(const bce_cse_words& batch) {
  for (int i = 0; i < 8; ++i) streams_[i]->packed(batch.words[i], batch.count[i]);
}

void ScanSession::feed_buckets(const bce_scan_buckets& batch) {
  std::vector<std::thread> pool;                                    // the eight collectors share nothing
  for (int i = 0; i < 8; ++i)
    if (batch.count[i] || batch.halvings[i])
      pool.emplace_back([this, &batch, i] {
        streams_[i]->bucketed(batch.syms[i], batch.count[i], batch.buckets[i], batch.nbuckets[i], batch.halvings[i]);
      });
  for (auto& t : pool) t.join();
}

ConfigTable ScanSession::finish() {
  // The reference's ScanCoder::init_ is a zero-initialised static (bce.cpp:833-834) that the
  // nine flush() calls fill: streams 0..7 (bce.cpp:1135-1136) and then the header coder (:1149).
  ConfigTable table{};
  for (auto& s : streams_) s->finish(table);
  ScanCollector header(-1);
  header.finish(table);
  return table;
}

}  // namespace bcehost
