// reads_io.hpp -- host side of the streamed `talc` command line: the incremental FASTA / FASTQ reader, the queue that
// hands batches from the reader to the writer, and the 70-column FASTA formatter.  No CUDA in here: talc_main.cpp uses
// it around talc_stream_*, tests/hostemu/reads_io_test.cpp drives it on the CPU (tests/test_reads_io.py).
#pragma once
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <deque>
#include <iostream>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

// ------------------------------------------------------------------------------------------------ streamed input
// io.cpp:26-48 (SeqAn readRecords, SURVEY B.6): FASTA or FASTQ by the first byte; ids = header without marker;
// sequence letters must be ACGTN (either case), anything else is a parse error.  The file is read in pieces; a
// batch ends at a record boundary once it holds --batch-reads reads or --batch-bases bases.
struct Batch {
  uint64_t seq = 0;
  std::vector<std::string> ids;
  std::vector<uint8_t> bases;
  std::vector<uint64_t> offs{0};
};

class ReadParser {
 public:
  explicit ReadParser(const std::string& path) : f_(fopen(path.c_str(), "rb")) { buf_.resize(16u << 20); }
  ~ReadParser() { if (f_) fclose(f_); }
  bool is_open() const { return f_ != nullptr; }
  // fills `b` with up to maxReads reads / about maxBases bases; returns false on a parse error.  b.ids.empty()
  // afterwards means the input is exhausted.  Lines are taken straight from the read buffer (memchr for the end of
  // line, one table-driven pass to validate + drop blanks, bulk append): the reader has to keep several GPUs fed.
  bool next_batch(Batch& b, size_t maxReads, size_t maxBases) {
    b.ids.clear();
    b.bases.clear();
    b.offs.assign(1, 0);
    b.bases.reserve(std::min<size_t>(maxBases, (size_t)1 << 30) + (1u << 20));  // a hint, not a limit
    if (pendingHeader_) {  // FASTA: the header that ended the previous batch opens this one
      b.ids.push_back(header_);
      pendingHeader_ = false;
      open_ = true;
    }
    const char* p;
    size_t n;
    while (get_line(p, n)) {
      if (first_) {
        if (n == 0) continue;
        if (p[0] == '>') fastq_ = false;
        else if (p[0] == '@') fastq_ = true;
        else return false;
        first_ = false;
      }
      if (!fastq_) {
        if (n && p[0] == '>') {
          if (open_) {
            b.offs.push_back(b.bases.size());
            if (b.ids.size() >= maxReads || b.bases.size() >= maxBases) {
              header_.assign(p + 1, n - 1);
              pendingHeader_ = true;
              open_ = false;
              return true;
            }
          }
          b.ids.emplace_back(p + 1, n - 1);
          open_ = true;
        } else if (!push_seq(b, p, n)) {
          std::cout << "ERROR: Unexpected character found" << std::endl;
          return false;
        }
      } else {
        if (n == 0) continue;
        if (p[0] != '@') return false;
        b.ids.emplace_back(p + 1, n - 1);
        if (!get_line(p, n) || !push_seq(b, p, n)) { std::cout << "ERROR: Unexpected character found" << std::endl; return false; }
        if (!get_line(p, n) || !get_line(p, n)) return false;
        b.offs.push_back(b.bases.size());
        if (b.ids.size() >= maxReads || b.bases.size() >= maxBases) return true;
      }
    }
    if (!fastq_ && open_) { b.offs.push_back(b.bases.size()); open_ = false; }
    return true;
  }

 private:
  // 1: a sequence letter (ACGTN either case), 2: blank to drop, 0: anything else is a parse error (SURVEY B.6)
  static const unsigned char* klass() {
    static unsigned char t[256];
    static bool init = false;
    if (!init) {
      memset(t, 0, sizeof t);
      for (const char* q = "ACGTNacgtn"; *q; ++q) t[(unsigned char)*q] = 1;
      t[(unsigned char)' '] = t[(unsigned char)'\t'] = 2;
      init = true;
    }
    return t;
  }
  static bool push_seq(Batch& b, const char* p, size_t n) {
    const unsigned char* t = klass();
    unsigned char all = 1;
    for (size_t i = 0; i < n; ++i) all &= t[(unsigned char)p[i]];  // 1 iff every byte is a sequence letter
    if (all == 1) {  // the common line: one bulk append
      b.bases.insert(b.bases.end(), (const uint8_t*)p, (const uint8_t*)p + n);
      return true;
    }
    for (size_t i = 0; i < n; ++i) {
      const unsigned char k = t[(unsigned char)p[i]];
      if (k == 1) b.bases.push_back((uint8_t)p[i]);
      else if (k == 0) return false;
    }
    return true;
  }
  // next line without its terminator ("\n" or "\r\n") as a view into the read buffer (valid until the next call);
  // a line cut by the end of the buffer is moved to its front and completed by the next fread
  bool get_line(const char*& line, size_t& n) {
    for (;;) {
      const char* p = buf_.data() + pos_;
      const void* nl = memchr(p, '\n', len_ - pos_);
      if (nl) {
        n = (size_t)((const char*)nl - p);
        line = p;
        pos_ += n + 1;
        while (n && line[n - 1] == '\r') --n;
        return true;
      }
      if (eof_) {
        if (pos_ == len_) return false;
        n = len_ - pos_;
        line = p;
        pos_ = len_;
        while (n && line[n - 1] == '\r') --n;
        return true;
      }
      const size_t tail = len_ - pos_;  // incomplete line: keep it, read more behind it
      if (tail && pos_) memmove(&buf_[0], p, tail);
      if (tail + (1u << 20) > buf_.size()) buf_.resize(buf_.size() * 2);  // a line longer than the buffer
      pos_ = 0;
      len_ = tail;
      const size_t got = fread(&buf_[len_], 1, buf_.size() - len_, f_);
      if (got == 0) eof_ = true;
      len_ += got;
    }
  }
  FILE* f_;
  std::string buf_, header_;
  size_t pos_ = 0, len_ = 0;
  bool eof_ = false, first_ = true, fastq_ = false, open_ = false, pendingHeader_ = false;
};

// ids of the batches in flight, handed from the reader to the writer in order
struct IdQueue {
  std::mutex mu;
  std::condition_variable cv;
  std::deque<std::shared_ptr<Batch>> q;
  bool done = false;
  void push(std::shared_ptr<Batch> b) {
    { std::lock_guard<std::mutex> lk(mu); q.push_back(std::move(b)); }
    cv.notify_all();
  }
  void finish() {
    { std::lock_guard<std::mutex> lk(mu); done = true; }
    cv.notify_all();
  }
  std::shared_ptr<Batch> pop() {
    std::unique_lock<std::mutex> lk(mu);
    cv.wait(lk, [&] { return done || !q.empty(); });
    if (q.empty()) return nullptr;
    auto b = q.front();
    q.pop_front();
    return b;
  }
};

// one corrected batch as 70-column FASTA records (io.cpp:50-75), formatted by up to `threads` workers
static void format_fasta(const Batch& b, const uint8_t* out, const uint64_t* ooffs, int threads, std::vector<std::string>& parts) {
  const size_t n = b.ids.size();
  const int nt = (int)std::max<size_t>(1, std::min<size_t>((size_t)threads, n / 2048 + 1));
  parts.assign(nt, std::string());
  auto work = [&](int t) {
    std::string& buf = parts[t];
    const size_t r0 = n * t / nt, r1 = n * (t + 1) / nt;
    buf.reserve((size_t)((ooffs[r1] - ooffs[r0]) * 1.02) + (r1 - r0) * 48 + 64);
    for (size_t r = r0; r < r1; ++r) {
      const uint8_t* s = out + ooffs[r];
      const size_t len = ooffs[r + 1] - ooffs[r];
      buf += '>';
      buf += b.ids[r];
      buf += '\n';
      if (len == 0) buf += '\n';
      for (size_t j = 0; j < len; j += 70) {
        buf.append((const char*)s + j, std::min<size_t>(70, len - j));
        buf += '\n';
      }
    }
  };
  if (nt == 1) { work(0); return; }
  std::vector<std::thread> th;
  for (int t = 0; t < nt; ++t) th.emplace_back(work, t);
  for (auto& x : th) x.join();
}

// --trim / --split: the pieces of one corrected batch as 70-column FASTA records, appended to buf.  pieceOff / bounds
// hold every supported stretch of each read ([start, end) in output coordinates: talc_stream_pieces of a batch
// corrected with TALC_PIECES_SPLIT and min_len 1).  trim: one record per read, from its first stretch's start to its
// last stretch's end, under the read's own header; split: one record per stretch, headed ">{name}_{start}_{end}{rest}"
// with name the id up to its first blank and rest the remainder of the header.  Pieces shorter than minLen are dropped,
// and a read without a piece has no record.  tally: reads with a record, records and bases written.
struct PieceTally {
  uint64_t reads = 0, pieces = 0, bases = 0;
};
static void format_pieces(const Batch& b, const uint8_t* out, const uint64_t* ooffs, const uint64_t* pieceOff, const uint32_t* bounds,
                          bool split, uint32_t minLen, std::string& buf, PieceTally& tally) {
  auto record = [&](const std::string& id, const char* suffix, const uint8_t* s, uint64_t len) {
    const size_t cut = split ? std::min(id.find_first_of(" \t"), id.size()) : id.size();
    buf += '>';
    buf.append(id, 0, cut);
    buf += suffix;
    buf.append(id, cut, std::string::npos);
    buf += '\n';
    for (uint64_t j = 0; j < len; j += 70) {
      buf.append((const char*)s + j, (size_t)std::min<uint64_t>(70, len - j));
      buf += '\n';
    }
    ++tally.pieces;
    tally.bases += len;
  };
  for (size_t r = 0; r < b.ids.size(); ++r) {
    const uint64_t p0 = pieceOff[r], p1 = pieceOff[r + 1];
    const uint8_t* s = out + ooffs[r];
    const uint64_t before = tally.pieces;
    if (!split) {
      if (p1 > p0 && bounds[2 * (p1 - 1) + 1] - bounds[2 * p0] >= minLen)
        record(b.ids[r], "", s + bounds[2 * p0], bounds[2 * (p1 - 1) + 1] - bounds[2 * p0]);
    } else {
      for (uint64_t p = p0; p < p1; ++p) {
        const uint32_t a = bounds[2 * p], e = bounds[2 * p + 1];
        if (e - a < minLen) continue;
        const std::string suffix = "_" + std::to_string(a) + "_" + std::to_string(e);
        record(b.ids[r], suffix.c_str(), s + a, e - a);
      }
    }
    tally.reads += tally.pieces > before;
  }
}
