// hts_io.hpp — minimal BGZF/BAM, VCF (text, plain or gzip/bgzip), FASTA(+.fai) and GTF2
// readers. zlib is the only dependency (no htslib / rust-htslib in this image).
//
// These readers restate only the *observable* behaviour the reference relies on at its
// call sites (SURVEY.md Appendix C):
//   - bam::Record::{pos,mapq,seq,qual,qname,cigar}, CigarStringView::{end_pos,read_pos}
//     used at reference src/microphasing.rs:78-139,297-343
//   - bam::RecordBuffer::fetch  (reference src/microphasing.rs:905-920)
//   - bcf::buffer::RecordBuffer::fetch (reference src/microphasing.rs:932-942)
//   - bio::io::fasta::IndexedReader::{fetch,read} (reference src/microphasing.rs:895-901)
//   - bio::io::gff::Reader(GTF2) (reference src/microphasing.rs:1982-2124)
// Header-only, C++17. Used by the product host code and by the oracle's input side.
#pragma once
#include <zlib.h>

#include "fast_inflate.hpp"

#include <atomic>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <exception>
#include <algorithm>
#include <functional>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <deque>
#include <fstream>
#include <map>
#include <memory>
#include <set>
#include <sstream>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

namespace mphio {

struct IoError : std::runtime_error {
  using std::runtime_error::runtime_error;
};

// ---------------------------------------------------------------- file slurp
inline std::vector<uint8_t> read_file(const std::string& path) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) throw IoError("cannot open " + path);
  std::vector<uint8_t> buf;
  uint8_t tmp[1 << 16];
  size_t n;
  while ((n = fread(tmp, 1, sizeof tmp, f)) > 0) buf.insert(buf.end(), tmp, tmp + n);
  fclose(f);
  return buf;
}

// a byte vector whose resize() does not zero the new bytes: inflated batches are overwritten completely, and clearing
// 16 MB per batch first cost more than framing its records
template <class T>
struct DefaultInitAllocator : std::allocator<T> {
  template <class U> struct rebind { using other = DefaultInitAllocator<U>; };
  using std::allocator<T>::allocator;
  template <class U> void construct(U* p) noexcept(std::is_nothrow_default_constructible<U>::value) { ::new (static_cast<void*>(p)) U; }
  template <class U, class... Args> void construct(U* p, Args&&... args) { ::new (static_cast<void*>(p)) U(std::forward<Args>(args)...); }
};
using RawBytes = std::vector<uint8_t, DefaultInitAllocator<uint8_t>>;


// ---------------------------------------------------------------- BGZF
// Streaming BGZF block reader: each block is an independent gzip member with a BC extra
// subfield holding the block size. inflate is done with raw deflate (windowBits -15).
// BGZF: a series of gzip members of <= 64 KiB each. With threads > 1 a producer thread reads batches of raw blocks
// and inflates them with a small pool while the consumer parses the previous batch (rank 3 of SURVEY.md §8(f):
// BGZF inflate is the first end-to-end bottleneck of the file drivers). threads == 1 is the plain sequential reader.
// The product's file drivers switch the BGZF reader to its own DEFLATE decoder; the test-only oracle, which shares this
// header, leaves it off and keeps zlib, so the two arms do not share the decoder.
inline std::atomic<bool>& fast_inflate_enabled() {
  static std::atomic<bool> on{false};
  return on;
}

// one raw block of a batch: compressed payload at cbuf + coff (clen bytes), inflated to out + ooff (isize bytes)
struct BgzfRaw {
  size_t coff, clen, ooff, isize;
};
// Optional replacement for the host inflate of a whole batch (the CUDA library installs the device-side inflate,
// kernels/inflate_kernels.cu): fills out[0, obytes) from the n blocks or throws, in which case the batch - and every later
// one - is inflated on the host. Only used for files of at least `min_bytes`, with batches of `batch_blocks` blocks.
using BgzfBatchInflater = std::function<void(const uint8_t* cbuf, size_t cbytes, const BgzfRaw* raws, size_t n, uint8_t* out, size_t obytes)>;
struct BgzfInflaterSpec {
  BgzfBatchInflater fn;
  size_t batch_blocks = 4096, min_bytes = size_t(8) << 20;
};
// where the blocks of a handed-over chunk came from: the block at file offset `coff` starts at chunk offset `ooff`, so a
// byte at chunk offset o has the virtual offset coff << 16 | (o - ooff) of the last span with ooff <= o
struct BgzfSpan {
  uint64_t coff;
  int64_t ooff;
};

class BgzfReader {
 public:
  using Raw = BgzfRaw;
  using BatchInflater = BgzfBatchInflater;
  using InflaterSpec = BgzfInflaterSpec;

  // batch_blocks: BGZF blocks per batch of the threaded reader (read-ahead is up to three batches)
  explicit BgzfReader(const std::string& path, unsigned threads = 1, InflaterSpec inflater = InflaterSpec(), size_t batch_blocks = 256)
      : path_(path), threads_(threads ? threads : 1), batch_blocks_(std::max<size_t>(1, batch_blocks)) {
    f_ = fopen(path.c_str(), "rb");
    if (!f_) throw IoError("cannot open " + path);
    if (fseek(f_, 0, SEEK_END) == 0) {
      const long sz = ftell(f_);
      if (sz > 0) file_bytes_ = size_t(sz);
      fseek(f_, 0, SEEK_SET);
    }
    if (inflater.fn && threads_ > 1 && file_bytes_ >= inflater.min_bytes) {
      inflater_ = std::move(inflater.fn);
      batch_blocks_ = std::max<size_t>(256, inflater.batch_blocks);
    }
    if (threads_ > 1) producer_ = std::thread([this] { produce(); });
  }
  bool device_inflate_used() const { return device_batches_.load() != 0; }
  ~BgzfReader() {
    stop_producer();
    if (f_) fclose(f_);
    if (getenv("MPH_IO_TRACE"))  // measurement hook: what reading the file cost
      fprintf(stderr, "[mph io] BGZF %s: %zu seeks, %zu compressed bytes read, %zu blocks inflated\n", path_.c_str(), seeks_,
              size_t(cbytes_read_.load()), size_t(blocks_inflated_.load()));
  }
  BgzfReader(const BgzfReader&) = delete;
  BgzfReader& operator=(const BgzfReader&) = delete;

  unsigned threads() const { return threads_; }
  size_t file_bytes() const { return file_bytes_; }  // compressed size (0 if unknown), a hint for buffer reservations
  // hands over everything that is inflated and unread (the rest of the current block / the next batch); false at EOF
  bool next_chunk(RawBytes& out) {
    if (pos_ == block_.size() && !(threads_ > 1 ? next_batch() : next_block())) return false;
    if (pos_ == 0) {
      out.swap(block_);
      block_.clear();
    } else {
      out.assign(block_.begin() + long(pos_), block_.end());
      block_.clear();
    }
    pos_ = 0;
    return true;
  }

  // hands over everything inflated (the current block / batch) with its spans; the unread bytes start at `begin`
  bool next_chunk(RawBytes& out, size_t& begin, std::vector<BgzfSpan>& spans) {
    if (pos_ == block_.size() && !(threads_ > 1 ? next_batch() : next_block())) return false;
    out.swap(block_);
    spans.swap(spans_);
    begin = pos_;
    block_.clear();
    spans_.clear();
    pos_ = 0;
    return true;
  }

  // Continues at a virtual offset (coff << 16 | offset inside the inflated block): drops the read-ahead, restarts the
  // reading at the block's file offset and the inflated stream at the offset inside it.
  void seek(uint64_t voff) {
    stop_producer();
    const uint64_t coff = voff >> 16;
    if (coff >= file_bytes_ || fseeko(f_, off_t(coff), SEEK_SET) != 0) throw IoError("seek past the end of " + path_);
    next_coff_ = seek_coff_ = coff;
    ready_.clear();
    stop_ = drained_ = false;
    block_.clear();
    spans_.clear();
    pos_ = 0;
    skip_ = size_t(voff & 0xFFFF);
    skip_pending_ = true;
    ++seeks_;
    if (threads_ > 1) producer_ = std::thread([this] { produce(); });
  }

  // read exactly n bytes; returns false on clean EOF at a record boundary (0 bytes read)
  bool read(void* dst, size_t n) {
    uint8_t* d = static_cast<uint8_t*>(dst);
    size_t got = 0;
    while (got < n) {
      if (pos_ == block_.size()) {
        if (!(threads_ > 1 ? next_batch() : next_block())) {
          if (got == 0) return false;
          throw IoError("truncated BGZF stream in " + path_);
        }
        continue;
      }
      size_t take = std::min(n - got, block_.size() - pos_);
      memcpy(d + got, block_.data() + pos_, take);
      pos_ += take;
      got += take;
    }
    return true;
  }

 private:
  void stop_producer() {
    if (!producer_.joinable()) return;
    {
      std::lock_guard<std::mutex> lk(mu_);
      stop_ = true;
    }
    cv_.notify_all();
    producer_.join();
  }
  // the first block after a seek starts at the seek's in-block offset, which must lie inside it
  void apply_skip() {
    if (!skip_pending_) return;
    skip_pending_ = false;
    const size_t first_isize = spans_.size() > 1 ? size_t(spans_[1].ooff - spans_[0].ooff) : block_.size();
    if (spans_.empty() || spans_[0].coff != seek_coff_ || skip_ > first_isize) throw IoError("virtual offset past the end of its BGZF block in " + path_);
    pos_ = skip_;
  }
  // reads one raw block (compressed payload appended to cbuf); false at end of file
  bool read_raw(std::vector<uint8_t>& cbuf, Raw& r, uint64_t* coff = nullptr) {
    if (coff) *coff = next_coff_;
    uint8_t hdr[18];
    size_t n = fread(hdr, 1, 18, f_);
    if (n == 0) return false;
    if (n != 18 || hdr[0] != 31 || hdr[1] != 139 || hdr[2] != 8 || !(hdr[3] & 4)) throw IoError("not a BGZF file: " + path_);
    uint16_t xlen = hdr[10] | (hdr[11] << 8);
    // the BC subfield is normally the first (and only) one
    std::vector<uint8_t> extra(xlen);
    memcpy(extra.data(), hdr + 12, std::min<size_t>(6, xlen));
    if (xlen > 6 && fread(extra.data() + 6, 1, xlen - 6, f_) != size_t(xlen - 6)) throw IoError("truncated BGZF header in " + path_);
    int bsize = -1;
    for (size_t o = 0; o + 4 <= extra.size();) {
      uint16_t slen = extra[o + 2] | (extra[o + 3] << 8);
      if (extra[o] == 'B' && extra[o + 1] == 'C' && slen == 2 && o + 6 <= extra.size()) bsize = extra[o + 4] | (extra[o + 5] << 8);
      o += 4 + slen;
    }
    if (bsize < 0) throw IoError("BGZF block without BC field in " + path_);
    if (size_t(bsize) + 1 < size_t(12) + xlen + 8) throw IoError("corrupt BGZF block size in " + path_);
    const size_t clen = size_t(bsize) + 1 - 12 - xlen - 8;  // compressed payload
    const size_t off = cbuf.size();
    cbuf.resize(off + clen + 8);
    if (fread(cbuf.data() + off, 1, clen + 8, f_) != clen + 8) throw IoError("truncated BGZF block in " + path_);
    uint32_t isize;
    memcpy(&isize, cbuf.data() + off + clen + 4, 4);
    r.coff = off; r.clen = clen; r.isize = isize; r.ooff = 0;
    next_coff_ += uint64_t(bsize) + 1;
    cbytes_read_ += uint64_t(bsize) + 1;
    return true;
  }
  void inflate_one(const uint8_t* in, size_t clen, uint8_t* out, size_t isize) const {
    if (isize == 0) return;
    blocks_inflated_.fetch_add(1, std::memory_order_relaxed);
    if (fast_inflate_enabled().load(std::memory_order_relaxed)) {
      // the reader's own decoder (io/fast_inflate.hpp, ~1.3x zlib on BAM blocks); whatever it rejects goes through zlib below
      static thread_local std::unique_ptr<FastInflate> fast;
      if (!fast) fast.reset(new FastInflate);
      if (fast->run(in, clen, out, isize)) return;
    }
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, -15) != Z_OK) throw IoError("zlib init failed");
    zs.next_in = const_cast<uint8_t*>(in);
    zs.avail_in = uInt(clen);
    zs.next_out = out;
    zs.avail_out = uInt(isize);
    int rc = inflate(&zs, Z_FINISH);
    inflateEnd(&zs);
    if (rc != Z_STREAM_END) throw IoError("BGZF inflate failed in " + path_);
  }
  bool next_block() {
    for (;;) {
      cbuf_.clear();
      Raw r;
      uint64_t coff;
      if (!read_raw(cbuf_, r, &coff)) return false;
      block_.resize(r.isize);
      spans_.assign(1, BgzfSpan{coff, 0});
      pos_ = 0;
      inflate_one(cbuf_.data() + r.coff, r.clen, block_.data(), r.isize);
      apply_skip();
      if (pos_ == block_.size()) continue;  // EOF marker / empty block, or a seek to the end of a block
      return true;
    }
  }

  // ---- threaded path: producer fills `ready_` (at most two batches ahead), consumer swaps them into block_
  struct Batch {
    RawBytes data;
    std::vector<BgzfSpan> spans;
    bool eof = false;
    std::exception_ptr err;
  };
  // raw (still compressed) blocks of one batch
  struct RawBatch {
    std::vector<uint8_t> cbuf;
    std::vector<Raw> raws;
    std::vector<uint64_t> coffs;  // file offset of each block
    size_t total = 0;
    bool eof = false;
    std::exception_ptr err;
  };
  void read_raw_batch(RawBatch& rb) {
    rb.cbuf.clear();
    rb.raws.clear();
    rb.coffs.clear();
    rb.total = 0;
    rb.eof = false;
    rb.err = nullptr;
    try {
      while (rb.raws.size() < batch_blocks_) {
        Raw r;
        uint64_t coff;
        if (!read_raw(rb.cbuf, r, &coff)) { rb.eof = true; break; }
        r.ooff = rb.total;
        rb.total += r.isize;
        rb.raws.push_back(r);
        rb.coffs.push_back(coff);
      }
    } catch (...) {
      rb.err = std::current_exception();
      rb.eof = true;
    }
  }
  // The producer reads the raw blocks of batch N + 1 from the file while its pool inflates batch N (the read is a copy out of
  // the page cache at a few GB/s: done between the inflates it was a third of the loader's wall time).
  void produce() {
    RawBatch cur, nxt;
    read_raw_batch(cur);
    for (;;) {
      {
        std::lock_guard<std::mutex> lk(mu_);
        if (stop_) return;
      }
      Batch b;
      b.eof = cur.eof;
      for (size_t i = 0; i < cur.raws.size(); ++i) b.spans.push_back(BgzfSpan{cur.coffs[i], int64_t(cur.raws[i].ooff)});
      bool have_next = false;
      try {
        b.data.resize(cur.total);
        std::atomic<size_t> next{0};
        std::vector<std::exception_ptr> errs(threads_);
        auto work = [&](unsigned ti) {
          try {
            for (;;) {
              const size_t i = next.fetch_add(1);
              if (i >= cur.raws.size()) break;
              inflate_one(cur.cbuf.data() + cur.raws[i].coff, cur.raws[i].clen, b.data.data() + cur.raws[i].ooff, cur.raws[i].isize);
            }
          } catch (...) {
            errs[ti] = std::current_exception();
          }
        };
        bool on_device = false;
        if (inflater_ && !cur.raws.empty()) {
          // the installed batch inflater (device side) runs on a helper thread while this one reads the next raw batch
          std::exception_ptr dev_err;
          std::thread helper([&] {
            try {
              inflater_(cur.cbuf.data(), cur.cbuf.size(), cur.raws.data(), cur.raws.size(), b.data.data(), cur.total);
            } catch (...) {
              dev_err = std::current_exception();
            }
          });
          if (!cur.eof) { read_raw_batch(nxt); have_next = true; }
          helper.join();
          if (dev_err) inflater_ = nullptr;  // not available / failed: this batch and the rest go through zlib
          else { on_device = true; device_batches_ += 1; blocks_inflated_ += cur.raws.size(); }
        }
        if (!on_device) {
          std::vector<std::thread> pool;
          for (unsigned ti = 1; ti < threads_; ++ti) pool.emplace_back(work, ti);
          if (!cur.eof && !have_next) { read_raw_batch(nxt); have_next = true; }  // overlaps the inflate of `cur`
          work(0);
          for (auto& t : pool) t.join();
          for (auto& e : errs)
            if (e) std::rethrow_exception(e);
        }
        if (cur.err) std::rethrow_exception(cur.err);  // what was read before the failure has been inflated; the failure ends the stream
      } catch (...) {
        b.err = std::current_exception();
        b.eof = true;
      }
      const bool last = b.eof;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return stop_ || ready_.size() < 2; });
        if (stop_) return;
        ready_.push_back(std::move(b));
      }
      cv_.notify_all();
      if (last) return;
      if (!have_next) read_raw_batch(nxt);
      std::swap(cur, nxt);
    }
  }
  bool next_batch() {
    for (;;) {
      Batch b;
      {
        std::unique_lock<std::mutex> lk(mu_);
        if (drained_) return false;
        cv_.wait(lk, [&] { return !ready_.empty(); });
        b = std::move(ready_.front());
        ready_.pop_front();
        if (b.eof) drained_ = true;
      }
      cv_.notify_all();
      if (b.err) std::rethrow_exception(b.err);
      block_ = std::move(b.data);
      spans_ = std::move(b.spans);
      pos_ = 0;
      if (!spans_.empty()) apply_skip();
      if (pos_ < block_.size()) return true;
      if (drained_) return false;
    }
  }

  std::string path_;
  FILE* f_ = nullptr;
  std::vector<uint8_t> cbuf_;
  RawBytes block_;
  std::vector<BgzfSpan> spans_;  // of block_
  size_t pos_ = 0;
  uint64_t next_coff_ = 0, seek_coff_ = 0;  // file offset of the next raw block / of the last seek
  size_t skip_ = 0;
  bool skip_pending_ = false;
  unsigned threads_ = 1;
  size_t file_bytes_ = 0;
  std::thread producer_;
  std::mutex mu_;
  std::condition_variable cv_;
  std::deque<Batch> ready_;
  bool stop_ = false, drained_ = false;
  BatchInflater inflater_;
  size_t batch_blocks_;
  std::atomic<size_t> device_batches_{0};
  size_t seeks_ = 0;
  std::atomic<uint64_t> cbytes_read_{0};
  mutable std::atomic<uint64_t> blocks_inflated_{0};
};

// ---------------------------------------------------------------- BAM
enum CigarOp : uint32_t { C_M = 0, C_I = 1, C_D = 2, C_N = 3, C_S = 4, C_H = 5, C_P = 6, C_EQ = 7, C_X = 8 };

struct BamRecord {
  int32_t tid = -1;
  int32_t pos = -1;
  uint8_t mapq = 0;
  uint16_t flag = 0;
  uint32_t l_seq = 0;
  std::string qname;             // without the trailing NUL
  std::vector<uint32_t> cigar;   // BAM encoding: len<<4 | op
  std::vector<uint8_t> seq4;     // 4-bit packed, high nibble first
  std::vector<uint8_t> qual;     // raw phred
  std::vector<uint8_t> aux;      // raw aux block (tests/fixture tooling use MD)

  bool is_unmapped() const { return flag & 4; }
  // bam::Record::seq()[i] -> ASCII from "=ACMGRSVTWYHKDBN"
  uint8_t base(uint32_t i) const {
    static const char* dec = "=ACMGRSVTWYHKDBN";
    uint8_t b = seq4[i >> 1];
    return uint8_t(dec[(i & 1) ? (b & 15) : (b >> 4)]);
  }
  // CigarStringView::end_pos(): pos + sum of reference-consuming op lengths (M,D,N,=,X)
  int64_t end_pos() const {
    int64_t e = pos;
    for (uint32_t c : cigar) {
      uint32_t op = c & 15, len = c >> 4;
      if (op == C_M || op == C_D || op == C_N || op == C_EQ || op == C_X) e += len;
    }
    return e;
  }
};

// CigarStringView::read_pos(ref_pos, include_softclips=false, include_dels=false).
// Returns: 1 = Some(qpos) (written to *out), 0 = None, -1 = Err.
// Restated from rust-htslib 0.36 bam/record.rs (crate not vendored under /root/reference;
// semantics pinned indirectly by the somatic fixtures, SURVEY.md Appendix C).
inline int cigar_read_pos(const std::vector<uint32_t>& cigar, int64_t read_start, int64_t ref_pos, uint32_t* out) {
  int64_t rpos = read_start;  // reference position
  int64_t qpos = 0;           // position within read
  size_t j = 0;               // index into cigar operation vector
  const size_t n = cigar.size();
  // find the first operation that refers to qpos = 0 (i.e. to bases in record.seq())
  for (size_t i = 0; i < n; ++i) {
    uint32_t op = cigar[i] & 15;
    if (op == C_M || op == C_X || op == C_EQ || op == C_I || op == C_S) {
      j = i;  // include_softclips == false: a leading S is consumed by the main loop
      break;
    }
    if (op == C_D || op == C_N) return -1;  // D/N before any op describing read sequence
    if (op == C_H && i > 0 && i + 1 < n) return -1;  // hard clip between operations
    if ((op == C_P || op == C_H) && i + 1 == n) return 0;  // only pads / hard clips
    // otherwise: leading H / P, consumes nothing
  }
  while (rpos <= ref_pos && j < n) {
    uint32_t op = cigar[j] & 15;
    int64_t l = cigar[j] >> 4;
    switch (op) {
      case C_M:
      case C_X:
      case C_EQ:
        if (rpos <= ref_pos && rpos + l > ref_pos) {
          *out = uint32_t(qpos + (ref_pos - rpos));
          return 1;
        }
        rpos += l;
        qpos += l;
        ++j;
        break;
      case C_S:
      case C_I:
        qpos += l;
        ++j;
        break;
      case C_N:
      case C_D:  // include_dels == false
        rpos += l;
        ++j;
        break;
      case C_P:
        ++j;
        break;
      case C_H:
        if (j + 1 < n) return -1;
        return 0;
      default:
        return -1;
    }
  }
  return 0;
}

struct BamFile {
  std::string header_text;
  std::vector<std::string> ref_names;
  std::vector<int64_t> ref_lens;
  std::unordered_map<std::string, int> tid_of;

  explicit BamFile(const std::string& path, unsigned inflate_threads = 1, BgzfReader::InflaterSpec inflater = BgzfReader::InflaterSpec(),
                   size_t batch_blocks = 256)
      : path_(path), rd_(path, inflate_threads, std::move(inflater), batch_blocks) {
    char magic[4];
    if (!rd_.read(magic, 4) || memcmp(magic, "BAM\1", 4) != 0) throw IoError("not a BAM file: " + path);
    auto must = [&](void* dst, size_t n) { if (!rd_.read(dst, n)) throw IoError("truncated BAM header: " + path); };
    int32_t l_text;
    must(&l_text, 4);
    if (l_text < 0 || l_text > (1 << 30)) throw IoError("corrupt BAM header: " + path);
    header_text.resize(size_t(l_text));
    if (l_text) must(&header_text[0], size_t(l_text));
    int32_t n_ref;
    must(&n_ref, 4);
    if (n_ref < 0 || n_ref > (1 << 24)) throw IoError("corrupt BAM header: " + path);
    for (int i = 0; i < n_ref; ++i) {
      int32_t l_name;
      must(&l_name, 4);
      if (l_name <= 0 || l_name > (1 << 16)) throw IoError("corrupt BAM header: " + path);
      std::string nm(size_t(l_name), 0);
      must(&nm[0], size_t(l_name));
      if (!nm.empty() && nm.back() == 0) nm.pop_back();
      int32_t l_ref;
      must(&l_ref, 4);
      tid_of[nm] = i;
      ref_names.push_back(nm);
      ref_lens.push_back(l_ref);
    }
  }

  unsigned inflate_threads() const { return rd_.threads(); }
  bool device_inflate_used() const { return rd_.device_inflate_used(); }
  size_t file_bytes() const { return rd_.file_bytes(); }
  // raw record stream after the header, in chunks (a record may straddle two chunks): for callers that frame and
  // parse the records themselves, in parallel
  bool next_chunk(RawBytes& out) { return rd_.next_chunk(out); }
  // the same with where the bytes came from (virtual offsets), and a jump to a virtual offset: the indexed read buffer
  bool next_chunk(RawBytes& out, size_t& begin, std::vector<BgzfSpan>& spans) { return rd_.next_chunk(out, begin, spans); }
  void seek(uint64_t voff) { rd_.seek(voff); }
  const std::string& path() const { return path_; }

  // next alignment record; false on EOF
  bool next(BamRecord& r) {
    int32_t bs;
    if (!rd_.read(&bs, 4)) return false;
    if (bs < 32 || bs > (1 << 29)) throw IoError("corrupt BAM record");  // the fixed part alone is 32 bytes
    buf_.resize(size_t(bs));
    if (!rd_.read(buf_.data(), size_t(bs))) throw IoError("truncated BAM record");
    const uint8_t* p = buf_.data();
    auto i32 = [&](size_t o) { int32_t v; memcpy(&v, p + o, 4); return v; };
    auto u16 = [&](size_t o) { uint16_t v; memcpy(&v, p + o, 2); return v; };
    r.tid = i32(0);
    r.pos = i32(4);
    uint8_t l_read_name = p[8];
    r.mapq = p[9];
    uint16_t n_cigar = u16(12);
    r.flag = u16(14);
    const int32_t l_seq = i32(16);
    // the variable part must fit the record: name, CIGAR, packed bases, qualities (the threaded loader checks the same)
    if (l_seq < 0 || 32 + size_t(l_read_name) + 4 * size_t(n_cigar) + (size_t(l_seq) + 1) / 2 + size_t(l_seq) > size_t(bs))
      throw IoError("corrupt BAM record");
    r.l_seq = uint32_t(l_seq);
    size_t o = 32;
    r.qname.assign(reinterpret_cast<const char*>(p + o), l_read_name ? l_read_name - 1 : 0);
    o += l_read_name;
    r.cigar.resize(n_cigar);
    if (n_cigar) memcpy(r.cigar.data(), p + o, 4 * size_t(n_cigar));
    o += 4 * size_t(n_cigar);
    size_t sb = (r.l_seq + 1) / 2;
    r.seq4.assign(p + o, p + o + sb);
    o += sb;
    r.qual.assign(p + o, p + o + r.l_seq);
    o += r.l_seq;
    r.aux.assign(p + o, p + bs);
    return true;
  }

 private:
  std::string path_;
  BgzfReader rd_;
  std::vector<uint8_t> buf_;
};

// ---------------------------------------------------------------- line reader (plain or gzip)
class LineReader {
 public:
  explicit LineReader(const std::string& path) {
    gz_ = gzopen(path.c_str(), "rb");
    if (!gz_) throw IoError("cannot open " + path);
    gzbuffer(gz_, 1 << 18);
  }
  ~LineReader() {
    if (gz_) gzclose(gz_);
  }
  // raw bytes (binary BCF); returns the number of bytes read
  size_t read_bytes(void* dst, size_t n) {
    size_t got = 0;
    while (got < n && !pre_.empty()) { static_cast<char*>(dst)[got++] = pre_.front(); pre_.erase(pre_.begin()); }
    while (got < n) {
      const int r = gzread(gz_, static_cast<char*>(dst) + got, unsigned(std::min<size_t>(n - got, 1u << 30)));
      if (r <= 0) break;
      got += size_t(r);
    }
    return got;
  }
  // gives bytes back to the stream (the format sniffing of VcfFile)
  void unread(const char* p, size_t n) { pre_.insert(pre_.begin(), p, p + n); }
  bool getline(std::string& line) {
    line.clear();
    while (!pre_.empty()) {
      const char c = pre_.front();
      pre_.erase(pre_.begin());
      if (c == '\n') {
        if (!line.empty() && line.back() == '\r') line.pop_back();
        return true;
      }
      line.push_back(c);
    }
    char buf[1 << 14];
    for (;;) {
      if (!gzgets(gz_, buf, sizeof buf)) return !line.empty();
      size_t n = strlen(buf);
      if (n && buf[n - 1] == '\n') {
        line.append(buf, n - 1);
        if (!line.empty() && line.back() == '\r') line.pop_back();
        return true;
      }
      line.append(buf, n);
    }
  }

 private:
  gzFile gz_;
  std::string pre_;
};

inline std::vector<std::string> split(const std::string& s, char d) {
  std::vector<std::string> out;
  size_t b = 0;
  for (;;) {
    size_t e = s.find(d, b);
    if (e == std::string::npos) {
      out.emplace_back(s.substr(b));
      break;
    }
    out.emplace_back(s.substr(b, e - b));
    b = e + 1;
  }
  return out;
}

// ---------------------------------------------------------------- VCF (text)
struct VcfRecord {
  int rid = -1;
  int64_t pos = 0;  // 0-based
  std::string ref;
  std::vector<std::string> alts;
  // INFO access mirrors bcf::Record::info(tag): *_defined = tag declared in the header
  bool somatic_flag = false;   // INFO/SOMATIC present (only meaningful if declared as Flag)
  bool has_ann = false;        // INFO/ANN key present on this record
  std::string ann_first;       // first comma-separated ANN entry
  bool has_svlen = false;
  std::vector<int64_t> svlen;  // INT64_MIN marks a missing value
};

struct VcfFile {
  std::vector<std::string> contigs;
  std::unordered_map<std::string, int> rid_of;
  bool somatic_defined = false, ann_defined = false, svlen_defined = false;

  // The reference opens its variants with bcf::Reader::from_path (src/main.rs:75), which takes text VCF (plain or
  // BGZF / gzip) and binary BCF2 alike; so does this reader: the first bytes of the (inflated) stream tell which.
  explicit VcfFile(const std::string& path) : lr_(path) {
    char magic[5];
    const size_t got = lr_.read_bytes(magic, 5);
    if (got == 5 && memcmp(magic, "BCF\2", 4) == 0) {
      if (magic[4] != 1 && magic[4] != 2) throw IoError("unsupported BCF minor version in " + path);
      bcf_ = true;
      uint32_t l_text = 0;
      if (lr_.read_bytes(&l_text, 4) != 4) throw IoError("truncated BCF header in " + path);
      std::string text(l_text, '\0');
      if (lr_.read_bytes(&text[0], l_text) != l_text) throw IoError("truncated BCF header in " + path);
      size_t b = 0;
      while (b < text.size()) {
        size_t e = text.find('\n', b);
        if (e == std::string::npos) e = text.size();
        std::string line = text.substr(b, e - b);
        while (!line.empty() && (line.back() == '\0' || line.back() == '\r')) line.pop_back();
        b = e + 1;
        if (line.rfind("##", 0) == 0) header_line(line);
      }
      return;
    }
    lr_.unread(magic, got);
    std::string line;
    while (lr_.getline(line)) {
      if (line.rfind("##", 0) == 0) {
        header_line(line);
        continue;
      }
      if (!line.empty() && line[0] == '#') break;  // #CHROM line
      pending_ = line;
      have_pending_ = true;
      break;
    }
  }

  // htslib: name2rid fails for contigs absent from the header; text VCFs whose records
  // use undeclared contigs get them appended on the fly (with a warning) by htslib.
  int name2rid(const std::string& c) const {
    auto it = rid_of.find(c);
    return it == rid_of.end() ? -1 : it->second;
  }

  bool next(VcfRecord& r) {
    if (bcf_) return next_bcf(r);
    std::string line;
    for (;;) {
      if (have_pending_) {
        line.swap(pending_);
        have_pending_ = false;
      } else if (!lr_.getline(line)) {
        return false;
      }
      if (line.empty() || line[0] == '#') continue;
      break;
    }
    // CHROM POS ID REF ALT QUAL FILTER INFO ...
    size_t f[9];
    size_t nf = 0, b = 0;
    f[nf++] = 0;
    while (nf < 9 && (b = line.find('\t', b)) != std::string::npos) f[nf++] = ++b;
    if (nf < 5) throw IoError("malformed VCF line: " + line.substr(0, 80));
    auto field = [&](size_t i) -> std::string {
      if (i >= nf) return std::string();
      size_t s = f[i];
      size_t e = (i + 1 < nf) ? f[i + 1] - 1 : line.find('\t', s);
      if (e == std::string::npos) e = line.size();
      return line.substr(s, e - s);
    };
    std::string chrom = field(0);
    int rid = name2rid(chrom);
    if (rid < 0) rid = add_contig(chrom);
    r.rid = rid;
    r.pos = std::stoll(field(1)) - 1;
    r.ref = field(3);
    r.alts.clear();
    std::string alt = field(4);
    if (alt != ".") r.alts = split(alt, ',');
    r.somatic_flag = r.has_ann = r.has_svlen = false;
    r.ann_first.clear();
    r.svlen.clear();
    std::string info = field(7);
    if (!info.empty() && info != ".") {
      size_t s = 0;
      while (s <= info.size()) {
        size_t e = info.find(';', s);
        if (e == std::string::npos) e = info.size();
        size_t eq = info.find('=', s);
        if (eq == std::string::npos || eq > e) eq = e;
        size_t klen = eq - s;
        if (klen == 7 && info.compare(s, 7, "SOMATIC") == 0) {
          r.somatic_flag = true;
        } else if (klen == 3 && info.compare(s, 3, "ANN") == 0) {
          r.has_ann = true;
          std::string v = eq < e ? info.substr(eq + 1, e - eq - 1) : std::string();
          size_t c = v.find(',');
          r.ann_first = c == std::string::npos ? v : v.substr(0, c);
        } else if (klen == 5 && info.compare(s, 5, "SVLEN") == 0) {
          r.has_svlen = true;
          std::string v = eq < e ? info.substr(eq + 1, e - eq - 1) : std::string();
          for (auto& t : split(v, ',')) r.svlen.push_back(t == "." || t.empty() ? INT64_MIN : std::stoll(t));
        }
        s = e + 1;
      }
    }
    return true;
  }

 private:
  int add_contig(const std::string& c) {
    auto it = rid_of.find(c);
    if (it != rid_of.end()) return it->second;
    int id = int(contigs.size());
    contigs.push_back(c);
    rid_of[c] = id;
    return id;
  }

  // value of `key=` inside a ##XXX=<...> header line ("" if absent)
  static std::string header_attr(const std::string& line, const char* key) {
    const std::string k = std::string(key) + "=";
    size_t p = line.find("<" + k);
    if (p == std::string::npos) p = line.find("," + k);
    if (p == std::string::npos) return std::string();
    p += 1 + k.size();
    const size_t e = line.find_first_of(",>", p);
    return line.substr(p, e == std::string::npos ? std::string::npos : e - p);
  }

  // one ## line of a VCF / BCF header: contigs, the INFO tags the path reads, and BCF's two dictionaries (the contig
  // dictionary, and the FILTER / INFO / FORMAT id dictionary with PASS at 0; an IDX= attribute overrides the position)
  void header_line(const std::string& line) {
    if (line.rfind("##contig=<", 0) == 0) {
      const std::string id = header_attr(line, "ID");
      if (id.empty()) return;
      const int rid = add_contig(id);
      const std::string idx = header_attr(line, "IDX");
      const size_t at = idx.empty() ? bcf_contig_rid_.size() : size_t(std::stoul(idx));
      if (bcf_contig_rid_.size() <= at) bcf_contig_rid_.resize(at + 1, -1);
      bcf_contig_rid_[at] = rid;
      return;
    }
    const bool is_info = line.rfind("##INFO=<", 0) == 0;
    if (!is_info && line.rfind("##FILTER=<", 0) != 0 && line.rfind("##FORMAT=<", 0) != 0) return;
    const std::string id = header_attr(line, "ID");
    if (id.empty()) return;
    if (is_info) {
      if (id == "SOMATIC") somatic_defined = line.find("Type=Flag") != std::string::npos;
      if (id == "ANN") ann_defined = true;
      if (id == "SVLEN") svlen_defined = true;
    }
    if (bcf_dict_.empty()) bcf_dict_.push_back("PASS");
    const std::string idx = header_attr(line, "IDX");
    size_t at;
    if (!idx.empty()) at = size_t(std::stoul(idx));
    else {
      auto it = std::find(bcf_dict_.begin(), bcf_dict_.end(), id);
      at = it == bcf_dict_.end() ? bcf_dict_.size() : size_t(it - bcf_dict_.begin());
    }
    if (bcf_dict_.size() <= at) bcf_dict_.resize(at + 1);
    bcf_dict_[at] = id;
  }

  // ---- BCF2 records (VCF specification, section 6): typed values over a little-endian byte block
  struct Cursor {
    const uint8_t* p;
    const uint8_t* end;
    void need(size_t n) const { if (size_t(end - p) < n) throw IoError("truncated BCF record"); }
    template <class T> T get() { need(sizeof(T)); T v; memcpy(&v, p, sizeof(T)); p += sizeof(T); return v; }
    // reads one integer of BCF type 1 / 2 / 3; *missing / *eov tell the reserved values
    int64_t get_int(int type, bool* missing, bool* eov) {
      *missing = *eov = false;
      if (type == 1) { const int8_t v = get<int8_t>(); *missing = v == INT8_MIN; *eov = v == INT8_MIN + 1; return v; }
      if (type == 2) { const int16_t v = get<int16_t>(); *missing = v == INT16_MIN; *eov = v == INT16_MIN + 1; return v; }
      if (type == 3) { const int32_t v = get<int32_t>(); *missing = v == INT32_MIN; *eov = v == INT32_MIN + 1; return v; }
      throw IoError("BCF: integer expected");
    }
    // descriptor byte (+ overflow length): type and number of elements
    void desc(int* type, size_t* len) {
      const uint8_t d = get<uint8_t>();
      *type = d & 15;
      *len = d >> 4;
      if (*len == 15) {
        int t; size_t l;
        desc(&t, &l);
        if (l != 1) throw IoError("BCF: malformed length");
        bool m, e;
        const int64_t v = get_int(t, &m, &e);
        if (v < 0) throw IoError("BCF: negative length");
        *len = size_t(v);
      }
    }
    static size_t width(int type) {
      switch (type) { case 0: return 0; case 1: return 1; case 2: return 2; case 3: return 4; case 5: return 4; case 7: return 1; }
      throw IoError("BCF: unknown value type");
    }
    void skip_value() { int t; size_t l; desc(&t, &l); need(width(t) * l); p += width(t) * l; }
    std::string get_string() {
      int t; size_t l;
      desc(&t, &l);
      if (t == 0) return std::string();
      if (t != 7) throw IoError("BCF: string expected");
      need(l);
      std::string s(reinterpret_cast<const char*>(p), l);
      p += l;
      while (!s.empty() && s.back() == '\0') s.pop_back();
      return s;
    }
  };

  bool next_bcf(VcfRecord& r) {
    uint32_t lens[2];
    const size_t got = lr_.read_bytes(lens, 8);
    if (got == 0) return false;
    if (got != 8) throw IoError("truncated BCF record");
    if (lens[0] < 24 || lens[0] > (1u << 30) || lens[1] > (1u << 30)) throw IoError("corrupt BCF record");
    buf_.resize(size_t(lens[0]) + lens[1]);
    if (lr_.read_bytes(buf_.data(), buf_.size()) != buf_.size()) throw IoError("truncated BCF record");
    Cursor c{buf_.data(), buf_.data() + lens[0]};
    const int32_t chrom = c.get<int32_t>(), pos = c.get<int32_t>();
    c.get<int32_t>();  // rlen
    c.get<float>();    // QUAL
    const uint32_t n_allele_info = c.get<uint32_t>();
    c.get<uint32_t>();  // n_fmt << 24 | n_sample
    const uint32_t n_info = n_allele_info & 0xFFFFu, n_allele = n_allele_info >> 16;
    if (chrom < 0 || size_t(chrom) >= bcf_contig_rid_.size() || bcf_contig_rid_[size_t(chrom)] < 0) throw IoError("BCF record on an undeclared contig");
    r.rid = bcf_contig_rid_[size_t(chrom)];
    r.pos = pos;
    c.get_string();  // ID
    r.ref.clear();
    r.alts.clear();
    for (uint32_t a = 0; a < n_allele; ++a) {
      std::string al = c.get_string();
      if (a == 0) r.ref = std::move(al);
      else r.alts.push_back(std::move(al));
    }
    c.skip_value();  // FILTER
    r.somatic_flag = r.has_ann = r.has_svlen = false;
    r.ann_first.clear();
    r.svlen.clear();
    for (uint32_t i = 0; i < n_info; ++i) {
      int kt; size_t kl;
      c.desc(&kt, &kl);
      if (kl != 1) throw IoError("BCF: malformed INFO key");
      bool m, e;
      const int64_t key = c.get_int(kt, &m, &e);
      const std::string* name = key >= 0 && size_t(key) < bcf_dict_.size() ? &bcf_dict_[size_t(key)] : nullptr;
      if (name && *name == "SOMATIC") {
        r.somatic_flag = true;  // a Flag is present by being listed (its value is empty or a single 1)
        c.skip_value();
      } else if (name && *name == "ANN") {
        r.has_ann = true;
        const std::string v = c.get_string();
        const size_t comma = v.find(',');
        r.ann_first = comma == std::string::npos ? v : v.substr(0, comma);
      } else if (name && *name == "SVLEN") {
        r.has_svlen = true;
        int t; size_t l;
        c.desc(&t, &l);
        for (size_t x = 0; x < l; ++x) {
          bool miss, eov;
          const int64_t v = c.get_int(t, &miss, &eov);
          if (eov) continue;
          r.svlen.push_back(miss ? INT64_MIN : v);
        }
      } else {
        c.skip_value();
      }
    }
    return true;
  }

  LineReader lr_;
  std::string pending_;
  bool have_pending_ = false;
  bool bcf_ = false;
  std::vector<std::string> bcf_dict_;   // FILTER / INFO / FORMAT ids by dictionary index
  std::vector<int> bcf_contig_rid_;     // contig dictionary index -> rid
  std::vector<uint8_t> buf_;
};

// ---------------------------------------------------------------- FASTA + .fai
// bio::io::fasta::IndexedReader: fetch(name, start, stop) 0-based half-open, read() strips
// line terminators and preserves case; out-of-range stop is an error.
class FastaIndexed {
 public:
  explicit FastaIndexed(const std::string& path) : path_(path) {
    std::ifstream fai(path + ".fai");
    if (!fai) throw IoError("cannot open " + path + ".fai");
    std::string line;
    while (std::getline(fai, line)) {
      if (line.empty()) continue;
      auto t = split(line, '\t');
      if (t.size() < 5) throw IoError("malformed .fai line");
      Entry e{std::stoull(t[1]), std::stoull(t[2]), std::stoull(t[3]), std::stoull(t[4])};
      idx_[t[0]] = e;
    }
    f_ = fopen(path.c_str(), "rb");
    if (!f_) throw IoError("cannot open " + path);
  }
  ~FastaIndexed() {
    if (f_) fclose(f_);
  }
  bool has(const std::string& name) const { return idx_.count(name) != 0; }
  uint64_t length(const std::string& name) const { return idx_.at(name).len; }

  void fetch(const std::string& name, uint64_t start, uint64_t stop, std::vector<uint8_t>& out) {
    auto it = idx_.find(name);
    if (it == idx_.end()) throw IoError("Unknown sequence name: " + name);
    const Entry& e = it->second;
    if (start > stop) throw IoError("Invalid query interval");
    if (stop > e.len) throw IoError("FASTA read interval was out of bounds");
    out.clear();
    out.reserve(stop - start);
    if (start == stop) return;
    uint64_t line = start / e.line_bases, col = start % e.line_bases;
    uint64_t off = e.offset + line * e.line_bytes + col;
    if (fseeko(f_, off_t(off), SEEK_SET) != 0) throw IoError("seek failed in " + path_);
    uint64_t need = stop - start;
    // bytes spanned on disk
    uint64_t last = stop - 1;
    uint64_t last_off = e.offset + (last / e.line_bases) * e.line_bytes + last % e.line_bases;
    std::vector<uint8_t> raw(last_off - off + 1);
    if (fread(raw.data(), 1, raw.size(), f_) != raw.size()) throw IoError("short read in " + path_);
    uint64_t c = col;
    for (size_t i = 0; i < raw.size() && out.size() < need;) {
      uint64_t take = std::min<uint64_t>(e.line_bases - c, need - out.size());
      out.insert(out.end(), raw.begin() + i, raw.begin() + i + take);
      i += take + (e.line_bytes - e.line_bases);
      c = 0;
    }
  }

 private:
  struct Entry {
    uint64_t len, offset, line_bases, line_bytes;
  };
  std::string path_;
  std::map<std::string, Entry> idx_;
  FILE* f_ = nullptr;
};

// ---------------------------------------------------------------- GTF2
struct GtfRecord {
  std::string seqname, feature, frame;
  uint64_t start = 0, end = 0;  // 1-based inclusive, as in the file
  char strand = '.';
  // bio::io::gff attributes() is a multimap; .get(k) yields the first value
  std::vector<std::pair<std::string, std::string>> attrs;
  const std::string* get(const char* k) const {
    for (auto& kv : attrs)
      if (kv.first == k) return &kv.second;
    return nullptr;
  }
};

// Parses one GTF2 line (bio 0.34 gff::Reader with GffType::GTF2: key/value separated by
// ' ', entries terminated by ';', surrounding quotes stripped). Returns false for
// comment / blank lines.
inline bool parse_gtf_line(const std::string& line, GtfRecord& r) {
  if (line.empty() || line[0] == '#') return false;
  auto t = split(line, '\t');
  if (t.size() < 9) throw IoError("malformed GTF line: " + line.substr(0, 80));
  r.seqname = t[0];
  r.feature = t[2];
  r.start = std::stoull(t[3]);
  r.end = std::stoull(t[4]);
  r.strand = t[6].empty() ? '.' : t[6][0];
  r.frame = t[7];
  r.attrs.clear();
  const std::string& a = t[8];
  size_t i = 0;
  while (i < a.size()) {
    while (i < a.size() && (a[i] == ' ' || a[i] == ';')) ++i;
    if (i >= a.size()) break;
    size_t ks = i;
    while (i < a.size() && a[i] != ' ' && a[i] != ';') ++i;
    std::string key = a.substr(ks, i - ks);
    while (i < a.size() && a[i] == ' ') ++i;
    std::string val;
    if (i < a.size() && a[i] == '"') {
      size_t e = a.find('"', i + 1);
      if (e == std::string::npos) e = a.size();
      val = a.substr(i + 1, e - i - 1);
      i = e + 1;
    } else {
      size_t vs = i;
      while (i < a.size() && a[i] != ';') ++i;
      val = a.substr(vs, i - vs);
      while (!val.empty() && val.back() == ' ') val.pop_back();
    }
    r.attrs.emplace_back(std::move(key), std::move(val));
    while (i < a.size() && a[i] != ';') ++i;
  }
  return true;
}

}  // namespace mphio
