// ingest.hpp — host side of the `somatic` sub-command up to the device boundary:
// GTF streaming and gene assembly (reference src/microphasing.rs:1982-2125), the per-gene read /
// variant / reference fetch (:894-942, src/common.rs:71-175) and hand-over to the Packer.
// rust-htslib's bam::RecordBuffer / bcf::buffer::RecordBuffer fetch semantics are restated from the
// crate's published behaviour (SURVEY.md Appendix C); the crate is not vendored under /root/reference.
#pragma once
#include <sys/mman.h>

#include <atomic>
#include <chrono>
#include <functional>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <deque>
#include <istream>
#include <memory>

#include "../io/bam_index.hpp"
#include "../io/hts_io.hpp"
#include "batch.hpp"

namespace mph {

inline uint64_t fnv1a(const std::string& s) {
  uint64_t h = 1469598103934665603ull;
  for (unsigned char c : s) { h ^= c; h *= 1099511628211ull; }
  return h;
}

// bam::RecordBuffer::fetch over a coordinate-sorted BAM: held in memory per contig, or read through its index
class ReadBuffer {
 public:
  // one alignment record. Sequence and qualities are NOT copied: the pointers go into the inflated BGZF batches, which the
  // buffer keeps alive (the threaded loader) or into the buffer's arenas (the sequential loader); CIGARs are copied into
  // aligned 32-bit storage.
  struct Rec {
    int32_t tid, pos;
    uint32_t end;  // CigarStringView::end_pos()
    uint32_t l_seq, n_cigar;
    uint16_t flag;
    uint8_t mapq;
    uint64_t qname_hash;
    const uint8_t* seq_p;   // BAM 4-bit bases
    const uint8_t* qual_p;  // raw phred
    const uint32_t* cig_p;
    bool is_unmapped() const { return flag & 4; }
  };

  explicit ReadBuffer(mphio::BamFile& bam) : bam_(bam) {
    tid_range_.assign(bam.ref_names.size(), {0, 0});
    if (bam.file_bytes()) recs_.reserve(bam.file_bytes() / 64 + 1024);  // ~100 compressed bytes per 150 bp record; untouched pages cost nothing
    if (bam.inflate_threads() > 1) {
      load_parallel(bam.inflate_threads());
    } else {
      // sequential loader (one core / MPH_IO_THREADS=1): records are copied into arenas; the arenas move while they grow,
      // so the records hold offsets until the load is over
      mphio::BamRecord r;
      while (bam.next(r)) {
        if (r.tid < 0 || size_t(r.tid) >= tid_range_.size()) continue;
        Rec x;
        x.tid = r.tid; x.pos = int32_t(r.pos); x.end = uint32_t(r.end_pos()); x.l_seq = r.l_seq; x.n_cigar = uint32_t(r.cigar.size());
        x.flag = r.flag; x.mapq = r.mapq; x.qname_hash = fnv1a_bytes(r.qname.data(), r.qname.size());
        x.seq_p = reinterpret_cast<const uint8_t*>(uintptr_t(seq_.size()));
        x.qual_p = reinterpret_cast<const uint8_t*>(uintptr_t(qual_.size()));
        x.cig_p = reinterpret_cast<const uint32_t*>(uintptr_t(cig_.size()));
        seq_.append(r.seq4.data(), r.seq4.size());
        qual_.append(r.qual.data(), r.qual.size());
        cig_.append(r.cigar.data(), r.cigar.size());
        recs_.append(&x, 1);
      }
      for (size_t i = 0; i < recs_.size(); ++i) {
        Rec& x = recs_[i];
        x.seq_p = seq_.data() + uintptr_t(x.seq_p);
        x.qual_p = qual_.data() + uintptr_t(x.qual_p);
        x.cig_p = cig_.data() + uintptr_t(x.cig_p);
      }
    }
    index_by_tid();
  }

  // Indexed mode: nothing is loaded up front. A re-fetch finds where to start through the index - a seek, or a read
  // forward when that start lies a little ahead of what has been read - and every fetch reads on lazily, only as far as
  // its end plus the one overflow record. Records point into the inflated batches; a batch is dropped by the buffer once
  // no record of the current fetch lies in it, and freed once no gene pins it (pins()).
  ReadBuffer(mphio::BamFile& bam, const mphio::BamIndex& index)
      : bam_(bam), index_(&index), read_on_bytes_(bam.inflate_threads() > 1 ? uint64_t(4) << 20 : uint64_t(64) << 10) {}

  // keeps an inflated batch alive
  using Pin = std::shared_ptr<const void>;

 private:
  // a growable array whose new elements are NOT value-initialised: the loader overwrites every byte it adds, and
  // zero-filling half a gigabyte first was a fifth of the load time
  template <class T>
  struct Arena {
    T* p = nullptr;
    size_t n = 0, cap = 0;
    Arena() = default;
    Arena(const Arena&) = delete;
    Arena& operator=(const Arena&) = delete;
    ~Arena() { free(p); }
    void reserve(size_t want) {
      if (want <= cap) return;
      T* q = static_cast<T*>(realloc(p, want * sizeof(T)));
      if (!q) throw std::bad_alloc();
      p = q;
      cap = want;
#ifdef MADV_HUGEPAGE
      // first touch of a few hundred MB costs one page fault per 4 KB otherwise: a third of the decode time
      if (want * sizeof(T) >= (size_t(8) << 20)) {
        const uintptr_t a = (reinterpret_cast<uintptr_t>(p) + 4095) & ~uintptr_t(4095);
        const uintptr_t e = (reinterpret_cast<uintptr_t>(p) + want * sizeof(T)) & ~uintptr_t(4095);
        if (e > a) madvise(reinterpret_cast<void*>(a), e - a, MADV_HUGEPAGE);
      }
#endif
    }
    void grow_to(size_t size) {
      if (size > cap) reserve(std::max(size, cap + cap / 2 + 4096));
      n = size;
    }
    void append(const T* src, size_t k) {
      const size_t at = n;
      grow_to(n + k);
      if (k) memcpy(p + at, src, k * sizeof(T));
    }
    size_t size() const { return n; }
    T* data() { return p; }
    const T* data() const { return p; }
    T& operator[](size_t i) { return p[i]; }
    const T& operator[](size_t i) const { return p[i]; }
  };

  // per contig: its records' range in recs_ (a coordinate-sorted BAM keeps each contig together; otherwise the records
  // are brought into contig order first, keeping the file order within a contig)
  void index_by_tid() {
    bool grouped = true;
    std::vector<uint8_t> seen(tid_range_.size(), 0);
    for (size_t i = 0; i < recs_.size() && grouped; ++i)
      if (i == 0 || recs_[i].tid != recs_[i - 1].tid) {
        if (seen[size_t(recs_[i].tid)]) grouped = false;
        seen[size_t(recs_[i].tid)] = 1;
      }
    if (!grouped) std::stable_sort(recs_.data(), recs_.data() + recs_.size(), [](const Rec& a, const Rec& b) { return a.tid < b.tid; });
    for (size_t i = 0; i < recs_.size();) {
      size_t j = i;
      while (j < recs_.size() && recs_[j].tid == recs_[i].tid) ++j;
      tid_range_[size_t(recs_[i].tid)] = {i, j};
      i = j;
    }
  }

  // decodes one framed record (p = first byte after the length prefix, bs = the prefix) in place; its CIGAR goes to `cig`
  static void decode_record(const uint8_t* p, int32_t bs, uint32_t* cig, Rec& x) {
    auto i32 = [&](size_t q) { int32_t v; memcpy(&v, p + q, 4); return v; };
    auto u16 = [&](size_t q) { uint16_t v; memcpy(&v, p + q, 2); return v; };
    x.tid = i32(0);
    x.pos = i32(4);
    const uint8_t l_read_name = p[8];
    x.mapq = p[9];
    x.n_cigar = u16(12);
    x.flag = u16(14);
    const int32_t l_seq = i32(16);
    if (l_seq < 0 || 32 + size_t(l_read_name) + 4 * size_t(x.n_cigar) + (size_t(l_seq) + 1) / 2 + size_t(l_seq) > size_t(bs)) throw mphio::IoError("corrupt BAM record");
    x.l_seq = uint32_t(l_seq);
    size_t q = 32;
    x.qname_hash = fnv1a_bytes(reinterpret_cast<const char*>(p + q), l_read_name ? l_read_name - 1 : 0);
    q += l_read_name;
    x.cig_p = cig;
    if (x.n_cigar) memcpy(cig, p + q, 4 * size_t(x.n_cigar));
    int64_t e = x.pos;  // CigarStringView::end_pos(): reference-consuming operations M, D, N, =, X
    for (uint32_t z = 0; z < x.n_cigar; ++z) {
      const uint32_t c = cig[z], op = c & 15;
      if (op == mphio::C_M || op == mphio::C_D || op == mphio::C_N || op == mphio::C_EQ || op == mphio::C_X) e += c >> 4;
    }
    x.end = uint32_t(e);
    q += 4 * size_t(x.n_cigar);
    x.seq_p = p + q;
    x.qual_p = p + q + (x.l_seq + 1) / 2;
  }

  // Threaded loader. The inflated batches are kept (records point into them: nothing but the CIGARs is copied).
  // Record boundaries are a dependent chain of length prefixes - one cache miss per record when a single thread walks it -
  // so every batch is cut into segments of ~1 MB that are framed and parsed in parallel: the first segment starts at the
  // known boundary, the others GUESS theirs (the first offset at which a few consecutive plausible record headers line
  // up) and walk on from there. The calling thread then checks, segment by segment, that the walk of everything before
  // ends exactly on the segment's guess; by induction every accepted boundary is a real one. A segment whose guess does
  // not match (or that found none) is framed again from the right offset on the calling thread. The parsed records of a
  // segment are copied into the record array once their position is known (also on the pool, beside the next batch).
  void load_parallel(unsigned threads) {
    struct Seg {
      const uint8_t* base = nullptr;  // the batch
      size_t size = 0;                // its bytes
      size_t lo = 0, hi = 0;          // records that START in [lo, hi) belong to this segment
      bool known = false;             // lo is a record boundary
      size_t guess = size_t(-1);      // first record start found (lo if known)
      size_t end = 0;                 // where the walk stopped: the first record start >= hi, or an incomplete record
      bool incomplete = false;        // ... the record at `end` does not fit the batch
      std::vector<Rec> recs;
      std::unique_ptr<uint32_t[]> cig;
      size_t rec0 = 0;
    };
    const int32_t n_ref = int32_t(tid_range_.size());
    // a record header that could be real (the checks htslib-based splitters use): false positives cost a fallback, nothing else
    auto plausible = [n_ref](const uint8_t* base, size_t size, size_t o) -> bool {
      if (o + 36 > size) return false;
      auto i32 = [&](size_t q) { int32_t v; memcpy(&v, base + o + q, 4); return v; };
      const int32_t bs = i32(0), tid = i32(4), pos = i32(8), l_seq = i32(20), ntid = i32(24), npos = i32(28);
      uint16_t n_cigar;
      memcpy(&n_cigar, base + o + 16, 2);
      const uint8_t l_name = base[o + 12];
      if (bs < 32 || bs > (1 << 26) || tid < -1 || tid >= n_ref || pos < -1 || ntid < -1 || ntid >= n_ref || npos < -1 || l_seq < 0 || l_name == 0) return false;
      if (32 + size_t(l_name) + 4 * size_t(n_cigar) + (size_t(l_seq) + 1) / 2 + size_t(l_seq) > size_t(bs)) return false;
      const size_t nul = o + 36 + l_name - 1;
      return nul >= size || base[nul] == 0;
    };
    // frames and parses the records starting in [from, sg.hi); fills sg.recs / sg.cig / sg.end / sg.incomplete
    auto walk = [](Seg& sg, size_t from) {
      std::vector<uint32_t> off;
      size_t o = from, n_cig = 0;
      sg.incomplete = false;
      while (o < sg.hi) {
        if (o + 4 > sg.size) { sg.incomplete = true; break; }
        int32_t bs;
        memcpy(&bs, sg.base + o, 4);
        if (bs < 32) throw mphio::IoError("corrupt BAM record");
        if (o + 4 + size_t(bs) > sg.size) { sg.incomplete = true; break; }
        uint16_t nc;
        memcpy(&nc, sg.base + o + 16, 2);
        if (32 + 4 * size_t(nc) > size_t(bs)) throw mphio::IoError("corrupt BAM record");
        n_cig += nc;
        off.push_back(uint32_t(o + 4));
        o += 4 + size_t(bs);
      }
      sg.end = o;
      sg.recs.resize(off.size());
      sg.cig.reset(new uint32_t[n_cig + 1]);
      uint32_t* cig = sg.cig.get();
      for (size_t i = 0; i < off.size(); ++i) {
        const uint8_t* p = sg.base + off[i];
        int32_t bs;
        memcpy(&bs, p - 4, 4);
        decode_record(p, bs, cig, sg.recs[i]);
        cig += sg.recs[i].n_cigar;
      }
    };
    struct Pool {
      std::mutex mu;
      std::condition_variable cv_work, cv_idle;
      std::deque<std::function<void()>> queue;
      size_t running = 0;
      bool closed = false;
      std::exception_ptr err;
      std::vector<std::thread> threads;
    } pool;
    auto worker = [&] {
      for (;;) {
        std::function<void()> job;
        {
          std::unique_lock<std::mutex> lk(pool.mu);
          pool.cv_work.wait(lk, [&] { return pool.closed || !pool.queue.empty(); });
          if (pool.queue.empty()) return;
          job = std::move(pool.queue.front());
          pool.queue.pop_front();
          ++pool.running;
        }
        try {
          job();
        } catch (...) {
          std::lock_guard<std::mutex> lk(pool.mu);
          if (!pool.err) pool.err = std::current_exception();
        }
        {
          std::lock_guard<std::mutex> lk(pool.mu);
          --pool.running;
        }
        pool.cv_idle.notify_all();
      }
    };
    auto submit = [&](std::function<void()> job) {
      {
        std::lock_guard<std::mutex> lk(pool.mu);
        pool.queue.push_back(std::move(job));
      }
      pool.cv_work.notify_one();
    };
    auto wait_idle = [&] {
      std::unique_lock<std::mutex> lk(pool.mu);
      pool.cv_idle.wait(lk, [&] { return pool.queue.empty() && pool.running == 0; });
      if (pool.err) std::rethrow_exception(pool.err);
    };
    auto shutdown = [&] {
      {
        std::lock_guard<std::mutex> lk(pool.mu);
        pool.closed = true;
      }
      pool.cv_work.notify_all();
      for (auto& t : pool.threads) t.join();
      pool.threads.clear();
    };
    // the inflate pool of the BGZF reader uses `threads` threads of its own; a few more for the parse are enough
    unsigned n_workers = std::max(2u, std::min(threads / 4, 6u));
    if (const char* e = getenv("MPH_PARSE_THREADS")) n_workers = unsigned(std::max(1, atoi(e)));
    for (unsigned ti = 0; ti < n_workers; ++ti) pool.threads.emplace_back(worker);
    const bool trace = getenv("MPH_IO_TRACE") != nullptr;  // measurement hook: where the loader's wall time goes
    double t_wait = 0, t_frame = 0, t_check = 0;
    size_t n_fallback = 0, n_segs = 0;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto since = [](std::chrono::steady_clock::time_point a) { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count(); };
    constexpr size_t SEG_BYTES = size_t(1) << 20;
    const bool bad_guess_hook = getenv("MPH_IO_BAD_GUESS") != nullptr;  // test hook: every guessed boundary is discarded -> all segments go through the checker's re-framing
    std::mutex cig_mu;
    // appends the records of a framed segment: the copy itself runs on the pool
    std::deque<std::unique_ptr<Seg>> in_flight;  // segments whose copy may still be running
    auto append = [&](std::unique_ptr<Seg> sgp) {
      Seg& sg = *sgp;
      if (sg.recs.empty()) return;
      const size_t n = sg.recs.size();
      if (recs_.size() + n > recs_.cap) {
        wait_idle();  // the record array must not move while copies into it are running
        in_flight.clear();
        recs_.reserve(std::max(recs_.size() + n, recs_.cap + recs_.cap / 2 + 4096));
      }
      sg.rec0 = recs_.size();
      recs_.grow_to(recs_.size() + n);
      Seg* raw = sgp.get();
      in_flight.push_back(std::move(sgp));
      submit([this, raw, &cig_mu] {
        memcpy(static_cast<void*>(recs_.data() + raw->rec0), raw->recs.data(), raw->recs.size() * sizeof(Rec));
        std::vector<Rec>().swap(raw->recs);
        std::lock_guard<std::mutex> lk(cig_mu);
        cig_blocks_.push_back(std::move(raw->cig));
      });
    };
    try {
      std::vector<uint8_t> carry;  // the head of a record whose tail is in the next batch
      // the batch whose segments are being framed on the pool while the calling thread waits for the next inflated batch
      struct Pending {
        std::vector<std::unique_ptr<Seg>> segs;
        const uint8_t* base = nullptr;
        size_t size = 0, o = 0;
        std::atomic<size_t> left{0};
        std::mutex mu;
        std::condition_variable cv;
        bool active = false;
      } pend;
      auto start_batch = [&](const uint8_t* base, size_t size, size_t o) {
        pend.segs.clear();
        pend.base = base; pend.size = size; pend.o = o;
        for (size_t lo = o; lo < size;) {
          const size_t hi = std::min(size, (lo / SEG_BYTES + 1) * SEG_BYTES);
          std::unique_ptr<Seg> sg(new Seg);
          sg->base = base; sg->size = size; sg->lo = lo; sg->hi = hi; sg->known = lo == o;
          pend.segs.push_back(std::move(sg));
          lo = hi;
        }
        n_segs += pend.segs.size();
        pend.left = pend.segs.size();
        pend.active = true;
        for (auto& sgp : pend.segs) {
          Seg* sg = sgp.get();
          Pending* pd = &pend;
          submit([sg, pd, &plausible, &walk, bad_guess_hook] {
            struct Done {
              Pending* pd;
              ~Done() { std::lock_guard<std::mutex> lk(pd->mu); if (--pd->left == 0) pd->cv.notify_all(); }
            } done{pd};
            size_t start = sg->lo;
            if (!sg->known) {
              start = size_t(-1);
              for (size_t p = sg->lo; p < sg->hi; ++p) {
                if (!plausible(sg->base, sg->size, p)) continue;
                size_t q = p;  // a few records further on must look like records as well
                bool ok = true;
                for (int k = 0; k < 4 && ok; ++k) {
                  int32_t bs;
                  memcpy(&bs, sg->base + q, 4);
                  q += 4 + size_t(bs);
                  if (q + 36 > sg->size) break;
                  ok = plausible(sg->base, sg->size, q);
                }
                if (ok) { start = p; break; }
              }
            }
            sg->guess = start;
            if (start == size_t(-1)) return;
            if (sg->known) { walk(*sg, start); return; }
            // a guessed boundary may be wrong: whatever the walk from it runs into is not an error of the file. The
            // checker frames the segment again from the real boundary, and a corrupt record is reported from there.
            try {
              if (bad_guess_hook) throw mphio::IoError("test hook");
              walk(*sg, start);
            } catch (const mphio::IoError&) {
              sg->guess = size_t(-1);
              sg->recs.clear();
            }
          });
        }
      };
      // waits for the pending batch, checks the chain of boundaries in order, hands the records over, leaves the tail in `carry`
      auto finish_batch = [&] {
        if (!pend.active) return;
        pend.active = false;
        auto t0 = now();
        {
          std::unique_lock<std::mutex> lk(pend.mu);
          pend.cv.wait(lk, [&] { return pend.left.load() == 0; });
        }
        {
          std::lock_guard<std::mutex> lk(pool.mu);
          if (pool.err) std::rethrow_exception(pool.err);
        }
        t_frame += since(t0);
        t0 = now();
        size_t expect = pend.o;
        bool final_incomplete = false;
        for (auto& sgp : pend.segs) {
          Seg& sg = *sgp;
          if (final_incomplete || expect >= sg.hi) continue;  // the segment lies inside a record that started earlier
          if (sg.guess != expect) {  // wrong or missing guess: frame it again from the right boundary
            ++n_fallback;
            walk(sg, expect);
          }
          expect = sg.end;
          final_incomplete = sg.incomplete;
          append(std::move(sgp));
        }
        if (expect < pend.size) carry.assign(pend.base + expect, pend.base + pend.size);
        pend.segs.clear();
        t_check += since(t0);
      };
      bool more = true;
      while (more) {
        auto t0 = now();
        mphio::RawBytes chunk;
        more = bam_.next_chunk(chunk);  // (the previous batch is being framed on the pool meanwhile)
        t_wait += since(t0);
        finish_batch();
        if (!more) chunk.clear();
        if (chunk.size() > 0xFFFFFF00ull) throw mphio::IoError("inflated BGZF batch too large");
        size_t o = 0;
        if (!carry.empty()) {
          // finish the record that started in the previous batch
          if (carry.size() < 4) {
            const size_t take = std::min(4 - carry.size(), chunk.size());
            carry.insert(carry.end(), chunk.begin(), chunk.begin() + long(take));
            o += take;
          }
          if (carry.size() >= 4) {
            int32_t bs;
            memcpy(&bs, carry.data(), 4);
            if (bs < 32) throw mphio::IoError("corrupt BAM record");
            const size_t need = 4 + size_t(bs);
            const size_t take = std::min(need - carry.size(), chunk.size() - o);
            carry.insert(carry.end(), chunk.begin() + long(o), chunk.begin() + long(o + take));
            o += take;
            if (carry.size() == need) {
              straddlers_.emplace_back(std::move(carry));
              carry.clear();
              std::unique_ptr<Seg> sg(new Seg);
              sg->base = straddlers_.back().data(); sg->size = straddlers_.back().size(); sg->lo = 0; sg->hi = sg->size;
              walk(*sg, 0);
              append(std::move(sg));
            }
          }
          if (!more && !carry.empty()) throw mphio::IoError("truncated BAM record");
        }
        const uint8_t* base = chunk.data();
        const size_t size = chunk.size();
        if (size) chunks_.push_back(std::move(chunk));  // the buffer itself does not move: pointers into it stay valid
        if (o < size) start_batch(base, size, o);
      }
      finish_batch();
      if (!carry.empty()) throw mphio::IoError("truncated BAM record");
      wait_idle();
      in_flight.clear();
      shutdown();
      if (pool.err) std::rethrow_exception(pool.err);
      if (trace)
        fprintf(stderr, "[mph io] BAM load: waiting for inflated batches %.1f ms, parallel framing + header parse %.1f, boundary check + hand-over %.1f (%zu segments, %zu framed again)\n",
                t_wait, t_frame, t_check, n_segs, n_fallback);
    } catch (...) {
      try { shutdown(); } catch (...) {}
      throw;
    }
    // records of contigs the header does not know are dropped (compaction in place keeps the file order)
    size_t keep = 0;
    for (size_t i = 0; i < recs_.size(); ++i)
      if (recs_[i].tid >= 0 && size_t(recs_[i].tid) < tid_range_.size()) recs_[keep++] = recs_[i];
    recs_.grow_to(keep);
  }

 public:
  const uint8_t* seq4(const Rec& r) const { return r.seq_p; }
  const uint8_t* qual(const Rec& r) const { return r.qual_p; }
  const uint32_t* cigar(const Rec& r) const { return r.cig_p; }
  size_t n_records() const { return recs_.size(); }

  // bam::RecordBuffer::fetch (rust-htslib 0.36) over the in-memory records: the mapped records with pos < end, kept
  // across calls for overlapping / adjacent queries. An indexed re-fetch yields every record that overlaps `start`
  // (htslib's iterator: pos < region end and end_pos > region start) and the buffer's loop has no start test of its own,
  // so reads that begin left of the gene and reach into it are buffered; without a re-fetch the records left of `start`
  // are dropped from the front.
  const std::deque<const Rec*>& fetch(const std::string& chrom, uint64_t start, uint64_t end) {
    if (overflow_) { inner_.push_back(overflow_); overflow_ = nullptr; }
    auto it = bam_.tid_of.find(chrom);
    if (it == bam_.tid_of.end()) throw std::runtime_error("sequence " + chrom + " not found in BAM header");
    const int tid = it->second;
    struct View {
      const Rec* p;
      size_t n;
      size_t size() const { return n; }
      const Rec& operator[](size_t i) const { return p[i]; }
    };
    const bool refetch = inner_.empty() || uint64_t(inner_.back()->pos) < start || inner_.front()->tid != tid ||
                         uint64_t(inner_.front()->pos) > start;
    if (index_) return fetch_indexed(tid, start, end, refetch);
    const View v{recs_.data() + tid_range_[size_t(tid)].first, tid_range_[size_t(tid)].second - tid_range_[size_t(tid)].first};
    if (refetch) {
      inner_.clear();
      tid_ = tid;
      cur_ = 0;
      // an index query starts at the first record overlapping `start`
      while (cur_ < v.size() && uint64_t(v[cur_].pos) < start && (v[cur_].is_unmapped() || uint64_t(v[cur_].end) <= start)) ++cur_;
    } else {
      while (!inner_.empty() && uint64_t(inner_.front()->pos) < start) inner_.pop_front();
    }
    while (tid_ == tid && cur_ < v.size()) {
      const Rec* r = &v[cur_++];
      if (r->is_unmapped()) continue;
      const uint64_t pos = uint64_t(r->pos);
      if (pos >= end) { overflow_ = r; break; }
      if (pos >= start || (refetch && uint64_t(r->end) > start)) inner_.push_back(r);
    }
    return inner_;
  }

  // indexed mode: the batches the records of the last fetch (and its overflow record) point into; empty otherwise
  std::vector<Pin> pins() const { return std::vector<Pin>(live_.begin(), live_.begin() + long(std::min(live_.size(), bi_ + 1))); }

 private:
  // ---- indexed mode
  // one inflated batch and the records that start in it; a record that began in the previous batch is completed in `head`
  struct Block {
    mphio::RawBytes data;
    std::vector<uint8_t> head;
    std::vector<Rec> recs;
    std::vector<uint64_t> voff;  // virtual offset of each record
    std::unique_ptr<uint32_t[]> cig;
  };

  const std::deque<const Rec*>& fetch_indexed(int tid, uint64_t start, uint64_t end, bool refetch) {
    if (refetch) {
      inner_.clear();
      tid_ = tid;
      position(index_->first_offset(tid, int64_t(std::min<uint64_t>(start, uint64_t(INT64_MAX)))));
    } else {
      while (!inner_.empty() && uint64_t(inner_.front()->pos) < start) inner_.pop_front();
    }
    // the whole-file loop over the contig's records, which end where the next contig's begin
    for (const Rec* r; (r = peek()) && r->tid == tid_;) {
      ++ri_;
      if (r->is_unmapped()) continue;
      const uint64_t pos = uint64_t(r->pos);
      if (pos >= end) { overflow_ = r; break; }
      if (pos >= start || (refetch && uint64_t(r->end) > start)) inner_.push_back(r);
    }
    // batches before the one holding the earliest record still needed go (the genes that point into them pin them)
    const Rec* keep = !inner_.empty() ? inner_.front() : overflow_;
    size_t b = bi_;
    for (size_t i = 0; keep && i < bi_; ++i)
      if (keep >= live_[i]->recs.data() && keep < live_[i]->recs.data() + live_[i]->recs.size()) { b = i; break; }
    live_.erase(live_.begin(), live_.begin() + long(std::min(b, live_.size())));
    bi_ -= std::min(b, bi_);
    return inner_;
  }

  // moves the cursor to the first record at or after virtual offset t (BamIndex::NONE: the contig has none to give)
  void position(uint64_t t) {
    contig_done_ = t == mphio::BamIndex::NONE;
    if (contig_done_) return;
    if (!live_.empty() && !live_.front()->voff.empty() && t >= live_.front()->voff.front() && t < stream_voff_) {
      for (size_t b = 0; b < live_.size(); ++b) {  // among the records read since the last seek
        const auto& v = live_[b]->voff;
        auto it = std::lower_bound(v.begin(), v.end(), t);
        if (it != v.end()) { bi_ = b; ri_ = size_t(it - v.begin()); return; }
      }
    }
    live_.clear();
    bi_ = ri_ = 0;
    if (!eof_ && t >= stream_voff_ && (t >> 16) - (stream_voff_ >> 16) <= read_on_bytes_) {
      while (read_block()) {
        const auto& v = live_.back()->voff;
        auto it = std::lower_bound(v.begin(), v.end(), t);
        if (it != v.end()) {
          live_.erase(live_.begin(), live_.end() - 1);
          ri_ = size_t(it - v.begin());
          return;
        }
      }
      live_.clear();  // no record at or after t
      return;
    }
    carry_.clear();
    eof_ = false;
    try {
      bam_.seek(t);
    } catch (const mphio::IoError& e) {
      throw mphio::IoError(std::string(e.what()) + " (offset from " + index_->path() + ")");
    }
    stream_voff_ = t;
  }

  // the record under the cursor, reading on as needed; nullptr at the end of the file or of a contig without records
  const Rec* peek() {
    if (contig_done_) return nullptr;
    for (;;) {
      if (bi_ < live_.size()) {
        if (ri_ < live_[bi_]->recs.size()) return &live_[bi_]->recs[ri_];
        if (bi_ + 1 < live_.size()) { ++bi_; ri_ = 0; continue; }
      }
      if (!read_block()) return nullptr;
    }
  }

  // frames and decodes the next inflated batch into a block at the end of live_; false at the end of the file
  bool read_block() {
    if (eof_) return false;
    std::shared_ptr<Block> blk(new Block);
    size_t o = 0;
    std::vector<mphio::BgzfSpan> spans;
    if (!bam_.next_chunk(blk->data, o, spans)) {
      eof_ = true;
      if (!carry_.empty()) throw mphio::IoError("truncated BAM record");
      return false;
    }
    const uint8_t* base = blk->data.data();
    const size_t size = blk->data.size();
    size_t si = 0;
    auto voff_at = [&](size_t at) {
      while (si + 1 < spans.size() && spans[si + 1].ooff <= int64_t(at)) ++si;
      return spans[si].coff << 16 | uint64_t(int64_t(at) - spans[si].ooff);
    };
    std::vector<std::pair<const uint8_t*, uint64_t>> at;  // record bytes after the length prefix, virtual offset
    size_t n_cig = 0;
    auto frame = [&](const uint8_t* p, size_t avail, uint64_t voff) -> size_t {  // 0: incomplete
      if (avail < 4) return 0;
      int32_t bs;
      memcpy(&bs, p, 4);
      if (bs < 32) throw mphio::IoError("corrupt BAM record");
      if (avail < 4 + size_t(bs)) return 0;
      uint16_t nc;
      memcpy(&nc, p + 16, 2);
      if (32 + 4 * size_t(nc) > size_t(bs)) throw mphio::IoError("corrupt BAM record");
      n_cig += nc;
      at.emplace_back(p + 4, voff);
      return 4 + size_t(bs);
    };
    if (!carry_.empty()) {  // the record that began in the previous batch: its length prefix first, then the rest
      size_t take = std::min(size_t(4) - std::min<size_t>(4, carry_.size()), size - o);
      carry_.insert(carry_.end(), base + o, base + o + take);
      o += take;
      if (carry_.size() >= 4) {
        int32_t bs;
        memcpy(&bs, carry_.data(), 4);
        if (bs < 32) throw mphio::IoError("corrupt BAM record");
        take = std::min(4 + size_t(bs) - carry_.size(), size - o);
        carry_.insert(carry_.end(), base + o, base + o + take);
        o += take;
        if (carry_.size() == 4 + size_t(bs)) {
          blk->head.swap(carry_);
          carry_.clear();
          frame(blk->head.data(), blk->head.size(), carry_voff_);
        }
      }
    }
    while (carry_.empty()) {
      const size_t n = frame(base + o, size - o, voff_at(o));
      if (!n) break;
      o += n;
    }
    if (carry_.empty() && o < size) {
      carry_voff_ = voff_at(o);
      carry_.assign(base + o, base + size);
    }
    stream_voff_ = carry_.empty() ? voff_at(size) : carry_voff_;
    blk->recs.resize(at.size());
    blk->voff.resize(at.size());
    blk->cig.reset(new uint32_t[n_cig + 1]);
    uint32_t* cig = blk->cig.get();
    for (size_t i = 0; i < at.size(); ++i) {
      int32_t bs;
      memcpy(&bs, at[i].first - 4, 4);
      decode_record(at[i].first, bs, cig, blk->recs[i]);
      cig += blk->recs[i].n_cigar;
      blk->voff[i] = at[i].second;
    }
    live_.push_back(std::move(blk));
    return true;
  }

  static uint64_t fnv1a_bytes(const char* p, size_t n) {
    uint64_t h = 1469598103934665603ull;
    for (size_t i = 0; i < n; ++i) { h ^= uint8_t(p[i]); h *= 1099511628211ull; }
    return h;
  }
  mphio::BamFile& bam_;
  Arena<Rec> recs_;                                     // every mapped-to-a-known-contig record, contig by contig, file order
  std::vector<std::pair<size_t, size_t>> tid_range_;    // per contig: [first, last) in recs_
  Arena<uint8_t> seq_, qual_;                           // sequential loader only
  Arena<uint32_t> cig_;
  std::deque<mphio::RawBytes> chunks_;                  // threaded loader: the inflated batches the records point into,
  std::deque<std::vector<uint8_t>> straddlers_;         // the records that straddle two batches,
  std::vector<std::unique_ptr<uint32_t[]>> cig_blocks_; // and the CIGARs, one aligned block per slice of records
  std::deque<const Rec*> inner_;
  const Rec* overflow_ = nullptr;
  int tid_ = -1;
  size_t cur_ = 0;
  // indexed mode
  const mphio::BamIndex* index_ = nullptr;
  // A start at most this many compressed bytes ahead of what has been read is reached by reading on instead of a seek.
  // A seek of the sequential reader costs nothing, one of the threaded reader throws away its read-ahead (three batches).
  uint64_t read_on_bytes_ = 0;
  std::deque<std::shared_ptr<Block>> live_;  // the batches read since the last seek that may still be needed
  size_t bi_ = 0, ri_ = 0;                    // cursor: block in live_, record in it
  std::vector<uint8_t> carry_;                // the head of a record whose tail is in the next batch
  uint64_t carry_voff_ = 0, stream_voff_ = 0; // its virtual offset; that of the first byte not yet framed
  bool eof_ = false, contig_done_ = false;
};

// bcf::Reader (streaming) + bcf::buffer::RecordBuffer::fetch
class VariantBuffer {
 public:
  explicit VariantBuffer(mphio::VcfFile& vcf) : vcf_(vcf) {}
  const std::deque<mphio::VcfRecord>& fetch(const std::string& chrom, uint64_t start, uint64_t end) {
    const int rid = vcf_.name2rid(chrom);
    if (rid < 0) throw std::runtime_error("contig " + chrom + " not found in VCF header");
    if (!ring_.empty()) {
      if (ring_.back().rid != rid) { ring_.swap(ring2_); ring2_.clear(); }
      else drain_left(rid, start);
    } else if (!ring2_.empty()) {
      ring_.swap(ring2_); ring2_.clear();
      drain_left(rid, start);
    }
    if (!ring2_.empty()) return ring_;
    if (have_overflow_) {
      const uint64_t pos = uint64_t(overflow_.pos);
      if (pos >= start) {
        if (pos <= end) { ring_.push_back(overflow_); have_overflow_ = false; }
        else return ring_;
      } else {
        have_overflow_ = false;
      }
    }
    mphio::VcfRecord rec;
    while (vcf_.next(rec)) {
      const uint64_t pos = uint64_t(rec.pos);
      if (rec.rid == rid) {
        if (pos >= end) { overflow_ = rec; have_overflow_ = true; break; }
        if (pos >= start) ring_.push_back(rec);
      } else if (rec.rid > rid) {
        ring2_.push_back(rec);
        break;
      }
    }
    return ring_;
  }

 private:
  void drain_left(int rid, uint64_t start) {
    while (!ring_.empty() && ring_.front().rid == rid && uint64_t(ring_.front().pos) < start) ring_.pop_front();
  }
  mphio::VcfFile& vcf_;
  std::deque<mphio::VcfRecord> ring_, ring2_;
  mphio::VcfRecord overflow_;
  bool have_overflow_ = false;
};

// Variant::new (common.rs:71-175)
inline std::vector<HostVariant> alleles_of(const mphio::VcfFile& vcf, const mphio::VcfRecord& rec, bool warn_only) {
  auto warn_or_error = [&](const std::string& msg) {
    fprintf(stderr, "%s\n", msg.c_str());
    if (!warn_only) throw Fatal(msg);
  };
  const bool germline = !(vcf.somatic_defined && rec.somatic_flag);
  std::string ann;
  if (vcf.ann_defined) {
    if (!rec.has_ann) throw Fatal("called `Option::unwrap()` on a `None` value (INFO/ANN declared in the header but absent)");
    ann = rec.ann_first;
  }
  std::string pc;
  for (auto& f : mphio::split(ann, '|'))
    if (f.find("p.") != std::string::npos) { pc = f; break; }
  std::vector<HostVariant> out;
  if (rec.pos < 0 || rec.pos > 0xFFFFFFF0ll) throw Unsupported("variant position beyond 32 bits");
  for (const std::string& a : rec.alts) {
    HostVariant v;
    v.pos = uint32_t(rec.pos);
    v.germline = germline;
    v.prot_change = pc;
    if (a.size() == 1 && rec.ref.size() > 1) {
      v.kind = MPH_DEL;
      v.len = uint32_t(rec.ref.size() - 1);
      out.push_back(v);
    } else if (a.size() > 1 && rec.ref.size() == 1) {
      if (a[0] == '<') {
        if (a == "<DEL>") {
          std::string where = " contig " + std::to_string(rec.rid) + " pos " + std::to_string(rec.pos);
          if (!vcf.svlen_defined || !rec.has_svlen) warn_or_error("Found no 'SVLEN' info tag for <DEL> alternative allele at" + where);
          else if (rec.svlen.size() > 1) warn_or_error("microphaser does not handle multiallelic records. Please normalize, e.g. with `bcftools norm -m-`.");
          else if (rec.svlen[0] == INT64_MIN) warn_or_error("Found no 'SVLEN' info tag for <DEL> alternative allele on" + where);
          else {
            const int64_t l = rec.svlen[0] < 0 ? -rec.svlen[0] : rec.svlen[0];
            if (l > 0x7FFFFFFF) throw Unsupported("deletion longer than 2^31");
            v.kind = MPH_DEL;
            v.len = uint32_t(l);
            out.push_back(v);
          }
        } else {
          warn_or_error("Alternative allele type '" + a + "' not yet supported.");
        }
      } else {
        v.kind = MPH_INS;
        v.ins = a;
        v.len = uint32_t(a.size() - 1);
        out.push_back(v);
      }
    } else if (a.size() == 1 && rec.ref.size() == 1) {
      v.kind = MPH_SNV;
      v.alt = uint8_t(a[0]);
      out.push_back(v);
    } else {
      fprintf(stderr, "Unsupported variant %s -> %s\n", rec.ref.c_str(), a.c_str());
    }
  }
  return out;
}

struct ParsedGene {
  HostGene gene;
  std::string biotype;
};

// GTF streaming rules of `phase` (:1982-2125): gene / transcript / CDS / start_codon / three_prime_utr
inline std::vector<ParsedGene> read_gtf(std::istream& in, int mode = 0) {
  std::vector<ParsedGene> genes;
  bool start_codon_found = false, three_prime_found = false;
  std::string last_chrom = "not_yet_set";
  uint64_t last_start = 0;
  std::string line;
  mphio::GtfRecord r;
  auto need = [](const mphio::GtfRecord& rec, const char* k, const char* msg) -> const std::string& {
    const std::string* v = rec.get(k);
    if (!v) throw Fatal(msg);
    return *v;
  };
  auto frame_of = [](const std::string& f) -> uint32_t {
    if (f == ".") return 0;
    if (f.empty()) throw Fatal("ParseIntError (GTF frame)");
    uint32_t v = 0;
    for (char c : f) {
      if (c < '0' || c > '9') throw Fatal("ParseIntError (GTF frame)");
      v = v * 10 + uint32_t(c - '0');
    }
    return v;
  };
  auto cur_tx = [&](const char* m1, const char* m2) -> HostTranscript& {
    if (genes.empty()) throw Fatal(m1);
    if (genes.back().gene.transcripts.empty()) throw Fatal(m2);
    return genes.back().gene.transcripts.back();
  };
  while (std::getline(in, line)) {
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (!mphio::parse_gtf_line(line, r)) continue;
    if (r.end > 0xFFFFFF00ull) throw Unsupported("coordinate beyond 32 bits");
    if (r.feature == "gene") {
      if (!genes.empty()) {
        last_chrom = genes.back().gene.chrom;
        last_start = genes.back().gene.start;
      }
      const std::string& gene_name = need(r, "gene_name", "missing gene_name in GTF");
      if (last_chrom == r.seqname && !(last_start <= r.start))
        throw Fatal("Your GTF file is not sorted correctly. Gene " + gene_name + " starts at " + std::to_string(r.start) +
                    ", while previous gene record started at " + std::to_string(last_start) + ".");
      ParsedGene pg;
      pg.gene.id = need(r, "gene_id", "missing gene_id in GTF");
      pg.gene.name = gene_name;
      pg.gene.chrom = r.seqname;
      pg.gene.start = uint32_t(r.start - 1);
      pg.gene.end = uint32_t(r.end);
      frame_of(r.frame);
      pg.biotype = need(r, "gene_biotype", "missing gene_biotype in GTF");
      genes.push_back(std::move(pg));
    } else if (r.feature == "transcript") {
      start_codon_found = false;
      three_prime_found = false;
      if (genes.empty()) throw Fatal("no gene record before transcript in GTF");
      HostTranscript t;
      t.id = need(r, "transcript_id", "missing transcript_id attribute in GTF");
      need(r, "transcript_biotype", "missing transcript_biotype in GTF");
      if (r.strand == '+') t.reverse = false;
      else if (r.strand == '-') t.reverse = true;
      else throw Fatal("missing strand information in GTF");
      genes.back().gene.transcripts.push_back(std::move(t));
    } else if (r.feature == "CDS") {
      HostTranscript& t = cur_tx("no gene record before exon in GTF", "no transcript record before exon in GTF");
      t.exons.push_back(HostExon{uint32_t(r.start - 1), uint32_t(r.end), frame_of(r.frame)});
    } else if (r.feature == "start_codon") {
      if (start_codon_found) continue;
      start_codon_found = true;
      HostTranscript& t = cur_tx("no gene record before start_codon in GTF", "no transcript record before start codon in GTF");
      if (t.exons.empty()) throw Fatal("no exon record before start codon in GTF");
      if (r.strand == '+') t.exons.back().start = uint32_t(r.start - 1);
      else t.exons.back().end = uint32_t(r.end);
    } else if (r.feature == "three_prime_utr" && mode == 0) {  // normal mode ignores UTR rows (normal_microphasing.rs:1405-1432)
      HostTranscript& t = cur_tx("no gene record before exon in GTF", "no transcript record before exon in GTF");
      if (three_prime_found) {
        t.exons.push_back(HostExon{uint32_t(r.start - 1), uint32_t(r.end), frame_of(r.frame)});
      } else {
        three_prime_found = true;
        if (t.exons.empty()) throw Fatal("no exon record before start codon in GTF");
        if (r.strand == '+') t.exons.back().end = uint32_t(r.end);
        else t.exons.back().start = uint32_t(r.start - 1);
      }
    }
  }
  return genes;
}

struct IngestOptions {
  uint32_t window_len = 27;
  bool warn_only = false;
  uint32_t min_mapq = 5;  // somatic: rec.mapq() < 5 is skipped (:910); normal mode has no filter
  int mode = 0;
};

// Everything phase_gene fetches for one gene (:894-942), held until it is packed.
struct GeneInput {
  HostGene gene;
  std::vector<HostRead> reads;  // point into records owned by the ReadBuffer
  // lazy form (file drivers): the buffered records themselves; `reads` is built from them when the gene is packed, which
  // happens on the packing threads instead of the single thread that walks the GTF
  std::vector<const ReadBuffer::Rec*> recs;
  std::vector<ReadBuffer::Pin> pins;  // indexed mode: the inflated batches `recs` point into, released once packed
  size_t n_reads = 0;
  uint32_t max_read_len = 0;
  void materialize() {
    if (!reads.empty() || recs.empty()) return;
    reads.reserve(recs.size());
    for (const ReadBuffer::Rec* rec : recs) {
      HostRead h;
      h.start = uint32_t(rec->pos);
      h.end = rec->end;
      h.l_seq = rec->l_seq;
      h.seq4 = rec->seq_p;
      h.qual = rec->qual_p;
      h.cigar = rec->cig_p;
      h.n_cigar = rec->n_cigar;
      h.qname_hash = rec->qname_hash;
      reads.push_back(h);
    }
    std::vector<const ReadBuffer::Rec*>().swap(recs);
  }
  std::vector<std::vector<HostVariant>> sites;
  std::vector<uint8_t> refseq;
};

// the buffered reads of the gene that pass the mapq filter (:905-920)
inline void fetch_reads(GeneInput& gi, ReadBuffer& reads, const IngestOptions& opt) {
  const HostGene& g = gi.gene;
  const auto& rb = reads.fetch(g.chrom, g.start, g.end);
  gi.recs.reserve(rb.size());
  for (auto& rec : rb) {
    if (rec->mapq < opt.min_mapq) continue;
    if (rec->l_seq > gi.max_read_len) gi.max_read_len = rec->l_seq;
    gi.recs.push_back(rec);
  }
  gi.n_reads = gi.recs.size();
  gi.pins = reads.pins();
}

// variant_tree.insert(rec.pos(), Variant::new(rec)): a later record at the same position replaces the earlier (:937)
inline void fetch_variants(GeneInput& gi, VariantBuffer& variants, const mphio::VcfFile& vcf, const IngestOptions& opt) {
  const HostGene& g = gi.gene;
  std::map<uint32_t, std::vector<HostVariant>> tree;
  for (auto& rec : variants.fetch(g.chrom, g.start, g.end)) tree[uint32_t(rec.pos)] = alleles_of(vcf, rec, opt.warn_only);
  for (auto& kv : tree)
    if (!kv.second.empty()) gi.sites.push_back(std::move(kv.second));
}

// One gene in the reference's one-pass order (:894-942): reference slice, reads, variants. The indexed paths fetch gene
// by gene like this, so that nothing of a gene is held longer than it takes to pack it.
inline GeneInput fetch_gene(HostGene&& g, ReadBuffer& reads, VariantBuffer& variants, const mphio::VcfFile& vcf, mphio::FastaIndexed& fasta,
                            const IngestOptions& opt) {
  GeneInput gi;
  gi.gene = std::move(g);
  fasta.fetch(gi.gene.chrom, gi.gene.start, uint64_t(gi.gene.end) + 100, gi.refseq);  // end_overflow (:895-901)
  fetch_reads(gi, reads, opt);
  fetch_variants(gi, variants, vcf, opt);
  return gi;
}

// Streams the GTF and fetches reads / variants / reference for every protein-coding gene, in GTF order.
// `reads_ready()` returns the loaded ReadBuffer, blocking until it is there: the file drivers load the BAM on another thread
// while this one parses the GTF and fetches the reference slices and variants (a third of the per-gene work), and only the
// read fetch waits for it. Errors keep the order of the one-pass loop (per gene: reference, reads, variants), and a failure
// of the BAM load itself comes before all of them, as it did when the buffer was built first.
template <class ReadsReady>
inline std::vector<GeneInput> ingest_genes_with(std::istream& gtf, ReadsReady&& reads_ready, mphio::VcfFile& vcf, mphio::FastaIndexed& fasta,
                                                const IngestOptions& opt, bool lazy_reads) {
  std::vector<ParsedGene> genes;
  try {
    genes = read_gtf(gtf, opt.mode);
  } catch (...) {
    reads_ready();  // a broken BAM is reported first
    throw;
  }
  VariantBuffer variants(vcf);
  std::vector<GeneInput> out;
  std::exception_ptr stashed;
  size_t stash_gene = size_t(-1);
  int stash_stage = 0;  // 0: reference fetch, 2: variants
  for (auto& pg : genes) {
    if (pg.biotype != "protein_coding") continue;  // :1964
    GeneInput gi;
    gi.gene = std::move(pg.gene);
    const HostGene& g = gi.gene;
    int stage = 0;
    try {
      fasta.fetch(g.chrom, g.start, uint64_t(g.end) + 100, gi.refseq);  // end_overflow (:895-901)
      stage = 2;
      fetch_variants(gi, variants, vcf, opt);
    } catch (...) {
      stashed = std::current_exception();
      stash_gene = out.size();
      stash_stage = stage;
      out.push_back(std::move(gi));
      break;
    }
    out.push_back(std::move(gi));
  }
  ReadBuffer& reads = reads_ready();
  for (size_t i = 0; i < out.size(); ++i) {
    GeneInput& gi = out[i];
    if (i == stash_gene && stash_stage == 0) std::rethrow_exception(stashed);
    fetch_reads(gi, reads, opt);
    if (!lazy_reads) gi.materialize();
    if (i == stash_gene) std::rethrow_exception(stashed);
  }
  return out;
}

inline std::vector<GeneInput> ingest_genes(std::istream& gtf, ReadBuffer& reads, mphio::VcfFile& vcf, mphio::FastaIndexed& fasta,
                                           const IngestOptions& opt, bool lazy_reads = false) {
  return ingest_genes_with(gtf, [&]() -> ReadBuffer& { return reads; }, vcf, fasta, opt, lazy_reads);
}

// Loads the BAM on a thread of its own; get() joins it and hands the buffer over (or rethrows what the load threw).
class ReadBufferLoader {
 public:
  explicit ReadBufferLoader(mphio::BamFile& bam) {
    thread_ = std::thread([this, &bam] {
      try {
        buf_.reset(new ReadBuffer(bam));
      } catch (...) {
        err_ = std::current_exception();
      }
    });
  }
  ~ReadBufferLoader() {
    if (thread_.joinable()) thread_.join();
  }
  ReadBuffer& get() {
    if (thread_.joinable()) thread_.join();
    if (err_) std::rethrow_exception(err_);
    return *buf_;
  }

 private:
  std::thread thread_;
  std::unique_ptr<ReadBuffer> buf_;
  std::exception_ptr err_;
};

// Contiguous gene ranges balanced by read count, one per device (SURVEY.md §8(e)): shard k is
// genes [cut[k], cut[k+1]). Shards are independent; their records are concatenated in shard order.
inline std::vector<size_t> partition_genes(const std::vector<GeneInput>& genes, size_t n_shards) {
  std::vector<size_t> cut(n_shards + 1, genes.size());
  cut[0] = 0;
  uint64_t total = 0;
  for (auto& g : genes) total += g.n_reads + 1;
  uint64_t acc = 0;
  size_t k = 1;
  for (size_t i = 0; i < genes.size() && k < n_shards; ++i) {
    acc += genes[i].n_reads + 1;
    while (k < n_shards && acc * n_shards >= total * k) cut[k++] = i + 1;
  }
  return cut;
}

inline void pack_genes(std::vector<GeneInput>& genes, size_t lo, size_t hi, Packer& packer) {
  for (size_t i = lo; i < hi; ++i) {
    GeneInput& gi = genes[i];
    gi.materialize();
    packer.add_gene(gi.gene, gi.reads, gi.max_read_len, gi.sites, std::move(gi.refseq));
    std::vector<HostRead>().swap(gi.reads);
    std::vector<ReadBuffer::Pin>().swap(gi.pins);  // the packer copied what it ships
  }
}

// The protein-coding genes of a parsed GTF, fetched one by one through the BAM index in GTF order and handed to
// `on_gene(GeneInput&&)`; the walk stops when that returns false.
template <class OnGene>
inline void walk_indexed_genes(std::vector<ParsedGene> genes, mphio::BamFile& bam, const mphio::BamIndex& index, mphio::VcfFile& vcf,
                               mphio::FastaIndexed& fasta, const IngestOptions& opt, OnGene&& on_gene) {
  ReadBuffer reads(bam, index);
  VariantBuffer variants(vcf);
  for (ParsedGene& pg : genes) {
    if (pg.biotype != "protein_coding") continue;  // :1964
    if (!on_gene(fetch_gene(std::move(pg.gene), reads, variants, vcf, fasta, opt))) return;
  }
}

// Builds the batch for every protein-coding gene of the GTF, in GTF order. With an index next to the BAM the reads are
// fetched through it gene by gene; without one the whole file is loaded first.
inline void ingest(std::istream& gtf, mphio::BamFile& bam, mphio::VcfFile& vcf, mphio::FastaIndexed& fasta, const IngestOptions& opt,
                   Packer& packer) {
  const std::string bai = mphio::BamIndex::locate(bam.path());
  if (!bai.empty()) {
    const mphio::BamIndex index(bai, bam.ref_names.size(), bam.file_bytes());
    std::vector<GeneInput> one(1);
    walk_indexed_genes(read_gtf(gtf, opt.mode), bam, index, vcf, fasta, opt, [&](GeneInput&& gi) {
      one[0] = std::move(gi);
      pack_genes(one, 0, 1, packer);
      return true;
    });
    return;
  }
  ReadBufferLoader loader(bam);
  std::vector<GeneInput> genes = ingest_genes_with(gtf, [&]() -> ReadBuffer& { return loader.get(); }, vcf, fasta, opt, true);
  pack_genes(genes, 0, genes.size(), packer);
}

}  // namespace mph
