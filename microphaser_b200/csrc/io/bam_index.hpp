// bam_index.hpp — the BAM index (.bai, SAM specification §5.2) and the one query the indexed read buffer makes of it:
// where a read of [beg, contig end) has to start. htslib's hts_itr_query restated for that region only. CSI and CRAM
// indices are not read.
//
// The index is outside input: every count is checked against the bytes that are left, every offset against the size of
// the BAM it indexes. A malformed index is an IoError naming the index file, never a silent fall-back to a scan: a wrong
// offset would mean wrong reads.
#pragma once
#include <unistd.h>

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "hts_io.hpp"

namespace mphio {

class BamIndex {
 public:
  static constexpr uint64_t NONE = ~uint64_t(0);  // first_offset(): the region holds no record

  // the index htslib would open for `bam_path`: <bam>.bai, then <bam without .bam>.bai; "" if there is none
  static std::string locate(const std::string& bam_path) {
    std::string p = bam_path + ".bai";
    if (access(p.c_str(), R_OK) == 0) return p;
    if (bam_path.size() > 4 && bam_path.compare(bam_path.size() - 4, 4, ".bam") == 0) {
      p = bam_path.substr(0, bam_path.size() - 4) + ".bai";
      if (access(p.c_str(), R_OK) == 0) return p;
    }
    return std::string();
  }

  // n_ref: contigs in the BAM header; bam_bytes: compressed size of the BAM (every offset must point inside it)
  BamIndex(const std::string& path, size_t n_ref, uint64_t bam_bytes) : path_(path) {
    const std::vector<uint8_t> buf = read_file(path);
    size_t o = 0;
    auto bad = [&](const char* what) { return IoError("malformed BAM index " + path + ": " + what); };
    auto need = [&](uint64_t n, const char* what) { if (n > buf.size() - o) throw bad(what); };
    auto i32 = [&](const char* what) { need(4, what); int32_t v; memcpy(&v, buf.data() + o, 4); o += 4; return v; };
    auto u64 = [&]() { uint64_t v; memcpy(&v, buf.data() + o, 8); o += 8; return v; };
    need(4, "truncated magic");
    if (memcmp(buf.data(), "BAI\1", 4) != 0) throw bad("bad magic");
    o = 4;
    const int32_t nr = i32("truncated reference count");
    if (nr < 0 || size_t(nr) != n_ref)
      throw bad(("indexes " + std::to_string(nr) + " references, the BAM header has " + std::to_string(n_ref)).c_str());
    refs_.resize(size_t(nr));
    auto check_off = [&](uint64_t v, bool is_end) {
      // a start must point into a block; an end may point at the end of the file
      if ((v >> 16) > bam_bytes || (!is_end && (v >> 16) == bam_bytes)) throw bad("offset past the end of the BAM");
    };
    for (auto& ref : refs_) {
      const int32_t n_bin = i32("truncated bin count");
      if (n_bin < 0 || uint64_t(n_bin) * 8 > buf.size() - o) throw bad("bin count larger than the file");
      for (int32_t b = 0; b < n_bin; ++b) {
        need(4, "truncated bin");
        uint32_t bin;
        memcpy(&bin, buf.data() + o, 4);
        o += 4;
        const int32_t n_chunk = i32("truncated chunk count");
        if (n_chunk < 0 || uint64_t(n_chunk) * 16 > buf.size() - o) throw bad("chunk count larger than the file");
        if (bin == PSEUDO_BIN) {  // samtools' per-reference statistics: two pairs that are not chunks
          if (n_chunk != 2) throw bad("pseudo-bin without two entries");
          o += 32;
          continue;
        }
        if (bin > MAX_BIN) throw bad("bin number out of range");
        auto& chunks = ref.bins[bin];
        for (int32_t c = 0; c < n_chunk; ++c) {
          const uint64_t beg = u64(), end = u64();
          check_off(beg, false);
          check_off(end, true);
          if (end < beg) throw bad("chunk ends before it begins");
          chunks.emplace_back(beg, end);
        }
      }
      const int32_t n_intv = i32("truncated linear index size");
      if (n_intv < 0 || uint64_t(n_intv) * 8 > buf.size() - o) throw bad("linear index larger than the file");
      ref.lin.resize(size_t(n_intv));
      for (auto& v : ref.lin) {
        v = u64();
        check_off(v, false);
      }
    }
    // an optional count of unplaced reads follows; nothing after it is read
  }

  const std::string& path() const { return path_; }

  // Virtual offset from which a read of [beg, end of contig tid) starts (hts_itr_query): the linear-index floor of the
  // 16 kb window holding `beg`, then the smallest chunk start, clamped to that floor, among the bins overlapping the
  // region whose chunks end past the floor. Every record that overlaps the region lies at or after it. NONE when no
  // chunk qualifies: no record of the contig reaches `beg`.
  uint64_t first_offset(int tid, int64_t beg) const {
    if (tid < 0 || size_t(tid) >= refs_.size()) return NONE;
    const Ref& ref = refs_[size_t(tid)];
    beg = std::max<int64_t>(0, std::min<int64_t>(beg, MAX_POS - 1));
    uint64_t floor = 0;
    if (!ref.lin.empty()) floor = ref.lin[std::min(size_t(beg >> 14), ref.lin.size() - 1)];
    uint64_t best = NONE;
    // Every bin of a level from the one holding `beg` on overlaps the region, which runs to the end of the contig. A bin
    // holds the records that start and end inside its interval, so in a sorted BAM all records of a later bin of the same
    // level come after all records of an earlier one: per level, the first bin with a chunk past the floor has the minimum.
    const uint32_t first[] = {0, 1, 9, 73, 585, 4681, MAX_BIN + 1};
    const int shift[] = {29, 26, 23, 20, 17, 14};
    for (int l = 0; l < 6; ++l)
      for (auto it = ref.bins.lower_bound(first[l] + uint32_t(beg >> shift[l])); it != ref.bins.end() && it->first < first[l + 1]; ++it) {
        bool found = false;
        for (auto& c : it->second)
          if (c.second > floor) {
            best = std::min(best, std::max(c.first, floor));
            found = true;
          }
        if (found) break;
      }
    return best;
  }

 private:
  static constexpr uint32_t PSEUDO_BIN = 37450, MAX_BIN = 37449;
  static constexpr int64_t MAX_POS = int64_t(1) << 29;  // the largest position a BAI describes
  struct Ref {
    std::map<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>> bins;
    std::vector<uint64_t> lin;
  };
  std::string path_;
  std::vector<Ref> refs_;
};

}  // namespace mphio
