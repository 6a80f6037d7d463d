// TEST INFRASTRUCTURE ONLY — the indexed ReadBuffer against the whole-file one.
//   index_fetch fetch <bam> <whole-file io threads> <indexed io threads>   queries "chrom start end" on stdin
//     runs every query through both buffers, fails on the first difference, and prints the records of each query as
//     "pos end flag mapq qname_hash digest" (digest: FNV-1a of the decoded bases, '|', the CIGAR text) for the caller's
//     own restatement of the fetch rule
//   index_fetch load <bam> <bai>     loads the index only: "ok", or the IoError and exit status 1
#include <cstdio>
#include <iostream>
#include <sstream>

#include "../../microphaser_b200/csrc/host/ingest.hpp"

static uint64_t digest(const mph::ReadBuffer::Rec& r) {
  static const char* dec = "=ACMGRSVTWYHKDBN";
  std::string s;
  for (uint32_t i = 0; i < r.l_seq; ++i) s += dec[(i & 1) ? (r.seq_p[i >> 1] & 15) : (r.seq_p[i >> 1] >> 4)];
  s += '|';
  for (uint32_t i = 0; i < r.n_cigar; ++i) s += std::to_string(r.cig_p[i] >> 4) + "MIDNSHP=X"[r.cig_p[i] & 15];
  return mph::fnv1a(s);
}

int main(int argc, char** argv) {
  try {
    const std::string mode = argv[1];
    if (mode == "load") {
      mphio::BamFile bam(argv[2], 1);
      mphio::BamIndex idx(argv[3], bam.ref_names.size(), bam.file_bytes());
      for (size_t t = 0; t < bam.ref_names.size(); ++t) idx.first_offset(int(t), 0);
      printf("ok\n");
      return 0;
    }
    mphio::fast_inflate_enabled().store(true);
    mphio::BamFile whole_bam(argv[2], unsigned(atoi(argv[3])));
    mph::ReadBuffer whole(whole_bam);
    const std::string bai = mphio::BamIndex::locate(argv[2]);
    if (bai.empty()) { fprintf(stderr, "no index\n"); return 2; }
    mphio::BamFile idx_bam(argv[2], unsigned(atoi(argv[4])), mphio::BgzfInflaterSpec(), 8);
    mphio::BamIndex idx(bai, idx_bam.ref_names.size(), idx_bam.file_bytes());
    mph::ReadBuffer indexed(idx_bam, idx);
    std::string chrom;
    uint64_t start, end;
    size_t q = 0, n = 0;
    while (std::cin >> chrom >> start >> end) {
      const std::deque<const mph::ReadBuffer::Rec*> a = whole.fetch(chrom, start, end);
      const auto& b = indexed.fetch(chrom, start, end);
      const auto pins = indexed.pins();
      if (a.size() != b.size()) { printf("query %zu (%s %llu %llu): %zu vs %zu records\n", q, chrom.c_str(), (unsigned long long)start, (unsigned long long)end, a.size(), b.size()); return 1; }
      printf("q %zu %zu\n", q, a.size());
      for (size_t i = 0; i < a.size(); ++i, ++n) {
        const auto& x = *a[i];
        const auto& y = *b[i];
        bool ok = x.tid == y.tid && x.pos == y.pos && x.end == y.end && x.l_seq == y.l_seq && x.n_cigar == y.n_cigar && x.flag == y.flag && x.mapq == y.mapq && x.qname_hash == y.qname_hash;
        ok = ok && memcmp(x.seq_p, y.seq_p, (x.l_seq + 1) / 2) == 0 && memcmp(x.qual_p, y.qual_p, x.l_seq) == 0 && memcmp(x.cig_p, y.cig_p, 4 * x.n_cigar) == 0;
        if (!ok) { printf("query %zu record %zu differs\n", q, i); return 1; }
        printf("%d %u %u %u %llu %llu\n", x.pos, x.end, x.flag, x.mapq, (unsigned long long)x.qname_hash, (unsigned long long)digest(x));
      }
      ++q;
    }
    printf("done %zu queries, %zu records, 0 differences\n", q, n);
    return 0;
  } catch (const std::exception& e) {
    printf("error: %s\n", e.what());
    return 1;
  }
}
