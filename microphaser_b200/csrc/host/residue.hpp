// residue.hpp — the serial part of the reference's window loop that stays on the host.
//
// The device returns, per *interesting* window (one that contains variants, a stop codon, or sits
// at an exon boundary), the observation count, the haplotype histogram and the assembled
// sequences. What is left is inherently sequential per transcript and touches only those few
// windows: the frameshift_frequencies map threaded through print_haplotypes
// (reference src/microphasing.rs:370,496-500,604-631,703-718), the ORF termination tests
// (:1465-1488), record construction (:720-837), the emission predicate (:839-875) and the
// splice-junction merge (:1497-1908, src/common.rs:376-568).
#pragma once
#include <charconv>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <memory>
#include <optional>
#include <string>
#include <string_view>
#include <tuple>
#include <vector>

#include "../io/fmt_util.hpp"
#include "batch.hpp"
#include "../core/record_core.h"

namespace mph {

// what comes back from the device for one batch
struct PhaseRaw {
  std::vector<uint32_t> iw;       // interesting window indices, ascending
  std::vector<MphWinOut> iw_out;  // per interesting window
  std::vector<MphHap> iw_hap0;    // per interesting window: assembly of haplotype 0
  std::vector<MphHist> hist;      // extra histogram keys (whole arena)
  std::vector<MphHap> hapx;       // per extra key
  std::vector<uint8_t> seq;       // sequence arena: slots of 2 * seq_cap bytes (normal mode: seq_cap bytes)
  std::vector<uint32_t> iw_voff;  // per interesting window (empty without replayed transcripts): offset of its matrix columns in vlist, 0xFFFFFFFF = own variants
  std::vector<uint32_t> seg_err;  // per segment (empty without replayed transcripts): 1 + iteration at which the reference panics
  std::vector<uint32_t> vlist;    // column lists: count, then variant indices in print_haplotypes order
  std::vector<uint64_t> win_id;   // normal mode only, per enumerated window: leading 64 bits of the record id of the reference window (0 = not hashed)
  std::vector<uint32_t> win_depth;  // normal mode only, per enumerated window: depth | (plain window starts / ends with a stop codon) << 31
  // device-class transcripts (core/record_core.h): their records come from the record kernels, already in the reference's order
  std::vector<MphRec> recs;
  std::vector<uint8_t> rec_seq;      // sequence bytes the records point into
  std::vector<MphRecSrc> rec_aux;    // second source of the merged records
  uint64_t dev_windows = 0, dev_read_windows = 0;  // statistics over their live windows (emulator only; the library sums on the device)
  uint32_t seg_base = 0;          // seg_err[0] belongs to this segment
  uint32_t win_base = 0;          // win_depth[0] / win_id[0] belong to this window
  uint32_t err = 0;
  uint64_t sum_depth = 0;         // over every enumerated window
};

// A string with N characters of inline storage, heap beyond that.  The record id is 16 characters and a
// window sequence usually 27 — both just past what std::string keeps inline — and every record carries three.
template <size_t N>
class InlineStr {
 public:
  InlineStr() { buf_[0] = 0; }
  InlineStr(std::string_view v) { assign(v); }
  InlineStr(const std::string& v) { assign(std::string_view(v)); }
  InlineStr(const char* v) { assign(std::string_view(v)); }
  InlineStr(const InlineStr& o) { assign(o.view()); }
  InlineStr(InlineStr&& o) noexcept { take(o); }
  InlineStr& operator=(const InlineStr& o) {
    if (this != &o) assign(o.view());
    return *this;
  }
  InlineStr& operator=(InlineStr&& o) noexcept {
    if (this != &o) take(o);
    return *this;
  }
  InlineStr& operator=(std::string_view v) { assign(v); return *this; }
  InlineStr& operator=(const std::string& v) { assign(std::string_view(v)); return *this; }

  // `v` must not alias this string's own storage
  void assign(std::string_view v) {
    char* d = reset(v.size());
    if (!v.empty()) memcpy(d, v.data(), v.size());
  }
  void assign(const char* p, size_t n) { assign(std::string_view(p, n)); }
  // sets the length; the characters are zero until written through operator[]
  void resize(size_t n) { memset(reset(n), 0, n); }
  void clear() { reset(0); }

  size_t size() const { return n_; }
  bool empty() const { return n_ == 0; }
  const char* data() const { return n_ <= N ? buf_ : big_.get(); }
  const char* c_str() const { return data(); }
  char& operator[](size_t i) { return (n_ <= N ? buf_ : big_.get())[i]; }
  const char& operator[](size_t i) const { return data()[i]; }
  std::string_view view() const { return std::string_view(data(), n_); }
  operator std::string_view() const { return view(); }
  operator std::string() const { return std::string(data(), n_); }

  friend bool operator==(const InlineStr& a, const InlineStr& b) { return a.view() == b.view(); }
  friend bool operator!=(const InlineStr& a, const InlineStr& b) { return a.view() != b.view(); }

 private:
  // storage for n characters plus the terminator, contents unspecified
  char* reset(size_t n) {
    char* d = buf_;
    if (n > N) {
      if (!big_ || n > cap_) {
        big_.reset(new char[n + 1]);
        cap_ = n;
      }
      d = big_.get();
    }
    n_ = n;
    d[n] = 0;
    return d;
  }
  void take(InlineStr& o) noexcept {
    n_ = o.n_;
    cap_ = o.cap_;
    big_ = std::move(o.big_);
    memcpy(buf_, o.buf_, sizeof buf_);
    o.n_ = 0;
    o.cap_ = 0;
    o.buf_[0] = 0;
  }
  size_t n_ = 0, cap_ = 0;
  std::unique_ptr<char[]> big_;
  char buf_[N + 1];
};
using IdStr = InlineStr<23>;
using SeqStr = InlineStr<39>;

// src/common.rs:350-373
struct InfoRecord {
  IdStr id;
  uint32_t tx = 0;
  uint64_t offset = 0, frame = 0;
  double freq = 0;
  uint32_t depth = 0, nvar = 0, nsomatic = 0, nvariant_sites = 0, nsomvariant_sites = 0;
  std::string variant_sites, somatic_positions, somatic_aa_change, germline_positions, germline_aa_change;
  SeqStr normal_sequence, mutant_sequence;
};

struct OutRecord {
  InfoRecord info;       // the TSV row
  SeqStr mt;             // mutant FASTA sequence (stdout), valid if has_mt && !mt_same
  SeqStr wt;             // normal FASTA sequence (--normal-output), valid if has_wt && !wt_same
  bool has_mt = false, has_wt = false;
  // the FASTA line is byte-identical to the TSV column (the common case): it is not stored twice
  bool mt_same = false, wt_same = false;
  const SeqStr& mt_str() const { return mt_same ? info.mutant_sequence : mt; }
  const SeqStr& wt_str() const { return wt_same ? info.normal_sequence : wt; }
};

struct ResidueStats {
  uint64_t windows = 0;       // main-ORF print_haplotypes calls the reference would make
  uint64_t read_windows = 0;  // sum of depth over them
};

namespace detail {

// Walks the '|'-separated fields of a column the way `str::split('|')` does ("" yields one empty field).
struct BarFields {
  std::string_view s;
  size_t pos = 0;
  bool done = false;
  explicit BarFields(std::string_view v) : s(v) {}
  bool next(std::string_view& out) {
    if (done) return false;
    const size_t e = s.find('|', pos);
    if (e == std::string_view::npos) { out = s.substr(pos); done = true; }
    else { out = s.substr(pos, e - pos); pos = e + 1; }
    return true;
  }
};
inline uint64_t parse_u64(std::string_view p) {
  if (p.empty()) throw Fatal("ParseIntError");
  uint64_t v = 0;
  for (char c : p) {
    if (c < '0' || c > '9') throw Fatal("ParseIntError");
    v = v * 10 + uint64_t(c - '0');
  }
  return v;
}
inline void bar_append(std::string& dst, bool& first, std::string_view field) {
  if (!first) dst.push_back('|');
  first = false;
  dst.append(field);
}
// Keeps the (position, aa change) pairs of one record whose position passes `keep` (common.rs:399-478):
// the walk stops at the first empty position field; indexing the change column past its end panics.
template <class Keep>
inline uint32_t merge_fields(std::string_view positions, std::string_view changes, std::string& out_pos, bool& first_pos,
                             std::string& out_aa, bool& first_aa, Keep keep) {
  BarFields pf(positions), af(changes);
  std::string_view p, aa;
  bool have_aa = af.next(aa);
  uint32_t kept = 0;
  while (pf.next(p)) {
    if (p.empty()) break;
    if (keep(parse_u64(p))) {
      if (!have_aa) throw Fatal("index out of bounds");
      bar_append(out_pos, first_pos, p);
      bar_append(out_aa, first_aa, aa);
      ++kept;
    }
    have_aa = af.next(aa);
  }
  return kept;
}

// IDRecord::update (common.rs:376-526)
inline InfoRecord merge_records(const InfoRecord& self, const InfoRecord& rec, bool forward, const std::string& tx_id, uint64_t offset,
                                uint64_t frame, double freq, const std::string& wt_seq, const std::string& mt_seq, uint64_t wlen) {
  InfoRecord o;
  o.id = mphfmt::record_id(reinterpret_cast<const uint8_t*>(mt_seq.data()), mt_seq.size(), tx_id, offset, forward ? 'F' : 'R');
  bool f_sp = true, f_saa = true, f_gp = true, f_gaa = true;
  uint32_t nsom = 0;
  nsom += merge_fields(self.somatic_positions, self.somatic_aa_change, o.somatic_positions, f_sp, o.somatic_aa_change, f_saa,
                       [&](uint64_t pv) { return forward ? (self.offset + offset <= pv) : (self.offset + wlen - offset >= pv); });
  nsom += merge_fields(rec.somatic_positions, rec.somatic_aa_change, o.somatic_positions, f_sp, o.somatic_aa_change, f_saa,
                       [&](uint64_t pv) { return forward ? (rec.offset + offset >= pv) : (rec.offset + wlen - 3 - offset <= pv); });
  uint32_t nvariants = nsom;
  nvariants += merge_fields(self.germline_positions, self.germline_aa_change, o.germline_positions, f_gp, o.germline_aa_change, f_gaa,
                            [&](uint64_t pv) { return self.offset + offset <= pv; });
  nvariants += merge_fields(rec.germline_positions, rec.germline_aa_change, o.germline_positions, f_gp, o.germline_aa_change, f_gaa,
                            [&](uint64_t pv) { return rec.offset >= pv - offset; });
  o.tx = self.tx;
  o.offset = forward ? self.offset + offset : rec.offset + wlen + 3 - offset;
  o.frame = frame;
  o.freq = freq;
  o.depth = (rec.depth == 0 || self.depth == 0) ? 0 : (rec.depth + self.depth) / 2;
  o.nvar = nvariants;
  o.nsomatic = nsom;
  o.nvariant_sites = self.nvariant_sites + rec.nvariant_sites;
  o.nsomvariant_sites = self.nsomvariant_sites + rec.nsomvariant_sites;
  // "self|rec" with one leading and one trailing '|' removed (common.rs:497-503)
  std::string& vr = o.variant_sites;
  vr.reserve(self.variant_sites.size() + rec.variant_sites.size() + 1);
  vr = self.variant_sites;
  vr.push_back('|');
  vr += rec.variant_sites;
  if (!vr.empty() && vr.front() == '|') vr.erase(0, 1);
  if (!vr.empty() && vr.back() == '|') vr.pop_back();
  o.normal_sequence = wt_seq;
  o.mutant_sequence = mt_seq;
  return o;
}

// IDRecord::add_freq (common.rs:528-568)
inline InfoRecord add_freq(InfoRecord r, double f) {
  const uint32_t new_nvar = r.nvar == 0 ? r.nvar : (f > 0.0 ? r.nvar - 1 : r.nvar);
  r.nsomatic = new_nvar < r.nsomatic ? r.nsomatic - 1 : r.nsomatic;
  r.nvar = new_nvar;
  r.freq = r.freq > 0.5 ? r.freq : r.freq + f;
  return r;
}

}  // namespace detail

// the variant columns print_haplotypes sees for one window: the window's own variants [va, va + n), or the
// explicit list the serial replay recorded (stale columns, core/replay_core.h)
struct WinVars {
  const uint32_t* list = nullptr;
  uint32_t va = 0, n = 0;
  uint32_t at(uint32_t c) const { return list ? list[c] : va + c; }
};

class Residue {
 public:
  Residue(const Batch& b, const PhaseRaw& raw) : b_(b), raw_(raw) {
    const char* tr = getenv("MPH_TRACE");
    if (tr && *tr) trace_ = fopen(tr, "w");
  }
  ~Residue() {
    if (trace_) fclose(trace_);
  }

  // Processes transcripts [tx_lo, tx_hi) and appends their records in the reference's order.
  void run(uint32_t tx_lo, uint32_t tx_hi, std::vector<OutRecord>& out, ResidueStats& stats) {
    // records are a few hundred bytes each: size the vector once from the number of interesting windows of the range
    // instead of letting it double its way up (about one record per three such windows on variant-dense input)
    if (tx_lo < tx_hi && b_.txs[tx_lo].seg_lo < b_.txs[tx_hi - 1].seg_hi) {
      const MphSegment& s0 = b_.segs[b_.txs[tx_lo].seg_lo];
      const MphSegment& s1 = b_.segs[b_.txs[tx_hi - 1].seg_hi - 1];
      auto lo = std::lower_bound(raw_.iw.begin(), raw_.iw.end(), s0.win_base);
      auto hi = std::lower_bound(lo, raw_.iw.end(), s1.win_base + s1.n_win);
      out.reserve(out.size() + size_t(hi - lo) / 3 + 16);
    }
    for (uint32_t t = tx_lo; t < tx_hi; ++t) {
      const TxMeta& tm = b_.txs[t];
      if (tm.seg_hi > tm.seg_lo && (b_.segs[tm.seg_lo].flags & MPH_SF_DEVREC)) continue;  // built on the device
      run_transcript(t, out, stats);
    }
  }

 private:
  using FrameFreqs = std::map<uint64_t, std::pair<double, bool>>;
  struct HapSeq {  // HaplotypeSeq (:141-145): only the record is ever read
    InfoRecord rec;
    // A haplotype whose mutant and normal sequence are both the plain reference window cannot produce a
    // merged record on its own (:1887 writes only mt != wt); its strings are built only if the other side
    // of the junction carries a variant.
    bool lazy = false;
    const MphSegment* sg = nullptr;
    const MphHap* h = nullptr;
    uint32_t k = 0;
    WinVars wv;
  };

  struct Key {
    uint64_t hap, frame;
    uint64_t count;
    const MphHap* info;
  };

  // index of window `widx` in the interesting-window list; the serial loop asks in ascending order within one
  // segment, so the previous answer (or its successor) is almost always the next one
  size_t find_iw(uint32_t widx) {
    const uint32_t* iw = raw_.iw.data();
    for (size_t c = iw_hint_; c < iw_hi_ && c < iw_hint_ + 2; ++c)
      if (iw[c] == widx) return iw_hint_ = c;
    const uint32_t* it = std::lower_bound(iw + iw_lo_, iw + iw_hi_, widx);
    if (it == iw + iw_hi_ || *it != widx) return SIZE_MAX;
    return iw_hint_ = size_t(it - iw);
  }

  std::string arena(const MphHap& h, bool germ) const {
    if (!(h.flags & MPH_HF_SEQ)) throw std::logic_error("internal: sequence not shipped for a haplotype that needs it");
    if (h.flags & MPH_HF_OVERFLOW) throw Unsupported("assembled haplotype longer than the sequence slot");
    const uint8_t* p = raw_.seq.data() + h.seq_off + (germ ? b_.seq_cap : 0);
    return std::string(reinterpret_cast<const char*>(p), germ ? h.germ_len : h.seq_len);
  }

  // print_haplotypes (:353-879) with the matrix scan and the sequence walk replaced by device results
  // what print_haplotypes hands back (:878): the haplotype list is materialised only for windows a
  // splice merge can read (exon boundaries); elsewhere only its length matters (:1437)
  struct HapList {
    std::vector<HapSeq> v;
    size_t n = 0;
    bool partial = false;
    bool empty() const { return n == 0; }
  };

  HapList print(uint32_t t, const MphSegment& sg, uint32_t k, size_t iwi, uint64_t frame_in, FrameFreqs& ff,
                            bool is_first_exon_window, std::vector<OutRecord>& out) {
    const TxMeta& tm = b_.txs[t];
    const GeneMeta& gm = b_.genes[tm.gene];
    const bool rev = tm.reverse;
    const MphGeom g = mph_geom(sg, k);
    WinVars wv;
    wv.va = mph_var_lb(b_.vars.data(), sg.var_lo, sg.var_hi, g.s);
    wv.n = mph_var_lb(b_.vars.data(), sg.var_lo, sg.var_hi, g.e) - wv.va;
    if (!raw_.iw_voff.empty() && raw_.iw_voff[iwi] != 0xFFFFFFFFu) {
      const uint32_t off = raw_.iw_voff[iwi];
      wv.n = raw_.vlist[off];
      wv.list = raw_.vlist.data() + off + 1;
    }
    const uint32_t nv = wv.n;
    const MphWinOut& wo = raw_.iw_out[iwi];
    const MphHap& h0 = raw_.iw_hap0[iwi];
    const uint64_t window_len = sg.ewl;
    const bool is_short_exon = (sg.flags & MPH_SF_SHORT) != 0;
    uint64_t frame = frame_in;
    // histogram for this frame (:383-411) from the fine keys (hap, obs.frame.0, obs.frame.1 != 0)
    // device keys arrive sorted by (hap, obs.frame.0, obs.frame.1 != 0); projecting them onto this frame's
    // (hap, frame) key keeps the order, equal keys become adjacent -> a small sorted vector, no tree
    std::vector<Key>& keybuf = key_scratch_;  // reused across windows; a window may have any number of keys
    keybuf.clear();
    size_t n_keys = 0;
    uint64_t frame_depth = 0;
    auto add = [&](uint64_t hap, uint32_t fr, uint64_t count, const MphHap* info) {
      const uint64_t f0 = fr & 0x7FFFFFFFu;
      const bool f1nz = (fr >> 31) != 0;
      if (frame > 0 && f0 != frame && f1nz) return;
      frame_depth += count;
      const uint64_t kf = frame > 0 ? frame : f0;
      for (size_t q = n_keys; q-- > 0;) {
        if (keybuf[q].hap == hap && keybuf[q].frame == kf) { keybuf[q].count += count; return; }
        if (keybuf[q].hap != hap) break;
      }
      keybuf.push_back(Key{hap, kf, count, info});
      ++n_keys;
    };
    if (wo.c0 > 0) add(0, 0, wo.c0, &h0);
    for (uint32_t x = 0; x < wo.n_extra; ++x) {
      const MphHist& e = raw_.hist[wo.extra_off + x];
      const MphHap* info = e.hap == 0 ? &h0 : &raw_.hapx[wo.extra_off + x];
      add(e.hap, e.frame, e.count, info);
    }
    // within one hap the projected frames may be out of order only when frame > 0 collapses them (then they are equal)
    for (size_t q = 1; q < n_keys; ++q) {
      Key kq = keybuf[q];
      size_t z = q;
      while (z > 0 && (keybuf[z - 1].hap > kq.hap || (keybuf[z - 1].hap == kq.hap && keybuf[z - 1].frame > kq.frame))) { keybuf[z] = keybuf[z - 1]; --z; }
      keybuf[z] = kq;
    }
    const bool has_frameshift = frame > 0;
    if (n_keys == 0) { keybuf.push_back(Key{0, 0, 0, &h0}); ++n_keys; }
    if (trace_) {  // same line format as the oracle's MPH_ORACLE_TRACE
      fprintf(trace_, "W\t%s\t%llu\t%llu\t%llu\t%u\t%llu\t%u", tm.id.c_str(), (unsigned long long)g.s, (unsigned long long)g.e,
              (unsigned long long)frame_in, wo.depth, (unsigned long long)frame_depth, nv);
      for (size_t q = 0; q < n_keys; ++q)
        fprintf(trace_, "\t%llu:%llu:%llu", (unsigned long long)keybuf[q].hap, (unsigned long long)keybuf[q].frame, (unsigned long long)keybuf[q].count);
      fputc('\n', trace_);
    }
    HapList haplotypes_vec;
    uint64_t shift_in_window = 0;
    const bool boundary = is_boundary(sg, k);
    for (size_t q = 0; q < n_keys; ++q) {
      const Key& key = keybuf[q];
      const MphHap& h = *key.info;
      if (h.flags & MPH_HF_REFRANGE) throw Fatal("index out of bounds: refseq");  // the reference panics when it reaches this walk
      const uint64_t haplotype_frame = key.frame;
      const bool indel = (h.flags & MPH_HF_INDEL) != 0, insertion = (h.flags & MPH_HF_INSERTION) != 0;
      bool shift_is_set = false;
      const double freq = key.count == 0 ? 0.0 : double(key.count) / double(frame_depth);
      const uint32_t depth = wo.depth;
      // replay of the frameshift side effects of the sequence walk (:482-502): the visited
      // variants are variants[0 .. n_prof) in order, profile != 0 <=> the haplotype carries it
      for (uint32_t c = 0; c < uint32_t(h.n_prof) + h.brk && c < 32; ++c) {
        const MphVar& v = b_.vars[wv.at(c)];
        const uint64_t vfs = (v.flags & MPH_VF_FS_MASK) >> MPH_VF_FS_SHIFT;
        shift_in_window = shift_in_window > 0 ? shift_in_window : vfs;
        if (c == h.n_prof || ((h.profile >> (2 * c)) & 3)) {  // c == n_prof: the variant the walk broke on
          if (shift_in_window > 0) {
            shift_is_set = true;
            ff[vfs] = {freq, !(v.flags & MPH_VF_GERMLINE)};
            ff[0] = {1.0 - freq, false};
          }
        }
      }
      double frame_frequency = freq;
      if (shift_is_set && frame == 0) frame = shift_in_window;
      ff.try_emplace(frame, 0.0, false);
      if (shift_in_window == 0) frame_frequency = freq * ff.at(frame).first;
      if (shift_in_window == 0 && haplotype_frame > 0 && frame == 0) frame_frequency = 0.0;
      const bool germ_eq = (h.flags & MPH_HF_GERM_EQ) != 0;
      bool germ_cleared = false;
      if ((indel && insertion) || (shift_in_window == 0 && (ff.at(frame).second || (has_frameshift && !germ_eq)))) germ_cleared = true;
      const uint64_t seq_len = h.seq_len;
      const uint64_t germ_len = germ_cleared ? 0 : h.germ_len;
      const uint64_t this_window_len = seq_len < window_len ? seq_len : window_len;
      const uint64_t normal_window_len = indel ? (germ_len < window_len ? germ_len : window_len) : this_window_len;
      const bool stop_gain = (h.flags & MPH_HF_STOP) != 0;
      const bool seqs_equal = germ_cleared ? seq_len == 0 : germ_eq;  // germline_seq == seq after clearing
      // does anything below need the actual bytes?
      const bool emit = (h.n_som > 0 || has_frameshift) && !is_short_exon && !seqs_equal && frame_frequency > 0.0 && (!stop_gain || has_frameshift);
      // bytes are needed for emitted records and for the windows a splice merge can read (:1497-1908);
      // an indel haplotype also needs them for the stop-codon side condition (:707)
      // a boundary haplotype that is the plain reference on both streams is kept lazily (see HapSeq)
      const bool lazy = boundary && !emit && (nv == 0 || key.hap == 0) && seqs_equal && !germ_cleared;
      const bool need_rec = (emit || boundary) && !lazy;
      const bool want_seq = need_rec || (stop_gain && indel);
      // views into the reference arena / the downloaded sequence arena: nothing is copied until a record is built
      std::string_view seq, germline_seq;
      if (want_seq) {
        if (nv == 0 || key.hap == 0) {
          // no variant applied: seq == germline_seq == refseq[s..e) (:464-471,594-599), the host has those bytes
          if (g.s < sg.ref_pos0 || uint64_t(g.e) - sg.ref_pos0 > sg.ref_len) throw Fatal("slice index out of range: refseq");
          seq = std::string_view(reinterpret_cast<const char*>(b_.ref.data()) + sg.ref_off + (g.s - sg.ref_pos0), g.e - g.s);
          if (!germ_cleared) germline_seq = seq;
        } else {
          if (!(h.flags & MPH_HF_SEQ)) throw std::logic_error("internal: sequence not shipped for an emitted / boundary haplotype");
          if (h.flags & MPH_HF_OVERFLOW) throw Unsupported("assembled haplotype longer than the sequence slot");
          const char* base = reinterpret_cast<const char*>(raw_.seq.data()) + h.seq_off;
          seq = std::string_view(base, h.seq_len);
          if (!germ_cleared) germline_seq = std::string_view(base + b_.seq_cap, h.germ_len);
        }
      }
      const bool have_seq = want_seq;
      auto slice = [](std::string_view s, uint64_t a, uint64_t e) -> std::string_view {
        if (a > e || e > s.size()) throw Fatal("slice index out of range");
        return s.substr(size_t(a), size_t(e - a));
      };
      std::string_view normal_peptide, neopeptide;
      bool peptides_differ;  // normal_peptide != neopeptide (:707)
      if (have_seq) {
        if (germline_seq.empty()) normal_peptide = std::string_view();
        else if (g.spos == 1) normal_peptide = slice(germline_seq, g.gap, germline_seq.size());
        else if (g.spos == 0) normal_peptide = slice(germline_seq, 0, normal_window_len);
        else normal_peptide = germline_seq;
        if (g.spos == 1) neopeptide = slice(seq, g.gap, seq.size());
        else if (g.spos == 0) neopeptide = insertion ? seq : slice(seq, 0, this_window_len);
        else neopeptide = seq;
        peptides_differ = normal_peptide != neopeptide;
      } else {
        // the sequence walk compared the two slices itself (valid while germline_seq is cleared for indel + insertion only)
        const bool k3_valid = key.hap != 0 && germ_cleared == (indel && insertion);
        if (indel && !k3_valid) throw std::logic_error("internal: indel haplotype without shipped sequence");
        peptides_differ = k3_valid ? (h.flags & MPH_HF_PEPDIFF) != 0 : !seqs_equal;
      }
      bool remove_peptide = false;
      if (stop_gain && g.spos != 2 && (window_len == this_window_len || indel) && !is_first_exon_window &&
          (peptides_differ || !indel || std::fabs(freq - 1.0) < std::numeric_limits<double>::epsilon())) {
        (void)have_seq;
        remove_peptide = true;
        if (frame == 0) ff[frame] = {0.0, false};
        else ff.erase(frame);
      }
      // meta information (:720-769)
      // built only for a haplotype that is written or that a junction merge can read (two windows in three need neither)
      const bool have_rec = need_rec || lazy;
      std::optional<InfoRecord> rec_slot;
      if (have_rec) rec_slot.emplace();
      InfoRecord& rec = have_rec ? *rec_slot : unused_rec_;
      if (have_rec) {
        rec.tx = t;
        rec.offset = g.spos == 0 ? uint64_t(g.s) + 1 : uint64_t(g.s) + 1 + g.gap;
        rec.frame = frame;
        rec.freq = frame_frequency;
        rec.depth = depth;
      }
      if (need_rec) {
        fill_meta(rec, wv, h);
        // the id of a record that is not written is never read (IDRecord::update derives a new one)
        if (emit) {
          if ((h.flags & MPH_HF_ID) && key.hap != 0) {  // hashed on the device next to the sequence walk
            static const char* hx = "0123456789abcdef";
            rec.id.resize(16);
            for (int q = 0; q < 15; ++q) rec.id[q] = hx[(h.id64 >> (60 - 4 * q)) & 15];
            rec.id[15] = rev ? 'R' : 'F';
          } else {
            rec.id = mphfmt::record_id(reinterpret_cast<const uint8_t*>(seq.data()), seq.size(), tm.id, g.s, rev ? 'R' : 'F');
          }
        }
        rec.normal_sequence.assign(normal_peptide);
        rec.mutant_sequence.assign(neopeptide);
      }
      if (!remove_peptide || frame == 0) {
        haplotypes_vec.n += 1;
        if (boundary) {
          HapSeq& hs = haplotypes_vec.v.emplace_back();
          if (emit) hs.rec = rec;  // the written record keeps its own copy
          else hs.rec = std::move(rec);
          if (lazy) {
            hs.lazy = true; hs.sg = &sg; hs.h = &h; hs.k = k; hs.wv = wv;
          } else {
            hs.rec.normal_sequence.assign(germline_seq);
            hs.rec.mutant_sequence.assign(seq);
          }
        } else {
          haplotypes_vec.partial = true;
        }
      }
      if (emit) {
        // the FASTA lines (:846-873) are the TSV columns again unless an insertion / indel changed the slice bounds
        std::string_view mt_line, wt_line;
        bool has_mt = false, has_wt = false;
        if (g.spos == 1) { mt_line = slice(seq, g.gap, seq.size()); has_mt = true; }
        else if (g.spos == 0) { mt_line = slice(seq, 0, this_window_len); has_mt = true; }
        if (!germline_seq.empty()) {
          if (g.spos == 1) { wt_line = slice(germline_seq, g.gap, germline_seq.size()); has_wt = true; }
          else if (g.spos == 0) { wt_line = slice(germline_seq, 0, this_window_len); has_wt = true; }
        }
        auto put = [](std::string_view line, std::string_view column, SeqStr& dst, bool& same) {
          same = line.data() == column.data() && line.size() == column.size();
          if (!same) dst.assign(line);
        };
        OutRecord& o = out.emplace_back();  // built in place: nothing below throws
        if (has_mt) { put(mt_line, neopeptide, o.mt, o.mt_same); o.has_mt = true; }
        if (has_wt) { put(wt_line, normal_peptide, o.wt, o.wt_same); o.has_wt = true; }
        o.info = std::move(rec);
      }
    }
    (void)gm;
    return haplotypes_vec;
  }

  // variant-site metadata of one haplotype (:720-769)
  void fill_meta(InfoRecord& rec, const WinVars& wv, const MphHap& h) const {
    const uint32_t nv = wv.n;
    uint32_t n_variantsites = 0, n_som_variantsites = 0;
    // the columns are written in place
    std::string &s_pc = rec.somatic_aa_change, &g_pc = rec.germline_aa_change, &s_pos = rec.somatic_positions, &g_pos = rec.germline_positions,
                &sites = rec.variant_sites;
    s_pc.clear(); g_pc.clear(); s_pos.clear(); g_pos.clear(); sites.clear();
    bool fs = true, fg = true, fsite = true;
    char buf[24];
    auto put = [&](std::string& dst, bool& first, uint64_t v) {
      if (!first) dst.push_back('|');
      first = false;
      auto r = std::to_chars(buf, buf + sizeof buf, v);
      dst.append(buf, r.ptr);
    };
    bool fspc = true, fgpc = true;
    for (uint32_t c = 0; c < nv; ++c) {
      const MphVar& v = b_.vars[wv.at(c)];
      if (c < h.n_prof && c < 32) {
        const unsigned code = unsigned((h.profile >> (2 * c)) & 3);
        if (code == 2) {
          put(s_pos, fs, uint64_t(v.pos) + 1);
          if (!fspc) s_pc.push_back('|');
          fspc = false;
          s_pc += b_.var_prot[wv.at(c)];
        } else if (code == 1) {
          put(g_pos, fg, uint64_t(v.pos) + 1);
          if (!fgpc) g_pc.push_back('|');
          fgpc = false;
          g_pc += b_.var_prot[wv.at(c)];
        }
      }
      if (c == 0 || v.pos != b_.vars[wv.at(c - 1)].pos) {
        ++n_variantsites;
        put(sites, fsite, uint64_t(v.pos) + 1);
        if (!(v.flags & MPH_VF_GERMLINE)) ++n_som_variantsites;
      }
    }
    rec.nvar = h.n_var;
    rec.nsomatic = h.n_som;
    rec.nvariant_sites = n_variantsites;
    rec.nsomvariant_sites = n_som_variantsites;
  }

  // builds the strings of a lazily kept boundary haplotype (plain reference window on both streams)
  void materialize(HapSeq& hs) const {
    if (!hs.lazy) return;
    const MphSegment& sg = *hs.sg;
    const MphGeom g = mph_geom(sg, hs.k);
    if (g.s < sg.ref_pos0 || uint64_t(g.e) - sg.ref_pos0 > sg.ref_len) throw Fatal("slice index out of range: refseq");
    fill_meta(hs.rec, hs.wv, *hs.h);
    hs.rec.mutant_sequence.assign(reinterpret_cast<const char*>(b_.ref.data()) + sg.ref_off + (g.s - sg.ref_pos0), g.e - g.s);
    hs.rec.normal_sequence = hs.rec.mutant_sequence;
    hs.lazy = false;
  }

  static bool is_boundary(const MphSegment& sg, uint32_t k) {
    if (sg.n_win == 0) return false;
    if (sg.flags & MPH_SF_HAS_FS) return true;
    if (k < sg.k_first || (k - sg.k_first) % sg.k_stride) return false;
    return mph_is_boundary(sg, (k - sg.k_first) / sg.k_stride);
  }

  void run_transcript(uint32_t t, std::vector<OutRecord>& out, ResidueStats& stats) {
    const TxMeta& tm = b_.txs[t];
    const GeneMeta& gm = b_.genes[tm.gene];
    const bool fwd = !tm.reverse;
    const uint64_t window_len = b_.window_len;
    std::map<uint64_t, uint64_t> frameshifts;
    if (fwd) frameshifts[0] = 0;
    else frameshifts[gm.end] = 0;
    std::vector<HapSeq> prev_hap_vec, hap_vec;
    bool prev_partial = false, hap_partial = false;  // the list came from a window whose haplotypes were not materialised
    FrameFreqs ff;
    ff[0] = {1.0, false};
    uint64_t exon_rest = 0;
    for (uint32_t si = tm.seg_lo; si < tm.seg_hi; ++si) {
      if (frameshifts.empty()) break;
      const MphSegment& sg = b_.segs[si];
      const bool is_short_exon = (sg.flags & MPH_SF_SHORT) != 0;
      const bool is_first_exon = (sg.flags & MPH_SF_FIRST_EXON) != 0;
      const bool is_last_exon = (sg.flags & MPH_SF_LAST_EXON) != 0;
      const bool has_fs = (sg.flags & MPH_SF_HAS_FS) != 0;
      const uint64_t current_exon_offset = sg.ceo;
      const uint64_t exon_window_len = sg.ewl;
      exon_rest = 0;
      // Iterations the serial loop has to visit: every iteration when frameshifting variants can
      // open further reading frames, otherwise only the interesting main-ORF windows (all other
      // iterations leave the state untouched).
      std::vector<uint32_t>& ks = ks_scratch_;
      ks.clear();
      {
        // this segment's slice of the (ascending) list: it usually starts where the previous segment's slice ended,
        // and it cannot hold more entries than the segment has windows
        const uint32_t* iw = raw_.iw.data();
        const size_t n_iw = raw_.iw.size();
        size_t lo = std::min(iw_hi_, n_iw);
        if ((lo > 0 && iw[lo - 1] >= sg.win_base) || (lo < n_iw && iw[lo] < sg.win_base))
          lo = size_t(std::lower_bound(iw, iw + n_iw, sg.win_base) - iw);
        const size_t hi = size_t(std::lower_bound(iw + lo, iw + std::min(n_iw, lo + size_t(sg.n_win)), sg.win_base + sg.n_win) - iw);
        iw_lo_ = iw_hint_ = lo;
        iw_hi_ = hi;
      }
      if (has_fs) {
        for (uint32_t k = 0; k < sg.n_iter; ++k) ks.push_back(k);
      } else {
        for (size_t c = iw_lo_; c < iw_hi_; ++c) ks.push_back(sg.k_first + (raw_.iw[c] - sg.win_base) * sg.k_stride);
      }
      uint32_t prev_vb_fs = 0, prev_va_fs = 0;
      bool fs_init = false;
      uint64_t live_windows_end = sg.n_win;  // windows of this segment the reference reaches
      bool stopped = false;
      // the replay found an iteration at which the reference panics (shrink_left past the matrix columns :220-222,
      // inverted BTreeMap range): the loop gets there unless the ORF has ended before
      const uint32_t panic_k = raw_.seg_err.empty() ? 0xFFFFFFFFu : raw_.seg_err[si - raw_.seg_base] - 1u;
      for (uint32_t k : ks) {
        if (frameshifts.empty()) { stopped = true; break; }
        if (k >= panic_k) throw Fatal("drain: range end out of bounds");
        const MphGeom g = mph_geom(sg, k);
        const uint64_t offset = fwd ? uint64_t(sg.off0) + k : uint64_t(sg.off0) - k;
        const bool is_first_exon_window = k == 0;
        const uint64_t rest = fwd ? sg.exon_end - (offset + exon_window_len) : offset - sg.exon_start;
        const bool is_last_exon_window = rest < 3;
        if (has_fs) {
          // newly collected variants (:1280-1342): frameshift map bookkeeping
          const uint32_t va = mph_var_lb(b_.vars.data(), sg.var_lo, sg.var_hi, g.s);
          const uint32_t vb = mph_var_lb(b_.vars.data(), sg.var_lo, sg.var_hi, g.e);
          uint32_t na, nb;  // index range of the new variants, in collection order
          if (!fs_init || k == 0) { na = va; nb = vb; }
          else if (fwd) { na = std::max(prev_vb_fs, va); nb = vb; }
          else { na = va; nb = std::min(prev_va_fs, vb); }
          fs_init = true;
          prev_va_fs = va; prev_vb_fs = vb;
          auto handle = [&](const MphVar& v) {
            const uint64_t s = (v.flags & MPH_VF_FS_MASK) >> MPH_VF_FS_SHIFT;
            if ((s % 3) > 0) {
              std::vector<uint64_t> previous;
              for (auto& kv : frameshifts) previous.push_back(kv.second + s);
              const uint64_t end_pos = v.kind == MPH_DEL ? uint64_t(v.pos) + v.len - 1 : v.pos;
              for (uint64_t s_ : previous) frameshifts[fwd ? end_pos : uint64_t(v.pos)] = s_ % 3;
            }
          };
          if (fwd) for (uint32_t j = na; j < nb; ++j) handle(b_.vars[j]);
          else for (uint32_t j = nb; j > na; --j) handle(b_.vars[j - 1]);
        }
        uint64_t stopped_frameshift = 3;
        std::vector<std::pair<uint64_t, uint64_t>>& active = active_scratch_;  // snapshot: the map is not mutated while iterating (:1347-1350)
        active.clear();
        if (fwd) { for (auto it = frameshifts.begin(); it != frameshifts.end() && it->first < offset; ++it) active.push_back(*it); }
        else { for (auto it = frameshifts.lower_bound(offset + exon_window_len); it != frameshifts.end(); ++it) active.push_back(*it); }
        uint64_t frameshift_count = 0;
        bool main_orf = false;
        for (auto& kf : active) {
          const uint64_t key = kf.first, frameshift = kf.second;
          ++frameshift_count;
          if (frameshift == 0) main_orf = true;
          const uint64_t coding_shift = fwd ? offset - sg.exon_start : sg.exon_end - offset;
          const bool has_frameshift = frameshift > 0;
          if (coding_shift % 3 == (frameshift + current_exon_offset) % 3 || is_short_exon) {
            if (!has_frameshift) {
              exon_rest = rest;
              if (exon_window_len < 3) exon_rest = exon_window_len;
            }
            if (k < sg.k_first || (k - sg.k_first) % sg.k_stride != 0) throw std::logic_error("internal: window was not enumerated");
            const uint32_t widx = sg.win_base + (k - sg.k_first) / sg.k_stride;
            const size_t iwi = find_iw(widx);
            if (iwi == SIZE_MAX) throw std::logic_error("internal: window summary missing");
            if (has_fs && frameshift == 0) {
              stats.windows += 1;
              stats.read_windows += raw_.iw_out[iwi].depth;
            }
            auto res = print(t, sg, k, iwi, frameshift, ff, is_first_exon_window, out);
            if (res.empty() || !ff.count(frameshift)) stopped_frameshift = key;
            if (exon_rest < 3 && (!is_short_exon || is_first_exon) && !has_frameshift) { prev_hap_vec = std::move(res.v); prev_partial = res.partial; }
            else { hap_vec = std::move(res.v); hap_partial = res.partial; }
            if (frameshift != 0 && ff.count(frameshift) && ff.at(frameshift).first == 0.0) stopped_frameshift = key;
          }
        }
        if (frameshift_count == 0 || !main_orf || !ff.count(0)) {
          frameshifts.clear();
          live_windows_end = live_index(sg, k);
          stopped = true;
          break;
        }
        if (stopped_frameshift != 3) {
          auto it = frameshifts.find(stopped_frameshift);
          if (it == frameshifts.end()) throw Fatal("called `Option::unwrap()` on a `None` value");
          if (it->second != 0) frameshifts.erase(it);
        }
        if (frameshifts.empty()) { live_windows_end = live_index(sg, k); stopped = true; break; }
        if (ff.at(0).first == 0.0 && frameshifts.size() == 1) {
          frameshifts.clear();
          live_windows_end = live_index(sg, k);
          stopped = true;
          break;
        }
        const bool at_splice_side = fwd ? offset - current_exon_offset == sg.exon_start
                                        : offset + exon_window_len + current_exon_offset == sg.exon_end;
        // a junction without a variant in either window merges reference-only lists and writes nothing (:1801-1810,1887):
        // the packer marks the others (MPH_SF_JOIN_HEAD) and only their lists are kept
        const bool junction = at_splice_side && !is_first_exon && (sg.flags & MPH_SF_JOIN_HEAD);
        if (junction) {
          if (prev_partial || hap_partial) throw Unsupported("transcript " + tm.id + ": splice merge needs a window that is not at an exon boundary");
          prev_partial = hap_partial = false;
        }
        if (junction)
          splice_merge(t, sg, offset, is_short_exon, is_last_exon, is_last_exon_window, exon_rest, frameshifts, ff, hap_vec, prev_hap_vec, out);
        (void)window_len;
      }
      if (!stopped && !frameshifts.empty() && panic_k != 0xFFFFFFFFu) throw Fatal("drain: range end out of bounds");
      // statistics: main-ORF windows the reference evaluates in this segment (depth is summed on the
      // device over exactly these windows)
      if (!has_fs) {
        stats.windows += live_windows_end;
        seg_live_.push_back({si, uint32_t(live_windows_end)});
      }
      if (stopped) break;
    }
  }

  // number of enumerated windows of `sg` up to and including iteration k
  static uint64_t live_index(const MphSegment& sg, uint32_t k) {
    if (k < sg.k_first) return 0;
    return uint64_t((k - sg.k_first) / sg.k_stride) + 1;
  }

  // :1505-1908
  void splice_merge(uint32_t t, const MphSegment& sg, uint64_t offset, bool is_short_exon, bool is_last_exon, bool is_last_exon_window,
                    uint64_t exon_rest, const std::map<uint64_t, uint64_t>& frameshifts, FrameFreqs& ff, std::vector<HapSeq>& hap_vec,
                    std::vector<HapSeq>& prev_hap_vec, std::vector<OutRecord>& out) {
    const TxMeta& tm = b_.txs[t];
    const bool fwd = !tm.reverse;
    const uint64_t window_len = b_.window_len;
    const uint64_t exon_window_len = sg.ewl;
    {
      bool all_lazy = true;
      for (auto& x : hap_vec) all_lazy = all_lazy && x.lazy;
      for (auto& x : prev_hap_vec) all_lazy = all_lazy && x.lazy;
      if (all_lazy && !(sg.flags & MPH_SF_HAS_FS) && !(is_short_exon && !is_last_exon)) {
        // every combination has mt == wt: the window slide below writes nothing (:1801-1810,1887)
        if (is_short_exon) prev_hap_vec.clear();
        return;
      }
      for (auto& x : hap_vec) materialize(x);
      for (auto& x : prev_hap_vec) materialize(x);
    }
    const std::vector<HapSeq>& first_hap_vec = fwd ? hap_vec : prev_hap_vec;
    const std::vector<HapSeq>& sec_hap_vec = fwd ? prev_hap_vec : hap_vec;
    struct OutVal { std::string mt; InfoRecord rec; std::string wt; };
    std::map<std::tuple<uint64_t, std::string, std::string>, OutVal> output_map;
    std::vector<HapSeq> new_hap_vec;
    const double eps = std::numeric_limits<double>::epsilon();
    for (const HapSeq& hapseq : first_hap_vec) {
      const InfoRecord& record = hapseq.rec;
      const std::string_view wt_sequence = record.normal_sequence, mt_sequence = record.mutant_sequence;
      for (const HapSeq& prev_hapseq : sec_hap_vec) {
        const InfoRecord& prev_record = prev_hapseq.rec;
        const std::string_view prev_wt_sequence = prev_record.normal_sequence, prev_mt_sequence = prev_record.mutant_sequence;
        auto cat = [](std::string_view a, std::string_view b) {
          std::string r;
          r.reserve(a.size() + b.size());
          r.append(a);
          r.append(b);
          return r;
        };
        const std::string new_wt_sequence = cat(prev_wt_sequence, wt_sequence);
        std::vector<std::string> new_mt_sequences;
        if (wt_sequence != mt_sequence) {
          new_mt_sequences.push_back(cat(prev_wt_sequence, mt_sequence));
          if (prev_wt_sequence != prev_mt_sequence) {
            new_mt_sequences.push_back(cat(prev_mt_sequence, wt_sequence));
            new_mt_sequences.push_back(cat(prev_mt_sequence, mt_sequence));
          }
        } else {
          new_mt_sequences.push_back(cat(prev_mt_sequence, mt_sequence));
        }
        if (is_short_exon && !is_last_exon) {
          const double out_freq = std::fabs(record.freq - prev_record.freq) < eps ? record.freq : record.freq * prev_record.freq;
          HapSeq nh;
          nh.rec = detail::merge_records(prev_record, record, fwd, tm.id, 0, record.frame, out_freq, new_wt_sequence, new_wt_sequence, window_len);
          new_hap_vec.push_back(std::move(nh));
        }
        for (const std::string& new_mt_sequence : new_mt_sequences) {
          if (is_short_exon && !is_last_exon) {
            const double out_freq = std::fabs(record.freq - prev_record.freq) < eps ? record.freq : record.freq * prev_record.freq;
            HapSeq nh;
            nh.rec = detail::merge_records(prev_record, record, fwd, tm.id, 0, record.frame, out_freq, new_wt_sequence, new_mt_sequence, window_len);
            new_hap_vec.push_back(std::move(nh));
            continue;
          }
          std::vector<std::pair<uint64_t, uint64_t>> active;
          if (fwd) { for (auto it = frameshifts.begin(); it != frameshifts.end() && it->first < offset; ++it) active.push_back(*it); }
          else { for (auto it = frameshifts.lower_bound(offset + exon_window_len); it != frameshifts.end(); ++it) active.push_back(*it); }
          for (auto& pf : active) {
            const uint64_t pos = pf.first, frameshift = pf.second;
            ff.try_emplace(frameshift, 0.0, false);
            const bool shift_in_window = fwd ? pos >= prev_record.offset : pos < record.offset + exon_window_len;
            const bool somatic_shift = ff.at(frameshift).second;
            const double frameshift_freq = ff.at(frameshift).first;
            const double ff0 = ff.at(0).first;
            const double main_orf_freq = ff0 == 0.0 ? frameshift_freq : ff0;
            const double shift_orf_freq = shift_in_window ? frameshift_freq : (ff0 == 0.0 ? frameshift_freq : ff0);
            const double variant_freq_record = fwd ? record.freq / main_orf_freq : record.freq / shift_orf_freq;
            const double variant_freq_prev_record = fwd ? prev_record.freq / shift_orf_freq : prev_record.freq / main_orf_freq;
            const double freq_record = ff0 == 0.0 ? frameshift_freq : variant_freq_record * frameshift_freq;
            const double freq_prev_record = ff0 == 0.0 ? frameshift_freq : variant_freq_prev_record * frameshift_freq;
            const double out_freq = std::fabs(record.freq - prev_record.freq) < eps ? freq_record : freq_record * freq_prev_record;
            const uint64_t out_shift = shift_in_window ? 0 : frameshift;
            uint64_t splice_offset = 3 - out_shift;
            if (!fwd && exon_rest < 3) splice_offset += exon_rest;
            size_t end_offset = 3 + size_t(out_shift);
            if (is_last_exon_window) end_offset = 0;
            if (uint64_t(new_mt_sequence.size()) < 2 * window_len) {
              if (fwd) splice_offset = 0;
              else end_offset = 0;
            }
            auto sub = [](const std::string& s, uint64_t a, uint64_t e) -> std::string_view {
              if (a > e || e > s.size()) throw Fatal("slice index out of range");
              return std::string_view(s).substr(size_t(a), size_t(e - a));
            };
            while (splice_offset + window_len <= uint64_t(new_mt_sequence.size() - end_offset)) {
              // most windows across a junction are identical in both sequences: compare views, build strings only to emit
              std::string_view wt_view;
              if (splice_offset + window_len <= uint64_t(new_wt_sequence.size())) {
                if (fwd) wt_view = sub(new_wt_sequence, splice_offset, splice_offset + window_len);
                else wt_view = sub(new_wt_sequence, new_wt_sequence.size() - end_offset - size_t(window_len), new_wt_sequence.size() - end_offset);
              }
              const std::string_view mt_view = fwd ? sub(new_mt_sequence, splice_offset, splice_offset + window_len)
                                                   : sub(new_mt_sequence, new_mt_sequence.size() - end_offset - size_t(window_len),
                                                         new_mt_sequence.size() - end_offset);
              if (out_shift > 0 && wt_view == mt_view && somatic_shift) wt_view = std::string_view();
              if (wt_view == mt_view || (wt_view.empty() && frameshift == 0)) {
                if (fwd) splice_offset += 3;
                else end_offset += 3;
                continue;
              }
              const std::string out_wt_seq(wt_view), out_mt_seq(mt_view);
              const uint64_t out_offset = fwd ? splice_offset : uint64_t(end_offset);
              InfoRecord out_record = fwd ? detail::merge_records(prev_record, record, true, tm.id, out_offset, frameshift, out_freq, out_wt_seq, out_mt_seq, window_len)
                                          : detail::merge_records(record, prev_record, false, tm.id, out_offset, frameshift, out_freq, out_wt_seq, out_mt_seq, window_len);
              auto slot = output_map.try_emplace(std::make_tuple(out_offset, out_mt_seq, out_wt_seq)).first;
              const double old_freq = slot->second.rec.freq;  // 0.0 in a fresh slot
              slot->second = OutVal{out_mt_seq, detail::add_freq(std::move(out_record), old_freq), out_wt_seq};
              if (fwd) splice_offset += 3;
              else end_offset += 3;
            }
          }
        }
      }
    }
    if (is_short_exon && !is_last_exon) {
      prev_hap_vec = std::move(new_hap_vec);
    } else {
      for (auto& kv : output_map) {
        OutVal& v = kv.second;
        if (v.mt != v.wt) {
          OutRecord o;
          if (window_len > v.mt.size()) throw Fatal("slice index out of range");
          o.mt = v.mt.substr(0, size_t(window_len));
          o.has_mt = true;
          if (!v.wt.empty()) {
            if (window_len > v.wt.size()) throw Fatal("slice index out of range");
            o.wt = v.wt.substr(0, size_t(window_len));
            o.has_wt = true;
          }
          o.info = std::move(v.rec);  // the map dies with this call
          out.push_back(std::move(o));
        }
      }
      if (is_short_exon) prev_hap_vec = std::move(new_hap_vec);
    }
  }

 public:
  // (segment, number of windows the reference reaches) — used to sum depth over live windows only
  std::vector<std::pair<uint32_t, uint32_t>> seg_live_;

 private:
  const Batch& b_;
  const PhaseRaw& raw_;
  FILE* trace_ = nullptr;
  std::vector<std::pair<uint64_t, uint64_t>> active_scratch_;
  InfoRecord unused_rec_;  // what `rec` names in print() for a haplotype that needs no record; never written
  size_t iw_lo_ = 0, iw_hi_ = 0, iw_hint_ = 0;  // this segment's slice of raw_.iw and the last lookup (find_iw)
  std::vector<uint32_t> ks_scratch_;
  std::vector<Key> key_scratch_;  // print(): the window's keys projected onto one frame
};

}  // namespace mph
