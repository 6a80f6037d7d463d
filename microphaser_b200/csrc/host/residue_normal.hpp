// residue_normal.hpp — host residue of the `normal` (healthy peptidome) mode.
//
// The device returns the observation count of every enumerated window and, for windows that hold
// variants, the haplotype histogram with the assembled sequences. What stays on the host is the
// record construction of print_haplotypes (reference src/normal_microphasing.rs:509-645), the
// frameshift / ORF bookkeeping of the window loop (:1039-1141) and the splice-junction merge
// (:1145-1250, IDRecord::{update,add_freq} :104-180). Unlike the somatic mode every window of a
// non-short exon writes a record, so this pass is proportional to the output size.
#pragma once
#include "residue.hpp"

namespace mph {

class ResidueNormal {
 public:
  ResidueNormal(const Batch& b, const PhaseRaw& raw) : b_(b), raw_(raw) {}

  void run(uint32_t tx_lo, uint32_t tx_hi, std::vector<OutRecord>& out, ResidueStats& stats) {
    for (uint32_t t = tx_lo; t < tx_hi; ++t) {
      const TxMeta& tm = b_.txs[t];
      if (tm.seg_hi > tm.seg_lo && (b_.segs[tm.seg_lo].flags & MPH_SF_DEVREC)) continue;  // built on the device (core/record_core.h)
      run_transcript(t, out, stats);
    }
  }

 private:
  struct HapSeq {  // HaplotypeSeq (:182-186)
    std::string sequence;
    InfoRecord rec;
  };

  size_t find_iw(uint32_t widx) const {
    auto it = std::lower_bound(raw_.iw.begin(), raw_.iw.end(), widx);
    if (it == raw_.iw.end() || *it != widx) return SIZE_MAX;
    return size_t(it - raw_.iw.begin());
  }

  // IDRecord::update (:105-146)
  InfoRecord update(const InfoRecord& self, const InfoRecord& rec, uint64_t off, const std::string& seq, const std::string& tx_id, bool rev) const {
    InfoRecord o;
    o.id = mphfmt::record_id(reinterpret_cast<const uint8_t*>(seq.data()), seq.size(), tx_id, off, rev ? 'R' : 'F');
    o.tx = self.tx;
    o.offset = off + self.offset;
    o.frame = self.frame;
    o.freq = self.freq * rec.freq;
    o.depth = self.depth;
    o.nvar = self.nvar + rec.nvar;
    o.nsomatic = self.nsomatic + rec.nsomatic;
    o.nvariant_sites = self.nvariant_sites + rec.nvariant_sites;
    o.nsomvariant_sites = self.nsomvariant_sites + rec.nsomvariant_sites;
    o.variant_sites = self.variant_sites + rec.variant_sites;
    o.somatic_positions = self.somatic_positions + rec.somatic_positions;
    o.somatic_aa_change = self.somatic_aa_change + rec.somatic_aa_change;
    o.germline_positions = self.germline_positions + rec.germline_positions;
    o.germline_aa_change = self.germline_aa_change + rec.germline_aa_change;
    o.mutant_sequence = seq;
    return o;
  }
  // IDRecord::add_freq (:148-179); the u32 subtraction wraps like the release build
  static InfoRecord add_freq(const InfoRecord& r, double f) {
    InfoRecord o = r;
    const uint32_t new_nvar = f > 0.0 ? r.nvar - 1u : r.nvar;
    o.nsomatic = new_nvar < r.nsomatic ? r.nsomatic - 1u : r.nsomatic;
    o.nvar = new_nvar;
    o.freq = r.freq + f;
    return o;
  }

  // variant-site metadata (:509-560): 0-based positions; sites are only counted while the walk
  // produced a profile entry for the variant
  void fill_meta(InfoRecord& rec, const WinVars& wv, const MphHap& h) const {
    const uint32_t nv = wv.n;
    uint32_t n_sites = 0, n_som_sites = 0;
    std::string s_pc, g_pc, s_pos, g_pos, sites;
    bool fs = true, fg = true, fsite = true, fspc = true, fgpc = true;
    char buf[24];
    auto put = [&](std::string& dst, bool& first, uint64_t v) {
      if (!first) dst.push_back('|');
      first = false;
      auto r = std::to_chars(buf, buf + sizeof buf, v);
      dst.append(buf, r.ptr);
    };
    for (uint32_t c = 0; c < nv && c < h.n_prof; ++c) {
      const MphVar& v = b_.vars[wv.at(c)];
      const unsigned code = c < 32 ? unsigned((h.profile >> (2 * c)) & 3) : 0;
      if (code == 2) {
        put(s_pos, fs, v.pos);
        if (!fspc) s_pc.push_back('|');
        fspc = false;
        s_pc += b_.var_prot[wv.at(c)];
      } else if (code == 1) {
        put(g_pos, fg, v.pos);
        if (!fgpc) g_pc.push_back('|');
        fgpc = false;
        g_pc += b_.var_prot[wv.at(c)];
      }
      if (c == 0 || v.pos != b_.vars[wv.at(c - 1)].pos) {
        ++n_sites;
        put(sites, fsite, v.pos);
        if (!(v.flags & MPH_VF_GERMLINE)) ++n_som_sites;
      }
    }
    rec.nvar = h.n_var;
    rec.nsomatic = h.n_som;
    rec.nvariant_sites = n_sites;
    rec.nsomvariant_sites = n_som_sites;
    rec.variant_sites = std::move(sites);
    rec.somatic_positions = std::move(s_pos);
    rec.somatic_aa_change = std::move(s_pc);
    rec.germline_positions = std::move(g_pos);
    rec.germline_aa_change = std::move(g_pc);
  }

  // print_haplotypes (:341-647) with the matrix scan and the sequence walk replaced by device results
  std::vector<HapSeq> print(uint32_t t, const MphSegment& sg, uint32_t k, uint32_t widx, uint64_t frame, bool keep, std::vector<OutRecord>& out,
                            size_t* n_res) {
    const TxMeta& tm = b_.txs[t];
    const bool rev = tm.reverse;
    const MphGeom g = mph_geom(sg, k);
    WinVars wv;
    wv.va = mph_var_lb(b_.vars.data(), sg.var_lo, sg.var_hi, g.s);
    wv.n = mph_var_lb(b_.vars.data(), sg.var_lo, sg.var_hi, g.e) - wv.va;
    size_t iwi = SIZE_MAX;
    if (sg.flags & MPH_SF_REPLAY) {
      // replayed transcript: the matrix columns are what the replay recorded, not the variants inside the window
      iwi = find_iw(widx);
      wv.n = 0;
      if (iwi != SIZE_MAX && !raw_.iw_voff.empty() && raw_.iw_voff[iwi] != 0xFFFFFFFFu) {
        const uint32_t off = raw_.iw_voff[iwi];
        wv.n = raw_.vlist[off];
        wv.list = raw_.vlist.data() + off + 1;
      }
    }
    const uint32_t nv = wv.n;
    const bool is_short_exon = (sg.flags & MPH_SF_SHORT) != 0;
    const uint64_t window_len = sg.ewl;
    const uint32_t wd = raw_.win_depth[widx - raw_.win_base];
    const uint32_t depth = wd & 0x7FFFFFFFu;
    std::vector<Key>& keybuf = key_scratch_;  // reused across windows; a window may have any number of keys
    keybuf.clear();
    MphHap plain;
    if (nv == 0) {
      memset(&plain, 0, sizeof plain);
      plain.flags = (wd >> 31) ? MPH_NF_STOP : 0;
      plain.seq_len = uint16_t(g.e - g.s);
      keybuf.push_back(Key{0, depth, &plain});
    } else {
      if (iwi == SIZE_MAX) iwi = find_iw(widx);
      if (iwi == SIZE_MAX) throw std::logic_error("internal: window summary missing");
      const MphWinOut& wo = raw_.iw_out[iwi];
      if (wo.c0 > 0) keybuf.push_back(Key{0, wo.c0, &raw_.iw_hap0[iwi]});
      for (uint32_t x = 0; x < wo.n_extra; ++x) {
        const MphHist& e = raw_.hist[wo.extra_off + x];
        keybuf.push_back(Key{e.hap, e.count, &raw_.hapx[wo.extra_off + x]});
      }
      if (keybuf.empty()) keybuf.push_back(Key{0, 0, &raw_.iw_hap0[iwi]});
    }
    std::vector<HapSeq> res;
    *n_res = 0;
    for (size_t q = 0; q < keybuf.size(); ++q) {
      const Key& key = keybuf[q];
      const MphHap& h = *key.info;
      if (h.flags & MPH_NF_REFRANGE) throw Fatal("index out of bounds: refseq");  // the reference panics when it reaches this walk
      const double freq = double(key.count) / double(depth);  // NaN without observations (:397)
      const bool stop_gain = (h.flags & MPH_NF_STOP) != 0;
      if (stop_gain && g.spos != 2) continue;
      if (h.flags & MPH_NF_OVERFLOW) throw Unsupported("assembled haplotype longer than the sequence slot");
      std::string seq;
      if (key.hap == 0) {
        if (g.s < sg.ref_pos0 || uint64_t(g.e) - sg.ref_pos0 > sg.ref_len) throw Fatal("slice index out of range: refseq");
        seq.assign(reinterpret_cast<const char*>(b_.ref.data()) + sg.ref_off + (g.s - sg.ref_pos0), g.e - g.s);
      } else {
        if (!(h.flags & MPH_NF_SEQ)) throw std::logic_error("internal: sequence not shipped");
        seq.assign(reinterpret_cast<const char*>(raw_.seq.data()) + h.seq_off, h.seq_len);
      }
      const bool insertion = (h.flags & MPH_NF_INSERTION) != 0;
      const uint64_t this_window_len = seq.size() < window_len ? uint64_t(seq.size()) : window_len;
      auto slice = [&](uint64_t a, uint64_t e) -> std::string {
        if (a > e || e > seq.size()) throw Fatal("slice index out of range");
        return seq.substr(size_t(a), size_t(e - a));
      };
      OutRecord o;
      InfoRecord& rec = o.info;
      if (g.spos == 1) rec.mutant_sequence = slice(g.gap, seq.size());
      else if (g.spos == 0) rec.mutant_sequence = insertion ? seq : slice(0, this_window_len);
      else rec.mutant_sequence = seq;
      {
        // ids are hashed on the device: per window for the reference haplotype, per key for the others
        uint64_t id64 = 0;
        bool have = false;
        if (key.hap == 0) { have = !raw_.win_id.empty() && raw_.win_id[widx - raw_.win_base] != 0; if (have) id64 = raw_.win_id[widx - raw_.win_base]; }
        else if (h.flags & MPH_NF_ID) { have = true; id64 = h.id64; }
        if (have) {
          static const char* hx = "0123456789abcdef";
          rec.id.resize(16);
          for (int q2 = 0; q2 < 15; ++q2) rec.id[q2] = hx[(id64 >> (60 - 4 * q2)) & 15];
          rec.id[15] = rev ? 'R' : 'F';
        } else {
          rec.id = mphfmt::record_id(reinterpret_cast<const uint8_t*>(seq.data()), seq.size(), tm.id, g.s, rev ? 'R' : 'F');
        }
      }
      rec.tx = t;
      rec.offset = g.s;
      rec.frame = frame;
      rec.freq = freq;
      rec.depth = depth;
      if (nv) fill_meta(rec, wv, h);
      ++*n_res;
      if (keep) {
        HapSeq hs;
        hs.rec = rec;
        hs.rec.mutant_sequence = seq;
        hs.sequence = seq;
        res.push_back(std::move(hs));
      }
      if (!is_short_exon) {
        if (g.spos == 1) { o.mt = rec.mutant_sequence; o.has_mt = true; }
        else if (g.spos == 0) {
          if (window_len > seq.size()) throw Fatal("slice index out of range");
          o.mt = seq.substr(0, size_t(window_len));
          o.has_mt = true;
        }
        out.push_back(std::move(o));
      }
    }
    return res;
  }

  static bool is_boundary(const MphSegment& sg, uint32_t k) {
    if (sg.n_win == 0) return false;
    if (sg.flags & (MPH_SF_HAS_FS | MPH_SF_SHORT)) return true;
    // a junction merge reads the latest list stored on either side (:1116-1120): the first window, the
    // last one, and - when the next exon's first window is also its last - the one before the last
    const uint32_t i = (k - sg.k_first) / sg.k_stride;
    return i == 0 || i + 2 >= sg.n_win;
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
      uint32_t prev_vb_fs = 0, prev_va_fs = 0;
      bool fs_init = false;
      const uint32_t n_steps = has_fs ? sg.n_iter : sg.n_win;
      // iteration at which the reference panics (found by the replay); reached unless the ORF ended before
      const uint32_t panic_k = raw_.seg_err.empty() ? 0xFFFFFFFFu : raw_.seg_err[si - raw_.seg_base] - 1u;
      bool left_early = false;
      for (uint32_t step = 0; step < n_steps; ++step) {
        if (frameshifts.empty()) { left_early = true; break; }
        const uint32_t k = has_fs ? step : sg.k_first + step * sg.k_stride;
        if (k >= panic_k) throw Fatal("drain: range end out of bounds");
        const MphGeom g = mph_geom(sg, k);
        const uint64_t offset = fwd ? uint64_t(sg.off0) + k : uint64_t(sg.off0) - k;
        const uint64_t rest = fwd ? sg.exon_end - (offset + exon_window_len) : offset - sg.exon_start;
        const bool is_last_exon_window = rest < 3;
        if (has_fs) {
          // variants collected at this iteration (:1018-1049) in collection order
          const uint32_t va = mph_var_lb(b_.vars.data(), sg.var_lo, sg.var_hi, g.s);
          const uint32_t vb = mph_var_lb(b_.vars.data(), sg.var_lo, sg.var_hi, g.e);
          uint32_t na, nb;
          if (!fs_init || k == 0) { na = va; nb = vb; }
          else if (fwd) { na = std::max(prev_vb_fs, va); nb = vb; }
          else { na = va; nb = std::min(prev_va_fs, vb); }
          fs_init = true;
          prev_va_fs = va; prev_vb_fs = vb;
          auto handle = [&](const MphVar& v) {
            const uint64_t s = (v.flags & MPH_VF_FS_MASK) >> MPH_VF_FS_SHIFT;
            if (s > 0) {  // no "% 3", no strand split (:1039-1049)
              std::vector<uint64_t> previous;
              for (auto& kv : frameshifts) previous.push_back(kv.second + s);
              const uint64_t end_pos = v.kind == MPH_DEL ? uint64_t(v.pos) + v.len - 1 : v.pos;
              for (uint64_t s_ : previous) frameshifts[end_pos] = s_;
            }
          };
          if (fwd) for (uint32_t j = na; j < nb; ++j) handle(b_.vars[j]);
          else for (uint32_t j = nb; j > na; --j) handle(b_.vars[j - 1]);
        }
        uint64_t stopped_frameshift = 3;
        std::vector<std::pair<uint64_t, uint64_t>> active;
        if (fwd) { for (auto it = frameshifts.begin(); it != frameshifts.end() && it->first < offset; ++it) active.push_back(*it); }
        else { for (auto it = frameshifts.lower_bound(offset + exon_window_len); it != frameshifts.end(); ++it) active.push_back(*it); }
        uint64_t frameshift_count = 0;
        bool main_orf = false;
        for (auto& kf : active) {
          const uint64_t key = kf.first, frameshift = kf.second;
          if (frameshift == 0) main_orf = true;
          ++frameshift_count;
          const uint64_t coding_shift = fwd ? offset - sg.exon_start : sg.exon_end - offset;
          if (coding_shift % 3 == (frameshift + current_exon_offset) % 3 || is_short_exon) {
            if (frameshift == 0) {
              exon_rest = rest;
              if (exon_window_len < 3) exon_rest = exon_window_len;
            }
            if (k < sg.k_first || (k - sg.k_first) % sg.k_stride != 0) throw std::logic_error("internal: window was not enumerated");
            const uint32_t widx = sg.win_base + (k - sg.k_first) / sg.k_stride;
            if (frameshift == 0) {
              stats.windows += 1;
              stats.read_windows += raw_.win_depth[widx - raw_.win_base] & 0x7FFFFFFFu;
            }
            size_t n_res = 0;
            auto res = print(t, sg, k, widx, frameshift, is_boundary(sg, k), out, &n_res);
            if (n_res == 0) stopped_frameshift = key;
            if (exon_rest < 3 && (!is_short_exon || is_first_exon)) prev_hap_vec = std::move(res);
            else hap_vec = std::move(res);
          }
        }
        if (frameshift_count == 0 || !main_orf) {
          frameshifts.clear();
          left_early = true;
          break;
        }
        frameshifts.erase(stopped_frameshift);  // :1130 — unconditional
        if (frameshifts.empty()) { left_early = true; break; }
        const bool at_splice_side = fwd ? offset - current_exon_offset == sg.exon_start
                                        : offset + exon_window_len + current_exon_offset == sg.exon_end;
        if (at_splice_side && !is_first_exon)
          splice_merge(t, fwd, is_short_exon, is_last_exon, is_last_exon_window, exon_rest, window_len, hap_vec, prev_hap_vec, out);
        if (is_short_exon) break;
      }
      if (!left_early && !frameshifts.empty() && panic_k != 0xFFFFFFFFu) throw Fatal("drain: range end out of bounds");
    }
  }

  // :1145-1250
  void splice_merge(uint32_t t, bool fwd, bool is_short_exon, bool is_last_exon, bool is_last_exon_window, uint64_t exon_rest, uint64_t window_len,
                    std::vector<HapSeq>& hap_vec, std::vector<HapSeq>& prev_hap_vec, std::vector<OutRecord>& out) {
    const TxMeta& tm = b_.txs[t];
    const std::vector<HapSeq>& first_hap_vec = fwd ? hap_vec : prev_hap_vec;
    const std::vector<HapSeq>& sec_hap_vec = fwd ? prev_hap_vec : hap_vec;
    std::map<std::pair<uint64_t, std::string>, std::pair<std::string, InfoRecord>> output_map;
    std::vector<HapSeq> new_hap_vec;
    for (const HapSeq& hapseq : first_hap_vec) {
      for (const HapSeq& prev_hapseq : sec_hap_vec) {
        const InfoRecord& record = hapseq.rec;
        const InfoRecord& prev_record = prev_hapseq.rec;
        const std::string joined = prev_hapseq.sequence + hapseq.sequence;
        if (is_short_exon) {
          HapSeq nh;
          nh.sequence = joined;
          nh.rec = update(prev_record, record, 0, joined, tm.id, !fwd);
          new_hap_vec.push_back(std::move(nh));
        }
        uint64_t splice_offset = 3;
        if (!fwd && exon_rest < 3) splice_offset += exon_rest;
        size_t end_offset = 3;
        if (is_last_exon_window) end_offset = 0;
        if (uint64_t(joined.size()) < 2 * window_len) {
          if (fwd) splice_offset = 0;
          else end_offset = 0;
        }
        while (splice_offset + window_len <= uint64_t(joined.size() - end_offset)) {
          if (splice_offset + window_len > joined.size()) throw Fatal("slice index out of range");
          std::string out_seq = joined.substr(size_t(splice_offset), size_t(window_len));
          InfoRecord out_record = update(prev_record, record, splice_offset, out_seq, tm.id, !fwd);
          auto id_tuple = std::make_pair(splice_offset, out_seq);
          auto it = output_map.find(id_tuple);
          const double old_freq = it != output_map.end() ? it->second.second.freq : 0.0;
          output_map[id_tuple] = std::make_pair(out_seq, add_freq(out_record, old_freq));
          splice_offset += 3;
        }
      }
    }
    if (is_short_exon && !is_last_exon) {
      prev_hap_vec = std::move(new_hap_vec);
    } else {
      for (auto& kv : output_map) {
        OutRecord o;
        const std::string& out_seq = kv.second.first;
        if (window_len > out_seq.size()) throw Fatal("slice index out of range");
        o.mt = out_seq.substr(0, size_t(window_len));
        o.has_mt = true;
        o.info = kv.second.second;
        out.push_back(std::move(o));
      }
    }
  }

  struct Key { uint64_t hap; uint64_t count; const MphHap* info; };
  const Batch& b_;
  const PhaseRaw& raw_;
  std::vector<Key> key_scratch_;  // print(): the window's keys
};

}  // namespace mph
