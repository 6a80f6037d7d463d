// record_core.h — record emission on the device: what print_haplotypes does with a window's histogram
// (reference src/microphasing.rs:604-875), ORF termination (:1465-1488) and the splice-junction merge
// (:1497-1908, IDRecord::update / add_freq src/common.rs:376-568), restated per item as host+device
// inline functions. The kernels of kernels/record_kernels.cu wrap them in the parallel structure; the
// test-only CPU emulator (tests/emu) wraps the same functions in plain loops.
//
// Which transcripts take this path ("device class", MPH_SF_DEVREC, decided by the packer): no frameshifting
// variant in the gene, no short exon, no skipped exon, at least two windows per exon, no serial replay. For those
// the state the reference threads through consecutive print_haplotypes calls collapses:
//   * `frameshifts` holds the single main-ORF entry (:953-957) and every enumerated window is in frame;
//   * `frameshift_frequencies` is {0: (1.0, false)} until the first haplotype with a premature stop sets it to
//     (0.0, false) (:703-718); the later haplotypes of that window then have frequency 0 and the transcript ends
//     after it (:1480-1488). Whether a haplotype removes the peptide does not depend on that state, so the first
//     such window of a transcript is a minimum over independent per-window tests.
//   * a junction merge (:1497-1908) reads the haplotype lists of exactly two windows - the first window of the
//     exon and the last window of the previous one - and runs with frameshift 0 and frequency 1.0 for the ORF.
// Everything else (frameshifts, short exons, replayed transcripts) stays with the host residue.
#pragma once
#include <math.h>

#include "phase_core.h"

// record flags
enum {
  MPH_RC_HAS_MT = 1,   // a line goes to the mutant FASTA (:846-858)
  MPH_RC_HAS_WT = 2,   // a line goes to the normal FASTA (:859-873)
  MPH_RC_MERGED = 4,   // produced by a junction merge: two sources, `aux` names the second
  MPH_RC_REVERSE = 8,
};

// One record as the device hands it over, 64 B. The text columns are rendered on the host from these fields:
// the position / amino-acid-change lists are the variants [var_ref, var_ref + n_win) of the source window whose
// profile code is 2 (somatic) or 1 (germline) and whose `keep` bit is set.
typedef struct {
  uint64_t id64;      // leading 64 bits of sha1(format!("{:?}{}{}", seq, transcript, offset)) (:667-675)
  double freq;
  uint32_t tx;
  uint32_t offset;    // `offset` column
  uint32_t depth;
  uint32_t seq_off;   // record sequence arena: max(neo_len, mt_len) mutant bytes, then max(norm_len, wt_len) normal bytes
  uint32_t var_ref;   // source A: first variant of its window
  uint32_t keep;      // source A: bit c <-> visited variant c passes the merge's position filter (all ones for a plain record)
  uint64_t profile;   // source A: 2 bits per visited variant, 0 absent, 1 germline, 2 somatic
  uint64_t n_prof : 7, n_win : 7;  // source A: visited variants, variants in the window (both <= 64)
  uint64_t nvar : 8, nsomatic : 8, nsites : 8, nsomsites : 8;
  uint64_t flags : 6;  // MPH_RC_*
  uint64_t rank : 12;  // merged: position among the junction's records in output_map order (< MPH_RC_JUNCTION_RECS)
  uint8_t neo_len, mt_len, norm_len, wt_len;  // `mutant_sequence` column, mutant FASTA line, `normal_sequence` column, normal FASTA line
  uint32_t aux;       // merged: index of source B in the aux array
} MphRec;
#define MPH_RC_JUNCTION_RECS 4096  // records one splice junction may write (the width of `rank`); more raise MPH_E_RECS_PER_LIST
#ifdef __cplusplus
static_assert(sizeof(MphRec) == 64, "MphRec is 64 B");
#endif

typedef struct {  // source B of a merged record, 24 B
  uint64_t profile;
  uint32_t var_ref, keep;
  uint8_t n_prof, n_win;
  uint8_t pad[6];
} MphRecSrc;

enum { MPH_RC_SEQ_SLOT = 64 };  // bytes of sequence a merged record owns in the merge arena (2 x window_len <= 64)

typedef struct {
  const MphSegment* segs;
  const MphVar* vars;
  const uint8_t* ref;
  const MphWinOut* win_out;
  const MphHap* hap0;
  const MphHist* hist;
  const MphHap* hapx;
  const uint8_t* seq;  // K3's arena for device-class transcripts: slots of 2 * seq_cap bytes (seq, germline_seq)
  uint32_t seq_cap;
  const uint8_t* tx_id_bytes;
  const uint32_t* tx_id_off;
} MphRecCtx;

// ---- keys of a window in print_haplotypes order (:383,434): haplotype 0 first, then the extra keys (sorted by K2)
typedef struct {
  uint64_t hap;
  uint32_t count;
  const MphHap* h;
} MphKeyRef;

MPH_HD uint32_t mph_rc_nkeys(const MphWinOut& wo) {
  const uint32_t n = (wo.c0 > 0 ? 1u : 0u) + wo.n_extra;
  return n ? n : 1u;  // an empty histogram still visits haplotype 0 with count 0 (:386)
}
MPH_HD MphKeyRef mph_rc_key(const MphRecCtx& c, const MphWinOut& wo, uint32_t widx, uint32_t q) {
  MphKeyRef k;
  if (wo.c0 > 0 || wo.n_extra == 0) {
    if (q == 0) { k.hap = 0; k.count = wo.c0; k.h = &c.hap0[widx]; return k; }
    q -= 1;
  }
  const uint32_t idx = wo.extra_off + q;
  k.hap = c.hist[idx].hap;
  k.count = c.hist[idx].count;
  k.h = k.hap == 0 ? &c.hap0[widx] : &c.hapx[idx];
  return k;
}
MPH_HD uint64_t mph_rc_frame_depth(const MphRecCtx& c, const MphWinOut& wo) {
  uint64_t d = wo.c0;
  for (uint32_t x = 0; x < wo.n_extra; ++x) d += c.hist[wo.extra_off + x].count;
  return d;
}

// ---- one haplotype of one window (:604-718, :839-844), device class
typedef struct {
  double freq;        // count / frame_depth (:404)
  uint8_t remove;     // remove_peptide (:703-718)
  uint8_t emit_ok;    // the emission predicate (:839-844) but for `freq > 0`
  uint8_t cleared;    // germline_seq was cleared (:624-631)
  uint32_t err;       // MPH_E_* bits the reference's panics map to
  uint32_t twl, nwl;  // this_window_len, normal_window_len (:651-660)
} MphKeyEval;

MPH_HD MphKeyEval mph_rc_eval(const MphSegment& sg, const MphGeom& g, uint32_t k, const MphKeyRef& key, uint64_t frame_depth) {
  MphKeyEval e;
  const MphHap& h = *key.h;
  e.err = 0;
  if (h.flags & MPH_HF_REFRANGE) e.err |= MPH_E_REF_RANGE;  // the reference panics when it reaches this walk
  e.freq = key.count == 0 ? 0.0 : (double)key.count / (double)frame_depth;
  const bool indel = (h.flags & MPH_HF_INDEL) != 0, insertion = (h.flags & MPH_HF_INSERTION) != 0;
  e.cleared = indel && insertion;
  const uint32_t seq_len = h.seq_len, germ_len = e.cleared ? 0u : h.germ_len, wl = sg.ewl;
  e.twl = seq_len < wl ? seq_len : wl;
  e.nwl = indel ? (germ_len < wl ? germ_len : wl) : e.twl;
  const bool stop_gain = (h.flags & MPH_HF_STOP) != 0;
  const bool seqs_equal = e.cleared ? seq_len == 0 : (h.flags & MPH_HF_GERM_EQ) != 0;
  e.emit_ok = h.n_som > 0 && !seqs_equal && !stop_gain;
  const bool pepdiff = key.hap == 0 ? false : (h.flags & MPH_HF_PEPDIFF) != 0;
  e.remove = stop_gain && g.spos != 2 && (wl == e.twl || indel) && k != 0 &&
             (pepdiff || !indel || fabs(e.freq - 1.0) < 2.220446049250313e-16);
  if (key.hap != 0 && (h.flags & MPH_HF_SLICE_ERR)) e.err |= MPH_E_SLICE;
  return e;
}

// first haplotype of the window that removes the peptide, 0xFFFFFFFF if none
MPH_HD uint32_t mph_rc_window_stop(const MphRecCtx& c, const MphSegment& sg, uint32_t i, uint32_t widx) {
  const MphWinOut wo = c.win_out[widx];
  const uint32_t k = sg.k_first + i * sg.k_stride;
  const MphGeom g = mph_geom(sg, k);
  const uint64_t fd = mph_rc_frame_depth(c, wo);
  const uint32_t nk = mph_rc_nkeys(wo);
  for (uint32_t q = 0; q < nk; ++q) {
    const MphKeyRef key = mph_rc_key(c, wo, widx, q);
    if (mph_rc_eval(sg, g, k, key, fd).remove) return q;
  }
  return 0xFFFFFFFFu;
}

// variant sites of a window (:757-769): distinct positions, and how many of them start with a somatic allele
MPH_HD void mph_rc_sites(const MphVar* vars, uint32_t va, uint32_t n, uint32_t* nsites, uint32_t* nsom) {
  uint32_t a = 0, b = 0;
  for (uint32_t c = 0; c < n; ++c)
    if (c == 0 || vars[va + c].pos != vars[va + c - 1].pos) {
      ++a;
      if (!(vars[va + c].flags & MPH_VF_GERMLINE)) ++b;
    }
  *nsites = a;
  *nsom = b;
}

// sequences of one haplotype as print_haplotypes holds them after the clearing step: `mt` = seq, `wt` = germline_seq
typedef struct {
  const uint8_t* mt;
  const uint8_t* wt;
  uint32_t mt_len, wt_len;
  uint32_t err;
} MphHapSeqs;

MPH_HD MphHapSeqs mph_rc_seqs(const MphRecCtx& c, const MphSegment& sg, const MphGeom& g, const MphKeyRef& key) {
  MphHapSeqs s;
  s.err = 0;
  const MphHap& h = *key.h;
  if (key.hap == 0) {  // no variant applied: both are refseq[s..e) (:464-471,594-599)
    s.mt = s.wt = c.ref + sg.ref_off + (g.s - sg.ref_pos0);
    s.mt_len = s.wt_len = g.e - g.s;
    if (g.s < sg.ref_pos0 || (uint64_t)g.e - sg.ref_pos0 > sg.ref_len) { s.err |= MPH_E_REF_RANGE; s.mt_len = s.wt_len = 0; }
    return s;
  }
  if (!(h.flags & MPH_HF_SEQ)) { s.err |= MPH_E_INTERNAL; s.mt = s.wt = c.ref; s.mt_len = s.wt_len = 0; return s; }
  if (h.flags & MPH_HF_OVERFLOW) s.err |= MPH_E_SEQ_SLOT;
  s.mt = c.seq + h.seq_off;
  s.wt = s.mt + c.seq_cap;
  s.mt_len = h.seq_len < c.seq_cap ? h.seq_len : c.seq_cap;
  const bool cleared = (h.flags & MPH_HF_INDEL) && (h.flags & MPH_HF_INSERTION);
  s.wt_len = cleared ? 0u : (h.germ_len < c.seq_cap ? h.germ_len : c.seq_cap);
  return s;
}

// number of records a live window writes itself (:839-875); q_stop = first removing haplotype of the window
MPH_HD uint32_t mph_rc_window_count(const MphRecCtx& c, const MphSegment& sg, uint32_t i, uint32_t widx, uint32_t q_stop, uint32_t* seq_bytes,
                                    uint32_t* err) {
  const MphWinOut wo = c.win_out[widx];
  const uint32_t k = sg.k_first + i * sg.k_stride;
  const MphGeom g = mph_geom(sg, k);
  const uint64_t fd = mph_rc_frame_depth(c, wo);
  const uint32_t nk = mph_rc_nkeys(wo);
  uint32_t n = 0, bytes = 0;
  for (uint32_t q = 0; q < nk; ++q) {
    const MphKeyRef key = mph_rc_key(c, wo, widx, q);
    const MphKeyEval e = mph_rc_eval(sg, g, k, key, fd);
    *err |= e.err;
    if (!(e.emit_ok && e.freq > 0.0 && q <= q_stop)) continue;  // after the removing haplotype the ORF frequency is 0 (:423)
    ++n;
    bytes += (uint32_t)key.h->seq_len + (uint32_t)key.h->germ_len;  // upper bound: the slices are parts of seq and germline_seq
  }
  *seq_bytes = bytes;
  return n;
}

// Writes the records of a live window at recs[0 .. n) and their bytes into seq_arena from seq_base on (the caller
// reserved the bytes mph_rc_window_count returned). Returns the number of records written.
MPH_HD uint32_t mph_rc_window_emit(const MphRecCtx& c, const MphSegment& sg, uint32_t i, uint32_t widx, uint32_t q_stop, MphRec* recs,
                                   uint8_t* seq_arena, uint32_t seq_base, uint32_t* err) {
  const MphWinOut wo = c.win_out[widx];
  const uint32_t k = sg.k_first + i * sg.k_stride;
  const MphGeom g = mph_geom(sg, k);
  const uint64_t fd = mph_rc_frame_depth(c, wo);
  const uint32_t nk = mph_rc_nkeys(wo);
  const bool rev = (sg.flags & MPH_SF_REVERSE) != 0;
  const uint32_t va = mph_var_lb(c.vars, sg.var_lo, sg.var_hi, g.s);
  const uint32_t nv = mph_var_lb(c.vars, va, sg.var_hi, g.e) - va;
  uint32_t nsites, nsom_sites;
  mph_rc_sites(c.vars, va, nv, &nsites, &nsom_sites);
  uint32_t n = 0, pos = seq_base;
  for (uint32_t q = 0; q < nk; ++q) {
    const MphKeyRef key = mph_rc_key(c, wo, widx, q);
    const MphKeyEval e = mph_rc_eval(sg, g, k, key, fd);
    if (!(e.emit_ok && e.freq > 0.0 && q <= q_stop)) continue;
    const MphHap& h = *key.h;
    const MphHapSeqs s = mph_rc_seqs(c, sg, g, key);
    *err |= s.err;
    // slices of :677-693 (TSV columns) and :846-873 (FASTA lines); a = common start of all four
    const uint32_t a = g.spos == 1 ? g.gap : 0u;
    const bool insertion = (h.flags & MPH_HF_INSERTION) != 0;
    uint32_t neo_b, mt_b, norm_b = 0, wt_b = 0;
    if (g.spos == 1) { neo_b = mt_b = s.mt_len; if (a > s.mt_len) *err |= MPH_E_SLICE; }
    else { mt_b = e.twl; neo_b = insertion ? s.mt_len : e.twl; }
    uint8_t flags = MPH_RC_HAS_MT | (rev ? MPH_RC_REVERSE : 0);
    if (s.wt_len > 0) {
      flags |= MPH_RC_HAS_WT;
      if (g.spos == 1) { norm_b = wt_b = s.wt_len; if (a > s.wt_len) *err |= MPH_E_SLICE; }
      else {
        norm_b = e.nwl;
        wt_b = e.twl;
        if (e.nwl > s.wt_len || e.twl > s.wt_len) *err |= MPH_E_SLICE;
      }
    }
    if (*err & (MPH_E_SLICE | MPH_E_REF_RANGE | MPH_E_INTERNAL | MPH_E_SEQ_SLOT)) { neo_b = mt_b = norm_b = wt_b = a; }
    const uint32_t mut_n = (neo_b > mt_b ? neo_b : mt_b) - a, nrm_n = norm_b > wt_b ? norm_b - a : (wt_b > a ? wt_b - a : 0u);
    if (mut_n > 255 || nrm_n > 255) *err |= MPH_E_SEQ_SLOT;
    MphRec r;
    r.id64 = h.id64;
    if (!(h.flags & MPH_HF_ID)) *err |= MPH_E_INTERNAL;
    r.freq = e.freq;  // the ORF frequency is 1.0 up to the removing haplotype (:423)
    r.tx = sg.tx;
    r.offset = g.spos == 0 ? g.s + 1u : g.s + 1u + g.gap;
    r.depth = wo.depth;
    r.seq_off = pos;
    r.var_ref = va;
    r.keep = 0xFFFFFFFFu;
    r.profile = h.profile;
    r.n_prof = h.n_prof;
    r.n_win = (uint8_t)nv;
    r.nvar = h.n_var;
    r.nsomatic = h.n_som;
    r.nsites = (uint8_t)nsites;
    r.nsomsites = (uint8_t)nsom_sites;
    r.flags = flags;
    r.rank = 0;
    r.neo_len = (uint8_t)(neo_b - a);
    r.mt_len = (uint8_t)(mt_b - a);
    r.norm_len = (uint8_t)(norm_b > a ? norm_b - a : 0u);
    r.wt_len = (uint8_t)(wt_b > a ? wt_b - a : 0u);
    r.aux = 0xFFFFFFFFu;
    for (uint32_t t = 0; t < mut_n && mut_n <= 255; ++t) seq_arena[pos + t] = s.mt[a + t];
    pos += mut_n <= 255 ? mut_n : 0u;
    for (uint32_t t = 0; t < nrm_n && nrm_n <= 255; ++t) seq_arena[pos + t] = s.wt[a + t];
    pos += nrm_n <= 255 ? nrm_n : 0u;
    recs[n++] = r;
  }
  return n;
}

// ================================================================================================ junction merge
// One entry of a haplotype list (HaplotypeSeq :141-145 with its IDRecord) as the merge reads it.
typedef struct {
  MphHapSeqs s;
  double freq;
  uint32_t offset, depth;
  uint32_t var_ref;
  uint64_t profile;
  uint8_t n_prof, n_win, nsites, nsomsites;
  uint8_t same;      // wt == mt
  uint8_t aligned;   // wt and mt have the same length (<= 64): `diff` marks the positions where they differ
  uint64_t diff;
} MphListEntry;

// byte x of the concatenation a + b
MPH_HD uint8_t mph_rc_cat(const uint8_t* a, uint32_t an, const uint8_t* b, uint32_t x) { return x < an ? a[x] : b[x - an]; }

// The byte-level steps of the merge. One thread does them with plain loops (the emulator; a lone device thread); the
// merge kernel runs one warp per junction with every lane executing the same control flow, and replaces these steps by
// lane-parallel versions (kernels/record_kernels.cu: MphWarpOps) - the single-thread latency of ~50 dependent byte loads
// per step is what made a junction's chain long.
struct MphSerialOps {
  struct Win {  // one candidate's mutant and wild-type window
    uint8_t mt[MPH_RC_SEQ_SLOT / 2], wt[MPH_RC_SEQ_SLOT / 2];
  };
  static MPH_HD bool leader() { return true; }
  static MPH_HD void sync() {}  // orders the leader's stores before the other lanes' loads
  static MPH_HD uint64_t diff_mask(const uint8_t* a, const uint8_t* b, uint32_t n) {  // n <= 64
    uint64_t m = 0;
    for (uint32_t x = 0; x < n; ++x)
      if (a[x] != b[x]) m |= (uint64_t)1 << x;
    return m;
  }
  static MPH_HD bool window_equal(const uint8_t* ma, uint32_t man, const uint8_t* mb, uint64_t ms, const uint8_t* wa, uint32_t wan,
                                  const uint8_t* wb, uint64_t ws, uint32_t wl) {
    for (uint32_t x = 0; x < wl; ++x)
      if (mph_rc_cat(ma, man, mb, (uint32_t)(ms + x)) != mph_rc_cat(wa, wan, wb, (uint32_t)(ws + x))) return false;
    return true;
  }
  static MPH_HD void load(Win& w, const uint8_t* ma, uint32_t man, const uint8_t* mb, uint64_t ms, const uint8_t* wa, uint32_t wan,
                          const uint8_t* wb, uint64_t ws, uint32_t wl) {
    for (uint32_t x = 0; x < wl; ++x) { w.mt[x] = mph_rc_cat(ma, man, mb, (uint32_t)(ms + x)); w.wt[x] = mph_rc_cat(wa, wan, wb, (uint32_t)(ws + x)); }
  }
  static MPH_HD bool equals_slot(const Win& w, const uint8_t* sq, uint32_t wl) {
    for (uint32_t x = 0; x < wl; ++x)
      if (sq[x] != w.mt[x] || sq[wl + x] != w.wt[x]) return false;
    return true;
  }
  static MPH_HD void store(const Win& w, uint8_t* sq, uint32_t wl) {
    for (uint32_t x = 0; x < wl; ++x) { sq[x] = w.mt[x]; sq[wl + x] = w.wt[x]; }
  }
  static MPH_HD bool slot_less(const uint8_t* sy, const uint8_t* sx, uint32_t n) {  // sy < sx over n bytes
    for (uint32_t t = 0; t < n; ++t)
      if (sy[t] != sx[t]) return sy[t] < sx[t];
    return false;
  }
};

template <class Ops>
MPH_HD MphListEntry mph_rc_entry(const MphRecCtx& c, const MphSegment& sg, uint32_t i, uint32_t widx, uint32_t q, uint32_t* err) {
  MphListEntry en;
  const MphWinOut wo = c.win_out[widx];
  const uint32_t k = sg.k_first + i * sg.k_stride;
  const MphGeom g = mph_geom(sg, k);
  const MphKeyRef key = mph_rc_key(c, wo, widx, q);
  const uint64_t fd = mph_rc_frame_depth(c, wo);
  en.freq = key.count == 0 ? 0.0 : (double)key.count / (double)fd;
  en.s = mph_rc_seqs(c, sg, g, key);
  *err |= en.s.err;
  en.offset = g.spos == 0 ? g.s + 1u : g.s + 1u + g.gap;
  en.depth = wo.depth;
  const uint32_t va = mph_var_lb(c.vars, sg.var_lo, sg.var_hi, g.s);
  const uint32_t nv = mph_var_lb(c.vars, va, sg.var_hi, g.e) - va;
  uint32_t ns, nss;
  mph_rc_sites(c.vars, va, nv, &ns, &nss);
  en.var_ref = va;
  en.profile = key.h->profile;
  en.n_prof = key.h->n_prof;
  en.n_win = (uint8_t)nv;
  en.nsites = (uint8_t)ns;
  en.nsomsites = (uint8_t)nss;
  en.diff = 0;
  en.aligned = en.s.mt_len == en.s.wt_len && en.s.mt_len <= 64;
  if (en.s.mt == en.s.wt && en.s.mt_len == en.s.wt_len) {
    en.same = 1;
  } else if (en.aligned) {
    en.diff = Ops::diff_mask(en.s.mt, en.s.wt, en.s.mt_len);
    en.same = en.diff == 0;
  } else {
    en.same = 0;  // different lengths
  }
  return en;
}

// IDRecord::update's position filters (common.rs:399-478) over one source; returns kept somatic / germline counts
MPH_HD void mph_rc_keep(const MphVar* vars, const MphListEntry& e, bool is_self, bool forward, uint64_t offset, uint64_t wlen, uint32_t* keep,
                        uint32_t* nsom, uint32_t* ngerm) {
  uint32_t m = 0, a = 0, b = 0;
  const uint64_t eo = e.offset;
  for (uint32_t cidx = 0; cidx < e.n_prof && cidx < 32; ++cidx) {
    const uint32_t code = (uint32_t)((e.profile >> (2 * cidx)) & 3);
    if (!code) continue;
    const uint64_t pv = (uint64_t)vars[e.var_ref + cidx].pos + 1;
    bool kp;
    if (code == 2) {
      if (is_self) kp = forward ? (eo + offset <= pv) : (eo + wlen - offset >= pv);
      else kp = forward ? (eo + offset >= pv) : (eo + wlen - 3 - offset <= pv);
    } else {
      if (is_self) kp = eo + offset <= pv;
      else kp = eo >= pv - offset;  // u64 arithmetic as in the reference: wraps when pv < offset
    }
    if (kp) { m |= 1u << cidx; if (code == 2) ++a; else ++b; }
  }
  *keep = m;
  *nsom = a;
  *ngerm = b;
}

// Junction merge of a device-class transcript (:1505-1908): `cur` = first window of segment sj, `prv` = last window of
// the previous segment sp. Two modes: count (recs == nullptr) returns an upper bound of the records (no de-duplication),
// fill writes the de-duplicated records to recs / aux / seq (slot x owns seq[x * MPH_RC_SEQ_SLOT ..)) with their ranks
// in output_map order and returns their number. `cap` bounds the fill.
template <class Ops>
MPH_HD uint32_t mph_rc_merge_t(const MphRecCtx& c, const MphSegment& sp, const MphSegment& sj, uint32_t window_len, MphRec* recs, MphRecSrc* aux,
                             uint8_t* seq, uint32_t aux_base, uint32_t seq_base, uint32_t cap, uint32_t* err) {
  const bool fwd = (sj.flags & MPH_SF_REVERSE) == 0;
  const uint32_t w_cur = sj.win_base, i_prv = sp.n_win - 1, w_prv = sp.win_base + i_prv;
  const uint32_t n_cur = mph_rc_nkeys(c.win_out[w_cur]), n_prv = mph_rc_nkeys(c.win_out[w_prv]);
  // first_hap_vec / sec_hap_vec (:1511-1516): forward = (current, previous exon), reverse = (previous exon, current)
  const uint32_t n_first = fwd ? n_cur : n_prv, n_sec = fwd ? n_prv : n_cur;
  const uint64_t wl = window_len;
  const double eps = 2.220446049250313e-16;
  uint32_t n_out = 0;
  // the two lists are small (haplotype 0 plus the few variant haplotypes of a window): build their entries once
  enum { LIST_CACHE = 6 };
  MphListEntry first_c[LIST_CACHE], sec_c[LIST_CACHE];
  for (uint32_t a = 0; a < n_first && a < LIST_CACHE; ++a) first_c[a] = fwd ? mph_rc_entry<Ops>(c, sj, 0, w_cur, a, err) : mph_rc_entry<Ops>(c, sp, i_prv, w_prv, a, err);
  for (uint32_t b = 0; b < n_sec && b < LIST_CACHE; ++b) sec_c[b] = fwd ? mph_rc_entry<Ops>(c, sp, i_prv, w_prv, b, err) : mph_rc_entry<Ops>(c, sj, 0, w_cur, b, err);
  for (uint32_t a = 0; a < n_first; ++a) {
    const MphListEntry record = a < LIST_CACHE ? first_c[a] : (fwd ? mph_rc_entry<Ops>(c, sj, 0, w_cur, a, err) : mph_rc_entry<Ops>(c, sp, i_prv, w_prv, a, err));
    const bool rec_same = record.same != 0;
    for (uint32_t b = 0; b < n_sec; ++b) {
      const MphListEntry prev = b < LIST_CACHE ? sec_c[b] : (fwd ? mph_rc_entry<Ops>(c, sp, i_prv, w_prv, b, err) : mph_rc_entry<Ops>(c, sj, 0, w_cur, b, err));
      const bool prev_same = prev.same != 0;
      if (rec_same && prev_same) continue;  // every window of mt + mt equals wt + wt: nothing is written (:1795-1810)
      const uint32_t n_mts = rec_same ? 1u : (prev_same ? 1u : 3u);
      const double out_freq = fabs(record.freq - prev.freq) < eps ? record.freq : record.freq * prev.freq;
      // new_wt = prev.wt + record.wt
      const uint8_t* wa = prev.s.wt; const uint32_t wan = prev.s.wt_len; const uint8_t* wb = record.s.wt; const uint64_t wn = (uint64_t)wan + record.s.wt_len;
      // when neither side changes length, new_mt and new_wt are aligned and differ exactly where the chosen sides differ
      const bool masks = record.aligned && prev.aligned && wn <= 64;
      for (uint32_t m = 0; m < n_mts; ++m) {
        // new_mt_sequences (:1541-1556): wt != mt: [prev.wt + mt, prev.mt + wt, prev.mt + mt]; else [prev.mt + mt]
        const uint8_t *ma, *mb; uint32_t man, mbn;
        bool prev_mt, rec_mt;
        if (rec_same) { prev_mt = true; rec_mt = true; }
        else if (m == 0) { prev_mt = false; rec_mt = true; }
        else if (m == 1) { prev_mt = true; rec_mt = false; }
        else { prev_mt = true; rec_mt = true; }
        ma = prev_mt ? prev.s.mt : prev.s.wt; man = prev_mt ? prev.s.mt_len : prev.s.wt_len;
        mb = rec_mt ? record.s.mt : record.s.wt; mbn = rec_mt ? record.s.mt_len : record.s.wt_len;
        const uint64_t mn = (uint64_t)man + mbn;
        const uint64_t dmask = masks ? ((prev_mt ? prev.diff : 0) | ((rec_mt ? record.diff : 0) << wan)) : 0;
        if (masks && dmask == 0) continue;
        uint64_t splice_offset = 3, end_offset = 3;  // frameshift 0, exon_rest >= 3 and not the exon's last window in this class
        if (mn < 2 * wl) { if (fwd) splice_offset = 0; else end_offset = 0; }
        uint32_t guard = 0;
        while (splice_offset + wl <= mn - end_offset) {  // u64: wraps like the reference's usize when mn < end_offset
          if (++guard > 4096) { *err |= MPH_E_SLICE; break; }
          // window [ms, ms + wl) of new_mt and [ws, ws + wl) of new_wt
          uint64_t ms, ws = 0;
          bool have_wt = splice_offset + wl <= wn;
          if (fwd) { ms = splice_offset; ws = splice_offset; if (ms + wl > mn) { *err |= MPH_E_SLICE; break; } }
          else {
            if (mn < end_offset + wl) { *err |= MPH_E_SLICE; break; }
            ms = mn - end_offset - wl;
            if (have_wt) { if (wn < end_offset + wl) { *err |= MPH_E_SLICE; break; } ws = wn - end_offset - wl; }
          }
          bool equal = have_wt;
          if (masks && have_wt) {
            equal = ((dmask >> ms) & ((wl >= 64 ? ~(uint64_t)0 : (((uint64_t)1 << wl) - 1)))) == 0;
          } else {
            equal = equal && Ops::window_equal(ma, man, mb, ms, wa, wan, wb, ws, (uint32_t)wl);
          }
          if (equal || !have_wt) {  // non mutated site, or no wild type at frameshift 0 (:1795-1810)
            if (fwd) splice_offset += 3; else end_offset += 3;
            continue;
          }
          const uint64_t out_offset = fwd ? splice_offset : end_offset;
          if (!recs) {
            ++n_out;
          } else {
            // key (out_offset, mt, wt): look for the slot (:1877-1901); a repeat replaces the record and folds the old frequency in (add_freq)
            typename Ops::Win win;
            Ops::load(win, ma, man, mb, ms, wa, wan, wb, ws, (uint32_t)wl);
            uint32_t slot = 0;
            for (; slot < n_out; ++slot) {
              if (recs[slot].aux != (uint32_t)out_offset) continue;  // aux holds the key's offset until the final pass
              if (Ops::equals_slot(win, seq + seq_base + (size_t)slot * MPH_RC_SEQ_SLOT, (uint32_t)wl)) break;
            }
            double old_freq = 0.0;
            if (slot == n_out) {
              if (n_out >= cap) { *err |= MPH_E_REC_OVERFLOW; return n_out; }
              ++n_out;
              Ops::store(win, seq + seq_base + (size_t)slot * MPH_RC_SEQ_SLOT, (uint32_t)wl);
              Ops::sync();
            } else {
              old_freq = recs[slot].freq;
            }
            // IDRecord::update (common.rs:376-526): forward = prev.update(record), reverse = record.update(prev)
            const MphListEntry& self = fwd ? prev : record;
            const MphListEntry& other = fwd ? record : prev;
            uint32_t ka, kb, sa, sb, ga, gb;
            mph_rc_keep(c.vars, self, true, fwd, out_offset, wl, &ka, &sa, &ga);
            mph_rc_keep(c.vars, other, false, fwd, out_offset, wl, &kb, &sb, &gb);
            MphRec r;
            r.id64 = out_offset;  // the id is hashed afterwards, one thread per record (mph_rc_merged_id): sha1 needs the key's offset
            r.tx = sj.tx;
            r.offset = (uint32_t)(fwd ? self.offset + out_offset : other.offset + wl + 3 - out_offset);
            r.depth = (other.depth == 0 || self.depth == 0) ? 0u : (other.depth + self.depth) / 2u;
            uint32_t nsom = sa + sb, nvar = nsom + ga + gb;
            // add_freq (common.rs:528-568), also applied to a fresh slot with 0.0
            const uint32_t new_nvar = nvar == 0 ? 0u : (old_freq > 0.0 ? nvar - 1 : nvar);
            nsom = new_nvar < nsom ? nsom - 1 : nsom;
            r.freq = out_freq > 0.5 ? out_freq : out_freq + old_freq;
            r.nvar = (uint8_t)new_nvar;
            r.nsomatic = (uint8_t)nsom;
            r.nsites = (uint8_t)(self.nsites + other.nsites);
            r.nsomsites = (uint8_t)(self.nsomsites + other.nsomsites);
            r.seq_off = seq_base + slot * MPH_RC_SEQ_SLOT;
            r.var_ref = self.var_ref; r.keep = ka; r.profile = self.profile; r.n_prof = self.n_prof; r.n_win = self.n_win;
            r.flags = (uint8_t)(MPH_RC_MERGED | MPH_RC_HAS_MT | MPH_RC_HAS_WT | (fwd ? 0 : MPH_RC_REVERSE));
            r.rank = 0;
            r.neo_len = r.mt_len = r.norm_len = r.wt_len = (uint8_t)wl;
            r.aux = (uint32_t)out_offset;
            if (Ops::leader()) recs[slot] = r;
            MphRecSrc x;
            x.profile = other.profile; x.var_ref = other.var_ref; x.keep = kb; x.n_prof = other.n_prof; x.n_win = other.n_win;
            for (int z = 0; z < 6; ++z) x.pad[z] = 0;
            if (Ops::leader()) aux[slot] = x;
            Ops::sync();
          }
          if (fwd) splice_offset += 3; else end_offset += 3;
        }
      }
    }
  }
  if (recs) {
    // ranks in output_map order: (out_offset, mt bytes, wt bytes) (:1518-1521); then aux takes its final meaning
    if (n_out > MPH_RC_JUNCTION_RECS) { *err |= MPH_E_RECS_PER_LIST; return 0; }
    for (uint32_t x = 0; x < n_out; ++x) {
      uint32_t rank = 0;
      const uint8_t* sx = seq + seq_base + (size_t)x * MPH_RC_SEQ_SLOT;
      for (uint32_t y = 0; y < n_out; ++y) {
        if (y == x) continue;
        const uint8_t* sy = seq + seq_base + (size_t)y * MPH_RC_SEQ_SLOT;
        bool less;  // y < x ?
        if (recs[y].aux != recs[x].aux) less = recs[y].aux < recs[x].aux;
        else less = Ops::slot_less(sy, sx, (uint32_t)(2 * wl));
        if (less) ++rank;
      }
      if (Ops::leader()) recs[x].rank = rank;
    }
    Ops::sync();
    if (Ops::leader())
      for (uint32_t x = 0; x < n_out; ++x) recs[x].aux = aux_base + x;
    Ops::sync();
  }
  return n_out;
}

MPH_HD uint32_t mph_rc_merge(const MphRecCtx& c, const MphSegment& sp, const MphSegment& sj, uint32_t window_len, MphRec* recs, MphRecSrc* aux,
                             uint8_t* seq, uint32_t aux_base, uint32_t seq_base, uint32_t cap, uint32_t* err) {
  return mph_rc_merge_t<MphSerialOps>(c, sp, sj, window_len, recs, aux, seq, aux_base, seq_base, cap, err);
}

// record id of a merged record (common.rs:385-391: sha1 over the mutant window, the transcript id and the key's offset,
// which mph_rc_merge left in id64); `mt` = the record's mutant window in the merge arena
MPH_HD void mph_rc_merged_id(const MphRecCtx& c, MphRec* r, const uint8_t* mt, uint32_t window_len) {
  const uint32_t t0 = c.tx_id_off[r->tx], tlen = c.tx_id_off[r->tx + 1] - t0;
  r->id64 = mph_record_id64(mt, window_len, c.tx_id_bytes + t0, tlen, (uint32_t)r->id64);
}

// ================================================================================================ `normal` mode
// Record emission of the healthy-peptidome pass (reference src/normal_microphasing.rs; line numbers below refer to that
// file) for device-class transcripts. Every window of a non-short exon writes a record per haplotype that does not start
// (forward) / end (reverse) with a stop codon (:493-507,629-644); a window whose haplotypes all stop ends the transcript
// (:1128-1131: the main-ORF entry is removed unconditionally). A junction merge (:1145-1250) slides over prev + cur of
// every pair of listed haplotypes and writes every window, not only the mutated ones.
enum {
  MPH_RC_NORMAL = 16,  // record of the normal mode: 0-based positions, sites limited to the visited variants, 32-bit counts of merged records in `keep`
  MPH_RC_REFSEQ = 32,  // the sequence is the reference window itself: seq_off indexes the batch's reference arena (nothing is shipped)
};

typedef struct {
  const uint32_t* win_depth;          // per window: depth | (plain window begins / ends with a stop codon) << 31
  const unsigned long long* win_id;   // per window: id of the reference window
} MphNrmCtx;

MPH_HD uint32_t mph_nrc_nkeys(const MphRecCtx& c, uint32_t widx, uint32_t nv) {
  if (nv == 0) return 1;
  return mph_rc_nkeys(c.win_out[widx]);
}

// key q of a window; for a window without variants the single reference haplotype is described by `plain`
MPH_HD MphKeyRef mph_nrc_key(const MphRecCtx& c, const MphNrmCtx& n, const MphGeom& g, uint32_t widx, uint32_t nv, uint32_t q, MphHap* plain) {
  if (nv == 0) {
    const uint32_t wd = n.win_depth[widx];
    plain->flags = (wd >> 31) ? MPH_NF_STOP : 0u;
    plain->seq_len = (uint16_t)(g.e - g.s);
    plain->germ_len = 0; plain->n_var = 0; plain->n_som = 0; plain->n_prof = 0; plain->brk = 0; plain->seq_off = 0xFFFFFFFFu; plain->profile = 0; plain->id64 = 0;
    MphKeyRef k;
    k.hap = 0; k.count = wd & 0x7FFFFFFFu; k.h = plain;
    return k;
  }
  return mph_rc_key(c, c.win_out[widx], widx, q);
}

// number of haplotypes of the window that are written / listed (n_res of print_haplotypes, :629-644); MPH_E_* bits in *err
MPH_HD uint32_t mph_nrc_window_count(const MphRecCtx& c, const MphNrmCtx& n, const MphSegment& sg, uint32_t i, uint32_t widx, uint32_t* seq_bytes,
                                     uint32_t* err) {
  const uint32_t k = sg.k_first + i * sg.k_stride;
  const MphGeom g = mph_geom(sg, k);
  const uint32_t va = mph_var_lb(c.vars, sg.var_lo, sg.var_hi, g.s);
  const uint32_t nv = mph_var_lb(c.vars, va, sg.var_hi, g.e) - va;
  const uint32_t nk = mph_nrc_nkeys(c, widx, nv);
  uint32_t cnt = 0, bytes = 0;
  for (uint32_t q = 0; q < nk; ++q) {
    MphHap plain;
    const MphKeyRef key = mph_nrc_key(c, n, g, widx, nv, q, &plain);
    if (key.h->flags & MPH_NF_REFRANGE) *err |= MPH_E_REF_RANGE;
    if ((key.h->flags & MPH_NF_STOP) && g.spos != 2) continue;
    if (key.h->flags & MPH_NF_OVERFLOW) *err |= MPH_E_SEQ_SLOT;
    ++cnt;
    if (key.hap != 0) bytes += key.h->seq_len;
  }
  *seq_bytes = bytes;
  return cnt;
}

// sequence of one listed haplotype (`seq` of print_haplotypes): the reference window or the assembled bytes
MPH_HD void mph_nrc_seq(const MphRecCtx& c, const MphSegment& sg, const MphGeom& g, const MphKeyRef& key, const uint8_t** p, uint32_t* len, uint32_t* err) {
  if (key.hap == 0) {
    *p = c.ref + sg.ref_off + (g.s - sg.ref_pos0);
    *len = g.e - g.s;
    if (g.s < sg.ref_pos0 || (uint64_t)g.e - sg.ref_pos0 > sg.ref_len) { *err |= MPH_E_REF_RANGE; *len = 0; }
    return;
  }
  if (!(key.h->flags & MPH_NF_SEQ)) { *err |= MPH_E_INTERNAL; *p = c.ref; *len = 0; return; }
  *p = c.seq + key.h->seq_off;
  *len = key.h->seq_len < c.seq_cap ? key.h->seq_len : c.seq_cap;
}

// writes the window's records; returns their number (= mph_nrc_window_count)
MPH_HD uint32_t mph_nrc_window_emit(const MphRecCtx& c, const MphNrmCtx& n, const MphSegment& sg, uint32_t i, uint32_t widx, MphRec* recs,
                                    uint8_t* seq_arena, uint32_t seq_base, uint32_t* err) {
  const uint32_t k = sg.k_first + i * sg.k_stride;
  const MphGeom g = mph_geom(sg, k);
  const bool rev = (sg.flags & MPH_SF_REVERSE) != 0;
  const uint32_t va = mph_var_lb(c.vars, sg.var_lo, sg.var_hi, g.s);
  const uint32_t nv = mph_var_lb(c.vars, va, sg.var_hi, g.e) - va;
  const uint32_t nk = mph_nrc_nkeys(c, widx, nv);
  const uint32_t depth = n.win_depth[widx] & 0x7FFFFFFFu;
  uint32_t cnt = 0, pos = seq_base;
  for (uint32_t q = 0; q < nk; ++q) {
    MphHap plain;
    const MphKeyRef key = mph_nrc_key(c, n, g, widx, nv, q, &plain);
    const MphHap& h = *key.h;
    if ((h.flags & MPH_NF_STOP) && g.spos != 2) continue;
    const uint8_t* sp;
    uint32_t sl;
    mph_nrc_seq(c, sg, g, key, &sp, &sl, err);
    const bool insertion = (h.flags & MPH_NF_INSERTION) != 0;
    const uint32_t twl = sl < sg.ewl ? sl : sg.ewl;
    // peptide_sequence column (:485-492) and FASTA line (:629-644): both start at `a`
    uint32_t a = 0, neo_b, mt_b;
    if (g.spos == 1) { a = g.gap; neo_b = mt_b = sl; if (a > sl) { *err |= MPH_E_SLICE; a = sl; } }
    else if (g.spos == 0) { neo_b = insertion ? sl : twl; mt_b = sg.ewl; if (sg.ewl > sl) { *err |= MPH_E_SLICE; mt_b = sl; } }
    else { neo_b = sl; mt_b = 0; }
    const uint32_t stored = (neo_b > mt_b ? neo_b : mt_b) - a;
    if (stored > 255) { *err |= MPH_E_SEQ_SLOT; }
    MphRec r;
    r.id64 = key.hap == 0 ? (uint64_t)n.win_id[widx] : h.id64;
    if (key.hap != 0 && !(h.flags & MPH_NF_ID)) *err |= MPH_E_INTERNAL;
    r.freq = (double)key.count / (double)depth;  // NaN without observations (:397)
    r.tx = sg.tx;
    r.offset = g.s;
    r.depth = depth;
    r.var_ref = va;
    r.keep = 0xFFFFFFFFu;
    r.profile = h.profile;
    r.n_prof = nv ? h.n_prof : 0;
    r.n_win = (uint8_t)nv;
    r.nvar = h.n_var;
    r.nsomatic = h.n_som;
    {
      const uint32_t lim = nv < r.n_prof ? nv : r.n_prof;  // sites are counted while the walk produced a profile entry (:509-560)
      uint32_t ns = 0, nss = 0;
      mph_rc_sites(c.vars, va, lim, &ns, &nss);
      r.nsites = (uint8_t)ns;
      r.nsomsites = (uint8_t)nss;
    }
    r.flags = (uint8_t)(MPH_RC_NORMAL | (g.spos != 2 ? MPH_RC_HAS_MT : 0) | (rev ? MPH_RC_REVERSE : 0));
    r.rank = 0;
    r.neo_len = (uint8_t)(neo_b - a);
    r.mt_len = (uint8_t)(mt_b > a ? mt_b - a : 0u);
    r.norm_len = r.wt_len = 0;
    r.aux = 0xFFFFFFFFu;
    if (key.hap == 0) {
      r.flags |= MPH_RC_REFSEQ;
      r.seq_off = sg.ref_off + (g.s - sg.ref_pos0) + a;
    } else {
      r.seq_off = pos;
      for (uint32_t t = 0; t < stored && stored <= 255; ++t) seq_arena[pos + t] = sp[a + t];
      pos += stored <= 255 ? stored : 0u;
    }
    recs[cnt++] = r;
  }
  return cnt;
}

// all haplotypes of the window stop (n_res == 0): the transcript ends here
MPH_HD bool mph_nrc_window_stops(const MphRecCtx& c, const MphNrmCtx& n, const MphSegment& sg, uint32_t i, uint32_t widx) {
  uint32_t bytes = 0, err = 0;
  return mph_nrc_window_count(c, n, sg, i, widx, &bytes, &err) == 0;
}

// One listed haplotype for the merge (HaplotypeSeq :182-186): its full sequence and the counts of its record.
typedef struct {
  const uint8_t* seq;
  uint32_t len;
  double freq;
  uint32_t offset, depth, var_ref;
  uint64_t profile;
  uint32_t nvar, nsomatic;
  uint8_t n_prof, n_win, nsites, nsomsites;
} MphNrmEntry;

// the a-th listed haplotype of a window (haplotypes that stop are not listed); returns false past the end
MPH_HD bool mph_nrc_entry(const MphRecCtx& c, const MphNrmCtx& n, const MphSegment& sg, uint32_t i, uint32_t widx, uint32_t a, MphNrmEntry* en,
                          MphHap* plain, uint32_t* err) {
  const uint32_t k = sg.k_first + i * sg.k_stride;
  const MphGeom g = mph_geom(sg, k);
  const uint32_t va = mph_var_lb(c.vars, sg.var_lo, sg.var_hi, g.s);
  const uint32_t nv = mph_var_lb(c.vars, va, sg.var_hi, g.e) - va;
  const uint32_t nk = mph_nrc_nkeys(c, widx, nv);
  const uint32_t depth = n.win_depth[widx] & 0x7FFFFFFFu;
  uint32_t seen = 0;
  for (uint32_t q = 0; q < nk; ++q) {
    const MphKeyRef key = mph_nrc_key(c, n, g, widx, nv, q, plain);
    if ((key.h->flags & MPH_NF_STOP) && g.spos != 2) continue;
    if (seen++ != a) continue;
    mph_nrc_seq(c, sg, g, key, &en->seq, &en->len, err);
    en->freq = (double)key.count / (double)depth;
    en->offset = g.s;
    en->depth = depth;
    en->var_ref = va;
    en->profile = key.h->profile;
    en->n_prof = nv ? key.h->n_prof : 0;
    en->n_win = (uint8_t)nv;
    en->nvar = key.h->n_var;
    en->nsomatic = key.h->n_som;
    const uint32_t lim = nv < en->n_prof ? nv : en->n_prof;
    uint32_t ns = 0, nss = 0;
    mph_rc_sites(c.vars, va, lim, &ns, &nss);
    en->nsites = (uint8_t)ns;
    en->nsomsites = (uint8_t)nss;
    return true;
  }
  return false;
}

// Junction merge of the normal mode (:1145-1250) for a device-class transcript: `cur` = first window of sj, `prv` = last window
// of sp. recs == nullptr counts (upper bound, no de-duplication); otherwise fills like mph_rc_merge_t. Only the window's
// bytes are the key here ((splice_offset, out_seq), :1216), and every window is written.
template <class Ops>
MPH_HD uint32_t mph_nrc_merge_t(const MphRecCtx& c, const MphNrmCtx& n, const MphSegment& sp, const MphSegment& sj, uint32_t window_len, MphRec* recs,
                                MphRecSrc* aux, uint8_t* seq, uint32_t aux_base, uint32_t seq_base, uint32_t cap, uint32_t* err) {
  const bool fwd = (sj.flags & MPH_SF_REVERSE) == 0;
  const uint32_t w_cur = sj.win_base, i_prv = sp.n_win - 1, w_prv = sp.win_base + i_prv;
  const uint64_t wl = window_len;
  uint32_t n_out = 0;
  for (uint32_t a = 0;; ++a) {
    MphNrmEntry record;  // from first_hap_vec: forward = current window, reverse = previous exon's last window
    MphHap plain_a;
    if (!(fwd ? mph_nrc_entry(c, n, sj, 0, w_cur, a, &record, &plain_a, err) : mph_nrc_entry(c, n, sp, i_prv, w_prv, a, &record, &plain_a, err))) break;
    for (uint32_t b = 0;; ++b) {
      MphNrmEntry prev;
      MphHap plain_b;
      if (!(fwd ? mph_nrc_entry(c, n, sp, i_prv, w_prv, b, &prev, &plain_b, err) : mph_nrc_entry(c, n, sj, 0, w_cur, b, &prev, &plain_b, err))) break;
      const uint64_t jn = (uint64_t)prev.len + record.len;  // joined = prev.sequence + record.sequence
      uint64_t splice_offset = 3, end_offset = 3;           // exon_rest >= 3 and not the exon's last window in this class
      if (jn < 2 * wl) { if (fwd) splice_offset = 0; else end_offset = 0; }
      uint32_t guard = 0;
      while (splice_offset + wl <= jn - end_offset) {  // u64: wraps like the reference's usize
        if (++guard > 4096 || splice_offset + wl > jn) { *err |= MPH_E_SLICE; break; }
        if (!recs) { ++n_out; splice_offset += 3; continue; }
        typename Ops::Win win;
        Ops::load(win, prev.seq, prev.len, record.seq, splice_offset, prev.seq, prev.len, record.seq, splice_offset, (uint32_t)wl);
        uint32_t slot = 0;
        for (; slot < n_out; ++slot) {
          if (recs[slot].aux != (uint32_t)splice_offset) continue;  // aux holds the key's offset until the final pass
          if (Ops::equals_slot(win, seq + seq_base + (size_t)slot * MPH_RC_SEQ_SLOT, (uint32_t)wl)) break;
        }
        double old_freq = 0.0;
        if (slot == n_out) {
          if (n_out >= cap) { *err |= MPH_E_REC_OVERFLOW; return n_out; }
          ++n_out;
          Ops::store(win, seq + seq_base + (size_t)slot * MPH_RC_SEQ_SLOT, (uint32_t)wl);
          Ops::sync();
        } else {
          old_freq = recs[slot].freq;
        }
        // IDRecord::update (:105-146): self = prev_record, rec = record; then add_freq (:148-179) with the slot's old frequency
        MphRec r;
        r.id64 = splice_offset;  // hashed afterwards (mph_rc_merged_id)
        r.tx = sj.tx;
        r.offset = (uint32_t)(splice_offset + prev.offset);
        r.depth = prev.depth;
        uint32_t nvar = prev.nvar + record.nvar, nsom = prev.nsomatic + record.nsomatic;
        const uint32_t new_nvar = old_freq > 0.0 ? nvar - 1u : nvar;  // u32 arithmetic wraps like the release build
        nsom = new_nvar < nsom ? nsom - 1u : nsom;
        r.freq = prev.freq * record.freq + old_freq;
        r.nvar = (uint8_t)new_nvar;
        r.nsomatic = (uint8_t)nsom;
        r.keep = new_nvar;  // the 32-bit counts of a merged normal-mode record: nvar here, nsomatic in the second source's `keep`
        r.nsites = (uint8_t)(prev.nsites + record.nsites);
        r.nsomsites = (uint8_t)(prev.nsomsites + record.nsomsites);
        r.seq_off = seq_base + slot * MPH_RC_SEQ_SLOT;
        r.var_ref = prev.var_ref; r.profile = prev.profile; r.n_prof = prev.n_prof; r.n_win = prev.n_win;
        r.flags = (uint8_t)(MPH_RC_NORMAL | MPH_RC_MERGED | MPH_RC_HAS_MT | (fwd ? 0 : MPH_RC_REVERSE));
        r.rank = 0;
        r.neo_len = r.mt_len = (uint8_t)wl;
        r.norm_len = r.wt_len = 0;
        r.aux = (uint32_t)splice_offset;
        if (Ops::leader()) recs[slot] = r;
        MphRecSrc x;
        x.profile = record.profile; x.var_ref = record.var_ref; x.keep = nsom; x.n_prof = record.n_prof; x.n_win = record.n_win;
        for (int z = 0; z < 6; ++z) x.pad[z] = 0;
        if (Ops::leader()) aux[slot] = x;
        Ops::sync();
        splice_offset += 3;
      }
    }
  }
  if (recs) {
    // ranks in output_map order: (splice_offset, out_seq) (:1216-1222); then aux takes its final meaning
    if (n_out > MPH_RC_JUNCTION_RECS) { *err |= MPH_E_RECS_PER_LIST; return 0; }
    for (uint32_t x = 0; x < n_out; ++x) {
      uint32_t rank = 0;
      const uint8_t* sx = seq + seq_base + (size_t)x * MPH_RC_SEQ_SLOT;
      for (uint32_t y = 0; y < n_out; ++y) {
        if (y == x) continue;
        const uint8_t* sy = seq + seq_base + (size_t)y * MPH_RC_SEQ_SLOT;
        bool less;
        if (recs[y].aux != recs[x].aux) less = recs[y].aux < recs[x].aux;
        else less = Ops::slot_less(sy, sx, (uint32_t)wl);
        if (less) ++rank;
      }
      if (Ops::leader()) recs[x].rank = rank;
    }
    Ops::sync();
    if (Ops::leader())
      for (uint32_t x = 0; x < n_out; ++x) recs[x].aux = aux_base + x;
    Ops::sync();
  }
  return n_out;
}
