// replay_core.h — serial replay of the ObservationMatrix for transcripts the closed form of
// phase_core.h does not cover (reference src/microphasing.rs; line numbers refer to that file):
//   * an observation survives from one exon into the next (cleanup_reads :259-278 keeps it), e.g. a
//     spliced read or an intron shorter than a read;
//   * the "stale column" of reverse-strand exons: at the last iteration `offset == old_offset`
//     (:1159) suppresses the removal of the variants at exon.start + window_len, which then stay in
//     the matrix — shifted through every later shrink_left — for the rest of the transcript.
// Both make the matrix state depend on the whole history of the transcript, so the replay runs the
// reference's own sequence of matrix operations (cleanup_reads, shrink_left, push_read,
// extend_right :220-343 in the order of the window loop :1119-1343) with one observation list per
// transcript. It emits, for every enumerated window, what the closed-form kernel emits (depth and
// the (haplotype, frame) histogram) plus the matrix's variant columns, which no longer equal the
// variants inside the window.
//
// Shared by the CUDA kernel k_replay (one warp per transcript, csrc/kernels/phase_kernels.cu) and the
// test-only CPU emulator. All functions are MPH_HD.
#pragma once
#include "phase_core.h"

#define MPH_RP_MAXCOLS 64
#define MPH_RP_KEYS 32

// One replay unit, 48 B: a run of consecutive exons of one transcript that no observation crosses the
// ends of. The matrix columns at its start do not depend on reads, so the packer computes them with a
// read-free pass over the transcript and the units of one transcript replay in parallel.
typedef struct {
  uint32_t seg_lo, seg_hi;    // its segments
  uint32_t read_lo, read_hi;  // the gene's reads
  uint32_t obs_off, obs_cap;  // slice of the observation scratch arrays
  uint32_t sl_va, sl_vb;      // start-loss variant range of the first exon (:1305-1316)
  uint32_t dq_off, dq_n;      // matrix columns when the unit starts (variant indices, oldest first) in the dq arena
  uint32_t last_vars;         // last_window_vars when the unit starts (:1024)
  uint32_t pad;
} MphReplayTx;

typedef struct MphReplayCtx {
  // inputs (same arrays as the closed-form kernels)
  const uint32_t* read_start; const uint32_t* read_end; const uint8_t* read_flags;
  const uint32_t* read_vlo; const uint8_t* read_nv; const uint32_t* read_vr;  // per read, expanded by K1 from the compact side table (read_vr = its entry)
  const uint32_t* vr_seq_off; const uint32_t* vr_cig_off; const uint16_t* vr_lseq; const uint16_t* vr_ncig;
  const uint8_t* bases; const uint32_t* cigars;
  const uint64_t* call_S; const uint64_t* call_B;
  const uint32_t* pairs; uint32_t n_pairs;  // (read, partner) interleaved, sorted by read
  const MphVar* vars; const MphSegment* segs; const uint32_t* seg_chunk0;
  const uint32_t* stopmap; const uint8_t* ref;
  const uint32_t* dq_init;  // arena of initial column lists
  uint32_t batch;           // somatic only: iterations that neither change the columns nor emit a window are folded into the next one that does
  uint32_t mode;            // 0 somatic, 1 normal (src/normal_microphasing.rs: every re-offered copy of a read is kept, no quality test)
  const uint8_t* tx_id_bytes; const uint32_t* tx_id_off;  // normal mode: record id of the reference window
  uint32_t* win_depth; unsigned long long* win_id;        // normal mode outputs
  uint32_t* o_last;         // normal mode, per gene read: index of its latest entry (entries are (read, haplotype, copies))
  // scratch: observation list
  uint32_t* o_read; uint64_t* o_hap; uint32_t* o_frame; uint8_t* o_flags;
  uint8_t* o_inmat;  // per gene read (obs_off + read - read_lo): the read is an observation right now
  // outputs
  MphWinOut* win_out; MphHist* hist; uint32_t* hist_win; uint32_t hist_cap;
  uint32_t key_cap = MPH_RP_KEYS;  // keys of the window table before a window is sorted in the arena instead (0 under MPH_FORCE_WIDE=2)
  MphHap* hap0; uint8_t* win_flag;
  uint32_t* win_voff;  // per window: offset of its column list in vlist (entry 0 = count), 0xFFFFFFFF = the window's own variants
  uint32_t* vlist; uint32_t vlist_cap;
  uint32_t* seg_err;   // per segment: 1 + iteration at which the reference panics (drain out of range, inverted range), 0 = none
  uint32_t* counters;  // CTR_* of phase_kernels.cuh
  unsigned long long* sum_depth;
} MphReplayCtx;

enum { MPH_RP_CTR_HIST = 0, MPH_RP_CTR_ERR = 3, MPH_RP_CTR_VLIST = 5 };

#ifdef __CUDA_ARCH__
#define MPH_RP_ADD(p, v) atomicAdd((p), (v))
#define MPH_RP_OR(p, v) atomicOr((p), (v))
#define MPH_RP_ADD64(p, v) atomicAdd((p), (unsigned long long)(v))
#else
static inline uint32_t mph_rp_add_host(uint32_t* p, uint32_t v) { const uint32_t o = *p; *p += v; return o; }
#define MPH_RP_ADD(p, v) mph_rp_add_host((p), (v))
#define MPH_RP_OR(p, v) (*(p) |= (v))
#define MPH_RP_ADD64(p, v) (*(p) += (unsigned long long)(v))
#endif

// supports_variant (:95-139) and bad_quality (:78-93) of one (read, variant) pair. Variants inside
// the alignment come from the K1 masks; a matrix column outside it (stale column) is evaluated here.
MPH_HD void mph_rp_eval(const MphReplayCtx& c, uint32_t r, uint32_t v, bool* sup, bool* bad, uint32_t* err) {
  const uint32_t vlo = c.read_vlo[r], nv = c.read_nv[r];
  if (v >= vlo && v - vlo < nv) {
    *sup = (c.call_S[r] >> (v - vlo)) & 1;
    *bad = (c.call_B[r] >> (v - vlo)) & 1;
    return;
  }
  const MphVar var = c.vars[v];
  const uint32_t start = c.read_start[r];
  *sup = false;
  *bad = false;
  if (start > var.pos) { *err |= MPH_E_REPLAY_PANIC; return; }  // "bug: read starts right of variant" (:160-167)
  // every read of a gene with replayed transcripts has an entry in the side table
  const uint32_t e = c.read_vr[r];
  const uint32_t l_seq = c.vr_lseq[e];
  const uint32_t soff = c.vr_seq_off[e];
  const uint32_t ncig = c.vr_ncig[e];
  const uint32_t* cig = c.cigars + c.vr_cig_off[e];
  if (var.kind == MPH_SNV) {
    const uint8_t* rec = c.bases + (size_t)soff;
    const uint32_t rel = var.pos - start;
    if (c.mode == 0 && rel < l_seq && mph_rec_low(rec, l_seq, rel)) { *bad = true; return; }
    uint32_t q;
    if (mph_read_pos(cig, ncig, l_seq, start, var.pos, &q) && q < l_seq) *sup = mph_rec_base4(rec, q) == var.alt4;
  } else {
    const uint32_t want = var.kind == MPH_INS ? 1u : 2u;
    for (uint32_t i = 0; i < ncig; ++i)
      if ((cig[i] & 15u) == want && (cig[i] >> 4) == var.len) { *sup = true; break; }
  }
}

// Observation::update_haplotype (:157-183) on packed state: frame = frame.0 | (frame.1 != 0) << 31, flags = bad_qual | start_loss << 1
MPH_HD void mph_rp_update(const MphReplayCtx& c, const MphReplayTx& t, uint32_t r, uint32_t i, uint32_t v, uint64_t* hap, uint32_t* frame,
                          uint8_t* flags, uint32_t* err) {
  const MphVar& var = c.vars[v];
  const uint32_t fs = (var.flags & MPH_VF_FS_MASK) >> MPH_VF_FS_SHIFT;
  bool sup, bad;
  mph_rp_eval(c, r, v, &sup, &bad, err);
  if (c.mode == 1) {  // normal_microphasing.rs:195-215: only the supported bit
    if (sup) *hap |= (uint64_t)1 << (i & 63u);
    return;
  }
  if (fs > 0 && var.pos != 0) *frame |= 0x80000000u;
  if (sup) {
    if (v >= t.sl_va && v < t.sl_vb) *flags |= 2;
    *hap |= (uint64_t)1 << (i & 63u);
    *frame = (*frame & 0x80000000u) | (((*frame & 0x7FFFFFFFu) + fs) & 0x7FFFFFFFu);
  }
  if (bad || (*flags & 3)) {
    *hap = 0;
    *flags |= 1;
  }
}

MPH_HD uint32_t mph_rp_partner(const MphReplayCtx& c, uint32_t r) {
  uint32_t lo = 0, hi = c.n_pairs;
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    if (c.pairs[2 * mid] < r) lo = mid + 1;
    else hi = mid;
  }
  return (lo < c.n_pairs && c.pairs[2 * lo] == r) ? c.pairs[2 * lo + 1] : 0xFFFFFFFFu;
}

// BTreeMap order of the keys (:383,434): haplotype, frame.0, frame.1 != 0
MPH_HD bool mph_rp_hist_less(const MphHist& a, const MphHist& b) {
  if (a.hap != b.hap) return a.hap < b.hap;
  const uint32_t fa = a.frame & 0x7FFFFFFFu, fb = b.frame & 0x7FFFFFFFu;
  if (fa != fb) return fa < fb;
  return (a.frame >> 31) < (b.frame >> 31);
}

// in-place heapsort of h[0, n) in that order (serial, no scratch)
MPH_HD void mph_rp_heapsort(MphHist* h, uint32_t n) {
  auto sift = [&](uint32_t root, uint32_t end) {
    for (;;) {
      uint32_t child = 2 * root + 1;
      if (child >= end) return;
      if (child + 1 < end && mph_rp_hist_less(h[child], h[child + 1])) ++child;
      if (!mph_rp_hist_less(h[root], h[child])) return;
      const MphHist tmp = h[root]; h[root] = h[child]; h[child] = tmp;
      root = child;
    }
  };
  for (uint32_t r = n / 2; r-- > 0;) sift(r, n);
  for (uint32_t end = n; end > 1; --end) {
    const MphHist tmp = h[0]; h[0] = h[end - 1]; h[end - 1] = tmp;
    sift(0, end - 1);
  }
}

// histogram + outputs of one enumerated window (the part of print_haplotypes :383-411 that reads the matrix)
MPH_HD void mph_rp_emit(const MphReplayCtx& c, const MphReplayTx& t, const MphSegment& sg, uint32_t si, uint32_t i, uint32_t k, const MphGeom& g,
                        uint32_t n_obs, const uint32_t* dq, uint32_t ncols, uint32_t* err) {
  const uint32_t widx = sg.win_base + i;
  MphHist table[MPH_RP_KEYS];
  uint32_t n_keys = 0, c0 = 0;
  const bool normal = c.mode == 1;
  uint32_t depth = normal ? 0u : n_obs;
  bool spill = false;    // more keys than the table holds
  for (uint32_t o = 0; o < n_obs; ++o) {
    if (c.o_flags[t.obs_off + o] & 1) continue;
    const uint64_t hap = c.o_hap[t.obs_off + o];
    const uint32_t wgt = normal ? c.o_frame[t.obs_off + o] : 1u;  // normal mode: copies of the read with this haplotype
    const uint32_t fr = normal ? 0u : c.o_frame[t.obs_off + o];
    if (normal) depth += wgt;
    if (hap == 0 && fr == 0) { c0 += wgt; continue; }
    if (spill) continue;
    uint32_t x = 0;
    for (; x < n_keys; ++x)
      if (table[x].hap == hap && table[x].frame == fr) break;
    if (x == n_keys) {
      if (n_keys == c.key_cap) { spill = true; continue; }
      table[x].hap = hap; table[x].frame = fr; table[x].count = 0;
      ++n_keys;
    }
    table[x].count += wgt;
  }
  const uint32_t code = ((c.seg_chunk0[si] + (i >> 5)) << 5) | (i & 31u);
  for (uint32_t a = 1; a < n_keys; ++a) {  // BTreeMap order (:383,434): haplotype, frame.0, frame.1 != 0
    const MphHist key = table[a];
    uint32_t b = a;
    while (b > 0 && mph_rp_hist_less(key, table[b - 1])) {
      table[b] = table[b - 1];
      --b;
    }
    table[b] = key;
  }
  MphWinOut wo;
  wo.depth = depth;
  wo.c0 = c0;
  wo.n_extra = n_keys;
  wo.extra_off = 0;
  if (spill) {
    // more keys than the table holds (the block tier's serial statement): the window's distinct keys, counted without
    // scratch (a key is listed at its first observation, with the weights of all its observations), are sorted in the key arena
    auto counted = [&](uint32_t o) {
      return !(c.o_flags[t.obs_off + o] & 1) && (c.o_hap[t.obs_off + o] != 0 || (!normal && c.o_frame[t.obs_off + o] != 0));
    };
    auto same = [&](uint32_t o, uint32_t q) {
      return c.o_hap[t.obs_off + o] == c.o_hap[t.obs_off + q] && (normal || c.o_frame[t.obs_off + o] == c.o_frame[t.obs_off + q]);
    };
    auto first = [&](uint32_t o) {
      for (uint32_t q = 0; q < o; ++q)
        if (counted(q) && same(o, q)) return false;
      return true;
    };
    uint32_t n_fold = 0;
    for (uint32_t o = 0; o < n_obs; ++o) n_fold += (counted(o) && first(o)) ? 1u : 0u;
    wo.n_extra = 0;
    if (n_fold > MPH_BLOCK_KEYS) {
      *err |= MPH_E_KEYS_PER_WINDOW;
    } else {
      const uint32_t off = MPH_RP_ADD(&c.counters[MPH_RP_CTR_HIST], n_fold);
      if (off + n_fold <= c.hist_cap) {
        MphHist* h = c.hist + off;
        uint32_t y = 0;
        for (uint32_t o = 0; o < n_obs; ++o) {
          if (!counted(o) || !first(o)) continue;
          MphHist e;
          e.hap = c.o_hap[t.obs_off + o];
          e.frame = normal ? 0u : c.o_frame[t.obs_off + o];
          e.count = 0;
          for (uint32_t q = o; q < n_obs; ++q)
            if (counted(q) && same(o, q)) e.count += normal ? c.o_frame[t.obs_off + q] : 1u;
          c.hist_win[off + y] = code;
          h[y++] = e;
        }
        mph_rp_heapsort(h, n_fold);
        wo.n_extra = n_fold;
        wo.extra_off = off;
      } else {
        *err |= MPH_E_HIST_OVERFLOW;
      }
    }
  } else if (n_keys) {
    const uint32_t off = MPH_RP_ADD(&c.counters[MPH_RP_CTR_HIST], n_keys);
    if (off + n_keys <= c.hist_cap) {
      wo.extra_off = off;
      for (uint32_t a = 0; a < n_keys; ++a) {
        c.hist[off + a] = table[a];
        c.hist_win[off + a] = code;
      }
    } else {
      *err |= MPH_E_HIST_OVERFLOW;
      wo.n_extra = 0;
    }
  }
  c.win_out[widx] = wo;
  MPH_RP_ADD64(c.sum_depth, depth);
  // the matrix columns in print_haplotypes order (:372-378): the deque, reversed on the reverse strand
  const bool rev = (sg.flags & MPH_SF_REVERSE) != 0;
  uint32_t n_walk = 0;
  {
    const uint32_t off = MPH_RP_ADD(&c.counters[MPH_RP_CTR_VLIST], ncols + 1);
    if (off + ncols + 1 <= c.vlist_cap) {
      c.vlist[off] = ncols;
      for (uint32_t j = 0; j < ncols; ++j) c.vlist[off + 1 + j] = rev ? dq[ncols - 1 - j] : dq[j];
      c.win_voff[widx] = off;
    } else {
      *err |= MPH_E_VLIST_OVERFLOW;
    }
    // variants the sequence walk visits (:473-476): j only advances while variants[j].pos == i
    uint32_t j = 0;
    for (uint32_t p = g.s; p < g.e && j < ncols; ++p)
      while (j < ncols && c.vars[rev ? dq[ncols - 1 - j] : dq[j]].pos == p) ++j;
    n_walk = j;
  }
  MphHap h0;
  if (normal) {
    *err |= mph_nrm_plain(sg, g, c.ref, n_walk, &h0);
    c.win_depth[widx] = depth | ((ncols == 0 && (h0.flags & MPH_NF_STOP)) ? 0x80000000u : 0u);
    unsigned long long id = 0;
    if (!(h0.flags & MPH_NF_REFRANGE)) {
      const uint32_t t0 = c.tx_id_off[sg.tx];
      id = mph_record_id64(c.ref + sg.ref_off + (g.s - sg.ref_pos0), g.e - g.s, c.tx_id_bytes + t0, c.tx_id_off[sg.tx + 1] - t0, g.s);
    }
    c.win_id[widx] = id;
    c.win_flag[widx] = ncols > 0 ? 1 : 0;  // the residue reads a window without columns from win_depth / win_id alone
  } else {
    *err |= mph_plain_hap(sg, g, c.stopmap, c.ref, n_walk, &h0);
    c.win_flag[widx] = 1;
  }
  if (ncols > 32) *err |= MPH_E_VARS_PER_WINDOW;
  c.hap0[widx] = h0;
  (void)k;
}

// the window loop of phase_gene (:944-1939) reduced to its matrix operations
MPH_HD void mph_replay_tx(const MphReplayCtx& c, const MphReplayTx& t) {
  uint32_t err = 0;
  uint32_t dq[MPH_RP_MAXCOLS];
  uint32_t ncols = t.dq_n <= MPH_RP_MAXCOLS ? t.dq_n : 0, n_obs = 0;
  if (t.dq_n > MPH_RP_MAXCOLS) err |= MPH_E_VARS_PER_WINDOW;
  for (uint32_t j = 0; j < ncols; ++j) dq[j] = c.dq_init[t.dq_off + j];
  uint64_t last_window_vars = t.last_vars;
  uint32_t* o_read = c.o_read + t.obs_off;
  uint64_t* o_hap = c.o_hap + t.obs_off;
  uint32_t* o_frame = c.o_frame + t.obs_off;
  uint8_t* o_flags = c.o_flags + t.obs_off;
  uint8_t* in_mat = c.o_inmat + t.obs_off;
  const bool normal = c.mode == 1;
  uint32_t* o_last = normal ? c.o_last + t.obs_off : nullptr;  // indexed by read - read_lo (obs_cap >= number of gene reads)
  const uint32_t n_gene_reads = t.read_hi - t.read_lo;
  if (normal) { for (uint32_t x = 0; x < n_gene_reads; ++x) o_last[x] = 0xFFFFFFFFu; }
  else { for (uint32_t x = 0; x < t.obs_cap; ++x) in_mat[x] = 0; }
  bool panicked = false;
  auto shrink_left = [&](uint64_t n) -> bool {  // :220-229
    if (n > ncols) { panicked = true; return false; }  // drain(..k) out of range
    for (uint32_t j = (uint32_t)n; j < ncols; ++j) dq[j - n] = dq[j];
    ncols -= (uint32_t)n;
    const uint64_t mask = ncols >= 64 ? ~(uint64_t)0 : (((uint64_t)1 << ncols) - 1);
    for (uint32_t o = 0; o < n_obs; ++o) o_hap[o] &= mask;
    return true;
  };
  for (uint32_t si = t.seg_lo; si < t.seg_hi && !(err & MPH_E_REPLAY_PANIC); ++si) {
    const MphSegment& sg = c.segs[si];
    const bool rev = (sg.flags & MPH_SF_REVERSE) != 0;
    const bool is_short = (sg.flags & MPH_SF_SHORT) != 0;
    if (!shrink_left(last_window_vars)) { c.seg_err[si] = 1; break; }  // :1024
    last_window_vars = 0;
    uint64_t old_offset = sg.off0, old_end = (uint64_t)sg.off0 + sg.ewl;
    bool reached_end = false;
    bool deferred = false;   // folded iterations are waiting to be offered
    uint32_t pushed_s = 0;   // forward strand: window start of the last iteration whose reads were offered
    MphGeom g_prev = mph_geom(sg, 0);
    // cleanup_reads (:259-278, call sites :1255-1262)
    auto do_cleanup = [&](const MphGeom& gg) {
      uint32_t w = 0;
      for (uint32_t o = 0; o < n_obs; ++o) {
        const uint32_t r = o_read[o];
        // somatic: cleanup_reads(splice_side_offset + 1) (:1257); normal: cleanup_reads(splice_side_offset) (normal_microphasing.rs:1001)
        const bool keep = rev ? c.read_start[r] < gg.s + (normal ? 0u : 1u) : c.read_end[r] >= gg.e;
        if (keep) {
          if (w != o) { o_read[w] = r; o_hap[w] = o_hap[o]; o_frame[w] = o_frame[o]; o_flags[w] = o_flags[o]; }
          if (normal) o_last[r - t.read_lo] = w;  // entries of one read keep their order
          ++w;
        } else if (normal) {
          o_last[r - t.read_lo] = 0xFFFFFFFFu;
        } else {
          in_mat[r - t.read_lo] = 0;
        }
      }
      n_obs = w;
    };
    // candidate reads (:1191-1249) and push_read (:297-343); `lo` = smallest start that is offered
    auto do_push = [&](const MphGeom& gg, uint32_t lo) {
      const uint32_t r0 = mph_u32_lb(c.read_start, t.read_lo, t.read_hi, lo);
      const uint32_t r1 = mph_u32_lb(c.read_start, r0, t.read_hi, gg.s + 1u);
      for (uint32_t r = r0; r < r1; ++r) {
        if (c.read_end[r] < gg.e) continue;
        if (normal) {
          // push_read of the normal mode (:301-331): no `contains`, columns numbered oldest-first, nothing is rejected;
          // consecutive copies of a read with the same haplotype share one entry
          uint64_t hap = 0;
          uint32_t fr0 = 0;
          uint8_t fl0 = 0;
          for (uint32_t i = 0; i < ncols; ++i) mph_rp_update(c, t, r, i, dq[i], &hap, &fr0, &fl0, &err);
          const uint32_t e = o_last[r - t.read_lo];
          if (e != 0xFFFFFFFFu && o_hap[e] == hap) { o_frame[e] += 1; continue; }
          if (n_obs >= t.obs_cap) { err |= MPH_E_REPLAY_INPUT; continue; }
          o_read[n_obs] = r; o_hap[n_obs] = hap; o_frame[n_obs] = 1; o_flags[n_obs] = 0;
          o_last[r - t.read_lo] = n_obs;
          ++n_obs;
          continue;
        }
        if (rev) {
          // `contains` (:281-294): an observation with the same start and qname is already in the matrix
          bool dup = in_mat[r - t.read_lo] != 0;
          if (!dup && (c.read_flags[r] & MPH_RF_PARTNER)) {
            // the reads sharing (start, qname) form a cycle of partner edges: two of them point at each other
            uint32_t q = mph_rp_partner(c, r);
            for (uint32_t hops = 0; !dup && q != 0xFFFFFFFFu && q != r && hops < 4096; ++hops) {
              dup = q >= t.read_lo && q < t.read_hi && in_mat[q - t.read_lo] != 0;
              q = mph_rp_partner(c, q);
            }
          }
          if (dup) continue;
        }
        uint64_t hap = 0;
        uint32_t frame = 0;
        uint8_t fl = 0;
        for (uint32_t i = 0; i < ncols; ++i) mph_rp_update(c, t, r, i, dq[ncols - 1 - i], &hap, &frame, &fl, &err);
        if (fl & 1) continue;  // rejected at push (:338)
        if (n_obs >= t.obs_cap) { err |= MPH_E_REPLAY_INPUT; continue; }
        o_read[n_obs] = r; o_hap[n_obs] = hap; o_frame[n_obs] = frame; o_flags[n_obs] = fl;
        in_mat[r - t.read_lo] = 1;
        ++n_obs;
      }
    };
    for (uint32_t k = 0; k < sg.n_iter; ++k) {
      const uint64_t offset = rev ? (uint64_t)sg.off0 - k : (uint64_t)sg.off0 + k;
      const MphGeom g = mph_geom(sg, k);
      const uint64_t rest = rev ? offset - sg.exon_start : sg.exon_end - (offset + sg.ewl);
      const bool is_last_exon_window = rest < 3, is_first_exon_window = k == 0;
      auto cnt = [&](uint64_t a, uint64_t b) -> uint64_t {  // variant_tree.range(a..b) (:1119-1170); a > b panics in the reference
        if (a > b) { panicked = true; return 0; }
        const uint32_t ia = mph_var_lb(c.vars, sg.var_lo, sg.var_hi, (uint32_t)a);
        return mph_var_lb(c.vars, ia, sg.var_hi, (uint32_t)b) - ia;
      };
      const uint32_t va = mph_var_lb(c.vars, sg.var_lo, sg.var_hi, g.s);
      const uint32_t vb = mph_var_lb(c.vars, va, sg.var_hi, g.e);
      const uint64_t nvars = vb - va;
      uint64_t added_vars, deleted_vars;
      if (is_first_exon_window) added_vars = nvars;
      else if (is_short || reached_end) added_vars = 0;
      else if (g.s > old_offset) added_vars = cnt(old_end, g.e);
      else added_vars = cnt(g.s, old_offset);
      if (offset == old_offset || is_short) deleted_vars = 0;
      else if (g.s > old_offset) deleted_vars = cnt(old_offset, g.s);
      else deleted_vars = cnt(g.e, old_end);
      if (is_last_exon_window) reached_end = true;
      if (panicked) { c.seg_err[si] = k + 1; break; }
      // Folding (somatic mode): an iteration that neither adds nor removes a column and is not an enumerated window only
      // offers reads; offering them later - all at once, just before the next iteration that does something - gives the
      // same matrix, because a read offered at a folded iteration and still alive afterwards passes the same tests against
      // the same columns. The first two iterations are never folded (the candidate range changes shape there).
      const uint64_t skip_cnt = nvars - added_vars;  // wraps like the release build: nothing is added then
      const uint32_t n_new_now = skip_cnt <= nvars ? (uint32_t)(nvars - skip_cnt) : 0u;
      const bool emit_now = k >= sg.k_first && (k - sg.k_first) % sg.k_stride == 0 && (k - sg.k_first) / sg.k_stride < sg.n_win;
      const bool fold = c.batch && !normal && k >= 2 && !emit_now && n_new_now == 0 && deleted_vars == 0 && !is_short;
      if (fold) {
        deferred = true;
        g_prev = g;
        last_window_vars = nvars;
        old_offset = g.s;
        old_end = g.e;
        continue;
      }
      if (deferred && deleted_vars > 0) {  // the folded reads must meet the columns as they were before this iteration's shrink_left
        do_cleanup(g_prev);
        do_push(g_prev, rev ? (g_prev.s > sg.K ? g_prev.s - sg.K : 0u) : pushed_s + 1u);
        pushed_s = g_prev.s;
      }
      deferred = false;
      do_cleanup(g);
      if (!shrink_left(deleted_vars)) { c.seg_err[si] = k + 1; break; }
      {
        const bool wide = rev || offset == (uint64_t)sg.exon_start + sg.ceo;
        uint32_t lo = wide ? (g.s > sg.K ? g.s - sg.K : 0u) : g.s;
        if (!wide && c.batch && !normal && k >= 2) lo = pushed_s + 1u;  // everything since the last offered start
        do_push(g, lo);
        pushed_s = g.s;
      }
      // newly collected variants (:1280-1296): the window's variants in collection order minus the first nvars - added_vars
      {
        const uint64_t skip = nvars - added_vars;  // wraps like the release build: nothing is added then
        const uint32_t n_new = skip <= nvars ? (uint32_t)(nvars - skip) : 0u;
        if (n_new) {
          if (ncols + n_new > MPH_RP_MAXCOLS) { err |= MPH_E_VARS_PER_WINDOW; break; }
          // extend_right (:232-256)
          for (uint32_t o = 0; o < n_obs; ++o) {
            uint64_t hap = o_hap[o] << (n_new & 63u);
            uint32_t frame = o_frame[o];
            uint8_t fl = o_flags[o];
            for (uint32_t i = 0; i < n_new; ++i) {
              const uint32_t x = (uint32_t)skip + (n_new - 1 - i);  // new_variants.rev(): the newest first
              const uint32_t v = rev ? vb - 1 - x : va + x;
              mph_rp_update(c, t, o_read[o], i, v, &hap, &frame, &fl, &err);
            }
            o_hap[o] = hap; o_frame[o] = frame; o_flags[o] = fl;
          }
          for (uint32_t x = (uint32_t)skip; x < (uint32_t)nvars; ++x) dq[ncols++] = rev ? vb - 1 - x : va + x;
        }
      }
      last_window_vars = nvars;
      if (k >= sg.k_first && (k - sg.k_first) % sg.k_stride == 0) {
        const uint32_t i = (k - sg.k_first) / sg.k_stride;
        if (i < sg.n_win) mph_rp_emit(c, t, sg, si, i, k, g, n_obs, dq, ncols, &err);
      }
      old_offset = g.s;
      old_end = g.e;
      if (is_short) break;
    }
    if (panicked) break;
    if (deferred) {  // folded iterations at the end of the exon: their reads may survive into the next one
      do_cleanup(g_prev);
      do_push(g_prev, rev ? (g_prev.s > sg.K ? g_prev.s - sg.K : 0u) : pushed_s + 1u);
    }
  }
  if (err) MPH_RP_OR(&c.counters[MPH_RP_CTR_ERR], err);
}
