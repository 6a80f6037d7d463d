// phase_kernels.cu — hand-written sm_100a kernels of the per-window phasing path (somatic mode).
//
//   K1 k_allele_call   thread per entry of the variant-read side table: supports_variant / bad_quality bitmasks
//                      over the variants inside the read (reference src/microphasing.rs:78-139), expanded to
//                      per-read arrays; reads without an entry were zero-filled before. Packed 4-bit bases are
//                      touched only where a variant lies.
//   K2 k_window_hist   CTA per group of <= 128 consecutive windows of one exon, two phases: thread = read builds a
//                      difference array over the windows for the plain reads (run ends by arithmetic on the window
//                      grid) and a list of the reads that carry allele calls; thread = window prefix-sums it into
//                      depth and evaluates the closed form of the ObservationMatrix (:157-343) for the listed reads
//                      only; haplotype keys go to per-window shared-memory tables (:383-411). k_window_hist_wide
//                      redoes windows whose keys overflow a table, one warp per window, and k_window_hist_block
//                      (block_kernels.cu) the few whose keys overflow that warp's table, one CTA per window.
//   K3 k_assemble      thread per extra haplotype key: sequence walk (:458-603), stop codon test (:42-76,
//                      :694-697) and the SHA-1 record id (:667-675) while the bytes are in registers / L1.
//   K4 k_flag_count / k_block_scan / k_scatter   stable compaction of the interesting windows so the
//                      host sees them in the reference's order.
//   K5 k_live_depth    statistics only: sum of depth over the windows the reference reaches.
//
// The serial replay of irregular transcripts lives in replay_kernels.cu, the `normal` mode in normal_kernels.cu.
// No tensor cores: nothing here is a dense contraction; the path is integer / byte work bounded by
// HBM and L2 bandwidth and by instruction issue in K2.
#include "phase_kernels.cuh"
#include <cstdlib>

#include "kernel_common.cuh"

namespace mphk {

using namespace detail;

namespace {

// ------------------------------------------------------------------ K0: reads off the bus
// A read crosses the bus as 1 B (distance to the previous start; its reference span is the batch's span unless an exception
// list names it) or 2 B (distance, span: batches of reads of all lengths); one warp per run prefix-sums the distances and
// writes the start / end arrays every later kernel uses. Exceptions (other spans, flags) are patched in after.
__global__ void __launch_bounds__(128) k_read_decode(const DeviceBatch d) {
  const uint32_t j = d.run0 + blockIdx.x * 4 + (threadIdx.x >> 5);
  const uint32_t lane = threadIdx.x & 31;
  if (j >= d.run1) return;
  const uint2 run = d.rd_runs[j];
  const uint32_t hi = j + 1 < d.run1 ? d.rd_runs[j + 1].x : d.r1;
  uint32_t pos = run.y;
  for (uint32_t base = run.x; base < hi; base += 32) {
    const uint32_t r = base + lane;
    uint32_t x = r < hi ? d.rd_delta[r] : 0u;
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(FULL, x, o);
      if (lane >= (uint32_t)o) x += y;
    }
    if (r < hi) {
      d.read_start_w[r] = pos + x;
      d.read_end_w[r] = pos + x + (d.rd_span ? (uint32_t)d.rd_span[r] : d.modal_span);
    }
    pos += __shfl_sync(FULL, x, 31);
  }
}

__global__ void __launch_bounds__(256) k_read_patch(const DeviceBatch d) {
  const uint32_t t = blockIdx.x * 256 + threadIdx.x;
  const uint32_t ns = d.sx1 - d.sx0, nf = d.fx1 - d.fx0;
  if (t < ns) { const uint2 e = d.rd_span_exc[d.sx0 + t]; d.read_end_w[e.x] = e.y; }
  else if (t < ns + nf) { const uint2 e = d.rd_flag_exc[d.fx0 + t - ns]; d.read_flags_w[e.x] = (uint8_t)e.y; }
}

// side table off the bus: one warp per run prefix-sums the read / variant-index distances, record sizes and CIGAR counts
__global__ void __launch_bounds__(128) k_side_decode(const DeviceBatch d) {
  const uint32_t j = d.vrun0 + blockIdx.x * 4 + (threadIdx.x >> 5);
  const uint32_t lane = threadIdx.x & 31;
  if (j >= d.vrun1) return;
  const MphSideRun run = d.vs_runs[j];
  const uint32_t hi = j + 1 < d.vrun1 ? d.vs_runs[j + 1].entry : d.vr1;
  uint32_t read = run.read, vlo = run.vlo, so = run.seq_off, co = run.cig_off;
  for (uint32_t base = run.entry; base < hi; base += 32) {
    const uint32_t e = base + lane;
    const bool in = e < hi;
    uint32_t a = in ? d.vs_read_d[e] : 0u, b = in ? d.vs_vlo_d[e] : 0u, c = in ? d.vs_size[e] : 0u;
    const uint32_t nc = in ? d.vs_ncig[e] : 0u;
    uint32_t g = nc < 255u ? nc : 0u;
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t ya = __shfl_up_sync(FULL, a, o), yb = __shfl_up_sync(FULL, b, o), yc = __shfl_up_sync(FULL, c, o), yg = __shfl_up_sync(FULL, g, o);
      if (lane >= (uint32_t)o) { a += ya; b += yb; c += yc; g += yg; }
    }
    if (in) {
      d.vr_read_w[e] = read + a;
      d.vr_vlo_w[e] = vlo + b;
      d.vr_seq_off_w[e] = so + c - d.vs_size[e];                 // exclusive sums for the two offsets
      d.vr_cig_off_w[e] = co + g - (nc < 255u ? nc : 0u);
      d.vr_ncig_w[e] = (uint16_t)nc;
    }
    read += __shfl_sync(FULL, a, 31); vlo += __shfl_sync(FULL, b, 31); so += __shfl_sync(FULL, c, 31); co += __shfl_sync(FULL, g, 31);
  }
}

__global__ void __launch_bounds__(256) k_side_patch(const DeviceBatch d) {
  const uint32_t t = d.nx0 + blockIdx.x * 256 + threadIdx.x;
  if (t < d.nx1) { const uint2 e = d.vs_ncig_exc[t]; d.vr_ncig_w[e.x] = (uint16_t)e.y; }
}

// ------------------------------------------------------------------ K1
__global__ void __launch_bounds__(256) k_allele_call(const DeviceBatch d) {
  const uint32_t e = d.vr0 + blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= d.vr1) return;
  const uint32_t r = d.vr_read[e];
  MphRead rd;
  rd.start = d.read_start[r];
  rd.end = d.read_end[r];
  rd.vlo = d.vr_vlo[e];
  rd.l_seq = d.vr_lseq[e];
  rd.nv = d.vr_nv[e];
  rd.n_cig = d.vr_ncig[e];
  const uint8_t* bases = d.bases + (size_t)d.vr_seq_off[e];
  const uint32_t* cig = d.cigars + d.vr_cig_off[e];
  const MphCall c = mph_call_read(rd, bases, cig, d.vars, d.mode == 0);
  d.call_S[r] = c.S;
  d.call_B[r] = c.B;
  d.call_flags[r] = (uint8_t)(((c.S | c.B) != 0) ? 1u : 0u);  // bit0: the read needs the full pair evaluation
  d.read_vlo[r] = rd.vlo;
  d.read_nv[r] = (uint8_t)rd.nv;
  d.read_vr[r] = e;
  if (d.read_flags[r] & MPH_RF_OVERFLOW) raise(d, MPH_E_VARS_PER_WINDOW);
}

// ------------------------------------------------------------------ K2
__device__ __forceinline__ uint32_t partner_lookup(const DeviceBatch& d, uint32_t r) {
  uint32_t lo = 0, hi = d.n_pairs;
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    if (d.pairs[mid].x < r) lo = mid + 1;
    else hi = mid;
  }
  return (lo < d.n_pairs && d.pairs[lo].x == r) ? d.pairs[lo].y : NONE;
}


// One (read, window) pair with the read flagged by K1 (allele calls, bad bases or a duplicate qname).
__device__ __forceinline__ MphPair eval_flagged(const DeviceBatch& d, const MphSegment& sg, bool rev, uint32_t k, const MphGeom& g, uint32_t va,
                                                uint32_t vb, uint32_t r, uint32_t st, uint32_t en, uint32_t cf, uint32_t vlo, uint64_t S, uint64_t B) {
  MphPair p;
  if (!rev) return mph_fwd_state(sg, d.vars, k, g, va, vb, st, en, vlo, S, B);
  p.member = 0; p.bad = 0; p.hap = 0; p.frame = 0;
  if (st > g.s || en < g.e) return p;
  const uint64_t Bx = B | (S & mph_range_mask(sg.sl_va, sg.sl_vb, vlo));
  uint32_t ke = mph_rev_entry(sg, d.vars, k, st, en, vlo, Bx);
  if (ke != NONE && (cf & 2u)) {
    // `contains` (:281-294): of two reads sharing (start, qname) only the first to enter stays
    const uint32_t q = partner_lookup(d, r);
    if (q != NONE) {
      const uint32_t qs = d.read_start[q], qe = d.read_end[q], qv = d.read_vlo[q];
      if (qs <= g.s && qe >= g.e) {
        const bool qc = (d.call_flags[q] & 1u) != 0;  // S / B are only written for reads with a call
        const uint64_t Bq = qc ? (d.call_B[q] | (d.call_S[q] & mph_range_mask(sg.sl_va, sg.sl_vb, qv))) : 0;
        const uint32_t kq = mph_rev_entry(sg, d.vars, k, qs, qe, qv, Bq);
        if (kq != NONE && (kq < ke || (kq == ke && q < r))) ke = NONE;
      }
    }
  }
  if (ke != NONE) p = mph_rev_state(sg, d.vars, k, g, va, vb, st, en, vlo, S, B, ke);
  return p;
}

// Wide variant: one warp per window, lanes over the candidate reads, keys in a 32-entry table.
// Used only for windows whose key count overflows the per-lane table of k_window_hist. A window with more keys than the
// table holds walks its reads a second time and hands its counted observations to k_window_hist_block (spill_window).
__device__ void window_hist_warp(const DeviceBatch& d, const MphSegment& sg, uint32_t ch_seg, uint32_t i, uint32_t code, MphHist* table, int lane) {
  const bool rev = (sg.flags & MPH_SF_REVERSE) != 0;
  const uint32_t k = sg.k_first + i * sg.k_stride;
  const uint32_t widx = sg.win_base + i;
  const MphGeom g = mph_geom(sg, k);
  const uint32_t va = mph_var_lb(d.vars, sg.var_lo, sg.var_hi, g.s);
  const uint32_t vb = mph_var_lb(d.vars, va, sg.var_hi, g.e);
  uint32_t rlo, rhi;
  mph_candidate_range(sg, d.read_start, g, &rlo, &rhi);
  // the observation of read r (member / counted = member and not bad_qual) with its key
  auto observe = [&](uint32_t r, bool* member, bool* counted, uint64_t* hap, uint32_t* frame) {
    *member = false; *counted = false; *hap = 0; *frame = 0;
    if (r >= rhi) return;
    const uint32_t st = d.read_start[r], en = d.read_end[r];
    if (en < g.e) return;
    const uint32_t cf = d.call_flags[r] | ((d.read_flags[r] & MPH_RF_PARTNER) ? 2u : 0u);
    const uint64_t S = (cf & 1u) ? d.call_S[r] : 0, B = (cf & 1u) ? d.call_B[r] : 0;  // S / B are only written for reads with a call
    const MphPair p = eval_flagged(d, sg, rev, k, g, va, vb, r, st, en, cf, d.read_vlo[r], S, B);
    *member = p.member != 0;
    *counted = *member && !p.bad;
    *hap = p.hap;
    *frame = p.frame;
  };
  const uint32_t key_cap = d.force_wide == 2 ? 0u : (uint32_t)K2_TABLE;
  uint32_t depth = 0, c0 = 0, n_keys = 0, n_spill = 0;
  bool spill = false;  // lane 0: a key did not fit the table
  for (uint32_t base = rlo; base < rhi; base += 32) {
    bool member, counted;
    uint64_t hap;
    uint32_t frame;
    observe(base + lane, &member, &counted, &hap, &frame);
    depth += __popc(__ballot_sync(FULL, member));
    const bool zero_key = counted && hap == 0 && frame == 0;
    c0 += __popc(__ballot_sync(FULL, zero_key));
    unsigned pending = __ballot_sync(FULL, counted && !zero_key);
    n_spill += __popc(pending);
    if (__shfl_sync(FULL, (int)spill, 0)) continue;
    while (pending) {
      const int leader = __ffs(pending) - 1;
      const uint64_t lh = __shfl_sync(FULL, hap, leader);
      const uint32_t lf = __shfl_sync(FULL, frame, leader);
      const unsigned same = __ballot_sync(FULL, counted && !zero_key && hap == lh && frame == lf);
      if (lane == 0 && !spill) {
        uint32_t t = 0;
        for (; t < n_keys; ++t)
          if (table[t].hap == lh && table[t].frame == lf) break;
        if (t == n_keys) {
          if (n_keys < key_cap) {
            table[t].hap = lh;
            table[t].frame = lf;
            table[t].count = 0;
            ++n_keys;
          } else {
            spill = true;
          }
        }
        if (!spill) table[t].count += __popc(same);
      }
      pending &= ~same;
    }
  }
  if (__shfl_sync(FULL, (int)spill, 0)) {
    // second walk: the counted observations outside the (0, 0) key, in read order, to the spill arena
    uint32_t off = 0;
    if (lane == 0) off = atomicAdd(&d.counters[CTR_SPILL], n_spill);
    off = __shfl_sync(FULL, off, 0);
    if ((uint64_t)off + n_spill <= d.spill_cap) {
      uint32_t y = off;
      for (uint32_t base = rlo; base < rhi; base += 32) {
        bool member, counted;
        uint64_t hap;
        uint32_t frame;
        observe(base + lane, &member, &counted, &hap, &frame);
        const bool emit = counted && !(hap == 0 && frame == 0);
        const unsigned bal = __ballot_sync(FULL, emit);
        if (emit) {
          MphHist e;
          e.hap = hap; e.count = 1; e.frame = frame;
          d.spill[y + __popc(bal & ((1u << lane) - 1u))] = e;
        }
        y += __popc(bal);
      }
      if (lane == 0) {
        MphSpillWin q;
        q.code = code; q.off = off; q.n = n_spill; q.devrec = (sg.flags & MPH_SF_DEVREC) ? 1u : 0u;
        d.spq[atomicAdd(&d.counters[CTR_SPQ], 1u)] = q;
      }
    } else if (lane == 0) {
      raise(d, MPH_E_SPILL_OVERFLOW);
    }
    n_keys = 0;  // k_window_hist_block writes the keys and sets n_extra / extra_off
  }
  if (lane == 0) {
    for (uint32_t a = 1; a < n_keys; ++a) {  // keys in the reference's BTreeMap order (:383,434)
      const MphHist key = table[a];
      uint32_t b = a;
      while (b > 0 && hist_less(key, table[b - 1])) {
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
    if (n_keys) {
      const bool devrec = (sg.flags & MPH_SF_DEVREC) != 0;
      uint32_t off = atomicAdd(&d.counters[devrec ? CTR_HISTD : CTR_HIST], n_keys);
      const bool fits = off + n_keys <= d.hist_cap;
      if (devrec && fits) off = d.hist_cap - off - n_keys;
      if (fits) {
        wo.extra_off = off;
        for (uint32_t a = 0; a < n_keys; ++a) {
          d.hist[off + a] = table[a];
          d.hist_win[off + a] = code;
        }
      } else {
        raise(d, MPH_E_HIST_OVERFLOW);
        wo.n_extra = 0;
      }
    }
    d.win_out[widx] = wo;
    atomicAdd(d.sum_depth, (unsigned long long)depth);
    MphHap h0;
    const uint32_t err = mph_plain_hap(sg, g, d.stopmap, d.ref, vb - va, &h0);
    d.win_flag[widx] = (sg.flags & MPH_SF_DEVREC) ? 2 : 1;  // it has extra keys, hence it is interesting
    if (sg.flags & MPH_SF_DEVREC) d.win_seg[widx] = ch_seg;
    d.hap0[widx] = h0;
    raise(d, err);
  }
  __syncwarp();
}

__global__ void __launch_bounds__(K2_WARPS * 32) k_window_hist_wide(const DeviceBatch d) {
  __shared__ MphHist table[K2_WARPS][K2_TABLE];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t n = d.counters[CTR_OVF];
  for (uint32_t o = blockIdx.x * K2_WARPS + warp; o < n; o += gridDim.x * K2_WARPS) {
    const uint32_t code = d.ovf_list[o];
    const MphChunk ch = d.chunks[code >> 5];
    const MphSegment sg = d.segs[ch.seg];
    window_hist_warp(d, sg, ch.seg, ch.i_first + (code & 31u), code, table[warp], lane);
  }
}

// K2a k_read_runs: thread per (segment, read) pair of the packer-resolved candidate ranges, a pure streaming kernel.
// A read without allele calls / bad bases / duplicate qname is an observation of a *contiguous* run of the segment's
// windows (membership is monotone in the iteration number). The run's ends come from arithmetic on the window grid
// (windows sit k_stride iterations apart) corrected against mph_geom, and the read adds +1 at the run's first window and
// -1 after its last one to a per-window difference array in global memory (no-return atomics: L2 reductions). Reads that
// carry an allele call, and the rare ones that need the full closed form, are appended to the segment's list.
// Every read is visited once per exon it can overlap (round 1 visited it once per 32-window chunk, with three binary
// searches over the window table each time).
constexpr int RR_THREADS = 256;
constexpr int RR_IPT = 4;  // work items per thread
constexpr int RR_ITEMS = RR_THREADS * RR_IPT;

// first segment of every K2a block: last segment whose items start at or before the block's first item. One thread per
// block searches here, in parallel, so that k_read_runs does not start every CTA with a 17-step dependent search behind a
// barrier (a fifth of its stall samples in the round-2 ncu capture).
__global__ void __launch_bounds__(256) k_read_runs_plan(const DeviceBatch d, uint32_t n_blocks) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_blocks) return;
  const uint32_t first = d.it0 + b * RR_ITEMS;
  uint32_t lo = d.s0, hi = d.s1;
  while (hi - lo > 1) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    if (d.seg_work_off[mid] <= first) lo = mid;
    else hi = mid;
  }
  d.rr_seg0[b] = lo;
}

__global__ void __launch_bounds__(RR_THREADS) k_read_runs(const DeviceBatch d) {
  const uint32_t it0 = d.it0, it1 = d.it1;
  const uint32_t first = it0 + blockIdx.x * RR_ITEMS;
  uint32_t seg = d.rr_seg0[blockIdx.x];
  uint32_t a_r[RR_IPT], a_seg[RR_IPT], a_st[RR_IPT], a_en[RR_IPT], a_cf[RR_IPT];
#pragma unroll
  for (int u = 0; u < RR_IPT; ++u) {
    const uint32_t item = first + u * RR_THREADS + threadIdx.x;
    a_r[u] = NONE;
    if (item < it1) {
      while (item >= d.seg_work_off[seg + 1]) ++seg;  // consecutive items: the same segment or one of the next few
      const uint32_t r = d.seg_work[seg].rlo + (item - d.seg_work_off[seg]);
      a_r[u] = r;
      a_seg[u] = seg;
      a_st[u] = d.read_start[r];
      a_en[u] = d.read_end[r];
      a_cf[u] = (uint32_t)d.call_flags[r] | ((d.read_flags[r] & MPH_RF_PARTNER) ? 2u : 0u);
    }
  }
#pragma unroll
  for (int u = 0; u < RR_IPT; ++u) {
    const uint32_t r = a_r[u];
    if (r == NONE) continue;
    const uint32_t si = a_seg[u], st = a_st[u], en = a_en[u], cf = a_cf[u];
    const MphSegment& sg = d.segs[si];
    const uint32_t flags = sg.flags;
    const bool rev = (flags & MPH_SF_REVERSE) != 0, has_fs = (flags & MPH_SF_HAS_FS) != 0;
    int cls;
    if (cf == 0 && !has_fs) {
      cls = 1;
    } else {
      const uint32_t vlo = d.read_vlo[r];
      const uint64_t S = (cf & 1u) ? d.call_S[r] : 0, B = (cf & 1u) ? d.call_B[r] : 0;  // S / B are only written for reads with a call
      const uint64_t Bx = B | (S & mph_range_mask(sg.sl_va, sg.sl_vb, vlo));
      const MphSegWork sw = d.seg_work[si];
      if (Bx == 0 && !(cf & 2u) && !has_fs) cls = (S != 0 && sw.vb1 > sw.va0) ? 2 : 1;
      else cls = 3;
    }
    if (cls == 2 && sg.n_win > 0xFFFFu) cls = 3;  // the run does not fit the list entry: full closed form per window
    bool counted = false;
    uint32_t run_lo = 0, run_hi = 0;
    if (cls != 3) {
      // Run of windows [ilo, ihi] of this segment at which the read is an observation. Here the segment has no
      // frameshift enumeration (those reads are all class 3), so windows sit 3 iterations apart (k = kf + 3 i) and only
      // the exon's first and last window deviate from s = off0 +- k, e = s + ewl (mph_geom).
      const int n = (int)sg.n_win;
      const int off0 = (int)sg.off0, ewl = (int)sg.ewl, kf = (int)sg.k_first;
      const int ist = (int)st, ien = (int)en;
      const MphGeom g_first = mph_geom(sg, (uint32_t)kf), g_last = mph_geom(sg, (uint32_t)(kf + (n - 1) * (int)sg.k_stride));
      // a segment without frameshift enumeration has one window (short exon) or windows exactly 3 iterations apart
      auto fdiv = [](int x) { return x >= 0 ? x / 3 : -((-x + 2) / 3); };  // floor(x / 3)
      auto cdiv = [&](int x) { return -fdiv(-x); };                        // ceil(x / 3)
      auto clampi = [](int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); };
      int ilo, ihi;
      if (n == 1) {
        // the single window of the segment: the membership test itself
        const uint32_t s0 = sg.off0 - sg.ceo;
        bool member;
        if (!rev) member = en >= g_first.e && (kf == 0 ? (st <= s0 && (int64_t)st >= (int64_t)s0 - (int64_t)sg.K) : (st <= s0 ? (int64_t)st >= (int64_t)s0 - (int64_t)sg.K : (st > sg.off0 && ist - off0 <= kf)));
        else member = st <= g_first.s && en >= g_first.e && (int64_t)st + sg.K >= (int64_t)g_first.s;
        ilo = member ? 0 : 1;
        ihi = 0;
      } else if (!rev) {
        // e is non-decreasing: e(i) = off0 + k + ewl for i < n - 1, the last window ends at g_last.e
        if (en >= g_last.e) ihi = n - 1;
        else ihi = ien >= off0 + ewl + kf ? clampi(fdiv(ien - off0 - ewl - kf), -1, n - 2) : -1;
        const uint32_t s0 = sg.off0 - sg.ceo;
        if (st <= s0) ilo = ((int64_t)st >= (int64_t)s0 - (int64_t)sg.K) ? 0 : n;  // offered at iteration 0 (:1227-1248)
        else if (st <= sg.off0) ilo = n;                                           // never offered
        else ilo = clampi(cdiv(ist - off0 - kf), 0, n);                            // first window at or after the offering iteration
      } else {
        // s is non-increasing: s(i) = off0 - k for i < n - 1, the last window starts at g_last.s
        if (st <= g_last.s) ihi = n - 1;
        else ihi = ist <= off0 - kf ? clampi(fdiv(off0 - kf - ist), -1, n - 2) : -1;
        // first window with e <= en: e(0) = g_first.e, e(i) = off0 - k + ewl for i >= 1 (non-increasing)
        int a;
        if (g_first.e <= en) a = 0;
        else a = clampi(cdiv(off0 - kf + ewl - ien), 1, n);
        // first window with s <= st + K
        const int64_t lim64 = (int64_t)st + sg.K;
        const int lim = lim64 > 0x7FFFFFFF ? 0x7FFFFFFF : (int)lim64;
        int b = clampi(cdiv(off0 - kf - lim), 0, n);
        if (b > n - 2) b = ((int64_t)g_last.s <= lim64) ? n - 1 : n;
        if (n == 1) b = ((int64_t)g_first.s <= lim64) ? 0 : 1;
        ilo = a > b ? a : b;
      }
      if (ilo <= ihi) {
        counted = true;
        run_lo = (uint32_t)ilo;
        run_hi = (uint32_t)ihi;
        atomicAdd(&d.win_diff[sg.win_base + ilo], 1);
        if (ihi + 1 < n) atomicAdd(&d.win_diff[sg.win_base + ihi + 1], -1);
      }
    }
    // the segment's list: full-closed-form reads from the front, reads that only add haplotype keys (with their run) from the back
    if (cls == 3) {
      d.seg_list[d.seg_work_off[si] + atomicAdd(&d.seg_list_n[si], 1u)] = make_uint2(r, 0u);
    } else if (cls == 2 && counted) {
      d.seg_list[d.seg_work_off[si + 1] - 1u - atomicAdd(&d.seg_list2_n[si], 1u)] = make_uint2(r, run_lo | (run_hi << 16));
    }
  }
}

// K2b k_window_hist: warp per chunk (<= 32 consecutive windows of one exon), lane = window. Depth and the (hap 0, frame 0)
// count are the prefix sum of K2a's difference array; only the reads K2a listed for the segment are evaluated per window
// (closed form of the ObservationMatrix), and their haplotype keys go to per-lane shared-memory tables.
constexpr int K2_LANE_KEYS = 4;
constexpr int K2B_WARPS = 4;

// MINB: CTAs per SM the register allocation aims at (8 -> 64 registers, 10 -> 48 with a few spilled words); both are
// compiled and MPH_K2B_MINB picks one at run time (the default is the one measured faster on B200, see DESIGN.md section 5).
template <int MINB>
__global__ void __launch_bounds__(K2B_WARPS * 32, MINB) k_window_hist(const DeviceBatch d) {
  // per-lane key tables, [key][lane] so that a warp touches 32 distinct banks
  __shared__ uint64_t t_hap[K2B_WARPS][K2_LANE_KEYS][32];
  __shared__ uint32_t t_cnt[K2B_WARPS][K2_LANE_KEYS][32];
  __shared__ uint32_t t_frm[K2B_WARPS][K2_LANE_KEYS][32];
  __shared__ MphSegment s_seg[K2B_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t chunk = d.c0 + blockIdx.x * K2B_WARPS + warp;
  if (chunk >= d.c1) return;
  const MphChunk ch = d.chunks[chunk];
  if (lane < (int)(sizeof(MphSegment) / 4)) reinterpret_cast<uint32_t*>(&s_seg[warp])[lane] = reinterpret_cast<const uint32_t*>(&d.segs[ch.seg])[lane];
  __syncwarp();
  const MphSegment& sg = s_seg[warp];
  if (sg.flags & MPH_SF_REPLAY) return;  // the whole transcript goes through k_replay
  const bool rev = (sg.flags & MPH_SF_REVERSE) != 0;
  const int n = (int)ch.n;
  const bool active = lane < n;
  const uint32_t i = ch.i_first + (active ? lane : 0);
  const uint32_t k = sg.k_first + i * sg.k_stride;
  const MphGeom g = mph_geom(sg, k);
  // prefix sum of the difference array: the windows of this segment before the chunk, then the chunk itself
  int carry = 0;
  for (uint32_t j = lane; j < ch.i_first; j += 32) carry += d.win_diff[sg.win_base + j];
  for (int o = 16; o; o >>= 1) carry += __shfl_xor_sync(FULL, carry, o);
  int run = active ? d.win_diff[sg.win_base + i] : 0;
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(FULL, run, o);
    if (lane >= o) run += y;
  }
  run += carry;
  const bool chunk_has_var = ch.vb1 > ch.va0;  // four chunks in five have none: no searches, no key-only list
  const uint32_t va = chunk_has_var ? mph_var_lb(d.vars, ch.va0, ch.vb1, g.s) : ch.va0;
  const uint32_t vb = chunk_has_var ? mph_var_lb(d.vars, va, ch.vb1, g.e) : ch.va0;
  const uint32_t nvar = vb - va;
  if (active && nvar > 64) raise(d, MPH_E_VARS_PER_WINDOW);
  const uint32_t my_s = active ? g.s : 0u;
  const uint32_t my_e = active ? g.e : 0xFFFFFFFFu;  // inactive lanes: nothing encloses e = 0xFFFFFFFF
  uint32_t depth_x = 0, n_keys = 0;  // depth_x: observations counted here (reads that need the closed form)
  int c0_adj = 0;
  bool overflow = false;
  auto add_key = [&](uint64_t hap, uint32_t frame) {
    uint32_t q = 0;
    for (; q < n_keys; ++q)
      if (t_hap[warp][q][lane] == hap && t_frm[warp][q][lane] == frame) break;
    if (q == n_keys) {
      if (n_keys == K2_LANE_KEYS || d.force_wide) { overflow = true; return; }
      t_hap[warp][q][lane] = hap;
      t_frm[warp][q][lane] = frame;
      t_cnt[warp][q][lane] = 0;
      ++n_keys;
    }
    t_cnt[warp][q][lane] += 1;
  };
  // the listed reads of the segment (lane = window); the list order varies from run to run, the sorted keys do not.
  // (1) reads that need the full closed form (bad bases, duplicate qname, frameshift enumeration): every window
  const uint32_t list3_n = d.seg_list_n[ch.seg];
  const uint2* list = d.seg_list + d.seg_work_off[ch.seg];
  for (uint32_t x0 = 0; x0 < list3_n; x0 += 32) {
    uint32_t mine_r = 0, mine_st = 0, mine_en = 0;
    if (x0 + lane < list3_n) { mine_r = list[x0 + lane].x; mine_st = d.read_start[mine_r]; mine_en = d.read_end[mine_r]; }
    const uint32_t cnt = min(32u, list3_n - x0);
    for (uint32_t x = 0; x < cnt; ++x) {
      const uint32_t r = __shfl_sync(FULL, mine_r, x);
      const uint32_t st = __shfl_sync(FULL, mine_st, x), en = __shfl_sync(FULL, mine_en, x);
      if (en < my_e || st > my_s) continue;
      const uint32_t cf = (uint32_t)d.call_flags[r] | ((d.read_flags[r] & MPH_RF_PARTNER) ? 2u : 0u);
      const uint64_t S = (cf & 1u) ? d.call_S[r] : 0, B = (cf & 1u) ? d.call_B[r] : 0;
      const MphPair p = eval_flagged(d, sg, rev, k, g, va, vb, r, st, en, cf, d.read_vlo[r], S, B);
      depth_x += p.member;
      if (p.member && !p.bad) {
        if (p.hap == 0 && p.frame == 0) c0_adj += 1;
        else add_key(p.hap, p.frame);
      }
    }
  }
  // (2) reads already counted as plain observations over a run of windows: the windows with variants need their haplotype
  uint32_t single_cnt = 0;  // windows with exactly one variant: their only possible extra key is haplotype 1 - a counter, no table
  const bool single = nvar == 1;
  if (chunk_has_var) {
    const uint32_t list2_n = d.seg_list2_n[ch.seg];
    const uint2* list2 = d.seg_list + d.seg_work_off[ch.seg + 1] - list2_n;
    for (uint32_t x0 = 0; x0 < list2_n; x0 += 32) {
      // one coalesced load of 32 entries; each lane fetches its entry's allele calls once, the windows get them by shuffle
      uint32_t mine_run = 0xFFFFu, mine_vlo = 0, mine_Slo = 0, mine_Shi = 0;
      if (x0 + lane < list2_n) {
        const uint2 e = list2[x0 + lane];
        const uint64_t S = d.call_S[e.x];
        mine_run = e.y; mine_vlo = d.read_vlo[e.x]; mine_Slo = (uint32_t)S; mine_Shi = (uint32_t)(S >> 32);
      }
      // skip the batch if none of its runs reaches a window with variants of this chunk
      const uint32_t lo_i = mine_run & 0xFFFFu, hi_i = mine_run >> 16;
      const bool touches = lo_i <= hi_i && hi_i >= ch.i_first && lo_i < ch.i_first + (uint32_t)n;
      if (!__any_sync(FULL, touches)) continue;
      const uint32_t cnt = min(32u, list2_n - x0);
      for (uint32_t x = 0; x < cnt; ++x) {
        const uint32_t rr = __shfl_sync(FULL, mine_run, x);
        const uint32_t vlo = __shfl_sync(FULL, mine_vlo, x);
        const uint64_t S = (uint64_t)__shfl_sync(FULL, mine_Slo, x) | ((uint64_t)__shfl_sync(FULL, mine_Shi, x) << 32);
        const bool in_run = nvar != 0 && active && i >= (rr & 0xFFFFu) && i <= (rr >> 16);
        if (single) {
          // bit (va - vlo) of S, if the variant is among the read's own
          const uint32_t sh = va - vlo;
          const uint32_t bit = (in_run && va >= vlo && sh < 64u) ? (uint32_t)((S >> sh) & 1u) : 0u;
          single_cnt += bit;
          continue;
        }
        if (!in_run) continue;
        const uint64_t bits = mph_window_bits(S, vlo, va, nvar);
        const uint64_t hap = rev ? bits : (mph_bitrev64(bits) >> (64 - nvar));
        if (hap != 0) {
          c0_adj -= 1;
          add_key(hap, 0);
        }
      }
    }
  }
  if (single_cnt) {  // fold the counter into the key table (it may already hold haplotype 1 from a closed-form read)
    c0_adj -= (int)single_cnt;
    uint32_t q = 0;
    for (; q < n_keys; ++q)
      if (t_hap[warp][q][lane] == 1 && t_frm[warp][q][lane] == 0) break;
    if (q == n_keys) {
      if (n_keys == K2_LANE_KEYS || d.force_wide) overflow = true;
      else { t_hap[warp][q][lane] = 1; t_frm[warp][q][lane] = 0; t_cnt[warp][q][lane] = 0; ++n_keys; }
    }
    if (q < K2_LANE_KEYS && !overflow) t_cnt[warp][q][lane] += single_cnt;
  }
  const uint32_t depth = (uint32_t)run + depth_x;
  const uint32_t c0 = (uint32_t)(run + c0_adj);
  // each lane sorts its keys (reference BTreeMap order :383,434)
  for (uint32_t a = 1; a < n_keys; ++a) {
    MphHist key;
    key.hap = t_hap[warp][a][lane]; key.frame = t_frm[warp][a][lane]; key.count = t_cnt[warp][a][lane];
    uint32_t b = a;
    while (b > 0) {
      MphHist prev;
      prev.hap = t_hap[warp][b - 1][lane]; prev.frame = t_frm[warp][b - 1][lane]; prev.count = t_cnt[warp][b - 1][lane];
      if (!hist_less(key, prev)) break;
      t_hap[warp][b][lane] = prev.hap; t_frm[warp][b][lane] = prev.frame; t_cnt[warp][b][lane] = prev.count;
      --b;
    }
    t_hap[warp][b][lane] = key.hap; t_frm[warp][b][lane] = key.frame; t_cnt[warp][b][lane] = key.count;
  }
  const bool ovf = active && overflow;
  const uint32_t mine = (active && !ovf) ? n_keys : 0;
  // warp-aggregated allocation in the key arena
  uint32_t incl = mine;
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(FULL, incl, o);
    if (lane >= o) incl += y;
  }
  const uint32_t total = __shfl_sync(FULL, incl, 31);
  uint32_t base_off = 0;
  const bool devrec_keys = (sg.flags & MPH_SF_DEVREC) != 0;
  if (lane == 0 && total) base_off = atomicAdd(&d.counters[devrec_keys ? CTR_HISTD : CTR_HIST], total);
  base_off = __shfl_sync(FULL, base_off, 0);
  const bool fits = base_off + total <= d.hist_cap;
  if (lane == 0 && total && !fits) raise(d, MPH_E_HIST_OVERFLOW);
  if (devrec_keys && fits) base_off = d.hist_cap - base_off - total;  // device-class keys grow from the back of the arena
  if (active && !ovf) {
    MphWinOut wo;
    wo.depth = depth;
    wo.c0 = c0;
    wo.n_extra = fits ? mine : 0;
    wo.extra_off = base_off + incl - mine;
    if (fits)
      for (uint32_t a = 0; a < mine; ++a) {
        MphHist h;
        h.hap = t_hap[warp][a][lane]; h.frame = t_frm[warp][a][lane]; h.count = t_cnt[warp][a][lane];
        d.hist[wo.extra_off + a] = h;
        d.hist_win[wo.extra_off + a] = (chunk << 5) | (uint32_t)lane;
      }
    const uint32_t widx = sg.win_base + i;
    d.win_out[widx] = wo;
    // Haplotype 0 needs no sequence walk (no variant is applied): stop test from the bitmap, and the
    // "interesting" decision. Only the extra keys (hap != 0) go through K3.
    MphHap h0;
    const uint32_t err = mph_plain_hap(sg, g, d.stopmap, d.ref, nvar, &h0);
    const bool boundary = mph_is_boundary(sg, i);
    const bool interesting = nvar > 0 || (h0.flags & MPH_HF_STOP) || boundary || wo.n_extra > 0;
    const bool devrec = (sg.flags & MPH_SF_DEVREC) != 0;  // 2: the record kernels take the window, 1: the host residue does
    d.win_flag[widx] = interesting ? (devrec ? 2 : 1) : 0;
    if (interesting) {
      d.hap0[widx] = h0;
      if (devrec) d.win_seg[widx] = ch.seg;
    }
    raise(d, err);
  }
  if (ovf) {
    const uint32_t o = atomicAdd(&d.counters[CTR_OVF], 1u);
    d.ovf_list[o] = (chunk << 5) | (uint32_t)lane;
  }
  unsigned long long dsum = (active && !ovf) ? depth : 0;
  for (int o = 16; o; o >>= 1) dsum += __shfl_down_sync(FULL, dsum, o);
  if (lane == 0 && dsum) atomicAdd(d.sum_depth, dsum);
}

// ------------------------------------------------------------------ K3
// One thread per extra histogram key (haplotype != 0): the sequence walk of print_haplotypes
// (:458-603) into thread-local buffers, then the stop test; the bytes are kept only for haplotypes
// that can be written (n_somatic > 0) or merged across a splice junction (boundary windows).
// `part`: ASM_ALL walks both ends of the key arena; ASM_DEVICE_CLASS only the keys of device-class transcripts (the back),
// while the serial replay may still be appending host-class keys at the front on its side stream; ASM_HOST_CLASS only the
// front, after the replay (capi.cu).
__global__ void __launch_bounds__(128) k_assemble(const DeviceBatch d, const int part) {
  uint32_t n_front = min(d.counters[CTR_HIST], d.hist_cap);
  const uint32_t n_back_all = min(d.counters[CTR_HISTD], d.hist_cap);
  if (n_front + n_back_all > d.hist_cap) {  // the two ends of the key arena met: the host retries with a larger one
    if (blockIdx.x == 0 && threadIdx.x == 0) raise(d, MPH_E_HIST_OVERFLOW);
    return;
  }
  uint32_t n_back = n_back_all;
  if (part == ASM_DEVICE_CLASS) n_front = 0;
  if (part == ASM_HOST_CLASS) n_back = 0;
  const uint32_t n = n_front + n_back;
  uint8_t seq[MAX_SEQ_CAP], germ[MAX_SEQ_CAP];
  const uint32_t cap = d.seq_cap;
  for (uint32_t y = blockIdx.x * blockDim.x + threadIdx.x; y < n; y += gridDim.x * blockDim.x) {
    const uint32_t x = y < n_front ? y : d.hist_cap - n_back + (y - n_front);
    const uint64_t hap = d.hist[x].hap;
    if (hap == 0) continue;  // a (hap 0, frame != 0) key shares the window's haplotype-0 record
    const uint32_t code = d.hist_win[x];
    // (a front that grew into the back while this launch walks it - ASM_DEVICE_CLASS beside the replay - is caught by the
    // ASM_HOST_CLASS launch, which raises the overflow; until then a clobbered key must not send the walk out of bounds)
    if ((code >> 5) >= d.n_chunks) continue;
    const MphChunk ch = d.chunks[code >> 5];
    const MphSegment sg = d.segs[ch.seg];
    const uint32_t i = ch.i_first + (code & 31u);
    const uint32_t k = sg.k_first + i * sg.k_stride;
    const MphGeom g = mph_geom(sg, k);
    const uint32_t va = mph_var_lb(d.vars, ch.va0, ch.vb1, g.s);
    const uint32_t vb = mph_var_lb(d.vars, va, ch.vb1, g.e);
    const bool replayed = (sg.flags & MPH_SF_REPLAY) != 0;
    const bool boundary = mph_is_boundary(sg, i) || replayed;
    MphHap out;
    uint32_t err;
    if (!replayed) {
      err = mph_assemble(sg, g, d.vars, va, vb, d.ref, d.ins_bytes, hap, seq, germ, cap, &out);
    } else {
      // the walk runs over the matrix columns the replay recorded, gathered into a dense array
      MphVar cols[MPH_RP_MAXCOLS];
      const uint32_t off = d.win_voff[sg.win_base + i];
      const uint32_t ncol = off == NONE ? 0u : min(d.vlist[off], (uint32_t)MPH_RP_MAXCOLS);
      for (uint32_t j = 0; j < ncol; ++j) cols[j] = d.vars[d.vlist[off + 1 + j]];
      err = mph_assemble(sg, g, cols, 0, ncol, d.ref, d.ins_bytes, hap, seq, germ, cap, &out);
    }
    // record id (:667-675): SHA-1 over the debug rendering of the assembled bytes, hashed while they are in registers / L1
    if ((out.n_som > 0 || (sg.flags & MPH_SF_HAS_FS)) && out.seq_len <= cap) {
      const uint32_t t0 = d.tx_id_off[sg.tx];
      out.id64 = mph_record_id64(seq, out.seq_len, d.tx_id_bytes + t0, d.tx_id_off[sg.tx + 1] - t0, g.s);
      out.flags |= MPH_HF_ID;
    }
    if (boundary || out.n_som > 0) {
      // device-class transcripts keep their sequences on the device (the record kernels read them), the others are downloaded
      const bool devrec = (sg.flags & MPH_SF_DEVREC) != 0;
      uint8_t* arena = devrec ? d.seq_dev : d.seq;
      const uint32_t arena_cap = devrec ? d.seq_dev_cap_bytes : d.seq_cap_bytes;
      const uint32_t off = atomicAdd(&d.counters[devrec ? CTR_SEQD : CTR_SEQ], 2 * cap);
      if (off + 2 * cap <= arena_cap) {
        const uint32_t sl = out.seq_len < cap ? out.seq_len : cap, gl = out.germ_len < cap ? out.germ_len : cap;
        for (uint32_t t = 0; t < sl; ++t) arena[off + t] = seq[t];
        for (uint32_t t = 0; t < gl; ++t) arena[off + cap + t] = germ[t];
        out.seq_off = off;
        out.flags |= MPH_HF_SEQ;
      } else {
        err |= MPH_E_SEQ_OVERFLOW;
      }
    }
    d.hapx[x] = out;
    raise(d, err);
  }
}

// ------------------------------------------------------------------ K4: stable compaction
constexpr int SCAN_THREADS = 1024;

__global__ void __launch_bounds__(SCAN_THREADS) k_flag_count(const DeviceBatch d) {
  const uint32_t w = d.w0 + blockIdx.x * SCAN_THREADS + threadIdx.x;
  const int f = (w < d.w1) && d.win_flag[w] == 1;  // 2 = device-class transcript: its records are built by the record kernels
  const int n = __syncthreads_count(f);
  if (threadIdx.x == 0) d.block_counts[blockIdx.x] = (uint32_t)n;
}

// exclusive scan of block_counts in place (one CTA), total -> counters[CTR_NIW]
__global__ void __launch_bounds__(SCAN_THREADS) k_block_scan(const DeviceBatch d, uint32_t n_blocks) {
  __shared__ uint32_t warp_sums[32];
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (uint32_t base = 0; base < n_blocks; base += SCAN_THREADS) {
    const uint32_t idx = base + threadIdx.x;
    const uint32_t v = idx < n_blocks ? d.block_counts[idx] : 0;
    uint32_t x = v;
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(FULL, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
      uint32_t s = warp_sums[lane];
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(FULL, s, o);
        if (lane >= o) s += y;
      }
      warp_sums[lane] = s;
    }
    __syncthreads();
    const uint32_t before = carry + (warp ? warp_sums[warp - 1] : 0) + (x - v);
    if (idx < n_blocks) d.block_counts[idx] = before;
    __syncthreads();
    if (threadIdx.x == SCAN_THREADS - 1) carry = before + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) d.counters[CTR_NIW] = carry;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scatter(const DeviceBatch d) {
  __shared__ uint32_t warp_sums[32];
  const uint32_t w = d.w0 + blockIdx.x * SCAN_THREADS + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool f = (w < d.w1) && d.win_flag[w] == 1;
  const unsigned bal = __ballot_sync(FULL, f);
  if (lane == 0) warp_sums[warp] = __popc(bal);
  __syncthreads();
  if (warp == 0) {
    uint32_t s = warp_sums[lane];
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(FULL, s, o);
      if (lane >= o) s += y;
    }
    warp_sums[lane] = s;
  }
  __syncthreads();
  if (f) {
    const uint32_t pos = d.block_counts[blockIdx.x] + (warp ? warp_sums[warp - 1] : 0) + __popc(bal & ((1u << lane) - 1));
    d.iw[pos] = w;
    d.iw_out[pos] = d.win_out[w];
    d.iw_hap0[pos] = d.hap0[w];
    if (d.win_voff) d.iw_voff[pos] = d.win_voff[w];
  }
}

}  // namespace

void launch_read_decode(const DeviceBatch& d, cudaStream_t st) {
  if (d.run1 > d.run0) MPH_LAUNCH(k_read_decode, ((d.run1 - d.run0 + 3) / 4, 128, 0, st), d);
  const uint32_t n = (d.sx1 - d.sx0) + (d.fx1 - d.fx0);
  if (n) MPH_LAUNCH(k_read_patch, ((n + 255) / 256, 256, 0, st), d);
  if (d.vrun1 > d.vrun0) MPH_LAUNCH(k_side_decode, ((d.vrun1 - d.vrun0 + 3) / 4, 128, 0, st), d);
  if (d.nx1 > d.nx0) MPH_LAUNCH(k_side_patch, ((d.nx1 - d.nx0 + 255) / 256, 256, 0, st), d);
}
void launch_allele_call(const DeviceBatch& d, cudaStream_t st) {
  if (d.vr1 > d.vr0) MPH_LAUNCH(k_allele_call, ((d.vr1 - d.vr0 + 255) / 256, 256, 0, st), d);
}
void launch_window_hist(const DeviceBatch& d, cudaStream_t st) {
  if (d.c1 <= d.c0) return;
  const uint32_t nc = d.c1 - d.c0;
  if (d.mode == 1) return launch_window_hist_normal(d, st);
  if (d.it1 > d.it0) {
    const uint32_t nb = (d.it1 - d.it0 + RR_ITEMS - 1) / RR_ITEMS;
    MPH_LAUNCH(k_read_runs_plan, ((nb + 255) / 256, 256, 0, st), d, nb);
    MPH_LAUNCH(k_read_runs, (nb, RR_THREADS, 0, st), d);
  }
  static const int minb = [] { const char* e = getenv("MPH_K2B_MINB"); return e ? atoi(e) : 8; }();
  if (minb >= 10) MPH_LAUNCH(k_window_hist<10>, ((nc + K2B_WARPS - 1) / K2B_WARPS, K2B_WARPS * 32, 0, st), d);
  else MPH_LAUNCH(k_window_hist<8>, ((nc + K2B_WARPS - 1) / K2B_WARPS, K2B_WARPS * 32, 0, st), d);
  // windows with more distinct haplotypes than a lane table holds (rare): one warp per window
  MPH_LAUNCH(k_window_hist_wide, (148 * 8, K2_WARPS * 32, 0, st), d);
  launch_window_hist_block(d, st, SPQ_K2);  // ... and those with more keys than a warp table holds: one CTA per window
}
void launch_assemble(const DeviceBatch& d, cudaStream_t st, int part) {
  if (d.c1 > d.c0 && d.mode == 1) launch_assemble_normal(d, st);
  else if (d.c1 > d.c0) MPH_LAUNCH(k_assemble, (148 * 8, 128, 0, st), d, part);  // grid-stride over the key arena (its size lives on the device)
}
void launch_compact(const DeviceBatch& d, cudaStream_t st) {
  const uint32_t nb = (d.w1 - d.w0 + SCAN_THREADS - 1) / SCAN_THREADS;
  if (nb) MPH_LAUNCH(k_flag_count, (nb, SCAN_THREADS, 0, st), d);
  MPH_LAUNCH(k_block_scan, (1, SCAN_THREADS, 0, st), d, nb);
  if (nb) MPH_LAUNCH(k_scatter, (nb, SCAN_THREADS, 0, st), d);
}
thread_local uint64_t g_kernel_launches = 0;
uint64_t kernel_launches_on_this_thread() { return g_kernel_launches; }
uint32_t read_runs_blocks(uint64_t n_items) { return uint32_t((n_items + RR_ITEMS - 1) / RR_ITEMS); }

}  // namespace mphk
