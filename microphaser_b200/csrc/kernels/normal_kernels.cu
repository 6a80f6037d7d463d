// normal_kernels.cu — window and assembly kernels of the `normal` mode (reference src/normal_microphasing.rs).
#include "kernel_common.cuh"

namespace mphk {

using namespace detail;

namespace {

// ------------------------------------------------------------------ normal mode (src/normal_microphasing.rs)
// The matrix of the normal mode keeps every copy of a re-offered read on the reverse strand
// (cleanup_reads(splice_side_offset) :1001, no `contains`), so an observation count is a ramp in the
// iteration number: a read contributes k - kc + 1 copies from its entry iteration kc until the window
// start reaches its own start, where the older copies are dropped. Phase A therefore keeps two
// difference arrays (slope and constant); the histogram only needs the reads that support an allele.
constexpr int KN_LANE_KEYS = 6;

__device__ __forceinline__ void normal_window_out(const DeviceBatch& d, const MphSegment& sg, uint32_t seg, const MphGeom& g, uint32_t widx, uint32_t nvar,
                                                  uint32_t depth) {
  MphHap h0;
  const uint32_t err = mph_nrm_plain(sg, g, d.ref, nvar, &h0);
  d.win_depth[widx] = depth | ((nvar == 0 && (h0.flags & MPH_NF_STOP)) ? 0x80000000u : 0u);
  // every window's reference haplotype is written by the host (:509-645): its record id is hashed here
  unsigned long long id = 0;
  if (!(h0.flags & MPH_NF_REFRANGE)) {
    const uint32_t t0 = d.tx_id_off[sg.tx];
    id = mph_record_id64(d.ref + sg.ref_off + (g.s - sg.ref_pos0), g.e - g.s, d.tx_id_bytes + t0, d.tx_id_off[sg.tx + 1] - t0, g.s);
  }
  d.win_id[widx] = id;
  // device-class transcripts: the record kernels take every window (they find its segment in win_seg); the host sees none of them
  const bool devrec = (sg.flags & MPH_SF_DEVREC) != 0;
  d.win_flag[widx] = nvar > 0 ? (devrec ? 2 : 1) : 0;
  d.win_seg[widx] = devrec ? seg : NONE;
  if (nvar) d.hap0[widx] = h0;
  raise(d, err);
}

// entry iteration of a reverse-strand read (first k with s(k) <= start + K and e(k) <= end), independent of the window
__device__ __forceinline__ uint32_t normal_rev_kc(const MphSegment& sg, uint32_t st, uint32_t en) {
  const uint64_t lim = (uint64_t)st + sg.K;
  uint32_t kc = sg.off0 > lim ? (uint32_t)(sg.off0 - lim) : 0;
  if (mph_geom(sg, 0).e > en) {
    const uint64_t t = (uint64_t)sg.off0 + sg.ewl;
    const uint32_t k2 = t > en ? (uint32_t)(t - en) : 1;
    if (k2 > kc) kc = k2;
    if (kc == 0) kc = 1;
  }
  kc = kc >= 2 ? kc - 2 : 0;
  for (; kc < sg.n_iter; ++kc) {
    const MphGeom gc = mph_geom(sg, kc);
    if (gc.s <= lim && gc.e <= en) break;
  }
  return kc;
}

// one warp per window whose keys overflow a lane table; a window with more keys than the warp table holds walks its reads a
// second time and hands its haplotypes to k_window_hist_block (as in window_hist_warp of phase_kernels.cu)
__device__ void window_hist_warp_normal(const DeviceBatch& d, const MphSegment& sg, uint32_t ch_seg, uint32_t i, uint32_t code, MphHist* table, int lane) {
  const bool rev = (sg.flags & MPH_SF_REVERSE) != 0;
  const uint32_t k = sg.k_first + i * sg.k_stride;
  const uint32_t widx = sg.win_base + i;
  const MphGeom g = mph_geom(sg, k);
  const uint32_t va = mph_var_lb(d.vars, sg.var_lo, sg.var_hi, g.s);
  const uint32_t vb = mph_var_lb(d.vars, va, sg.var_hi, g.e);
  uint32_t rlo, rhi;
  mph_candidate_range(sg, d.read_start, g, &rlo, &rhi);
  // the copies of read r in the matrix; S != 0: they need their haplotypes
  auto observe = [&](uint32_t r, uint32_t* copies, uint32_t* kp_last, uint32_t* vlo, uint64_t* S) {
    *copies = 0; *kp_last = k; *vlo = 0; *S = 0;
    if (r >= rhi) return;
    const uint32_t st = d.read_start[r], en = d.read_end[r];
    if (!rev) {
      const uint32_t kp = mph_nrm_fwd_entry(sg, k, g, st, en);
      if (kp != NONE) { *copies = 1; *kp_last = kp; }
    } else {
      uint32_t kc;
      *copies = mph_nrm_rev_copies(sg, k, g, st, en, &kc);
    }
    if (*copies && (d.call_flags[r] & 1u)) { *S = d.call_S[r]; *vlo = d.read_vlo[r]; }  // S is only written for reads with a call
  };
  const uint32_t key_cap = d.force_wide == 2 ? 0u : (uint32_t)K2_TABLE;
  uint32_t depth = 0, c0 = 0, n_keys = 0, n_spill = 0;
  bool spill = false;  // lane 0: a key did not fit the table
  for (uint32_t base = rlo; base < rhi; base += 32) {
    uint32_t copies, kp_last, vlo;
    uint64_t S;
    observe(base + lane, &copies, &kp_last, &vlo, &S);
    uint32_t cs = copies;
    for (int o = 16; o; o >>= 1) cs += __shfl_xor_sync(FULL, cs, o);
    depth += cs;
    const uint32_t plain = (S == 0) ? copies : 0;
    uint32_t ps = plain;
    for (int o = 16; o; o >>= 1) ps += __shfl_xor_sync(FULL, ps, o);
    c0 += ps;
    uint32_t todo = (S != 0) ? copies : 0, maxc = todo;
    for (int o = 16; o; o >>= 1) maxc = max(maxc, __shfl_xor_sync(FULL, maxc, o));
    for (uint32_t c = 0; c < maxc; ++c) {
      const bool have = c < todo;
      uint64_t hap = 0;
      if (have) hap = mph_nrm_hap(sg, d.vars, rev ? k - c : kp_last, k, va, vb, vlo, S);
      c0 += __popc(__ballot_sync(FULL, have && hap == 0));
      unsigned pending = __ballot_sync(FULL, have && hap != 0);
      n_spill += __popc(pending);
      if (__shfl_sync(FULL, (int)spill, 0)) continue;
      while (pending) {
        const int leader = __ffs(pending) - 1;
        const uint64_t lh = __shfl_sync(FULL, hap, leader);
        const unsigned same = __ballot_sync(FULL, have && hap == lh);
        if (lane == 0 && !spill) {
          uint32_t t = 0;
          for (; t < n_keys; ++t)
            if (table[t].hap == lh) break;
          if (t == n_keys) {
            if (n_keys < key_cap) {
              table[t].hap = lh;
              table[t].frame = 0;
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
  }
  if (__shfl_sync(FULL, (int)spill, 0)) {
    uint32_t off = 0;
    if (lane == 0) off = atomicAdd(&d.counters[CTR_SPILL], n_spill);
    off = __shfl_sync(FULL, off, 0);
    if ((uint64_t)off + n_spill <= d.spill_cap) {
      uint32_t y = off;
      for (uint32_t base = rlo; base < rhi; base += 32) {
        uint32_t copies, kp_last, vlo;
        uint64_t S;
        observe(base + lane, &copies, &kp_last, &vlo, &S);
        uint32_t todo = (S != 0) ? copies : 0, maxc = todo;
        for (int o = 16; o; o >>= 1) maxc = max(maxc, __shfl_xor_sync(FULL, maxc, o));
        for (uint32_t c = 0; c < maxc; ++c) {
          const bool have = c < todo;
          uint64_t hap = 0;
          if (have) hap = mph_nrm_hap(sg, d.vars, rev ? k - c : kp_last, k, va, vb, vlo, S);
          const bool emit = have && hap != 0;
          const unsigned bal = __ballot_sync(FULL, emit);
          if (emit) {
            MphHist e;
            e.hap = hap; e.count = 1; e.frame = 0;
            d.spill[y + __popc(bal & ((1u << lane) - 1u))] = e;
          }
          y += __popc(bal);
        }
      }
      if (lane == 0) {
        MphSpillWin q;
        q.code = code; q.off = off; q.n = n_spill; q.devrec = 0;  // normal mode: every key sits at the front of the arena
        d.spq[atomicAdd(&d.counters[CTR_SPQ], 1u)] = q;
      }
    } else if (lane == 0) {
      raise(d, MPH_E_SPILL_OVERFLOW);
    }
    n_keys = 0;  // k_window_hist_block writes the keys and sets n_extra / extra_off
  }
  if (lane == 0) {
    for (uint32_t a = 1; a < n_keys; ++a) {  // ascending haplotype value (VecMap iteration order :383)
      const MphHist key = table[a];
      uint32_t b = a;
      while (b > 0 && key.hap < table[b - 1].hap) {
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
      const uint32_t off = atomicAdd(&d.counters[CTR_HIST], n_keys);
      if (off + n_keys <= d.hist_cap) {
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
    normal_window_out(d, sg, ch_seg, g, widx, vb - va, depth);
  }
  __syncwarp();
}

__global__ void __launch_bounds__(K2_WARPS * 32) k_window_hist_wide_normal(const DeviceBatch d) {
  __shared__ MphHist table[K2_WARPS][K2_TABLE];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t n = d.counters[CTR_OVF];
  for (uint32_t o = blockIdx.x * K2_WARPS + warp; o < n; o += gridDim.x * K2_WARPS) {
    const uint32_t code = d.ovf_list[o];
    const MphChunk ch = d.chunks[code >> 5];
    const MphSegment sg = d.segs[ch.seg];
    window_hist_warp_normal(d, sg, ch.seg, ch.i_first + (code & 31u), code, table[warp], lane);
  }
}

__global__ void __launch_bounds__(K2_WARPS * 32) k_window_hist_normal(const DeviceBatch d) {
  __shared__ uint64_t t_hap[K2_WARPS][KN_LANE_KEYS][32];
  __shared__ uint32_t t_cnt[K2_WARPS][KN_LANE_KEYS][32];
  __shared__ MphSegment s_seg[K2_WARPS];
  __shared__ uint32_t s_s[K2_WARPS][32], s_e[K2_WARPS][32];
  __shared__ int s_add[K2_WARPS][34], s_slope[K2_WARPS][34];
  __shared__ uint32_t s_list[K2_WARPS][K2_LIST];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t chunk = d.c0 + blockIdx.x * K2_WARPS + warp;
  if (chunk >= d.c1) return;
  const MphChunk ch = d.chunks[chunk];
  if (lane < (int)(sizeof(MphSegment) / 4)) reinterpret_cast<uint32_t*>(&s_seg[warp])[lane] = reinterpret_cast<const uint32_t*>(&d.segs[ch.seg])[lane];
  s_add[warp][lane] = 0;
  s_slope[warp][lane] = 0;
  if (lane < 2) { s_add[warp][32 + lane] = 0; s_slope[warp][32 + lane] = 0; }
  __syncwarp();
  const MphSegment& sg = s_seg[warp];
  if (sg.flags & MPH_SF_REPLAY) return;  // the whole transcript goes through k_replay_normal
  const bool rev = (sg.flags & MPH_SF_REVERSE) != 0;
  const int n = (int)ch.n;
  const bool active = lane < n;
  const uint32_t i = ch.i_first + (active ? lane : 0);
  const uint32_t k = sg.k_first + i * sg.k_stride;
  const MphGeom g = mph_geom(sg, k);
  const uint32_t va = mph_var_lb(d.vars, ch.va0, ch.vb1, g.s);
  const uint32_t vb = mph_var_lb(d.vars, va, ch.vb1, g.e);
  const uint32_t nvar = vb - va;
  if (active && nvar > 64) raise(d, MPH_E_VARS_PER_WINDOW);
  const bool chunk_has_var = ch.vb1 > ch.va0;
  s_s[warp][lane] = g.s;
  s_e[warp][lane] = g.e;
  const uint32_t s0 = sg.off0 - sg.ceo;
  const uint32_t rlo = ch.rlo, rhi = ch.rhi;
  const int64_t c1_lo = (int64_t)s0 - (int64_t)sg.K;
  const int k_base = (int)(sg.k_first + ch.i_first * sg.k_stride);  // iteration number of lane 0
  uint32_t n_keys = 0;
  int c0_adj = 0;
  bool overflow = false;
  __syncwarp();
  auto add_key = [&](uint64_t hap) {
    uint32_t t = 0;
    for (; t < n_keys; ++t)
      if (t_hap[warp][t][lane] == hap) break;
    if (t == n_keys) {
      if (n_keys == KN_LANE_KEYS || d.force_wide) { overflow = true; return; }
      t_hap[warp][t][lane] = hap;
      t_cnt[warp][t][lane] = 0;
      ++n_keys;
    }
    t_cnt[warp][t][lane] += 1;
  };
  // phase B body (lane = window): copies of the listed reads, one haplotype per copy
  auto process_list = [&](uint32_t list_n) {
    if (!active || nvar == 0) return;
    for (uint32_t x = 0; x < list_n; ++x) {
      const uint32_t r = s_list[warp][x];
      const uint32_t st = d.read_start[r], en = d.read_end[r], vlo = d.read_vlo[r];
      const uint64_t S = d.call_S[r];
      if (!rev) {
        const uint32_t kp = mph_nrm_fwd_entry(sg, k, g, st, en);
        if (kp == NONE) continue;
        const uint64_t hap = mph_nrm_hap(sg, d.vars, kp, k, va, vb, vlo, S);
        if (hap) { c0_adj -= 1; add_key(hap); }
      } else {
        uint32_t kc;
        const uint32_t copies = mph_nrm_rev_copies(sg, k, g, st, en, &kc);
        for (uint32_t c = 0; c < copies; ++c) {
          const uint64_t hap = mph_nrm_hap(sg, d.vars, k - c, k, va, vb, vlo, S);
          if (hap) { c0_adj -= 1; add_key(hap); }
        }
      }
    }
  };
  // ---- phase A (lane = read)
  uint32_t list_n = 0;
  const uint32_t* ss = s_s[warp];
  const uint32_t* se = s_e[warp];
  for (uint32_t base = rlo; base < rhi; base += 32) {
    const uint32_t r = base + lane;
    bool need = false;
    if (r < rhi) {
      const uint32_t st = d.read_start[r], en = d.read_end[r];
      int ilo = 1, ihi = 0;
      if (!rev) {
        int a = 0, b = n;  // e non-decreasing: windows with e <= en form a prefix
        while (a < b) { const int m = (a + b) >> 1; if (se[m] <= en) a = m + 1; else b = m; }
        ihi = a - 1;
        if (st <= s0) {
          ilo = ((int64_t)st >= c1_lo) ? 0 : n;
        } else if (st <= sg.off0) {
          ilo = n;
        } else {
          const uint32_t k_ins = st - sg.off0;
          const uint32_t t = k_ins > sg.k_first ? (k_ins - sg.k_first + sg.k_stride - 1) / sg.k_stride : 0;
          ilo = t > ch.i_first ? (int)min(t - ch.i_first, (uint32_t)n) : 0;
        }
        if (ilo <= ihi) {
          atomicAdd(&s_add[warp][ilo], 1);
          atomicAdd(&s_add[warp][ihi + 1], -1);
          need = true;
        }
      } else {
        const uint32_t kc = normal_rev_kc(sg, st, en);
        const uint32_t t = kc > sg.k_first ? (kc - sg.k_first + sg.k_stride - 1) / sg.k_stride : 0;
        ilo = t > ch.i_first ? (int)min(t - ch.i_first, (uint32_t)n) : 0;
        int a = 0, b = n;  // s non-increasing: windows with s >= st form a prefix
        while (a < b) { const int m = (a + b) >> 1; if (ss[m] >= st) a = m + 1; else b = m; }
        ihi = a - 1;
        a = 0; b = n;      // windows with s > st
        while (a < b) { const int m = (a + b) >> 1; if (ss[m] > st) a = m + 1; else b = m; }
        const int iramp = a - 1;
        if (ilo <= iramp) {  // copies(j) = stride * j + (k_base - kc + 1)
          const int cst = k_base - (int)kc + 1;
          atomicAdd(&s_slope[warp][ilo], (int)sg.k_stride);
          atomicAdd(&s_slope[warp][iramp + 1], -(int)sg.k_stride);
          atomicAdd(&s_add[warp][ilo], cst);
          atomicAdd(&s_add[warp][iramp + 1], -cst);
          need = true;
        }
        const int elo = max(ilo, iramp + 1);
        if (elo <= ihi) {  // window start == read start: the older copies have just been dropped
          atomicAdd(&s_add[warp][elo], 1);
          atomicAdd(&s_add[warp][ihi + 1], -1);
          need = true;
        }
      }
      need = need && chunk_has_var && (d.call_flags[r] & 1u) && d.call_S[r] != 0;
    }
    const unsigned nm = __ballot_sync(FULL, need);
    if (nm) {
      if (list_n + __popc(nm) > K2_LIST) {
        __syncwarp();
        process_list(list_n);
        list_n = 0;
        __syncwarp();
      }
      if (need) s_list[warp][list_n + __popc(nm & ((1u << lane) - 1))] = r;
      list_n += __popc(nm);
      __syncwarp();
    }
  }
  __syncwarp();
  process_list(list_n);
  // ---- phase B: prefix sums of the two difference arrays
  int run = s_add[warp][lane], slope = s_slope[warp][lane];
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(FULL, run, o), z = __shfl_up_sync(FULL, slope, o);
    if (lane >= o) { run += y; slope += z; }
  }
  const uint32_t depth = (uint32_t)(run + slope * lane);
  const uint32_t c0 = (uint32_t)((int)depth + c0_adj);
  for (uint32_t a = 1; a < n_keys; ++a) {  // ascending haplotype value
    const uint64_t kh = t_hap[warp][a][lane];
    const uint32_t kc = t_cnt[warp][a][lane];
    uint32_t b = a;
    while (b > 0 && kh < t_hap[warp][b - 1][lane]) {
      t_hap[warp][b][lane] = t_hap[warp][b - 1][lane];
      t_cnt[warp][b][lane] = t_cnt[warp][b - 1][lane];
      --b;
    }
    t_hap[warp][b][lane] = kh;
    t_cnt[warp][b][lane] = kc;
  }
  const bool ovf = active && overflow;
  const uint32_t mine = (active && !ovf) ? n_keys : 0;
  uint32_t incl = mine;
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(FULL, incl, o);
    if (lane >= o) incl += y;
  }
  const uint32_t total = __shfl_sync(FULL, incl, 31);
  uint32_t base_off = 0;
  if (lane == 0 && total) base_off = atomicAdd(&d.counters[CTR_HIST], total);
  base_off = __shfl_sync(FULL, base_off, 0);
  const bool fits = base_off + total <= d.hist_cap;
  if (lane == 0 && total && !fits) raise(d, MPH_E_HIST_OVERFLOW);
  if (active && !ovf) {
    MphWinOut wo;
    wo.depth = depth;
    wo.c0 = c0;
    wo.n_extra = fits ? mine : 0;
    wo.extra_off = base_off + incl - mine;
    if (fits)
      for (uint32_t a = 0; a < mine; ++a) {
        MphHist h;
        h.hap = t_hap[warp][a][lane]; h.frame = 0; h.count = t_cnt[warp][a][lane];
        d.hist[wo.extra_off + a] = h;
        d.hist_win[wo.extra_off + a] = (chunk << 5) | (uint32_t)lane;
      }
    const uint32_t widx = sg.win_base + i;
    d.win_out[widx] = wo;
    normal_window_out(d, sg, ch.seg, g, widx, nvar, depth);
  }
  if (ovf) {
    const uint32_t o = atomicAdd(&d.counters[CTR_OVF], 1u);
    d.ovf_list[o] = (chunk << 5) | (uint32_t)lane;
  }
  unsigned long long dsum = (active && !ovf) ? depth : 0;
  for (int o = 16; o; o >>= 1) dsum += __shfl_down_sync(FULL, dsum, o);
  if (lane == 0 && dsum) atomicAdd(d.sum_depth, dsum);
}

// thread per haplotype key != 0: the sequence walk of the normal-mode print_haplotypes (:403-507);
// every haplotype of a variant window is written by the host, so every sequence is kept
__global__ void __launch_bounds__(128) k_assemble_normal(const DeviceBatch d) {
  const uint32_t n = min(d.counters[CTR_HIST], d.hist_cap);
  uint8_t seq[MAX_SEQ_CAP];
  const uint32_t cap = d.seq_cap;
  for (uint32_t x = blockIdx.x * blockDim.x + threadIdx.x; x < n; x += gridDim.x * blockDim.x) {
    const MphHist key = d.hist[x];
    const uint32_t code = d.hist_win[x];
    const MphChunk ch = d.chunks[code >> 5];
    const MphSegment sg = d.segs[ch.seg];
    const uint32_t i = ch.i_first + (code & 31u);
    const uint32_t k = sg.k_first + i * sg.k_stride;
    const MphGeom g = mph_geom(sg, k);
    const uint32_t va = mph_var_lb(d.vars, ch.va0, ch.vb1, g.s);
    const uint32_t vb = mph_var_lb(d.vars, va, ch.vb1, g.e);
    const uint32_t depth = d.win_out[sg.win_base + i].depth;
    MphHap out;
    uint32_t err;
    if (!(sg.flags & MPH_SF_REPLAY)) {
      err = mph_nrm_assemble(sg, g, d.vars, va, vb, d.ref, d.ins_bytes, key.hap, key.count == depth, seq, cap, &out);
    } else {
      MphVar cols[MPH_RP_MAXCOLS];
      const uint32_t off = d.win_voff[sg.win_base + i];
      const uint32_t ncol = off == NONE ? 0u : min(d.vlist[off], (uint32_t)MPH_RP_MAXCOLS);
      for (uint32_t j = 0; j < ncol; ++j) cols[j] = d.vars[d.vlist[off + 1 + j]];
      err = mph_nrm_assemble(sg, g, cols, 0, ncol, d.ref, d.ins_bytes, key.hap, key.count == depth, seq, cap, &out);
    }
    if (out.seq_len <= cap) {
      const uint32_t t0 = d.tx_id_off[sg.tx];
      out.id64 = mph_record_id64(seq, out.seq_len, d.tx_id_bytes + t0, d.tx_id_off[sg.tx + 1] - t0, g.s);
      out.flags |= MPH_NF_ID;
    }
    const uint32_t off = atomicAdd(&d.counters[CTR_SEQ], cap);
    if (off + cap <= d.seq_cap_bytes) {
      const uint32_t sl = out.seq_len < cap ? out.seq_len : cap;
      for (uint32_t t = 0; t < sl; ++t) d.seq[off + t] = seq[t];
      out.seq_off = off;
      out.flags |= MPH_NF_SEQ;
    } else {
      err |= MPH_E_SEQ_OVERFLOW;
    }
    d.hapx[x] = out;
    raise(d, err);
  }
}

}  // namespace

void launch_window_hist_normal(const DeviceBatch& d, cudaStream_t st) {
  const uint32_t nc = d.c1 - d.c0;
  MPH_LAUNCH(k_window_hist_normal, ((nc + K2_WARPS - 1) / K2_WARPS, K2_WARPS * 32, 0, st), d);
  // windows with more distinct haplotypes than a lane table holds (rare): one warp per window
  MPH_LAUNCH(k_window_hist_wide_normal, (148 * 8, K2_WARPS * 32, 0, st), d);
  launch_window_hist_block(d, st, SPQ_K2);  // ... and those with more keys than a warp table holds: one CTA per window
}
void launch_assemble_normal(const DeviceBatch& d, cudaStream_t st) {
  MPH_LAUNCH(k_assemble_normal, (148 * 8, 128, 0, st), d);  // grid-stride over the key arena (its size lives on the device)
}

}  // namespace mphk
