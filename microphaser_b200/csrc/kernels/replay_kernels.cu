// replay_kernels.cu — serial replay of the ObservationMatrix for the transcripts the closed form does not cover
// (core/replay_core.h states the steps; reference src/microphasing.rs:220-343,1119-1343 and, for the normal mode,
// src/normal_microphasing.rs:238-331,1001).
#include "kernel_common.cuh"

namespace mphk {

using namespace detail;

namespace {

// ------------------------------------------------------------------ serial replay
// One warp per irregular transcript. The matrix operations of one transcript are a strict sequence
// (core/replay_core.h: mph_replay_tx is the single-threaded statement of the same steps and what the
// CPU emulator runs); within one step the observations are independent, so the lanes stride over
// them. The observation list lives in shared memory (it spills to a global scratch slice if a
// window is deeper than RP_OBS), the segment's variant positions are cached in shared memory, and
// the read cursors move incrementally, so an iteration costs one global round trip.
static_assert((int)MPH_RP_CTR_HIST == (int)CTR_HIST && (int)MPH_RP_CTR_ERR == (int)CTR_ERR && (int)MPH_RP_CTR_VLIST == (int)CTR_VLIST,
              "mph_replay_tx counts in the kernels' counter words");
constexpr int RP_WARPS = 1;
constexpr int RP_OBS = 512;
constexpr int RP_READS = 640;  // reads of one exon's candidate range cached in shared memory (single-exon units)
constexpr int RP_POS = 256;
constexpr int RP_STOPW = 24;  // stop-codon bitmap words cached per segment

struct RpShared {
  uint64_t o_hap[RP_OBS];
  uint32_t o_read[RP_OBS], o_key[RP_OBS], o_frame[RP_OBS];
  uint8_t o_flags[RP_OBS];
  uint32_t rs[RP_READS], re[RP_READS];
  uint8_t rf[RP_READS], im[RP_READS];
  uint32_t pos[RP_POS];
  uint32_t stop[RP_STOPW];
  uint32_t dq[MPH_RP_MAXCOLS], dqpos[MPH_RP_MAXCOLS];
  MphHist table[MPH_RP_KEYS];
  MphSegment sg;
};

// first index in [lo, hi) with a[idx] >= target (hi if none): the tile around the previous answer is tried before a binary search;
// two lower bounds over the same array with their loads issued together (one round trip in the common case)
__device__ __forceinline__ void warp_lb2(const uint32_t* __restrict__ a, uint32_t lo, uint32_t hi, uint32_t t0, uint32_t t1, uint32_t* c0, uint32_t* c1,
                                         int lane) {
  uint32_t g0 = *c0 > lo + 16u ? *c0 - 16u : lo, g1 = *c1 > lo + 16u ? *c1 - 16u : lo;
  if (g0 > hi) g0 = hi;
  if (g1 > hi) g1 = hi;
  const uint32_t i0 = g0 + lane, i1 = g1 + lane;
  const uint32_t v0 = i0 < hi ? a[i0] : 0xFFFFFFFFu, v1 = i1 < hi ? a[i1] : 0xFFFFFFFFu;
  const uint32_t p0 = g0 > lo ? a[g0 - 1] : 0u, p1 = g1 > lo ? a[g1 - 1] : 0u;
  const unsigned b0 = __ballot_sync(FULL, i0 >= hi || v0 >= t0), b1 = __ballot_sync(FULL, i1 >= hi || v1 >= t1);
  *c0 = ((g0 == lo || p0 < t0) && b0) ? g0 + (uint32_t)__ffs(b0) - 1u : mph_u32_lb(a, lo, hi, t0);
  *c1 = ((g1 == lo || p1 < t1) && b1) ? g1 + (uint32_t)__ffs(b1) - 1u : mph_u32_lb(a, lo, hi, t1);
}

__device__ __forceinline__ void replay_unit(const DeviceBatch& d, const uint32_t ti, RpShared& sh, const int lane) {
  const MphReplayTx t = d.replay[ti];
  MphReplayCtx c;
  c.read_start = d.read_start; c.read_end = d.read_end; c.read_flags = d.read_flags;
  c.read_vlo = d.read_vlo; c.read_nv = d.read_nv; c.read_vr = d.read_vr;
  c.vr_seq_off = d.vr_seq_off; c.vr_cig_off = d.vr_cig_off; c.vr_lseq = d.vr_lseq; c.vr_ncig = d.vr_ncig;
  c.bases = d.bases; c.cigars = d.cigars; c.call_S = d.call_S; c.call_B = d.call_B;
  c.pairs = reinterpret_cast<const uint32_t*>(d.pairs); c.n_pairs = d.n_pairs;
  c.vars = d.vars; c.segs = d.segs; c.seg_chunk0 = d.seg_chunk0; c.stopmap = d.stopmap; c.ref = d.ref;
  c.dq_init = d.dq_init;
  c.mode = 0; c.tx_id_bytes = nullptr; c.tx_id_off = nullptr; c.win_depth = nullptr; c.win_id = nullptr; c.o_last = nullptr; c.seg_err = d.seg_err;
  c.o_read = nullptr; c.o_hap = nullptr; c.o_frame = nullptr; c.o_flags = nullptr; c.o_inmat = d.o_inmat;
  c.win_out = d.win_out; c.hist = d.hist; c.hist_win = d.hist_win; c.hist_cap = d.hist_cap;
  c.key_cap = d.force_wide == 2 ? 0u : (uint32_t)MPH_RP_KEYS;
  c.hap0 = d.hap0; c.win_flag = d.win_flag; c.win_voff = d.win_voff; c.vlist = d.vlist; c.vlist_cap = d.vlist_cap;
  c.counters = d.counters; c.sum_depth = d.sum_depth;
  // observation list: shared memory first, generic pointers so that it can move to the global scratch slice
  uint64_t* o_hap = sh.o_hap;
  uint32_t *o_read = sh.o_read, *o_key = sh.o_key, *o_frame = sh.o_frame;
  uint8_t* o_flags = sh.o_flags;
  uint32_t o_cap = RP_OBS;
  // read-side arrays, indexed by the global read number: global memory, or (single-exon units whose candidate
  // range fits) shared-memory copies addressed through shifted pointers
  const uint32_t* rs = d.read_start;
  const uint32_t* re = d.read_end;
  const uint8_t* rf = d.read_flags;
  uint8_t* in_mat = d.o_inmat + t.obs_off - t.read_lo;
  uint32_t r_lo = t.read_lo, r_hi = t.read_hi;
  bool reads_cached = false;
  if (t.seg_hi - t.seg_lo == 1) {
    const MphSegment sg0 = d.segs[t.seg_lo];
    const MphGeom ga = mph_geom(sg0, 0), gz = mph_geom(sg0, sg0.n_iter ? sg0.n_iter - 1 : 0);
    const bool rv = (sg0.flags & MPH_SF_REVERSE) != 0;
    const uint32_t s_lo = rv ? min(ga.s, gz.s) : ga.s, s_hi = max(ga.s, gz.s);
    const uint32_t c_lo = mph_u32_lb(d.read_start, t.read_lo, t.read_hi, s_lo > sg0.K ? s_lo - sg0.K : 0u);
    const uint32_t c_hi = mph_u32_lb(d.read_start, c_lo, t.read_hi, s_hi + 1u);
    if (c_hi - c_lo <= RP_READS) {
      for (uint32_t x = lane; x < c_hi - c_lo; x += 32) {
        const uint32_t r = c_lo + x;
        sh.rs[x] = d.read_start[r]; sh.re[x] = d.read_end[r]; sh.rf[x] = d.read_flags[r]; sh.im[x] = 0;
      }
      rs = sh.rs - c_lo; re = sh.re - c_lo; rf = sh.rf - c_lo; in_mat = sh.im - c_lo;
      c.read_start = rs; c.read_end = re; c.read_flags = rf;
      r_lo = c_lo; r_hi = c_hi;
      reads_cached = true;
    }
  }
  if (!reads_cached)
    for (uint32_t x = lane; x < t.obs_cap; x += 32) in_mat[t.read_lo + x] = 0;
  uint32_t err = 0, ncols = t.dq_n <= MPH_RP_MAXCOLS ? t.dq_n : 0u, n_obs = 0;
  if (t.dq_n > MPH_RP_MAXCOLS) err |= MPH_E_VARS_PER_WINDOW;
  const uint32_t key_cap = d.force_wide == 2 ? 0u : (uint32_t)MPH_RP_KEYS;
  for (uint32_t j = lane; j < ncols; j += 32) sh.dq[j] = d.dq_init[t.dq_off + j];
  uint64_t last_window_vars = t.last_vars;
  uint32_t cur_lo = r_lo, cur_hi = r_lo;
  uint32_t vl_cur = 0, vl_end = 0;        // slice of the column-list arena owned by this warp
  unsigned long long depth_sum = 0;       // lane 0
  uint32_t key_bound = 0;                 // forward: min end over the observations, reverse: max start (cleanup is skipped when it cannot remove anything)
  for (uint32_t j = lane; j < ncols; j += 32) sh.dqpos[j] = d.vars[sh.dq[j]].pos;
  __syncwarp();

  bool panicked = false;  // uniform: the reference panics here (drain out of range, inverted BTreeMap range)
  auto shrink_left = [&](uint64_t n) -> bool {  // :220-229
    if (n > ncols) { panicked = true; return false; }
    if (n) {
      const uint32_t a = lane + (uint32_t)n, b = lane + 32 + (uint32_t)n;
      const uint32_t x0 = a < ncols ? sh.dq[a] : 0u, x1 = b < ncols ? sh.dq[b] : 0u;
      const uint32_t y0 = a < ncols ? sh.dqpos[a] : 0u, y1 = b < ncols ? sh.dqpos[b] : 0u;
      __syncwarp();
      if (a < ncols) { sh.dq[lane] = x0; sh.dqpos[lane] = y0; }
      if (b < ncols) { sh.dq[lane + 32] = x1; sh.dqpos[lane + 32] = y1; }
      ncols -= (uint32_t)n;
      const uint64_t mask = ncols >= 64 ? ~(uint64_t)0 : (((uint64_t)1 << ncols) - 1);
      for (uint32_t o = lane; o < n_obs; o += 32) o_hap[o] &= mask;
      __syncwarp();
    }
    return true;
  };

  for (uint32_t si = t.seg_lo; si < t.seg_hi; ++si) {
    __syncwarp();
    if (lane < (int)(sizeof(MphSegment) / 4)) reinterpret_cast<uint32_t*>(&sh.sg)[lane] = reinterpret_cast<const uint32_t*>(&d.segs[si])[lane];
    __syncwarp();
    const MphSegment& sg = sh.sg;
    const bool rev = (sg.flags & MPH_SF_REVERSE) != 0;
    const bool is_short = (sg.flags & MPH_SF_SHORT) != 0;
    // variant positions of the exon: every window of the segment lies inside [exon_start, exon_end]
    const uint32_t vs_lo = mph_var_lb(d.vars, sg.var_lo, sg.var_hi, sg.exon_start);
    const uint32_t vs_hi = mph_var_lb(d.vars, vs_lo, sg.var_hi, sg.exon_end + 1u);
    const uint32_t n_pos = vs_hi - vs_lo;
    const bool cached = n_pos <= RP_POS;
    if (cached)
      for (uint32_t x = lane; x < n_pos; x += 32) sh.pos[x] = d.vars[vs_lo + x].pos;
    // stop-codon bitmap words of the segment's reference slice
    const uint32_t sw0 = sg.ref_off >> 5, sw_n = ((sg.ref_off + sg.ref_len) >> 5) - sw0 + 3;
    const bool stop_cached = sw_n <= RP_STOPW;
    if (stop_cached && lane < (int)sw_n) sh.stop[lane] = d.stopmap[sw0 + lane];
    const uint32_t* stopmap_seg = stop_cached ? sh.stop - sw0 : d.stopmap;
    __syncwarp();
    auto lbpos = [&](uint64_t x) -> uint32_t {  // first variant index with pos >= x
      if (!cached || x < sg.exon_start || x > (uint64_t)sg.exon_end + 1u) return mph_var_lb(d.vars, sg.var_lo, sg.var_hi, (uint32_t)x);
      uint32_t lo = 0, hi = n_pos;
      while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (sh.pos[mid] < (uint32_t)x) lo = mid + 1;
        else hi = mid;
      }
      return vs_lo + lo;
    };
    if (!shrink_left(last_window_vars)) {  // :1024
      if (lane == 0) d.seg_err[si] = 1;
      break;
    }
    last_window_vars = 0;
    uint64_t old_offset = sg.off0, old_end = (uint64_t)sg.off0 + sg.ewl;
    bool reached_end = false;
    uint32_t prev_va = vs_lo, prev_vb = vs_lo;
    uint32_t emit_k = sg.k_first, emit_i = 0;  // next enumerated window
    bool deferred = false;            // folded iterations are waiting to be offered
    uint32_t pushed_s = 0;            // forward strand: window start of the last iteration whose reads were offered
    uint32_t prev_s = 0, prev_e = 0;  // geometry of the last folded iteration
    // cleanup_reads (:259-278): in-place compaction, a tile is read completely before it is written
    auto do_cleanup = [&](uint32_t gs, uint32_t ge) {
     if (n_obs && (rev ? key_bound > gs : key_bound < ge)) {
      uint32_t w = 0, kb = rev ? 0u : 0xFFFFFFFFu;
      for (uint32_t base = 0; base < n_obs; base += 32) {
        const uint32_t o = base + lane;
        const bool valid = o < n_obs;
        uint32_t r = 0, key = 0, fr = 0;
        uint64_t hp = 0;
        uint8_t fl = 0;
        if (valid) { r = o_read[o]; key = o_key[o]; hp = o_hap[o]; fr = o_frame[o]; fl = o_flags[o]; }
        const bool keep = valid && (rev ? key < gs + 1u : key >= ge);
        if (valid && !keep) in_mat[r] = 0;
        const unsigned bal = __ballot_sync(FULL, keep);
        __syncwarp();
        if (keep) {
          const uint32_t p = w + __popc(bal & ((1u << lane) - 1));
          o_read[p] = r; o_key[p] = key; o_hap[p] = hp; o_frame[p] = fr; o_flags[p] = fl;
          kb = rev ? max(kb, key) : min(kb, key);
        }
        w += __popc(bal);
        __syncwarp();
      }
      n_obs = w;
      key_bound = rev ? __reduce_max_sync(FULL, kb) : __reduce_min_sync(FULL, kb);
    }
    };
    // candidate reads (:1191-1249) and push_read (:297-343); `lo` = smallest start that is offered
    auto do_push = [&](uint32_t gs, uint32_t ge, uint32_t lo) {
      warp_lb2(rs, r_lo, r_hi, lo, gs + 1u, &cur_lo, &cur_hi, lane);
      if (cur_hi < cur_lo) cur_hi = cur_lo;
      for (uint32_t base4 = cur_lo; base4 < cur_hi; base4 += 128) {
       // the loads of four tiles are issued before any of them is processed
       uint32_t en4[4];
       uint8_t im4[4], rf4[4];
#pragma unroll
       for (int j = 0; j < 4; ++j) {
         const uint32_t rj = base4 + 32 * j + lane;
         const bool in = rj < cur_hi;
         en4[j] = in ? re[rj] : 0u;
         im4[j] = (in && rev) ? in_mat[rj] : (uint8_t)0;
         rf4[j] = (in && rev) ? rf[rj] : (uint8_t)0;
       }
#pragma unroll
       for (int j = 0; j < 4; ++j) {
        const uint32_t base = base4 + 32 * j;
        if (base >= cur_hi) break;
        const uint32_t r = base + lane;
        bool cand = r < cur_hi && en4[j] >= ge;
        if (cand && rev) {
          // `contains` (:281-294): the read itself or the read sharing its (start, qname) is in the matrix already
          bool dup = im4[j] != 0;
          if (!dup && (rf4[j] & MPH_RF_PARTNER)) {
            // the reads sharing (start, qname) form a cycle of partner edges (two of them point at each other). Whatever makes
            // one of them a duplicate makes this read one as well, so only their own push test matters
            uint32_t q = mph_rp_partner(c, r);
            for (uint32_t hops = 0; !dup && q != NONE && q != r && hops < 4096; ++hops) {
              if (q >= r_lo && q < r_hi) {
                dup = in_mat[q] != 0;
                if (!dup && q < r && q >= cur_lo && re[q] >= ge) {  // offered just before r in this same iteration
                  uint64_t hq = 0;
                  uint32_t fq = 0;
                  uint8_t lq = 0;
                  for (uint32_t i = 0; i < ncols; ++i) mph_rp_update(c, t, q, i, sh.dq[ncols - 1 - i], &hq, &fq, &lq, &err);
                  dup = !(lq & 1);
                }
              }
              q = mph_rp_partner(c, q);
            }
          }
          cand = !dup;
        }
        uint64_t hap = 0;
        uint32_t frame = 0;
        uint8_t fl = 0;
        if (cand) {
          for (uint32_t i = 0; i < ncols; ++i) mph_rp_update(c, t, r, i, sh.dq[ncols - 1 - i], &hap, &frame, &fl, &err);
          if (fl & 1) cand = false;  // rejected at push (:338)
        }
        const unsigned bal = __ballot_sync(FULL, cand);
        const uint32_t n_in = __popc(bal);
        bool drop = false;  // uniform
        if (n_in && n_obs + n_in > o_cap) {
          if (o_hap == sh.o_hap && n_obs + n_in <= t.obs_cap) {  // move the list to its global scratch slice
            uint64_t* g_hap = d.o_hap + t.obs_off;
            uint32_t *g_read = d.o_read + t.obs_off, *g_key = d.o_key + t.obs_off, *g_frame = d.o_frame + t.obs_off;
            uint8_t* g_flags = d.o_flags + t.obs_off;
            for (uint32_t o = lane; o < n_obs; o += 32) { g_hap[o] = o_hap[o]; g_read[o] = o_read[o]; g_key[o] = o_key[o]; g_frame[o] = o_frame[o]; g_flags[o] = o_flags[o]; }
            o_hap = g_hap; o_read = g_read; o_key = g_key; o_frame = g_frame; o_flags = g_flags;
            o_cap = t.obs_cap;
            __syncwarp();
          } else {
            err |= MPH_E_REPLAY_INPUT;
            drop = true;
          }
        }
        if (n_in && !drop) {
          uint32_t kk = rev ? 0u : 0xFFFFFFFFu;
          if (cand) {
            const uint32_t p = n_obs + __popc(bal & ((1u << lane) - 1));
            kk = rev ? rs[r] : en4[j];
            o_read[p] = r; o_key[p] = kk; o_hap[p] = hap; o_frame[p] = frame; o_flags[p] = fl;
            in_mat[r] = 1;
          }
          if (rev) key_bound = n_obs ? max(key_bound, __reduce_max_sync(FULL, kk)) : __reduce_max_sync(FULL, kk);
          else key_bound = n_obs ? min(key_bound, __reduce_min_sync(FULL, kk)) : __reduce_min_sync(FULL, kk);
          n_obs += n_in;
        }
        __syncwarp();
       }
      }
    };
    for (uint32_t k = 0; k < sg.n_iter; ++k) {
      const uint64_t offset = rev ? (uint64_t)sg.off0 - k : (uint64_t)sg.off0 + k;
      const MphGeom g = mph_geom(sg, k);
      const uint64_t rest = rev ? offset - sg.exon_start : sg.exon_end - (offset + sg.ewl);
      const bool is_last_exon_window = rest < 3, is_first_exon_window = k == 0;
      // for k >= 1 old_offset / old_end are the previous window's start / end, so every variant_tree.range count
      // (:1119-1170) is a difference of the previous and the current lower bounds; an inverted range panics
      uint32_t va, vb;
      if (k == 0 || !cached) { va = lbpos(g.s); vb = lbpos(g.e); }
      else {
        va = prev_va; vb = prev_vb;
        while (va < vs_hi && sh.pos[va - vs_lo] < g.s) ++va;
        while (va > vs_lo && sh.pos[va - 1 - vs_lo] >= g.s) --va;
        while (vb < vs_hi && sh.pos[vb - vs_lo] < g.e) ++vb;
        while (vb > vs_lo && sh.pos[vb - 1 - vs_lo] >= g.e) --vb;
      }
      const uint64_t nvars = vb - va;
      uint64_t added_vars, deleted_vars;
      if (is_first_exon_window) added_vars = nvars;
      else if (is_short || reached_end) added_vars = 0;
      else if (g.s > old_offset) { if (old_end > g.e) panicked = true; added_vars = vb - prev_vb; }
      else { if (g.s > old_offset) panicked = true; added_vars = prev_va - va; }
      if (offset == old_offset || is_short) deleted_vars = 0;
      else if (g.s > old_offset) deleted_vars = va - prev_va;
      else { if (g.e > old_end) panicked = true; deleted_vars = prev_vb - vb; }
      prev_va = va; prev_vb = vb;
      if (is_last_exon_window) reached_end = true;
      if (panicked) {
        if (lane == 0) d.seg_err[si] = k + 1;
        break;
      }
      // Folding: an iteration that neither adds nor removes a column and is not an enumerated window only offers reads;
      // offering them all at once just before the next iteration that does something gives the same matrix (a read
      // offered at a folded iteration and still alive afterwards passes the same tests against the same columns). The
      // first two iterations are never folded: the candidate range changes shape there. core/replay_core.h states it.
      const uint64_t skip_cnt = nvars - added_vars;  // wraps like the release build: nothing is added then
      const uint32_t n_new_now = skip_cnt <= nvars ? (uint32_t)(nvars - skip_cnt) : 0u;
      const bool emit_now = k == emit_k && emit_i < sg.n_win;
      if (k >= 2 && !emit_now && n_new_now == 0 && deleted_vars == 0 && !is_short) {
        deferred = true;
        prev_s = g.s; prev_e = g.e;
        last_window_vars = nvars;
        old_offset = g.s;
        old_end = g.e;
        continue;
      }
      if (deferred && deleted_vars > 0) {  // the folded reads must meet the columns as they were before this iteration's shrink_left
        do_cleanup(prev_s, prev_e);
        do_push(prev_s, prev_e, rev ? (prev_s > sg.K ? prev_s - sg.K : 0u) : pushed_s + 1u);
        pushed_s = prev_s;
      }
      deferred = false;
      do_cleanup(g.s, g.e);
      if (!shrink_left(deleted_vars)) {
        if (lane == 0) d.seg_err[si] = k + 1;
        break;
      }
      {
        const bool wide = rev || offset == (uint64_t)sg.exon_start + sg.ceo;
        uint32_t lo = wide ? (g.s > sg.K ? g.s - sg.K : 0u) : g.s;
        if (!wide && k >= 2) lo = pushed_s + 1u;  // everything since the last offered start
        do_push(g.s, g.e, lo);
        pushed_s = g.s;
      }
      // newly collected variants (:1280-1296) and extend_right (:232-256)
      {
        const uint64_t skip = nvars - added_vars;  // wraps like the release build: nothing is added then
        const uint32_t n_new = skip <= nvars ? (uint32_t)(nvars - skip) : 0u;
        if (n_new) {
          if (ncols + n_new > MPH_RP_MAXCOLS) { err |= MPH_E_VARS_PER_WINDOW; break; }
          for (uint32_t o = lane; o < n_obs; o += 32) {
            uint64_t hap = o_hap[o] << (n_new & 63u);
            uint32_t frame = o_frame[o];
            uint8_t fl = o_flags[o];
            const uint32_t r = o_read[o];
            for (uint32_t i = 0; i < n_new; ++i) {
              const uint32_t x = (uint32_t)skip + (n_new - 1 - i);
              mph_rp_update(c, t, r, i, rev ? vb - 1 - x : va + x, &hap, &frame, &fl, &err);
            }
            o_hap[o] = hap; o_frame[o] = frame; o_flags[o] = fl;
          }
          for (uint32_t x = (uint32_t)skip + lane; x < (uint32_t)nvars; x += 32) {
            const uint32_t v = rev ? vb - 1 - x : va + x;
            sh.dq[ncols + (x - (uint32_t)skip)] = v;
            sh.dqpos[ncols + (x - (uint32_t)skip)] = d.vars[v].pos;
          }
          ncols += n_new;
          __syncwarp();
        }
      }
      last_window_vars = nvars;
      if (k == emit_k && emit_i < sg.n_win) {
        // histogram of print_haplotypes (:383-411) and the window's outputs
        const uint32_t i = emit_i;
        emit_k += sg.k_stride;
        ++emit_i;
        const uint32_t widx = sg.win_base + i;
        uint32_t n_keys = 0, c0 = 0, n_spill = 0;
        bool spill = false;  // lane 0: a key did not fit the table (the window goes to k_window_hist_block)
        for (uint32_t base = 0; base < n_obs; base += 32) {
          const uint32_t o = base + lane;
          const bool valid = o < n_obs && !(o_flags[o] & 1);
          const uint64_t hap = valid ? o_hap[o] : 0;
          const uint32_t fr = valid ? o_frame[o] : 0;
          const bool zero_key = valid && hap == 0 && fr == 0;
          c0 += __popc(__ballot_sync(FULL, zero_key));
          unsigned pending = __ballot_sync(FULL, valid && !zero_key);
          n_spill += __popc(pending);
          if (__shfl_sync(FULL, (int)spill, 0)) continue;
          while (pending) {
            const int leader = __ffs(pending) - 1;
            const uint64_t lh = __shfl_sync(FULL, hap, leader);
            const uint32_t lf = __shfl_sync(FULL, fr, leader);
            const unsigned same = __ballot_sync(FULL, valid && !zero_key && hap == lh && fr == lf);
            if (lane == 0 && !spill) {
              uint32_t x = 0;
              for (; x < n_keys; ++x)
                if (sh.table[x].hap == lh && sh.table[x].frame == lf) break;
              if (x == n_keys) {
                if (n_keys < key_cap) {
                  sh.table[x].hap = lh; sh.table[x].frame = lf; sh.table[x].count = 0;
                  ++n_keys;
                } else {
                  spill = true;
                }
              }
              if (!spill) sh.table[x].count += __popc(same);
            }
            pending &= ~same;
          }
        }
        n_keys = __shfl_sync(FULL, n_keys, 0);
        if (__shfl_sync(FULL, (int)spill, 0)) {
          // the counted observations outside the (0, 0) key go to the spill arena; the window to the replay's queue
          uint32_t off = 0;
          if (lane == 0) off = atomicAdd(&d.counters[CTR_SPILL], n_spill);
          off = __shfl_sync(FULL, off, 0);
          if ((uint64_t)off + n_spill <= d.spill_cap) {
            uint32_t y = off;
            for (uint32_t base = 0; base < n_obs; base += 32) {
              const uint32_t o = base + lane;
              const bool valid = o < n_obs && !(o_flags[o] & 1);
              const uint64_t hap = valid ? o_hap[o] : 0;
              const uint32_t fr = valid ? o_frame[o] : 0;
              const bool emit = valid && !(hap == 0 && fr == 0);
              const unsigned bal = __ballot_sync(FULL, emit);
              if (emit) {
                MphHist e;
                e.hap = hap; e.count = 1; e.frame = fr;
                d.spill[y + __popc(bal & ((1u << lane) - 1u))] = e;
              }
              y += __popc(bal);
            }
            if (lane == 0) {
              MphSpillWin q;
              q.code = ((d.seg_chunk0[si] + (i >> 5)) << 5) | (i & 31u); q.off = off; q.n = n_spill; q.devrec = 0;  // replayed transcripts are host class
              d.spq_rp[atomicAdd(&d.counters[CTR_SPQR], 1u)] = q;
            }
          } else {
            err |= MPH_E_SPILL_OVERFLOW;
          }
          n_keys = 0;  // k_window_hist_block writes the keys and sets n_extra / extra_off
        }
        if (vl_cur + ncols + 1 > vl_end) {  // a fresh slice of the column-list arena (one atomic per ~256 entries)
          uint32_t got = 0;
          const uint32_t want = max(256u, ncols + 1);
          if (lane == 0) got = atomicAdd(&d.counters[CTR_VLIST], want);
          vl_cur = __shfl_sync(FULL, got, 0);
          vl_end = vl_cur + want;
        }
        const uint32_t voff = vl_cur;
        vl_cur += ncols + 1;
        if (lane == 0) {
          for (uint32_t a = 1; a < n_keys; ++a) {
            const MphHist key = sh.table[a];
            uint32_t b = a;
            while (b > 0 && hist_less(key, sh.table[b - 1])) { sh.table[b] = sh.table[b - 1]; --b; }
            sh.table[b] = key;
          }
          MphWinOut wo;
          wo.depth = n_obs; wo.c0 = c0; wo.n_extra = n_keys; wo.extra_off = 0;
          if (n_keys) {
            const uint32_t off = atomicAdd(&d.counters[CTR_HIST], n_keys);
            if (off + n_keys <= d.hist_cap) {
              wo.extra_off = off;
              const uint32_t code = ((d.seg_chunk0[si] + (i >> 5)) << 5) | (i & 31u);
              for (uint32_t a = 0; a < n_keys; ++a) { d.hist[off + a] = sh.table[a]; d.hist_win[off + a] = code; }
            } else {
              err |= MPH_E_HIST_OVERFLOW;
              wo.n_extra = 0;
            }
          }
          d.win_out[widx] = wo;
          depth_sum += n_obs;
          // variants the sequence walk visits (:473-476): j only advances while variants[j].pos == i
          uint32_t j = 0;
          for (uint32_t p = g.s; p < g.e && j < ncols; ++p)
            while (j < ncols && (rev ? sh.dqpos[ncols - 1 - j] : sh.dqpos[j]) == p) ++j;
          MphHap h0;
          err |= mph_plain_hap(sg, g, stopmap_seg, d.ref, j, &h0);
          if (ncols > 32) err |= MPH_E_VARS_PER_WINDOW;
          d.hap0[widx] = h0;
          d.win_flag[widx] = 1;
        }
        if (voff + ncols + 1 <= d.vlist_cap) {
          if (lane == 0) { d.vlist[voff] = ncols; d.win_voff[widx] = voff; }
          for (uint32_t j = lane; j < ncols; j += 32) d.vlist[voff + 1 + j] = rev ? sh.dq[ncols - 1 - j] : sh.dq[j];
        } else {
          err |= MPH_E_VLIST_OVERFLOW;
        }
        __syncwarp();
      }
      old_offset = g.s;
      old_end = g.e;
      if (is_short) break;
    }
    if (!panicked && deferred && si + 1 < t.seg_hi) {  // folded iterations at the end of the exon: their reads may survive into the next one
      do_cleanup(prev_s, prev_e);
      do_push(prev_s, prev_e, rev ? (prev_s > sg.K ? prev_s - sg.K : 0u) : pushed_s + 1u);
    }
    if (panicked || __any_sync(FULL, (err & (MPH_E_REPLAY_PANIC | MPH_E_VARS_PER_WINDOW)) != 0)) break;
  }
  if (lane == 0 && depth_sum) atomicAdd(d.sum_depth, depth_sum);
  raise(d, err);
}

// Persistent launch: a few single-warp CTAs per SM pull units from a queue (counters[CTR_RPQ]) until it is empty. A unit is
// a dependent chain of a few hundred iterations, so the kernel is as long as its longest warp whatever the grid; a small
// grid leaves the registers and shared memory of every SM to the window / record kernels that run beside it on the main
// stream (capi.cu: the replay and everything that depends on it form a side chain).
__global__ void __launch_bounds__(RP_WARPS * 32, 20) k_replay(const DeviceBatch d) {
  __shared__ RpShared sh_all[RP_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  RpShared& sh = sh_all[warp];
  for (;;) {
    uint32_t q = 0;
    if (lane == 0) q = atomicAdd(&d.counters[CTR_RPQ], 1u);
    q = __shfl_sync(FULL, q, 0);
    const uint32_t ti = d.rp0 + q;
    if (ti >= d.rp1) return;
    replay_unit(d, ti, sh, lane);
    __syncwarp();
  }
}

// Normal mode: the same replay with the normal-mode matrix (every re-offered copy is kept, entries are
// (read, haplotype, copies)). The normal-mode residue writes a record for every window, so this path is far from the
// critical one; lane 0 of a warp runs the single-threaded statement of core/replay_core.h per unit.
__global__ void __launch_bounds__(64) k_replay_normal(const DeviceBatch d) {
  const uint32_t ti = d.rp0 + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (ti >= d.rp1 || (threadIdx.x & 31)) return;
  MphReplayCtx c;
  c.read_start = d.read_start; c.read_end = d.read_end; c.read_flags = d.read_flags;
  c.read_vlo = d.read_vlo; c.read_nv = d.read_nv; c.read_vr = d.read_vr;
  c.vr_seq_off = d.vr_seq_off; c.vr_cig_off = d.vr_cig_off; c.vr_lseq = d.vr_lseq; c.vr_ncig = d.vr_ncig;
  c.bases = d.bases; c.cigars = d.cigars; c.call_S = d.call_S; c.call_B = d.call_B;
  c.pairs = reinterpret_cast<const uint32_t*>(d.pairs); c.n_pairs = d.n_pairs;
  c.vars = d.vars; c.segs = d.segs; c.seg_chunk0 = d.seg_chunk0; c.stopmap = d.stopmap; c.ref = d.ref; c.dq_init = d.dq_init;
  c.mode = 1; c.tx_id_bytes = d.tx_id_bytes; c.tx_id_off = d.tx_id_off; c.win_depth = d.win_depth; c.win_id = d.win_id; c.o_last = d.o_key;
  c.o_read = d.o_read; c.o_hap = d.o_hap; c.o_frame = d.o_frame; c.o_flags = d.o_flags; c.o_inmat = d.o_inmat;
  c.win_out = d.win_out; c.hist = d.hist; c.hist_win = d.hist_win; c.hist_cap = d.hist_cap;
  c.key_cap = d.force_wide == 2 ? 0u : (uint32_t)MPH_RP_KEYS;
  c.hap0 = d.hap0; c.win_flag = d.win_flag; c.win_voff = d.win_voff; c.vlist = d.vlist; c.vlist_cap = d.vlist_cap;
  c.seg_err = d.seg_err; c.counters = d.counters; c.sum_depth = d.sum_depth;
  mph_replay_tx(c, d.replay[ti]);
}

}  // namespace

void launch_replay(const DeviceBatch& d, cudaStream_t st, uint32_t max_ctas) {
  if (d.rp1 <= d.rp0) return;
  if (d.mode == 1) MPH_LAUNCH(k_replay_normal, ((d.rp1 - d.rp0 + 1) / 2, 64, 0, st), d);
  else MPH_LAUNCH(k_replay, (std::min<uint32_t>((d.rp1 - d.rp0 + RP_WARPS - 1) / RP_WARPS, max_ctas ? max_ctas : 0xFFFFFFFFu), RP_WARPS * 32, 0, st), d);
  // somatic: replayed windows with more keys than the warp's table holds (the normal-mode replay sorts them in the key arena)
  if (d.mode == 0) launch_window_hist_block(d, st, SPQ_REPLAY);
}

}  // namespace mphk
