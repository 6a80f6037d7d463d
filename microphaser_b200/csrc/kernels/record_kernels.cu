// record_kernels.cu — record emission on the device for the device-class transcripts (core/record_core.h):
// the emit predicate (reference src/microphasing.rs:839-844), ORF termination at the first premature stop
// (:703-718, :1480-1488), the splice-junction merge (:1497-1908, src/common.rs:376-568) and a stable,
// ordered compaction of the *records* — the host only renders text.
//
//   k_rc_flag_count / k_rc_scan / k_rc_scatter   compact the interesting windows of device-class transcripts
//   k_rc_stop     thread per such window: does one of its haplotypes remove the peptide? -> atomicMin per transcript
//   k_rc_count    thread per window: records it writes itself; lists the windows whose junction merge is due
//   k_rc_merge    warp per junction: the merge with its byte-level steps split over the lanes, into the merge arena
//   k_rc_ids      thread per merged record: its SHA-1 id
//   k_rc_scan     exclusive scan of the per-block record counts
//   k_rc_emit     thread per window: writes its records at their final, ordered positions
//
// All of it is integer / byte work on a few hundred thousand windows per shard; the kernels are latency bound and
// short next to K1-K3.
#include <cstdlib>

#include "kernel_common.cuh"
#include "phase_kernels.cuh"

#include "../core/record_core.h"

namespace mphk {

using namespace detail;

namespace {

constexpr int RC_THREADS = 512;

__device__ __forceinline__ MphRecCtx rec_ctx(const DeviceBatch& d) {
  MphRecCtx c;
  c.segs = d.segs; c.vars = d.vars; c.ref = d.ref; c.win_out = d.win_out; c.hap0 = d.hap0; c.hist = d.hist; c.hapx = d.hapx;
  c.seq = d.seq_dev; c.seq_cap = d.seq_cap; c.tx_id_bytes = d.tx_id_bytes; c.tx_id_off = d.tx_id_off;
  return c;
}

// block-wide exclusive scan of one value per thread (RC_THREADS threads); returns the exclusive prefix, *total = block sum
__device__ __forceinline__ uint32_t block_exclusive(uint32_t v, uint32_t* total) {
  __shared__ uint32_t warp_sums[RC_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t x = v;
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(FULL, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) warp_sums[warp] = x;
  __syncthreads();
  uint32_t before = 0, sum = 0;
  for (int w = 0; w < RC_THREADS / 32; ++w) {
    if (w < warp) before += warp_sums[w];
    sum += warp_sums[w];
  }
  __syncthreads();
  *total = sum;
  return before + x - v;
}

__global__ void __launch_bounds__(RC_THREADS) k_rc_flag_count(const DeviceBatch d) {
  const uint32_t w = d.w0 + blockIdx.x * RC_THREADS + threadIdx.x;
  const int f = (w < d.w1) && d.win_flag[w] == 2;
  const int n = __syncthreads_count(f);
  if (threadIdx.x == 0) d.rc_blocks[blockIdx.x] = (uint32_t)n;
}

// exclusive scan of blocks[0 .. n_blocks) in place (one CTA); total -> counters[ctr]
__global__ void __launch_bounds__(1024) k_rc_scan(const DeviceBatch d, uint32_t* blocks, uint32_t n_blocks, int ctr) {
  __shared__ uint32_t warp_sums[32];
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (uint32_t base = 0; base < n_blocks; base += 1024) {
    const uint32_t idx = base + threadIdx.x;
    const uint32_t v = idx < n_blocks ? blocks[idx] : 0;
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
    if (idx < n_blocks) blocks[idx] = before;
    __syncthreads();
    if (threadIdx.x == 1023) carry = before + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) d.counters[ctr] = carry;
}

__global__ void __launch_bounds__(RC_THREADS) k_rc_scatter(const DeviceBatch d) {
  const uint32_t w = d.w0 + blockIdx.x * RC_THREADS + threadIdx.x;
  const bool f = (w < d.w1) && d.win_flag[w] == 2;
  uint32_t total;
  const uint32_t before = block_exclusive(f ? 1u : 0u, &total);
  if (f) d.rw[d.rc_blocks[blockIdx.x] + before] = w;
}

__global__ void __launch_bounds__(RC_THREADS) k_rc_stop(const DeviceBatch d) {
  const uint32_t x = blockIdx.x * RC_THREADS + threadIdx.x;
  if (x >= d.counters[CTR_NRW]) return;
  const uint32_t w = d.rw[x];
  const MphSegment& sg = d.segs[d.win_seg[w]];
  const MphRecCtx c = rec_ctx(d);
  const uint32_t q = mph_rc_window_stop(c, sg, w - sg.win_base, w);
  d.rw_stopq[x] = q;
  if (q != NONE) atomicMin(&d.tx_stop[sg.tx], w);
}

__global__ void __launch_bounds__(RC_THREADS, 3) k_rc_count(const DeviceBatch d) {
  const uint32_t x = blockIdx.x * RC_THREADS + threadIdx.x;
  uint32_t n = 0, nb = 0;
  if (x < d.counters[CTR_NRW]) {
    const uint32_t w = d.rw[x];
    const uint32_t si = d.win_seg[w];
    const MphSegment& sg = d.segs[si];
    const uint32_t stop = d.tx_stop[sg.tx];
    uint32_t bytes = 0;
    if (w <= stop) {
      const MphRecCtx c = rec_ctx(d);
      const uint32_t i = w - sg.win_base;
      uint32_t err = 0;
      n = mph_rc_window_count(c, sg, i, w, d.rw_stopq[x], &bytes, &err);
      if (n > 0xFFFu) { err |= MPH_E_RECS_PER_LIST; n = 0; }
      // junction merge (:1497-1908): the transcript is still alive after the first window of a later exon; k_rc_merge does it
      const bool junction = i == 0 && !(sg.flags & MPH_SF_FIRST_EXON) && (sg.flags & MPH_SF_JOIN_HEAD) && w < stop && si > 0 && d.segs[si - 1].tx == sg.tx;
      if (junction) d.rw_junc[atomicAdd(&d.counters[CTR_NJ], 1u)] = x;
      raise(d, err);
    }
    d.rw_info[x] = n;
    d.rw_mbase[x] = 0;
    d.rw_bytes[x] = bytes;
    nb = bytes;
  }
  // block sums without a barrier (rc_blocks / rc_bblocks were zeroed by the host): records, and their sequence bytes
  for (int o = 16; o; o >>= 1) { n += __shfl_down_sync(FULL, n, o); nb += __shfl_down_sync(FULL, nb, o); }
  if ((threadIdx.x & 31) == 0 && n) atomicAdd(&d.rc_blocks[blockIdx.x], n);
  if ((threadIdx.x & 31) == 0 && nb) atomicAdd(&d.rc_bblocks[blockIdx.x], nb);
}

// lane-parallel byte steps of the merge: the 32 lanes of a warp run mph_rc_merge_t with identical arguments and identical
// control flow; only these steps split the bytes over the lanes
struct MphWarpOps {
  struct Win {
    uint8_t mt, wt;  // byte `lane` of the candidate's windows (window_len <= 32)
  };
  static __device__ __forceinline__ int lane() { return threadIdx.x & 31; }
  static __device__ __forceinline__ bool leader() { return lane() == 0; }
  static __device__ __forceinline__ void sync() { __syncwarp(); }
  static __device__ __forceinline__ uint64_t diff_mask(const uint8_t* a, const uint8_t* b, uint32_t n) {
    const uint32_t x = lane();
    const unsigned lo = __ballot_sync(FULL, x < n && a[x] != b[x]);
    const unsigned hi = __ballot_sync(FULL, x + 32 < n && a[x + 32] != b[x + 32]);
    return (uint64_t)lo | ((uint64_t)hi << 32);
  }
  static __device__ __forceinline__ bool window_equal(const uint8_t* ma, uint32_t man, const uint8_t* mb, uint64_t ms, const uint8_t* wa, uint32_t wan,
                                                      const uint8_t* wb, uint64_t ws, uint32_t wl) {
    const uint32_t x = lane();
    const bool ne = x < wl && mph_rc_cat(ma, man, mb, (uint32_t)(ms + x)) != mph_rc_cat(wa, wan, wb, (uint32_t)(ws + x));
    return !__any_sync(FULL, ne);
  }
  static __device__ __forceinline__ void load(Win& w, const uint8_t* ma, uint32_t man, const uint8_t* mb, uint64_t ms, const uint8_t* wa, uint32_t wan,
                                              const uint8_t* wb, uint64_t ws, uint32_t wl) {
    const uint32_t x = lane();
    w.mt = x < wl ? mph_rc_cat(ma, man, mb, (uint32_t)(ms + x)) : 0;
    w.wt = x < wl ? mph_rc_cat(wa, wan, wb, (uint32_t)(ws + x)) : 0;
  }
  static __device__ __forceinline__ bool equals_slot(const Win& w, const uint8_t* sq, uint32_t wl) {
    const uint32_t x = lane();
    const bool ne = x < wl && (sq[x] != w.mt || sq[wl + x] != w.wt);
    return !__any_sync(FULL, ne);
  }
  static __device__ __forceinline__ void store(const Win& w, uint8_t* sq, uint32_t wl) {
    const uint32_t x = lane();
    if (x < wl) { sq[x] = w.mt; sq[wl + x] = w.wt; }
  }
  static __device__ __forceinline__ bool slot_less(const uint8_t* sy, const uint8_t* sx, uint32_t n) {
    for (uint32_t base = 0; base < n; base += 32) {
      const uint32_t t = base + lane();
      const uint8_t a = t < n ? sy[t] : 0, b = t < n ? sx[t] : 0;
      const unsigned ne = __ballot_sync(FULL, a != b);
      if (ne) {
        const int first = __ffs(ne) - 1;
        return __shfl_sync(FULL, (int)a, first) < __shfl_sync(FULL, (int)b, first);
      }
    }
    return false;
  }
};

// junction merges (:1497-1908): one warp per junction; the records go to the merge arena, k_rc_emit places them
constexpr int RM_WARPS = 4;
__global__ void __launch_bounds__(RM_WARPS * 32, 8) k_rc_merge(const DeviceBatch d) {
  const int lane = threadIdx.x & 31;
  const uint32_t nj = d.counters[CTR_NJ];
  // the number of junctions lives on the device: the warps of a grid of a few CTAs per SM pull them from a queue (a merge
  // takes anything from a few hundred to tens of thousands of cycles, a static split leaves warps idle)
  for (;;) {
  uint32_t j = 0;
  if (lane == 0) j = atomicAdd(&d.counters[CTR_MQ], 1u);
  j = __shfl_sync(FULL, j, 0);
  if (j >= nj) return;
  const uint32_t x = d.rw_junc[j];
  const uint32_t w = d.rw[x];
  const uint32_t si = d.win_seg[w];
  const MphSegment& sg = d.segs[si];
  const MphSegment& sp = d.segs[si - 1];
  const MphRecCtx c = rec_ctx(d);
  uint32_t err = 0, nm = 0, mbase = 0;
  const uint32_t ub = mph_rc_merge_t<MphWarpOps>(c, sp, sg, d.window_len, nullptr, nullptr, nullptr, 0, 0, 0, &err);
  if (ub) {
    if (lane == 0) mbase = atomicAdd(&d.counters[CTR_MERGE], ub);
    mbase = __shfl_sync(FULL, mbase, 0);
    if (mbase + ub <= d.m_cap) {
      nm = mph_rc_merge_t<MphWarpOps>(c, sp, sg, d.window_len, d.m_recs + mbase, d.m_aux + mbase, d.m_seq, mbase, mbase * MPH_RC_SEQ_SLOT, ub, &err);
      for (uint32_t z = nm + lane; z < ub; z += 32) d.m_recs[mbase + z].flags = 0;  // slots the de-duplication left unused
    } else {
      err |= MPH_E_REC_OVERFLOW;
    }
  }
  if (nm > 0xFFFFFu) { err |= MPH_E_RECS_PER_LIST; nm = 0; }  // rw_info keeps 20 bits for them
  if (lane == 0) {
    d.rw_info[x] |= nm << 12;
    d.rw_mbase[x] = mbase;
    d.rw_bytes[x] += nm * 2u * d.window_len;
    if (nm) atomicAdd(&d.rc_blocks[x / RC_THREADS], nm);
    if (nm) atomicAdd(&d.rc_bblocks[x / RC_THREADS], nm * 2u * d.window_len);
    raise(d, err);
  }
  __syncwarp();
  }
}

// record ids of the junction records: one thread per slot of the merge arena (sha1 is ~4 k instructions per record; inside
// the merge it would run serially in the junction's thread)
__global__ void __launch_bounds__(128) k_rc_ids(const DeviceBatch d) {
  const uint32_t x = blockIdx.x * 128 + threadIdx.x;
  if (x >= min(d.counters[CTR_MERGE], d.m_cap)) return;
  MphRec r = d.m_recs[x];
  if (!(r.flags & MPH_RC_MERGED)) return;
  const MphRecCtx c = rec_ctx(d);
  mph_rc_merged_id(c, &r, d.m_seq + (size_t)x * MPH_RC_SEQ_SLOT, d.window_len);
  d.m_recs[x].id64 = r.id64;
}

__global__ void __launch_bounds__(RC_THREADS, 3) k_rc_emit(const DeviceBatch d) {
  if (blockIdx.x * RC_THREADS >= d.counters[CTR_NRW]) return;  // the grid covers the host's upper bound
  const uint32_t x = blockIdx.x * RC_THREADS + threadIdx.x;
  const bool live = x < d.counters[CTR_NRW];
  const uint32_t info = live ? d.rw_info[x] : 0u;
  const uint32_t n_own = info & 0xFFFu, nm = info >> 12;
  uint32_t total;
  const uint32_t before = block_exclusive(n_own + nm, &total);
  // the sequence bytes are placed by a scan as well, so that they lie in record order: the host copies the bytes of a block
  // of transcripts with one memcpy instead of one cache miss per record
  const uint32_t bytes = live ? d.rw_bytes[x] : 0u;
  const uint32_t before_bytes = block_exclusive(bytes, &total);
  if (!live || n_own + nm == 0) return;
  const uint32_t base = d.rc_blocks[blockIdx.x] + before;
  if (base + n_own + nm > d.rec_cap) { raise(d, MPH_E_REC_OVERFLOW); return; }
  const uint32_t sbase = d.rc_bblocks[blockIdx.x] + before_bytes;
  if (sbase + bytes > d.rec_seq_cap) { raise(d, MPH_E_REC_OVERFLOW); return; }
  const uint32_t w = d.rw[x];
  const MphSegment& sg = d.segs[d.win_seg[w]];
  const MphRecCtx c = rec_ctx(d);
  uint32_t err = 0;
  const uint32_t wrote = mph_rc_window_emit(c, sg, w - sg.win_base, w, d.rw_stopq[x], d.recs + base, d.rec_seq, sbase, &err);
  if (wrote != n_own) err |= MPH_E_INTERNAL;
  // the junction's records follow the window's own, in output_map order (:1877-1901)
  const uint32_t mbase = d.rw_mbase[x], wl = d.window_len;
  uint32_t spos = sbase + bytes - nm * 2u * wl;
  for (uint32_t m = 0; m < nm; ++m) {
    MphRec r = d.m_recs[mbase + m];
    const uint8_t* src = d.m_seq + (size_t)(mbase + m) * MPH_RC_SEQ_SLOT;
    for (uint32_t t = 0; t < 2u * wl; ++t) d.rec_seq[spos + t] = src[t];
    r.seq_off = spos;
    spos += 2u * wl;
    d.recs[base + n_own + r.rank] = r;
  }
  raise(d, err);
}

// ------------------------------------------------------------------ `normal` mode (src/normal_microphasing.rs)
// Every window of a device-class transcript writes records, so the kernels run over all windows of the slice (x = w - w0)
// instead of a compacted list; win_seg[w] names the window's segment (0xFFFFFFFF: host class).
__device__ __forceinline__ MphRecCtx rec_ctx_normal(const DeviceBatch& d, MphNrmCtx* n) {
  MphRecCtx c = rec_ctx(d);
  c.seq = d.seq;  // the normal-mode K3 has one sequence arena (slots of seq_cap bytes)
  n->win_depth = d.win_depth;
  n->win_id = d.win_id;
  return c;
}

__global__ void __launch_bounds__(RC_THREADS) k_nrc_stop(const DeviceBatch d) {
  const uint32_t w = d.w0 + blockIdx.x * RC_THREADS + threadIdx.x;
  if (w >= d.w1) return;
  const uint32_t si = d.win_seg[w];
  if (si == NONE) return;
  const MphSegment& sg = d.segs[si];
  MphNrmCtx n;
  const MphRecCtx c = rec_ctx_normal(d, &n);
  if (mph_nrc_window_stops(c, n, sg, w - sg.win_base, w)) atomicMin(&d.tx_stop[sg.tx], w);
}

__global__ void __launch_bounds__(RC_THREADS) k_nrc_count(const DeviceBatch d) {
  const uint32_t x = blockIdx.x * RC_THREADS + threadIdx.x, w = d.w0 + x;
  uint32_t cnt = 0, nb = 0;
  if (w < d.w1) {
    uint32_t bytes = 0;
    const uint32_t si = d.win_seg[w];
    if (si != NONE) {
      const MphSegment& sg = d.segs[si];
      const uint32_t stop = d.tx_stop[sg.tx];
      if (w <= stop) {
        MphNrmCtx n;
        const MphRecCtx c = rec_ctx_normal(d, &n);
        const uint32_t i = w - sg.win_base;
        uint32_t err = 0;
        cnt = mph_nrc_window_count(c, n, sg, i, w, &bytes, &err);
        if (cnt > 0xFFFu) { err |= MPH_E_RECS_PER_LIST; cnt = 0; }
        const bool junction = i == 0 && !(sg.flags & MPH_SF_FIRST_EXON) && w < stop && si > 0 && d.segs[si - 1].tx == sg.tx;
        if (junction) d.rw_junc[atomicAdd(&d.counters[CTR_NJ], 1u)] = x;
        raise(d, err);
      }
    }
    d.rw_info[x] = cnt;
    d.rw_mbase[x] = 0;
    d.rw_bytes[x] = bytes;
    nb = bytes;
  }
  for (int o = 16; o; o >>= 1) { cnt += __shfl_down_sync(FULL, cnt, o); nb += __shfl_down_sync(FULL, nb, o); }
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&d.rc_blocks[blockIdx.x], cnt);
  if ((threadIdx.x & 31) == 0 && nb) atomicAdd(&d.rc_bblocks[blockIdx.x], nb);
}

__global__ void __launch_bounds__(RM_WARPS * 32) k_nrc_merge(const DeviceBatch d) {
  const uint32_t j = blockIdx.x * RM_WARPS + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= d.counters[CTR_NJ]) return;
  const uint32_t x = d.rw_junc[j], w = d.w0 + x;
  const uint32_t si = d.win_seg[w];
  const MphSegment& sg = d.segs[si];
  const MphSegment& sp = d.segs[si - 1];
  MphNrmCtx n;
  const MphRecCtx c = rec_ctx_normal(d, &n);
  uint32_t err = 0, nm = 0, mbase = 0;
  const uint32_t ub = mph_nrc_merge_t<MphWarpOps>(c, n, sp, sg, d.window_len, nullptr, nullptr, nullptr, 0, 0, 0, &err);
  if (ub) {
    if (lane == 0) mbase = atomicAdd(&d.counters[CTR_MERGE], ub);
    mbase = __shfl_sync(FULL, mbase, 0);
    if (mbase + ub <= d.m_cap) {
      nm = mph_nrc_merge_t<MphWarpOps>(c, n, sp, sg, d.window_len, d.m_recs + mbase, d.m_aux + mbase, d.m_seq, mbase, mbase * MPH_RC_SEQ_SLOT, ub, &err);
      for (uint32_t z = nm + lane; z < ub; z += 32) d.m_recs[mbase + z].flags = 0;
    } else {
      err |= MPH_E_REC_OVERFLOW;
    }
  }
  if (nm > 0xFFFFFu) { err |= MPH_E_RECS_PER_LIST; nm = 0; }  // rw_info keeps 20 bits for them
  if (lane == 0) {
    d.rw_info[x] |= nm << 12;
    d.rw_mbase[x] = mbase;
    d.rw_bytes[x] += nm * d.window_len;
    if (nm) atomicAdd(&d.rc_blocks[x / RC_THREADS], nm);
    if (nm) atomicAdd(&d.rc_bblocks[x / RC_THREADS], nm * d.window_len);
    raise(d, err);
  }
}

__global__ void __launch_bounds__(RC_THREADS) k_nrc_emit(const DeviceBatch d) {
  const uint32_t x = blockIdx.x * RC_THREADS + threadIdx.x, w = d.w0 + x;
  const bool live = w < d.w1;
  const uint32_t info = live ? d.rw_info[x] : 0u;
  const uint32_t n_own = info & 0xFFFu, nm = info >> 12;
  uint32_t total;
  const uint32_t before = block_exclusive(n_own + nm, &total);
  const uint32_t bytes = live ? d.rw_bytes[x] : 0u;  // placed by a scan: record order (see k_rc_emit)
  const uint32_t before_bytes = block_exclusive(bytes, &total);
  if (!live || n_own + nm == 0) return;
  const uint32_t base = d.rc_blocks[blockIdx.x] + before;
  if (base + n_own + nm > d.rec_cap) { raise(d, MPH_E_REC_OVERFLOW); return; }
  const uint32_t sbase = d.rc_bblocks[blockIdx.x] + before_bytes;
  if (bytes && sbase + bytes > d.rec_seq_cap) { raise(d, MPH_E_REC_OVERFLOW); return; }
  const MphSegment& sg = d.segs[d.win_seg[w]];
  MphNrmCtx n;
  const MphRecCtx c = rec_ctx_normal(d, &n);
  uint32_t err = 0;
  const uint32_t wrote = mph_nrc_window_emit(c, n, sg, w - sg.win_base, w, d.recs + base, d.rec_seq, sbase, &err);
  if (wrote != n_own) err |= MPH_E_INTERNAL;
  const uint32_t mbase = d.rw_mbase[x], wl = d.window_len;
  uint32_t spos = sbase + bytes - nm * wl;
  for (uint32_t m = 0; m < nm; ++m) {
    MphRec r = d.m_recs[mbase + m];
    const uint8_t* src = d.m_seq + (size_t)(mbase + m) * MPH_RC_SEQ_SLOT;
    for (uint32_t t = 0; t < wl; ++t) d.rec_seq[spos + t] = src[t];
    r.seq_off = spos;
    spos += wl;
    d.recs[base + n_own + r.rank] = r;
  }
  raise(d, err);
}

// statistics: windows the reference reaches and the sum of depth over them (K5)
__global__ void __launch_bounds__(256) k_live_depth2(const DeviceBatch d) {
  const uint32_t chunk = d.c0 + blockIdx.x * 8 + (threadIdx.x >> 5);
  const uint32_t lane = threadIdx.x & 31;
  unsigned long long v = 0, nw = 0;
  if (chunk < d.c1) {
    const MphChunk ch = d.chunks[chunk];
    const MphSegment& sg = d.segs[ch.seg];
    if (lane < ch.n) {
      const uint32_t i = ch.i_first + lane;
      if (sg.flags & MPH_SF_DEVREC) {
        if (sg.win_base + i <= d.tx_stop[sg.tx]) { v = d.mode == 1 ? (d.win_depth[sg.win_base + i] & 0x7FFFFFFFu) : d.win_out[sg.win_base + i].depth; nw = 1; }
      } else if (d.mode == 0 && i < d.seg_live[ch.seg]) {
        v = d.win_out[sg.win_base + i].depth;
      }
    }
  }
  for (int o = 16; o; o >>= 1) { v += __shfl_down_sync(FULL, v, o); nw += __shfl_down_sync(FULL, nw, o); }
  if (lane == 0 && v) atomicAdd(d.live_depth, v);
  if (lane == 0 && nw) atomicAdd(d.live_depth + 1, nw);
}

}  // namespace

void launch_records(const DeviceBatch& d, cudaStream_t st) {
  if (d.w1 <= d.w0) return;
  const uint32_t nb = (d.w1 - d.w0 + RC_THREADS - 1) / RC_THREADS;
  if (d.mode == 1) {
    MPH_LAUNCH(k_nrc_stop, (nb, RC_THREADS, 0, st), d);
    cudaMemsetAsync(d.rc_blocks, 0, (size_t)nb * sizeof(uint32_t), st);
    cudaMemsetAsync(d.rc_bblocks, 0, (size_t)nb * sizeof(uint32_t), st);
    MPH_LAUNCH(k_nrc_count, (nb, RC_THREADS, 0, st), d);
    if (d.s1 > d.s0) MPH_LAUNCH(k_nrc_merge, ((d.s1 - d.s0 + RM_WARPS - 1) / RM_WARPS, RM_WARPS * 32, 0, st), d);
    MPH_LAUNCH(k_rc_ids, ((d.m_cap + 127) / 128, 128, 0, st), d);
    MPH_LAUNCH(k_rc_scan, (1, 1024, 0, st), d, d.rc_blocks, nb, CTR_NREC);
    MPH_LAUNCH(k_rc_scan, (1, 1024, 0, st), d, d.rc_bblocks, nb, CTR_RECSEQ);
    MPH_LAUNCH(k_nrc_emit, (nb, RC_THREADS, 0, st), d);
    return;
  }
  MPH_LAUNCH(k_rc_flag_count, (nb, RC_THREADS, 0, st), d);
  MPH_LAUNCH(k_rc_scan, (1, 1024, 0, st), d, d.rc_blocks, nb, CTR_NRW);
  MPH_LAUNCH(k_rc_scatter, (nb, RC_THREADS, 0, st), d);
  // the number of listed windows lives on the device: the grids cover the upper bound the host knows (interesting
  // windows of the slice cannot exceed its windows); threads beyond the count return at once
  const uint32_t nbl = nb;
  MPH_LAUNCH(k_rc_stop, (nbl, RC_THREADS, 0, st), d);
  cudaMemsetAsync(d.rc_blocks, 0, (size_t)nbl * sizeof(uint32_t), st);
  cudaMemsetAsync(d.rc_bblocks, 0, (size_t)nbl * sizeof(uint32_t), st);
  MPH_LAUNCH(k_rc_count, (nbl, RC_THREADS, 0, st), d);
  static const uint32_t merge_ctas = [] { const char* e = getenv("MPH_MERGE_CTAS"); return e ? (uint32_t)atoi(e) : 148u * 8u; }();  // 0: a warp per segment
  if (d.s1 > d.s0) MPH_LAUNCH(k_rc_merge, (std::min<uint32_t>((d.s1 - d.s0 + RM_WARPS - 1) / RM_WARPS, merge_ctas ? merge_ctas : 0xFFFFFFFFu), RM_WARPS * 32, 0, st), d);  // at most one junction per segment
  MPH_LAUNCH(k_rc_ids, ((d.m_cap + 127) / 128, 128, 0, st), d);
  MPH_LAUNCH(k_rc_scan, (1, 1024, 0, st), d, d.rc_blocks, nbl, CTR_NREC);
  MPH_LAUNCH(k_rc_scan, (1, 1024, 0, st), d, d.rc_bblocks, nbl, CTR_RECSEQ);
  MPH_LAUNCH(k_rc_emit, (nbl, RC_THREADS, 0, st), d);
}

void launch_live_depth(const DeviceBatch& d, cudaStream_t st) {
  if (d.c1 > d.c0) MPH_LAUNCH(k_live_depth2, ((d.c1 - d.c0 + 7) / 8, 256, 0, st), d);
}

}  // namespace mphk
