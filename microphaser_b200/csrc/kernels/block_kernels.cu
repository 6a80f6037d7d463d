// block_kernels.cu — third tier of the window histogram (reference src/microphasing.rs:383-411, the BTreeMap of
// print_haplotypes): windows with more distinct haplotype keys than a warp table holds (K2_TABLE, MPH_RP_KEYS).
//
// k_window_hist_wide / k_window_hist_wide_normal / k_replay leave such a window's counted observations in the spill arena
// (one MphHist per observation or per run of normal-mode copies, count = weight; the (0, 0) key stays in c0) and queue the
// window. k_window_hist_block runs one CTA per queued window: the shared buffer holds 2 * MPH_BLOCK_KEYS entries, the first
// half the window's distinct keys so far (sorted, with their counts), the second half the next chunk of observations. The
// whole buffer is bitonic-sorted in hist_less order and equal neighbours are folded back into the first half (a block scan
// numbers the distinct keys, shared atomics sum their counts). A window's depth is therefore unbounded; more than
// MPH_BLOCK_KEYS distinct keys raises MPH_E_KEYS_PER_WINDOW. The sorted keys go to the histogram arena exactly as the warp
// tiers write them (device class from the back, host class from the front), and win_out gets n_extra / extra_off.
#include "kernel_common.cuh"

#include <atomic>

namespace mphk {

using namespace detail;

namespace {

constexpr int BK_THREADS = 1024;
constexpr uint32_t BK_BUF = 2 * MPH_BLOCK_KEYS;
constexpr uint32_t BK_PER = BK_BUF / BK_THREADS;  // consecutive buffer entries per thread in the fold
constexpr size_t BK_SMEM = BK_BUF * sizeof(MphHist);  // 128 KB
static_assert(BK_BUF % BK_THREADS == 0, "the fold gives every thread the same number of entries");

// hist_less, with the empty entries (count 0) after every key
__device__ __forceinline__ bool bk_less(const MphHist& a, const MphHist& b) {
  if ((a.count == 0) != (b.count == 0)) return b.count == 0;
  return hist_less(a, b);
}

__device__ __forceinline__ bool same_key(const MphHist& a, const MphHist& b) { return a.hap == b.hap && a.frame == b.frame; }

// bitonic sort of buf[0, n), n a power of two
__device__ void bk_sort(MphHist* buf, uint32_t n) {
  for (uint32_t k = 2; k <= n; k <<= 1)
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t t = threadIdx.x; t < n / 2; t += BK_THREADS) {
        const uint32_t i = (t / j) * 2 * j + (t % j), l = i + j;
        const MphHist a = buf[i], b = buf[l];
        const bool asc = (i & k) == 0;
        if (asc ? bk_less(b, a) : bk_less(a, b)) { buf[i] = b; buf[l] = a; }
      }
      __syncthreads();
    }
}

// exclusive block-wide prefix sum of v; *total = the sum over the block
__device__ __forceinline__ uint32_t bk_scan(uint32_t v, uint32_t* warp_sums, uint32_t* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
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
  const uint32_t before = (warp ? warp_sums[warp - 1] : 0u) + x - v;
  *total = warp_sums[31];
  __syncthreads();
  return before;
}

__global__ void __launch_bounds__(BK_THREADS) k_window_hist_block(const DeviceBatch d, const MphSpillWin* __restrict__ queue, const uint32_t* n_queued) {
  extern __shared__ MphHist buf[];
  __shared__ uint32_t warp_sums[32];
  __shared__ uint32_t s_off;
  const uint32_t nq = *n_queued;
  for (uint32_t e = blockIdx.x; e < nq; e += gridDim.x) {
    const MphSpillWin w = queue[e];
    uint32_t n_uniq = 0;
    bool too_many = false;
    for (uint32_t p0 = 0; p0 < w.n; p0 += MPH_BLOCK_KEYS) {
      const uint32_t m = min(w.n - p0, (uint32_t)MPH_BLOCK_KEYS);
      uint32_t n = 64;
      while (n < n_uniq + m) n <<= 1;
      for (uint32_t x = threadIdx.x; x < n - n_uniq; x += BK_THREADS) {
        MphHist h;
        if (x < m) h = d.spill[w.off + p0 + x];
        else { h.hap = 0; h.frame = 0; h.count = 0; }
        buf[n_uniq + x] = h;
      }
      __syncthreads();
      bk_sort(buf, n);
      // fold: thread t owns entries [t * BK_PER, (t + 1) * BK_PER); a key starts where it differs from its left neighbour
      const uint32_t x0 = threadIdx.x * BK_PER;
      MphHist v[BK_PER];
      uint32_t head_bits = 0;
      MphHist left;
      left.count = 0;
      if (x0 > 0 && x0 < n) left = buf[x0 - 1];
#pragma unroll
      for (uint32_t u = 0; u < BK_PER; ++u) {
        if (x0 + u < n) v[u] = buf[x0 + u];
        else v[u].count = 0;
        if (v[u].count != 0 && (left.count == 0 || !same_key(left, v[u]))) head_bits |= 1u << u;
        left = v[u];
      }
      uint32_t total;
      uint32_t j = bk_scan(__popc(head_bits), warp_sums, &total);  // (its barriers order the loads above before the stores below)
      if (total > MPH_BLOCK_KEYS) { too_many = true; break; }  // uniform
      uint32_t jv[BK_PER];
#pragma unroll
      for (uint32_t u = 0; u < BK_PER; ++u) {
        if (head_bits & (1u << u)) { MphHist h = v[u]; h.count = 0; buf[j] = h; ++j; }
        jv[u] = j - 1;  // the key the entry folds into
      }
      __syncthreads();
#pragma unroll
      for (uint32_t u = 0; u < BK_PER; ++u)
        if (v[u].count) atomicAdd(&buf[jv[u]].count, v[u].count);
      __syncthreads();
      n_uniq = total;
    }
    if (too_many) {
      if (threadIdx.x == 0) raise(d, MPH_E_KEYS_PER_WINDOW);
      __syncthreads();
      continue;
    }
    const MphChunk ch = d.chunks[w.code >> 5];
    const uint32_t widx = d.segs[ch.seg].win_base + ch.i_first + (w.code & 31u);
    if (threadIdx.x == 0) {
      uint32_t off = atomicAdd(&d.counters[w.devrec ? CTR_HISTD : CTR_HIST], n_uniq);
      const bool fits = off + n_uniq <= d.hist_cap;
      if (w.devrec && fits) off = d.hist_cap - off - n_uniq;  // device-class keys grow from the back of the arena
      if (!fits) raise(d, MPH_E_HIST_OVERFLOW);
      s_off = fits ? off : NONE;
      d.win_out[widx].n_extra = fits ? n_uniq : 0u;
      d.win_out[widx].extra_off = fits ? off : 0u;
    }
    __syncthreads();
    const uint32_t off = s_off;
    if (off != NONE)
      for (uint32_t x = threadIdx.x; x < n_uniq; x += BK_THREADS) {
        d.hist[off + x] = buf[x];
        d.hist_win[off + x] = w.code;
      }
    __syncthreads();
  }
}

}  // namespace

void launch_window_hist_block(const DeviceBatch& d, cudaStream_t st, int queue) {
  // 128 KB of dynamic shared memory needs an opt-in per device
  static std::atomic<uint64_t> opted{0};
  int dev = 0;
  cudaGetDevice(&dev);
  const uint64_t bit = uint64_t(1) << (dev & 63);
  if (!(opted.load() & bit)) {
    cudaFuncSetAttribute(k_window_hist_block, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BK_SMEM);
    opted.fetch_or(bit);
  }
  // one CTA per SM walks the queue; its length lives on the device, so an empty queue costs one empty launch
  const MphSpillWin* q = queue == SPQ_REPLAY ? d.spq_rp : d.spq;
  const uint32_t* n = d.counters + (queue == SPQ_REPLAY ? CTR_SPQR : CTR_SPQ);
  MPH_LAUNCH(k_window_hist_block, (148, BK_THREADS, BK_SMEM, st), d, q, n);
}

}  // namespace mphk
