// capi.cu — implementation of include/microphaser_gpu.h: packer, device pipeline (H2D, K1-K4, D2H),
// host residue, writers and the file-level `somatic` driver. No CPU fallback: every phase call runs
// the CUDA kernels of kernels/phase_kernels.cu or fails.
#include <cuda_runtime.h>
#include <malloc.h>
#include <cstring>
#include <unistd.h>

#include <condition_variable>
#include <deque>
#include <mutex>
#include <unordered_map>
#include <chrono>
#include <cstdarg>
#include <fstream>
#include <iostream>
#include <memory>
#include <optional>
#include <thread>
#include <utility>

#include "../../include/microphaser_gpu.h"
#include "host/cli.hpp"
#include "host/peptides_host.hpp"
#include "host/records_host.hpp"
#include "host/shard_pipeline.hpp"
#include "host/synth_files.hpp"
#include "kernels/inflate_kernels.cuh"
#include "kernels/peptide_kernels.cuh"
#include "kernels/phase_kernels.cuh"

using namespace mph;

namespace {

thread_local std::string g_last_error;

struct CudaError : std::runtime_error {
  using std::runtime_error::runtime_error;
};

#define CU(call)                                                                                          \
  do {                                                                                                    \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess) throw CudaError(std::string(#call) + ": " + cudaGetErrorString(e_));          \
  } while (0)

template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;
  void ensure(size_t n) {
    if (n <= cap) return;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = n + n / 8 + 64;
    CU(cudaMalloc(&p, want * sizeof(T)));
    cap = want;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  ~DevBuf() { release(); }
};

// Device-side BGZF inflate for the file drivers (kernels/inflate_kernels.cu): the compressed batch goes up, one warp per
// block inflates it, the inflated batch comes back into the reader's buffer. Installed in the BGZF reader as its batch
// inflater; any failure (no memory, a block the decoder rejects) throws and the reader falls back to zlib on the host.
struct GpuInflater {
  int device = 0;
  cudaStream_t st = nullptr;
  DevBuf<uint8_t> d_in, d_out;
  DevBuf<MphRawBlock> d_blk;
  DevBuf<uint32_t> d_status;
  std::vector<MphRawBlock> h_blk;
  double ms_total = 0;
  size_t batches = 0, bytes_in = 0, bytes_out = 0;
  explicit GpuInflater(int dev) : device(dev) {}
  GpuInflater(const GpuInflater&) = delete;
  GpuInflater& operator=(const GpuInflater&) = delete;
  ~GpuInflater() {
    cudaSetDevice(device);
    if (st) cudaStreamDestroy(st);
  }
  void run(const uint8_t* cbuf, size_t cbytes, const mphio::BgzfRaw* raws, size_t n, uint8_t* out, size_t obytes) {
    const auto t0 = std::chrono::steady_clock::now();
    CU(cudaSetDevice(device));
    if (!st) CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    if (cbytes > 0xFFFFFF00ull || obytes > 0xFFFFFF00ull) throw std::runtime_error("BGZF batch too large for the device inflate");
    h_blk.resize(n);
    for (size_t i = 0; i < n; ++i) {
      if (raws[i].coff + raws[i].clen > cbytes || raws[i].ooff + raws[i].isize > obytes) throw std::runtime_error("BGZF block out of its batch");
      h_blk[i] = MphRawBlock{uint32_t(raws[i].coff), uint32_t(raws[i].clen), uint32_t(raws[i].ooff), uint32_t(raws[i].isize)};
    }
    d_in.ensure(cbytes + 16); d_out.ensure(obytes + 16); d_blk.ensure(n + 1); d_status.ensure(1);
    CU(cudaMemcpyAsync(d_in.p, cbuf, cbytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_blk.p, h_blk.data(), n * sizeof(MphRawBlock), cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(d_status.p, 0, sizeof(uint32_t), st));
    mphk::launch_bgzf_inflate(d_in.p, d_blk.p, uint32_t(n), d_out.p, d_status.p, st);
    CU(cudaGetLastError());
    uint32_t status = 0;
    if (obytes) CU(cudaMemcpyAsync(out, d_out.p, obytes, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&status, d_status.p, sizeof status, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (status) throw std::runtime_error("device inflate: DEFLATE error " + std::to_string(status));
    ms_total += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    batches += 1; bytes_in += cbytes; bytes_out += obytes;
  }
};

}  // namespace

struct mph_batch {
  Batch b;
  std::vector<uint2> pairs;
  bool pinned = false;
  std::vector<std::pair<void*, size_t>> registered;
  uint64_t h2d_bytes = 0;
  int span_mode = 0;  // bus form of the read spans (host/batch.hpp: bus_span_mode), fixed when the batch is finished
  ~mph_batch() {
    for (auto& r : registered) cudaHostUnregister(r.first);
  }
};

struct mph_packer {
  std::unique_ptr<Packer> p;
  int mode = 0;
};

// One block of consecutive transcripts of a result. Records of host-class transcripts arrive as text-ready OutRecords
// from the host residue; records of device-class transcripts stay in the compact form the record kernels produced
// (core/record_core.h) and are rendered when they are read or written.
struct ResultPart {
  std::vector<OutRecord> host;   // ascending transcript
  std::vector<MphRec> dev;       // ascending transcript; a transcript is in exactly one of the two
  std::vector<uint8_t> dev_seq;
  std::vector<MphRecSrc> dev_aux;
  std::vector<OutRecord> rendered;  // all records of the part in order, built on first access through mph_result_get
  std::once_flag once;
  size_t size() const { return host.size() + dev.size(); }
};

struct mph_result {
  int mode = 0;
  // records in the reference's order: the transcript blocks of the residue threads, kept as they were produced
  std::deque<ResultPart> parts;
  std::vector<uint64_t> part_base;  // prefix counts, parts.size() + 1 entries
  uint64_t size() const { return part_base.empty() ? 0 : part_base.back(); }
  std::vector<std::string> tx_id, gene_id, gene_name, chrom;
  std::vector<uint8_t> tx_reverse;
  // what rendering a device-built record needs of the batch
  std::vector<MphVar> vars;
  std::vector<std::string> var_prot;
  std::vector<uint8_t> ref;  // normal mode: the reference arena (records of reference windows point into it)

  RenderCtx ctx_of(const ResultPart& p) const {
    RenderCtx c;
    c.vars = vars.data(); c.var_prot = &var_prot; c.seq = p.dev_seq.data(); c.aux = p.dev_aux.data(); c.ref = ref.data();
    return c;
  }
  // calls f(const OutRecord&) for every record of the part in transcript order; device-built ones are rendered on the fly
  template <class F>
  void for_each(const ResultPart& p, F&& f) const {
    if (!p.rendered.empty() || p.size() == 0) { for (auto& r : p.rendered) f(r); return; }
    const RenderCtx rc = ctx_of(p);
    size_t h = 0, d = 0;
    while (h < p.host.size() || d < p.dev.size()) {
      const bool take_dev = h == p.host.size() || (d < p.dev.size() && p.dev[d].tx < p.host[h].info.tx);
      if (take_dev) { const OutRecord r = render_record(rc, p.dev[d++]); f(r); }
      else f(p.host[h++]);
    }
  }
  const OutRecord& at(uint64_t i) {
    const size_t pi = size_t(std::upper_bound(part_base.begin(), part_base.end(), i) - part_base.begin()) - 1;
    ResultPart& p = parts[pi];
    std::call_once(p.once, [&] {
      std::vector<OutRecord> all;
      all.reserve(p.size());
      for_each(p, [&](const OutRecord& r) { all.push_back(r); });
      p.rendered = std::move(all);
    });
    return p.rendered[size_t(i - part_base[pi])];
  }
};

struct mph_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;       // compute + device -> host
  cudaStream_t copy_stream = nullptr;  // host -> device of the next stage
  cudaStream_t replay_stream = nullptr;  // the serial replay of irregular transcripts runs beside the window kernels
  cudaEvent_t ev_rp[5] = {};           // K1 done (main) / replay start / replay done / host-class K3 start / side chain done
  int sm_count = 148;
  std::vector<cudaEvent_t> ev_copy;
  uint32_t stage_seg_lo = 0, stage_seg_hi = 0, stage_tx_lo = 0, stage_tx_hi = 0;
  bool replay_on_side = false;         // the last run_kernels put k_replay on replay_stream (its time comes from ev_rp)
  bool side_chain = false;             // ... followed there by the host-class K3 walk and K4 (somatic mode)
  bool kernels_done = false;           // mph_phase_resident ran for the uploaded batch: mph_phase_collect only downloads
  cudaEvent_t ev[10] = {};
  std::string last_error;
  const mph_batch* cur = nullptr;
  mphk::DeviceBatch d;
  DevBuf<uint32_t> read_start, read_end, read_vlo, read_vr, vr_read, vr_vlo, vr_seq_off, vr_cig_off, cigars, block_counts, iw, counters, seg_live, ovf_list, stopmap, hist_win, win_depth, seg_chunk0, dq_init, seg_err, tx_id_off, o_read, o_key, o_frame, win_voff, vlist, iw_voff, seg_work_off, seg_list_n, rr_seg0;
  DevBuf<uint16_t> vr_lseq, vr_ncig;
  DevBuf<uint8_t> tx_id_bytes;
  DevBuf<uint8_t> read_nv, vr_nv, read_flags, bases, ins_bytes, ref, call_flags, seq, win_flag, o_flags, o_inmat;
  DevBuf<MphReplayTx> replay;
  DevBuf<uint64_t> o_hap;
  DevBuf<uint2> pairs, seg_list, rd_runs, rd_span_exc, rd_flag_exc, vs_ncig_exc;
  DevBuf<uint8_t> rd_delta, rd_span, vs_vlo_d, vs_ncig;
  DevBuf<uint16_t> vs_read_d, vs_size;
  DevBuf<MphSideRun> vs_runs;
  DevBuf<MphVar> vars;
  DevBuf<MphSegment> segs;
  DevBuf<MphChunk> chunks;
  DevBuf<MphSegWork> seg_work;
  DevBuf<MphRec> recs, m_recs;
  DevBuf<MphRecSrc> m_aux;
  DevBuf<uint8_t> seq_dev, rec_seq, m_seq;
  DevBuf<uint32_t> win_seg, tx_stop, rw, rw_stopq, rw_info, rw_mbase, rw_bytes, rw_junc, rc_blocks, rc_bblocks;
  DevBuf<int> win_diff;
  DevBuf<uint64_t> call_S, call_B;
  DevBuf<MphWinOut> win_out, iw_out;
  DevBuf<MphHist> hist, spill;
  DevBuf<MphSpillWin> spq, spq_rp;
  DevBuf<MphHap> hap0, hapx, iw_hap0;
  DevBuf<unsigned long long> sums, win_id;
  mph_timing timing = {};
  std::unordered_map<const void*, size_t> pinned_dl;  // page-locked download buffers: data pointer -> bytes
  std::vector<PhaseRaw> raws;  // download buffers per stage, reused across calls (no page faults after the first)
  // secondary path: normal-peptidome hash set (open addressing, 5-bit packed peptides)
  DevBuf<unsigned long long> set_table;
  DevBuf<uint32_t> set_idx;    // peptides longer than 12 letters: slots index set_bytes (kernels/peptide_kernels.cu)
  DevBuf<uint8_t> set_bytes;
  uint64_t set_mask = 0;
  uint32_t set_k = 0;
  uint64_t set_distinct = 0;
};

namespace {

int fail(mph_ctx* ctx, int code, const std::string& msg) {
  g_last_error = msg;
  if (ctx) ctx->last_error = msg;
  return code;
}

template <class F>
int guarded(mph_ctx* ctx, F&& f) {
  try {
    f();
    return MPH_OK;
  } catch (const CudaError& e) {
    return fail(ctx, MPH_ERR_CUDA, e.what());
  } catch (const Fatal& e) {
    return fail(ctx, MPH_ERR_PANIC, e.what());
  } catch (const Unsupported& e) {
    return fail(ctx, MPH_ERR_UNSUPPORTED, e.what());
  } catch (const std::logic_error& e) {
    return fail(ctx, MPH_ERR_INTERNAL, e.what());
  } catch (const std::exception& e) {
    return fail(ctx, MPH_ERR_INPUT, e.what());
  }
}

void finish_batch(mph_batch* mb, bool pin) {
  Batch& b = mb->b;
  if (b.seq_cap > 256) throw Unsupported("insertion / deletion alleles too long for the device sequence slot");
  mb->pairs.clear();
  for (auto& e : b.pair_edges) mb->pairs.push_back(make_uint2(e.first, e.second));
  std::sort(mb->pairs.begin(), mb->pairs.end(), [](const uint2& a, const uint2& c) { return a.x < c.x; });
  auto bytes = [](auto& v) { return v.size() * sizeof(v[0]); };
  mb->span_mode = bus_span_mode(b);
  mb->h2d_bytes = bytes(b.rd_delta) + (mb->span_mode ? bytes(b.rd_mspan_exc) : bytes(b.rd_span) + bytes(b.rd_span_exc)) + bytes(b.rd_runs) + bytes(b.rd_flag_exc) + bytes(b.vs_read_d) + bytes(b.vs_vlo_d) + bytes(b.vs_size) +
                  bytes(b.vs_ncig) + bytes(b.vs_runs) + bytes(b.vs_ncig_exc) + bytes(b.vr_lseq) + bytes(b.vr_nv) + bytes(b.bases) + bytes(b.cigars) +
                  bytes(b.vars) + bytes(b.ins_bytes) + bytes(b.segs) + bytes(b.chunks) + bytes(b.seg_work) + bytes(b.seg_work_off) + bytes(b.ref) + bytes(b.stopmap) + bytes(mb->pairs) +
                  bytes(b.tx_id_bytes) + bytes(b.tx_id_off) + bytes(b.replay) + bytes(b.replay_dq) + (b.replay.empty() ? 0 : bytes(b.seg_chunk0));
  if (pin) {
    auto reg = [&](auto& v) {
      if (v.empty()) return;
      if (cudaHostRegister(v.data(), v.size() * sizeof(v[0]), cudaHostRegisterDefault) == cudaSuccess)
        mb->registered.emplace_back(v.data(), v.size() * sizeof(v[0]));
      else
        cudaGetLastError();
    };
    reg(b.rd_delta); if (mb->span_mode) reg(b.rd_mspan_exc); else { reg(b.rd_span); reg(b.rd_span_exc); } reg(b.rd_runs); reg(b.rd_flag_exc); reg(b.vs_read_d); reg(b.vs_vlo_d); reg(b.vs_size); reg(b.vs_ncig); reg(b.vs_runs); reg(b.vs_ncig_exc); reg(b.vr_lseq);
    reg(b.vr_nv); reg(b.bases); reg(b.cigars); reg(b.vars); reg(b.ins_bytes); reg(b.segs); reg(b.chunks); reg(b.seg_work); reg(b.seg_work_off); reg(b.ref); reg(b.stopmap);
    reg(mb->pairs);
    reg(b.tx_id_bytes); reg(b.tx_id_off); reg(b.replay); reg(b.replay_dq); reg(b.seg_chunk0);
    mb->pinned = true;
  }
}

// ---- stages ---------------------------------------------------------------------------------
// A batch is cut at gene boundaries into stages. mph_phase_batch copies stage s + 1 to the device on the copy stream
// while the kernels and the download of stage s run on the compute stream and the host threads work on the residue of
// the stages already downloaded. The resident entry points (upload / phase_resident / collect) use one stage = everything.
struct Stage {
  GeneMark lo, hi;
  uint32_t pair_lo = 0, pair_hi = 0;  // slice of mb->pairs (sorted by read)
};

std::vector<Stage> plan_stages(const mph_batch* mb, unsigned want) {
  const Batch& b = mb->b;
  const size_t n_genes = b.marks.size() - 1;
  std::vector<Stage> out;
  if (want < 1) want = 1;
  size_t g = 0;
  // the first two and the last two stages are shorter (0.35 and 0.7 of a regular one): the host residue can start
  // earlier and less of it is left when the last copy has finished
  auto weight = [want](unsigned s) {
    const unsigned e = want - 1 - s;
    const unsigned m = s < e ? s : e;
    return m == 0 ? 0.35 : (m == 1 ? 0.7 : 1.0);
  };
  double total_w = 0, acc_w = 0;
  for (unsigned s = 0; s < want; ++s) total_w += weight(s);
  for (unsigned s = 0; s < want && g < n_genes; ++s) {
    acc_w += weight(s);
    const uint64_t target = want > 2 ? uint64_t(double(b.marks.back().reads) * acc_w / total_w) : b.marks.back().reads * (s + 1) / want;
    size_t ge = g + 1;
    while (ge < n_genes && b.marks[ge].reads < target) ++ge;
    if (s + 1 == want) ge = n_genes;
    Stage st;
    st.lo = b.marks[g];
    st.hi = b.marks[ge];
    auto by_read = [](const uint2& a, uint64_t r) { return a.x < r; };
    st.pair_lo = uint32_t(std::lower_bound(mb->pairs.begin(), mb->pairs.end(), st.lo.reads, by_read) - mb->pairs.begin());
    st.pair_hi = uint32_t(std::lower_bound(mb->pairs.begin(), mb->pairs.end(), st.hi.reads, by_read) - mb->pairs.begin());
    out.push_back(st);
    g = ge;
  }
  if (out.empty()) {
    Stage st;
    st.lo = b.marks.front();
    st.hi = b.marks.back();
    st.pair_hi = uint32_t(mb->pairs.size());
    out.push_back(st);
  }
  return out;
}

// device buffers for the whole batch and the pointers of the kernel argument; nothing is copied here
void prepare(mph_ctx* c, const mph_batch* mb) {
  const Batch& b = mb->b;
  CU(cudaSetDevice(c->device));
  if (b.n_windows > 0xFFFFFF00ull || b.n_reads() > 0xFFFFFF00ull) throw Unsupported("batch too large: split it into gene ranges");
  if (b.chunks.size() >= (1u << 27)) throw Unsupported("batch too large: split it into gene ranges");
  const size_t nr = b.n_reads(), nw = size_t(b.n_windows);
  const size_t nvr = b.vr_read.size();
  c->read_start.ensure(nr + 1); c->read_end.ensure(nr + 1); c->read_flags.ensure(nr + 1);
  c->rd_delta.ensure(nr + 1); if (!mb->span_mode) c->rd_span.ensure(nr + 1); c->rd_runs.ensure(b.rd_runs.size() + 1); c->rd_span_exc.ensure((mb->span_mode ? b.rd_mspan_exc.size() : b.rd_span_exc.size()) + 1);
  c->rd_flag_exc.ensure(b.rd_flag_exc.size() + 1);
  c->read_vlo.ensure(nr + 1); c->read_nv.ensure(nr + 1); c->read_vr.ensure(nr + 1);  // expanded on the device by K1
  c->vr_read.ensure(nvr + 1); c->vr_vlo.ensure(nvr + 1); c->vr_seq_off.ensure(nvr + 1); c->vr_cig_off.ensure(nvr + 1);
  c->vr_lseq.ensure(nvr + 1); c->vr_ncig.ensure(nvr + 1); c->vr_nv.ensure(nvr + 1);
  c->vs_read_d.ensure(nvr + 1); c->vs_vlo_d.ensure(nvr + 1); c->vs_size.ensure(nvr + 1); c->vs_ncig.ensure(nvr + 1);
  c->vs_runs.ensure(b.vs_runs.size() + 1); c->vs_ncig_exc.ensure(b.vs_ncig_exc.size() + 1);
  c->bases.ensure(b.bases.size() + 1); c->cigars.ensure(b.cigars.size() + 1); c->vars.ensure(b.vars.size() + 1); c->ins_bytes.ensure(b.ins_bytes.size() + 1);
  c->segs.ensure(b.segs.size() + 1); c->chunks.ensure(b.chunks.size() + 1); c->seg_work.ensure(b.seg_work.size() + 1); c->seg_work_off.ensure(b.seg_work_off.size() + 1);
  c->win_diff.ensure(nw + 1); c->seg_list.ensure(size_t(b.seg_work_off.back()) + 1); c->seg_list_n.ensure(2 * b.segs.size() + 2); c->rr_seg0.ensure(mphk::read_runs_blocks(b.seg_work_off.back()) + 2); c->ref.ensure(b.ref.size() + 1); c->stopmap.ensure(b.stopmap.size() + 1);
  c->pairs.ensure(mb->pairs.size() + 1); c->tx_id_bytes.ensure(b.tx_id_bytes.size() + 1); c->tx_id_off.ensure(b.tx_id_off.size() + 1);
  c->call_S.ensure(nr + 1); c->call_B.ensure(nr + 1); c->call_flags.ensure(nr + 1);
  c->win_out.ensure(nw + 1); c->hap0.ensure(nw + 1); c->win_flag.ensure(nw + 1);
  c->block_counts.ensure(nw / 1024 + 2);
  c->iw.ensure(nw + 1); c->iw_out.ensure(nw + 1); c->iw_hap0.ensure(nw + 1); c->ovf_list.ensure(nw + 1);
  c->spq.ensure(nw + 1); c->spq_rp.ensure(nw + 1);  // a window is queued at most once
  if (c->spill.cap == 0) c->spill.ensure(1 << 16);
  c->counters.ensure(mphk::CTR_COUNT); c->sums.ensure(3);
  {
    c->win_seg.ensure(nw + 1); c->tx_stop.ensure(b.txs.size() + 1);
    c->rw.ensure(nw + 1); c->rw_stopq.ensure(nw + 1); c->rw_info.ensure(nw + 1); c->rw_mbase.ensure(nw + 1); c->rw_bytes.ensure(nw + 1); c->rw_junc.ensure(b.segs.size() + 1);
    c->rc_blocks.ensure(nw / 256 + 4);  // (the record kernels use 512 windows per block)
    c->rc_bblocks.ensure(nw / 256 + 4);
    // somatic: about one record per 30 windows; normal: every window writes at least one
    const size_t rec_want = b.mode == 1 ? nw + nw / 4 + (1 << 14) : std::max<size_t>(nw / 16, 1 << 14);
    if (c->recs.cap < rec_want) { c->recs.ensure(rec_want); c->rec_seq.ensure(std::max<size_t>(c->rec_seq.cap, b.mode == 1 ? rec_want * 8 : rec_want * 64)); }
    if (c->m_recs.cap == 0) { c->m_recs.ensure(1 << 14); c->m_aux.ensure(c->m_recs.cap); c->m_seq.ensure(c->m_recs.cap * MPH_RC_SEQ_SLOT); }
  } c->seg_live.ensure(b.segs.size() + 1);
  if (c->hist.cap == 0) { c->hist.ensure(std::max<size_t>(nw / 2, 1 << 16)); c->hapx.ensure(c->hist.cap); }
  if (c->hapx.cap < c->hist.cap) c->hapx.ensure(c->hist.cap);
  if (c->hist_win.cap < c->hist.cap) c->hist_win.ensure(c->hist.cap);
  const size_t seq_want = (2 * b.segs.size() + nw / 8 + 4096) * 2 * b.seq_cap;
  if (c->seq.cap < seq_want) c->seq.ensure(seq_want);
  if (b.mode == 0 && c->seq_dev.cap < seq_want) c->seq_dev.ensure(seq_want);
  mphk::DeviceBatch& d = c->d;
  d.n_reads = uint32_t(nr); d.n_vars = uint32_t(b.vars.size()); d.n_segs = uint32_t(b.segs.size()); d.n_chunks = uint32_t(b.chunks.size());
  d.n_windows = uint32_t(nw); d.seq_cap = b.seq_cap;
  d.read_start = c->read_start.p; d.read_end = c->read_end.p; d.read_flags = c->read_flags.p;
  d.read_start_w = c->read_start.p; d.read_end_w = c->read_end.p; d.read_flags_w = c->read_flags.p;
  d.rd_delta = c->rd_delta.p; d.rd_span = mb->span_mode ? nullptr : c->rd_span.p; d.modal_span = b.modal_span; d.rd_runs = c->rd_runs.p; d.rd_span_exc = c->rd_span_exc.p; d.rd_flag_exc = c->rd_flag_exc.p;
  d.read_vlo = c->read_vlo.p; d.read_nv = c->read_nv.p; d.read_vr = c->read_vr.p;
  d.vr_read = c->vr_read.p; d.vr_vlo = c->vr_vlo.p; d.vr_seq_off = c->vr_seq_off.p; d.vr_cig_off = c->vr_cig_off.p;
  d.vr_lseq = c->vr_lseq.p; d.vr_ncig = c->vr_ncig.p; d.vr_nv = c->vr_nv.p;
  d.vr_read_w = c->vr_read.p; d.vr_vlo_w = c->vr_vlo.p; d.vr_seq_off_w = c->vr_seq_off.p; d.vr_cig_off_w = c->vr_cig_off.p; d.vr_ncig_w = c->vr_ncig.p;
  d.vs_read_d = c->vs_read_d.p; d.vs_vlo_d = c->vs_vlo_d.p; d.vs_size = c->vs_size.p; d.vs_ncig = c->vs_ncig.p; d.vs_runs = c->vs_runs.p;
  d.vs_ncig_exc = c->vs_ncig_exc.p;
  d.bases = c->bases.p; d.cigars = c->cigars.p; d.vars = c->vars.p;
  d.ins_bytes = c->ins_bytes.p; d.segs = c->segs.p; d.chunks = c->chunks.p; d.seg_work = c->seg_work.p; d.seg_work_off = c->seg_work_off.p;
  d.win_diff = c->win_diff.p; d.seg_list = c->seg_list.p; d.seg_list_n = c->seg_list_n.p; d.seg_list2_n = c->seg_list_n.p + b.segs.size() + 1; d.rr_seg0 = c->rr_seg0.p; d.ref = c->ref.p; d.stopmap = c->stopmap.p;
  d.call_S = reinterpret_cast<uint64_t*>(c->call_S.p); d.call_B = reinterpret_cast<uint64_t*>(c->call_B.p); d.call_flags = c->call_flags.p;
  d.win_out = c->win_out.p; d.hap0 = c->hap0.p; d.win_flag = c->win_flag.p; d.block_counts = c->block_counts.p;
  d.ovf_list = c->ovf_list.p; d.spq = c->spq.p; d.spq_rp = c->spq_rp.p;
  d.iw = c->iw.p; d.iw_out = c->iw_out.p; d.iw_hap0 = c->iw_hap0.p; d.counters = c->counters.p;
  d.sum_depth = c->sums.p; d.live_depth = c->sums.p + 1; d.seg_live = c->seg_live.p;
  d.window_len = b.window_len;
  d.win_seg = c->win_seg.p; d.tx_stop = c->tx_stop.p; d.rw = c->rw.p; d.rw_stopq = c->rw_stopq.p; d.rw_info = c->rw_info.p; d.rw_mbase = c->rw_mbase.p;
  d.rw_bytes = c->rw_bytes.p; d.rw_junc = c->rw_junc.p; d.rc_blocks = c->rc_blocks.p; d.rc_bblocks = c->rc_bblocks.p;
  d.tx_id_bytes = c->tx_id_bytes.p; d.tx_id_off = c->tx_id_off.p;
  d.n_replay = uint32_t(b.replay.size());
  d.win_voff = nullptr; d.iw_voff = nullptr;
  if (d.n_replay) {
    const size_t no = size_t(b.replay_obs) + 1;
    c->replay.ensure(b.replay.size() + 1); c->seg_chunk0.ensure(b.seg_chunk0.size() + 1); c->dq_init.ensure(b.replay_dq.size() + 1);
    c->o_read.ensure(no); c->o_key.ensure(no); c->o_hap.ensure(no); c->o_frame.ensure(no); c->o_flags.ensure(no); c->o_inmat.ensure(no);
    c->win_voff.ensure(nw + 1); c->iw_voff.ensure(nw + 1); c->seg_err.ensure(b.segs.size() + 1);
    if (c->vlist.cap == 0) c->vlist.ensure(1 << 16);
    d.replay = c->replay.p; d.seg_chunk0 = c->seg_chunk0.p; d.dq_init = c->dq_init.p;
    d.o_read = c->o_read.p; d.o_key = c->o_key.p; d.o_hap = reinterpret_cast<uint64_t*>(c->o_hap.p); d.o_frame = c->o_frame.p; d.o_flags = c->o_flags.p; d.o_inmat = c->o_inmat.p;
    d.win_voff = c->win_voff.p; d.iw_voff = c->iw_voff.p; d.seg_err = c->seg_err.p;
  }
  d.mode = uint32_t(b.mode);
  if (b.mode == 1) { c->win_depth.ensure(nw + 1); d.win_depth = c->win_depth.p; c->win_id.ensure(nw + 1); d.win_id = c->win_id.p; }
  c->cur = mb;
  c->timing = mph_timing{};
  c->timing.h2d_bytes = mb->h2d_bytes;
}

template <class T, class V>
void h2d_range(cudaStream_t st, DevBuf<T>& dst, const V& src, size_t lo, size_t hi) {
  if (hi > src.size()) hi = src.size();
  if (hi > lo) CU(cudaMemcpyAsync(dst.p + lo, src.data() + lo, (hi - lo) * sizeof(T), cudaMemcpyHostToDevice, st));
}

// host -> device copy of one stage's slices
void copy_stage(mph_ctx* c, const mph_batch* mb, const Stage& s, bool first, cudaStream_t st) {
  const Batch& b = mb->b;
  const size_t r0 = s.lo.reads, r1 = s.hi.reads;
  h2d_range(st, c->rd_delta, b.rd_delta, r0, r1);
  if (mb->span_mode) h2d_range(st, c->rd_span_exc, b.rd_mspan_exc, s.lo.mspan_exc, s.hi.mspan_exc);  // one span per batch + the reads that differ
  else { h2d_range(st, c->rd_span, b.rd_span, r0, r1); h2d_range(st, c->rd_span_exc, b.rd_span_exc, s.lo.span_exc, s.hi.span_exc); }
  h2d_range(st, c->rd_runs, b.rd_runs, s.lo.runs, s.hi.runs);
  h2d_range(st, c->rd_flag_exc, b.rd_flag_exc, s.lo.flag_exc, s.hi.flag_exc);
  const size_t e0 = s.lo.vr, e1 = s.hi.vr;
  h2d_range(st, c->vs_read_d, b.vs_read_d, e0, e1); h2d_range(st, c->vs_vlo_d, b.vs_vlo_d, e0, e1); h2d_range(st, c->vs_size, b.vs_size, e0, e1);
  h2d_range(st, c->vs_ncig, b.vs_ncig, e0, e1); h2d_range(st, c->vr_lseq, b.vr_lseq, e0, e1); h2d_range(st, c->vr_nv, b.vr_nv, e0, e1);
  h2d_range(st, c->vs_runs, b.vs_runs, s.lo.vruns, s.hi.vruns); h2d_range(st, c->vs_ncig_exc, b.vs_ncig_exc, s.lo.ncig_exc, s.hi.ncig_exc);
  h2d_range(st, c->bases, b.bases, s.lo.bases, s.hi.bases); h2d_range(st, c->cigars, b.cigars, s.lo.cigars, s.hi.cigars);
  h2d_range(st, c->vars, b.vars, s.lo.vars, s.hi.vars); h2d_range(st, c->ins_bytes, b.ins_bytes, s.lo.ins, s.hi.ins);
  h2d_range(st, c->segs, b.segs, s.lo.segs, s.hi.segs); h2d_range(st, c->chunks, b.chunks, s.lo.chunks, s.hi.chunks);
  h2d_range(st, c->seg_work, b.seg_work, s.lo.segs, s.hi.segs); h2d_range(st, c->seg_work_off, b.seg_work_off, s.lo.segs, s.hi.segs + 1);
  h2d_range(st, c->ref, b.ref, s.lo.ref, s.hi.ref);
  h2d_range(st, c->stopmap, b.stopmap, s.lo.ref / 32, s.hi.ref / 32 + 4);  // whole words; neighbouring stages rewrite the shared word with the same bits
  h2d_range(st, c->pairs, mb->pairs, s.pair_lo, s.pair_hi);
  if (first) { h2d_range(st, c->tx_id_bytes, b.tx_id_bytes, 0, b.tx_id_bytes.size()); h2d_range(st, c->tx_id_off, b.tx_id_off, 0, b.tx_id_off.size()); }
  if (!b.replay.empty()) {
    h2d_range(st, c->replay, b.replay, s.lo.replay, s.hi.replay); h2d_range(st, c->dq_init, b.replay_dq, s.lo.dq, s.hi.dq);
    h2d_range(st, c->seg_chunk0, b.seg_chunk0, s.lo.segs, s.hi.segs);
  }
}

void set_ranges(mph_ctx* c, const Stage& s) {
  mphk::DeviceBatch& d = c->d;
  d.r0 = uint32_t(s.lo.reads); d.r1 = uint32_t(s.hi.reads);
  d.vr0 = uint32_t(s.lo.vr); d.vr1 = uint32_t(s.hi.vr);
  d.c0 = uint32_t(s.lo.chunks); d.c1 = uint32_t(s.hi.chunks);
  d.s0 = uint32_t(s.lo.segs); d.s1 = uint32_t(s.hi.segs);
  d.run0 = uint32_t(s.lo.runs); d.run1 = uint32_t(s.hi.runs); d.sx0 = uint32_t(c->cur->span_mode ? s.lo.mspan_exc : s.lo.span_exc); d.sx1 = uint32_t(c->cur->span_mode ? s.hi.mspan_exc : s.hi.span_exc);
  d.fx0 = uint32_t(s.lo.flag_exc); d.fx1 = uint32_t(s.hi.flag_exc);
  d.vrun0 = uint32_t(s.lo.vruns); d.vrun1 = uint32_t(s.hi.vruns); d.nx0 = uint32_t(s.lo.ncig_exc); d.nx1 = uint32_t(s.hi.ncig_exc);
  d.it0 = c->cur->b.seg_work_off[s.lo.segs]; d.it1 = c->cur->b.seg_work_off[s.hi.segs];
  d.w0 = uint32_t(s.lo.windows); d.w1 = uint32_t(s.hi.windows);
  d.rp0 = uint32_t(s.lo.replay); d.rp1 = uint32_t(s.hi.replay);
  d.pairs = c->pairs.p + s.pair_lo; d.n_pairs = s.pair_hi - s.pair_lo;
}

// kernels K1-K4 over the slice set by set_ranges, on the compute stream
void run_kernels(mph_ctx* c) {
  if (!c->cur) throw std::runtime_error("no batch uploaded");
  mphk::DeviceBatch& d = c->d;
  { const char* fw = getenv("MPH_FORCE_WIDE"); d.force_wide = (fw && (*fw == '1' || *fw == '2')) ? uint32_t(*fw - '0') : 0u; }
  if (c->hist_win.cap < c->hist.cap) c->hist_win.ensure(c->hist.cap);
  d.hist = c->hist.p; d.hapx = c->hapx.p; d.hist_win = c->hist_win.p; d.hist_cap = uint32_t(std::min<size_t>(c->hist.cap, 0xFFFFFFF0u));
  d.spill = c->spill.p; d.spill_cap = uint32_t(std::min<size_t>(c->spill.cap, 0xFFFFFFF0u));
  d.seq = c->seq.p; d.seq_cap_bytes = uint32_t(std::min<size_t>(c->seq.cap, 0xFFFFFF00u));
  d.seq_dev = c->seq_dev.p; d.seq_dev_cap_bytes = uint32_t(std::min<size_t>(c->seq_dev.cap, 0xFFFFFF00u));
  d.recs = c->recs.p; d.rec_cap = uint32_t(std::min<size_t>(c->recs.cap, 0xFFFFFF00u));
  d.rec_seq = c->rec_seq.p; d.rec_seq_cap = uint32_t(std::min<size_t>(c->rec_seq.cap, 0xFFFFFF00u));
  d.m_recs = c->m_recs.p; d.m_aux = c->m_aux.p; d.m_seq = c->m_seq.p; d.m_cap = uint32_t(std::min<size_t>(c->m_recs.cap, 0x03FFFFFFu));
  CU(cudaMemsetAsync(c->counters.p, 0, mphk::CTR_COUNT * sizeof(uint32_t), c->stream));
  // normal mode: the record kernels visit every window and find its segment in win_seg; windows nobody claims (replayed
  // transcripts) must read as host class
  if (d.mode == 1 && d.w1 > d.w0) CU(cudaMemsetAsync(c->win_seg.p + d.w0, 0xFF, size_t(d.w1 - d.w0) * sizeof(uint32_t), c->stream));
  if (c->stage_tx_hi > c->stage_tx_lo)
    CU(cudaMemsetAsync(c->tx_stop.p + c->stage_tx_lo, 0xFF, size_t(c->stage_tx_hi - c->stage_tx_lo) * sizeof(uint32_t), c->stream));
  CU(cudaEventRecord(c->ev[2], c->stream));  // k1_ms covers the zero-fill below: it is the allele call of the reads without variants
  if (d.r1 > d.r0) {
    // reads without an entry in the side table: no allele call, no bad base, no variant inside
    const size_t n = size_t(d.r1 - d.r0);
    // (call_S / call_B are written by K1 for the reads of the side table only; every reader checks call_flags / read_nv first)
    CU(cudaMemsetAsync(c->call_flags.p + d.r0, 0, n, c->stream));
    CU(cudaMemsetAsync(c->read_flags.p + d.r0, 0, n, c->stream));
    CU(cudaMemsetAsync(c->read_nv.p + d.r0, 0, n, c->stream));
  }
  if (d.rp1 > d.rp0) {
    // K2 writes the flag of every window it owns; the replay only those it reaches (and, on its side stream, possibly after
    // the record kernels have looked): whatever an earlier batch left in the windows of replayed transcripts must not be read
    CU(cudaMemsetAsync(c->win_flag.p + d.w0, 0, size_t(d.w1 - d.w0), c->stream));
    d.vlist = c->vlist.p; d.vlist_cap = uint32_t(std::min<size_t>(c->vlist.cap, 0xFFFFFF00u));
    CU(cudaMemsetAsync(c->win_voff.p + d.w0, 0xFF, size_t(d.w1 - d.w0) * sizeof(uint32_t), c->stream));
    const uint32_t s0 = c->stage_seg_lo, s1 = c->stage_seg_hi;
    CU(cudaMemsetAsync(c->seg_err.p + s0, 0, size_t(s1 - s0) * sizeof(uint32_t), c->stream));
  } else if (d.n_replay) {
    CU(cudaMemsetAsync(c->win_voff.p + d.w0, 0xFF, size_t(d.w1 - d.w0) * sizeof(uint32_t), c->stream));
  }
  if (d.w1 > d.w0) CU(cudaMemsetAsync(c->win_diff.p + d.w0, 0, size_t(d.w1 - d.w0) * sizeof(int), c->stream));
  if (d.s1 > d.s0) {
    CU(cudaMemsetAsync(d.seg_list_n + d.s0, 0, size_t(d.s1 - d.s0) * sizeof(uint32_t), c->stream));
    CU(cudaMemsetAsync(d.seg_list2_n + d.s0, 0, size_t(d.s1 - d.s0) * sizeof(uint32_t), c->stream));
  }
  mphk::launch_read_decode(d, c->stream);  // K0: start / end / flags of the slice's reads from their 2-byte bus form
  mphk::launch_allele_call(d, c->stream);
  CU(cudaEventRecord(c->ev[3], c->stream));
  // The serial replay is a dependent chain per unit (a few hundred iterations, latency bound) over 1 % of the transcripts, all
  // of them host class: nothing on the main chain needs its results before the download. In the somatic mode it therefore
  // runs on its own stream, followed there by the K3 walk of the host-class keys and the compaction of the host-class windows
  // (K4), while the main stream goes on with the K3 walk of the device-class keys and the record kernels and joins at the end.
  // MPH_SIDE_REPLAY: "k1" (default) starts the side chain right after K1, so the replay overlaps K2, K3 and the record
  // kernels; "k2" starts it when K2 is done (K2 then runs alone); "0" puts everything on one stream, which is how bench.py
  // times the kernels one by one for its roofline line. MPH_REPLAY_PER_SM > 0 makes k_replay a persistent grid of that many
  // single-warp CTAs per SM (default: one CTA per unit). `normal` mode: the replay runs beside K2 and joins before K3.
  // Measured on B200 (whole-exome shard): DESIGN.md section 5.
  // (read per call, not cached: bench.py times the kernels alone for the roofline line by switching the side chain off)
  const int side_cfg = [] { const char* e = getenv("MPH_SIDE_REPLAY"); return !e ? 1 : (*e == '0' ? 0 : (strcmp(e, "k2") == 0 ? 2 : 1)); }();
  const uint32_t replay_per_sm = [] { const char* e = getenv("MPH_REPLAY_PER_SM"); const int v = e ? atoi(e) : 0; return uint32_t(v > 0 ? v : 0); }();
  const bool side = side_cfg != 0 && d.rp1 > d.rp0;
  const bool side_from_k1 = side && (side_cfg == 1 || d.mode == 1);
  const uint32_t replay_ctas = replay_per_sm * uint32_t(c->sm_count);
  if (side_from_k1) {
    CU(cudaEventRecord(c->ev_rp[0], c->stream));
    CU(cudaStreamWaitEvent(c->replay_stream, c->ev_rp[0], 0));
    CU(cudaEventRecord(c->ev_rp[1], c->replay_stream));
    mphk::launch_replay(d, c->replay_stream, replay_ctas);
    CU(cudaEventRecord(c->ev_rp[2], c->replay_stream));
  } else if (!side) {
    mphk::launch_replay(d, c->stream);
  }
  CU(cudaEventRecord(c->ev[8], c->stream));
  mphk::launch_window_hist(d, c->stream);
  CU(cudaEventRecord(c->ev[4], c->stream));
  c->replay_on_side = side;
  c->side_chain = side && d.mode == 0;
  if (c->side_chain) {
    // side chain: (the replay,) host-class keys (K2's and the replay's) and host-class windows
    CU(cudaStreamWaitEvent(c->replay_stream, c->ev[4], 0));
    if (!side_from_k1) {
      CU(cudaEventRecord(c->ev_rp[1], c->replay_stream));
      mphk::launch_replay(d, c->replay_stream, replay_ctas);
      CU(cudaEventRecord(c->ev_rp[2], c->replay_stream));
    }
    CU(cudaEventRecord(c->ev_rp[3], c->replay_stream));
    mphk::launch_assemble(d, c->replay_stream, mphk::ASM_HOST_CLASS);
    mphk::launch_compact(d, c->replay_stream);
    CU(cudaEventRecord(c->ev_rp[4], c->replay_stream));
    // main chain: device-class keys, record kernels
    mphk::launch_assemble(d, c->stream, mphk::ASM_DEVICE_CLASS);
    CU(cudaEventRecord(c->ev[5], c->stream));
    CU(cudaEventRecord(c->ev[6], c->stream));
    mphk::launch_records(d, c->stream);
    CU(cudaEventRecord(c->ev[7], c->stream));
    CU(cudaStreamWaitEvent(c->stream, c->ev_rp[4], 0));
  } else {
    if (side) CU(cudaStreamWaitEvent(c->stream, c->ev_rp[2], 0));  // normal mode: K3 needs the replay's keys
    mphk::launch_assemble(d, c->stream);
    CU(cudaEventRecord(c->ev[5], c->stream));
    mphk::launch_compact(d, c->stream);
    CU(cudaEventRecord(c->ev[6], c->stream));
    mphk::launch_records(d, c->stream);
    CU(cudaEventRecord(c->ev[7], c->stream));
  }
  CU(cudaEventRecord(c->ev[9], c->stream));
  CU(cudaGetLastError());
}

// per-kernel-group device times of the last run_kernels (CUDA events on the streams the kernels ran on), added to ctx->timing.
// With the side chain: replay_ms is k_replay alone on its stream, k4_ms the host-class K3 walk + compaction that follow it
// there, k2 / k3 / k5 the main chain (K3 = device-class keys); kernels_ms is the whole chain from the first kernel to the join.
void add_kernel_times(mph_ctx* c) {
  float ms;
  CU(cudaEventElapsedTime(&ms, c->ev[2], c->ev[3])); c->timing.k1_ms += ms;
  if (c->replay_on_side) { CU(cudaEventElapsedTime(&ms, c->ev_rp[1], c->ev_rp[2])); c->timing.replay_ms += ms; }
  else { CU(cudaEventElapsedTime(&ms, c->ev[3], c->ev[8])); c->timing.replay_ms += ms; }
  CU(cudaEventElapsedTime(&ms, c->ev[8], c->ev[4])); c->timing.k2_ms += ms;
  CU(cudaEventElapsedTime(&ms, c->ev[2], c->ev[9])); c->timing.kernels_ms += ms;
  CU(cudaEventElapsedTime(&ms, c->ev[4], c->ev[5])); c->timing.k3_ms += ms;
  if (c->side_chain) { CU(cudaEventElapsedTime(&ms, c->ev_rp[3], c->ev_rp[4])); c->timing.k4_ms += ms; }
  else { CU(cudaEventElapsedTime(&ms, c->ev[5], c->ev[6])); c->timing.k4_ms += ms; }
  CU(cudaEventElapsedTime(&ms, c->ev[6], c->ev[7])); c->timing.k5_ms += ms;
}

// resize of a download buffer that keeps it page-locked (device -> host copies into pageable memory go through a bounce
// buffer at a fraction of the link speed). The registration follows the allocation: dropped before a growth, renewed after.
template <class V>
void resize_pinned(mph_ctx* c, V& v, size_t n) {
  if (n > v.capacity()) {
    auto it = c->pinned_dl.find(v.data());
    if (it != c->pinned_dl.end()) {
      cudaHostUnregister(const_cast<void*>(it->first));
      c->pinned_dl.erase(it);
    }
    v.reserve(n + n / 4);  // the sizes of consecutive calls differ a little: avoid a re-registration per call
  }
  v.resize(n);
  const size_t bytes = v.capacity() * sizeof(v[0]);
  if (bytes >= (size_t(1) << 16) && !c->pinned_dl.count(v.data())) {
    if (cudaHostRegister(v.data(), bytes, cudaHostRegisterDefault) == cudaSuccess) c->pinned_dl[v.data()] = bytes;
    else cudaGetLastError();
  }
}

// an arena ran out during the last run_kernels (the counters say how much was asked for): grows it; true = run again
bool grow_arenas(mph_ctx* c, const uint32_t* ctr) {
  const uint32_t err = ctr[mphk::CTR_ERR];
  if (!(err & (MPH_E_HIST_OVERFLOW | MPH_E_SEQ_OVERFLOW | MPH_E_VLIST_OVERFLOW | MPH_E_REC_OVERFLOW | MPH_E_SPILL_OVERFLOW))) return false;
  if (err & MPH_E_SPILL_OVERFLOW) c->spill.ensure(size_t(ctr[mphk::CTR_SPILL]) * 2 + 1024);
  if (err & MPH_E_REC_OVERFLOW) {
    c->recs.ensure(std::max<size_t>(size_t(ctr[mphk::CTR_NREC]) * 2 + 1024, c->recs.cap));
    c->rec_seq.ensure(std::max<size_t>(size_t(ctr[mphk::CTR_RECSEQ]) * 2 + 4096, std::max(c->rec_seq.cap, c->recs.cap * 64)));
    c->m_recs.ensure(std::max<size_t>(size_t(ctr[mphk::CTR_MERGE]) * 2 + 1024, c->m_recs.cap));
    c->m_aux.ensure(c->m_recs.cap); c->m_seq.ensure(c->m_recs.cap * MPH_RC_SEQ_SLOT);
  }
  if (err & MPH_E_SEQ_OVERFLOW) c->seq_dev.ensure(size_t(ctr[mphk::CTR_SEQD]) * 2 + 4096);
  if (err & MPH_E_VLIST_OVERFLOW) c->vlist.ensure(size_t(ctr[mphk::CTR_VLIST]) * 2 + 1024);
  if (err & MPH_E_HIST_OVERFLOW) { c->hist.ensure((size_t(ctr[mphk::CTR_HIST]) + ctr[mphk::CTR_HISTD]) * 2 + 1024); c->hapx.ensure(c->hist.cap); }
  if (err & MPH_E_SEQ_OVERFLOW) c->seq.ensure(size_t(ctr[mphk::CTR_SEQ]) * 2 + 4096);
  return true;
}

// device -> host copy of what the kernels produced for the current slice; re-runs the kernels when an arena was too small
void fetch_stage(mph_ctx* c, const Stage& s, PhaseRaw& raw, uint64_t* n_iw_total) {
  const Batch& b = c->cur->b;
  uint32_t ctr[mphk::CTR_COUNT];
  for (int attempt = 0;; ++attempt) {
    CU(cudaMemcpyAsync(ctr, c->counters.p, sizeof ctr, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (grow_arenas(c, ctr) && attempt < 6) {
      run_kernels(c);
      continue;
    }
    break;
  }
  float ms;
  add_kernel_times(c);
  raw.err = ctr[mphk::CTR_ERR];
  if (raw.err & MPH_E_SLICE) throw Fatal("slice index out of range");
  if (raw.err & MPH_E_SEQ_SLOT) throw Unsupported("assembled haplotype longer than the sequence slot");
  if (raw.err & MPH_E_REF_RANGE) throw Fatal("slice index out of range: refseq");
  if (raw.err & MPH_E_VARS_PER_WINDOW) throw Unsupported("more than 32 variants in one window / 64 inside one read");
  if (raw.err & MPH_E_KEYS_PER_WINDOW) throw Unsupported(MPH_MSG_KEYS_PER_WINDOW);
  if (raw.err & MPH_E_RECS_PER_LIST) throw Unsupported(MPH_MSG_RECS_PER_LIST);
  if (raw.err & MPH_E_REPLAY_PANIC) throw Fatal("bug: read starts right of variant");
  if (raw.err) throw std::logic_error("device error bits " + std::to_string(raw.err));
  const uint32_t n_iw = ctr[mphk::CTR_NIW], n_hist = ctr[mphk::CTR_HIST], n_seq = ctr[mphk::CTR_SEQ];
  const uint32_t n_rec = ctr[mphk::CTR_NREC], n_recseq = ctr[mphk::CTR_RECSEQ], n_merge = ctr[mphk::CTR_MERGE];
  resize_pinned(c, raw.recs, n_rec); resize_pinned(c, raw.rec_seq, n_recseq); resize_pinned(c, raw.rec_aux, n_merge);
  resize_pinned(c, raw.iw, n_iw); resize_pinned(c, raw.iw_out, n_iw); resize_pinned(c, raw.iw_hap0, n_iw); resize_pinned(c, raw.hist, n_hist);
  resize_pinned(c, raw.hapx, n_hist); resize_pinned(c, raw.seq, n_seq);
  CU(cudaEventRecord(c->ev[0], c->stream));
  if (n_iw) {
    CU(cudaMemcpyAsync(raw.iw.data(), c->iw.p, n_iw * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(raw.iw_out.data(), c->iw_out.p, n_iw * sizeof(MphWinOut), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(raw.iw_hap0.data(), c->iw_hap0.p, n_iw * sizeof(MphHap), cudaMemcpyDeviceToHost, c->stream));
  }
  if (n_hist) {
    CU(cudaMemcpyAsync(raw.hist.data(), c->hist.p, n_hist * sizeof(MphHist), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(raw.hapx.data(), c->hapx.p, n_hist * sizeof(MphHap), cudaMemcpyDeviceToHost, c->stream));
  }
  if (n_seq) CU(cudaMemcpyAsync(raw.seq.data(), c->seq.p, n_seq, cudaMemcpyDeviceToHost, c->stream));
  if (n_rec) CU(cudaMemcpyAsync(raw.recs.data(), c->recs.p, size_t(n_rec) * sizeof(MphRec), cudaMemcpyDeviceToHost, c->stream));
  if (n_recseq) CU(cudaMemcpyAsync(raw.rec_seq.data(), c->rec_seq.p, n_recseq, cudaMemcpyDeviceToHost, c->stream));
  if (n_merge) CU(cudaMemcpyAsync(raw.rec_aux.data(), c->m_aux.p, size_t(n_merge) * sizeof(MphRecSrc), cudaMemcpyDeviceToHost, c->stream));
  const bool has_replay = c->d.n_replay != 0;
  const uint32_t n_vl = (c->d.rp1 > c->d.rp0) ? std::min<uint32_t>(ctr[mphk::CTR_VLIST], c->d.vlist_cap) : 0;
  resize_pinned(c, raw.iw_voff, has_replay ? n_iw : 0);
  resize_pinned(c, raw.vlist, n_vl);
  if (has_replay && n_iw) CU(cudaMemcpyAsync(raw.iw_voff.data(), c->iw_voff.p, n_iw * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
  if (n_vl) CU(cudaMemcpyAsync(raw.vlist.data(), c->vlist.p, size_t(n_vl) * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
  raw.seg_base = uint32_t(s.lo.segs);
  if (c->d.rp1 > c->d.rp0) {
    raw.seg_err.resize(size_t(s.hi.segs - s.lo.segs));
    if (!raw.seg_err.empty()) CU(cudaMemcpyAsync(raw.seg_err.data(), c->seg_err.p + s.lo.segs, raw.seg_err.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
  } else {
    raw.seg_err.clear();
  }
  const bool normal_mode = b.mode == 1;
  const size_t nw = size_t(s.hi.windows - s.lo.windows);
  raw.win_base = uint32_t(s.lo.windows);
  resize_pinned(c, raw.win_depth, normal_mode ? nw : 0);
  resize_pinned(c, raw.win_id, normal_mode ? nw : 0);
  if (normal_mode && nw) {
    CU(cudaMemcpyAsync(raw.win_depth.data(), c->win_depth.p + s.lo.windows, nw * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(raw.win_id.data(), c->win_id.p + s.lo.windows, nw * 8, cudaMemcpyDeviceToHost, c->stream));
  }
  CU(cudaEventRecord(c->ev[1], c->stream));
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
  c->timing.d2h_ms += ms;
  c->timing.d2h_bytes += sizeof ctr + size_t(n_iw) * (4 + sizeof(MphWinOut) + sizeof(MphHap)) + size_t(n_hist) * (sizeof(MphHist) + sizeof(MphHap)) + n_seq +
                         size_t(n_rec) * sizeof(MphRec) + n_recseq + size_t(n_merge) * sizeof(MphRecSrc) +
                         raw.win_depth.size() * 12 + (raw.iw_voff.size() + raw.vlist.size() + raw.seg_err.size()) * 4;
  *n_iw_total += n_iw;
}

// copies the device-built records of transcripts [tx_lo, tx_hi) with their bytes into a result part
void take_device_records(const PhaseRaw& raw, uint32_t tx_lo, uint32_t tx_hi, ResultPart& part) {
  auto by_tx = [](const MphRec& r, uint32_t t) { return r.tx < t; };
  const auto d0 = std::lower_bound(raw.recs.begin(), raw.recs.end(), tx_lo, by_tx);
  const auto d1 = std::lower_bound(d0, raw.recs.end(), tx_hi, by_tx);
  if (d0 == d1) return;
  part.dev.assign(d0, d1);
  // the sequence bytes: the somatic record kernels lay them out in record order, so a block of transcripts owns one
  // contiguous range (one memcpy; reading them record by record out of the freshly DMA-written download buffer was a cache
  // miss each and most of the host threads' time); any other layout is copied record by record
  size_t bytes = 0, n_aux = 0, lo = size_t(-1), hi = 0;
  for (const MphRec& r : part.dev) {
    if (!(r.flags & MPH_RC_REFSEQ)) {
      const size_t n = size_t(std::max(r.neo_len, r.mt_len)) + std::max(r.norm_len, r.wt_len);
      bytes += n;
      lo = std::min<size_t>(lo, r.seq_off);
      hi = std::max<size_t>(hi, size_t(r.seq_off) + n);
    }
    n_aux += (r.flags & MPH_RC_MERGED) ? 1 : 0;
  }
  part.dev_seq.resize(bytes);
  part.dev_aux.reserve(n_aux);
  const bool contiguous = bytes != 0 && hi - lo == bytes && hi <= raw.rec_seq.size();
  if (contiguous) memcpy(part.dev_seq.data(), raw.rec_seq.data() + lo, bytes);
  size_t pos = 0;
  for (MphRec& r : part.dev) {
    if (!(r.flags & MPH_RC_REFSEQ)) {  // (a reference window's bytes stay in the batch's reference arena)
      const size_t n = size_t(std::max(r.neo_len, r.mt_len)) + std::max(r.norm_len, r.wt_len);
      if (contiguous) {
        r.seq_off = uint32_t(r.seq_off - lo);
      } else {
        memcpy(part.dev_seq.data() + pos, raw.rec_seq.data() + r.seq_off, n);
        r.seq_off = uint32_t(pos);
        pos += n;
      }
    }
    if (r.flags & MPH_RC_MERGED) {
      part.dev_aux.push_back(raw.rec_aux[r.aux]);
      r.aux = uint32_t(part.dev_aux.size() - 1);
    }
  }
}

// host residue workers: transcripts are independent, blocks of them are taken from a queue that the stage loop fills
struct ResiduePool {
  struct Task { const PhaseRaw* raw; uint32_t tx_lo, tx_hi; size_t part; };
  const Batch& b;
  std::deque<ResultPart>& parts;
  std::vector<std::thread> threads;
  std::mutex mu;
  std::condition_variable cv;
  std::deque<Task> queue;
  bool closed = false;
  std::vector<ResidueStats> stats;
  std::vector<std::vector<std::pair<uint32_t, uint32_t>>> live;
  std::vector<std::exception_ptr> errs;
  std::vector<double> busy_ms;
  // measurement hook (MPH_TIMELINE): per task, the part it wrote, when it ended and how long it ran
  struct Trace { size_t part; double end_ms, ms; };
  std::vector<std::vector<Trace>> trace;
  bool tracing = false;
  std::chrono::steady_clock::time_point wall0;

  ResiduePool(const Batch& batch, std::deque<ResultPart>& out, unsigned n_thr)
      : b(batch), parts(out), stats(n_thr), live(n_thr), errs(n_thr), busy_ms(n_thr, 0.0), trace(n_thr) {
    for (unsigned ti = 0; ti < n_thr; ++ti) threads.emplace_back([this, ti] { run(ti); });
  }
  void run(unsigned ti) {
    for (;;) {
      Task t;
      {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return closed || !queue.empty(); });
        if (queue.empty()) return;
        t = queue.front();
        queue.pop_front();
      }
      if (errs[ti]) continue;  // keep draining so that finish() returns
      const auto t0 = std::chrono::steady_clock::now();
      try {
        if (b.mode == 1) {
          ResidueNormal r(b, *t.raw);
          r.run(t.tx_lo, t.tx_hi, parts[t.part].host, stats[ti]);
          take_device_records(*t.raw, t.tx_lo, t.tx_hi, parts[t.part]);
        } else {
          Residue r(b, *t.raw);
          r.run(t.tx_lo, t.tx_hi, parts[t.part].host, stats[ti]);
          live[ti].insert(live[ti].end(), r.seg_live_.begin(), r.seg_live_.end());
          // the device-built records of this block's transcripts: copied out of the (reused, page-locked) download buffers in
          // their compact form; they are rendered when the result is read or written
          take_device_records(*t.raw, t.tx_lo, t.tx_hi, parts[t.part]);
        }
      } catch (...) {
        errs[ti] = std::current_exception();
      }
      const auto t1 = std::chrono::steady_clock::now();
      busy_ms[ti] += std::chrono::duration<double, std::milli>(t1 - t0).count();
      if (tracing) trace[ti].push_back(Trace{t.part, std::chrono::duration<double, std::milli>(t1 - wall0).count(), std::chrono::duration<double, std::milli>(t1 - t0).count()});
    }
  }
  void push(const PhaseRaw* raw, uint32_t tx_lo, uint32_t tx_hi, size_t part) {
    {
      std::lock_guard<std::mutex> lk(mu);
      queue.push_back(Task{raw, tx_lo, tx_hi, part});
    }
    cv.notify_one();
  }
  void finish() {
    {
      std::lock_guard<std::mutex> lk(mu);
      closed = true;
    }
    cv.notify_all();
    for (auto& t : threads) t.join();
    threads.clear();
  }
  ~ResiduePool() {
    if (!threads.empty()) finish();
  }
};

unsigned residue_threads(uint32_t n_tx) {
  // host threads for the residue: MPH_HOST_THREADS, else all cores but one (a multi-GPU launcher gives every rank its
  // share). The spare core is for the calling thread, which queues the stages and waits on the stream: when it has to
  // compete with the workers every stage hand-over is late (measured on a 16-core B200 host: 21.5 -> 20.7 ms per call).
  const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  unsigned n_thr = std::min<unsigned>(hw >= 4 ? hw - 1 : hw, 32u);
  if (const char* ht = getenv("MPH_HOST_THREADS")) n_thr = std::max(1, atoi(ht));
  if (n_tx < 256) n_thr = 1;
  return n_thr;
}

// kernels + download + residue for the stages; `copied` tells whether the inputs are already on the device
void phase_stages(mph_ctx* c, const std::vector<Stage>& stages, bool copied, mph_result** out) {
  const mph_batch* mb = c->cur;
  const Batch& b = mb->b;
  const auto wall0 = std::chrono::steady_clock::now();
  const uint64_t launches0 = mphk::kernel_launches_on_this_thread();
  const size_t ns = stages.size();
  if (c->raws.size() < ns) c->raws.resize(ns);
  if (c->ev_copy.size() < ns + 1) {
    const size_t old = c->ev_copy.size();
    c->ev_copy.resize(ns + 1);
    for (size_t i = old; i < c->ev_copy.size(); ++i) CU(cudaEventCreate(&c->ev_copy[i]));
  }
  CU(cudaMemsetAsync(c->sums.p, 0, 3 * sizeof(unsigned long long), c->stream));
  // Host -> device copies go to the copy stream, the compute stream waits per stage. From pinned buffers they are all
  // queued now (asynchronous, back to back at link speed); from pageable buffers cudaMemcpyAsync blocks the caller, so
  // stage s + 1 is queued after the kernels of stage s have been launched.
  size_t copies_queued = 0;
  auto queue_copies = [&](size_t upto) {
    for (; copies_queued < upto && copies_queued < ns; ++copies_queued) {
      copy_stage(c, mb, stages[copies_queued], copies_queued == 0, c->copy_stream);
      CU(cudaEventRecord(c->ev_copy[copies_queued], c->copy_stream));
    }
  };
  if (!copied) {
    CU(cudaEventRecord(c->ev_copy[ns], c->copy_stream));
    queue_copies(mb->pinned ? ns : 1);
  }
  std::unique_ptr<mph_result> res(new mph_result);
  res->mode = b.mode;
  const uint32_t n_tx = uint32_t(b.txs.size());
  const unsigned n_thr = residue_threads(n_tx);
  // record blocks in transcript order: every stage contributes ceil(n / blk) of them. A stage is cut into at least four
  // blocks per worker (16 .. 128 transcripts each), so that the residue of the last, short stage still spreads over all
  // workers: that residue is the tail of the call that nothing overlaps.
  std::vector<uint32_t> blk(ns, 128);
  std::vector<size_t> part0(ns + 1, 0);
  for (size_t s = 0; s < ns; ++s) {
    const uint64_t n = stages[s].hi.txs - stages[s].lo.txs;
    blk[s] = uint32_t(std::min<uint64_t>(128, std::max<uint64_t>(16, n / (4 * uint64_t(n_thr)))));
    part0[s + 1] = part0[s] + size_t((n + blk[s] - 1) / blk[s]);
  }
  std::deque<ResultPart> parts(part0[ns]);
  // transcript metadata of the result: copied while the first host -> device copy is in flight
  res->tx_id.reserve(b.txs.size()); res->gene_id.reserve(b.txs.size()); res->gene_name.reserve(b.txs.size()); res->chrom.reserve(b.txs.size());
  res->tx_reverse.reserve(b.txs.size());
  res->vars = b.vars;
  res->var_prot = b.var_prot;
  if (b.mode == 1) res->ref = b.ref;
  for (auto& t : b.txs) {
    res->tx_id.push_back(t.id);
    res->gene_id.push_back(b.genes[t.gene].id);
    res->gene_name.push_back(b.genes[t.gene].name);
    res->chrom.push_back(b.genes[t.gene].chrom);
    res->tx_reverse.push_back(t.reverse ? 1 : 0);
  }
  uint64_t n_iw_total = 0;
  const bool timeline = getenv("MPH_TIMELINE") != nullptr;  // measurement hook
  {
    ResiduePool pool(b, parts, n_thr);
    pool.tracing = timeline;
    pool.wall0 = wall0;
    try {
      for (size_t s = 0; s < ns; ++s) {
        const Stage& st = stages[s];
        if (!copied) CU(cudaStreamWaitEvent(c->stream, c->ev_copy[s], 0));
        set_ranges(c, st);
        c->stage_seg_lo = uint32_t(st.lo.segs);
        c->stage_seg_hi = uint32_t(st.hi.segs);
        c->stage_tx_lo = uint32_t(st.lo.txs);
        c->stage_tx_hi = uint32_t(st.hi.txs);
        if (!(copied && c->kernels_done)) run_kernels(c);
        if (!copied) queue_copies(s + 2);
        fetch_stage(c, st, c->raws[s], &n_iw_total);
        if (timeline) fprintf(stderr, "[mph] stage %zu downloaded at %.2f ms\n", s, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count());
        size_t part = part0[s];
        for (uint32_t lo = uint32_t(st.lo.txs); lo < uint32_t(st.hi.txs); lo += blk[s], ++part)
          pool.push(&c->raws[s], lo, std::min<uint32_t>(uint32_t(st.hi.txs), lo + blk[s]), part);
      }
    } catch (...) {
      pool.finish();
      throw;
    }
    if (timeline) fprintf(stderr, "[mph] last stage queued at %.2f ms\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count());
    pool.finish();
    if (timeline) {
      fprintf(stderr, "[mph] residue finished at %.2f ms\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count());
      for (size_t s = 0; s < ns; ++s) {
        double busy = 0, last = 0;
        size_t n = 0;
        for (auto& tr : pool.trace)
          for (auto& e : tr)
            if (e.part >= part0[s] && e.part < part0[s + 1]) { busy += e.ms; last = std::max(last, e.end_ms); ++n; }
        fprintf(stderr, "[mph] residue of stage %zu: %zu blocks of %u transcripts, %.2f ms of worker time, last block done at %.2f ms\n", s, n, blk[s], busy, last);
      }
    }
    for (auto& e : pool.errs)
      if (e) std::rethrow_exception(e);
    ResidueStats stt;
    double busy = 0;
    for (unsigned ti = 0; ti < n_thr; ++ti) {
      stt.windows += pool.stats[ti].windows;
      stt.read_windows += pool.stats[ti].read_windows;
      busy += pool.busy_ms[ti];
    }
    c->timing.residue_ms = busy / n_thr;
    c->timing.windows = stt.windows;
    c->timing.read_windows = stt.read_windows;
    // statistics: depth summed on the device over the windows the reference reaches (the normal-mode residue visits
    // every window and sums the depth itself)
    {
      std::vector<uint32_t> live(b.segs.size() + 1, 0);
      for (auto& pl : pool.live)
        for (auto& sl : pl) live[sl.first] = sl.second;
      CU(cudaMemcpyAsync(c->seg_live.p, live.data(), live.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
      Stage all;
      all.lo = b.marks.front();
      all.hi = b.marks.back();
      all.pair_hi = uint32_t(mb->pairs.size());
      set_ranges(c, all);
      mphk::launch_live_depth(c->d, c->stream);
      unsigned long long sums[3];
      CU(cudaMemcpyAsync(sums, c->sums.p, sizeof sums, cudaMemcpyDeviceToHost, c->stream));
      CU(cudaStreamSynchronize(c->stream));
      c->timing.read_windows += sums[1];
      c->timing.windows += sums[2];  // live windows of the device-class transcripts (counted on the device)
    }
  }
  if (!copied) {
    float ms;
    CU(cudaEventElapsedTime(&ms, c->ev_copy[ns], c->ev_copy[ns - 1]));
    c->timing.h2d_ms = ms;
  }
  res->part_base.assign(1, 0);
  for (auto& p : parts) res->part_base.push_back(res->part_base.back() + p.size());
  res->parts = std::move(parts);
  c->timing.windows_enumerated = b.n_windows;
  c->timing.n_interesting = n_iw_total;
  c->timing.n_records = res->size();
  c->timing.kernel_launches = uint32_t(mphk::kernel_launches_on_this_thread() - launches0);  // counted at the launch sites (MPH_LAUNCH)
  c->timing.n_replay_units = uint32_t(b.replay.size());
  c->timing.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
  if (timeline) fprintf(stderr, "[mph] call finished at %.2f ms\n", c->timing.total_ms);
  *out = res.release();
}

// host buffers in, records out: the pipelined path
void phase_batch_impl(mph_ctx* c, const mph_batch* mb, mph_result** out) {
  c->cur = nullptr;
  prepare(c, mb);
  // stages of about 16 M reads: every stage pays the fixed latency of its kernel chain (the serial replay's longest unit, the
  // junction merges) and the chain of a stage starts only after the previous stage's download, so a few long stages beat
  // many short ones now that the copy is short (6 B per read) and almost no host work is left to hide behind it. Measured
  // on B200, whole-exome shard (35 M reads, 214 MB): 2 stages 11.1 ms, 3: 11.6, 4: 12.4, 6: 15.0, 8: 17.8 ms per call.
  unsigned want = unsigned(std::min<uint64_t>(12, std::max<uint64_t>(1, (mb->b.n_reads() + 8000000) / 16000000)));
  if (const char* e = getenv("MPH_STAGES")) want = unsigned(std::max(1, atoi(e)));
  const std::vector<Stage> stages = plan_stages(mb, want);
  c->kernels_done = false;
  // the context must not keep pointing at the caller's batch after the call, whichever way it ends: the batch may be
  // destroyed next, and a later mph_phase_resident / mph_phase_collect has to fail cleanly ("no batch uploaded")
  try {
    phase_stages(c, stages, false, out);
  } catch (...) {
    c->cur = nullptr;
    throw;
  }
  c->cur = nullptr;
}

void write_all(int fd, const std::string& s) {
  size_t off = 0;
  while (off < s.size()) {
    ssize_t n = ::write(fd, s.data() + off, s.size() - off);
    if (n <= 0) throw std::runtime_error("write failed");
    off += size_t(n);
  }
}

}  // namespace

// ---- secondary path helpers (device translation / hash set) ---------------------------------
namespace {

void dev_translate(mph_ctx* c, const uint8_t* nt, const uint64_t* off, const int8_t* frame, uint64_t n, uint8_t* aa, const uint64_t* aa_off, uint8_t* bad) {
  CU(cudaSetDevice(c->device));
  if (n == 0) return;
  DevBuf<uint8_t> d_nt, d_aa, d_bad;
  DevBuf<uint64_t> d_off, d_aoff;
  DevBuf<int8_t> d_fr;
  d_nt.ensure(off[n] + 1); d_aa.ensure(aa_off[n] + 1); d_bad.ensure(n); d_off.ensure(n + 1); d_aoff.ensure(n + 1); d_fr.ensure(n);
  try {
    if (off[n]) CU(cudaMemcpyAsync(d_nt.p, nt, off[n], cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_off.p, off, (n + 1) * 8, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_aoff.p, aa_off, (n + 1) * 8, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_fr.p, frame, n, cudaMemcpyHostToDevice, c->stream));
    mphk::launch_translate(d_nt.p, d_off.p, d_fr.p, n, d_aa.p, d_aoff.p, d_bad.p, c->stream);
    CU(cudaGetLastError());
    if (aa_off[n]) CU(cudaMemcpyAsync(aa, d_aa.p, aa_off[n], cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(bad, d_bad.p, n, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  } catch (...) {
    d_nt.release(); d_aa.release(); d_bad.release(); d_off.release(); d_aoff.release(); d_fr.release();
    throw;
  }
  d_nt.release(); d_aa.release(); d_bad.release(); d_off.release(); d_aoff.release(); d_fr.release();
}

void dev_set_load(mph_ctx* c, const uint8_t* peptides, uint32_t k, uint64_t n) {
  CU(cudaSetDevice(c->device));
  if (k == 0 || k > 255) throw Unsupported("peptide length must be 1..255");
  const bool longk = k > 12;  // 5 bits per letter fill a 64-bit key up to 12 letters; longer peptides are compared as bytes
  if (longk && n > 0xFFFFFFF0ull) throw Unsupported("more than 2^32 peptides of more than 12 letters");
  uint64_t slots = 1024;
  while (slots < 2 * n + 16) slots <<= 1;
  if (longk) c->set_idx.ensure(slots);
  else c->set_table.ensure(slots);
  c->set_mask = slots - 1;
  c->set_k = k;
  if (longk) CU(cudaMemsetAsync(c->set_idx.p, 0, slots * 4, c->stream));
  else CU(cudaMemsetAsync(c->set_table.p, 0, slots * 8, c->stream));
  c->sums.ensure(2);
  CU(cudaMemsetAsync(c->sums.p, 0, 16, c->stream));
  if (n && longk) {
    c->set_bytes.ensure(n * k);  // stays resident: the slots point into it
    CU(cudaMemcpyAsync(c->set_bytes.p, peptides, n * k, cudaMemcpyHostToDevice, c->stream));
    mphk::launch_set_insert_long(c->set_bytes.p, k, n, c->set_idx.p, c->set_mask, c->sums.p, c->stream);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
  } else if (n) {
    DevBuf<uint8_t> d_p;
    d_p.ensure(n * k);
    try {
      CU(cudaMemcpyAsync(d_p.p, peptides, n * k, cudaMemcpyHostToDevice, c->stream));
      mphk::launch_set_insert(d_p.p, k, n, c->set_table.p, c->set_mask, c->sums.p, c->stream);
      CU(cudaGetLastError());
      CU(cudaStreamSynchronize(c->stream));
    } catch (...) {
      d_p.release();
      throw;
    }
    d_p.release();
  }
  unsigned long long nd = 0;
  CU(cudaMemcpyAsync(&nd, c->sums.p, 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  c->set_distinct = nd;
}

void dev_set_probe(mph_ctx* c, const uint8_t* queries, uint32_t k, uint64_t n, uint8_t* hit) {
  CU(cudaSetDevice(c->device));
  if (c->set_k == 0) throw std::runtime_error("no peptide set loaded");
  if (n == 0) return;
  if (k != c->set_k) {  // a peptide of another length cannot be in the set
    memset(hit, 0, n);
    return;
  }
  DevBuf<uint8_t> d_q, d_h;
  d_q.ensure(n * k); d_h.ensure(n);
  try {
    CU(cudaMemcpyAsync(d_q.p, queries, n * k, cudaMemcpyHostToDevice, c->stream));
    CU(cudaEventRecord(c->ev[2], c->stream));
    if (k > 12) mphk::launch_set_probe_long(d_q.p, k, n, c->set_bytes.p, c->set_idx.p, c->set_mask, d_h.p, c->stream);
    else mphk::launch_set_probe(d_q.p, k, n, c->set_table.p, c->set_mask, d_h.p, c->stream);
    CU(cudaEventRecord(c->ev[3], c->stream));
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(hit, d_h.p, n, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    float probe_ms = 0;
    CU(cudaEventElapsedTime(&probe_ms, c->ev[2], c->ev[3]));
    c->timing.k1_ms = probe_ms;  // measurement: the probe kernel alone
  } catch (...) {
    d_q.release(); d_h.release();
    throw;
  }
  d_q.release(); d_h.release();
}

std::vector<std::string> dev_set_export(mph_ctx* c) {
  std::vector<std::string> out;
  if (c->set_k == 0 || c->set_distinct == 0) return out;
  const uint32_t k = c->set_k;
  DevBuf<uint8_t> d_o;
  d_o.ensure(c->set_distinct * k);
  std::vector<uint8_t> host(c->set_distinct * k);
  try {
    CU(cudaMemsetAsync(c->sums.p, 0, 16, c->stream));
    if (k > 12) mphk::launch_set_export_long(c->set_idx.p, c->set_mask + 1, c->set_bytes.p, k, d_o.p, c->sums.p, c->stream);
    else mphk::launch_set_export(c->set_table.p, c->set_mask + 1, k, d_o.p, c->sums.p, c->stream);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(host.data(), d_o.p, host.size(), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  } catch (...) {
    d_o.release();
    throw;
  }
  d_o.release();
  for (uint64_t i = 0; i < c->set_distinct; ++i) out.emplace_back(reinterpret_cast<const char*>(host.data() + i * k), k);
  return out;
}

// adapters for host/peptides_host.hpp
pep::TranslateFn make_translate(mph_ctx* c) {
  return [c](const std::vector<std::string>& nt, const std::vector<int8_t>& frame, std::vector<std::string>& aa, std::vector<uint8_t>& bad) {
    const uint64_t n = nt.size();
    std::vector<uint64_t> off(n + 1, 0), aoff(n + 1, 0);
    for (uint64_t i = 0; i < n; ++i) {
      off[i + 1] = off[i] + nt[i].size();
      aoff[i + 1] = aoff[i] + (nt[i].size() >= 2 ? nt[i].size() / 3 : 0);
    }
    std::vector<uint8_t> flat(off[n] + 1), out(aoff[n] + 1);
    for (uint64_t i = 0; i < n; ++i) memcpy(flat.data() + off[i], nt[i].data(), nt[i].size());
    bad.assign(n, 0);
    dev_translate(c, flat.data(), off.data(), frame.data(), n, out.data(), aoff.data(), bad.data());
    aa.resize(n);
    for (uint64_t i = 0; i < n; ++i) aa[i].assign(reinterpret_cast<const char*>(out.data() + aoff[i]), size_t(aoff[i + 1] - aoff[i]));
  };
}

std::vector<uint8_t> flatten_k(const std::vector<std::string>& v, uint32_t k, std::vector<uint64_t>& index) {
  std::vector<uint8_t> flat;
  for (uint64_t i = 0; i < v.size(); ++i)
    if (v[i].size() == k) {
      index.push_back(i);
      flat.insert(flat.end(), v[i].begin(), v[i].end());
    }
  return flat;
}

}  // namespace

extern "C" {

int mph_ctx_create(int device, mph_ctx** out) {
  if (!out) return fail(nullptr, MPH_ERR_INPUT, "out is NULL");
  *out = nullptr;
  std::unique_ptr<mph_ctx> c(new mph_ctx);
  int rc = guarded(nullptr, [&] {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) throw CudaError(std::string("no CUDA device: ") + cudaGetErrorString(e));
    if (device < 0 || device >= n) throw CudaError("device index out of range");
    c->device = device;
    // A result is a few hundred record blocks of ~100 KB that the host threads fill on every call and the caller frees
    // afterwards. With glibc's default trim threshold (128 KB) the freed heap tops go back to the kernel each time and the
    // next call pays a page fault per 4 KB again - most of the host threads' time once the records come from the device.
    // Keep freed memory in the heaps (MPH_KEEP_HEAP=0 leaves the process's malloc settings alone).
    {
      static std::once_flag heap_once;
      std::call_once(heap_once, [] {
        const char* e = getenv("MPH_KEEP_HEAP");
        if (e && *e == '0') return;
#ifdef M_TRIM_THRESHOLD
        mallopt(M_TRIM_THRESHOLD, 1 << 30);
        mallopt(M_MMAP_THRESHOLD, 1 << 28);
#endif
      });
    }
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c->replay_stream, cudaStreamNonBlocking));
    { int sms = 0; if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) c->sm_count = sms; }
    for (auto& e3 : c->ev_rp) CU(cudaEventCreate(&e3));
    for (auto& e2 : c->ev) CU(cudaEventCreate(&e2));
  });
  if (rc != MPH_OK) return rc;
  *out = c.release();
  return MPH_OK;
}

void mph_ctx_destroy(mph_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  for (auto& e : c->ev)
    if (e) cudaEventDestroy(e);
  for (auto& kv : c->pinned_dl) cudaHostUnregister(const_cast<void*>(kv.first));
  c->pinned_dl.clear();
  for (auto& e : c->ev_copy)
    if (e) cudaEventDestroy(e);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  for (auto& e : c->ev_rp)
    if (e) cudaEventDestroy(e);
  if (c->replay_stream) cudaStreamDestroy(c->replay_stream);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;  // the remaining device buffers are released by ~DevBuf
}

const char* mph_last_error(const mph_ctx* ctx) { return ctx ? ctx->last_error.c_str() : g_last_error.c_str(); }

int mph_packer_create(uint32_t window_len, int mode, mph_packer** out) {
  if (!out) return fail(nullptr, MPH_ERR_INPUT, "out is NULL");
  if (mode != 0 && mode != 1) return fail(nullptr, MPH_ERR_UNSUPPORTED, "mode must be 0 (somatic) or 1 (normal)");
  if (window_len == 0 || window_len % 3 != 0) return fail(nullptr, MPH_ERR_UNSUPPORTED, "window length must be a positive multiple of 3");
  *out = new mph_packer;
  (*out)->p.reset(new Packer(window_len, mode));
  (*out)->mode = mode;
  return MPH_OK;
}

void mph_packer_destroy(mph_packer* p) { delete p; }

int mph_packer_add_gene(mph_packer* p, const mph_gene_in* g) {
  if (!p || !g || !p->p) return fail(nullptr, MPH_ERR_INPUT, "null argument");
  return guarded(nullptr, [&] {
    HostGene hg;
    hg.id = g->gene_id ? g->gene_id : "";
    hg.name = g->gene_name ? g->gene_name : "";
    hg.chrom = g->chrom ? g->chrom : "";
    hg.start = g->gene_start;
    hg.end = g->gene_end;
    for (uint32_t t = 0; t < g->n_tx; ++t) {
      HostTranscript ht;
      ht.id = g->tx_id[t];
      ht.reverse = g->tx_reverse[t] != 0;
      for (uint32_t e = g->tx_exon_off[t]; e < g->tx_exon_off[t + 1]; ++e) ht.exons.push_back(HostExon{g->exon_start[e], g->exon_end[e], g->exon_frame[e]});
      hg.transcripts.push_back(std::move(ht));
    }
    std::vector<HostRead> reads(g->n_reads);
    for (uint32_t r = 0; r < g->n_reads; ++r) {
      HostRead& h = reads[r];
      h.start = g->read_start[r];
      h.end = g->read_end[r];
      h.l_seq = g->read_lseq[r];
      h.seq4 = g->seq4 + g->read_seq_off[r];
      h.qual = g->qual + g->read_qual_off[r];
      h.cigar = g->cigar + g->read_cigar_off[r];
      h.n_cigar = g->read_cigar_off[r + 1] - g->read_cigar_off[r];
      h.qname_hash = g->read_qname_hash ? g->read_qname_hash[r] : r;
    }
    std::vector<std::vector<HostVariant>> sites;
    for (uint32_t v = 0; v < g->n_vars; ++v) {
      HostVariant hv;
      hv.pos = g->var_pos[v];
      hv.kind = g->var_kind[v];
      hv.germline = g->var_germline[v] != 0;
      hv.alt = g->var_alt[v];
      hv.len = g->var_len[v];
      if (hv.kind == MPH_INS) hv.ins.assign(reinterpret_cast<const char*>(g->ins_bytes + g->var_ins_off[v]), g->var_ins_off[v + 1] - g->var_ins_off[v]);
      if (g->var_prot_change && g->var_prot_change[v]) hv.prot_change = g->var_prot_change[v];
      if (sites.empty() || sites.back().back().pos != hv.pos) sites.emplace_back();
      sites.back().push_back(std::move(hv));
    }
    std::vector<uint8_t> refseq(g->refseq, g->refseq + g->refseq_len);
    p->p->add_gene(hg, reads, g->max_read_len, sites, std::move(refseq));
  });
}

int mph_packer_finish(mph_packer* p, int pin, mph_batch** out) {
  if (!p || !out || !p->p) return fail(nullptr, MPH_ERR_INPUT, "null argument");
  std::unique_ptr<mph_batch> mb(new mph_batch);
  int rc = guarded(nullptr, [&] {
    mb->b = std::move(p->p->batch());
    p->p.reset();
    finish_batch(mb.get(), pin != 0);
  });
  if (rc != MPH_OK) return rc;
  *out = mb.release();
  return MPH_OK;
}

void mph_batch_destroy(mph_batch* b) { delete b; }

int mph_batch_get_view(const mph_batch* mb, mph_batch_view* v) {
  if (!mb || !v) return fail(nullptr, MPH_ERR_INPUT, "null argument");
  const Batch& b = mb->b;
  memset(v, 0, sizeof *v);
  v->window_len = b.window_len;
  v->n_reads = b.n_reads(); v->n_vars = b.vars.size(); v->n_segments = b.segs.size(); v->n_chunks = b.chunks.size();
  v->n_windows = b.n_windows; v->n_transcripts = b.txs.size(); v->n_genes = b.genes.size();
  v->read_start = b.read_start.data(); v->read_end = b.read_end.data(); v->read_flags = b.read_flags.data();
  v->n_variant_reads = b.vr_read.size();
  v->vr_read = b.vr_read.data(); v->vr_vlo = b.vr_vlo.data(); v->vr_seq_off = b.vr_seq_off.data(); v->vr_cig_off = b.vr_cig_off.data();
  v->vr_lseq = b.vr_lseq.data(); v->vr_ncig = b.vr_ncig.data(); v->vr_nv = b.vr_nv.data();
  v->bases = b.bases.data(); v->bases_bytes = b.bases.size(); v->cigars = b.cigars.data(); v->n_cigar_ops = b.cigars.size();
  v->vars = b.vars.data(); v->segments = b.segs.data(); v->chunks = b.chunks.data(); v->ref = b.ref.data(); v->ref_bytes = b.ref.size();
  v->h2d_bytes = mb->h2d_bytes;
  return MPH_OK;
}

int mph_batch_upload(mph_ctx* ctx, const mph_batch* batch) {
  if (!ctx || !batch) return fail(ctx, MPH_ERR_INPUT, "null argument");
  return guarded(ctx, [&] {
    ctx->cur = nullptr;  // stays null if the upload fails
    try {
      prepare(ctx, batch);
      const std::vector<Stage> all = plan_stages(batch, 1);
      CU(cudaEventRecord(ctx->ev[0], ctx->stream));
      copy_stage(ctx, batch, all[0], true, ctx->stream);
      CU(cudaEventRecord(ctx->ev[1], ctx->stream));
      CU(cudaStreamSynchronize(ctx->stream));
    } catch (...) {
      ctx->cur = nullptr;
      throw;
    }
    float ms;
    CU(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
    ctx->timing.h2d_ms = ms;
    ctx->kernels_done = false;
  });
}

int mph_phase_resident(mph_ctx* ctx) {
  if (!ctx) return fail(ctx, MPH_ERR_INPUT, "null argument");
  return guarded(ctx, [&] {
    if (!ctx->cur) throw std::runtime_error("no batch uploaded");
    CU(cudaSetDevice(ctx->device));
    const std::vector<Stage> all = plan_stages(ctx->cur, 1);
    set_ranges(ctx, all[0]);
    ctx->stage_seg_lo = 0;
    ctx->stage_seg_hi = uint32_t(all[0].hi.segs);
    ctx->stage_tx_lo = 0;
    ctx->stage_tx_hi = uint32_t(all[0].hi.txs);
    CU(cudaMemsetAsync(ctx->sums.p, 0, 3 * sizeof(unsigned long long), ctx->stream));
    // (an arena that is too small makes the kernels skip work: look at the overflow flags like mph_phase_collect does, so
    // that the step this entry point times is always the complete one)
    for (int attempt = 0;; ++attempt) {
      const uint64_t launches0 = mphk::kernel_launches_on_this_thread();
      run_kernels(ctx);
      ctx->timing.kernel_launches = uint32_t(mphk::kernel_launches_on_this_thread() - launches0);  // of the complete pass
      uint32_t ctr[mphk::CTR_COUNT];
      CU(cudaMemcpyAsync(ctr, ctx->counters.p, sizeof ctr, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaStreamSynchronize(ctx->stream));
      if (!(grow_arenas(ctx, ctr) && attempt < 6)) break;
    }
    ctx->timing.k1_ms = ctx->timing.k2_ms = ctx->timing.k3_ms = ctx->timing.k4_ms = ctx->timing.k5_ms = ctx->timing.replay_ms = ctx->timing.kernels_ms = 0;
    add_kernel_times(ctx);
    ctx->kernels_done = true;
  });
}

int mph_phase_collect(mph_ctx* ctx, mph_result** out) {
  if (!ctx || !out) return fail(ctx, MPH_ERR_INPUT, "null argument");
  *out = nullptr;
  return guarded(ctx, [&] {
    if (!ctx->cur) throw std::runtime_error("no resident run to collect");
    CU(cudaSetDevice(ctx->device));
    const std::vector<Stage> all = plan_stages(ctx->cur, 1);
    ctx->timing.k1_ms = ctx->timing.k2_ms = ctx->timing.k3_ms = ctx->timing.k4_ms = ctx->timing.k5_ms = ctx->timing.replay_ms = ctx->timing.kernels_ms = 0;
    ctx->timing.d2h_ms = 0;
    ctx->timing.d2h_bytes = 0;
    phase_stages(ctx, all, true, out);
  });
}

int mph_phase_batch(mph_ctx* ctx, const mph_batch* batch, mph_result** out) {
  if (!ctx || !batch || !out) return fail(ctx, MPH_ERR_INPUT, "null argument");
  *out = nullptr;
  return guarded(ctx, [&] { phase_batch_impl(ctx, batch, out); });
}

int mph_ctx_timing(const mph_ctx* ctx, mph_timing* out) {
  if (!ctx || !out) return fail(nullptr, MPH_ERR_INPUT, "null argument");
  *out = ctx->timing;
  return MPH_OK;
}

void mph_result_destroy(mph_result* r) { delete r; }
uint64_t mph_result_count(const mph_result* r) { return r ? r->size() : 0; }

int mph_result_get(const mph_result* r, uint64_t i, mph_record* o) {
  if (!r || !o || i >= r->size()) return fail(nullptr, MPH_ERR_INPUT, "record index out of range");
  const OutRecord& rec = const_cast<mph_result*>(r)->at(i);  // renders the record's part on first access
  const uint32_t t = rec.info.tx;
  o->id = rec.info.id.c_str();
  o->transcript = r->tx_id[t].c_str(); o->gene_id = r->gene_id[t].c_str(); o->gene_name = r->gene_name[t].c_str(); o->chrom = r->chrom[t].c_str();
  o->offset = rec.info.offset; o->frame = rec.info.frame; o->freq = rec.info.freq;
  o->depth = rec.info.depth; o->nvar = rec.info.nvar; o->nsomatic = rec.info.nsomatic;
  o->nvariant_sites = rec.info.nvariant_sites; o->nsomvariant_sites = rec.info.nsomvariant_sites;
  o->reverse = r->tx_reverse[t];
  o->variant_sites = rec.info.variant_sites.c_str(); o->somatic_positions = rec.info.somatic_positions.c_str();
  o->somatic_aa_change = rec.info.somatic_aa_change.c_str(); o->germline_positions = rec.info.germline_positions.c_str();
  o->germline_aa_change = rec.info.germline_aa_change.c_str(); o->normal_sequence = rec.info.normal_sequence.c_str();
  o->mutant_sequence = rec.info.mutant_sequence.c_str();
  o->fasta_mutant = rec.has_mt ? rec.mt_str().c_str() : nullptr;
  o->fasta_normal = rec.has_wt ? rec.wt_str().c_str() : nullptr;
  return MPH_OK;
}

int mph_result_write(const mph_result* r, int fd_fasta, int fd_tsv, int fd_normal, int* header_written) {
  if (!r) return fail(nullptr, MPH_ERR_INPUT, "null argument");
  return guarded(nullptr, [&] {
    static const char* header =
        "id\ttranscript\tgene_id\tgene_name\tchrom\toffset\tframe\tfreq\tdepth\tnvar\tnsomatic\tnvariant_sites\tnsomvariant_sites\t"
        "strand\tvariant_sites\tsomatic_positions\tsomatic_aa_change\tgermline_positions\tgermline_aa_change\tnormal_sequence\t"
        "mutant_sequence\n";
    static const char* header_normal =
        "id\ttranscript\tgene_id\tgene_name\tchrom\toffset\tframe\tfreq\tdepth\tnvar\tnsomatic\tnvariant_sites\tnsomvariant_sites\t"
        "strand\tvariant_sites\tsomatic_positions\tsomatic_aa_change\tgermline_positions\tgermline_aa_change\tpeptide_sequence\n";
    int hw = header_written ? *header_written : 0;
    const bool normal_mode = r->mode == 1;  // 20 columns, the last one is peptide_sequence (src/normal_microphasing.rs:80-102)
    // text of a run of parts; the parts are independent, so several host threads render and the chunks are written in order
    struct Chunk { std::string fa, tsv, nrm; };
    const size_t n_parts = r->parts.size();
    unsigned n_thr = std::max(1u, std::min<unsigned>(std::thread::hardware_concurrency(), 16u));
    if (const char* ht = getenv("MPH_HOST_THREADS")) n_thr = unsigned(std::max(1, atoi(ht)));
    if (r->size() < 20000) n_thr = 1;
    n_thr = unsigned(std::min<size_t>(n_thr, std::max<size_t>(1, n_parts)));
    std::vector<Chunk> chunks(n_thr);
    auto render = [&](unsigned ti) {
      Chunk& ck = chunks[ti];
      const size_t p0 = n_parts * ti / n_thr, p1 = n_parts * (ti + 1) / n_thr;
      char num[32];
      auto put_u = [&](std::string& dst, uint64_t v) { auto e = std::to_chars(num, num + sizeof num, v); dst.append(num, e.ptr); };
      for (size_t pi = p0; pi < p1; ++pi)
        r->for_each(r->parts[pi], [&](const OutRecord& rec) {
          const uint32_t t = rec.info.tx;
          std::string& fa = ck.fa; std::string& tsv = ck.tsv; std::string& nrm = ck.nrm;
          if (rec.has_mt) { fa += '>'; fa += rec.info.id; fa += '\n'; fa += rec.mt_str(); fa += '\n'; }
          if (rec.has_wt) { nrm += '>'; nrm += rec.info.id; nrm += '\n'; nrm += rec.wt_str(); nrm += '\n'; }
          // ids, transcript / gene names, numbers and sequences never need quoting; the free-text columns go through csv_field
          tsv += rec.info.id; tsv += '\t';
          mphfmt::csv_field(r->tx_id[t], '\t', tsv); tsv += '\t';
          mphfmt::csv_field(r->gene_id[t], '\t', tsv); tsv += '\t';
          mphfmt::csv_field(r->gene_name[t], '\t', tsv); tsv += '\t';
          mphfmt::csv_field(r->chrom[t], '\t', tsv); tsv += '\t';
          put_u(tsv, rec.info.offset); tsv += '\t';
          put_u(tsv, rec.info.frame); tsv += '\t';
          tsv += mphfmt::format_f64(rec.info.freq); tsv += '\t';
          put_u(tsv, rec.info.depth); tsv += '\t';
          put_u(tsv, rec.info.nvar); tsv += '\t';
          put_u(tsv, rec.info.nsomatic); tsv += '\t';
          put_u(tsv, rec.info.nvariant_sites); tsv += '\t';
          put_u(tsv, rec.info.nsomvariant_sites); tsv += '\t';
          tsv += r->tx_reverse[t] ? "Reverse" : "Forward"; tsv += '\t';
          mphfmt::csv_field(rec.info.variant_sites, '\t', tsv); tsv += '\t';
          mphfmt::csv_field(rec.info.somatic_positions, '\t', tsv); tsv += '\t';
          mphfmt::csv_field(rec.info.somatic_aa_change, '\t', tsv); tsv += '\t';
          mphfmt::csv_field(rec.info.germline_positions, '\t', tsv); tsv += '\t';
          mphfmt::csv_field(rec.info.germline_aa_change, '\t', tsv); tsv += '\t';
          if (!normal_mode) { mphfmt::csv_field(std::string(rec.info.normal_sequence), '\t', tsv); tsv += '\t'; }
          mphfmt::csv_field(std::string(rec.info.mutant_sequence), '\t', tsv);
          tsv += '\n';
        });
    };
    if (n_thr == 1) {
      render(0);
    } else {
      std::vector<std::thread> th;
      for (unsigned ti = 0; ti < n_thr; ++ti) th.emplace_back(render, ti);
      for (auto& t : th) t.join();
    }
    for (Chunk& ck : chunks) {
      if (fd_fasta >= 0) write_all(fd_fasta, ck.fa);
      if (fd_tsv >= 0 && !ck.tsv.empty()) {
        if (!hw) { write_all(fd_tsv, normal_mode ? header_normal : header); hw = 1; }
        write_all(fd_tsv, ck.tsv);
      }
      if (fd_normal >= 0) write_all(fd_normal, ck.nrm);
    }
    if (header_written) *header_written = hw;
  });
}

static void add_timing(mph_timing& a, const mph_timing& t) {
  a.h2d_ms += t.h2d_ms; a.k1_ms += t.k1_ms; a.k2_ms += t.k2_ms; a.k3_ms += t.k3_ms; a.k4_ms += t.k4_ms; a.d2h_ms += t.d2h_ms;
  a.residue_ms += t.residue_ms; a.total_ms += t.total_ms; a.replay_ms += t.replay_ms; a.k5_ms += t.k5_ms; a.pack_ms += t.pack_ms; a.kernels_ms += t.kernels_ms; a.h2d_bytes += t.h2d_bytes; a.d2h_bytes += t.d2h_bytes;
  a.windows += t.windows; a.read_windows += t.read_windows; a.windows_enumerated += t.windows_enumerated; a.n_interesting += t.n_interesting;
  a.n_records += t.n_records; a.kernel_launches += t.kernel_launches; a.n_replay_units += t.n_replay_units;
}

using FilePipeline = ShardPipeline<std::vector<GeneInput>, std::unique_ptr<mph_batch>, std::unique_ptr<mph_result>, mph_timing>;

// The file driver of the single- and multi-device entry points. Without an index the whole BAM is loaded and the genes
// are cut into balanced shards, a fixed run of consecutive shards per device. With an index next to the BAM this thread
// fetches the genes one by one in the reference's one-pass order (reference slice, reads, variants) and closes a shard
// every `reads_per_shard` reads for whichever device is free; it waits while workers + 1 shards are not yet written, so
// the reads held in memory follow the shard size, not the file size, and a failure of the walk (a corrupt block late in
// the BAM) is reported after the shards before it are written, as the reference, which streams, does.
static void run_files(const std::vector<mph_ctx*>& ctxs, const char* bam_path, const char* ref_path, const char* variants_path,
                      const char* gtf_path, const char* fasta_out_path, const char* tsv_path, const char* normal_path,
                      uint32_t window_len, int warn_only, int mode) {
  // BGZF inflate of the alignment file runs on a few host threads (MPH_IO_THREADS, default min(cores, 8))
  // BGZF inflate is the largest single host cost of the file driver (about 0.7 core-seconds per million 150 bp reads with zlib):
  // every core takes blocks
  unsigned io_threads = std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency()), 32u);
  if (const char* e = getenv("MPH_IO_THREADS")) io_threads = unsigned(std::max(1, atoi(e)));
  // host inflate: the reader's own decoder unless MPH_ZLIB_INFLATE=1
  {
    const char* z = getenv("MPH_ZLIB_INFLATE");
    mphio::fast_inflate_enabled().store(!(z && *z == '1'));
  }
  // MPH_GPU_INFLATE=1: the BGZF blocks of a large alignment file are inflated on the device (kernels/inflate_kernels.cu)
  // instead of by zlib on the host threads. Off by default: with one decoder thread per block every input byte and every
  // LZ77 copy is a dependent global-memory access, and the 7 436 blocks of the 183 MB sample take 287 ms (copies included)
  // against 113 ms for zlib on 16 cores (B200, round 2). It is bit-exact (the file-driver parity tests run with it), so it
  // stays as the base of the next step: blocks staged in shared memory and sub-block parallel decoding.
  std::shared_ptr<GpuInflater> gpu_inflate;
  mphio::BgzfInflaterSpec inflater;
  {
    const char* e = getenv("MPH_GPU_INFLATE");
    if (e && *e == '1' && io_threads > 1) {
      gpu_inflate = std::make_shared<GpuInflater>(ctxs[0]->device);
      inflater.fn = [gpu_inflate](const uint8_t* cbuf, size_t cbytes, const mphio::BgzfRaw* raws, size_t n, uint8_t* out, size_t obytes) {
        gpu_inflate->run(cbuf, cbytes, raws, n, out, obytes);
      };
      if (const char* bb = getenv("MPH_GPU_INFLATE_BLOCKS")) inflater.batch_blocks = size_t(std::max(256, atoi(bb)));
    }
  }
  // with an index next to the BAM the genes are streamed: reads are fetched through the index, and batches of 64 blocks
  // keep the read-ahead that a seek throws away small
  const std::string bai = mphio::BamIndex::locate(bam_path);
  mphio::BamFile bam(bam_path, io_threads, inflater, bai.empty() ? 256 : 64);
  std::unique_ptr<mphio::BamIndex> index;
  if (!bai.empty()) index.reset(new mphio::BamIndex(bai, bam.ref_names.size(), bam.file_bytes()));
  mphio::VcfFile vcf(variants_path);
  mphio::FastaIndexed fasta(ref_path);
  // the reference creates its output files before it starts phasing (src/main.rs:79-85)
  auto open_out = [](const char* p) -> int {
    if (std::string(p) == "-") return 1;
    FILE* f = fopen(p, "wb");
    if (!f) throw std::runtime_error(std::string("cannot create ") + p);
    int fd = dup(fileno(f));
    fclose(f);
    return fd;
  };
  const int fd_fa = open_out(fasta_out_path), fd_tsv = open_out(tsv_path), fd_n = normal_path ? open_out(normal_path) : -1;
  auto close_all = [&] {
    if (fd_fa > 2) close(fd_fa);
    if (fd_tsv > 2) close(fd_tsv);
    if (fd_n > 2) close(fd_n);
  };
  try {
    IngestOptions io;
    io.window_len = window_len;
    io.warn_only = warn_only != 0;
    io.mode = mode;
    if (mode == 1) io.min_mapq = 0;  // the normal mode keeps every read (src/normal_microphasing.rs:667-676)
    std::ifstream gf;
    std::istream* gin = &std::cin;
    if (std::string(gtf_path) != "-") {
      gf.open(gtf_path);
      if (!gf) throw std::runtime_error(std::string("cannot open ") + gtf_path);
      gin = &gf;
    }
    const size_t n_dev = ctxs.size();
    auto pack = [&](std::vector<GeneInput>& genes) {
      Packer packer(window_len, mode);
      pack_genes(genes, 0, genes.size(), packer);
      std::unique_ptr<mph_batch> batch(new mph_batch);
      batch->b = std::move(packer.batch());
      finish_batch(batch.get(), false);
      return batch;
    };
    auto phase = [&](size_t dv, std::unique_ptr<mph_batch>& batch, mph_timing& sum) {
      mph_result* res = nullptr;
      phase_batch_impl(ctxs[dv], batch.get(), &res);
      add_timing(sum, ctxs[dv]->timing);  // a device's timing is the sum over its shards
      return std::unique_ptr<mph_result>(res);
    };
    int hw = 0;  // the TSV header goes out with the first row only
    auto write = [&](std::unique_ptr<mph_result>& res) {
      if (mph_result_write(res.get(), fd_fa, fd_tsv, fd_n, &hw) != MPH_OK) throw std::runtime_error(g_last_error);
    };
    std::unique_ptr<ReadBufferLoader> loader;  // whole file: holds the reads the genes point into, so it outlives the pipeline
    std::optional<FilePipeline> pipe;
    std::exception_ptr err;  // a failure of the indexed walk; a failure in the pipeline replaces it, being reported first
    // packing threads per device: one per core up to 12, MPH_PACK_THREADS overrides it
    const size_t cores_per_dev = std::min<size_t>(12, std::max<size_t>(1, std::thread::hardware_concurrency() / n_dev));
    const char* pack_threads = getenv("MPH_PACK_THREADS");
    uint64_t reads_per_shard = mode == 1 ? 2000000ull : 8000000ull;
    const auto t_ingest0 = std::chrono::steady_clock::now();
    double ingest_ms;
    if (index) {
      std::vector<ParsedGene> parsed = read_gtf(*gin, mode);  // the unsorted-GTF panic comes before any output
      if (const char* e = getenv("MPH_SHARD_READS")) reads_per_shard = uint64_t(std::max(1, atoi(e)));
      const size_t n_workers = n_dev * (pack_threads ? size_t(std::max(1, atoi(pack_threads))) : cores_per_dev);
      pipe.emplace(n_dev, n_workers, n_workers + 1, pack, phase, write);
      std::vector<GeneInput> shard;
      uint64_t shard_reads = 0;
      try {
        walk_indexed_genes(std::move(parsed), bam, *index, vcf, fasta, io, [&](GeneInput&& gi) {
          shard_reads += gi.n_reads;
          shard.push_back(std::move(gi));
          if (shard_reads < reads_per_shard) return !pipe->failed();
          shard_reads = 0;
          return pipe->submit(std::exchange(shard, {}), FilePipeline::kAnyDevice);
        });
      } catch (...) {
        err = std::current_exception();  // the genes fetched before the failure are still phased and written
      }
      if (!shard.empty()) pipe->submit(std::move(shard), FilePipeline::kAnyDevice);
      ingest_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_ingest0).count();
    } else {
      loader.reset(new ReadBufferLoader(bam));  // the BAM loads on its own thread while this one parses the GTF and fetches reference slices and variants
      std::vector<GeneInput> genes = ingest_genes_with(*gin, [&]() -> ReadBuffer& { return loader->get(); }, vcf, fasta, io, true);
      ingest_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_ingest0).count();
      // one contiguous gene range per device, no exchange between shards (SURVEY.md §8(e)); a device's range is cut
      // further so that several host threads pack in parallel, while its phase calls run one after the other
      uint64_t total_reads = 0;
      for (auto& g : genes) total_reads += g.n_reads;
      const size_t per_dev = pack_threads ? size_t(std::max(1, atoi(pack_threads))) : total_reads > 200000 * n_dev ? cores_per_dev : 1;
      // more shards than packing threads when the input is large: a shard's records are written and freed as soon as all
      // earlier shards are out, which bounds the memory held in records (the normal mode writes one per window)
      size_t n_shards = std::max<size_t>(n_dev * per_dev, size_t((total_reads + reads_per_shard - 1) / reads_per_shard));
      n_shards = (n_shards + n_dev - 1) / n_dev * n_dev;  // the same number of consecutive shards per device
      const size_t shards_per_dev = n_shards / n_dev;
      const std::vector<size_t> cut = partition_genes(genes, n_shards);
      pipe.emplace(n_dev, std::min(n_shards, n_dev * per_dev), 0, pack, phase, write);
      for (size_t k = 0; k < n_shards; ++k) {
        std::vector<GeneInput> shard(std::make_move_iterator(genes.begin() + cut[k]), std::make_move_iterator(genes.begin() + cut[k + 1]));
        if (!pipe->submit(std::move(shard), k / shards_per_dev)) break;
      }
    }
    FilePipeline::Totals totals;
    try {
      pipe->finish(totals);
    } catch (...) {
      err = std::current_exception();
    }
    for (size_t dv = 0; dv < n_dev; ++dv) ctxs[dv]->timing = totals.per_dev[dv];
    // host stages of the file driver (the first context carries them)
    ctxs[0]->timing.ingest_ms = ingest_ms;
    ctxs[0]->timing.pack_ms = double(totals.pack_us) / 1000.0;
    ctxs[0]->timing.write_ms = double(totals.write_us) / 1000.0;
    if (err) std::rethrow_exception(err);
    if (gpu_inflate && getenv("MPH_IO_TRACE"))
      fprintf(stderr, "[mph io] device inflate: %zu batches, %.1f MB in, %.1f MB out, %.1f ms inside the inflater (copies + kernel)%s\n", gpu_inflate->batches,
              gpu_inflate->bytes_in / 1e6, gpu_inflate->bytes_out / 1e6, gpu_inflate->ms_total, bam.device_inflate_used() ? "" : " - not used (small file or fallback to zlib)");
  } catch (...) {
    close_all();
    throw;
  }
  close_all();
}

// What the mph_run_* file entry points share: a null argument is reported on `null_ctx`, a window length the packer
// cannot take and the run's own errors on the first context. Only the normal mode (mode 1) has no `normal_path`.
static int run_files_checked(mph_ctx* null_ctx, mph_ctx* const* ctxs, int n_ctx, const char* bam_path, const char* ref_path,
                             const char* variants_path, const char* gtf_path, const char* fasta_out_path, const char* tsv_path,
                             const char* normal_path, uint32_t window_len, int warn_only, int mode) {
  if (!ctxs || n_ctx < 1 || !bam_path || !ref_path || !variants_path || !gtf_path || !fasta_out_path || !tsv_path || (mode == 0 && !normal_path))
    return fail(null_ctx, MPH_ERR_INPUT, "null argument");
  if (window_len == 0 || window_len % 3 != 0) return fail(ctxs[0], MPH_ERR_UNSUPPORTED, "window length must be a positive multiple of 3");
  return guarded(ctxs[0], [&] {
    run_files(std::vector<mph_ctx*>(ctxs, ctxs + n_ctx), bam_path, ref_path, variants_path, gtf_path, fasta_out_path, tsv_path, normal_path,
              window_len, warn_only, mode);
  });
}

int mph_run_somatic(mph_ctx* ctx, const char* bam_path, const char* ref_path, const char* variants_path, const char* gtf_path,
                    const char* fasta_out_path, const char* tsv_path, const char* normal_path, uint32_t window_len, int warn_only) {
  if (!ctx) return fail(nullptr, MPH_ERR_INPUT, "null argument");
  return run_files_checked(ctx, &ctx, 1, bam_path, ref_path, variants_path, gtf_path, fasta_out_path, tsv_path, normal_path, window_len, warn_only, 0);
}

int mph_run_normal(mph_ctx* ctx, const char* bam_path, const char* ref_path, const char* variants_path, const char* gtf_path,
                   const char* fasta_out_path, const char* tsv_path, uint32_t window_len, int warn_only) {
  if (!ctx) return fail(nullptr, MPH_ERR_INPUT, "null argument");
  return run_files_checked(ctx, &ctx, 1, bam_path, ref_path, variants_path, gtf_path, fasta_out_path, tsv_path, nullptr, window_len, warn_only, 1);
}

int mph_run_somatic_multi(mph_ctx* const* ctxs, int n_ctx, const char* bam_path, const char* ref_path, const char* variants_path,
                          const char* gtf_path, const char* fasta_out_path, const char* tsv_path, const char* normal_path,
                          uint32_t window_len, int warn_only) {
  return run_files_checked(nullptr, ctxs, n_ctx, bam_path, ref_path, variants_path, gtf_path, fasta_out_path, tsv_path, normal_path, window_len,
                           warn_only, 0);
}

int mph_run_normal_multi(mph_ctx* const* ctxs, int n_ctx, const char* bam_path, const char* ref_path, const char* variants_path,
                         const char* gtf_path, const char* fasta_out_path, const char* tsv_path, uint32_t window_len, int warn_only) {
  return run_files_checked(nullptr, ctxs, n_ctx, bam_path, ref_path, variants_path, gtf_path, fasta_out_path, tsv_path, nullptr, window_len,
                           warn_only, 1);
}

int mph_translate(mph_ctx* ctx, const uint8_t* nt, const uint64_t* off, const int8_t* frame, uint64_t n, uint8_t* aa, const uint64_t* aa_off,
                  uint8_t* bad) {
  if (!ctx || !off || !aa_off || (n && (!nt || !frame || !aa || !bad))) return fail(ctx, MPH_ERR_INPUT, "null argument");
  return guarded(ctx, [&] { dev_translate(ctx, nt, off, frame, n, aa, aa_off, bad); });
}

int mph_set_load(mph_ctx* ctx, const uint8_t* peptides, uint32_t k, uint64_t n) {
  if (!ctx || (n && !peptides)) return fail(ctx, MPH_ERR_INPUT, "null argument");
  return guarded(ctx, [&] { dev_set_load(ctx, peptides, k, n); });
}

int mph_set_probe(mph_ctx* ctx, const uint8_t* queries, uint32_t k, uint64_t n, uint8_t* hit) {
  if (!ctx || (n && (!queries || !hit))) return fail(ctx, MPH_ERR_INPUT, "null argument");
  return guarded(ctx, [&] { dev_set_probe(ctx, queries, k, n, hit); });
}

int mph_run_filter(mph_ctx* ctx, const char* reference_bin, const char* tsv_in, const char* fasta_out_path, const char* normal_out,
                   const char* tsv_out, const char* removed_tsv, const char* removed_fasta, uint32_t peptide_length) {
  if (!ctx || !reference_bin || !tsv_in || !fasta_out_path || !normal_out || !tsv_out || !removed_tsv || !removed_fasta)
    return fail(ctx, MPH_ERR_INPUT, "null argument");
  return guarded(ctx, [&] {
    pep::FilterPaths io;
    io.tsv_in = tsv_in; io.normal_out = normal_out; io.tsv_out = tsv_out; io.removed_tsv = removed_tsv; io.removed_fasta = removed_fasta;
    FILE* fo = stdout;
    if (std::string(fasta_out_path) != "-") {
      fo = fopen(fasta_out_path, "wb");
      if (!fo) throw std::runtime_error(std::string("cannot create ") + fasta_out_path);
    }
    io.fasta_out = fo;
    try {
      // the reference deserialises the whole set up front (:245); items of another length or with non-letter bytes can never match
      std::vector<std::string> items = pep::read_peptide_set(reference_bin);
      std::vector<uint64_t> idx;
      std::vector<uint8_t> flat = flatten_k(items, peptide_length, idx);
      dev_set_load(ctx, flat.data(), peptide_length, idx.size());
      pep::ProbeFn probe = [&](const std::vector<std::string>& q, uint32_t k, std::vector<uint8_t>& hit) {
        hit.assign(q.size(), 0);
        std::vector<uint64_t> qi;
        std::vector<uint8_t> qf = flatten_k(q, k, qi);
        std::vector<uint8_t> h(qi.size() + 1, 0);
        dev_set_probe(ctx, qf.data(), k, qi.size(), h.data());
        for (size_t x = 0; x < qi.size(); ++x) hit[qi[x]] = h[x];
      };
      pep::run_filter(io, peptide_length, make_translate(ctx), probe);
    } catch (...) {
      if (fo != stdout) fclose(fo);
      throw;
    }
    if (fo != stdout) fclose(fo);
  });
}

int mph_run_build_reference(mph_ctx* ctx, const char* reference_fasta, const char* binary_out, const char* fasta_out_path, uint32_t peptide_length) {
  if (!ctx || !reference_fasta || !binary_out || !fasta_out_path) return fail(ctx, MPH_ERR_INPUT, "null argument");
  return guarded(ctx, [&] {
    FILE* fo = stdout;
    if (std::string(fasta_out_path) != "-") {
      fo = fopen(fasta_out_path, "wb");
      if (!fo) throw std::runtime_error(std::string("cannot create ") + fasta_out_path);
    }
    try {
      pep::DedupeFn dedupe = [&](const std::vector<std::string>& peptides, uint32_t k) {
        std::vector<uint64_t> idx;
        std::vector<uint8_t> flat = flatten_k(peptides, k, idx);
        dev_set_load(ctx, flat.data(), k, idx.size());
        return dev_set_export(ctx);
      };
      pep::run_build_reference(reference_fasta, binary_out, fo, peptide_length, make_translate(ctx), dedupe);
    } catch (...) {
      if (fo != stdout) fclose(fo);
      throw;
    }
    if (fo != stdout) fclose(fo);
  });
}

int mph_synth_batch(const mph_synth_params* sp, uint32_t window_len, int pin, mph_batch** out) {
  if (!sp || !out) return fail(nullptr, MPH_ERR_INPUT, "null argument");
  std::unique_ptr<mph_batch> mb(new mph_batch);
  int rc = guarded(nullptr, [&] {
    const char* me = getenv("MPH_SYNTH_MODE");  // measurement hook: 1 packs the same workload for the normal mode
    Packer packer(window_len, (me && *me == '1') ? 1 : 0);
    SynthParams p;
    p.seed = sp->seed; p.n_transcripts = sp->n_transcripts; p.exons = sp->exons_per_transcript; p.exon_min = sp->exon_len_min;
    p.exon_max = sp->exon_len_max; p.read_len = sp->read_len; p.coverage = sp->coverage; p.germline_per_kb = sp->germline_per_kb;
    p.somatic_per_kb = sp->somatic_per_kb; p.lowq_frac = sp->lowq_frac; p.indel_read_frac = sp->indel_read_frac;
    p.ins_var_frac = sp->ins_var_frac; p.del_var_frac = sp->del_var_frac;
    synth_into(packer, p);
    mb->b = std::move(packer.batch());
    finish_batch(mb.get(), pin != 0);
  });
  if (rc != MPH_OK) return rc;
  *out = mb.release();
  return MPH_OK;
}

int mph_synth_write_files(const mph_synth_params* sp, uint32_t window_len, const char* dir) {
  if (!sp || !dir) return fail(nullptr, MPH_ERR_INPUT, "null argument");
  return guarded(nullptr, [&] {
    SynthParams p;
    p.seed = sp->seed; p.n_transcripts = sp->n_transcripts; p.exons = sp->exons_per_transcript; p.exon_min = sp->exon_len_min;
    p.exon_max = sp->exon_len_max; p.read_len = sp->read_len; p.coverage = sp->coverage; p.germline_per_kb = sp->germline_per_kb;
    p.somatic_per_kb = sp->somatic_per_kb; p.lowq_frac = sp->lowq_frac; p.indel_read_frac = sp->indel_read_frac;
    p.ins_var_frac = sp->ins_var_frac; p.del_var_frac = sp->del_var_frac;
    synth_write_files(p, window_len, dir);
  });
}

}  // extern "C"
