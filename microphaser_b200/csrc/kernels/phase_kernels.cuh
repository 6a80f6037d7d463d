// phase_kernels.cuh — device-side view of one batch and the launch entry points of the phasing
// kernels (sm_100a). Definitions in phase_kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../core/layout.h"
#include "../core/replay_core.h"
#include "../core/record_core.h"

namespace mphk {

// everything the kernels read or write, all device pointers
struct DeviceBatch {
  // inputs
  uint32_t n_reads = 0, n_vars = 0, n_segs = 0, n_chunks = 0, n_windows = 0, seq_cap = 64, n_pairs = 0;
  // the slice of the batch one launch sequence works on (a stage of the copy / compute / residue pipeline, or everything)
  uint32_t r0 = 0, r1 = 0;    // reads
  uint32_t vr0 = 0, vr1 = 0;  // entries of the variant-read side table (K1)
  uint32_t c0 = 0, c1 = 0;    // chunks (K2b, K5)
  uint32_t s0 = 0, s1 = 0;    // segments
  uint32_t it0 = 0, it1 = 0;  // K2a work items (segment, read): seg_work_off[s0] .. seg_work_off[s1]
  uint32_t w0 = 0, w1 = 0;    // windows (K4)
  uint32_t rp0 = 0, rp1 = 0;  // replay units
  uint32_t mode = 0;        // 0 somatic, 1 normal (reference src/normal_microphasing.rs)
  // test hook MPH_FORCE_WIDE: 1 sends every window with extra keys through k_window_hist_wide; 2 also makes the wide kernels
  // and the replay spill such a window at its first extra key, so that every one of them goes through k_window_hist_block
  uint32_t force_wide = 0;
  const uint32_t* read_start = nullptr;  // rebuilt on the device by K0 from the 2-byte bus encoding below
  const uint32_t* read_end = nullptr;
  const uint8_t* read_flags = nullptr;
  uint32_t* read_start_w = nullptr;      // the same buffers, writable (K0)
  uint32_t* read_end_w = nullptr;
  uint8_t* read_flags_w = nullptr;
  const uint8_t* rd_delta = nullptr;     // per read: start - previous start (0 at the head of a run)
  const uint8_t* rd_span = nullptr;      // per read: end - start, 255 = see rd_span_exc; nullptr: every read spans modal_span unless rd_span_exc lists it
  uint32_t modal_span = 0;
  const uint2* rd_runs = nullptr;        // (first read, its start), ascending; a run ends where the next begins
  const uint2* rd_span_exc = nullptr;    // (read, end)
  const uint2* rd_flag_exc = nullptr;    // (read, flags)
  uint32_t run0 = 0, run1 = 0, sx0 = 0, sx1 = 0, fx0 = 0, fx1 = 0;  // the slice's runs / exceptions
  // compact side table: the reads K1 has work for
  const uint32_t* vr_read = nullptr;     // rebuilt on the device by K0 (k_side_decode) from the 9-byte bus form below
  const uint32_t* vr_vlo = nullptr;
  const uint32_t* vr_seq_off = nullptr;  // byte offset of the packed read record in `bases`
  const uint32_t* vr_cig_off = nullptr;
  const uint16_t* vr_lseq = nullptr;     // shipped as they are
  const uint16_t* vr_ncig = nullptr;
  const uint8_t* vr_nv = nullptr;
  uint32_t* vr_read_w = nullptr; uint32_t* vr_vlo_w = nullptr; uint32_t* vr_seq_off_w = nullptr; uint32_t* vr_cig_off_w = nullptr; uint16_t* vr_ncig_w = nullptr;
  const uint16_t* vs_read_d = nullptr;   // per entry: read index - previous entry's (0 at the head of a run)
  const uint8_t* vs_vlo_d = nullptr;     // per entry: first-variant index - previous entry's
  const uint16_t* vs_size = nullptr;     // per entry: bytes of its packed read record
  const uint8_t* vs_ncig = nullptr;      // per entry: CIGAR operations shipped (0 = one M over the read), 255 = see vs_ncig_exc
  const MphSideRun* vs_runs = nullptr;   // where the running sums restart
  const uint2* vs_ncig_exc = nullptr;    // (entry, CIGAR operations)
  uint32_t vrun0 = 0, vrun1 = 0, nx0 = 0, nx1 = 0;  // the slice's runs / exceptions
  // per read, expanded by K1 (read_nv is zeroed first; read_vlo / read_vr are only defined where read_nv != 0)
  uint32_t* read_vlo = nullptr;
  uint8_t* read_nv = nullptr;
  uint32_t* read_vr = nullptr;
  const uint2* pairs = nullptr;  // (read, partner) sorted by read — both directions; the current slice's pairs, n_pairs of them
  const uint8_t* bases = nullptr;
  const uint32_t* cigars = nullptr;
  const MphVar* vars = nullptr;
  const uint8_t* ins_bytes = nullptr;
  const MphSegment* segs = nullptr;
  const MphChunk* chunks = nullptr;
  const MphSegWork* seg_work = nullptr;   // per segment: candidate read / variant ranges (layout.h)
  const uint32_t* seg_work_off = nullptr; // running sum of the read range lengths, n_segs + 1 entries
  // K2a output
  int* win_diff = nullptr;        // per window: +1 where a plain observation's run of windows starts, -1 after its end
  // per segment, in [seg_work_off[seg], seg_work_off[seg + 1]): from the front the reads that need the full closed form (x = read),
  // from the back the reads that carry allele calls and were counted as plain observations (x = read, y = first | last << 16 window of their run)
  uint2* seg_list = nullptr;
  uint32_t* seg_list_n = nullptr;
  uint32_t* seg_list2_n = nullptr;
  uint32_t* rr_seg0 = nullptr;  // first segment of every k_read_runs block (k_read_runs_plan)
  const uint8_t* ref = nullptr;
  const uint32_t* stopmap = nullptr;  // 1 bit per ref byte: a stop codon starts here
  const uint8_t* tx_id_bytes = nullptr;  // transcript ids (record ids are hashed on the device)
  const uint32_t* tx_id_off = nullptr;
  // K1 output
  uint64_t* call_S = nullptr;
  uint64_t* call_B = nullptr;
  uint8_t* call_flags = nullptr;  // bit0: S|B != 0 or host flag PARTNER — the read needs the full pair evaluation
  // K2 output
  MphWinOut* win_out = nullptr;
  MphHist* hist = nullptr;
  uint32_t* hist_win = nullptr;  // per key: (chunk << 5 | lane) of its window
  uint32_t hist_cap = 0;          // keys of host-class windows fill the arena from the front (CTR_HIST, downloaded), those of
                                  // device-class transcripts from the back (CTR_HISTD, read by K3 and the record kernels only)
  uint32_t* ovf_list = nullptr;  // (chunk << 5 | lane) of windows whose keys overflow a lane table; chunk count must be < 2^27
  // block tier (layout.h MPH_BLOCK_KEYS): windows whose keys overflow a warp table. The wide kernels and the replay append their
  // counted observations to `spill` (counters[CTR_SPILL] entries) and queue them: K2's in spq (counters[CTR_SPQ]), the replay's
  // in spq_rp (counters[CTR_SPQR]); a window is queued at most once, so a queue of n_windows entries cannot overflow
  MphHist* spill = nullptr;
  uint32_t spill_cap = 0;
  MphSpillWin* spq = nullptr;
  MphSpillWin* spq_rp = nullptr;
  // K3 output
  MphHap* hap0 = nullptr;
  MphHap* hapx = nullptr;  // parallel to hist
  uint8_t* seq = nullptr;
  uint32_t seq_cap_bytes = 0;
  uint8_t* win_flag = nullptr;  // 1: interesting
  // K4 output
  uint32_t* block_counts = nullptr;
  uint32_t* iw = nullptr;
  MphWinOut* iw_out = nullptr;
  MphHap* iw_hap0 = nullptr;
  // counters: [0] hist_used [1] seq_used [2] n_interesting [3] err bits ; u64 sum_depth at +8
  uint32_t* counters = nullptr;
  unsigned long long* sum_depth = nullptr;
  unsigned long long* live_depth = nullptr;
  const uint32_t* seg_live = nullptr;  // per segment: number of windows the reference reaches
  // serial replay of irregular transcripts (core/replay_core.h)
  const MphReplayTx* replay = nullptr;
  uint32_t n_replay = 0;
  const uint32_t* seg_chunk0 = nullptr;
  const uint32_t* dq_init = nullptr;  // initial matrix columns of the replay units
  uint32_t* o_read = nullptr; uint32_t* o_key = nullptr; uint64_t* o_hap = nullptr; uint32_t* o_frame = nullptr; uint8_t* o_flags = nullptr; uint8_t* o_inmat = nullptr;
  uint32_t* win_voff = nullptr;  // per window: offset of the matrix column list in vlist, 0xFFFFFFFF = the window's own variants
  uint32_t* vlist = nullptr;
  uint32_t vlist_cap = 0;
  uint32_t* iw_voff = nullptr;   // K4: win_voff of the interesting windows
  uint32_t* seg_err = nullptr;   // per segment: 1 + iteration at which the reference panics, 0 = none
  // record kernels (record_kernels.cu, core/record_core.h): device-class transcripts
  uint32_t window_len = 27;
  uint32_t* win_seg = nullptr;      // per interesting window of a device-class transcript: its segment
  uint8_t* seq_dev = nullptr;       // K3's sequence arena for those transcripts (never downloaded); counter CTR_SEQD
  uint32_t seq_dev_cap_bytes = 0;
  uint32_t* tx_stop = nullptr;      // per transcript: first window with a haplotype that ends the ORF (0xFFFFFFFF: none)
  uint32_t* rw = nullptr;           // compacted interesting windows of device-class transcripts (counters[CTR_NRW] of them)
  uint32_t* rw_stopq = nullptr;     // per listed window: first haplotype that removes the peptide
  uint32_t* rw_info = nullptr;      // per listed window: own records | merged records << 12
  uint32_t* rw_mbase = nullptr;     // per listed window: first slot of its junction's records in the merge arena
  uint32_t* rw_bytes = nullptr;     // per listed window: sequence bytes its records need
  uint32_t* rw_junc = nullptr;      // listed windows (indices into rw) whose junction merge is due (counters[CTR_NJ])
  uint32_t* rc_blocks = nullptr;    // block sums / offsets of the two compactions
  uint32_t* rc_bblocks = nullptr;   // block sums / offsets of the records' sequence bytes (somatic mode: the bytes are laid out in record order)
  MphRec* recs = nullptr;           // ordered records (counters[CTR_NREC])
  uint32_t rec_cap = 0;
  uint8_t* rec_seq = nullptr;       // their sequence bytes (counters[CTR_RECSEQ])
  uint32_t rec_seq_cap = 0;
  MphRec* m_recs = nullptr;         // merge arena: junction records before they are placed (counters[CTR_MERGE] slots)
  MphRecSrc* m_aux = nullptr;
  uint8_t* m_seq = nullptr;         // MPH_RC_SEQ_SLOT bytes per slot
  uint32_t m_cap = 0;
  unsigned long long* win_id = nullptr;  // normal mode, per window: leading 64 bits of the record id of the unmodified reference window
  uint32_t* win_depth = nullptr;       // normal mode, per window: depth | (plain window begins / ends with a stop codon) << 31
};

enum { CTR_HIST = 0, CTR_SEQ = 1, CTR_NIW = 2, CTR_ERR = 3, CTR_OVF = 4, CTR_VLIST = 5, CTR_SEQD = 6, CTR_NRW = 7, CTR_MERGE = 8, CTR_NREC = 9, CTR_RECSEQ = 10, CTR_HISTD = 11, CTR_NJ = 12, CTR_RPQ = 13, CTR_MQ = 14, CTR_SPILL = 16, CTR_SPQ = 17, CTR_SPQR = 18, CTR_COUNT = 20 };

void launch_read_decode(const DeviceBatch& d, cudaStream_t st);
void launch_allele_call(const DeviceBatch& d, cudaStream_t st);
void launch_window_hist(const DeviceBatch& d, cudaStream_t st);
void launch_replay(const DeviceBatch& d, cudaStream_t st, uint32_t max_ctas = 0);  // replay_kernels.cu; max_ctas: size of the persistent grid (0 = one CTA per unit)
void launch_window_hist_normal(const DeviceBatch& d, cudaStream_t st);    // normal_kernels.cu (called by launch_window_hist in mode 1)
enum { SPQ_K2 = 0, SPQ_REPLAY = 1 };  // which queue of the block tier a launch consumes
void launch_window_hist_block(const DeviceBatch& d, cudaStream_t st, int queue);  // block_kernels.cu
void launch_assemble_normal(const DeviceBatch& d, cudaStream_t st);
enum { ASM_ALL = 0, ASM_DEVICE_CLASS = 1, ASM_HOST_CLASS = 2 };  // which end of the key arena a K3 launch walks
void launch_assemble(const DeviceBatch& d, cudaStream_t st, int part = ASM_ALL);
void launch_compact(const DeviceBatch& d, cudaStream_t st);
void launch_live_depth(const DeviceBatch& d, cudaStream_t st);            // record_kernels.cu
void launch_records(const DeviceBatch& d, cudaStream_t st);               // record_kernels.cu
uint64_t kernel_launches_on_this_thread();  // running count of the kernels the calling thread has launched (bench "gpu_launches")
uint32_t read_runs_blocks(uint64_t n_items);  // CTAs k_read_runs uses for that many (segment, read) items

}  // namespace mphk
