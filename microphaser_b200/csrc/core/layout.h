// layout.h — plain-old-data records shared by the host packer, the CUDA kernels and the
// test-only CPU emulator. Everything the device touches is a flat array of these.
//
// Vocabulary follows the reference (src/microphasing.rs): a *segment* is one exon of one
// transcript as the window loop sees it (:974-1029); *iteration* k of a segment is one pass of
// the `loop` at :1030 (offset = off0 ± k); a *window* is an iteration at which
// print_haplotypes (:1411) is called; an *observation* is a read held in the
// ObservationMatrix (:147-154).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define MPH_HD __host__ __device__ __forceinline__
#else
#define MPH_HD inline
#endif

enum { MPH_SNV = 0, MPH_INS = 1, MPH_DEL = 2 };

// variant flags
enum {
  MPH_VF_GERMLINE = 1,   // !INFO/SOMATIC (common.rs:75)
  MPH_VF_FS_SHIFT = 1,   // bits 1-2: Variant::frameshift() (common.rs:215-221)
  MPH_VF_FS_MASK = 6,
};

// One ALT allele (common.rs:38-59), 16 B. Per gene the records are sorted by (pos asc, then
// ALT order of the VCF line for forward-strand genes / reversed ALT order for reverse-strand
// genes) — exactly the order of `variants` inside print_haplotypes (:373-379).
typedef struct {
  uint32_t pos;      // 0-based
  uint32_t len;      // INS: alt.len()-1, DEL: ref.len()-1 or |SVLEN|
  uint8_t kind;      // MPH_SNV / MPH_INS / MPH_DEL
  uint8_t alt;       // SNV: raw ALT byte
  uint8_t flags;     // MPH_VF_*
  uint8_t alt4;      // SNV: 4-bit BAM code of `alt`, 0xFF if `alt` is not a BAM base letter
  uint32_t ins_off;  // INS: offset of the ALT allele bytes (len+1 of them) in the insertion arena
} MphVar;

// segment flags
enum {
  MPH_SF_REVERSE = 1,
  MPH_SF_SHORT = 2,       // is_short_exon (:999-1004)
  MPH_SF_FIRST_EXON = 4,  // exon_count == 1
  MPH_SF_LAST_EXON = 8,
  MPH_SF_HAS_FS = 16,     // the gene carries frameshifting variants: every iteration is a window
  MPH_SF_KEEP_PENULT = 64,  // the next exon's only window is first and last: its junction merge reads this exon's last-but-one window (:1401-1405)
  MPH_SF_JOIN_HEAD = 128,   // the junction at the exon's first window can produce records (a variant on either side): its list is kept
  MPH_SF_JOIN_TAIL = 256,   // the same for the junction after the exon's last window (and the last-but-one with KEEP_PENULT)
  MPH_SF_REPLAY = 32,     // the transcript goes through the serial replay (core/replay_core.h), not the closed form
  MPH_SF_DEVREC = 512,    // the transcript's records are built on the device (core/record_core.h); set on all its segments
};

// One processed exon of one transcript, 96 B.
typedef struct {
  uint32_t exon_start, exon_end;  // [start, end)
  uint32_t off0;                  // offset at iteration 0 (:1015-1019)
  uint32_t ewl;                   // exon_window_len (:1007-1013)
  uint32_t n_iter;                // iterations k = 0 .. n_iter-1
  uint32_t ceo;                   // current_exon_offset (:989-995)
  uint32_t flags;                 // MPH_SF_*
  uint32_t K;                     // max_read_len - ewl (:1196,1208)
  uint32_t read_lo, read_hi;      // the gene's reads (global indices, sorted by start, file order)
  uint32_t var_lo, var_hi;        // the gene's variants (global indices)
  uint32_t sl_va, sl_vb;          // variant index range with start-loss positions (:1305-1319); empty if none
  uint32_t max_span;              // max (end - start) over the gene's reads
  uint32_t ref_pos0;              // genomic position of ref arena byte ref_off
  uint32_t ref_off, ref_len;      // this segment's slice of the reference arena (exon + deletion margin)
  uint32_t tx;                    // transcript index
  uint32_t win_base;              // global index of this segment's first window
  uint32_t k_first, k_stride;     // windows are iterations k_first + i*k_stride, i = 0 .. n_win-1
  uint32_t n_win;
  uint32_t pad;
} MphSegment;

// A unit of K2/K3 work: n consecutive windows of one segment, 32 B. The read / variant index
// ranges the chunk can touch are data independent, so the packer resolves them once (it saves the
// kernels ~27 dependent binary-search loads per chunk).
typedef struct {
  uint32_t seg;
  uint32_t i_first;
  uint32_t n;
  uint32_t rlo, rhi;  // union of the windows' candidate reads (global read indices)
  uint32_t va0, vb1;  // variants with pos in [min s, max e) over the chunk's windows
  uint32_t pad;
} MphChunk;

// Per segment, 16 B: the union of its windows' candidate reads [rlo, rhi) and of the variants inside them [va0, vb1).
// The read-run kernel (K2a) visits every (segment, read) pair of these ranges exactly once.
typedef struct {
  uint32_t rlo, rhi;
  uint32_t va0, vb1;
} MphSegWork;

// Restart point of the side table's running sums on the bus (host: Batch::VRun), 20 B.
typedef struct {
  uint32_t entry, read, vlo, seq_off, cig_off;
} MphSideRun;

// Per-read fields, as the core functions see them in registers. In memory the reads are
// structure-of-arrays (include/microphaser_gpu.h: mph_batch_in.read_*).
//   seq_off : 16-byte units into the packed-base arena, where the read's record is
//             ceil(l_seq/2) B of BAM 4-bit bases followed by ceil(l_seq/8) B of (qual < 10) bits;
//             0xFFFFFFFF when nv == 0 (reads without variants ship no bases at all)
//   n_cig   : 0 => a single M of l_seq (no cigar shipped); else ops at cig_off in the cigar arena
typedef struct {
  uint32_t start;  // record.pos()
  uint32_t end;    // cigar().end_pos(), exclusive
  uint32_t vlo;    // global index of the first variant of the gene with pos >= start
  uint32_t l_seq;  // seq().len()
  uint32_t nv;     // variants with pos in [start, end), capped at 64
  uint32_t n_cig;
} MphRead;

enum {
  MPH_RF_OVERFLOW = 1,  // more than 64 variants inside the read
  MPH_RF_PARTNER = 2,   // another read of the gene has the same (start, qname): `contains` (:281-294)
};

// K1 output, 16 B per read: bit j <-> variant vlo + j.
typedef struct {
  uint64_t S;  // supports_variant (:95-139)
  uint64_t B;  // bad_quality (:78-93)
} MphCall;

// K2 output per window, 16 B.
typedef struct {
  uint32_t depth;      // ObservationMatrix::nrows() (:457) — observations incl. bad_qual ones
  uint32_t c0;         // count of the (haplotype 0, frame 0) key
  uint32_t extra_off;  // first extra histogram entry in the arena
  uint32_t n_extra;    // number of extra (non-(0,0)) keys
} MphWinOut;

// One extra histogram key, 16 B. Keys of a window are stored sorted by (hap, frame0, f1nz).
typedef struct {
  uint64_t hap;
  uint32_t count;
  uint32_t frame;  // bits 0-30: obs.frame.0, bit 31: obs.frame.1 != 0
} MphHist;

// K3 output per assembled haplotype (entry 0 of every window + every extra entry), 32 B.
enum {
  MPH_HF_STOP = 1,       // has_stop_codon(neopeptide) (:694-697)
  MPH_HF_INDEL = 2,      // :442
  MPH_HF_INSERTION = 4,  // :443
  MPH_HF_SEQ = 8,        // seq/germline_seq bytes were written to the sequence arena
  MPH_HF_GERM_EQ = 16,   // germline_seq == seq before any clearing (:624-631)
  MPH_HF_OVERFLOW = 32,  // assembled sequence longer than the per-haplotype arena slot
  MPH_HF_ID = 128,       // id64 holds the leading 64 bits of the record id's SHA-1 (:667-675)
  MPH_HF_REFRANGE = 64,  // the walk left the shipped reference slice: the reference panics if (and only if) it reaches this haplotype
  MPH_HF_PEPDIFF = 256,    // normal_peptide != neopeptide (:677-693,707) with frameshift-free clearing of germline_seq (:624-631)
  MPH_HF_SLICE_ERR = 512,  // one of the peptide slices of :677-693 is out of range (the reference panics there)
};
typedef struct {
  uint32_t flags;      // MPH_HF_*
  uint16_t seq_len;    // seq.len()
  uint16_t germ_len;   // germline_seq.len() before clearing
  uint8_t n_var;       // n_variants (:452)
  uint8_t n_som;       // n_somatic (:451)
  uint8_t n_prof;      // variant_profile.len() (:462)
  uint8_t brk;         // 1: the walk hit `break` at :549-552 on variants[n_prof] with its bit set
                       //    (its frameshift side effects :482-502 happened, its profile entry did not)
  uint32_t seq_off;    // byte offset into the sequence arena: seq then germline_seq
  uint64_t profile;    // 2 bits per visited variant: 0 absent, 1 germline, 2 somatic (:583-590)
  uint64_t id64;       // MPH_HF_ID: sha1(format!("{:?}{}{}", seq, transcript.id, offset)) bits 159..96; the id is its first 15 hex digits + strand initial
} MphHap;

// device error bits (sticky, OR-ed into one word)
enum {
  MPH_E_HIST_OVERFLOW = 1,   // histogram arena exhausted -> host retries with a larger arena
  MPH_E_SEQ_OVERFLOW = 2,    // sequence arena exhausted  -> host retries with a larger arena
  MPH_E_KEYS_PER_WINDOW = 4, // more than MPH_BLOCK_KEYS distinct keys in one window
  MPH_E_REF_RANGE = 8,       // reference index out of the shipped slice (reference: slice panic)
  MPH_E_VARS_PER_WINDOW = 16, // > 64 variants in one window (reference: shift overflow)
  MPH_E_REPLAY_PANIC = 32,    // serial replay: the reference panics here (drain out of range, read right of a variant, inverted range)
  MPH_E_VLIST_OVERFLOW = 64,  // column-list arena exhausted -> host retries with a larger arena
  MPH_E_REPLAY_INPUT = 128,   // serial replay: observation scratch too small or read bases not shipped (internal)
  MPH_E_SLICE = 256,          // record kernels: a sequence slice the reference takes is out of range (reference: slice panic)
  MPH_E_INTERNAL = 512,       // record kernels: a haplotype that is written lacks its sequence or id
  MPH_E_SEQ_SLOT = 1024,      // assembled haplotype longer than the sequence slot / a record length field
  MPH_E_REC_OVERFLOW = 2048,  // record / merge arena exhausted -> host retries with larger arenas
  MPH_E_SPILL_OVERFLOW = 4096, // spill arena of the block histogram tier exhausted -> host retries with a larger arena
  MPH_E_RECS_PER_LIST = 8192   // record kernels: more records from one window (4095) or one splice junction (MPH_RC_JUNCTION_RECS) than they index
};

// Third histogram tier: a window with more distinct keys than a warp table holds spills its counted observations
// (MphHist entries, count = weight) to the spill arena and queues itself; k_window_hist_block (one CTA per queued window)
// sorts and folds them in shared memory. MPH_BLOCK_KEYS distinct keys is what that buffer keeps: a window with more
// raises MPH_E_KEYS_PER_WINDOW. The kernel, the CPU emulator and the error message share this bound.
#define MPH_BLOCK_KEYS 4096
#define MPH_XSTR_(x) #x
#define MPH_XSTR(x) MPH_XSTR_(x)
#define MPH_MSG_KEYS_PER_WINDOW "more than " MPH_XSTR(MPH_BLOCK_KEYS) " distinct haplotypes in one window"
#define MPH_MSG_RECS_PER_LIST "more records from one window or one splice junction than a record list holds"

// One queued window of the block tier, 16 B.
typedef struct {
  uint32_t code;    // (chunk << 5 | lane) of the window, as in hist_win
  uint32_t off, n;  // its observations in the spill arena
  uint32_t devrec;  // 1: the keys go to the back of the histogram arena (device-class transcript, somatic mode)
} MphSpillWin;
