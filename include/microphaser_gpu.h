/* microphaser_gpu.h — C ABI of the B200-native per-window phasing path.
 *
 * The reference (koesterlab/microphaser, Rust) has no plugin or FFI interface: the path sits behind
 * in-crate calls. The seam this library replaces is
 *
 *   src/main.rs:91-101        run_somatic -> microphasing::phase(fasta, gtf, bcf, bam, writers.., window_len, flag)
 *   src/microphasing.rs:1943  phase(): GTF streaming, one phase_gene() per protein-coding gene
 *   src/microphasing.rs:882   phase_gene(): per-gene read/variant/reference fetch + the window loop
 *   src/microphasing.rs:212-879  ObservationMatrix::{new, cleanup_reads, shrink_left, push_read,
 *                                extend_right, print_haplotypes}
 *
 * A host (the reference's Rust driver through a `-sys` shim, or the C++ CLI of this repository)
 * keeps file parsing, hands genes / reads / variants to the packer below, and gets back the records
 * in the reference's emission order. Reads, variants and exon tables cross the boundary as flat
 * structure-of-arrays buffers; there are no torch or C++ types in any signature.
 *
 * Conventions: every function returns 0 on success or a negative MPH_ERR_* code; the message is
 * available from mph_last_error(). Nothing throws across the boundary. A context is bound to one
 * CUDA device and is not thread-safe: use one context per device per host thread (multi-GPU =
 * N contexts driven by N threads or processes). There is no CPU fallback: without a usable CUDA
 * device mph_ctx_create fails with MPH_ERR_CUDA.
 */
#ifndef MICROPHASER_GPU_H
#define MICROPHASER_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPH_OK 0
#define MPH_ERR_CUDA (-1)        /* no device / CUDA runtime failure */
#define MPH_ERR_INPUT (-2)       /* malformed or inconsistent input (I/O errors, bad arguments) */
#define MPH_ERR_PANIC (-3)       /* a condition on which the reference panics (exit status 101) */
#define MPH_ERR_UNSUPPORTED (-4) /* input needs the serial replay path (not implemented yet) */
#define MPH_ERR_INTERNAL (-5)

typedef struct mph_ctx mph_ctx;       /* one CUDA device + its buffers and stream */
typedef struct mph_packer mph_packer; /* builds a batch from genes */
typedef struct mph_batch mph_batch;   /* packed structure-of-arrays input (host, optionally pinned) */
typedef struct mph_result mph_result; /* ordered records of one batch */

/* ---- context ---------------------------------------------------------------------------- */
int mph_ctx_create(int device, mph_ctx** out);
void mph_ctx_destroy(mph_ctx* ctx);
/* message of the last failing call on this context (or of the last failing context-free call when
 * ctx is NULL); valid until the next call on the same thread */
const char* mph_last_error(const mph_ctx* ctx);

/* ---- packer: replaces the per-gene set-up of phase_gene (src/microphasing.rs:894-942) ---- */
/* mode 0 = somatic (reads with mapq < 5 are dropped by the caller, :910);
 * mode 1 = normal, the healthy-peptidome pass of src/normal_microphasing.rs:650-1279 (no mapq / base-quality
 * filter, every window of a non-short exon yields a record; mph_record.mutant_sequence then holds the
 * `peptide_sequence` column, normal_sequence is empty and offsets are 0-based as in the reference) */
int mph_packer_create(uint32_t window_len, int mode, mph_packer** out);
void mph_packer_destroy(mph_packer* p);

typedef struct {
  /* gene (src/common.rs:224-253); coordinates 0-based half-open */
  const char* gene_id;
  const char* gene_name;
  const char* chrom;
  uint32_t gene_start, gene_end;
  /* reference bases of [gene_start, gene_end + 100), case preserved (:895-901) */
  const uint8_t* refseq;
  uint32_t refseq_len;
  /* transcripts with at least one CDS exon, in GTF order; exons in GTF order (:1982-2125) */
  uint32_t n_tx;
  const char* const* tx_id;
  const uint8_t* tx_reverse;   /* 0 forward, 1 reverse */
  const uint32_t* tx_exon_off; /* n_tx + 1 offsets into exon_* */
  const uint32_t* exon_start;
  const uint32_t* exon_end;
  const uint32_t* exon_frame;  /* GTF frame column, '.' = 0 */
  /* reads held by the record buffer for this gene after the mapq filter, file order (:905-920) */
  uint32_t n_reads;
  uint32_t max_read_len;       /* max seq().len() over them (:913-915) */
  const uint32_t* read_start;  /* record.pos() */
  const uint32_t* read_end;    /* cigar().end_pos() */
  const uint32_t* read_lseq;
  const uint64_t* read_qname_hash;
  const uint32_t* read_seq_off; /* byte offset of the BAM 4-bit bases in seq4 */
  const uint8_t* seq4;
  const uint32_t* read_qual_off; /* byte offset of the raw phred qualities in qual */
  const uint8_t* qual;
  const uint32_t* read_cigar_off; /* n_reads + 1 offsets into cigar (BAM-encoded ops) */
  const uint32_t* cigar;
  /* variants: the variant_tree of the gene, ascending position, ALT alleles in VCF order (:932-942) */
  uint32_t n_vars;
  const uint32_t* var_pos;
  const uint8_t* var_kind;     /* 0 SNV, 1 insertion, 2 deletion (src/common.rs:38-59) */
  const uint8_t* var_germline; /* !INFO/SOMATIC */
  const uint8_t* var_alt;      /* SNV: ALT byte */
  const uint32_t* var_len;     /* insertion: alt.len()-1; deletion: ref.len()-1 or |SVLEN| */
  const uint32_t* var_ins_off; /* n_vars + 1 offsets into ins_bytes (whole ALT allele of insertions) */
  const uint8_t* ins_bytes;
  const char* const* var_prot_change; /* may be NULL */
} mph_gene_in;

int mph_packer_add_gene(mph_packer* p, const mph_gene_in* gene);
/* finishes the packer and hands the batch over; pin != 0 page-locks the buffers for async copies */
int mph_packer_finish(mph_packer* p, int pin, mph_batch** out);
void mph_batch_destroy(mph_batch* b);

/* read-only view of the packed structure-of-arrays buffers (what is copied to the device) */
typedef struct {
  uint32_t window_len;
  uint64_t n_reads, n_vars, n_segments, n_chunks, n_windows, n_transcripts, n_genes;
  const uint32_t* read_start;   /* per read, sorted by start within a gene */
  const uint32_t* read_end;
  const uint8_t* read_flags;
  /* compact side table: one entry per read that overlaps a variant (every read of a gene whose transcripts need the
   * serial replay): read index, first variant index, byte offset of its packed bases / offset of its CIGAR, lengths.
   * (On the bus the table travels as 9 B per entry - distances and record sizes - and is rebuilt on the device.) */
  uint64_t n_variant_reads;
  const uint32_t* vr_read;
  const uint32_t* vr_vlo;
  const uint32_t* vr_seq_off;
  const uint32_t* vr_cig_off;
  const uint16_t* vr_lseq;
  const uint16_t* vr_ncig;
  const uint8_t* vr_nv;
  const uint8_t* bases;   uint64_t bases_bytes;   /* packed read record per side-table entry: format byte, 2-bit or 4-bit bases, low-quality positions (csrc/core/phase_core.h) */
  const uint32_t* cigars; uint64_t n_cigar_ops;
  const void* vars;       /* MphVar[n_vars], 16 B each (csrc/core/layout.h) */
  const void* segments;   /* MphSegment[n_segments], 96 B each */
  const void* chunks;     /* MphChunk[n_chunks], 32 B each */
  const uint8_t* ref;     uint64_t ref_bytes;     /* per-exon reference slices */
  uint64_t h2d_bytes;     /* bytes copied host -> device per mph_phase_batch call */
} mph_batch_view;
int mph_batch_get_view(const mph_batch* b, mph_batch_view* out);

/* ---- the hot path: replaces the window loop of phase_gene (src/microphasing.rs:944-1939) ---- */
/* host buffers in, ordered records out: H2D copy, kernels K1-K4, D2H copy, host residue */
int mph_phase_batch(mph_ctx* ctx, const mph_batch* batch, mph_result** out);
/* the same work split for measurements with inputs resident in HBM */
int mph_batch_upload(mph_ctx* ctx, const mph_batch* batch);
int mph_phase_resident(mph_ctx* ctx);                     /* kernels K1-K4 only, on the context's stream */
int mph_phase_collect(mph_ctx* ctx, mph_result** out);    /* D2H + residue of the last resident run */

typedef struct {
  /* CUDA events on the library's streams, summed over the pipeline stages of one call; residue_ms: busy time of the
   * host threads / thread count; total_ms: wall clock of the call (the stages overlap, so it is less than the sum) */
  double h2d_ms, k1_ms, k2_ms, k3_ms, k4_ms, d2h_ms, residue_ms, total_ms;
  uint64_t h2d_bytes, d2h_bytes;
  uint64_t windows;       /* main-ORF windows the reference evaluates (print_haplotypes calls, frame 0) */
  uint64_t read_windows;  /* sum of depth over them */
  uint64_t windows_enumerated, n_interesting, n_records;
  uint32_t kernel_launches;
  uint32_t n_replay_units; /* replay units (runs of exons of irregular transcripts) that went through k_replay */
  double replay_ms;        /* k_replay, CUDA events; k2_ms is the closed-form window kernels alone */
  double k5_ms;            /* record kernels: ORF stop, emit predicate, junction merge, ordered compaction of the records */
  double pack_ms;          /* file drivers only: host time spent in the packer (wall clock, summed over the packing threads) */
  double ingest_ms;        /* file drivers only: BGZF inflate + BAM decode, GTF / VCF / FASTA parsing and the per-gene fetches (wall clock) */
  double write_ms;         /* file drivers only: rendering and writing the three output streams (wall clock, summed over the shards) */
  double kernels_ms;       /* CUDA events around the whole kernel chain of a run (first launch to last), summed over the stages; k_replay
                            * runs on a second stream beside K2, so this is less than the sum of the per-kernel figures */
} mph_timing;
int mph_ctx_timing(const mph_ctx* ctx, mph_timing* out);

/* ---- results ------------------------------------------------------------------------------ */
void mph_result_destroy(mph_result* r);
uint64_t mph_result_count(const mph_result* r);
typedef struct {
  const char* id;          /* 15 hex of SHA-1 + strand initial (:667-675) */
  const char* transcript; const char* gene_id; const char* gene_name; const char* chrom;
  uint64_t offset, frame;
  double freq;
  uint32_t depth, nvar, nsomatic, nvariant_sites, nsomvariant_sites;
  int reverse;
  const char* variant_sites; const char* somatic_positions; const char* somatic_aa_change;
  const char* germline_positions; const char* germline_aa_change;
  const char* normal_sequence; const char* mutant_sequence;
  const char* fasta_mutant;  /* NULL if no line goes to the mutant FASTA (:846-858) */
  const char* fasta_normal;  /* NULL if no line goes to the normal FASTA (:859-873) */
} mph_record;
int mph_result_get(const mph_result* r, uint64_t i, mph_record* out);
/* appends the three output streams in the reference's byte format (SURVEY.md Appendix B);
 * *tsv_header_written carries the "header with the first row" state across batches */
int mph_result_write(const mph_result* r, int fd_fasta, int fd_tsv, int fd_normal, int* tsv_header_written);

/* ---- file-level driver: replaces microphasing::phase (src/microphasing.rs:1943-2131) ------ */
/* `somatic` sub-command on real files; GTF is read from gtf_path ("-" = stdin), mutant FASTA goes
 * to fasta_out_path ("-" = stdout). With a BAM index next to the BAM (<bam>.bai, else <bam minus .bam>.bai)
 * the reads are fetched through it gene range by gene range and phased in shards as they close, so host
 * memory follows the shard size; a malformed index is MPH_ERR_INPUT. Without one the whole BAM is loaded
 * first. */
int mph_run_somatic(mph_ctx* ctx, const char* bam_path, const char* ref_path, const char* variants_path, const char* gtf_path,
                    const char* fasta_out_path, const char* tsv_path, const char* normal_path, uint32_t window_len,
                    int unsupported_allele_warning_only);

/* `normal` sub-command (src/normal_microphasing.rs:1281-1440): FASTA of every window's haplotypes and the 20-column TSV */
int mph_run_normal(mph_ctx* ctx, const char* bam_path, const char* ref_path, const char* variants_path, const char* gtf_path,
                   const char* fasta_out_path, const char* tsv_path, uint32_t window_len, int unsupported_allele_warning_only);

/* the same over several devices of one box: genes are split into n_ctx contiguous ranges balanced by
 * read count, every context phases its range on its own host thread, records are concatenated in
 * range order. With a BAM index the streamed shards go to whichever device is free as they close.
 * No collective is involved (shards are independent). */
int mph_run_somatic_multi(mph_ctx* const* ctxs, int n_ctx, const char* bam_path, const char* ref_path, const char* variants_path,
                          const char* gtf_path, const char* fasta_out_path, const char* tsv_path, const char* normal_path,
                          uint32_t window_len, int unsupported_allele_warning_only);

/* `normal` sub-command over several devices, sharded the same way (src/normal_microphasing.rs:1281-1440) */
int mph_run_normal_multi(mph_ctx* const* ctxs, int n_ctx, const char* bam_path, const char* ref_path, const char* variants_path,
                         const char* gtf_path, const char* fasta_out_path, const char* tsv_path, uint32_t window_len,
                         int unsupported_allele_warning_only);

/* ---- secondary path: `filter` / `build_reference` (src/peptides.rs) ------------------------------ */
/* to_protein (:128-146): n nucleotide sequences nt[off[i]..off[i+1]); frame[i] = +1 (forward) or -1 (reverse complement
 * first, :131-135). aa[aa_off[i]..aa_off[i+1]) receives floor(len/3) amino-acid letters ('X' = stop); bad[i] = 1 if a
 * codon is not in the table (the reference unwraps an Err there, :141). Constant-memory codon table on the device. */
int mph_translate(mph_ctx* ctx, const uint8_t* nt, const uint64_t* off, const int8_t* frame, uint64_t n, uint8_t* aa, const uint64_t* aa_off,
                  uint8_t* bad);
/* the normal peptidome as a device open-addressing hash set (deserialised HashSet<Vec<u8>> of :245): n peptides of k letters (up to 12: 5-bit packed
 * 64-bit keys; longer ones, e.g. the 13-25 of MHC-II runs: slots index the resident byte array and equality is a byte compare) */
int mph_set_load(mph_ctx* ctx, const uint8_t* peptides, uint32_t k, uint64_t n);
/* ref_set.contains(tumor_peptide) (:502, :684) for n queries of k letters; hit[i] = 1 if present */
int mph_set_probe(mph_ctx* ctx, const uint8_t* queries, uint32_t k, uint64_t n, uint8_t* hit);
/* peptides::filter (:234-709) and peptides::build (:148-186) end to end on files ("-" = stdout for the tumor / peptide FASTA) */
int mph_run_filter(mph_ctx* ctx, const char* reference_bin, const char* tsv_in, const char* fasta_out_path, const char* normal_out,
                   const char* tsv_out, const char* removed_tsv, const char* removed_fasta, uint32_t peptide_length);
int mph_run_build_reference(mph_ctx* ctx, const char* reference_fasta, const char* binary_out, const char* fasta_out_path, uint32_t peptide_length);

/* ---- synthetic workload (bench only): packs an exome-shaped batch natively ------------------ */
typedef struct {
  uint64_t seed;
  uint32_t n_transcripts, exons_per_transcript, exon_len_min, exon_len_max, read_len;
  double coverage, germline_per_kb, somatic_per_kb, lowq_frac, indel_read_frac;
  double ins_var_frac, del_var_frac; /* share of the variants that are 1-6 nt insertions / deletions (hypermutated config) */
} mph_synth_params;
int mph_synth_batch(const mph_synth_params* params, uint32_t window_len, int pin, mph_batch** out);
/* the same genes / reads / variants as real files in `dir`: ref.fa(.fai), annotation.gtf, variants.vcf, reads.bam */
int mph_synth_write_files(const mph_synth_params* params, uint32_t window_len, const char* dir);

#ifdef __cplusplus
}
#endif
#endif /* MICROPHASER_GPU_H */
