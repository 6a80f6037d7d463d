// cli.hpp — command-line surface of the reference (src/main.rs:34-265 and the clap YAML files):
//   microphaser somatic <tumor.bam> -r REF -b VCF [-w 27] [-t info.tsv] [-n normal.fasta] [-u] [-v]
// GTF on stdin, mutant FASTA on stdout. The device side is injected as a callable so the same
// front end serves the CUDA library (product) and the test-only CPU emulator.
#pragma once
#include <functional>
#include <iostream>
#include <map>
#include <set>

#include "ingest.hpp"
#include "records_host.hpp"
#include "writer.hpp"

namespace mph {

using PhaseFn = std::function<PhaseRaw(const Batch&)>;

struct CliArgs {
  std::map<std::string, std::string> opt;
  std::vector<std::string> pos;
  std::set<std::string> flags;
};
struct CliSpec {
  const char* lng;
  char shrt;
  bool value;
};

// BGZF inflate / record decode threads of the alignment reader: MPH_IO_THREADS, default 1 here (the library's file
// drivers default to min(cores, 8))
inline unsigned io_threads_env() {
  const char* e = getenv("MPH_IO_THREADS");
  return e ? unsigned(std::max(1, atoi(e))) : 1u;
}

inline CliArgs parse_cli(int argc, char** argv, int first, const std::vector<CliSpec>& specs) {
  CliArgs a;
  for (int i = first; i < argc; ++i) {
    std::string s = argv[i];
    const CliSpec* sp = nullptr;
    std::string val;
    bool have_val = false;
    if (s.rfind("--", 0) == 0) {
      std::string name = s.substr(2);
      size_t eq = name.find('=');
      if (eq != std::string::npos) { val = name.substr(eq + 1); name = name.substr(0, eq); have_val = true; }
      for (auto& x : specs) if (name == x.lng) sp = &x;
    } else if (s.size() >= 2 && s[0] == '-') {
      for (auto& x : specs) if (x.shrt && s[1] == x.shrt) sp = &x;
      if (sp && s.size() > 2) { val = s.substr(s[2] == '=' ? 3 : 2); have_val = true; }
    } else {
      a.pos.push_back(s);
      continue;
    }
    if (!sp) throw std::runtime_error("error: Found argument '" + s + "' which wasn't expected");
    if (sp->value) {
      if (!have_val) {
        if (i + 1 >= argc) throw std::runtime_error(std::string("error: The argument '--") + sp->lng + "' requires a value");
        val = argv[++i];
      }
      a.opt[sp->lng] = val;
    } else {
      a.flags.insert(sp->lng);
    }
  }
  return a;
}

inline int run_somatic(int argc, char** argv, const PhaseFn& phase) {
  CliArgs a = parse_cli(argc, argv, 2, {{"ref", 'r', true}, {"variants", 'b', true}, {"window-len", 'w', true}, {"tsv", 't', true},
                                        {"normal-output", 'n', true}, {"unsupported-allele-warning-only", 'u', false}, {"verbose", 'v', false}});
  if (a.pos.size() != 1 || !a.opt.count("ref") || !a.opt.count("variants"))
    throw std::runtime_error("error: The following required arguments were not provided: <tumor-sample> --ref <FILE> --variants <FILE>");
  mphio::BamFile bam(a.pos[0], io_threads_env());
  mphio::VcfFile vcf(a.opt["variants"]);
  mphio::FastaIndexed fasta(a.opt["ref"]);
  Outputs o;
  o.fasta = stdout;
  const std::string tsv = a.opt.count("tsv") ? a.opt["tsv"] : "info.tsv";
  const std::string nrm = a.opt.count("normal-output") ? a.opt["normal-output"] : "normal.fasta";
  o.normal = fopen(nrm.c_str(), "wb");
  if (!o.normal) throw std::runtime_error("cannot create " + nrm);
  o.tsv = fopen(tsv.c_str(), "wb");
  if (!o.tsv) throw std::runtime_error("cannot create " + tsv);
  IngestOptions io;
  io.window_len = a.opt.count("window-len") ? uint32_t(std::stoul(a.opt["window-len"])) : 27;
  io.warn_only = a.flags.count("unsupported-allele-warning-only") != 0;
  Packer packer(io.window_len);
  ingest(std::cin, bam, vcf, fasta, io, packer);
  Batch& b = packer.batch();
  PhaseRaw raw = phase(b);
  if (raw.err & MPH_E_REF_RANGE) throw Fatal("slice index out of range: refseq");
  if (raw.err & MPH_E_VARS_PER_WINDOW) throw Unsupported("more than 32 variants in one window / 64 in one read");
  if (raw.err & MPH_E_SLICE) throw Fatal("slice index out of range");
  if (raw.err & MPH_E_SEQ_SLOT) throw Unsupported("assembled haplotype longer than the sequence slot");
  if (raw.err & MPH_E_KEYS_PER_WINDOW) throw Unsupported(MPH_MSG_KEYS_PER_WINDOW);
  if (raw.err & MPH_E_RECS_PER_LIST) throw Unsupported(MPH_MSG_RECS_PER_LIST);
  if (raw.err) throw std::runtime_error("device error bits " + std::to_string(raw.err));
  Residue res(b, raw);
  std::vector<OutRecord> host_recs;
  ResidueStats st;
  res.run(0, uint32_t(b.txs.size()), host_recs, st);
  const std::vector<OutRecord> recs = ordered_records(b, raw, std::move(host_recs));
  write_records(b, recs, o);
  fclose(o.tsv);
  fclose(o.normal);
  fflush(stdout);
  return 0;
}

// microphaser normal <normal.bam> -r REF -b VCF [-w 27] [-t info.tsv] [-u] [-v]  (src/main.rs, src/cli.yaml `normal`)
inline int run_normal(int argc, char** argv, const PhaseFn& phase) {
  CliArgs a = parse_cli(argc, argv, 2, {{"ref", 'r', true}, {"variants", 'b', true}, {"window-len", 'w', true}, {"tsv", 't', true},
                                        {"unsupported-allele-warning-only", 'u', false}, {"verbose", 'v', false}});
  if (a.pos.size() != 1 || !a.opt.count("ref") || !a.opt.count("variants"))
    throw std::runtime_error("error: The following required arguments were not provided: <normal-sample> --ref <FILE> --variants <FILE>");
  mphio::BamFile bam(a.pos[0], io_threads_env());
  mphio::VcfFile vcf(a.opt["variants"]);
  mphio::FastaIndexed fasta(a.opt["ref"]);
  Outputs o;
  o.fasta = stdout;
  const std::string tsv = a.opt.count("tsv") ? a.opt["tsv"] : "info.tsv";
  o.tsv = fopen(tsv.c_str(), "wb");
  if (!o.tsv) throw std::runtime_error("cannot create " + tsv);
  IngestOptions io;
  io.window_len = a.opt.count("window-len") ? uint32_t(std::stoul(a.opt["window-len"])) : 27;
  io.warn_only = a.flags.count("unsupported-allele-warning-only") != 0;
  io.mode = 1;
  io.min_mapq = 0;
  Packer packer(io.window_len, 1);
  ingest(std::cin, bam, vcf, fasta, io, packer);
  Batch& b = packer.batch();
  PhaseRaw raw = phase(b);
  if (raw.err & MPH_E_REF_RANGE) throw Fatal("index out of bounds: refseq");
  if (raw.err & MPH_E_VARS_PER_WINDOW) throw Unsupported("more than 32 variants in one window / 64 in one read");
  if (raw.err & MPH_E_KEYS_PER_WINDOW) throw Unsupported(MPH_MSG_KEYS_PER_WINDOW);
  if (raw.err & MPH_E_RECS_PER_LIST) throw Unsupported(MPH_MSG_RECS_PER_LIST);
  if (raw.err) throw std::runtime_error("device error bits " + std::to_string(raw.err));
  if (raw.err & MPH_E_SLICE) throw Fatal("slice index out of range");
  if (raw.err & MPH_E_SEQ_SLOT) throw Unsupported("assembled haplotype longer than the sequence slot");
  ResidueNormal res(b, raw);
  std::vector<OutRecord> host_recs;
  ResidueStats st;
  res.run(0, uint32_t(b.txs.size()), host_recs, st);
  const std::vector<OutRecord> recs = ordered_records(b, raw, std::move(host_recs));
  write_records(b, recs, o);
  fclose(o.tsv);
  fflush(stdout);
  return 0;
}

inline int cli_main(int argc, char** argv, const PhaseFn& phase) {
  try {
    if (argc < 2) return 0;
    const std::string sub = argv[1];
    if (sub == "somatic") return run_somatic(argc, argv, phase);
    if (sub == "normal") return run_normal(argc, argv, phase);
    throw std::runtime_error("error: unknown subcommand " + sub);
  } catch (const Fatal& e) {
    fflush(stdout);
    fprintf(stderr, "thread 'main' panicked at '%s'\n", e.what());
    return 101;
  } catch (const Unsupported& e) {
    fflush(stdout);
    fprintf(stderr, "microphaser-b200: input needs the serial replay path, which is not implemented: %s\n", e.what());
    return 3;
  } catch (const std::exception& e) {
    fflush(stdout);
    fprintf(stderr, "%s\n", e.what());
    return 1;
  }
}

}  // namespace mph
