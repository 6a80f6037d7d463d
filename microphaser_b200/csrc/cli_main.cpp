// cli_main.cpp — `microphaser` command line with the reference's surface (src/main.rs:34-265,
// src/somatic_cli.yaml): GTF on stdin, mutant FASTA on stdout. Thin host over the C ABI of
// include/microphaser_gpu.h; the phasing itself runs on the GPU, there is no CPU fallback.
//   microphaser somatic <tumor.bam> --ref genome.fasta --variants tumor.vcf [-w 27] [--tsv info.tsv]
//                       [--normal-output normal.fasta] [-u] [-v]   < annotation.gtf > peptides.mt.fa
//   microphaser normal <normal.bam> --ref genome.fasta --variants normal.vcf [-w 27] [--tsv info.tsv] [-u] [-v] < annotation.gtf > peptides.wt.fa
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/microphaser_gpu.h"

namespace {

struct Spec { const char* lng; char shrt; bool value; };

// clap-style parsing: --name value, --name=value, -n value, -nvalue
bool parse_args(int argc, char** argv, const std::vector<Spec>& specs, std::map<std::string, std::string>& opt, std::vector<std::string>& pos) {
  for (int i = 2; i < argc; ++i) {
    std::string s = argv[i];
    const Spec* sp = nullptr;
    std::string val;
    bool have = false;
    if (s.rfind("--", 0) == 0) {
      std::string name = s.substr(2);
      size_t eq = name.find('=');
      if (eq != std::string::npos) { val = name.substr(eq + 1); name = name.substr(0, eq); have = true; }
      for (auto& x : specs) if (name == x.lng) sp = &x;
    } else if (s.size() >= 2 && s[0] == '-') {
      for (auto& x : specs) if (s[1] == x.shrt) sp = &x;
      if (sp && s.size() > 2) { val = s.substr(s[2] == '=' ? 3 : 2); have = true; }
    } else { pos.push_back(s); continue; }
    if (!sp) { fprintf(stderr, "error: Found argument '%s' which wasn't expected\n", s.c_str()); return false; }
    if (sp->value) {
      if (!have) { if (i + 1 >= argc) { fprintf(stderr, "error: The argument '--%s' requires a value\n", sp->lng); return false; } val = argv[++i]; }
      opt[sp->lng] = val;
    } else opt[sp->lng] = "1";
  }
  return true;
}

// exit status of a run; `unsupported` leads the message of MPH_ERR_UNSUPPORTED
int finish(mph_ctx* ctx, int rc, const char* unsupported) {
  int status = 0;
  if (rc == MPH_ERR_PANIC) { fprintf(stderr, "thread 'main' panicked at '%s'\n", mph_last_error(ctx)); status = 101; }
  else if (rc == MPH_ERR_UNSUPPORTED) { fprintf(stderr, "microphaser: %s: %s\n", unsupported, mph_last_error(ctx)); status = 3; }
  else if (rc != MPH_OK) { fprintf(stderr, "%s\n", mph_last_error(ctx)); status = 1; }
  return status;
}

// filter (src/filter_cli.yaml) and build_reference (src/build_ref_cli.yaml)
int run_secondary(const std::string& sub, int argc, char** argv) {
  std::map<std::string, std::string> opt;
  std::vector<std::string> pos;
  const bool filter = sub == "filter";
  if (filter) {
    if (!parse_args(argc, argv, {{"tsv", 't', true}, {"reference", 'r', true}, {"tsv-output", 'o', true}, {"similar-removed", 's', true},
                                 {"removed-peptides", 'p', true}, {"normal-output", 'n', true}, {"peptide-length", 'l', true}, {"verbose", 'v', false}}, opt, pos)) return 1;
    if (!opt.count("tsv") || !opt.count("reference")) { fprintf(stderr, "error: The following required arguments were not provided: --tsv <FILE> --reference <FILE>\n"); return 1; }
  } else {
    if (!parse_args(argc, argv, {{"reference", 'r', true}, {"output", 'o', true}, {"peptide-length", 'l', true}, {"verbose", 'v', false}}, opt, pos)) return 1;
    if (!opt.count("reference") || !opt.count("output")) { fprintf(stderr, "error: The following required arguments were not provided: --reference <FILE> --output <FILE>\n"); return 1; }
  }
  auto get = [&](const char* k, const char* d) { return opt.count(k) ? opt[k] : std::string(d); };
  const uint32_t l = uint32_t(strtoul(get("peptide-length", "9").c_str(), nullptr, 10));
  mph_ctx* ctx = nullptr;
  if (mph_ctx_create(getenv("MPH_DEVICE") ? atoi(getenv("MPH_DEVICE")) : 0, &ctx) != MPH_OK) { fprintf(stderr, "microphaser: %s\n", mph_last_error(nullptr)); return 1; }
  const int rc = filter ? mph_run_filter(ctx, opt["reference"].c_str(), opt["tsv"].c_str(), "-", get("normal-output", "normal.filtered.fa").c_str(),
                                         get("tsv-output", "info.filtered.tsv").c_str(), get("similar-removed", "info.removed.tsv").c_str(),
                                         get("removed-peptides", "peptides.removed.fasta").c_str(), l)
                        : mph_run_build_reference(ctx, opt["reference"].c_str(), opt["output"].c_str(), "-", l);
  const int st = finish(ctx, rc, "not supported by the GPU path");
  mph_ctx_destroy(ctx);
  return st;
}

}  // namespace

int main(int argc, char** argv) {
  if (argc < 2) return 0;
  const std::string sub = argv[1];
  if (sub == "filter" || sub == "build_reference") return run_secondary(sub, argc, argv);
  const bool normal_mode = sub == "normal";  // src/main.rs `normal`: same arguments without --normal-output
  if (sub != "somatic" && !normal_mode) {
    fprintf(stderr, "error: sub-command '%s' is not part of the GPU phasing path\n", sub.c_str());
    return 1;
  }
  std::map<std::string, std::string> opt;
  std::vector<std::string> pos;
  if (!parse_args(argc, argv, {{"ref", 'r', true}, {"variants", 'b', true}, {"window-len", 'w', true}, {"tsv", 't', true}, {"normal-output", 'n', true},
                               {"unsupported-allele-warning-only", 'u', false}, {"verbose", 'v', false}}, opt, pos)) return 1;
  const bool warn_only = opt.count("unsupported-allele-warning-only") != 0;
  if (pos.size() != 1 || !opt.count("ref") || !opt.count("variants")) {
    fprintf(stderr, "error: The following required arguments were not provided: <tumor-sample> --ref <FILE> --variants <FILE>\n");
    return 1;
  }
  const std::string tsv = opt.count("tsv") ? opt["tsv"] : "info.tsv";
  const std::string nrm = opt.count("normal-output") ? opt["normal-output"] : "normal.fasta";
  const uint32_t wl = opt.count("window-len") ? uint32_t(strtoul(opt["window-len"].c_str(), nullptr, 10)) : 27;
  // device selection stays out of the (frozen) command line: MPH_DEVICES=0,1,2,3 shards the genes over several GPUs
  std::vector<int> devices;
  if (const char* dl = getenv("MPH_DEVICES")) {
    for (const char* p = dl; *p;) {
      devices.push_back(atoi(p));
      while (*p && *p != ',') ++p;
      if (*p == ',') ++p;
    }
  }
  if (devices.empty()) devices.push_back(getenv("MPH_DEVICE") ? atoi(getenv("MPH_DEVICE")) : 0);
  std::vector<mph_ctx*> ctxs;
  int rc = MPH_OK;
  for (int dv : devices) {
    mph_ctx* c = nullptr;
    rc = mph_ctx_create(dv, &c);
    if (rc != MPH_OK) { fprintf(stderr, "microphaser: %s\n", mph_last_error(nullptr)); return 1; }
    ctxs.push_back(c);
  }
  mph_ctx* ctx = ctxs[0];
  if (normal_mode)
    rc = mph_run_normal(ctx, pos[0].c_str(), opt["ref"].c_str(), opt["variants"].c_str(), "-", "-", tsv.c_str(), wl, warn_only);
  else
    rc = mph_run_somatic_multi(ctxs.data(), int(ctxs.size()), pos[0].c_str(), opt["ref"].c_str(), opt["variants"].c_str(), "-", "-", tsv.c_str(),
                               nrm.c_str(), wl, warn_only);
  const int status = finish(ctx, rc, "input needs the serial replay path, which is not implemented");
  for (auto c : ctxs) mph_ctx_destroy(c);
  return status;
}
