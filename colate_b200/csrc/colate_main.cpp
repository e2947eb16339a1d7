// `Colate` command-line host, `--mode mut` on two precomputed .colate.in files.
// Mirrors the reference CLI (include/coal/Colate.cpp:6-116, flag table 11-45) and the control
// flow of mut() (include/coal/coal.cpp:3071-3863); all computation goes through the C ABI
// (include/colate_b200.h) onto the GPU.  There is no CPU fallback.
#include <sys/resource.h>
#include <sys/stat.h>
#include <sys/time.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <map>
#include <set>
#include <sstream>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "../../include/colate_b200.h"

namespace {

struct Options {
  std::map<std::string, std::string> kv;
  int count(const std::string& k) const { return kv.count(k) ? 1 : 0; }
  const std::string& get(const std::string& k) const { return kv.at(k); }
};

// option names of the reference's table (Colate.cpp:11-45); value-less: help, strandfilter
const char* kValueOpts[] = {"mode", "anc", "mut", "target_bcf", "reference_bcf", "target_mask", "reference_mask", "target_table",
                            "target_bam", "reference_bam", "target_tmp", "reference_tmp", "target_age", "reference_age", "ref_genome",
                            "anc_genome", "mask", "mask_cutoff", "chr", "bins", "lineage_bin", "outgroup_tmrca", "years_per_gen",
                            "coal", "seed", "num_bootstraps", "filters", "groups", "poplabels", "map", "input", "output",
                            // additions of this build
                            "num_bootstrap", "device", "devices", "pairs", "targets"};

void help()
{
  std::cout << "Usage:\n  Colate --mode mut --mut <prefix> --target_tmp <t.colate.in> --reference_tmp <r.colate.in> --bins x,y,step\n"
               "         [--chr <file>] [--target_mask <prefix>] [--reference_mask <prefix>] [--target_age <years>]\n"
               "         [--reference_age <years>] [--years_per_gen <float>] [--coal <file>] [--seed <int>]\n"
               "         [--num_bootstraps <int>] [--device <int> | --devices <i,j,...>] [--host_parse] -o <output prefix>\n"
               "  Colate --mode mut --mut <prefix> --pairs <file> --seed <int> (--bins x,y,step | --coal <file>) [--chr <file>]\n"
               "         [--ref_genome <prefix>] [--filters mapq,length,mismatches] [--years_per_gen <float>] [--num_bootstraps <int>]\n"
               "         [--devices <i,j,...>] [--host_parse]\n"
               "    a cohort in one job: every non-blank line of <file> not starting with '#' is one run\n"
               "      <target_tmp> <reference_tmp> <output_prefix> [target_age=<years>] [reference_age=<years>]\n"
               "      [target_mask=<prefix>] [reference_mask=<prefix>]\n"
               "      target_bam=<t.bam> reference_bam=<r.bam> <output_prefix> [same keys]     (needs --ref_genome)\n"
               "      target_bcf=<prefix> reference_bcf=<prefix> <output_prefix> [same keys]   (needs --chr)\n"
               "    with the shared flags; each line's .coal / .bin (and, for bam and bcf lines, .colate_mat) equal those of the\n"
               "    single-pair run with the same flags; every BAM file and BCF / VCF prefix is decoded once per device (a failing\n"
               "    input fails the lines that use it, the others complete, the exit status is 1)\n"
               "  Colate --mode mut --mut <prefix> --target_bam <t.bam> --reference_bam <r.bam> --ref_genome <prefix> (--bins x,y,step | --coal <file>)\n"
               "         [--chr <file>] [--target_mask <prefix>] [--reference_mask <prefix>] [--target_age <years>] [--reference_age <years>]\n"
               "         [--years_per_gen <float>] [--seed <int>] [--num_bootstraps <int>] [--filters mapq,length,mismatches] [--device <int>]\n"
               "         -o <output prefix>     (also writes <output prefix>.colate_mat; one device; no --strandfilter)\n"
               "  Colate --mode mut --mut <prefix> --chr <file> --target_bcf <prefix> --reference_bcf <prefix> [--ref_genome <prefix>]\n"
               "         (--bins x,y,step | --coal <file>) [--target_mask <prefix>] [--reference_mask <prefix>] [--target_age <years>]\n"
               "         [--reference_age <years>] [--years_per_gen <float>] [--seed <int>] [--num_bootstraps <int>] [--device <int>]\n"
               "         -o <output prefix>     (reads <prefix>_chr<c>.bcf per --chr entry, BCF or bgzipped VCF as for htslib;\n"
               "                                 also writes <output prefix>.colate_mat; one device)\n"
               "    a BCF / VCF <prefix> without any <prefix>_chr<c>.bcf that is itself a file is read as a whole genome: --chr entry\n"
               "    c reads its contig c or chr<c> (everywhere target_bcf / reference_bcf are read, --pairs and --targets lines too)\n"
               "  Colate --mode make_tmp --mut <prefix> --chr <file> --target_bcf <prefix> --ref_genome <prefix> [--target_mask <prefix>]\n"
               "         [--device <int>] -o <output prefix>     (writes <output prefix>.colate.in)\n"
               "  Colate --mode make_tmp --mut <prefix> --target_bam <t.bam> --ref_genome <prefix> [--chr <file>] [--target_mask <prefix>]\n"
               "         [--filters mapq,length,mismatches] [--device <int>] -o <output prefix>     (writes <output prefix>.colate.in)\n"
               "  Colate --mode make_tmp --mut <prefix> --target_table <file> --ref_genome <prefix> [--chr <file>] [--target_mask <prefix>] -o <output prefix>\n"
               "  Colate --mode make_tmp --mut <prefix> --ref_genome <prefix> --targets <file> [--chr <file>] [--filters mapq,length,mismatches]\n"
               "         [--device <int>]\n"
               "    many targets in one job: every non-blank line of <file> not starting with '#' is one target\n"
               "      (target_bam=<t.bam> | target_bcf=<prefix>) <output_prefix> [target_mask=<prefix>]\n"
               "    with the shared flags; each line's <output_prefix>.colate.in equals that of the single-target run (target_bcf needs --chr;\n"
               "    a failing line writes no file, the others complete, the exit status is 1)\n"
            << std::endl;
}

bool parse(int argc, char** argv, Options& o)
{
  std::set<std::string> val(std::begin(kValueOpts), std::end(kValueOpts));
  for (int i = 1; i < argc; i++) {
    std::string a = argv[i];
    std::string key, value;
    bool has_value = false;
    if (a.rfind("--", 0) == 0) {
      key = a.substr(2);
      size_t eq = key.find('=');
      if (eq != std::string::npos) { value = key.substr(eq + 1); key = key.substr(0, eq); has_value = true; }
    } else if (a == "-o") key = "output";
    else if (a == "-i") key = "input";
    else { std::cerr << "Option '" << a << "' does not exist" << std::endl; return false; }
    if (key == "help" || key == "strandfilter" || key == "host_parse") { o.kv[key] = "1"; continue; }   // host_parse: addition of this build
    if (!val.count(key)) {  // cxxopts::option_not_exists_exception in the reference (cxxopts.hpp:1180-1185)
      std::cerr << "Option '" << key << "' does not exist" << std::endl;
      return false;
    }
    if (!has_value) {
      if (i + 1 >= argc) { std::cerr << "Option '" << key << "' is missing an argument" << std::endl; return false; }
      value = argv[++i];
    }
    o.kv[key] = value;
  }
  return true;
}

int die(const std::string& what)
{
  std::cerr << what << ": " << colate_last_error() << std::endl;
  return 1;
}

bool file_exists(const std::string& p) { std::ifstream f(p); return f.good(); }

// COLATE_TIMING=1: wall-clock phases on stderr
struct Phases {
  bool on = getenv("COLATE_TIMING") != nullptr;
  double t0 = now(), last = t0;
  static double now() { timeval tv; gettimeofday(&tv, nullptr); return tv.tv_sec + 1e-6 * tv.tv_usec; }
  void tick(const char* what) { if (!on) return; const double t = now(); fprintf(stderr, "[timing] %-28s %8.3f s (total %.3f)\n", what, t - last, t - t0); last = t; }
};

// one GPU of the job: its handle, its contiguous range of the --chr list and what stage i found there
struct Dev {
  int id = 0;
  colate_handle* h = nullptr;
  int c_lo = 0, c_hi = 0;
  std::vector<int64_t> site_off;            // rows of its chromosomes (local offsets)
  std::vector<int32_t> pos;                 // their positions on the host (mask lookups only)
  int64_t n_used = 0, used_base = 0, extra_words = 0;
  int n_blocks = 0, block_base = 0;
  uint32_t mt_after[COLATE_MT_WORDS];
  int rc = 0;
  std::string err;
  bool fail(const std::string& what) { rc = 1; err = what + ": " + colate_last_error(); return false; }
};

// contiguous ranges of the --chr list per device, balanced by weight (rows or text bytes); every device keeps at least
// one chromosome while there are enough of them (same rule as colate_b200/dist.py: split_chromosomes)
std::vector<std::pair<int, int>> split_chromosomes(const std::vector<int64_t>& weight, int world)
{
  const int n = (int)weight.size();
  std::vector<double> cum(n + 1, 0.0);
  for (int c = 0; c < n; c++) cum[c + 1] = cum[c] + (double)weight[c];
  std::vector<int> bounds{0};
  for (int r = 1; r < world; r++) {
    const int lo = std::min(n, bounds.back() + 1);
    const int hi = std::min(n, std::max(lo, n - (world - r)));
    const double target = cum[n] * r / world;
    int best = lo;
    for (int c = lo; c <= hi; c++) if (std::fabs(cum[c] - target) < std::fabs(cum[best] - target)) best = c;
    bounds.push_back(best);
  }
  bounds.push_back(n);
  std::vector<std::pair<int, int>> out;
  for (int r = 0; r < world; r++) out.push_back({bounds[r], bounds[r + 1]});
  return out;
}

template <class F> void on_every_device(std::vector<Dev>& devs, F f)
{
  std::vector<std::thread> th;
  for (size_t g = 1; g < devs.size(); g++) th.emplace_back([&, g] { f(devs[g]); });
  f(devs[0]);
  for (auto& t : th) t.join();
}

bool all_ok(const std::vector<Dev>& devs)
{
  bool ok = true;
  for (auto& d : devs) if (d.rc) { std::cerr << "device " << d.id << ": " << d.err << std::endl; ok = false; }
  return ok;
}

// --filters mapq,length,mismatches (coal.cpp:3096: default "20,30,10")
bool parse_filters(const Options& o, int f[3])
{
  f[0] = 20; f[1] = 30; f[2] = 10;
  if (!o.count("filters")) return true;
  std::stringstream ss(o.get("filters"));
  std::string tok;
  int k = 0;
  while (std::getline(ss, tok, ',')) {
    if (k == 3 || tok.empty()) return false;
    char* end = nullptr;
    f[k++] = (int)strtol(tok.c_str(), &end, 10);
    if (*end) return false;
  }
  return k == 3;
}

// --ref_genome (fasta::Read, data.cpp:213-237): <prefix>_chr<name>.fa per --chr entry, or the file itself without --chr
struct RefGenome {
  std::vector<uint8_t*> seq;
  std::vector<int64_t> len;
  ~RefGenome() { for (uint8_t* p : seq) colate_free(p); }
  bool read(const Options& o, const std::vector<std::string>& name_chr)
  {
    for (auto& nm : name_chr) {
      const std::string f = o.count("chr") ? o.get("ref_genome") + "_chr" + nm + ".fa" : o.get("ref_genome");
      uint8_t* p = nullptr;
      const int64_t n = colate_read_fasta(f.c_str(), &p);
      if (n < 0) { std::cerr << colate_last_error() << std::endl; return false; }
      seq.push_back(p);
      len.push_back(n);
    }
    return true;
  }
};

// BAM inputs (--target_bam / --reference_bam): what this build does not restate is refused before any device is touched
bool bam_args_ok(const Options& o, bool need_both)
{
  auto bad = [](const std::string& what) { std::cerr << "Error: " << what << std::endl; return false; };
  if (o.count("strandfilter")) return bad("--strandfilter is not supported with BAM inputs (its read filter is not restated)");
  for (const char* k : {"target_tmp", "reference_tmp", "target_bcf", "reference_bcf", "target_table"})
    if (o.count(k)) return bad(std::string("--") + k + " cannot be mixed with BAM inputs");
  if (need_both && !(o.count("target_bam") && o.count("reference_bam")))
    return bad("--mode mut with BAM inputs needs both --target_bam and --reference_bam (bam/tmp and bam/bcf mixes are not supported)");
  if (o.count("pairs")) return bad("--pairs cannot be combined with BAM inputs");
  const std::string dev = o.count("devices") ? o.get("devices") : "";
  if (dev.find(',') != std::string::npos) return bad("BAM inputs run on one device (--device <i>)");
  if (!o.count("ref_genome")) return bad("BAM inputs need --ref_genome");
  int f[3];
  if (!parse_filters(o, f)) return bad("--filters takes three integers: mapq,length,mismatches");
  return true;
}

// BCF inputs (--target_bcf / --reference_bcf, one <prefix>_chr<c>.bcf per --chr entry): what this build does not restate is
// refused before any device is touched -- the bcf + bam, bcf-only and bam + bcf front-ends (parse_bamvcf, parse_vcf,
// parse_onebamvcf) are not pinned by any reference run, nor are bcf files without --chr
bool bcf_args_ok(const Options& o, bool need_both)
{
  auto bad = [](const std::string& what) { std::cerr << "Error: " << what << std::endl; return false; };
  for (const char* k : {"target_tmp", "reference_tmp", "target_bam", "reference_bam", "target_table"})
    if (o.count(k)) return bad(std::string("--") + k + " cannot be mixed with BCF inputs");
  if (need_both && !(o.count("target_bcf") && o.count("reference_bcf")))
    return bad("--mode mut with BCF inputs needs both --target_bcf and --reference_bcf (bcf/tmp, bcf/bam and single-bcf runs are not supported)");
  if (o.count("pairs")) return bad("--pairs cannot be combined with BCF inputs");
  const std::string dev = o.count("devices") ? o.get("devices") : "";
  if (dev.find(',') != std::string::npos) return bad("BCF inputs run on one device (--device <i>)");
  if (!o.count("chr")) return bad("BCF inputs need --chr (one <prefix>_chr<c>.bcf file per chromosome)");
  return true;
}

// A BCF / VCF input X (--target_bcf, --reference_bcf, target_bcf= / reference_bcf= lines): per-chromosome files X_chr<c>.bcf, as
// the reference opens them, when any of them exists; otherwise X itself when it is a regular file, read as a whole genome (one
// file, --chr entry c reading the contig c or chr<c>); otherwise the per-chromosome files, whose absence is reported as before.
struct GenotypeInput {
  bool whole = false;
  std::vector<std::string> files;   // the per-chromosome files, or X
};
GenotypeInput genotype_input(const std::string& x, const std::vector<std::string>& name_chr)
{
  GenotypeInput in;
  bool any = false;
  struct stat st;
  for (auto& nm : name_chr) {
    in.files.push_back(x + "_chr" + nm + ".bcf");
    any |= stat(in.files.back().c_str(), &st) == 0;
  }
  if (!any && stat(x.c_str(), &st) == 0 && S_ISREG(st.st_mode)) {
    in.whole = true;
    in.files.assign(1, x);
  }
  return in;
}

int run_mut(const Options& options)
{
  if (!options.count("mut") || !options.count("output")) {  // coal.cpp:3077-3086
    std::cout << "Not enough arguments supplied." << std::endl;
    std::cout << "Needed: mut, bins, output. Optional: target_tmp, reference_tmp, target_bcf, reference_bcf, target_bam, "
                 "reference_bam, ref_genome, target_age, reference_age, target_mask, reference_mask, coal, num_bootstrap, filters."
              << std::endl;
    help();
    std::cout << "Calculate coalescence rates for sample." << std::endl;
    exit(0);
  }
  const bool bam = options.count("target_bam") || options.count("reference_bam");
  if (bam && !bam_args_ok(options, true)) return 1;
  const bool bcf = options.count("target_bcf") || options.count("reference_bcf");
  if (bcf && !bcf_args_ok(options, true)) return 1;
  const bool counts_front_end = bam || bcf;   // every front-end but tmp/tmp: raw count weights, counts / 1e3, a .colate_mat
  std::cerr << "---------------------------------------------------------" << std::endl;
  std::cerr << "Calculating coalescence rates for (ancient) samples.." << std::endl;

  double ypg = 28.0;
  const bool has_ypg = options.count("years_per_gen");
  double age = colate_age_generations(options.count("target_age") ? options.get("target_age").c_str() : nullptr,
                                      options.count("reference_age") ? options.get("reference_age").c_str() : nullptr, has_ypg,
                                      has_ypg ? strtof(options.get("years_per_gen").c_str(), nullptr) : 0.0f, &ypg);
  std::cerr << age << std::endl;  // coal.cpp:3119
  const bool is_ancient = age > 0.0;
  std::cerr << "num_bins: " << COLATE_NUM_AGE_BINS << std::endl;
  if (!colate_libm_exact())
    std::cerr << "Warning: this host's libm is not glibc 2.39 with the FMA variants of exp/log/log1p. The EM on the GPU follows that\n"
                 "         libm op for op; the reference compiled and run on THIS host may differ in the last bits of every exp/log,\n"
                 "         which moves the ill-conditioned rates of the deepest epochs by up to ~1e-5 relative (DESIGN.md 5)." << std::endl;

  int seed = (int)(std::time(0) + getpid());  // coal.cpp:3158
  if (options.count("seed")) seed = atoi(options.get("seed").c_str());
  int R = 1;  // coal.cpp:3164; the README spells the flag --num_bootstrap, the code --num_bootstraps
  if (options.count("num_bootstraps")) R = atoi(options.get("num_bootstraps").c_str());
  else if (options.count("num_bootstrap")) R = atoi(options.get("num_bootstrap").c_str());
  if (R < 0) R = 0;
  const std::string out = options.get("output");

  // devices of this job: --devices 0,1,... (chromosomes are dealt to them for stage i, replicates for stages ii-iii; the
  // two small exchanges -- used rows / blocks per device, the block histograms -- go through this process' memory)
  std::vector<Dev> devs;
  {
    std::string list = options.count("devices") ? options.get("devices") : (options.count("device") ? options.get("device") : "0");
    std::stringstream ss(list);
    std::string tok;
    while (std::getline(ss, tok, ',')) if (!tok.empty()) { Dev d; d.id = atoi(tok.c_str()); devs.push_back(d); }
    if (devs.empty()) { Dev d; devs.push_back(d); }
  }
  const int G = (int)devs.size();

  Phases ph;
  // the CUDA contexts come up (about a second) while the main thread reads the input files
  std::vector<std::thread> init;
  for (int g = 0; g < G; g++) init.emplace_back([&, g] { if (colate_create(devs[g].id, &devs[g].h)) devs[g].fail("colate_create"); });
  struct Joiner { std::vector<std::thread>& t; ~Joiner() { for (auto& x : t) if (x.joinable()) x.join(); } } joiner{init};
  auto wait_for_devices = [&]() -> bool {
    for (auto& x : init) if (x.joinable()) x.join();
    return all_ok(devs);
  };
  std::vector<double> counts((size_t)std::max(R, 1) * 2 * COLATE_NUM_AGE_BINS, 0.0);
  std::vector<double> block_stats((size_t)COLATE_MAX_BLOCKS * 4 * COLATE_NUM_AGE_BINS);
  std::vector<int32_t> weights;
  int num_blocks = 0;
  bool from_cache = false;
  double cached_age_bin[COLATE_NUM_AGE_BINS];
  uint32_t mt[COLATE_MT_WORDS];
  colate_mt_seed((uint32_t)seed, mt);

  if (file_exists(out + ".colate_mat")) {  // stale-cache behaviour of coal.cpp:3169-3170, 3471-3499
    std::cerr << "Loading precomputed file " << out << ".colate_mat" << std::endl;
    std::ifstream is(out + ".colate_mat");
    for (int b = 0; b < COLATE_NUM_AGE_BINS; b++) is >> cached_age_bin[b];   // the reference overwrites age_bin[] with the file's values (coal.cpp:3481-3483)
    for (int i = 0; i < R; i++)
      for (int k = 0; k < 2 * COLATE_NUM_AGE_BINS; k++) is >> counts[(size_t)i * 2 * COLATE_NUM_AGE_BINS + k];
    from_cache = true;
  } else {
    if (!counts_front_end && !(options.count("target_tmp") && options.count("reference_tmp"))) {
      std::cerr << "This build reads --target_tmp/--reference_tmp (.colate.in), --target_bam/--reference_bam or --target_bcf/--reference_bcf "
                   "inputs." << std::endl;
      return 1;
    }
    // file lists, coal.cpp:3290-3316
    std::vector<std::string> name_chr, f_mut, f_tmask, f_rmask;
    if (options.count("chr")) {
      std::ifstream is(options.get("chr"));
      if (is.fail()) std::cerr << "Error while opening file " << options.get("chr") << std::endl;
      std::string line;
      while (std::getline(is, line)) {
        name_chr.push_back(line);
        f_mut.push_back(options.get("mut") + "_chr" + line + ".mut");
        if (options.count("target_mask")) f_tmask.push_back(options.get("target_mask") + "_chr" + line + ".fa");
        if (options.count("reference_mask")) f_rmask.push_back(options.get("reference_mask") + "_chr" + line + ".fa");
      }
    } else {
      name_chr.push_back("");
      f_mut.push_back(options.get("mut"));
      if (options.count("target_mask")) f_tmask.push_back(options.get("target_mask"));
      if (options.count("reference_mask")) f_rmask.push_back(options.get("reference_mask"));
    }
    const int n_chr = (int)name_chr.size();
    {
      std::set<std::string> uniq(name_chr.begin(), name_chr.end());
      if ((int)uniq.size() != n_chr) { std::cerr << "Duplicate chromosome names in --chr" << std::endl; return 1; }
    }
    // readers.  Plain-text .mut files are parsed on the GPU (colate_ingest_*: the bytes go to the device, one thread
    // per row); if any file only exists as .gz the host reader (zlib) takes over for all of them.
    std::vector<std::vector<char>> texts(n_chr);
    bool all_plain = !options.count("host_parse");
    for (int c = 0; c < n_chr && all_plain; c++) {
      FILE* f = fopen(f_mut[c].c_str(), "rb");
      if (!f) { all_plain = false; break; }
      fseek(f, 0, SEEK_END);
      const long sz = ftell(f);
      fseek(f, 0, SEEK_SET);
      texts[c].resize((size_t)std::max(sz, 0L));
      if (sz > 0 && fread(texts[c].data(), 1, (size_t)sz, f) != (size_t)sz) all_plain = false;
      fclose(f);
    }
    struct SitesHost { std::vector<int64_t> off; std::vector<int32_t> pos; std::vector<float> ab, ae; std::vector<uint32_t> meta; } sh;
    // the two .colate.in files.  One device: the file image goes to the GPU and is decoded there (colate_ingest_colate_in).
    // Several devices: decoded once on the host, the chromosome seek (coal.cpp:2125-2145) emulated on the WHOLE record
    // stream, and every device receives the records and ranges of its own chromosomes.
    std::vector<const char*> names;
    for (auto& s : name_chr) names.push_back(s.c_str());
    const std::string files[2] = {options.get(bam ? "target_bam" : bcf ? "target_bcf" : "target_tmp"),
                                  options.get(bam ? "reference_bam" : bcf ? "reference_bcf" : "reference_tmp")};
    GenotypeInput bcf_in[2];   // <prefix>_chr<c>.bcf, as the reference opens them, or one whole-genome file
    std::vector<const char*> bcf_paths[2];
    for (int g = 0; g < 2 && bcf; g++) {
      bcf_in[g] = genotype_input(files[g], name_chr);
      for (auto& f : bcf_in[g].files) bcf_paths[g].push_back(f.c_str());
    }
    const bool bcf_whole = bcf_in[0].whole || bcf_in[1].whole;
    struct GenomeHost { int64_t n = 0; std::vector<char> image; std::vector<int32_t> rc, bp, aaf, daf; std::vector<uint16_t> al; std::vector<int64_t> first, end; } gh[2];
    RefGenome refg;
    int filters[3];
    parse_filters(options, filters);
    if ((bam || (bcf && options.count("ref_genome"))) && !refg.read(options, name_chr)) return 1;
    for (int g = 0; g < 2 && !counts_front_end; g++) {
      FILE* f = fopen(files[g].c_str(), "rb");
      if (!f) { std::cerr << "Failed to open " << files[g] << std::endl; continue; }  // the reference only warns (coal.cpp:2093-2098)
      fseek(f, 0, SEEK_END);
      const long sz = ftell(f);
      fseek(f, 0, SEEK_SET);
      gh[g].image.resize((size_t)std::max(sz, 0L));
      if (sz > 0 && fread(gh[g].image.data(), 1, (size_t)sz, f) != (size_t)sz) std::cerr << "short read on " << files[g] << std::endl;
      fclose(f);
      if (G > 1) {
        const int64_t cap = (int64_t)gh[g].image.size() / 18 + 16;
        gh[g].rc.resize(cap); gh[g].bp.resize(cap); gh[g].aaf.resize(cap); gh[g].daf.resize(cap); gh[g].al.resize(cap);
        int64_t n = colate_read_colate_in(files[g].c_str(), n_chr, names.data(), cap, gh[g].rc.data(), gh[g].bp.data(), gh[g].aaf.data(),
                                          gh[g].daf.data(), gh[g].al.data());
        if (n < 0) { std::cerr << colate_last_error() << std::endl; n = 0; }
        gh[g].n = n;
        gh[g].first.resize(n_chr); gh[g].end.resize(n_chr);
        colate_chr_ranges(n_chr, n, gh[g].rc.data(), gh[g].first.data(), gh[g].end.data());
        std::vector<char>().swap(gh[g].image);
      }
    }
    ph.tick("read input files");
    if (!wait_for_devices()) return 1;
    ph.tick("wait for the CUDA context");
    if (!all_plain) {
      sh.off.assign(n_chr + 1, 0);
      for (int c = 0; c < n_chr; c++) {
        std::cerr << "parsing CHR: " << c + 1 << " / " << n_chr << std::endl;
        int64_t n = colate_read_mut(f_mut[c].c_str(), 0, nullptr, nullptr, nullptr, nullptr);
        if (n < 0) { std::cerr << colate_last_error() << std::endl; exit(1); }
        size_t o = sh.pos.size();
        sh.pos.resize(o + n); sh.ab.resize(o + n); sh.ae.resize(o + n); sh.meta.resize(o + n);
        if (colate_read_mut(f_mut[c].c_str(), n, sh.pos.data() + o, sh.ab.data() + o, sh.ae.data() + o, sh.meta.data() + o) < 0) {
          std::cerr << colate_last_error() << std::endl;
          exit(1);
        }
        sh.off[c + 1] = (int64_t)sh.pos.size();
      }
    }

    // chromosomes -> devices, balanced by text bytes / rows
    std::vector<int64_t> w(n_chr);
    for (int c = 0; c < n_chr; c++) w[c] = all_plain ? (int64_t)texts[c].size() : sh.off[c + 1] - sh.off[c];
    const auto parts = split_chromosomes(w, G);
    for (int g = 0; g < G; g++) { devs[g].c_lo = parts[g].first; devs[g].c_hi = parts[g].second; }
    for (int c = 0; c < n_chr; c++) std::cerr << "parsing CHR: " << c + 1 << " / " << n_chr << std::endl;

    // ---- per device: sites, genomes, masks, flag pass (coal.cpp:2148-2219)
    on_every_device(devs, [&](Dev& d) {
      const int nc = d.c_hi - d.c_lo;
      d.site_off.assign(nc + 1, 0);
      if (all_plain) {
        int64_t bytes = 0;
        for (int c = d.c_lo; c < d.c_hi; c++) bytes += (int64_t)texts[c].size();
        if (nc == 0) {
          const int64_t zero = 0;
          if (colate_set_sites(d.h, 0, &zero, nullptr, nullptr, nullptr, nullptr, 0)) { d.fail("colate_set_sites"); return; }
        } else {
          if (colate_ingest_begin(d.h, nc, bytes / 20 + nc)) { d.fail("colate_ingest_begin"); return; }
          for (int c = d.c_lo; c < d.c_hi; c++) {
            const int64_t n = colate_ingest_mut_text(d.h, texts[c].data(), (int64_t)texts[c].size(), 0);
            if (n < 0) { d.fail("colate_ingest_mut_text"); return; }
            d.site_off[c - d.c_lo + 1] = d.site_off[c - d.c_lo] + n;
            std::vector<char>().swap(texts[c]);
          }
          if (colate_ingest_end(d.h)) { d.fail("colate_ingest_end"); return; }
        }
        if (nc > 0 && (options.count("target_mask") || options.count("reference_mask"))) {   // the mask gather runs on host positions
          d.pos.resize((size_t)d.site_off[nc]);
          if (colate_ingest_fetch(d.h, 0, d.site_off[nc], d.pos.data(), nullptr, nullptr, nullptr)) { d.fail("colate_ingest_fetch"); return; }
        }
      } else {
        const int64_t s0 = sh.off[d.c_lo];
        for (int c = 0; c <= nc; c++) d.site_off[c] = sh.off[d.c_lo + c] - s0;
        if (colate_set_sites(d.h, nc, d.site_off.data(), sh.pos.data() + s0, sh.ab.data() + s0, sh.ae.data() + s0, sh.meta.data() + s0, 0)) {
          d.fail("colate_set_sites");
          return;
        }
        d.pos.assign(sh.pos.begin() + s0, sh.pos.begin() + sh.off[d.c_hi]);
      }
      // BAM genomes: the pileup of each file at the rows (parse_onebambam's bam_parser, coal.cpp:1799-2069); BCF genomes: the
      // decoder half of parse_vcfvcf (coal.cpp:997-1137) per genome.  Both front-ends: raw count weights and 1e3 normalisation
      if (counts_front_end && colate_set_option(d.h, "front_end", 1)) { d.fail("colate_set_option"); return; }
      // a whole-genome input reads --ref_genome resident on the device
      if (bcf_whole && !refg.seq.empty() && colate_set_ref_genome(d.h, n_chr, (const uint8_t* const*)refg.seq.data(), refg.len.data())) {
        d.fail("colate_set_ref_genome");
        return;
      }
      for (int g = 0; g < 2; g++) {
        if (bcf && bcf_in[g].whole) {
          if (colate_rows_from_bcf_genome(d.h, g == 0 ? 0 : -1, g == 1 ? 1 : -1, n_chr, names.data(), files[g].c_str(), refg.seq.empty() ? 0 : 1, 0)) {
            d.fail(files[g]);
            return;
          }
        } else if (bcf) {
          if (colate_rows_from_bcf(d.h, g, g == 0 ? COLATE_BCF_TARGET : COLATE_BCF_REFERENCE, n_chr, names.data(), bcf_paths[g].data(),
                                   refg.seq.empty() ? nullptr : (const uint8_t* const*)refg.seq.data(), refg.seq.empty() ? nullptr : refg.len.data(), 0,
                                   nullptr, nullptr)) {
            d.fail(files[g]);
            return;
          }
        } else if (bam) {
          if (colate_pileup_bam(d.h, g, files[g].c_str(), n_chr, names.data(), (const uint8_t* const*)refg.seq.data(), refg.len.data(), filters[0],
                                filters[1], filters[2], 0, nullptr)) {
            d.fail(files[g]);
            return;
          }
        } else if (G == 1) {
          if (colate_ingest_colate_in(d.h, g, gh[g].image.data(), (int64_t)gh[g].image.size(), n_chr, names.data(), 0) < 0) {
            d.fail("colate_ingest_colate_in");
            return;
          }
        } else {
          // records [r0, r1) cover the ranges of this device's chromosomes
          int64_t r0 = gh[g].n, r1 = 0;
          for (int c = d.c_lo; c < d.c_hi; c++)
            if (gh[g].first[c] >= 0) { r0 = std::min(r0, gh[g].first[c]); r1 = std::max(r1, gh[g].end[c]); }
          if (r1 < r0) { r0 = 0; r1 = 0; }
          std::vector<int64_t> first(nc + 1), end(nc + 1);
          for (int c = d.c_lo; c < d.c_hi; c++) {
            first[c - d.c_lo] = gh[g].first[c] >= 0 ? gh[g].first[c] - r0 : -1;
            end[c - d.c_lo] = gh[g].first[c] >= 0 ? gh[g].end[c] - r0 : -1;
          }
          if (colate_set_genome(d.h, g, r1 - r0, first.data(), end.data(), gh[g].bp.data() + r0, gh[g].aaf.data() + r0, gh[g].daf.data() + r0,
                                gh[g].al.data() + r0, 0)) {
            d.fail("colate_set_genome");
            return;
          }
        }
      }
      const std::vector<std::string>* masks[2] = {&f_tmask, &f_rmask};
      for (int g = 0; g < 2; g++) {
        if (masks[g]->empty() || nc == 0) continue;
        std::vector<uint32_t> bits(((size_t)d.site_off[nc] + 31) / 32 + 1, 0);
        for (int c = 0; c < nc; c++) {
          if (colate_mask_bits_from_fasta((*masks[g])[d.c_lo + c].c_str(), d.site_off[c + 1] - d.site_off[c], d.pos.data() + d.site_off[c],
                                          d.site_off[c], bits.data())) {
            d.fail("mask");
            return;
          }
        }
        if (colate_set_mask(d.h, g, bits.data(), 0)) { d.fail("colate_set_mask"); return; }
      }
      std::vector<int64_t> used(nc + 1);
      std::vector<int32_t> blocks(nc + 1);
      if (colate_stage1_flags(d.h, 0, 1, used.data(), blocks.data())) { d.fail("colate_stage1_flags"); return; }
      d.n_used = 0; d.n_blocks = 0;
      for (int c = 0; c < nc; c++) { d.n_used += used[c]; d.n_blocks += blocks[c]; }
    });
    if (!all_ok(devs)) exit(1);
    for (auto& g : gh) g = GenomeHost();
    ph.tick("sites, genomes, masks, flag pass");
    // ---- the exchange: every device's offset into the reference's generator stream and its first genomic block
    for (int g = 1; g < G; g++) {
      devs[g].used_base = devs[g - 1].used_base + devs[g - 1].n_used;
      devs[g].block_base = devs[g - 1].block_base + devs[g - 1].n_blocks;
    }
    num_blocks = devs[G - 1].block_base + devs[G - 1].n_blocks;
    if (num_blocks > COLATE_MAX_BLOCKS) { std::cerr << "more than 500 genomic blocks (the reference overruns its arrays, coal.cpp:3140)" << std::endl; return 1; }
    on_every_device(devs, [&](Dev& d) {
      if (colate_stage1_sample(d.h, mt, d.used_base, d.block_base, block_stats.data() + (size_t)d.block_base * 4 * COLATE_NUM_AGE_BINS, nullptr,
                               d.mt_after)) {
        d.fail("colate_stage1_sample");
        return;
      }
      d.extra_words = colate_last_stage1_extra_words(d.h);
    });
    if (!all_ok(devs)) return 1;
    if (G > 1)
      for (auto& d : devs)
        if (d.extra_words) {
          std::cerr << "This input has rows whose samples the reference redraws (age interval beyond the age grid, coal.cpp:2279-2294): "
                       "the generator offsets of the later chromosomes depend on them. Run it with one device." << std::endl;
          return 1;
        }
    memcpy(mt, devs[G - 1].mt_after, sizeof mt);   // the state after the last used row lives on the last device
    std::cerr << "Number of blocks: " << num_blocks << std::endl;
    ph.tick("stage i");
    if (R > 0) {
      weights.resize((size_t)R * num_blocks);
      colate_draw_block_weights(mt, R, num_blocks, weights.data());
    }
  }

  // epochs, coal.cpp:3503-3646
  std::vector<double> epochs(4096), rates_init(4096, 1.0 / 20000.0);
  int ep_null = 0, E;
  if (options.count("coal")) {
    E = colate_epochs_from_coal_file(options.get("coal").c_str(), age, epochs.data(), rates_init.data(), 4096);
    if (E < 0) return die("--coal");
    for (int e = 0; e < E; e++) std::cerr << rates_init[e] << " ";
    std::cerr << std::endl;
  } else {
    if (!options.count("bins")) { std::cerr << "Error: --bins or --coal is required." << std::endl; return 1; }
    E = colate_epochs_from_bins(options.get("bins").c_str(), age, ypg, epochs.data(), 4096, &ep_null);
    if (E < 0) { std::cerr << colate_last_error() << std::endl; exit(1); }
  }
  if (!wait_for_devices()) return 1;   // (the .colate_mat cache path gets here without having touched the devices)
  std::cerr << "Maximising likelihood using EM.. " << std::endl;
  std::vector<double> rates((size_t)std::max(R, 1) * E, 0.0), ll(std::max(R, 1));
  std::vector<int32_t> iters(std::max(R, 1), 0);
  if (R > 0) {
    // replicates -> devices round-robin; stage ii (block bootstrap, coal.cpp:3344-3451) and stage iii (EM, 3675-3827)
    on_every_device(devs, [&](Dev& d) {
      const int g = (int)(&d - devs.data());
      std::vector<int> mine;
      for (int r = g; r < R; r += G) mine.push_back(r);
      const int n = (int)mine.size();
      if (n == 0) return;
      std::vector<double> cn((size_t)n * 2 * COLATE_NUM_AGE_BINS), rt((size_t)n * E), l2(n);
      std::vector<int32_t> it(n);
      const double* cn_in = nullptr;
      if (from_cache) {
        if (colate_set_age_bins(d.h, cached_age_bin)) { d.fail("colate_set_age_bins"); return; }
        for (int k = 0; k < n; k++) memcpy(cn.data() + (size_t)k * 2 * COLATE_NUM_AGE_BINS, counts.data() + (size_t)mine[k] * 2 * COLATE_NUM_AGE_BINS, 2 * COLATE_NUM_AGE_BINS * 8);
        cn_in = cn.data();
      } else {
        std::vector<int32_t> w((size_t)n * num_blocks);
        for (int k = 0; k < n; k++) memcpy(w.data() + (size_t)k * num_blocks, weights.data() + (size_t)mine[k] * num_blocks, (size_t)num_blocks * 4);
        if (colate_stage2_bootstrap(d.h, n, num_blocks, w.data(), block_stats.data(), age, counts_front_end ? cn.data() : nullptr)) { d.fail("colate_stage2_bootstrap"); return; }
        for (int k = 0; k < n && counts_front_end; k++)
          memcpy(counts.data() + (size_t)mine[k] * 2 * COLATE_NUM_AGE_BINS, cn.data() + (size_t)k * 2 * COLATE_NUM_AGE_BINS, 2 * COLATE_NUM_AGE_BINS * 8);
      }
      if (colate_stage3_em(d.h, n, E, epochs.data(), rates_init.data(), cn_in, 100000, rt.data(), it.data(), l2.data())) { d.fail("colate_stage3_em"); return; }
      for (int k = 0; k < n; k++) {
        memcpy(rates.data() + (size_t)mine[k] * E, rt.data() + (size_t)k * E, (size_t)E * 8);
        iters[mine[k]] = it[k];
        ll[mine[k]] = l2[k];
      }
    });
    if (!all_ok(devs)) return 1;
    for (int i = 0; i < R; i++) std::cerr << "Bootstrap " << i + 1 << ": Total iterations " << iters[i] << std::endl;
  }
  if (counts_front_end && !from_cache) {   // every front-end but tmp/tmp keeps its bootstrap counts (coal.cpp:3336-3343, 3453-3465)
    double age_bin[COLATE_NUM_AGE_BINS];
    colate_age_bins(age_bin);
    if (colate_write_colate_mat((out + ".colate_mat").c_str(), R, age_bin, counts.data())) return die("write .colate_mat");
  }
  // .coal first: for ancient samples it zeroes rates[0..ep_null] (coal.cpp:3832-3834); the fp64 side
  // output then holds exactly the values the text was printed from
  ph.tick("stage ii + iii");
  if (colate_write_coal((out + ".coal").c_str(), R, E, epochs.data(), rates.data(), is_ancient, ep_null)) return die("write .coal");
  if (colate_write_bin((out + ".bin").c_str(), R, E, epochs.data(), rates.data(), iters.data())) return die("write .bin");
  for (auto& d : devs) colate_destroy(d.h);

  rusage usage;
  getrusage(RUSAGE_SELF, &usage);
  std::cerr << "CPU Time spent: " << usage.ru_utime.tv_sec << "." << std::setfill('0') << std::setw(6) << usage.ru_utime.tv_usec
            << "s; Max Memory usage: " << usage.ru_maxrss / 1000.0 << "Mb." << std::endl;
  std::cerr << "---------------------------------------------------------" << std::endl << std::endl;
  return 0;
}

// ---- --pairs: a cohort of target / reference runs in one job ------------------------------------------------------------
// Every line is the run `Colate --mode mut --target_tmp T --reference_tmp R -o OUT [--target_age ..] ...` (or its --target_bam /
// --reference_bam or --target_bcf / --reference_bcf form) with the shared flags, and its .coal / .bin (and, for BAM and BCF lines,
// .colate_mat) are those of that run.  The .mut text is parsed once per device, --ref_genome is read once and uploaded once per
// device, every genome (an input under one mask, a BCF prefix once per role) fills a slot of its own, every input file is decoded
// once per device (further slots of it are device copies, colate_copy_genome), all pairs consume prefixes of the one --seed
// generator stream (colate_set_stream_cache), and the EM of all pairs' replicates runs on their mixed epoch grids in one launch
// (colate_stage3_em_grids).
enum InputKind { kTmp = 0, kBam = 1, kBcf = 2 };

struct PairLine {
  int line = 0;
  int kind = kTmp;
  std::string input[2], out, age[2], mask[2];
  bool has_age[2] = {false, false};
  int genome[2] = {-1, -1};   // index into the job's genome list
  bool cached = false;        // <out>.colate_mat exists: the reference's stale-cache path
  // results
  std::string err;
  int num_blocks = 0, E = 0, ep_null = 0, grid = -1;
  int64_t n_used = 0;
  double age_gen = 0.0;
  std::vector<double> epochs, rates_init, counts, rates, ll;
  std::vector<int32_t> iters;
};

// one slot's content: an input file (a .colate.in, a BAM, a BCF / VCF prefix) under a mask; a BCF prefix per role (its rows are
// resolved by role), a BAM or a .colate.in for both roles alike (role 0)
struct GenomeKey {
  int kind = kTmp;
  std::string input;
  int role = 0;
  std::string mask;
  bool operator<(const GenomeKey& o) const { return std::tie(kind, input, role, mask) < std::tie(o.kind, o.input, o.role, o.mask); }
};

// the shared flags the pairs-file check needs
struct PairsFlags {
  bool has_chr = false, ref_genome = false, strandfilter = false;
  std::vector<std::string> name_chr;
};

// The pairs file, checked completely before any device is touched.  false: the message (naming the line) is on stderr.
bool read_pairs_file(const std::string& path, const PairsFlags& fl, std::vector<PairLine>& pl, std::vector<GenomeKey>& genomes)
{
  std::ifstream is(path);
  if (is.fail()) { std::cerr << "Error: cannot open the pairs file " << path << std::endl; return false; }
  std::map<GenomeKey, int> gidx;
  std::map<std::string, int> out_line;
  std::string text;
  int ln = 0;
  auto bad = [&](const std::string& what) { std::cerr << "Error in pairs file " << path << ", line " << ln << ": " << what << std::endl; return false; };
  // an input field: <file.colate.in>, or target_bam= / target_bcf= (field 0), reference_bam= / reference_bcf= (field 1)
  static const char* kInputKeys[2][2] = {{"target_bam=", "target_bcf="}, {"reference_bam=", "reference_bcf="}};
  auto input_key = [](const std::string& f, int role, int* kind) {
    for (int k = 0; k < 2; k++)
      if (f.rfind(kInputKeys[role][k], 0) == 0) { *kind = k == 0 ? kBam : kBcf; return (int)strlen(kInputKeys[role][k]); }
    return 0;
  };
  static const char* kKindName[3] = {".colate.in", "bam", "bcf"};
  while (std::getline(is, text)) {
    ln++;
    std::stringstream ss(text);
    std::vector<std::string> f;
    std::string tok;
    while (ss >> tok) f.push_back(tok);
    if (f.empty() || f[0][0] == '#') continue;
    if (f.size() < 3) return bad("expected <target_tmp> <reference_tmp> <output_prefix> [key=value ...], found " + std::to_string(f.size()) + " field(s)");
    PairLine p;
    p.line = ln;
    int kinds[2] = {kTmp, kTmp};
    for (int g = 0; g < 2; g++) {
      int k = kTmp;
      if (input_key(f[g], 1 - g, &k))
        return bad("'" + f[g].substr(0, f[g].find('=') + 1) + "' in field " + std::to_string(g + 1) + " (the first field is the target, the second the reference)");
      const int n = input_key(f[g], g, &k);
      if (n && n == (int)f[g].size()) return bad("'" + f[g] + "' is not of the form key=value");
      kinds[g] = k;
      p.input[g] = f[g].substr(n);
    }
    if (kinds[0] != kinds[1])
      return bad(std::string("a ") + kKindName[kinds[0]] + " target with a " + kKindName[kinds[1]] +
                 " reference (the reference's mixed front-ends are not supported: both inputs are .colate.in files, both target_bam= / "
                 "reference_bam=, or both target_bcf= / reference_bcf=)");
    p.kind = kinds[0];
    p.out = f[2];
    std::set<std::string> seen;
    for (size_t k = 3; k < f.size(); k++) {
      const size_t eq = f[k].find('=');
      if (eq == std::string::npos || eq == 0 || eq + 1 == f[k].size()) return bad("'" + f[k] + "' is not of the form key=value");
      const std::string key = f[k].substr(0, eq), val = f[k].substr(eq + 1);
      if (!seen.insert(key).second) return bad("'" + key + "' is given twice");
      if (key == "target_age") { p.age[0] = val; p.has_age[0] = true; }
      else if (key == "reference_age") { p.age[1] = val; p.has_age[1] = true; }
      else if (key == "target_mask") p.mask[0] = val;
      else if (key == "reference_mask") p.mask[1] = val;
      else if (key == "target_bam" || key == "target_bcf" || key == "reference_bam" || key == "reference_bcf")
        return bad("'" + key + "=' goes in field " + (key[0] == 't' ? "1" : "2") + " of the line");
      else
        return bad("unknown key '" + key + "' (known: target_age, reference_age, target_mask, reference_mask; target_bam, target_bcf in field 1, "
                   "reference_bam, reference_bcf in field 2)");
    }
    auto dup = out_line.find(p.out);
    if (dup != out_line.end()) return bad("output prefix " + p.out + " is already used on line " + std::to_string(dup->second));
    out_line[p.out] = ln;
    if (p.kind == kBam) {
      if (fl.strandfilter) return bad("--strandfilter is not supported with BAM inputs (its read filter is not restated)");
      if (!fl.ref_genome) return bad("BAM inputs need --ref_genome");
    }
    if (p.kind == kBcf && !fl.has_chr) return bad("BCF inputs need --chr (one <prefix>_chr<c>.bcf file per chromosome)");
    for (int g = 0; g < 2; g++) {
      const std::vector<std::string> files = p.kind == kBcf ? genotype_input(p.input[g], fl.name_chr).files : std::vector<std::string>{p.input[g]};
      for (auto& file : files) {
        FILE* fp = fopen(file.c_str(), "rb");
        if (!fp) return bad("cannot read " + file);
        fclose(fp);
      }
      const GenomeKey key{p.kind, p.input[g], p.kind == kBcf ? g : 0, p.mask[g]};
      auto it = gidx.find(key);
      if (it == gidx.end()) {
        if ((int)genomes.size() == COLATE_MAX_GENOMES)
          return bad("more than " + std::to_string(COLATE_MAX_GENOMES) +
                     " distinct genomes ((input, mask) combinations; a BCF prefix once per role) in one job");
        it = gidx.emplace(key, (int)genomes.size()).first;
        genomes.push_back(key);
      }
      p.genome[g] = it->second;
    }
    p.cached = file_exists(p.out + ".colate_mat");
    pl.push_back(p);
  }
  if (pl.empty()) { std::cerr << "Error: the pairs file " << path << " lists no pair" << std::endl; return false; }
  return true;
}

int run_cohort(const Options& options)
{
  const std::string pairs_path = options.get("pairs");
  for (const char* k : {"target_tmp", "reference_tmp", "output", "target_age", "reference_age", "target_mask", "reference_mask", "target_bcf",
                        "reference_bcf", "target_bam", "reference_bam", "device"})
    if (options.count(k)) {
      std::cerr << "Error: --" << (strcmp(k, "output") ? k : "output/-o") << " cannot be combined with --pairs (give it per line of the pairs file"
                << (strcmp(k, "device") ? "" : "; use --devices") << ")" << std::endl;
      return 1;
    }
  if (!options.count("mut")) { std::cerr << "Error: --pairs needs --mut" << std::endl; return 1; }
  if (!options.count("seed")) { std::cerr << "Error: --pairs needs --seed (all pairs share the generator stream of that seed)" << std::endl; return 1; }
  if (!options.count("bins") && !options.count("coal")) { std::cerr << "Error: --bins or --coal is required." << std::endl; return 1; }
  // file lists, coal.cpp:3290-3316
  std::vector<std::string> name_chr, f_mut;
  if (options.count("chr")) {
    std::ifstream is(options.get("chr"));
    if (is.fail()) std::cerr << "Error while opening file " << options.get("chr") << std::endl;
    std::string line;
    while (std::getline(is, line)) { name_chr.push_back(line); f_mut.push_back(options.get("mut") + "_chr" + line + ".mut"); }
  } else {
    name_chr.push_back("");
    f_mut.push_back(options.get("mut"));
  }
  PairsFlags fl;
  fl.has_chr = options.count("chr");
  fl.ref_genome = options.count("ref_genome");
  fl.strandfilter = options.count("strandfilter");
  fl.name_chr = name_chr;
  std::vector<PairLine> pl;
  std::vector<GenomeKey> genomes;
  if (!read_pairs_file(pairs_path, fl, pl, genomes)) return 1;
  bool any_bam = false, live_ref = false;   // live_ref: some pair to be computed reads --ref_genome
  for (auto& p : pl) {
    any_bam = any_bam || p.kind == kBam;
    if (!p.cached && (p.kind == kBam || (p.kind == kBcf && fl.ref_genome))) live_ref = true;
  }
  int filters[3];
  if (!parse_filters(options, filters) && any_bam) { std::cerr << "Error: --filters takes three integers: mapq,length,mismatches" << std::endl; return 1; }

  const int seed = atoi(options.get("seed").c_str());
  int R = 1;
  if (options.count("num_bootstraps")) R = atoi(options.get("num_bootstraps").c_str());
  else if (options.count("num_bootstrap")) R = atoi(options.get("num_bootstrap").c_str());
  if (R < 0) R = 0;
  const bool has_ypg = options.count("years_per_gen");
  const float ypg_flag = has_ypg ? strtof(options.get("years_per_gen").c_str(), nullptr) : 0.0f;
  std::vector<int> dev_ids;
  {
    std::stringstream ss(options.count("devices") ? options.get("devices") : "0");
    std::string tok;
    while (std::getline(ss, tok, ',')) if (!tok.empty()) dev_ids.push_back(atoi(tok.c_str()));
    if (dev_ids.empty()) dev_ids.push_back(0);
  }
  const int G = (int)dev_ids.size();
  std::cerr << "Cohort: " << pl.size() << " pairs, " << genomes.size() << " genomes, " << G << " device(s)" << std::endl;

  const int n_chr = (int)name_chr.size();
  {
    std::set<std::string> uniq(name_chr.begin(), name_chr.end());
    if ((int)uniq.size() != n_chr) { std::cerr << "Duplicate chromosome names in --chr" << std::endl; return 1; }
  }
  auto mask_file = [&](const std::string& prefix, int c) { return options.count("chr") ? prefix + "_chr" + name_chr[c] + ".fa" : prefix; };
  std::vector<const char*> names;
  for (auto& s : name_chr) names.push_back(s.c_str());
  bool any_live = false, any_mask = false;
  for (auto& p : pl)
    if (!p.cached) { any_live = true; any_mask = any_mask || !p.mask[0].empty() || !p.mask[1].empty(); }
  // the .mut text, read once for all devices: parsed on the GPU, or by the host reader (zlib) if a file only exists as .gz
  std::vector<std::vector<char>> texts(n_chr);
  bool all_plain = !options.count("host_parse");
  struct SitesHost { std::vector<int64_t> off; std::vector<int32_t> pos; std::vector<float> ab, ae; std::vector<uint32_t> meta; } sh;
  if (any_live) {
    for (int c = 0; c < n_chr && all_plain; c++) {
      FILE* f = fopen(f_mut[c].c_str(), "rb");
      if (!f) { all_plain = false; break; }
      fseek(f, 0, SEEK_END);
      const long sz = ftell(f);
      fseek(f, 0, SEEK_SET);
      texts[c].resize((size_t)std::max(sz, 0L));
      if (sz > 0 && fread(texts[c].data(), 1, (size_t)sz, f) != (size_t)sz) all_plain = false;
      fclose(f);
    }
    if (!all_plain) {
      sh.off.assign(n_chr + 1, 0);
      for (int c = 0; c < n_chr; c++) {
        const int64_t n = colate_read_mut(f_mut[c].c_str(), 0, nullptr, nullptr, nullptr, nullptr);
        if (n < 0) { std::cerr << colate_last_error() << std::endl; return 1; }
        const size_t o = sh.pos.size();
        sh.pos.resize(o + n); sh.ab.resize(o + n); sh.ae.resize(o + n); sh.meta.resize(o + n);
        if (colate_read_mut(f_mut[c].c_str(), n, sh.pos.data() + o, sh.ab.data() + o, sh.ae.data() + o, sh.meta.data() + o) < 0) {
          std::cerr << colate_last_error() << std::endl;
          return 1;
        }
        sh.off[c + 1] = (int64_t)sh.pos.size();
      }
    }
  }
  RefGenome refg;   // --ref_genome, read once for all devices (fasta::Read, data.cpp:213-237)
  if (live_ref && !refg.read(options, name_chr)) return 1;
  // the epoch grid of an age, coal.cpp:3503-3646
  auto grid_of_age = [&](PairLine& p, double ypg) -> bool {
    p.epochs.assign(4096, 0.0);
    p.rates_init.assign(4096, 1.0 / 20000.0);
    p.ep_null = 0;
    if (options.count("coal")) p.E = colate_epochs_from_coal_file(options.get("coal").c_str(), p.age_gen, p.epochs.data(), p.rates_init.data(), 4096);
    else p.E = colate_epochs_from_bins(options.get("bins").c_str(), p.age_gen, ypg, p.epochs.data(), 4096, &p.ep_null);
    if (p.E < 0) { p.err = std::string(options.count("coal") ? "--coal" : "--bins") + ": " + colate_last_error(); return false; }
    p.epochs.resize(p.E);
    p.rates_init.resize(p.E);
    return true;
  };
  uint32_t mt0[COLATE_MT_WORDS];
  colate_mt_seed((uint32_t)seed, mt0);
  constexpr int C2 = 2 * COLATE_NUM_AGE_BINS;
  constexpr int kEmBatch = 2048;   // replicates per EM launch
  std::vector<std::string> dev_err(G), dev_summary(G);
  std::vector<int64_t> n_bam(G, 0), n_bcf(G, 0);   // per device: BAM files piled, BCF / VCF files decoded

  // one host thread per device; pairs are dealt round-robin in file order
  auto work = [&](int g) {
    std::vector<PairLine*> mine;
    for (size_t k = g; k < pl.size(); k += G) mine.push_back(&pl[k]);
    if (mine.empty()) return;
    colate_handle* h = nullptr;
    auto dev_fail = [&](const std::string& what) {
      dev_err[g] = "device " + std::to_string(dev_ids[g]) + ": " + what + ": " + colate_last_error();
      for (PairLine* p : mine) if (p->err.empty()) p->err = dev_err[g];
    };
    if (colate_create(dev_ids[g], &h)) { dev_fail("colate_create"); return; }
    struct Destroy { colate_handle* h; ~Destroy() { colate_destroy(h); } } destroy{h};
    bool live = false, masked = false;
    for (PairLine* p : mine) if (!p->cached) { live = true; masked = masked || !p->mask[0].empty() || !p->mask[1].empty(); }
    if (live) {
      // sites (coal.cpp:2148-2176), then every genome this device needs, decoded into its own slot and masked there
      std::vector<int64_t> site_off(n_chr + 1, 0);
      std::vector<int32_t> pos;
      if (all_plain) {
        int64_t bytes = 0;
        for (auto& t : texts) bytes += (int64_t)t.size();
        if (colate_ingest_begin(h, n_chr, bytes / 20 + n_chr)) { dev_fail("colate_ingest_begin"); return; }
        for (int c = 0; c < n_chr; c++) {
          const int64_t n = colate_ingest_mut_text(h, texts[c].data(), (int64_t)texts[c].size(), 0);
          if (n < 0) { dev_fail("colate_ingest_mut_text"); return; }
          site_off[c + 1] = site_off[c] + n;
        }
        if (colate_ingest_end(h)) { dev_fail("colate_ingest_end"); return; }
        if (masked) {
          pos.resize((size_t)site_off[n_chr]);
          if (colate_ingest_fetch(h, 0, site_off[n_chr], pos.data(), nullptr, nullptr, nullptr)) { dev_fail("colate_ingest_fetch"); return; }
        }
      } else {
        site_off = sh.off;
        if (colate_set_sites(h, n_chr, sh.off.data(), sh.pos.data(), sh.ab.data(), sh.ae.data(), sh.meta.data(), 0)) { dev_fail("colate_set_sites"); return; }
        pos = sh.pos;
      }
      // --ref_genome once per device, where a pair of this device reads it
      bool dev_ref = false;
      for (PairLine* p : mine) dev_ref = dev_ref || (!p->cached && (p->kind == kBam || (p->kind == kBcf && fl.ref_genome)));
      if (dev_ref && colate_set_ref_genome(h, n_chr, (const uint8_t* const*)refg.seq.data(), refg.len.data())) { dev_fail("colate_set_ref_genome"); return; }
      std::map<int, int> slot_of;     // genome -> slot on this device, in the order the pairs first use them
      std::vector<int> order;
      for (PairLine* p : mine) {
        if (p->cached) continue;
        for (int k = 0; k < 2; k++)
          if (!slot_of.count(p->genome[k])) { slot_of[p->genome[k]] = (int)order.size(); order.push_back(p->genome[k]); }
      }
      std::map<int, std::string> genome_err;
      // BAM and BCF inputs: decoded once per device (both roles of a BCF prefix from one decode); the input's further slots (other
      // masks) are device copies of its first slot of the same role.  first[(input, role)] = that slot, or its error.
      std::map<std::pair<std::string, int>, int> first;
      std::map<std::string, std::string> input_err;
      for (const int gi : order) {
        const GenomeKey& gk = genomes[gi];
        const int slot = slot_of[gi];
        const std::string ik = std::to_string(gk.kind) + ":" + gk.input;   // the input file(s) of this genome
        if (gk.kind == kTmp) {
          std::vector<char> image;
          FILE* f = fopen(gk.input.c_str(), "rb");
          if (!f) { genome_err[gi] = "cannot read " + gk.input; continue; }
          fseek(f, 0, SEEK_END);
          const long sz = ftell(f);
          fseek(f, 0, SEEK_SET);
          image.resize((size_t)std::max(sz, 0L));
          const bool short_read = sz > 0 && fread(image.data(), 1, (size_t)sz, f) != (size_t)sz;
          fclose(f);
          if (short_read) { genome_err[gi] = "short read on " + gk.input; continue; }
          if (colate_ingest_colate_in(h, slot, image.data(), (int64_t)image.size(), n_chr, names.data(), 0) < 0) {
            genome_err[gi] = gk.input + ": " + colate_last_error();
            continue;
          }
        } else {
          if (!first.count({ik, gk.role}) && !input_err.count(ik)) {
            if (gk.kind == kBam) {
              n_bam[g]++;
              if (colate_pileup_bam(h, slot, gk.input.c_str(), n_chr, names.data(), nullptr, nullptr, filters[0], filters[1], filters[2], 0, nullptr))
                input_err[ik] = gk.input + ": " + colate_last_error();
              else
                first[{ik, 0}] = slot;
            } else {
              int rs[2] = {-1, -1};   // the first slot of each role of this prefix on this device
              for (const int gj : order)
                if (genomes[gj].kind == kBcf && genomes[gj].input == gk.input && rs[genomes[gj].role] < 0) rs[genomes[gj].role] = slot_of[gj];
              const GenotypeInput in = genotype_input(gk.input, name_chr);
              std::vector<const char*> fp;
              for (auto& x : in.files) fp.push_back(x.c_str());
              n_bcf[g] += (int64_t)in.files.size();
              if (in.whole ? colate_rows_from_bcf_genome(h, rs[0], rs[1], n_chr, names.data(), fp[0], fl.ref_genome ? 1 : 0, 0)
                           : colate_rows_from_bcf_roles(h, rs[0], rs[1], n_chr, names.data(), fp.data(), fl.ref_genome ? 1 : 0, 0))
                input_err[ik] = gk.input + ": " + colate_last_error();
              else
                for (int r = 0; r < 2; r++) if (rs[r] >= 0) first[{ik, r}] = rs[r];
            }
          }
          if (input_err.count(ik)) { genome_err[gi] = input_err[ik]; continue; }
          const int src = first[{ik, gk.role}];
          if (src != slot && colate_copy_genome(h, slot, src)) { genome_err[gi] = gk.input + ": " + colate_last_error(); continue; }
        }
        if (gk.mask.empty()) continue;
        std::vector<uint32_t> bits(((size_t)site_off[n_chr] + 31) / 32 + 1, 0);
        bool ok = true;
        for (int c = 0; c < n_chr && ok; c++)
          ok = !colate_mask_bits_from_fasta(mask_file(gk.mask, c).c_str(), site_off[c + 1] - site_off[c], pos.data() + site_off[c], site_off[c],
                                            bits.data());
        if (ok) ok = !colate_set_mask(h, slot, bits.data(), 0);
        if (!ok) genome_err[gi] = "mask " + gk.mask + ": " + colate_last_error();
      }
      // stages i-ii per pair (coal.cpp:3317-3451) and its epoch grid
      if (colate_set_stream_cache(h, 1)) { dev_fail("colate_set_stream_cache"); return; }
      for (PairLine* p : mine) {
        if (p->cached) continue;
        for (int k = 0; k < 2 && p->err.empty(); k++)
          if (genome_err.count(p->genome[k])) p->err = genome_err[p->genome[k]];
        if (!p->err.empty()) continue;
        double ypg = 28.0;
        p->age_gen = colate_age_generations(p->has_age[0] ? p->age[0].c_str() : nullptr, p->has_age[1] ? p->age[1].c_str() : nullptr, has_ypg, ypg_flag, &ypg);
        // BAM and BCF lines: raw count weights in stage i, counts / 1e3 from stage ii (as the single-pair run sets it)
        if (colate_set_option(h, "front_end", p->kind == kTmp ? 0 : 1)) { dev_fail("colate_set_option"); return; }
        uint32_t mt[COLATE_MT_WORDS];
        if (colate_stage1(h, slot_of[p->genome[0]], slot_of[p->genome[1]], mt0, &p->num_blocks, nullptr, nullptr, &p->n_used, mt)) {
          p->err = std::string("stage i: ") + colate_last_error();
          continue;
        }
        if (R > 0) {
          std::vector<int32_t> w((size_t)R * p->num_blocks);
          colate_draw_block_weights(mt, R, p->num_blocks, w.data());
          p->counts.assign((size_t)R * C2, 0.0);
          if (colate_stage2_bootstrap(h, R, p->num_blocks, w.data(), nullptr, p->age_gen, p->counts.data())) {
            p->err = std::string("stage ii: ") + colate_last_error();
            continue;
          }
        }
        if (R == 0) p->counts.assign(C2, 0.0);   // the .colate_mat of R = 0 holds the age grid alone
        grid_of_age(*p, ypg);
      }
      colate_set_stream_cache(h, 0);
      if (colate_set_option(h, "front_end", 0)) { dev_fail("colate_set_option"); return; }
      // stage iii: every replicate of every pair on its own grid, kEmBatch replicates per launch (coal.cpp:3675-3827)
      if (R > 0) {
        std::vector<PairLine*> run;
        for (PairLine* p : mine) if (!p->cached && p->err.empty()) run.push_back(p);
        for (size_t b0 = 0; b0 < run.size();) {
          size_t b1 = b0;
          while (b1 < run.size() && (int)(b1 - b0 + 1) * R <= std::max(kEmBatch, R)) b1++;
          std::map<std::vector<double>, int> gidx;   // grids (epochs then initial rates) of this launch
          std::vector<int32_t> grid_E, grid_of;
          std::vector<int64_t> grid_off;
          std::vector<double> ep, init, cn;
          for (size_t k = b0; k < b1; k++) {
            PairLine* p = run[k];
            std::vector<double> key(p->epochs);
            key.insert(key.end(), p->rates_init.begin(), p->rates_init.end());
            auto it = gidx.find(key);
            if (it == gidx.end()) {
              it = gidx.emplace(key, (int)grid_E.size()).first;
              grid_E.push_back(p->E);
              grid_off.push_back((int64_t)ep.size());
              ep.insert(ep.end(), p->epochs.begin(), p->epochs.end());
              init.insert(init.end(), p->rates_init.begin(), p->rates_init.end());
            }
            for (int r = 0; r < R; r++) grid_of.push_back(it->second);
            cn.insert(cn.end(), p->counts.begin(), p->counts.end());
          }
          const int n = (int)grid_of.size();
          const int E_max = *std::max_element(grid_E.begin(), grid_E.end());
          std::vector<double> rt((size_t)n * E_max), l2(n);
          std::vector<int32_t> itv(n);
          const bool ok = !colate_stage3_em_grids(h, n, grid_of.data(), (int)grid_E.size(), grid_E.data(), grid_off.data(), ep.data(), init.data(),
                                                  cn.data(), 100000, rt.data(), itv.data(), l2.data());
          for (size_t k = b0; k < b1; k++) {
            PairLine* p = run[k];
            if (!ok) { p->err = std::string("EM: ") + colate_last_error(); continue; }
            const size_t r0 = (k - b0) * R;
            p->rates.assign((size_t)R * p->E, 0.0);
            for (int r = 0; r < R; r++) memcpy(p->rates.data() + (size_t)r * p->E, rt.data() + (r0 + r) * E_max, (size_t)p->E * 8);
            p->iters.assign(itv.begin() + r0, itv.begin() + r0 + R);
            p->ll.assign(l2.begin() + r0, l2.begin() + r0 + R);
          }
          b0 = b1;
        }
      }
    }
    // pairs with <out>.colate_mat: stages i-ii are skipped and the EM runs on the age grid read back from that file
    // (coal.cpp:3169-3170, 3471-3499), in a launch of their own
    for (PairLine* p : mine) {
      if (!p->cached || !p->err.empty()) continue;
      double ypg = 28.0;
      p->age_gen = colate_age_generations(p->has_age[0] ? p->age[0].c_str() : nullptr, p->has_age[1] ? p->age[1].c_str() : nullptr, has_ypg, ypg_flag, &ypg);
      double cached_age_bin[COLATE_NUM_AGE_BINS];
      p->counts.assign((size_t)std::max(R, 1) * C2, 0.0);
      std::ifstream is(p->out + ".colate_mat");
      for (int b = 0; b < COLATE_NUM_AGE_BINS; b++) is >> cached_age_bin[b];
      for (int i = 0; i < R; i++)
        for (int k = 0; k < C2; k++) is >> p->counts[(size_t)i * C2 + k];
      if (!grid_of_age(*p, ypg) || R == 0) continue;
      p->rates.assign((size_t)R * p->E, 0.0);
      p->iters.assign(R, 0);
      p->ll.assign(R, 0.0);
      if (colate_set_age_bins(h, cached_age_bin) ||
          colate_stage3_em(h, R, p->E, p->epochs.data(), p->rates_init.data(), p->counts.data(), 100000, p->rates.data(), p->iters.data(), p->ll.data()))
        p->err = std::string("EM: ") + colate_last_error();
      if (colate_set_age_bins(h, nullptr)) { dev_fail("colate_set_age_bins"); return; }
    }
    int64_t cnt[4];
    colate_upload_counts(h, cnt);
    char line[256];
    snprintf(line, sizeof line, "device %d (handle %d of %d): BAM files piled %lld, BCF/VCF files decoded %lld, .mut texts parsed %lld (%lld rows), "
             "reference genome uploads %lld (%lld bytes)", dev_ids[g], g + 1, G, (long long)n_bam[g], (long long)n_bcf[g], (long long)cnt[0],
             (long long)cnt[1], (long long)cnt[2], (long long)cnt[3]);
    dev_summary[g] = line;
  };
  {
    std::vector<std::thread> th;
    for (int g = 1; g < G; g++) th.emplace_back(work, g);
    work(0);
    for (auto& t : th) t.join();
  }
  for (auto& e : dev_err) if (!e.empty()) std::cerr << e << std::endl;
  for (auto& x : dev_summary) if (!x.empty()) std::cerr << x << std::endl;
  // outputs in file order; a failed pair writes nothing.  BAM and BCF lines keep their bootstrap counts (coal.cpp:3336-3343,
  // 3453-3465), written first as the single-pair run does; a line from the stale cache leaves its .colate_mat as it is
  double age_bin[COLATE_NUM_AGE_BINS];
  colate_age_bins(age_bin);
  int n_failed = 0;
  for (auto& p : pl) {
    if (p.err.empty() && p.kind != kTmp && !p.cached && colate_write_colate_mat((p.out + ".colate_mat").c_str(), R, age_bin, p.counts.data()))
      p.err = std::string("writing the output: ") + colate_last_error();
    if (p.err.empty() && (colate_write_coal((p.out + ".coal").c_str(), R, p.E, p.epochs.data(), p.rates.data(), p.age_gen > 0.0, p.ep_null) ||
                          colate_write_bin((p.out + ".bin").c_str(), R, p.E, p.epochs.data(), p.rates.data(), p.iters.data())))
      p.err = std::string("writing the output: ") + colate_last_error();
    if (!p.err.empty()) {
      n_failed++;
      std::cerr << "pair on line " << p.line << " (" << p.out << ") FAILED: " << p.err << std::endl;
      continue;
    }
    std::cerr << "pair on line " << p.line << " (" << p.out << "): ";
    if (p.cached) std::cerr << "from " << p.out << ".colate_mat";
    else std::cerr << "blocks " << p.num_blocks << ", used rows " << p.n_used;
    std::cerr << ", iterations";
    for (int32_t it : p.iters) std::cerr << " " << it;
    std::cerr << std::endl;
  }
  if (n_failed) std::cerr << n_failed << " of " << pl.size() << " pairs failed" << std::endl;
  return n_failed ? 1 : 0;
}

// --mode make_tmp --target_bam (maketmp_bam, coal.cpp:2527-2680): the pileup of the BAM file at the .mut rows comes from the
// device (colate_pileup_bam), the .colate.in is written on the host from it (colate_maketmp_pileup)
int run_make_tmp_bam(const Options& options)
{
  std::cerr << options.get("target_bam") << ".." << std::endl;
  if (!bam_args_ok(options, false)) return 1;
  std::vector<std::string> name_chr, f_mut, f_mask;
  if (options.count("chr")) {
    std::ifstream is(options.get("chr"));
    if (is.fail()) std::cerr << "Error while opening file " << options.get("chr") << std::endl;
    std::string line;
    while (std::getline(is, line)) {
      name_chr.push_back(line);
      f_mut.push_back(options.get("mut") + "_chr" + line + ".mut");
      if (options.count("target_mask")) f_mask.push_back(options.get("target_mask") + "_chr" + line + ".fa");
    }
  } else {
    name_chr.push_back("");
    f_mut.push_back(options.get("mut"));
    if (options.count("target_mask")) f_mask.push_back(options.get("target_mask"));
  }
  const int n_chr = (int)name_chr.size();
  {
    std::set<std::string> uniq(name_chr.begin(), name_chr.end());
    if ((int)uniq.size() != n_chr) { std::cerr << "Duplicate chromosome names in --chr" << std::endl; return 1; }
  }
  int filters[3];
  parse_filters(options, filters);
  std::vector<int64_t> off(n_chr + 1, 0);
  std::vector<int32_t> pos;
  std::vector<float> ab, ae;
  std::vector<uint32_t> meta;
  for (int c = 0; c < n_chr; c++) {
    std::cerr << "parsing CHR: " << c + 1 << " / " << n_chr << std::endl;
    const int64_t n = colate_read_mut(f_mut[c].c_str(), 0, nullptr, nullptr, nullptr, nullptr);
    if (n < 0) { std::cerr << colate_last_error() << std::endl; return 1; }
    const size_t o = pos.size();
    pos.resize(o + n); ab.resize(o + n); ae.resize(o + n); meta.resize(o + n);
    if (colate_read_mut(f_mut[c].c_str(), n, pos.data() + o, ab.data() + o, ae.data() + o, meta.data() + o) < 0) {
      std::cerr << colate_last_error() << std::endl;
      return 1;
    }
    off[c + 1] = (int64_t)pos.size();
  }
  RefGenome refg;
  if (!refg.read(options, name_chr)) return 1;
  colate_handle* h = nullptr;
  if (colate_create(options.count("device") ? atoi(options.get("device").c_str()) : 0, &h)) return die("colate_create");
  struct Destroy { colate_handle* h; ~Destroy() { colate_destroy(h); } } destroy{h};
  std::vector<const char*> names, muts, masks;
  for (int c = 0; c < n_chr; c++) {
    names.push_back(name_chr[c].c_str());
    muts.push_back(f_mut[c].c_str());
    if (!f_mask.empty()) masks.push_back(f_mask[c].c_str());
  }
  std::vector<int32_t> counts((size_t)off[n_chr] * 4 + 4);
  if (colate_set_sites(h, n_chr, off.data(), pos.data(), ab.data(), ae.data(), meta.data(), 0)) return die("colate_set_sites");
  if (colate_pileup_bam(h, 0, options.get("target_bam").c_str(), n_chr, names.data(), (const uint8_t* const*)refg.seq.data(), refg.len.data(),
                        filters[0], filters[1], filters[2], 0, counts.data()))
    return die(options.get("target_bam"));
  const std::string out = options.get("output") + ".colate.in";
  if (colate_maketmp_pileup(n_chr, names.data(), muts.data(), counts.data(), off[n_chr], masks.empty() ? nullptr : masks.data(), out.c_str()) < 0) {
    std::cerr << colate_last_error() << std::endl;
    return 1;
  }
  rusage usage;
  getrusage(RUSAGE_SELF, &usage);
  std::cerr << "CPU Time spent: " << usage.ru_utime.tv_sec << "." << std::setfill('0') << std::setw(6) << usage.ru_utime.tv_usec
            << "s; Max Memory usage: " << usage.ru_maxrss / 1000.0 << "Mb." << std::endl;
  std::cerr << "---------------------------------------------------------" << std::endl << std::endl;
  return 0;
}

// --mode make_tmp --target_bcf (maketmp_vcf, coal.cpp:2325-2525): the records of every <prefix>_chr<c>.bcf are decoded on the
// device (colate_decode_bcf), the .colate.in is written on the host from them (colate_maketmp_records)
int run_make_tmp_bcf(const Options& options)
{
  std::cerr << options.get("target_bcf") << ".." << std::endl;
  if (!bcf_args_ok(options, false)) return 1;
  if (!options.count("ref_genome")) { std::cerr << "Option 'ref_genome' has no value" << std::endl; return 1; }   // cxxopts throws in the reference
  std::vector<std::string> name_chr, f_mut, f_ref, f_mask;
  {
    std::ifstream is(options.get("chr"));
    if (is.fail()) { std::cerr << "Error while opening file " << options.get("chr") << std::endl; return 1; }
    std::string line;
    while (std::getline(is, line)) {
      name_chr.push_back(line);
      f_mut.push_back(options.get("mut") + "_chr" + line + ".mut");
      f_ref.push_back(options.get("ref_genome") + "_chr" + line + ".fa");
      if (options.count("target_mask")) f_mask.push_back(options.get("target_mask") + "_chr" + line + ".fa");
    }
  }
  const int n_chr = (int)name_chr.size();
  if (n_chr == 0) { std::cerr << "Error: empty --chr list" << std::endl; return 1; }
  {
    std::set<std::string> uniq(name_chr.begin(), name_chr.end());
    if ((int)uniq.size() != n_chr) { std::cerr << "Duplicate chromosome names in --chr" << std::endl; return 1; }
  }
  const GenotypeInput in = genotype_input(options.get("target_bcf"), name_chr);
  colate_handle* h = nullptr;
  if (colate_create(options.count("device") ? atoi(options.get("device").c_str()) : 0, &h)) return die("colate_create");
  struct Destroy { colate_handle* h; ~Destroy() { colate_destroy(h); } } destroy{h};
  std::vector<int64_t> off(n_chr + 1, 0), rec_first(n_chr, 0), rec_n(n_chr, 0);
  std::vector<int32_t> pos, alt, n_hap(n_chr);
  std::vector<uint8_t> a0, a1, bi;
  if (in.whole) {   // one decode of the whole-genome file, every chromosome's records resident
    std::vector<const char*> nm;
    for (auto& x : name_chr) nm.push_back(x.c_str());
    if (colate_decode_bcf_genome(h, in.files[0].c_str(), n_chr, nm.data(), 0, rec_first.data(), rec_n.data(), n_hap.data())) return die(in.files[0]);
  }
  for (int c = 0; c < n_chr; c++) {
    std::cerr << "parsing CHR: " << c + 1 << " / " << n_chr << std::endl;
    const std::string& f = in.files[in.whole ? 0 : c];
    if (!in.whole && colate_decode_bcf(h, f.c_str(), 0, &rec_n[c], &n_hap[c])) return die(f);
    const int64_t n = rec_n[c];
    const size_t o = pos.size();
    pos.resize(o + n); a0.resize(o + n); a1.resize(o + n); alt.resize(o + n); bi.resize(o + n);
    if (colate_bcf_records(h, rec_first[c], n, pos.data() + o, a0.data() + o, a1.data() + o, alt.data() + o, bi.data() + o)) return die(f);
    off[c + 1] = off[c] + n;
  }
  std::vector<const char*> names, muts, refs, masks;
  for (int c = 0; c < n_chr; c++) {
    names.push_back(name_chr[c].c_str());
    muts.push_back(f_mut[c].c_str());
    refs.push_back(f_ref[c].c_str());
    if (!f_mask.empty()) masks.push_back(f_mask[c].c_str());
  }
  const std::string out = options.get("output") + ".colate.in";
  if (colate_maketmp_records(n_chr, names.data(), muts.data(), off.data(), pos.data(), a0.data(), a1.data(), alt.data(), bi.data(), n_hap.data(),
                             refs.data(), masks.empty() ? nullptr : masks.data(), out.c_str()) < 0) {
    std::cerr << colate_last_error() << std::endl;
    return 1;
  }
  rusage usage;
  getrusage(RUSAGE_SELF, &usage);
  std::cerr << "CPU Time spent: " << usage.ru_utime.tv_sec << "." << std::setfill('0') << std::setw(6) << usage.ru_utime.tv_usec
            << "s; Max Memory usage: " << usage.ru_maxrss / 1000.0 << "Mb." << std::endl;
  std::cerr << "---------------------------------------------------------" << std::endl << std::endl;
  return 0;
}

// ---- --targets: make_tmp for many BAM / BCF / VCF targets in one job --------------------------------------------------------
// Every line is the run `Colate --mode make_tmp --target_bam B | --target_bcf P [--target_mask M] -o OUT` with the shared flags, and
// its OUT.colate.in is that run's, byte for byte.  The .mut text is parsed once (on the GPU), --ref_genome is read and uploaded
// once, every distinct mask becomes per-row bits once; per target what remains is the BGZF inflation of its own file, its device
// decode (and pileup), and the device writer (colate_maketmp_write_pileup / _bcf).
struct TargetLine {
  int line = 0;
  bool bam = false;
  std::string input, out, mask;
  int mask_id = -1;
  int64_t records = -1;
  std::string err;
};

// The targets file, checked completely before any device is touched.  false: the message (naming the line) is on stderr.
bool read_targets_file(const std::string& path, const std::vector<std::string>& name_chr, bool has_chr, std::vector<TargetLine>& tl)
{
  std::ifstream is(path);
  if (is.fail()) { std::cerr << "Error: cannot open the targets file " << path << std::endl; return false; }
  std::map<std::string, int> out_line;
  std::string text;
  int ln = 0;
  auto bad = [&](const std::string& what) { std::cerr << "Error in targets file " << path << ", line " << ln << ": " << what << std::endl; return false; };
  while (std::getline(is, text)) {
    ln++;
    std::stringstream ss(text);
    std::vector<std::string> f;
    std::string tok;
    while (ss >> tok) f.push_back(tok);
    if (f.empty() || f[0][0] == '#') continue;
    if (f.size() < 2 || f.size() > 3)
      return bad("expected (target_bam=<file> | target_bcf=<prefix>) <output_prefix> [target_mask=<prefix>], found " + std::to_string(f.size()) + " field(s)");
    TargetLine t;
    t.line = ln;
    std::set<std::string> seen;
    int n_out = 0;
    for (auto& x : f) {
      const size_t eq = x.find('=');
      if (eq == std::string::npos) { t.out = x; n_out++; continue; }
      if (eq == 0 || eq + 1 == x.size()) return bad("'" + x + "' is not of the form key=value");
      const std::string key = x.substr(0, eq), val = x.substr(eq + 1);
      if (!seen.insert(key).second) return bad("'" + key + "' is given twice");
      if (key == "target_table") return bad("target_table= is not supported with --targets (the table variant of make_tmp runs on the host alone: use --target_table)");
      if (key == "target_bam" || key == "target_bcf") {
        if (!t.input.empty()) return bad("give exactly one of target_bam= and target_bcf=");
        t.bam = key == "target_bam";
        t.input = val;
      } else if (key == "target_mask") t.mask = val;
      else return bad("unknown key '" + key + "' (known: target_bam, target_bcf, target_mask)");
    }
    if (t.input.empty()) return bad("give exactly one of target_bam= and target_bcf=");
    if (n_out != 1) return bad("expected one output prefix, found " + std::to_string(n_out));
    auto dup = out_line.find(t.out);
    if (dup != out_line.end()) return bad("output prefix " + t.out + " is already used on line " + std::to_string(dup->second));
    out_line[t.out] = ln;
    if (t.bam) {
      FILE* fp = fopen(t.input.c_str(), "rb");
      if (!fp) return bad("cannot read " + t.input);
      fclose(fp);
    } else {
      if (!has_chr) return bad("target_bcf needs --chr (one <prefix>_chr<c>.bcf file per chromosome)");
      for (auto& fbcf : genotype_input(t.input, name_chr).files) {
        FILE* fp = fopen(fbcf.c_str(), "rb");
        if (!fp) return bad("cannot read " + fbcf);
        fclose(fp);
      }
    }
    tl.push_back(t);
  }
  if (tl.empty()) { std::cerr << "Error: the targets file " << path << " lists no target" << std::endl; return false; }
  return true;
}

int run_make_tmp_batch(const Options& options)
{
  auto bad = [](const std::string& what) { std::cerr << "Error: " << what << std::endl; return 1; };
  for (const char* k : {"target_bam", "target_bcf", "target_table", "target_mask", "output"})
    if (options.count(k))
      return bad(std::string("--") + (strcmp(k, "output") ? k : "output/-o") + " cannot be combined with --targets (give it per line of the targets file)");
  if (options.count("strandfilter")) return bad("--strandfilter is not supported with BAM inputs (its read filter is not restated)");
  if (!options.count("mut")) return bad("--targets needs --mut");
  if (!options.count("ref_genome")) return bad("--targets needs --ref_genome");
  int filters[3];
  if (!parse_filters(options, filters)) return bad("--filters takes three integers: mapq,length,mismatches");
  const std::string dev = options.count("devices") ? options.get("devices") : "";
  if (dev.find(',') != std::string::npos) return bad("--targets runs on one device (--device <i>): inflating the targets on the host bounds the job");
  const bool has_chr = options.count("chr");
  std::vector<std::string> name_chr, f_mut;
  if (has_chr) {
    std::ifstream is(options.get("chr"));
    if (is.fail()) return bad("cannot open " + options.get("chr"));
    std::string line;
    while (std::getline(is, line)) { name_chr.push_back(line); f_mut.push_back(options.get("mut") + "_chr" + line + ".mut"); }
    if (name_chr.empty()) return bad("empty --chr list");
  } else {
    name_chr.push_back("");
    f_mut.push_back(options.get("mut"));
  }
  const int n_chr = (int)name_chr.size();
  {
    std::set<std::string> uniq(name_chr.begin(), name_chr.end());
    if ((int)uniq.size() != n_chr) return bad("duplicate chromosome names in --chr");
  }
  std::vector<TargetLine> tl;
  if (!read_targets_file(options.get("targets"), name_chr, has_chr, tl)) return 1;
  std::vector<std::string> masks;   // distinct target_mask prefixes
  {
    std::map<std::string, int> mid;
    for (auto& t : tl) {
      if (t.mask.empty()) continue;
      auto it = mid.find(t.mask);
      if (it == mid.end()) { it = mid.emplace(t.mask, (int)masks.size()).first; masks.push_back(t.mask); }
      t.mask_id = it->second;
    }
  }
  Phases ph;
  std::cerr << "---------------------------------------------------------" << std::endl;
  std::cerr << "Calculating Colate tmp input files for " << tl.size() << " targets.." << std::endl;

  // the .mut text, read once: parsed on the GPU, or by the host reader (zlib) if a file only exists as .gz
  std::vector<std::vector<char>> texts(n_chr);
  bool all_plain = !options.count("host_parse");
  for (int c = 0; c < n_chr && all_plain; c++) {
    FILE* f = fopen(f_mut[c].c_str(), "rb");
    if (!f) { all_plain = false; break; }
    fseek(f, 0, SEEK_END);
    const long sz = ftell(f);
    fseek(f, 0, SEEK_SET);
    texts[c].resize((size_t)std::max(sz, 0L));
    if (sz > 0 && fread(texts[c].data(), 1, (size_t)sz, f) != (size_t)sz) all_plain = false;
    fclose(f);
  }
  struct { std::vector<int64_t> off; std::vector<int32_t> pos; std::vector<float> ab, ae; std::vector<uint32_t> meta, words; } sh;
  if (!all_plain) {
    texts.clear();
    sh.off.assign(n_chr + 1, 0);
    for (int c = 0; c < n_chr; c++) {
      const int64_t n = colate_read_mut(f_mut[c].c_str(), 0, nullptr, nullptr, nullptr, nullptr);
      if (n < 0) { std::cerr << colate_last_error() << std::endl; return 1; }
      const size_t o = sh.pos.size();
      sh.pos.resize(o + n); sh.ab.resize(o + n); sh.ae.resize(o + n); sh.meta.resize(o + n); sh.words.resize(o + n);
      if (colate_read_mut(f_mut[c].c_str(), n, sh.pos.data() + o, sh.ab.data() + o, sh.ae.data() + o, sh.meta.data() + o) < 0 ||
          colate_read_mut_words(f_mut[c].c_str(), n, sh.words.data() + o) < 0) {
        std::cerr << colate_last_error() << std::endl;
        return 1;
      }
      sh.off[c + 1] = (int64_t)sh.pos.size();
    }
  }
  ph.tick("read .mut");
  RefGenome refg;
  if (!refg.read(options, name_chr)) return 1;
  ph.tick("read --ref_genome");

  colate_handle* h = nullptr;
  if (colate_create(options.count("device") ? atoi(options.get("device").c_str()) : 0, &h)) return die("colate_create");
  struct Destroy { colate_handle* h; ~Destroy() { colate_destroy(h); } } destroy{h};
  std::vector<int64_t> site_off(n_chr + 1, 0);
  std::vector<int32_t> pos;
  if (all_plain) {
    int64_t bytes = 0;
    for (auto& t : texts) bytes += (int64_t)t.size();
    if (colate_ingest_begin(h, n_chr, bytes / 20 + n_chr)) return die("colate_ingest_begin");
    for (int c = 0; c < n_chr; c++) {
      const int64_t n = colate_ingest_mut_text(h, texts[c].data(), (int64_t)texts[c].size(), 0);
      if (n < 0) return die(f_mut[c]);
      site_off[c + 1] = site_off[c] + n;
    }
    if (colate_ingest_end(h)) return die("colate_ingest_end");
    texts.clear();
    pos.resize((size_t)site_off[n_chr]);
    if (colate_ingest_fetch(h, 0, site_off[n_chr], pos.data(), nullptr, nullptr, nullptr)) return die("colate_ingest_fetch");
  } else {
    site_off = sh.off;
    if (colate_set_sites(h, n_chr, sh.off.data(), sh.pos.data(), sh.ab.data(), sh.ae.data(), sh.meta.data(), 0)) return die("colate_set_sites");
    if (colate_set_maketmp_words(h, sh.words.data(), 0)) return die("colate_set_maketmp_words");
    pos = sh.pos;
  }
  // the device writer walks the rows as the reference's forward-only record cursor does: positions must ascend per chromosome
  for (int c = 0; c < n_chr; c++)
    for (int64_t m = site_off[c] + 1; m < site_off[c + 1]; m++)
      if (pos[m] < pos[m - 1]) {
        std::cerr << "Error: " << f_mut[c] << ": positions of a .mut file are not ascending (the reference's sequential reader needs sorted input)" << std::endl;
        return 1;
      }
  ph.tick("parse .mut");
  if (colate_set_ref_genome(h, n_chr, (const uint8_t* const*)refg.seq.data(), refg.len.data())) return die("colate_set_ref_genome");
  ph.tick("upload --ref_genome");
  // every distinct mask once: make_tmp pass bits per row
  std::vector<std::vector<uint32_t>> mask_bits(masks.size());
  std::vector<std::string> mask_err(masks.size());
  for (size_t k = 0; k < masks.size(); k++) {
    mask_bits[k].assign((size_t)site_off[n_chr] / 32 + 2, 0);
    for (int c = 0; c < n_chr && mask_err[k].empty(); c++) {
      const std::string f = has_chr ? masks[k] + "_chr" + name_chr[c] + ".fa" : masks[k];
      if (colate_maketmp_mask_bits(f.c_str(), site_off[c + 1] - site_off[c], pos.data() + site_off[c], site_off[c], mask_bits[k].data()))
        mask_err[k] = colate_last_error();
    }
  }
  ph.tick("masks");
  std::vector<const char*> names;
  for (auto& s : name_chr) names.push_back(s.c_str());
  for (auto& t : tl) {
    const std::string out = t.out + ".colate.in";
    const uint32_t* mb = t.mask_id >= 0 ? mask_bits[t.mask_id].data() : nullptr;
    if (t.mask_id >= 0 && !mask_err[t.mask_id].empty()) t.err = mask_err[t.mask_id];
    else if (t.bam) {
      if (colate_pileup_bam(h, 0, t.input.c_str(), n_chr, names.data(), nullptr, nullptr, filters[0], filters[1], filters[2], 0, nullptr))
        t.err = t.input + ": " + colate_last_error();
      else if ((t.records = colate_maketmp_write_pileup(h, 0, n_chr, names.data(), mb, out.c_str())) < 0)
        t.err = colate_last_error();
      if (ph.on && t.err.empty()) {
        double b[10], w[4];
        colate_last_bam_timing(h, b);
        colate_last_maketmp_timing(h, w);
        fprintf(stderr, "[timing] line %d bam: inflate %.3f s, walk %.3f s, pileup_bam %.3f s; writer kernels %.3f ms, d2h %.3f ms, write %.3f s\n",
                t.line, b[1], b[2], b[6], w[0], w[1], w[2]);
      }
    } else {
      const GenotypeInput in = genotype_input(t.input, name_chr);
      std::vector<const char*> fp;
      for (auto& f : in.files) fp.push_back(f.c_str());
      t.records = in.whole ? colate_maketmp_write_bcf_genome(h, n_chr, names.data(), fp[0], mb, 0, out.c_str())
                           : colate_maketmp_write_bcf(h, n_chr, names.data(), fp.data(), mb, 0, out.c_str());
      if (t.records < 0) t.err = t.input + ": " + colate_last_error();
      if (ph.on && t.err.empty()) {
        double b[10], w[4];
        colate_last_bcf_timing(h, b);
        colate_last_maketmp_timing(h, w);
        fprintf(stderr, "[timing] line %d bcf: inflate %.3f s, walk %.3f s, decode+write %.3f s; writer kernels %.3f ms, d2h %.3f ms, write %.3f s\n",
                t.line, b[1], b[2], b[6], w[0], w[1], w[2]);
      }
    }
    if (!t.err.empty()) remove(out.c_str());   // a failed line leaves no file, not even an older one
    ph.tick(("target on line " + std::to_string(t.line)).c_str());
  }
  if (ph.on) {
    int64_t cnt[4];
    colate_upload_counts(h, cnt);
    fprintf(stderr, "[timing] .mut texts parsed %lld (%lld rows), reference genome uploads %lld (%lld bytes)\n", (long long)cnt[0], (long long)cnt[1],
            (long long)cnt[2], (long long)cnt[3]);
  }
  int n_failed = 0;
  for (auto& t : tl) {
    if (t.err.empty()) std::cerr << "target on line " << t.line << " (" << t.out << "): " << t.records << " records written" << std::endl;
    else { n_failed++; std::cerr << "target on line " << t.line << " (" << t.out << ") FAILED: " << t.err << std::endl; }
  }
  if (n_failed) std::cerr << n_failed << " of " << tl.size() << " targets failed" << std::endl;
  std::cerr << "---------------------------------------------------------" << std::endl << std::endl;
  return n_failed ? 1 : 0;
}

// --mode make_tmp with --target_table (make_tmp(), coal.cpp:2923-3069 -> maketmp_table, 2682-2808): host-only
int run_make_tmp(const Options& options)
{
  if (options.count("targets")) return run_make_tmp_batch(options);
  if (!options.count("mut") || !options.count("output")) {
    std::cout << "Not enough arguments supplied." << std::endl;
    std::cout << "Needed: mut, ref_genome, output, either of target_bcf or target_bam. Optional: filters, target_mask, strandfilter, anc_genome." << std::endl;
    help();
    std::cout << "Calculate coalescence rates for sample." << std::endl;
    exit(0);
  }
  std::cerr << "---------------------------------------------------------" << std::endl;
  std::cerr << "Calculating Colate tmp input file for ";
  if (options.count("target_bcf")) return run_make_tmp_bcf(options);
  if (options.count("target_bam")) return run_make_tmp_bam(options);
  if (!options.count("target_table")) { std::cerr << std::endl; return 0; }   // the reference does nothing without an input either
  if (!options.count("ref_genome")) { std::cerr << std::endl << "Option 'ref_genome' has no value" << std::endl; return 1; }   // cxxopts throws in the reference
  std::cerr << options.get("target_table") << ".." << std::endl;
  std::vector<std::string> name_chr, f_mut, f_ref, f_mask;
  if (options.count("chr")) {
    std::ifstream is(options.get("chr"));
    if (is.fail()) std::cerr << "Error while opening file " << options.get("chr") << std::endl;
    std::string line;
    while (std::getline(is, line)) {
      name_chr.push_back(line);
      f_mut.push_back(options.get("mut") + "_chr" + line + ".mut");
      f_ref.push_back(options.get("ref_genome") + "_chr" + line + ".fa");
      if (options.count("target_mask")) f_mask.push_back(options.get("target_mask") + "_chr" + line + ".fa");
    }
  } else {
    name_chr.push_back("");
    f_mut.push_back(options.get("mut"));
    f_ref.push_back(options.get("ref_genome"));
    if (options.count("target_mask")) f_mask.push_back(options.get("target_mask"));
  }
  for (size_t c = 0; c < name_chr.size(); c++) {
    std::cerr << "parsing CHR: " << c + 1 << " / " << name_chr.size() << std::endl;
    if (!file_exists(f_ref[c]) && !file_exists(f_ref[c] + ".gz")) {   // fasta::Read exits (data.cpp:220-223); only its presence matters here
      std::cerr << "Error while opening file " << f_ref[c] << "." << std::endl;
      exit(1);
    }
  }
  std::vector<const char*> names, muts, masks;
  for (size_t c = 0; c < name_chr.size(); c++) {
    names.push_back(name_chr[c].c_str());
    muts.push_back(f_mut[c].c_str());
    if (!f_mask.empty()) masks.push_back(f_mask[c].c_str());
  }
  const std::string out = options.get("output") + ".colate.in";
  if (colate_maketmp_table((int)names.size(), names.data(), muts.data(), options.get("target_table").c_str(), masks.empty() ? nullptr : masks.data(), 1,
                           out.c_str()) < 0) {
    std::cerr << colate_last_error() << std::endl;
    exit(1);
  }
  rusage usage;
  getrusage(RUSAGE_SELF, &usage);
  std::cerr << "CPU Time spent: " << usage.ru_utime.tv_sec << "." << std::setfill('0') << std::setw(6) << usage.ru_utime.tv_usec
            << "s; Max Memory usage: " << usage.ru_maxrss / 1000.0 << "Mb." << std::endl;
  std::cerr << "---------------------------------------------------------" << std::endl << std::endl;
  return 0;
}

}  // namespace

int main(int argc, char* argv[])
{
  Options options;
  if (!parse(argc, argv, options)) return 1;
  if (!options.count("mode")) {
    std::cout << "Not enough arguments supplied." << std::endl;
    help();
    return 0;
  }
  const std::string mode = options.get("mode");
  int rc = 0;
  if (mode == "mut") rc = options.count("pairs") ? run_cohort(options) : run_mut(options);
  else if (mode == "make_tmp") rc = run_make_tmp(options);
  else {
    std::cout << "####### error #######" << std::endl;
    std::cout << "Invalid or missing mode." << std::endl;
    std::cout << "This build implements --mode mut (tmp/tmp, bam/bam or bcf/bcf inputs) and --mode make_tmp from a --target_table, a --target_bam "
                 "or a --target_bcf. The reference's other modes (preprocess_mut, calc_depth, print_tmp, CondCoalRates) are out of scope." << std::endl;
  }
  if (options.count("help")) help();
  return rc;
}
