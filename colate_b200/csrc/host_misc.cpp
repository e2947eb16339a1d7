// Host-side pieces of the path that are not kernels: error plumbing, the age grid and the
// exact bin thresholds, the per-row filter, the chromosome seek emulation, ages / epoch
// grid, and the readers / writers of the reference's file formats (SURVEY.md App. B).
#include "internal.h"
#include "exact_sum.cuh"

#include <zlib.h>

#include <algorithm>
#include <cerrno>
#include <cmath>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

namespace colate {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
int fail(int code, const std::string& msg) { g_err = msg; return code; }

// max(0,(int)round(log(x10)*C)+1), coal.cpp:2253/2265/2284; (int) as cvttsd2si
int bin_of_x10_host(double x10)
{
  double r = std::round(std::log(x10) * 10.0);
  int v = (r > -2147483649.0 && r < 2147483648.0) ? (int)r : INT_MIN;
  v = (int)((unsigned)v + 1u);
  return v > 0 ? v : 0;
}

static inline double from_bits(uint64_t b) { double d; memcpy(&d, &b, 8); return d; }
static inline uint64_t to_bits(double d) { uint64_t b; memcpy(&b, &d, 8); return b; }

bool bin_thresholds(double* thr10)
{
  bool monotone = true;
  thr10[0] = 0.0;
  for (int k = 1; k <= NBINS; k++) {
    // positive doubles order like their bit patterns
    uint64_t lo = to_bits(1e-3), hi = to_bits(1e12);   // f(lo) < k <= f(hi)
    while (hi - lo > 1) {
      uint64_t mid = lo + (hi - lo) / 2;
      if (bin_of_x10_host(from_bits(mid)) >= k) hi = mid; else lo = mid;
    }
    thr10[k] = from_bits(hi);
    for (int d = 1; d <= 16; d++) {
      if (bin_of_x10_host(from_bits(hi - d)) >= k) monotone = false;
      if (bin_of_x10_host(from_bits(hi + d)) < k) monotone = false;
    }
  }
  return monotone;
}

bool age_thresholds(double* thrA, double* thrP, uint16_t* lut)
{
  bool monotone = true;
  thrA[0] = 0.0;
  for (int k = 1; k <= NBINS; k++) {
    uint64_t lo = to_bits(1e-4), hi = to_bits(1e11);
    while (hi - lo > 1) {
      uint64_t mid = lo + (hi - lo) / 2;
      if (bin_of_x10_host(10 * from_bits(mid)) >= k) hi = mid; else lo = mid;
    }
    thrA[k] = from_bits(hi);
    for (int d = 1; d <= 16; d++) {
      if (bin_of_x10_host(10 * from_bits(hi - d)) >= k) monotone = false;
      if (bin_of_x10_host(10 * from_bits(hi + d)) < k) monotone = false;
    }
  }
  thrA[NBINS + 1] = HUGE_VAL;
  for (int p = 0; p < 192; p++) thrP[p] = HUGE_VAL;
  for (int k = 0; k <= NBINS; k++) thrP[slot_of_bin(k)] = thrA[k + 1];
  for (int c = 0; c < LUT_N; c++) {
    const double edge = from_bits((uint64_t)(uint32_t)((c + LUT_BASE) << LUT_SHIFT) << 32);
    int k = 0;
    while (k < NBINS && edge >= thrA[k + 1]) k++;
    // at most one threshold inside a cell (a cell is at most a factor 1 + 1/32 wide, a bin e^0.1);
    // bit 15 says whether there is one (then the device compares against thrP[slot]), the first
    // and last cells are clamp targets and always compare
    const double next = from_bits((uint64_t)(uint32_t)((c + 1 + LUT_BASE) << LUT_SHIFT) << 32);
    if (k + 2 <= NBINS && next > thrA[k + 2]) monotone = false;
    const bool inside = (k < NBINS && next > thrA[k + 1]) || c == 0 || c == LUT_N - 1;
    lut[c] = (uint16_t)(slot_of_bin(k) | (inside ? 0x8000 : 0));
  }
  return monotone;
}

// ---- gz/plain file slurp (igzstream semantics: gzopen reads plain files transparently) ----
bool slurp(const std::string& path, std::vector<char>& buf)
{
  gzFile f = gzopen(path.c_str(), "rb");
  if (!f) return false;
  gzbuffer(f, 1 << 20);
  buf.clear();
  size_t cap = 1 << 22;
  buf.resize(cap);
  size_t n = 0;
  for (;;) {
    if (n == cap) { cap *= 2; buf.resize(cap); }
    int got = gzread(f, buf.data() + n, (unsigned)std::min<size_t>(cap - n, 1u << 30));
    if (got < 0) { gzclose(f); return false; }
    if (got == 0) break;
    n += (size_t)got;
  }
  gzclose(f);
  buf.resize(n);
  return true;
}

bool slurp_or_gz(const std::string& path, std::vector<char>& buf)
{
  // Mutations::Read(filename) / fasta::Read: try <path>, then <path>.gz
  FILE* probe = fopen(path.c_str(), "rb");
  if (probe) { fclose(probe); return slurp(path, buf); }
  return slurp(path + ".gz", buf);
}


// ---- .colate.in images in memory -------------------------------------------------------------
// Sequential decode of a record stream {i32 lchrom, chrom, i32 bp, anc, der, i32 AAF, i32 DAF} (coal.cpp:2505-2514),
// the way the reference freads it (coal.cpp:2126-2133): a truncated last record ends the stream.
// bp == nullptr: count only.
int64_t decode_colate_in_host(const char* buf, int64_t sz, const std::vector<std::string>& names, int64_t cap,
                              int32_t* rec_chrom, int32_t* bp, int32_t* aaf, int32_t* daf, uint16_t* alleles)
{
  const int n_chr = (int)names.size();
  int64_t n = 0;
  size_t o = 0;
  int last_id = -1;
  std::string last_name;
  while (o + 4 <= (size_t)sz) {
    int32_t l;
    memcpy(&l, buf + o, 4);
    if (l < 0 || l >= 1024 || o + 4 + (size_t)l + 14 > (size_t)sz) break;  // truncated tail
    if (bp) {
      if (n >= cap) return fail(COLATE_ERR_ARG, "colate_read_colate_in: capacity too small");
      const char* nm = buf + o + 4;
      int id;
      if (last_id >= 0 && last_name.size() == (size_t)l && memcmp(last_name.data(), nm, l) == 0) id = last_id;
      else {
        id = n_chr;
        for (int c = 0; c < n_chr; c++)
          if (names[c].size() == (size_t)l && memcmp(names[c].data(), nm, l) == 0) { id = c; break; }
        last_id = id;
        last_name.assign(nm, l);
      }
      const char* r = nm + l;
      rec_chrom[n] = id;
      memcpy(&bp[n], r, 4);
      alleles[n] = (uint16_t)((unsigned char)r[4] | ((unsigned char)r[5] << 8));
      memcpy(&aaf[n], r + 6, 4);
      memcpy(&daf[n], r + 10, 4);
    }
    n++;
    o += 4 + (size_t)l + 14;
  }
  return n;
}

// Run structure of an image WITHOUT walking it record by record: a run = consecutive records with the same
// {lchrom, chrom} header, hence the same width.  From a record at a known boundary the run's end is located by
// galloping + bisection over "does the header at boundary + j * width equal this run's header".  The probes only
// look at O(log n) records per run, so the result is a HYPOTHESIS: it is exactly the sequential reader's
// segmentation iff every record inside every run carries its run's header (by induction each record then starts
// where the previous one ends) -- which the device decoder checks for all records in parallel (k_decode_colate_in);
// if the check fails the caller falls back to decode_colate_in_host.
int64_t colate_in_runs(const char* buf, int64_t sz, const std::vector<std::string>& names, std::vector<ColateInRun>& runs)
{
  const int n_chr = (int)names.size();
  runs.clear();
  int64_t o = 0, n = 0;
  while (o + 4 <= sz) {
    int32_t l;
    memcpy(&l, buf + o, 4);
    if (l < 0 || l >= 1024 || o + 4 + (int64_t)l + 14 > sz) break;  // truncated tail
    const int64_t w = 18 + (int64_t)l;
    const int hl = 4 + l;
    const int64_t bound = (sz - o) / w;                             // complete records of this width that fit
    auto same = [&](int64_t j) { return memcmp(buf + o + j * w, buf + o, hl) == 0; };
    int64_t good = 0, badj = bound;                                 // header(good) matches; badj: first known mismatch (or the bound)
    for (int64_t j = 1; j < bound; j *= 2) {
      if (same(j)) good = j; else { badj = j; break; }
    }
    while (badj - good > 1) {
      const int64_t mid = good + (badj - good) / 2;
      if (same(mid)) good = mid; else badj = mid;
    }
    int id = n_chr;
    for (int c = 0; c < n_chr; c++)
      if (names[c].size() == (size_t)l && memcmp(names[c].data(), buf + o + 4, l) == 0) { id = c; break; }
    runs.push_back(ColateInRun{o, (int32_t)w, id, good + 1, n});
    n += good + 1;
    o += (good + 1) * w;
  }
  return n;
}

// colate_chr_ranges() on the run-length form
void chr_ranges_runs(int n_chr, const std::vector<ColateInRun>& runs, int64_t* chr_first, int64_t* chr_end)
{
  const int64_t n_rec = runs.empty() ? 0 : runs.back().rec_base + runs.back().n_rec;
  auto chrom_of = [&](int64_t k) {   // run index holding record k
    size_t lo = 0, hi = runs.size();
    while (hi - lo > 1) { size_t mid = (lo + hi) / 2; if (runs[mid].rec_base <= k) lo = mid; else hi = mid; }
    return lo;
  };
  int64_t cur = -1, next = 0;
  for (int c = 0; c < n_chr; c++) {
    bool have = cur >= 0 && runs[chrom_of(cur)].chr_id == c;
    if (!have) {
      // the reader advances record by record until it holds one of chromosome c (or hits the end of the file)
      size_t r = next < n_rec ? chrom_of(next) : runs.size();
      while (r < runs.size() && runs[r].chr_id != c) r++;
      if (r < runs.size()) { cur = std::max(next, runs[r].rec_base); next = cur + 1; have = true; }
      else if (n_rec > 0) { cur = n_rec - 1; next = n_rec; }          // fread failed: it keeps its last record
    }
    if (have) {
      size_t r = chrom_of(cur);
      int64_t e = runs[r].rec_base + runs[r].n_rec;
      while (r + 1 < runs.size() && runs[r + 1].chr_id == c) { r++; e = runs[r].rec_base + runs[r].n_rec; }
      chr_first[c] = cur;
      chr_end[c] = e;
      cur = e - 1;
      next = e;
    } else {
      chr_first[c] = -1;
      chr_end[c] = -1;
    }
  }
}

// one data line of a .mut file, [p, nl) with *nl == '\n' (mutations.cpp:70-250; the columns the path uses)
// std::stoi / std::stof as libstdc++ implements them (__gnu_cxx::__stoa over strtol / strtof): false where they throw
// -- no conversion (invalid_argument), ERANGE or a value outside int (out_of_range).  The text is NUL-terminated
// somewhere behind the field; conversion stops at the field's ';' (or ' ') by itself.
static bool stoi_like(const char* s, int* v)
{
  char* end = nullptr;
  errno = 0;
  const long x = strtol(s, &end, 10);
  if (end == s || errno == ERANGE || x < INT_MIN || x > INT_MAX) return false;
  *v = (int)x;
  return true;
}
static bool stof_like(const char* s, float* v)
{
  char* end = nullptr;
  errno = 0;
  const float x = strtof(s, &end);
  if (end == s || errno == ERANGE) return false;
  *v = x;
  return true;
}

// One data line of a .mut file, [p, nl) with *nl == '\n' and a NUL somewhere behind it, field by field as
// Mutations::Read walks it (mutations.cpp:70-250).  false = the reference does not survive the line: a field it
// converts with std::stoi (snp, pos, dist, tree, every branch index, is_flipped, every frequency column: it prints
// "Error reading following line in mut file" and exits, mutations.cpp:84-88 ...) or std::stof (the two ages: the
// exception is not caught) cannot be converted, or fields are missing (it reads past the end of the line).
bool parse_mut_line_fields(const char* p, const char* nl, int32_t* pos, float* age_begin, float* age_end, uint32_t* meta, int* flipped_out,
                           int* n_branch_out, char* type16 /*[16], may be null*/)
{
  // snp;pos;dist;rs-id;tree;branches;is_not_mapping;is_flipped;age_begin;age_end;type;upstream;downstream;freq...
  const char* f[11];
  const char* q = p;
  int nf = 0;
  f[nf++] = q;
  while (q < nl && nf < 11) { if (*q == ';') f[nf++] = q + 1; q++; }
  if (nf < 10) return false;
  int v = 0, ps = 0, fl = 0;
  if (!stoi_like(f[0], &v) || !stoi_like(f[1], &ps) || !stoi_like(f[2], &v) || !stoi_like(f[4], &v)) return false;
  *pos = ps;
  int nb = 0;
  for (const char* b = f[5]; b < f[6] - 1;) {          // tokens between single spaces (mutations.cpp:144-160)
    while (b < f[6] - 1 && *b == ' ') b++;
    if (b < f[6] - 1) {
      if (!stoi_like(b, &v)) return false;
      nb++;
      while (b < f[6] - 1 && *b != ' ') b++;
    }
  }
  if (!stoi_like(f[7], &fl)) return false;
  const int flipped = fl != 0;
  float ab, ae;
  if (nf < 11 && memchr(f[9], ';', nl - f[9]) == nullptr) return false;   // age_end must end with ';' (mutations.cpp:207-210)
  if (!stof_like(f[8], &ab) || !stof_like(f[9], &ae)) return false;
  *age_begin = ab;
  *age_end = ae;
  char mt[16] = "NA";
  if (nf >= 11) {
    // mutation type runs to the next ';' or the end of the line (mutations.cpp:216-223)
    const char* e = f[10];
    size_t k = 0;
    while (e < nl && *e != ';' && k + 1 < sizeof mt) mt[k++] = *e++;
    mt[k] = 0;
    if (e < nl && *e != ';') { mt[0] = 'N'; mt[1] = 'N'; mt[2] = 0; }  // longer than any valid code
    while (e < nl && *e != ';') e++;
    // upstream; downstream; then frequency columns, each converted with std::stoi (mutations.cpp:224-250)
    if (e < nl && e + 1 < nl) {
      const char* g = e + 1;
      for (int k2 = 0; k2 < 2; k2++) {                 // both must end with ';'
        const char* sc = (const char*)memchr(g, ';', nl - g);
        if (!sc) return false;
        g = sc + 1;
      }
      while (g < nl) {
        if (!stoi_like(g, &v)) return false;
        const char* sc = (const char*)memchr(g, ';', nl - g);
        g = sc ? sc + 1 : nl;
      }
    }
  }
  *meta = colate_site_meta(flipped, nb, ab, ae, mt);
  if (flipped_out) *flipped_out = flipped;
  if (n_branch_out) *n_branch_out = nb;
  if (type16) memcpy(type16, mt, 16);
  return true;
}

bool parse_mut_line_host(const char* p, const char* nl, int32_t* pos, float* age_begin, float* age_end, uint32_t* meta)
{
  return parse_mut_line_fields(p, nl, pos, age_begin, age_end, meta, nullptr, nullptr, nullptr);
}

}  // namespace colate

using namespace colate;

extern "C" {

const char* colate_last_error(void) { return g_err.c_str(); }
const char* colate_version(void) { return "colate_b200 0.1 (sm_100a)"; }

void colate_age_bins(double* age_bin)
{
  double C = 10;
  age_bin[0] = 0.0;
  for (int bin = 0; bin < NBINS - 1; bin++) age_bin[bin + 1] = std::exp(bin / C) / 10.0;
}

int colate_test_bin_thresholds(double* thr10) { return bin_thresholds(thr10) ? 0 : 1; }
double colate_test_add_repeated(double acc, double w, int c) { return exsum::add_repeated(acc, w, c); }
int64_t colate_test_stream_phys(int64_t o, int64_t off) { return stream_phys(o, off); }

uint32_t colate_site_meta(int flipped, int n_branch, float age_begin, float age_end, const char* mutation_type)
{
  if (!(flipped == 0 && n_branch == 1 && age_begin < age_end && age_end >= 0)) return 0;
  const char* slash = strchr(mutation_type, '/');
  size_t n = strlen(mutation_type);
  size_t la = slash ? (size_t)(slash - mutation_type) : n;
  size_t ld = slash ? n - la - 1 : 0;
  if (la != 1 || ld != 1) return 0;  // empty, or not one of the single-letter codes
  char a = mutation_type[0], d = mutation_type[2];
  if (!(a == 'A' || a == 'C' || a == 'G' || a == 'T' || a == '0')) return 0;
  if (!(d == 'A' || d == 'C' || d == 'G' || d == 'T' || d == '1')) return 0;
  return 1u | ((uint32_t)(unsigned char)a << 8) | ((uint32_t)(unsigned char)d << 16);
}

int colate_chr_ranges(int n_chr, int64_t n_rec, const int32_t* rec_chrom, int64_t* chr_first, int64_t* chr_end)
{
  int64_t cur = -1, next = 0;  // cur: record currently held by the reader (-1: none yet)
  for (int c = 0; c < n_chr; c++) {
    while (!(cur >= 0 && rec_chrom[cur] == c)) {
      if (next >= n_rec) break;          // fread fails: the reader keeps its last record
      cur = next++;
    }
    if (cur >= 0 && rec_chrom[cur] == c) {
      int64_t e = cur + 1;
      while (e < n_rec && rec_chrom[e] == c) e++;
      chr_first[c] = cur;
      chr_end[c] = e;
      // whatever part of the run the row loop leaves unread is skipped by the next seek
      cur = e - 1;
      next = e;
    } else {
      chr_first[c] = -1;
      chr_end[c] = -1;
    }
  }
  return 0;
}

double colate_age_generations(const char* target_age, const char* reference_age, int has_years_per_gen,
                              float years_per_gen, double* years_per_gen_out)
{
  // coal.cpp:3105-3118: std::stof of the two strings, float flag for years_per_gen
  double ta = 0, ra = 0;
  if (target_age) ta = strtof(target_age, nullptr);
  if (reference_age) ra = strtof(reference_age, nullptr);
  double ypg = 28.0;
  if (has_years_per_gen) ypg = years_per_gen;
  if (years_per_gen_out) *years_per_gen_out = ypg;
  return std::max(ta, ra) / ypg;
}

int colate_epochs_from_bins(const char* bins, double age, double years_per_gen, double* epochs, int cap, int* ep_null)
{
  // coal.cpp:3553-3630
  const double log_10 = std::log(10);
  double log_age = std::log(age * years_per_gen) / log_10;
  std::string s(bins);
  double v[3];
  size_t i = 0;
  for (int t = 0; t < 3; t++) {
    if (t > 0 && i >= s.size()) return fail(COLATE_ERR_ARG, "Error: epochs format is wrong. Specify x,y,stepsize.");
    std::string tok;
    while (i < s.size() && s[i] != ',') tok += s[i++];
    i++;
    char* end = nullptr;
    v[t] = strtof(tok.c_str(), &end);
    if (end == tok.c_str()) return fail(COLATE_ERR_ARG, "--bins: not a number: '" + tok + "'");
  }
  const double lower = v[0], upper = v[1], step = v[2];
  if (!(step > 0)) return fail(COLATE_ERR_ARG, "--bins: stepsize must be positive");
  int ne = 0;
  *ep_null = 0;
  epochs[ne++] = 0.0;
  if (log_age < lower && age != 0.0) { epochs[ne++] = age; log_age = -1; }
  double boundary = lower;
  while (boundary < upper) {
    if (ne + 3 > cap) return fail(COLATE_ERR_ARG, "--bins: too many epochs");
    if (boundary > log_age && log_age != -1) {
      epochs[ne++] = age;
      if (boundary - log_age < 0.25 * step) boundary += step;
      log_age = -1;
    } else {
      if (log_age != -1) (*ep_null)++;
      epochs[ne++] = std::exp(log_10 * boundary) / years_per_gen;
    }
    boundary += step;
  }
  epochs[ne++] = std::exp(log_10 * upper) / years_per_gen;
  epochs[ne] = std::max(1e8, 10 * epochs[ne - 1]) / years_per_gen;
  ne++;
  return ne;
}

int colate_epochs_from_coal_file(const char* path, double age, double* epochs, double* rates_init, int cap)
{
  // coal.cpp:3508-3549 (epoch line) and 3638-3646 (initial rates)
  std::vector<char> buf;
  if (!slurp(path, buf)) return fail(COLATE_ERR_IO, std::string("cannot read ") + path);
  std::string all(buf.begin(), buf.end());
  size_t l1 = all.find('\n');
  if (l1 == std::string::npos) return fail(COLATE_ERR_IO, "--coal: missing epoch line");
  size_t l2 = all.find('\n', l1 + 1);
  std::string line = all.substr(l1 + 1, (l2 == std::string::npos ? all.size() : l2) - l1 - 1);
  int ne = 0, ep = 0;
  std::string tmp;
  auto push = [&](const std::string& tok) -> bool {
    char* end = nullptr;
    float f = strtof(tok.c_str(), &end);
    if (end == tok.c_str()) return false;
    if (ne + 2 > cap) return false;
    if (ep == 1 && age < f && age != 0.0) { epochs[ne++] = age; ep++; }
    if (ep != 1 || age == 0.0) { epochs[ne++] = f; ep++; }
    return true;
  };
  for (size_t i = 0; i < line.size(); i++) {
    if (line[i] == ' ' || line[i] == '\t') {
      if (!push(tmp)) return fail(COLATE_ERR_IO, "--coal: malformed epoch line");
      tmp.clear();
    } else tmp += line[i];
  }
  if (!tmp.empty() && !push(tmp)) return fail(COLATE_ERR_IO, "--coal: malformed epoch line");
  if (ne < 2 || epochs[0] != 0) return fail(COLATE_ERR_IO, "--coal: first epoch must be 0");
  for (int e = 1; e < ne; e++)
    if (!(epochs[e] > epochs[e - 1])) return fail(COLATE_ERR_IO, "--coal: epochs must increase");
  // `is >> dummy >> dummy` then one rate per epoch
  const char* p = (l2 == std::string::npos) ? "" : all.c_str() + l2 + 1;
  char* end = nullptr;
  for (int k = 0; k < 2; k++) { strtod(p, &end); if (end == p) return fail(COLATE_ERR_IO, "--coal: missing rates"); p = end; }
  for (int e = 0; e < ne; e++) {
    double r = strtod(p, &end);
    if (end == p) return fail(COLATE_ERR_IO, "--coal: missing rates");
    rates_init[e] = r;
    p = end;
  }
  return ne;
}

// ---- readers ------------------------------------------------------------------------------
int64_t colate_read_mut(const char* path, int64_t cap, int32_t* pos, float* age_begin, float* age_end, uint32_t* meta)
{
  std::vector<char> buf;
  if (!slurp_or_gz(path, buf)) return fail(COLATE_ERR_IO, std::string("Error while reading ") + path + "(.gz).");
  buf.push_back('\n');
  buf.push_back('\0');
  const char* p = buf.data();
  const char* endp = buf.data() + buf.size() - 1;
  // header line
  const char* nl = (const char*)memchr(p, '\n', endp - p);
  if (!nl) return 0;
  p = nl + 1;
  int64_t n = 0;
  while (p < endp) {
    nl = (const char*)memchr(p, '\n', endp - p);
    if (!nl) break;
    if (nl == p) {  // std::getline returns an empty line; the reference would fault on it
      if (nl + 1 >= endp) break;
      return fail(COLATE_ERR_IO, std::string("empty line in ") + path);
    }
    if (pos) {
      if (n >= cap) return fail(COLATE_ERR_ARG, "colate_read_mut: capacity too small");
      if (!parse_mut_line_host(p, nl, &pos[n], &age_begin[n], &age_end[n], &meta[n]))
        return fail(COLATE_ERR_IO, std::string("Error reading following line in mut file: ") + std::string(p, nl));
    }
    n++;
    p = nl + 1;
  }
  return n;
}

int64_t colate_read_colate_in(const char* path, int n_chr, const char* const* chr_names, int64_t cap,
                              int32_t* rec_chrom, int32_t* bp, int32_t* aaf, int32_t* daf, uint16_t* alleles)
{
  FILE* f = fopen(path, "rb");
  if (!f) return fail(COLATE_ERR_IO, std::string("Failed to open ") + path);
  fseek(f, 0, SEEK_END);
  long sz = ftell(f);
  fseek(f, 0, SEEK_SET);
  std::vector<char> buf((size_t)sz);
  if (sz > 0 && fread(buf.data(), 1, (size_t)sz, f) != (size_t)sz) { fclose(f); return fail(COLATE_ERR_IO, "short read"); }
  fclose(f);
  std::vector<std::string> names(chr_names, chr_names + n_chr);
  return colate::decode_colate_in_host(buf.data(), sz, names, cap, rec_chrom, bp, aaf, daf, alleles);
}

int colate_mask_bits_from_fasta(const char* path, int64_t n, const int32_t* pos, int64_t row0, uint32_t* pass_bits)
{
  std::vector<char> buf;
  if (!slurp_or_gz(path, buf)) return fail(COLATE_ERR_IO, std::string("Error while opening file ") + path + ".");
  // data.cpp:213-237: drop the first line, concatenate the rest upper-cased
  size_t i = 0;
  while (i < buf.size() && buf[i] != '\n') i++;
  i++;
  size_t len = 0;
  for (; i < buf.size(); i++) {
    char c = buf[i];
    if (c == '\n') continue;
    if (c >= 'a' && c <= 'z') c -= 32;
    buf[len++] = c;
  }
  for (int64_t k = 0; k < n; k++) {
    int32_t b = pos[k];
    bool pass = true;
    if ((uint64_t)(int64_t)b < (uint64_t)len) {       // int vs size_t compare, coal.cpp:2169
      if (b >= 1 && buf[b - 1] != 'P') pass = false;
    }
    int64_t m = row0 + k;
    if (pass) pass_bits[m >> 5] |= (1u << (m & 31));
    else pass_bits[m >> 5] &= ~(1u << (m & 31));
  }
  return 0;
}

// ---- writers ------------------------------------------------------------------------------
int colate_write_coal(const char* path, int R, int E, const double* epochs, double* rates, int is_ancient, int ep_null)
{
  // coal.cpp:3660-3672, 3830-3844; operator<<(double) with default flags == "%g"
  FILE* f = fopen(path, "w");
  if (!f) return fail(COLATE_ERR_IO, std::string("cannot write ") + path);
  fprintf(f, "0\n");
  if (is_ancient) {
    fprintf(f, "0 ");
    for (int e = ep_null + 1; e < E; e++) fprintf(f, "%g ", epochs[e]);
  } else {
    for (int e = 0; e < E; e++) fprintf(f, "%g ", epochs[e]);
  }
  fprintf(f, "\n");
  for (int i = 0; i < R; i++) {
    double* r = rates + (size_t)i * E;
    fprintf(f, "0 %d ", i);
    if (is_ancient) {
      for (int j = 0; j <= ep_null && j < E; j++) r[j] = 0;
      for (int e = ep_null; e < E; e++) fprintf(f, "%g ", r[e]);
    } else {
      for (int e = 0; e < E; e++) fprintf(f, "%g ", r[e]);
    }
    fprintf(f, "\n");
  }
  fclose(f);
  return 0;
}

int colate_write_colate_mat(const char* path, int R, const double* age_bin, const double* counts)
{
  // coal.cpp:3336-3343 (grid line) and 3453-3465 (two lines per replicate), operator<<(double) with default flags == "%g"
  if (!path || R <= 0 || !age_bin || !counts) return fail(COLATE_ERR_ARG, "colate_write_colate_mat: bad arguments");
  FILE* f = fopen(path, "w");
  if (!f) return fail(COLATE_ERR_IO, std::string("cannot write ") + path);
  for (int b = 0; b < colate::NBINS; b++) fprintf(f, "%g ", age_bin[b]);
  fprintf(f, "\n");
  for (int i = 0; i < 2 * R; i++) {
    for (int b = 0; b < colate::NBINS; b++) fprintf(f, "%g ", counts[(size_t)i * colate::NBINS + b]);
    fprintf(f, "\n");
  }
  fclose(f);
  return 0;
}

int colate_write_bin(const char* path, int R, int E, const double* epochs, const double* rates, const int32_t* iters)
{
  FILE* f = fopen(path, "wb");
  if (!f) return fail(COLATE_ERR_IO, std::string("cannot write ") + path);
  const char magic[8] = {'C', 'O', 'L', 'A', 'T', 'E', 'B', '1'};
  int32_t hdr[2] = {R, E};
  fwrite(magic, 1, 8, f);
  fwrite(hdr, 4, 2, f);
  fwrite(epochs, 8, (size_t)E, f);
  fwrite(rates, 8, (size_t)R * E, f);
  fwrite(iters, 4, (size_t)R, f);
  fclose(f);
  return 0;
}

}  // extern "C"

extern "C" int64_t colate_test_colate_in_runs(const char* buf, int64_t sz, int n_chr, const char* const* chr_names, int cap_runs,
                                              int64_t* runs4, int64_t* chr_first, int64_t* chr_end)
{
  std::vector<std::string> names(chr_names, chr_names + n_chr);
  std::vector<colate::ColateInRun> runs;
  const int64_t n = colate::colate_in_runs(buf, sz, names, runs);
  if ((int)runs.size() > cap_runs) return -1;
  for (size_t i = 0; i < runs.size(); i++) {
    runs4[4 * i] = runs[i].byte_off; runs4[4 * i + 1] = runs[i].width; runs4[4 * i + 2] = runs[i].chr_id; runs4[4 * i + 3] = runs[i].n_rec;
  }
  colate::chr_ranges_runs(n_chr, runs, chr_first, chr_end);
  return n | ((int64_t)runs.size() << 40);
}

// ---- make_tmp from a table (SURVEY.md 8f, N4) ------------------------------------------------------
// fasta::Read (data.cpp:213-237): header line dropped, the rest upper-cased and concatenated
static bool read_fasta_seq(const std::string& path, std::vector<char>& seq)
{
  if (!slurp_or_gz(path, seq)) return false;
  size_t i = 0;
  while (i < seq.size() && seq[i] != '\n') i++;
  i++;
  size_t len = 0;
  for (; i < seq.size(); i++) {
    char c = seq[i];
    if (c == '\n') continue;
    if (c >= 'a' && c <= 'z') c -= 32;
    seq[len++] = c;
  }
  seq.resize(len);
  return true;
}

extern "C" int64_t colate_read_fasta(const char* path, uint8_t** seq_out)
{
  using colate::fail;
  if (!path || !seq_out) return fail(COLATE_ERR_ARG, "colate_read_fasta: bad arguments");
  *seq_out = nullptr;
  std::vector<char> seq;
  if (!read_fasta_seq(path, seq)) return fail(COLATE_ERR_IO, std::string("Error while opening file ") + path + ".");
  uint8_t* p = (uint8_t*)malloc(seq.size() + 1);
  if (!p) return fail(COLATE_ERR_ARG, "colate_read_fasta: out of host memory");
  memcpy(p, seq.data(), seq.size());
  *seq_out = p;
  return (int64_t)seq.size();
}

extern "C" void colate_free(void* p) { free(p); }

// maketmp_table (coal.cpp:2682-2808): a .colate.in record stream for a haploid target given as a whitespace-separated
// table of (chromosome, position, allele) triples in --chr order.  For every row of the .mut files that is not
// flipped, maps to one branch and has single-letter allele codes (no age condition here), passes the optional mask
// (positions at or beyond the mask end are DROPPED here, unlike in mode mut) and has a table entry at its position,
// one record {lchrom, chrom, bp, anc, der, AAF = 1 - DAF, DAF} is written; with a reference genome (always the case
// through the CLI) the entry must carry the ancestral or the derived allele.  The table cursor is the reference's
// `is >> chr >> bp >> allele` stream: it persists across chromosomes, and once it runs dry nothing matches any more.
extern "C" int64_t colate_maketmp_table(int n_chr, const char* const* chr_names, const char* const* mut_files, const char* table_file,
                                        const char* const* target_masks, int has_ref_genome, const char* out_file)
{
  using colate::fail;
  if (n_chr <= 0 || !chr_names || !mut_files || !table_file || !out_file) return fail(COLATE_ERR_ARG, "colate_maketmp_table: bad arguments");
  std::vector<char> tab;
  if (!colate::slurp(table_file, tab)) return fail(COLATE_ERR_IO, std::string("Error while opening file ") + table_file);
  FILE* fp = fopen(out_file, "wb");
  if (!fp) return fail(COLATE_ERR_IO, std::string("cannot write ") + out_file);
  // token cursor over the table with the semantics of three chained formatted extractions
  size_t tp = 0;
  bool dry = false;                                   // a past extraction failed: the stream stays failed
  std::string chr_table, allele;
  long bp_target = -1;
  auto token = [&](std::string& out) -> bool {
    while (tp < tab.size() && isspace((unsigned char)tab[tp])) tp++;
    out.clear();                                      // operator>>(string) erases first
    if (tp >= tab.size()) return false;
    size_t b = tp;
    while (tp < tab.size() && !isspace((unsigned char)tab[tp])) tp++;
    out.assign(tab.data() + b, tp - b);
    return true;
  };
  auto next_triple = [&]() -> bool {
    if (dry) return false;
    std::string t;
    if (!token(chr_table)) { dry = true; return false; }
    if (!token(t)) { dry = true; return false; }
    char* end = nullptr;
    const long v = strtol(t.c_str(), &end, 10);
    if (end == t.c_str()) { bp_target = 0; dry = true; return false; }     // failed int extraction stores 0
    bp_target = v;
    if (!token(allele)) { dry = true; return false; }
    return true;
  };
  int64_t n_written = 0;
  for (int chr = 0; chr < n_chr; chr++) {
    const std::string name = chr_names[chr];
    std::vector<char> mask;
    const bool has_mask = target_masks && target_masks[chr];
    if (has_mask && !read_fasta_seq(target_masks[chr], mask)) { fclose(fp); return fail(COLATE_ERR_IO, std::string("Error while opening file ") + target_masks[chr] + "."); }
    std::vector<char> buf;
    if (!colate::slurp_or_gz(mut_files[chr], buf)) { fclose(fp); return fail(COLATE_ERR_IO, std::string("Error while reading ") + mut_files[chr] + "(.gz)."); }
    buf.push_back('\n');
    buf.push_back('\0');
    if (bp_target == -1) next_triple();
    while (chr_table != name) { if (!next_triple()) break; }
    const char* p = buf.data();
    const char* endp = buf.data() + buf.size() - 1;
    const char* nl = (const char*)memchr(p, '\n', endp - p);   // header line
    p = nl ? nl + 1 : endp;
    while (p < endp) {
      nl = (const char*)memchr(p, '\n', endp - p);
      if (!nl) break;
      if (nl == p) { if (nl + 1 >= endp) break; fclose(fp); return fail(COLATE_ERR_IO, std::string("empty line in ") + mut_files[chr]); }
      int32_t bp_mut; float ab, ae; uint32_t meta; int flipped, nb; char type[16];
      if (!colate::parse_mut_line_fields(p, nl, &bp_mut, &ab, &ae, &meta, &flipped, &nb, type)) {
        fclose(fp);
        return fail(COLATE_ERR_IO, std::string("Error reading following line in mut file: ") + std::string(p, nl));
      }
      p = nl + 1;
      if (!(flipped == 0 && nb == 1)) continue;
      // single-letter codes: ancestral in {A,C,G,T,0}, derived in {A,C,G,T,1} (type[] holds at most 15 characters: anything longer is not a code)
      const char* slash = strchr(type, '/');
      if (!slash || slash - type != 1 || strlen(slash + 1) != 1) continue;
      const char a = type[0], d = type[2];
      if (!(a == 'A' || a == 'C' || a == 'G' || a == 'T' || a == '0')) continue;
      if (!(d == 'A' || d == 'C' || d == 'G' || d == 'T' || d == '1')) continue;
      if (has_mask) {
        if ((uint64_t)(int64_t)bp_mut >= (uint64_t)mask.size()) continue;
        if (bp_mut >= 1 && mask[bp_mut - 1] != 'P') continue;
      }
      if (chr_table == name && bp_target < bp_mut)
        while (!dry && chr_table == name && bp_target < bp_mut) next_triple();
      if (!(chr_table == name && bp_target == bp_mut)) continue;
      int32_t daf = 0;
      const bool is_anc = allele.size() == 1 && allele[0] == a, is_der = allele.size() == 1 && allele[0] == d;
      if (has_ref_genome) {
        if (!(is_anc || is_der)) continue;
        if (is_der) daf = 1;
      } else if (!is_anc) daf = 1;
      const int32_t lchrom = (int32_t)name.size(), aaf = 1 - daf;
      fwrite(&lchrom, 4, 1, fp);
      fwrite(name.data(), 1, name.size(), fp);
      fwrite(&bp_mut, 4, 1, fp);
      fwrite(&a, 1, 1, fp);
      fwrite(&d, 1, 1, fp);
      fwrite(&aaf, 4, 1, fp);
      fwrite(&daf, 4, 1, fp);
      n_written++;
    }
  }
  fclose(fp);
  return n_written;
}

// ---- make_tmp from genotype records (SURVEY.md 8f N4, the vcf variant on pre-decoded arrays) -----------------------
// maketmp_vcf (coal.cpp:2325-2525): a .colate.in record stream from the genotype records of one sample set at the rows of the
// .mut files.  The BCF decoding (htslib, vcf_parser) stays with the caller; its output per record is the 1-based position, the
// first two alleles (the letter if the allele string is one character, 0 if it is empty, 0xff otherwise), the sum of the allele
// indices over the n_hap[chr] haplotypes (bcf_gt_allele, coal.cpp:2434, 2467) and whether every index is <= 1.
// The reference walks the file with a cursor (2397-2403): it reads on only while the record's position is below the row's, so a
// record is matched iff it is the first one at or after the row's position, and a cursor that has run off the end stays on the
// last record.  Row filter (2365, 2381-2395): not flipped, one branch, ancestral exactly one of A C G T 0 and derived exactly one
// of A C G T 1; a mask drops rows at or beyond its end or not 'P'.  A matched record (2406-2487) gives DAF = N when it shows
// the derived allele alone and nobody carries an alternative, the (flipped) allele sum when its alleles are the row's, and
// drops the row otherwise; an unmatched row is read off the reference genome (2489-2503).
extern "C" int64_t colate_maketmp_records(int n_chr, const char* const* chr_names, const char* const* mut_files, const int64_t* rec_off,
                                          const int32_t* rec_pos, const uint8_t* rec_a0, const uint8_t* rec_a1, const int32_t* rec_alt_sum,
                                          const uint8_t* rec_biallelic, const int32_t* n_hap, const char* const* ref_genomes,
                                          const char* const* target_masks, const char* out_file)
{
  using colate::fail;
  if (n_chr <= 0 || !chr_names || !mut_files || !rec_off || !rec_pos || !rec_a0 || !rec_a1 || !rec_alt_sum || !rec_biallelic || !n_hap || !out_file)
    return fail(COLATE_ERR_ARG, "colate_maketmp_records: bad arguments");
  for (int chr = 0; chr < n_chr; chr++)
    if (rec_off[chr + 1] <= rec_off[chr]) return fail(COLATE_ERR_ARG, "colate_maketmp_records: a chromosome without genotype records (the reference reads the first record unconditionally, coal.cpp:2362)");
  FILE* fp = fopen(out_file, "wb");
  if (!fp) return fail(COLATE_ERR_IO, std::string("cannot write ") + out_file);
  int64_t n_written = 0;
  for (int chr = 0; chr < n_chr; chr++) {
    const std::string name = chr_names[chr];
    std::vector<char> mask, refg;
    const bool has_mask = target_masks && target_masks[chr];
    const bool has_refg = ref_genomes && ref_genomes[chr];
    if (has_mask && !read_fasta_seq(target_masks[chr], mask)) { fclose(fp); return fail(COLATE_ERR_IO, std::string("Error while opening file ") + target_masks[chr] + "."); }
    if (has_refg && !read_fasta_seq(ref_genomes[chr], refg)) { fclose(fp); return fail(COLATE_ERR_IO, std::string("Error while opening file ") + ref_genomes[chr] + "."); }
    std::vector<char> buf;
    if (!colate::slurp_or_gz(mut_files[chr], buf)) { fclose(fp); return fail(COLATE_ERR_IO, std::string("Error while reading ") + mut_files[chr] + "(.gz)."); }
    buf.push_back('\n');
    buf.push_back('\0');
    const char* p = buf.data();
    const char* endp = buf.data() + buf.size() - 1;
    const char* nl = (const char*)memchr(p, '\n', endp - p);   // header line
    p = nl ? nl + 1 : endp;
    int64_t cur = rec_off[chr];                                 // the record the reference's reader holds
    const int64_t rec_end = rec_off[chr + 1];
    int32_t bp_target = rec_pos[cur];
    const int32_t N = n_hap[chr];
    while (p < endp) {
      nl = (const char*)memchr(p, '\n', endp - p);
      if (!nl) break;
      if (nl == p) { if (nl + 1 >= endp) break; fclose(fp); return fail(COLATE_ERR_IO, std::string("empty line in ") + mut_files[chr]); }
      int32_t bp_mut; float ab, ae; uint32_t meta; int flipped, nb; char type[16];
      if (!colate::parse_mut_line_fields(p, nl, &bp_mut, &ab, &ae, &meta, &flipped, &nb, type)) {
        fclose(fp);
        return fail(COLATE_ERR_IO, std::string("Error reading following line in mut file: ") + std::string(p, nl));
      }
      p = nl + 1;
      if (!(flipped == 0 && nb == 1)) continue;
      if (!(type[0] != '\0' && type[1] == '/' && type[2] != '\0' && type[3] == '\0')) continue;   // both alleles one letter
      const char a = type[0], d = type[2];
      if (!(a == 'A' || a == 'C' || a == 'G' || a == 'T' || a == '0')) continue;
      if (!(d == 'A' || d == 'C' || d == 'G' || d == 'T' || d == '1')) continue;
      if (has_mask) {
        if ((uint64_t)(int64_t)bp_mut >= (uint64_t)mask.size()) continue;
        if (bp_mut >= 1 && mask[bp_mut - 1] != 'P') continue;
      }
      if (bp_target < bp_mut)
        while (cur + 1 < rec_end) {
          bp_target = rec_pos[++cur];
          if (bp_target >= bp_mut) break;
        }
      int32_t daf = 0;
      if (bp_target == bp_mut) {
        const uint8_t t0 = rec_a0[cur], t1 = rec_a1[cur];
        const uint8_t ua = (uint8_t)a, ud = (uint8_t)d;
        if (t0 == ud && t1 == 0) {                       // the derived allele alone: shared by everybody unless someone carries an alternative
          if (!rec_biallelic[cur] || rec_alt_sum[cur] != 0) continue;
          daf = N;
        } else if ((t0 == ua && t1 == ud) || (t0 == ud && t1 == ua)) {
          if (!rec_biallelic[cur]) continue;
          daf = (t0 == ud && t1 == ua) ? N - rec_alt_sum[cur] : rec_alt_sum[cur];
        } else continue;
      } else {
        if (!has_refg || bp_mut < 1 || (uint64_t)(bp_mut - 1) >= (uint64_t)refg.size()) continue;
        const char g = refg[bp_mut - 1];
        if (d == g) daf = N;
        else if (a == g) daf = 0;
        else continue;
      }
      const int32_t aaf = N - daf;
      if (aaf < 0) { fclose(fp); return fail(COLATE_ERR_ARG, "colate_maketmp_records: allele sum above the number of haplotypes (the reference asserts, coal.cpp:2511)"); }
      const int32_t lchrom = (int32_t)name.size();
      fwrite(&lchrom, 4, 1, fp);
      fwrite(name.data(), 1, name.size(), fp);
      fwrite(&bp_mut, 4, 1, fp);
      fwrite(&a, 1, 1, fp);
      fwrite(&d, 1, 1, fp);
      fwrite(&aaf, 4, 1, fp);
      fwrite(&daf, 4, 1, fp);
      n_written++;
    }
  }
  fclose(fp);
  return n_written;
}

// ---- make_tmp from a pileup (SURVEY.md 8f N4, the bam variant on pre-decoded arrays) ------------------------------
// maketmp_bam (coal.cpp:2527-2680): a .colate.in record stream from the pileup of one BAM file at the rows of the .mut
// files.  The BAM decoding (htslib, bam_parser) stays with the caller; `counts` is its output: for every DATA ROW of the
// .mut files in --chr order, the reads showing A, C, G, T at the row's position (bam_parser::count_alleles at bp_mut - 1, zeros
// where the position is not covered).  Row filter as the reference: not flipped, one branch, ancestral exactly one of
// A C G T 0 and a non-empty derived string (no age condition, no condition on the derived code: coal.cpp:2568, 2584-2587);
// the optional mask drops positions at or beyond its end (2589-2595); AAF / DAF are the counts of the one-letter ancestral /
// derived alleles (2616-2633), a record is written iff one of them is positive (2641-2646; no limit on the number of alleles).
extern "C" int64_t colate_maketmp_pileup(int n_chr, const char* const* chr_names, const char* const* mut_files, const int32_t* counts,
                                         int64_t n_rows, const char* const* target_masks, const char* out_file)
{
  using colate::fail;
  if (n_chr <= 0 || !chr_names || !mut_files || !counts || !out_file) return fail(COLATE_ERR_ARG, "colate_maketmp_pileup: bad arguments");
  FILE* fp = fopen(out_file, "wb");
  if (!fp) return fail(COLATE_ERR_IO, std::string("cannot write ") + out_file);
  auto idx = [](char c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1; };
  int64_t n_written = 0, row = 0;
  for (int chr = 0; chr < n_chr; chr++) {
    const std::string name = chr_names[chr];
    std::vector<char> mask;
    const bool has_mask = target_masks && target_masks[chr];
    if (has_mask && !read_fasta_seq(target_masks[chr], mask)) { fclose(fp); return fail(COLATE_ERR_IO, std::string("Error while opening file ") + target_masks[chr] + "."); }
    std::vector<char> buf;
    if (!colate::slurp_or_gz(mut_files[chr], buf)) { fclose(fp); return fail(COLATE_ERR_IO, std::string("Error while reading ") + mut_files[chr] + "(.gz)."); }
    buf.push_back('\n');
    buf.push_back('\0');
    const char* p = buf.data();
    const char* endp = buf.data() + buf.size() - 1;
    const char* nl = (const char*)memchr(p, '\n', endp - p);   // header line
    p = nl ? nl + 1 : endp;
    while (p < endp) {
      nl = (const char*)memchr(p, '\n', endp - p);
      if (!nl) break;
      if (nl == p) { if (nl + 1 >= endp) break; fclose(fp); return fail(COLATE_ERR_IO, std::string("empty line in ") + mut_files[chr]); }
      int32_t bp_mut; float ab, ae; uint32_t meta; int flipped, nb; char type[16];
      if (!colate::parse_mut_line_fields(p, nl, &bp_mut, &ab, &ae, &meta, &flipped, &nb, type)) {
        fclose(fp);
        return fail(COLATE_ERR_IO, std::string("Error reading following line in mut file: ") + std::string(p, nl));
      }
      p = nl + 1;
      if (row >= n_rows) { fclose(fp); return fail(COLATE_ERR_ARG, "colate_maketmp_pileup: fewer count rows than .mut rows"); }
      const int32_t* c = counts + 4 * row++;
      if (!(flipped == 0 && nb == 1)) continue;
      // type[] holds the first 15 characters of the mutation type: enough for "one-letter ancestral, '/', first derived letter,
      // is the derived string longer than one letter"
      const char* slash = strchr(type, '/');
      if (!slash || slash - type != 1 || slash[1] == '\0') continue;       // ancestral one letter, derived non-empty
      const char a = type[0], d = type[2];
      if (!(a == 'A' || a == 'C' || a == 'G' || a == 'T' || a == '0')) continue;
      if (has_mask) {
        if ((uint64_t)(int64_t)bp_mut >= (uint64_t)mask.size()) continue;
        if (bp_mut >= 1 && mask[bp_mut - 1] != 'P') continue;
      }
      const int reads = c[0] + c[1] + c[2] + c[3];
      if (reads <= 0) continue;
      int32_t aaf = 0, daf = 0;
      if (idx(a) >= 0) aaf = c[idx(a)];
      if (slash[2] == '\0' && idx(d) >= 0) daf = c[idx(d)];              // the derived string must be the single letter
      if (!(aaf > 0 || daf > 0)) continue;
      const int32_t lchrom = (int32_t)name.size();
      fwrite(&lchrom, 4, 1, fp);
      fwrite(name.data(), 1, name.size(), fp);
      fwrite(&bp_mut, 4, 1, fp);
      fwrite(&a, 1, 1, fp);
      fwrite(&d, 1, 1, fp);
      fwrite(&aaf, 4, 1, fp);
      fwrite(&daf, 4, 1, fp);
      n_written++;
    }
  }
  fclose(fp);
  if (row != n_rows) return fail(COLATE_ERR_ARG, "colate_maketmp_pileup: more count rows than .mut rows");
  return n_written;
}
