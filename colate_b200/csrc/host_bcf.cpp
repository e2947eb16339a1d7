// BCF input, host side: the BCF2 container (VCF specification v4.3, 6.3) over BGZF (bgzf.h).  The reference reads BCF through
// htslib (vcf_parser, include/vcf/htslib.cpp); of a record parse_vcfvcf and maketmp_vcf use the position, the first two alleles
// and the GT values (coal.cpp:997-1137, 2397-2487), which the device decodes (kernels_bcf.cu).  The host inflates the blocks,
// parses the header for the sample count and the dictionary index of GT, and walks the records by l_shared / l_indiv.
#include "bcf_reader.h"

#include <sys/time.h>

#include <algorithm>
#include <cstring>
#include <map>
#include <thread>

#include "internal.h"

namespace colate {

namespace {
inline uint32_t rd32(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }
inline double now_s() { timeval tv; gettimeofday(&tv, nullptr); return tv.tv_sec + 1e-6 * tv.tv_usec; }

// value of key=<...> inside a structured header line's <...> (quoted values are skipped over), "" if absent
std::string field(const std::string& body, const std::string& key)
{
  size_t i = 0;
  while (i < body.size()) {
    const size_t eq = body.find('=', i);
    if (eq == std::string::npos) break;
    const std::string k = body.substr(i, eq - i);
    size_t j = eq + 1;
    if (j < body.size() && body[j] == '"') {
      j++;
      while (j < body.size() && body[j] != '"') j += body[j] == '\\' ? 2 : 1;
      j = std::min(body.size(), j + 1);
    } else {
      while (j < body.size() && body[j] != ',') j++;
    }
    if (k == key) return body.substr(eq + 1, j - eq - 1);
    i = j + 1;
  }
  return "";
}
}  // namespace

// Header text -> sample count and GT's dictionary index (-1: no ##FORMAT=<ID=GT line).  The dictionary holds the FILTER, INFO
// and FORMAT IDs (one entry per ID, shared by the three kinds): PASS is 0, the others are numbered in order of first appearance
// unless the line carries IDX=, which sets the number (htslib's bcf_hdr_add_hrec; bcftools writes IDX=, hand-written headers do not).
void header_text(const char* text, size_t n, int* n_sample, int* gt_key)
{
  std::map<std::string, long> dict{{"PASS", 0}};
  long next = 1;
  *n_sample = 0;
  *gt_key = -1;
  size_t i = 0;
  while (i < n && text[i]) {
    size_t e = i;
    while (e < n && text[e] && text[e] != '\n') e++;
    std::string line(text + i, e - i);
    if (!line.empty() && line.back() == '\r') line.pop_back();
    i = e + 1;
    if (line.rfind("#CHROM", 0) == 0) {
      int tabs = 0;
      for (char ch : line) tabs += ch == '\t';
      *n_sample = std::max(0, tabs - 8);      // #CHROM POS ID REF ALT QUAL FILTER INFO FORMAT sample...
      continue;
    }
    bool is_format = line.rfind("##FORMAT=<", 0) == 0;
    if (!is_format && line.rfind("##INFO=<", 0) != 0 && line.rfind("##FILTER=<", 0) != 0) continue;
    const size_t lt = line.find('<');
    const std::string body = line.substr(lt + 1, line.size() >= lt + 2 && line.back() == '>' ? line.size() - lt - 2 : std::string::npos);
    const std::string id = field(body, "ID");
    const std::string idx = field(body, "IDX");
    long k;
    auto it = dict.find(id);
    if (it != dict.end()) k = it->second;
    else {
      k = idx.empty() ? next : strtol(idx.c_str(), nullptr, 10);
      dict[id] = k;
    }
    next = std::max(next, k + 1);
    if (is_format && id == "GT") *gt_key = (int)k;
  }
}

int BcfReader::open(const std::string& path, int threads)
{
  if (int rc = open_bgzf(path, "BCF", threads)) return rc;
  return read_header();
}

int BcfReader::read_header()
{
  if (int rc = need_header_bytes(5, 0)) return rc;
  if (memcmp(carry_.data(), "BCF\2", 4) != 0 || (carry_[4] != 1 && carry_[4] != 2))
    return err("not a BCF file (magic BCF\\2\\1 or BCF\\2\\2 missing)", 0, false);
  if (int rc = need_header_bytes(9, 5)) return rc;
  const uint32_t l_text = rd32(carry_.data() + 5);
  if (l_text > (1u << 30)) return err("BCF header with l_text over 1 GiB", 5, false);
  const size_t o = 9 + (size_t)l_text;
  if (int rc = need_header_bytes(o, 5)) return rc;
  header_text((const char*)carry_.data() + 9, l_text, &n_sample, &gt_key);
  if (gt_key < 0) return err("BCF header without a ##FORMAT=<ID=GT line", 9, false);
  drop_header(o);
  return 0;
}

int BcfReader::fill(uint8_t* buf, size_t target, BcfWindow& w)
{
  size_t n = 0;
  if (int rc = fill_window(buf, target, &n, &w.ustart)) return rc;
  const double t0 = now_s();
  w.n_bytes = n;
  w.rec_off.clear();
  w.rec_pos.clear();
  size_t o = 0;
  while (o + 8 <= n) {
    const uint64_t l_shared = rd32(buf + o), l_indiv = rd32(buf + o + 4);
    const uint64_t at = w.ustart + o;
    if (l_shared < 24) return err("BCF record with l_shared " + std::to_string(l_shared) + " (< 24)", at, false);
    if (o + 8 + l_shared + l_indiv > n) break;              // partial record: carried into the next window
    const uint8_t* r = buf + o + 8;
    const int32_t chrom = (int32_t)rd32(r), pos = (int32_t)rd32(r + 4);
    const int ns = (int)(rd32(r + 20) & 0xffffffu);
    if (ns != n_sample)
      return err("BCF record with " + std::to_string(ns) + " samples (the header has " + std::to_string(n_sample) + ")", at, false);
    if (n_records == 0) {
      contig = chrom;
      first_pos = pos;
    } else {
      if (chrom != contig)
        return err("BCF record on contig " + std::to_string(chrom) + " after records on contig " + std::to_string(contig) +
                       " (a per-chromosome file holds one contig)", at, false);
      if (pos < last_pos)
        return fail(COLATE_ERR_ORDER, path_ + ": BCF records not sorted by position (POS " + std::to_string(pos + 1) + " after " +
                                          std::to_string(last_pos + 1) + ") at inflated byte offset " + std::to_string(at));
    }
    last_pos = pos;
    n_records++;
    w.rec_off.push_back((int64_t)o);
    w.rec_pos.push_back(pos);
    o += 8 + l_shared + l_indiv;
  }
  carry_tail(buf, o, n, w.ustart);
  walk_s += now_s() - t0;
  if (at_end() && !carry_.empty()) return err("BCF record runs past the end of the data", carry_uoff_, false);
  if (at_end() && n_records == 0) return err("BCF file without records (the reference reads a first record unconditionally)", carry_uoff_, false);
  return 0;
}

}  // namespace colate

// Host-only scan of a BCF file (no GPU): record count, first and last POS (0-based), the records' contig, the header's sample
// count and GT key, with every host check of colate_rows_from_bcf.
extern "C" int colate_bcf_scan(const char* path, int64_t window_bytes, int64_t* n_records, int32_t* first_pos, int32_t* last_pos,
                               int32_t* contig, int32_t* n_sample, int32_t* gt_key)
{
  using namespace colate;
  if (!path) return fail(COLATE_ERR_ARG, "colate_bcf_scan: bad arguments");
  BcfReader rd;
  if (int rc = rd.open(path, (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency())))) return rc;
  const size_t target = window_bytes > 0 ? (size_t)window_bytes : (size_t)64 << 20;
  std::vector<uint8_t> buf;
  BcfWindow w;
  for (;;) {
    const size_t need = rd.next_window_bytes(target);
    if (need == 0) break;
    if (buf.size() < need) buf.resize(need);
    if (int rc = rd.fill(buf.data(), target, w)) return rc;
  }
  if (rd.n_records == 0) return rd.err("BCF file without records (the reference reads a first record unconditionally)", 0, false);
  if (n_records) *n_records = rd.n_records;
  if (first_pos) *first_pos = rd.first_pos;
  if (last_pos) *last_pos = rd.last_pos;
  if (contig) *contig = rd.contig;
  if (n_sample) *n_sample = rd.n_sample;
  if (gt_key) *gt_key = rd.gt_key;
  return 0;
}
