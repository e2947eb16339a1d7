// Bgzipped text VCF input, host side (vcf_reader.h), and the format detection shared by every genotype-file reader.  The
// reference opens <prefix>_chr<c>.bcf with htslib's bcf_open, which reads BGZF text VCF into the same bcf1_t as BCF; the host
// walks the lines for CHROM and POS, the device parses the rest (k_vcf_decode).
#include "vcf_reader.h"

#include <sys/time.h>

#include <algorithm>
#include <cstring>
#include <thread>

#include "internal.h"

namespace colate {

namespace {
inline double now_s() { timeval tv; gettimeofday(&tv, nullptr); return tv.tv_sec + 1e-6 * tv.tv_usec; }
const char kVcfMagic[] = "##fileformat=VCF";
const char* const kFixed[8] = {"#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO"};
}  // namespace

int open_genotypes(const std::string& path, int threads, std::unique_ptr<GenotypeReader>* out)
{
  BgzfFile f;
  if (int rc = f.open_bgzf(path, "BCF", threads)) return rc;
  const uint8_t* p;
  size_t got;
  if (int rc = f.peek(5, &p, &got)) return rc;
  bool vcf = false;
  if (got == 5 && memcmp(p, "BCF\2", 4) != 0) {
    if (int rc = f.peek(sizeof kVcfMagic - 1, &p, &got)) return rc;
    vcf = got == sizeof kVcfMagic - 1 && memcmp(p, kVcfMagic, got) == 0;
  }
  if (vcf) out->reset(new VcfReader);
  else out->reset(new BcfReader);
  (*out)->adopt(f);
  return (*out)->read_header();
}

int VcfReader::read_header()
{
  format_ = "VCF";
  record_newlines = true;
  // whole lines from the start of carry_: ## lines until the #CHROM line
  size_t o = 0, from = 0, end = 0;
  for (;;) {
    const uint8_t* nl = carry_.size() > from ? (const uint8_t*)memchr(carry_.data() + from, '\n', carry_.size() - from) : nullptr;
    if (!nl && !at_end()) {
      from = carry_.size();
      const uint8_t* p;
      size_t got;
      if (int rc = peek(carry_.size() + 1, &p, &got)) return rc;
      continue;
    }
    const size_t e = nl ? (size_t)(nl - carry_.data()) : carry_.size();
    const char* l = (const char*)carry_.data() + o;
    if (e == o && !nl) return err("VCF header without a #CHROM line", o, false);
    if (e - o >= 6 && memcmp(l, "#CHROM", 6) == 0) {
      end = nl ? e + 1 : e;
      break;
    }
    if (e - o < 2 || l[0] != '#' || l[1] != '#' || !nl)
      return err("VCF header without a #CHROM line (a line that is neither ## nor #CHROM)", o, false);
    o = from = e + 1;
  }
  int ns = 0;
  header_text((const char*)carry_.data(), end, &ns, &gt_key);
  if (gt_key < 0) return err("VCF header without a ##FORMAT=<ID=GT line", 0, false);
  std::vector<std::string> cols(1);
  for (size_t i = o; i < end && carry_[i] != '\n'; i++) {
    if (carry_[i] == '\t') cols.emplace_back();
    else cols.back() += (char)carry_[i];
  }
  for (int c = 0; c < 8; c++)
    if (c >= (int)cols.size() || cols[c] != kFixed[c])
      return err("VCF #CHROM line whose first eight columns are not CHROM POS ID REF ALT QUAL FILTER INFO", o, false);
  if (cols.size() == 8) return err("VCF file without samples (the #CHROM line ends at INFO)", o, false);
  if (cols[8] != "FORMAT") return err("VCF #CHROM line whose ninth column is not FORMAT", o, false);
  if (cols.size() == 9) return err("VCF #CHROM line with FORMAT but no sample", o, false);
  n_sample = (int)cols.size() - 9;
  drop_header(end);
  return 0;
}

// one record line buf[o, e) (newline excluded): CHROM and POS
int VcfReader::line(const uint8_t* buf, size_t o, size_t e, BcfWindow& w)
{
  const uint64_t at = w.ustart + o;
  if (e == o) return err("empty VCF line", at, false);
  if (buf[e - 1] == '\r') return err("VCF line ending in \\r\\n (CRLF is not read)", at, false);
  const uint8_t* t1 = (const uint8_t*)memchr(buf + o, '\t', e - o);
  if (!t1) return err("VCF line without a POS column", at, false);
  const size_t ce = (size_t)(t1 - buf);
  size_t q = ce + 1;
  int64_t v = 0;
  bool ok = q < e && buf[q] != '\t';
  for (; ok && q < e && buf[q] != '\t'; q++) {
    const unsigned d = buf[q] - '0';
    ok = d <= 9 && (v = v * 10 + d) <= 2147483646;
  }
  if (!ok) return err("VCF POS that is not a plain decimal in [0, 2147483646]", at, false);
  const int32_t pos = (int32_t)(v - 1);
  if (n_records == 0) {
    chrom.assign((const char*)buf + o, ce - o);
    first_pos = pos;
  } else {
    if (ce - o != chrom.size() || memcmp(buf + o, chrom.data(), ce - o) != 0)
      return err("VCF record on contig " + std::string((const char*)buf + o, ce - o) + " after records on contig " + chrom +
                     " (a per-chromosome file holds one contig)", at, false);
    if (pos < last_pos)
      return fail(COLATE_ERR_ORDER, path_ + ": VCF records not sorted by position (POS " + std::to_string(v) + " after " +
                                        std::to_string((int64_t)last_pos + 1) + ") at inflated byte offset " + std::to_string(at));
  }
  last_pos = pos;
  n_records++;
  w.rec_off.push_back((int64_t)o);
  w.rec_pos.push_back(pos);
  return 0;
}

int VcfReader::fill(uint8_t* buf, size_t target, BcfWindow& w)
{
  size_t n = 0;
  const size_t n_carry = carry_.size();
  if (int rc = fill_window(buf, target, &n, &w.ustart)) return rc;
  const double t0 = now_s();
  w.n_bytes = n;
  w.rec_off.clear();
  w.rec_pos.clear();
  const bool last = at_end();
  // newlines: in the carried bytes (a cut line, or after the header what its blocks held past it) found here, in the inflated
  // blocks listed by the inflate threads (BgzfFile::newlines)
  size_t o = 0, k = 0;
  while (o < n) {
    const uint8_t* nl = o < n_carry ? (const uint8_t*)memchr(buf + o, '\n', n_carry - o) : nullptr;
    const bool found = nl || k < newlines.size();
    if (!found && !last) break;                               // partial line: carried into the next window
    const size_t e = nl ? (size_t)(nl - buf) : found ? (size_t)newlines[k++] : n;   // the last line may lack its newline
    if (int rc = line(buf, o, e, w)) return rc;
    o = found ? e + 1 : e;
  }
  w.text_end = (int64_t)o;
  carry_tail(buf, o, n, w.ustart);
  walk_s += now_s() - t0;
  if (at_end() && n_records == 0) return err("VCF file without records (the reference reads a first record unconditionally)", carry_uoff_, false);
  return 0;
}

}  // namespace colate

// Host-only scan of a bgzipped text VCF (no GPU): record count, first and last POS (0-based, as htslib's bcf1_t.pos), the header's
// sample count and the records' CHROM (NUL-terminated, cut to chrom_cap - 1 bytes), with every host check of colate_rows_from_bcf.
// A BCF file is refused here (colate_bcf_scan reads it).
extern "C" int colate_vcf_scan(const char* path, int64_t window_bytes, int64_t* n_records, int32_t* first_pos, int32_t* last_pos,
                               int32_t* n_sample, char* chrom, int64_t chrom_cap)
{
  using namespace colate;
  if (!path || (chrom && chrom_cap <= 0)) return fail(COLATE_ERR_ARG, "colate_vcf_scan: bad arguments");
  std::unique_ptr<GenotypeReader> rd;
  if (int rc = open_genotypes(path, (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency())), &rd)) return rc;
  if (!rd->text) return rd->err("a BCF file, not text VCF (colate_bcf_scan reads it)", 0, false);
  const size_t target = window_bytes > 0 ? (size_t)window_bytes : (size_t)64 << 20;
  std::vector<uint8_t> buf;
  BcfWindow w;
  for (;;) {
    const size_t need = rd->next_window_bytes(target);
    if (need == 0) break;
    if (buf.size() < need) buf.resize(need);
    if (int rc = rd->fill(buf.data(), target, w)) return rc;
  }
  if (rd->n_records == 0) return rd->err("VCF file without records (the reference reads a first record unconditionally)", 0, false);
  const std::string& c = static_cast<VcfReader&>(*rd).chrom;
  if (n_records) *n_records = rd->n_records;
  if (first_pos) *first_pos = rd->first_pos;
  if (last_pos) *last_pos = rd->last_pos;
  if (n_sample) *n_sample = rd->n_sample;
  if (chrom) {
    const size_t k = std::min(c.size(), (size_t)chrom_cap - 1);
    memcpy(chrom, c.data(), k);
    chrom[k] = 0;
  }
  return 0;
}
