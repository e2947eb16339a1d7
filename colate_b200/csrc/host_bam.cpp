// BAM input, host side: BGZF (SAM/BAM format specification 4.1) and the BAM container (4.2).  The reference reads BAM
// through htslib (bam_parser, include/vcf/htslib.cpp); of a record its pileup uses pos, mapq, l_seq, the packed sequence and
// the qualities, which the device decodes (kernels_bam.cu).  The host finds the blocks, inflates them in parallel, parses the
// header, matches the --chr list and walks the records by block_size to find their boundaries and contigs.
#include "bam_reader.h"

#include <sys/time.h>

#include <algorithm>
#include <cstring>
#include <thread>

#include "internal.h"

namespace colate {

namespace {
inline uint16_t rd16(const uint8_t* p) { return (uint16_t)(p[0] | p[1] << 8); }
inline uint32_t rd32(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }
inline double now_s() { timeval tv; gettimeofday(&tv, nullptr); return tv.tv_sec + 1e-6 * tv.tv_usec; }
}  // namespace

int BamReader::open(const std::string& path, int n_chr, const char* const* chr_names, int threads)
{
  if (int rc = open_bgzf(path, "BAM", threads)) return rc;
  return parse_header(n_chr, chr_names);
}

int BamReader::parse_header(int n_chr, const char* const* chr_names)
{
  if (int rc = need_header_bytes(4, 0)) return rc;
  if (memcmp(carry_.data(), "BAM\1", 4) != 0) return err("not a BAM file (magic BAM\\1 missing)", 0, false);
  if (int rc = need_header_bytes(8, 4)) return rc;
  const uint32_t l_text = rd32(carry_.data() + 4);
  if (l_text > (1u << 30)) return err("BAM header with l_text over 1 GiB", 4, false);
  size_t o = 8 + (size_t)l_text;
  if (int rc = need_header_bytes(o + 4, 4)) return rc;
  const int32_t n_ref = (int32_t)rd32(carry_.data() + o);
  if (n_ref < 0) return err("BAM header with a negative n_ref", o, false);
  o += 4;
  for (int32_t r = 0; r < n_ref; r++) {
    if (int rc = need_header_bytes(o + 4, o)) return rc;
    const uint32_t l_name = rd32(carry_.data() + o);
    if (l_name == 0 || l_name > (1u << 20)) return err("BAM header with a bad l_name", o, false);
    if (int rc = need_header_bytes(o + 4 + l_name + 4, o)) return rc;
    const char* nm = (const char*)carry_.data() + o + 4;
    ref_names_.emplace_back(nm, strnlen(nm, l_name));
    o += 4 + l_name + 4;
  }
  drop_header(o);
  listed_of_ref_.assign(n_ref, -1);
  ref_of_listed_.assign(n_chr, -1);
  done_.assign(n_chr, 0);
  for (int c = 0; c < n_chr; c++) {
    const std::string a = chr_names[c], b = "chr" + a;
    listed_names_.push_back(a);
    for (int32_t r = 0; r < n_ref; r++) {
      if (!contig_matches(ref_names_[r], a)) continue;
      if (ref_of_listed_[c] >= 0)
        return fail(COLATE_ERR_IO, path_ + ": contig " + a + " of the --chr list appears in the BAM header as both " + ref_names_[ref_of_listed_[c]] +
                                       " and " + ref_names_[r]);
      if (listed_of_ref_[r] >= 0) return fail(COLATE_ERR_ARG, path_ + ": header contig " + ref_names_[r] + " matches two --chr entries");
      ref_of_listed_[c] = r;
      listed_of_ref_[r] = c;
    }
    if (ref_of_listed_[c] < 0) return fail(COLATE_ERR_IO, path_ + ": contig " + a + " of the --chr list is not in the BAM header (neither " + a + " nor " + b + ")");
  }
  return 0;
}

int BamReader::fill(uint8_t* buf, size_t target, BamWindow& w)
{
  size_t n = 0;
  if (int rc = fill_window(buf, target, &n, &w.ustart)) return rc;
  const double t0 = now_s();
  w.n_bytes = n;
  w.rec_off.clear(); w.rec_chr.clear(); w.rec_pos.clear(); w.rec_lseq.clear();
  size_t o = 0;
  while (o + 4 <= n) {
    const uint32_t bs = rd32(buf + o);
    const uint64_t at = w.ustart + o;
    if (bs < 32) return err("BAM record with block_size " + std::to_string(bs) + " (< 32)", at, false);
    if (o + 4 + (size_t)bs > n) break;                    // partial record: carried into the next window
    const uint8_t* r = buf + o + 4;
    const int32_t ref = (int32_t)rd32(r), pos = (int32_t)rd32(r + 4), l_seq = (int32_t)rd32(r + 16);
    const uint32_t l_read_name = r[8], n_cigar = rd16(r + 12);
    if (l_seq < 0 || 32 + (uint64_t)l_read_name + 4ull * n_cigar + (uint64_t)(l_seq + 1) / 2 + (uint64_t)l_seq > bs)
      return err("BAM record whose fields run past its block_size", at, false);
    if (ref < -1 || ref >= (int32_t)listed_of_ref_.size()) return err("BAM record with refID " + std::to_string(ref) + " outside the header", at, false);
    const int c = ref >= 0 ? listed_of_ref_[ref] : -1;
    if (c >= 0) {
      // (checked here, before any launch: the counting kernels index the reference genome at pos + i)
      if (pos < 0) return fail(COLATE_ERR_ORDER, path_ + ": a record of contig " + ref_names_[ref] + " has the negative position " + std::to_string(pos) +
                                                     " at inflated byte offset " + std::to_string(at));
      if (c != cur_) {
        if (done_[c] || c < cur_)
          return err("records of contig " + ref_names_[ref] + " are not contiguous or not in --chr order (after " +
                         (cur_ >= 0 ? ref_names_[ref_of_listed_[cur_]] : std::string("?")) + ")", at, false);
        if (cur_ >= 0) done_[cur_] = 1;
        cur_ = c;
      }
      w.rec_off.push_back((int64_t)o);
      w.rec_chr.push_back(c);
      w.rec_pos.push_back(pos);
      w.rec_lseq.push_back(l_seq);
    }
    o += 4 + (size_t)bs;
  }
  carry_tail(buf, o, n, w.ustart);
  walk_s += now_s() - t0;
  if (at_end() && !carry_.empty()) return err("BAM record runs past the end of the data", carry_uoff_, false);
  return 0;
}

}  // namespace colate

// Host-only scan of a BAM file (no GPU): per --chr entry the number of records, the first and last position and the header
// contig it matched.  Same BGZF checks, header parse, contig matching and record walk as colate_pileup_bam.
extern "C" int colate_bam_scan(const char* path, int n_chr, const char* const* chr_names, int64_t window_bytes, int64_t* n_records,
                               int32_t* first_pos, int32_t* last_pos, int32_t* ref_id)
{
  using namespace colate;
  if (!path || n_chr <= 0 || !chr_names) return fail(COLATE_ERR_ARG, "colate_bam_scan: bad arguments");
  BamReader rd;
  if (int rc = rd.open(path, n_chr, chr_names, (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency())))) return rc;
  std::vector<int64_t> n(n_chr, 0);
  std::vector<int32_t> first(n_chr, -1), last(n_chr, -1);
  const size_t target = window_bytes > 0 ? (size_t)window_bytes : (size_t)64 << 20;
  std::vector<uint8_t> buf;
  BamWindow w;
  for (;;) {
    const size_t need = rd.next_window_bytes(target);
    if (need == 0) break;
    if (buf.size() < need) buf.resize(need);
    if (int rc = rd.fill(buf.data(), target, w)) return rc;
    for (size_t k = 0; k < w.rec_off.size(); k++) {
      const int c = w.rec_chr[k];
      if (n[c]++ == 0) first[c] = w.rec_pos[k];
      last[c] = w.rec_pos[k];
    }
  }
  for (int c = 0; c < n_chr; c++) {
    if (n_records) n_records[c] = n[c];
    if (first_pos) first_pos[c] = first[c];
    if (last_pos) last_pos[c] = last[c];
    if (ref_id) ref_id[c] = rd.ref_of_listed(c);
  }
  return 0;
}
