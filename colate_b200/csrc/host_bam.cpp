// BAM input, host side: BGZF (SAM/BAM format specification 4.1) and the BAM container (4.2).  The reference reads BAM
// through htslib (bam_parser, include/vcf/htslib.cpp); of a record its pileup uses pos, mapq, l_seq, the packed sequence and
// the qualities, which the device decodes (kernels_bam.cu).  The host finds the blocks, inflates them in parallel, parses the
// header, matches the --chr list and walks the records by block_size to find their boundaries and contigs.
#include "bam_reader.h"

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/time.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cstring>
#include <mutex>
#include <thread>

#include "internal.h"

namespace colate {

namespace {
inline uint16_t rd16(const uint8_t* p) { return (uint16_t)(p[0] | p[1] << 8); }
inline uint32_t rd32(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }
inline double now_s() { timeval tv; gettimeofday(&tv, nullptr); return tv.tv_sec + 1e-6 * tv.tv_usec; }
}  // namespace

BamReader::~BamReader()
{
  if (map_) munmap((void*)map_, size_);
  if (fd_ >= 0) close(fd_);
}

int BamReader::err(const std::string& what, uint64_t off, bool compressed)
{
  return fail(COLATE_ERR_IO, path_ + ": " + what + " at " + (compressed ? "byte offset " : "inflated byte offset ") + std::to_string(off));
}

int BamReader::open(const std::string& path, int n_chr, const char* const* chr_names, int threads)
{
  path_ = path;
  n_threads = std::max(1, threads);
  const double t0 = now_s();
  fd_ = ::open(path.c_str(), O_RDONLY);
  if (fd_ < 0) return fail(COLATE_ERR_IO, "cannot open " + path);
  struct stat st;
  if (fstat(fd_, &st) != 0) return fail(COLATE_ERR_IO, "cannot stat " + path);
  size_ = (size_t)st.st_size;
  if (size_ > 0) {
    void* m = mmap(nullptr, size_, PROT_READ, MAP_PRIVATE, fd_, 0);
    if (m == MAP_FAILED) return fail(COLATE_ERR_IO, "cannot map " + path);
    map_ = (const uint8_t*)m;
    madvise(m, size_, MADV_SEQUENTIAL);
  }
  // block index: every header gives BSIZE, every footer ISIZE; the inflated offsets are their prefix sum
  uint64_t o = 0, u = 0;
  while (o < size_) {
    const uint8_t* p = map_ + o;
    if (size_ - o < 18) return err("truncated BGZF block header", o, true);
    if (p[0] != 31 || p[1] != 139 || p[2] != 8) return err("not a gzip member (BGZF block expected)", o, true);
    if (!(p[3] & 4)) return err("gzip member without the BGZF 'BC' extra subfield (plain gzip is not BAM)", o, true);
    const size_t xlen = rd16(p + 10);
    if (12 + xlen > size_ - o) return err("truncated BGZF block header", o, true);
    long bsize = -1;
    for (size_t x = 12; x + 4 <= 12 + xlen;) {
      const size_t slen = rd16(p + x + 2);
      if (p[x] == 66 && p[x + 1] == 67 && slen == 2 && x + 6 <= 12 + xlen) bsize = rd16(p + x + 4);
      x += 4 + slen;
    }
    if (bsize < 0) return err("gzip member without the BGZF 'BC' extra subfield (plain gzip is not BAM)", o, true);
    const size_t total = (size_t)bsize + 1;
    if (total < 12 + xlen + 8) return err("BGZF block size smaller than its header", o, true);
    if (total > size_ - o) return err("truncated BGZF block", o, true);
    BgzfBlock b;
    b.coff = o;
    b.data = (uint32_t)(12 + xlen);
    b.clen = (uint32_t)(total - 12 - xlen - 8);
    b.crc = rd32(p + total - 8);
    b.isize = rd32(p + total - 4);
    b.uoff = u;
    if (b.isize > 65536) return err("BGZF block with ISIZE over 64 KiB", o, true);
    blocks_.push_back(b);
    u += b.isize;
    o += total;
  }
  index_s += now_s() - t0;
  return parse_header(n_chr, chr_names);
}

// raw deflate of blocks [b0, b1) into dst (block b at dst + uoff(b) - uoff(b0)), n_threads threads; CRC32 and ISIZE checked
int BamReader::inflate_blocks(size_t b0, size_t b1, uint8_t* dst)
{
  if (b1 <= b0) return 0;
  const double t0 = now_s();
  std::atomic<size_t> next{b0};
  std::mutex mu;
  size_t bad = SIZE_MAX;
  std::string bad_what;
  auto work = [&]() {
    z_stream s;
    memset(&s, 0, sizeof s);
    if (inflateInit2(&s, -15) != Z_OK) { std::lock_guard<std::mutex> g(mu); if (b0 < bad) { bad = b0; bad_what = "zlib inflateInit2 failed"; } return; }
    uint8_t dummy;
    for (size_t b; (b = next.fetch_add(1)) < b1;) {
      const BgzfBlock& k = blocks_[b];
      uint8_t* out = dst + (k.uoff - blocks_[b0].uoff);
      inflateReset(&s);
      s.next_in = (Bytef*)(map_ + k.coff + k.data);
      s.avail_in = k.clen;
      s.next_out = k.isize ? out : &dummy;
      s.avail_out = k.isize;
      const int r = inflate(&s, Z_FINISH);
      const char* what = nullptr;
      if (r != Z_STREAM_END) what = (r == Z_BUF_ERROR && s.avail_out == 0) ? "BGZF block inflates to more than its ISIZE" : "corrupt deflate data in BGZF block";
      else if (s.avail_out != 0) what = "BGZF block inflates to less than its ISIZE";
      else if (crc32(0, out, k.isize) != k.crc) what = "BGZF block CRC32 mismatch";
      if (what) {
        std::lock_guard<std::mutex> g(mu);
        if (b < bad) { bad = b; bad_what = what; }
      }
    }
    inflateEnd(&s);
  };
  const int nt = (int)std::min<size_t>(n_threads, b1 - b0);
  std::vector<std::thread> th;
  for (int t = 1; t < nt; t++) th.emplace_back(work);
  work();
  for (auto& t : th) t.join();
  inflate_s += now_s() - t0;
  if (bad != SIZE_MAX) return err(bad_what, blocks_[bad].coff, true);
  return 0;
}

// the first n inflated bytes in carry_ (the header is parsed from there); `at` names the field that needs them
int BamReader::need_header_bytes(size_t n, size_t at)
{
  while (carry_.size() < n && next_block_ < blocks_.size()) {
    const size_t o = carry_.size();
    carry_.resize(o + blocks_[next_block_].isize);
    if (int rc = inflate_blocks(next_block_, next_block_ + 1, carry_.data() + o)) return rc;
    next_block_++;
  }
  return carry_.size() >= n ? 0 : err("BAM header runs past the end of the data", at, false);
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
  carry_.erase(carry_.begin(), carry_.begin() + o);
  carry_uoff_ = o;
  // --chr entry <name> = header contig <name> or chr<name> (bam_parser, htslib.cpp:388)
  listed_of_ref_.assign(n_ref, -1);
  ref_of_listed_.assign(n_chr, -1);
  done_.assign(n_chr, 0);
  for (int c = 0; c < n_chr; c++) {
    const std::string a = chr_names[c], b = "chr" + a;
    listed_names_.push_back(a);
    for (int32_t r = 0; r < n_ref; r++) {
      if (ref_names_[r] != a && ref_names_[r] != b) continue;
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

size_t BamReader::next_window_bytes(size_t target) const
{
  size_t n = carry_.size();
  size_t b = next_block_;
  if (b == blocks_.size()) return n;
  do n += blocks_[b++].isize; while (b < blocks_.size() && n < target);
  return n;
}

int BamReader::fill(uint8_t* buf, size_t target, BamWindow& w)
{
  size_t b1 = next_block_;
  size_t n = carry_.size();
  if (b1 < blocks_.size()) do n += blocks_[b1++].isize; while (b1 < blocks_.size() && n < target);
  if (!carry_.empty()) memcpy(buf, carry_.data(), carry_.size());
  if (int rc = inflate_blocks(next_block_, b1, buf + carry_.size())) return rc;
  next_block_ = b1;
  const double t0 = now_s();
  w.n_bytes = n;
  w.ustart = carry_uoff_;
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
  carry_.assign(buf + o, buf + n);
  carry_uoff_ = w.ustart + o;
  walk_s += now_s() - t0;
  if (next_block_ == blocks_.size() && !carry_.empty()) return err("BAM record runs past the end of the data", carry_uoff_, false);
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
