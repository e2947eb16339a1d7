// BGZF blocks on the host (SAM/BAM format specification 4.1), for the BAM (host_bam.cpp), BCF (host_bcf.cpp) and text VCF
// (host_vcf.cpp) readers.
#include "bgzf.h"

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

BgzfFile::~BgzfFile()
{
  if (map_) munmap((void*)map_, size_);
  if (fd_ >= 0) close(fd_);
}

bool contig_matches(const std::string& contig, const std::string& entry) { return contig == entry || contig == "chr" + entry; }

int BgzfFile::err(const std::string& what, uint64_t off, bool compressed)
{
  return fail(COLATE_ERR_IO, path_ + ": " + what + " at " + (compressed ? "byte offset " : "inflated byte offset ") + std::to_string(off));
}

int BgzfFile::open_bgzf(const std::string& path, const char* format, int threads)
{
  path_ = path;
  format_ = format;
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
  const std::string plain = "gzip member without the BGZF 'BC' extra subfield (plain gzip is not " + format_ + ")";
  uint64_t o = 0, u = 0;
  while (o < size_) {
    const uint8_t* p = map_ + o;
    if (size_ - o < 18) return err("truncated BGZF block header", o, true);
    if (p[0] != 31 || p[1] != 139 || p[2] != 8) return err("not a gzip member (BGZF block expected)", o, true);
    if (!(p[3] & 4)) return err(plain, o, true);
    const size_t xlen = rd16(p + 10);
    if (12 + xlen > size_ - o) return err("truncated BGZF block header", o, true);
    long bsize = -1;
    for (size_t x = 12; x + 4 <= 12 + xlen;) {
      const size_t slen = rd16(p + x + 2);
      if (p[x] == 66 && p[x + 1] == 67 && slen == 2 && x + 6 <= 12 + xlen) bsize = rd16(p + x + 4);
      x += 4 + slen;
    }
    if (bsize < 0) return err(plain, o, true);
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
  return 0;
}

// raw deflate of blocks [b0, b1) into dst (block b at dst + uoff(b) - uoff(b0)), n_threads threads; CRC32 and ISIZE checked
int BgzfFile::inflate_blocks(size_t b0, size_t b1, uint8_t* dst, bool scan_newlines)
{
  if (b1 <= b0) return 0;
  const double t0 = now_s();
  if (scan_newlines && block_nl_.size() < b1 - b0) block_nl_.resize(b1 - b0);
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
      } else if (scan_newlines) {
        std::vector<uint32_t>& nl = block_nl_[b - b0];
        nl.clear();
        for (const uint8_t* q = out; (q = (const uint8_t*)memchr(q, '\n', out + k.isize - q)); q++) nl.push_back((uint32_t)(q - out));
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

int BgzfFile::need_header_bytes(size_t n, size_t at)
{
  const uint8_t* p;
  size_t got;
  if (int rc = peek(n, &p, &got)) return rc;
  return got >= n ? 0 : err(format_ + " header runs past the end of the data", at, false);
}

int BgzfFile::peek(size_t n, const uint8_t** p, size_t* got)
{
  while (carry_.size() < n && next_block_ < blocks_.size()) {
    const size_t o = carry_.size();
    carry_.resize(o + blocks_[next_block_].isize);
    if (int rc = inflate_blocks(next_block_, next_block_ + 1, carry_.data() + o)) return rc;
    next_block_++;
  }
  *p = carry_.data();
  *got = std::min(n, carry_.size());
  return 0;
}

void BgzfFile::adopt(BgzfFile& o)
{
  std::swap(path_, o.path_);
  std::swap(format_, o.format_);
  std::swap(carry_, o.carry_);
  std::swap(carry_uoff_, o.carry_uoff_);
  std::swap(fd_, o.fd_);
  std::swap(map_, o.map_);
  std::swap(size_, o.size_);
  std::swap(blocks_, o.blocks_);
  std::swap(next_block_, o.next_block_);
  std::swap(index_s, o.index_s);
  std::swap(inflate_s, o.inflate_s);
  std::swap(n_threads, o.n_threads);
}

void BgzfFile::drop_header(size_t o)
{
  carry_.erase(carry_.begin(), carry_.begin() + o);
  carry_uoff_ = o;
}

size_t BgzfFile::next_window_bytes(size_t target) const
{
  size_t n = carry_.size();
  size_t b = next_block_;
  if (b == blocks_.size()) return n;
  do n += blocks_[b++].isize; while (b < blocks_.size() && n < target);
  return n;
}

int BgzfFile::fill_window(uint8_t* buf, size_t target, size_t* n_out, uint64_t* ustart)
{
  size_t b1 = next_block_;
  size_t n = carry_.size();
  if (b1 < blocks_.size()) do n += blocks_[b1++].isize; while (b1 < blocks_.size() && n < target);
  if (!carry_.empty()) memcpy(buf, carry_.data(), carry_.size());
  if (int rc = inflate_blocks(next_block_, b1, buf + carry_.size(), record_newlines)) return rc;
  if (record_newlines) {
    newlines.clear();
    for (size_t b = next_block_; b < b1; b++) {
      const int64_t base = (int64_t)(carry_.size() + (blocks_[b].uoff - blocks_[next_block_].uoff));
      for (uint32_t x : block_nl_[b - next_block_]) newlines.push_back(base + x);
    }
  }
  next_block_ = b1;
  *n_out = n;
  *ustart = carry_uoff_;
  return 0;
}

void BgzfFile::carry_tail(const uint8_t* buf, size_t o, size_t n, uint64_t ustart)
{
  carry_.assign(buf + o, buf + n);
  carry_uoff_ = ustart + o;
}

}  // namespace colate
