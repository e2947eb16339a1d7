// BGZF (SAM/BAM format specification 4.1) on the host, shared by the BAM, the BCF and the text VCF readers: the file is memory-mapped, its
// blocks are indexed from their headers and footers, windows of blocks are inflated with raw zlib on a thread pool straight
// into the caller's (pinned) buffer, and every block's CRC32 and ISIZE is checked.  A window starts with the bytes the
// previous one left over (a record that straddles the window end), so the container readers only ever see whole records.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

namespace colate {

struct BgzfBlock {
  uint64_t coff;      // byte offset of the block in the file
  uint32_t data;      // offset of the deflate data inside the block
  uint32_t clen;      // deflate data bytes
  uint32_t crc, isize;
  uint64_t uoff;      // offset of the block's first inflated byte in the inflated stream
};

// A --chr entry <name> reads the contig <name> or chr<name> (bam_parser, htslib.cpp:388): BAM, and whole-genome BCF / VCF.
bool contig_matches(const std::string& contig, const std::string& entry);

class BgzfFile {
 public:
  ~BgzfFile();
  // Opens and indexes the blocks.  `format` names the container in messages ("BAM", "BCF").  0 or COLATE_ERR_IO (message set).
  int open_bgzf(const std::string& path, const char* format, int n_threads);
  // Bytes the next window needs: the carried bytes plus whole blocks up to at least `target` inflated bytes (at least one
  // block).  0: nothing is left.
  size_t next_window_bytes(size_t target) const;
  // Copies the carried bytes to buf and inflates the blocks of the next window after them (capacity >= next_window_bytes).
  // *n: bytes in buf; *ustart: inflated-stream offset of buf[0].
  int fill_window(uint8_t* buf, size_t target, size_t* n, uint64_t* ustart);
  // The window's bytes [o, n) are an incomplete record: they start the next window.
  void carry_tail(const uint8_t* buf, size_t o, size_t n, uint64_t ustart);
  bool at_end() const { return next_block_ == blocks_.size(); }
  // Inflates blocks until the first n bytes of the stream (or all of it, if shorter) are held: *p, *got.  For sniffing the format.
  int peek(size_t n, const uint8_t** p, size_t* got);
  // Takes over o's file, index and carried bytes (o is left closed).  A format sniffed on one reader is read by another.
  void adopt(BgzfFile& o);
  uint64_t inflated_size() const { return blocks_.empty() ? 0 : blocks_.back().uoff + blocks_.back().isize; }
  // "<path>: <what> at [inflated ]byte offset <off>" as COLATE_ERR_IO
  int err(const std::string& what, uint64_t off, bool compressed);
  double index_s = 0, inflate_s = 0;   // wall time of the phases so far
  int n_threads = 1;
  // Text readers: fill_window also lists the newlines of the blocks it inflates (window offsets, ascending), each inflate thread
  // scanning the block it has just inflated while the block is in cache.  The carried bytes at the window's start are not scanned.
  bool record_newlines = false;
  std::vector<int64_t> newlines;

 protected:
  // the first n inflated bytes in carry_ (a header is parsed from there); `at` names the field that needs them
  int need_header_bytes(size_t n, size_t at);
  // the header is parsed: drop its o bytes from carry_
  void drop_header(size_t o);
  int inflate_blocks(size_t b0, size_t b1, uint8_t* dst, bool scan_newlines = false);
  std::string path_, format_;
  std::vector<uint8_t> carry_;     // inflated bytes not yet consumed (header, then a partial record)
  uint64_t carry_uoff_ = 0;        // inflated-stream offset of carry_[0]

 private:
  int fd_ = -1;
  const uint8_t* map_ = nullptr;
  size_t size_ = 0;
  std::vector<BgzfBlock> blocks_;
  size_t next_block_ = 0;
  std::vector<std::vector<uint32_t>> block_nl_;   // inflate_blocks(scan_newlines): '\n' offsets in block b0 + i
};

}  // namespace colate
