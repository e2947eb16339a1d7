// BAM input on the host (SAM/BAM format specification, sections 4.1 BGZF and 4.2 BAM): the BGZF block index, parallel
// inflation, the header, contig matching and the record walk.  The device decodes the records (kernels_bam.cu).
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

// Whole records of the listed contigs in one window of the inflated stream.  rec_off: offset of the record's block_size field
// in the window; rec_chr: index in the --chr list; rec_pos / rec_lseq: the record's pos and l_seq (row ranges, chunk sizes).
struct BamWindow {
  size_t n_bytes = 0;
  uint64_t ustart = 0;      // inflated-stream offset of the window's first byte
  std::vector<int64_t> rec_off;
  std::vector<int32_t> rec_chr, rec_pos, rec_lseq;
};

class BamReader {
 public:
  ~BamReader();
  // Opens, indexes the BGZF blocks, parses the header and matches the listed contigs.  0 or COLATE_ERR_IO / _ARG (message set).
  int open(const std::string& path, int n_chr, const char* const* chr_names, int n_threads);
  // Bytes the next window needs: the carried partial record plus whole blocks up to at least `target` inflated bytes
  // (at least one block).  0: nothing is left.
  size_t next_window_bytes(size_t target) const;
  // Inflates the next window into buf (capacity >= next_window_bytes(target)) and walks its records.
  int fill(uint8_t* buf, size_t target, BamWindow& w);
  int32_t ref_of_listed(int c) const { return ref_of_listed_[c]; }
  double index_s = 0, inflate_s = 0, walk_s = 0;   // wall time of the phases so far
  int n_threads = 1;

 private:
  int err(const std::string& what, uint64_t off, bool compressed);
  int inflate_blocks(size_t b0, size_t b1, uint8_t* dst);
  int need_header_bytes(size_t n, size_t at);
  int parse_header(int n_chr, const char* const* chr_names);
  std::string path_;
  int fd_ = -1;
  const uint8_t* map_ = nullptr;
  size_t size_ = 0;
  std::vector<BgzfBlock> blocks_;
  size_t next_block_ = 0;
  std::vector<uint8_t> carry_;     // inflated bytes not yet consumed (header, then a partial record)
  uint64_t carry_uoff_ = 0;        // inflated-stream offset of carry_[0]
  std::vector<std::string> ref_names_;
  std::vector<int32_t> listed_of_ref_, ref_of_listed_;
  std::vector<char> done_;         // listed contigs whose records are behind us
  int cur_ = -1;                   // listed contig of the records being walked
  std::vector<std::string> listed_names_;
};

}  // namespace colate
