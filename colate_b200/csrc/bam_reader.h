// BAM input on the host (SAM/BAM format specification, sections 4.1 BGZF and 4.2 BAM): the BGZF block index, parallel
// inflation, the header, contig matching and the record walk.  The device decodes the records (kernels_bam.cu).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "bgzf.h"

namespace colate {

// Whole records of the listed contigs in one window of the inflated stream.  rec_off: offset of the record's block_size field
// in the window; rec_chr: index in the --chr list; rec_pos / rec_lseq: the record's pos and l_seq (row ranges, chunk sizes).
struct BamWindow {
  size_t n_bytes = 0;
  uint64_t ustart = 0;      // inflated-stream offset of the window's first byte
  std::vector<int64_t> rec_off;
  std::vector<int32_t> rec_chr, rec_pos, rec_lseq;
};

class BamReader : public BgzfFile {
 public:
  // Opens, indexes the BGZF blocks, parses the header and matches the listed contigs.  0 or COLATE_ERR_IO / _ARG (message set).
  int open(const std::string& path, int n_chr, const char* const* chr_names, int n_threads);
  // Inflates the next window into buf (capacity >= next_window_bytes(target)) and walks its records.
  int fill(uint8_t* buf, size_t target, BamWindow& w);
  int32_t ref_of_listed(int c) const { return ref_of_listed_[c]; }
  double walk_s = 0;   // wall time of the record walk so far (BgzfFile: index_s, inflate_s)

 private:
  int parse_header(int n_chr, const char* const* chr_names);
  std::vector<std::string> ref_names_;
  std::vector<int32_t> listed_of_ref_, ref_of_listed_;
  std::vector<char> done_;         // listed contigs whose records are behind us
  int cur_ = -1;                   // listed contig of the records being walked
  std::vector<std::string> listed_names_;
};

}  // namespace colate
