// BCF input on the host (VCF specification v4.3, section 6.3 "BCF2"): the magic, the header text (sample count, the dictionary
// index of GT) and the record walk by l_shared / l_indiv over BGZF windows (bgzf.h).  The device decodes the records
// (kernels_bcf.cu).  One file holds one chromosome: the reference opens <prefix>_chr<c>.bcf per --chr entry and never
// looks at CHROM, so a file whose records name more than one contig is refused.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "bgzf.h"

namespace colate {

// Whole records of one window of the inflated stream.  rec_off: offset of the record's l_shared field in the window;
// rec_pos: its POS (0-based).
struct BcfWindow {
  size_t n_bytes = 0;
  uint64_t ustart = 0;      // inflated-stream offset of the window's first byte
  std::vector<int64_t> rec_off;
  std::vector<int32_t> rec_pos;
};

class BcfReader : public BgzfFile {
 public:
  // Opens, indexes the BGZF blocks and parses the header.  0 or COLATE_ERR_IO (message set).
  int open(const std::string& path, int n_threads);
  // Inflates the next window into buf (capacity >= next_window_bytes(target)) and walks its records: every record's n_sample
  // must be the header's, its CHROM the file's first record's, its POS at least the previous record's (COLATE_ERR_ORDER).
  // At the end of the file a file without records is refused.
  int fill(uint8_t* buf, size_t target, BcfWindow& w);
  int n_sample = 0, gt_key = -1;
  int32_t contig = -1;                         // CHROM of the records
  int64_t n_records = 0;
  int32_t first_pos = -1, last_pos = -1;       // 0-based
  double walk_s = 0;                           // wall time of the record walk so far (BgzfFile: index_s, inflate_s)
};

}  // namespace colate
