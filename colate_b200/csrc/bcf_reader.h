// BCF input on the host (VCF specification v4.3, section 6.3 "BCF2"): the magic, the header text (sample count, the dictionary
// index of GT) and the record walk by l_shared / l_indiv over BGZF windows (bgzf.h).  The device decodes the records
// (kernels_bcf.cu).  One file holds one chromosome: the reference opens <prefix>_chr<c>.bcf per --chr entry and never
// looks at CHROM, so a file whose records name more than one contig is refused.
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "bgzf.h"

namespace colate {

// Whole records of one window of the inflated stream.  rec_off: offset of the record's l_shared field in the window;
// rec_pos: its POS (0-based).  Text VCF (vcf_reader.h): rec_off is the offset of the line's first byte, and the window's
// lines end at the next line's offset or, for the last one, at text_end (the newline included, if there is one).
struct BcfWindow {
  size_t n_bytes = 0;
  uint64_t ustart = 0;      // inflated-stream offset of the window's first byte
  std::vector<int64_t> rec_off;
  std::vector<int32_t> rec_pos;
  int64_t text_end = 0;
};

// A per-chromosome genotype file as htslib's bcf_open reads it: BCF (BcfReader) or bgzipped text VCF (VcfReader).
class GenotypeReader : public BgzfFile {
 public:
  virtual ~GenotypeReader() = default;
  // Parses the header from the start of the inflated stream.  0 or COLATE_ERR_IO (message set).
  virtual int read_header() = 0;
  // Inflates the next window into buf (capacity >= next_window_bytes(target)) and walks its records: every record's CHROM
  // must be the file's first record's, its POS at least the previous record's (COLATE_ERR_ORDER).  At the end of the file a
  // file without records is refused.
  virtual int fill(uint8_t* buf, size_t target, BcfWindow& w) = 0;
  bool text = false;                           // VcfReader
  int n_sample = 0;
  int64_t n_records = 0;
  int32_t first_pos = -1, last_pos = -1;       // 0-based
  double walk_s = 0;                           // wall time of the record walk so far (BgzfFile: index_s, inflate_s)
};

class BcfReader : public GenotypeReader {
 public:
  // Opens, indexes the BGZF blocks and parses the header.  0 or COLATE_ERR_IO (message set).
  int open(const std::string& path, int n_threads);
  // The magic BCF\2\1 or BCF\2\2, the header text.
  int read_header() override;
  // GenotypeReader::fill; also every record's n_sample must be the header's.
  int fill(uint8_t* buf, size_t target, BcfWindow& w) override;
  int gt_key = -1;
  int32_t contig = -1;                         // CHROM of the records
};

// Opens a genotype file and picks its reader from the first inflated bytes, as htslib detects the format: BCF\2\1 or
// BCF\2\2 is BCF, "##fileformat=VCF" is text VCF, anything else is refused with BcfReader's message.  Files that are not
// BGZF (plain gzip, uncompressed BCF or VCF) are refused by BgzfFile::open_bgzf as before.
int open_genotypes(const std::string& path, int n_threads, std::unique_ptr<GenotypeReader>* out);

// Header text -> sample count (tabs after the #CHROM line's eighth column, less one for FORMAT) and GT's dictionary index (-1:
// no ##FORMAT=<ID=GT line) (host_bcf.cpp).
void header_text(const char* text, size_t n, int* n_sample, int* gt_key);

}  // namespace colate
