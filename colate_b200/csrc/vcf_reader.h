// Bgzipped text VCF input on the host (VCF specification v4.3, section 1): the header (the ## lines and the #CHROM line) and
// the walk over the record lines, which reads CHROM and POS only.  The device parses the rest of every line (k_vcf_decode,
// kernels_bcf.cu).  htslib's bcf_open reads such a file wherever the reference opens <prefix>_chr<c>.bcf, so the same
// per-chromosome rules as BCF apply: one contig per file, positions ascending.
#pragma once
#include <string>

#include "bcf_reader.h"

namespace colate {

class VcfReader : public GenotypeReader {
 public:
  VcfReader() { text = true; }
  // The ## lines up to the #CHROM line.  Refused: no #CHROM line, a #CHROM line whose first eight columns are not CHROM POS
  // ID REF ALT QUAL FILTER INFO, or that has no FORMAT and sample columns, or FORMAT and no sample; no ##FORMAT=<ID=GT line.
  int read_header() override;
  // GenotypeReader::fill over lines: rec_off = the line's first byte, text_end = the end of the window's last whole line.
  // Also refused: an empty line, a line ending in \r\n, a POS that is not a plain decimal in [0, 2^31 - 2].  A line cut by the
  // window's end starts the next window; the file's last line may lack its newline.
  int fill(uint8_t* buf, size_t target, BcfWindow& w) override;
  int gt_key = -1;       // dictionary index of GT, as BcfReader (only its presence matters here)
  std::string chrom;     // CHROM of the records

 private:
  int line(const uint8_t* buf, size_t o, size_t e, BcfWindow& w);
};

}  // namespace colate
