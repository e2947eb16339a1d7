// Genotype matrices (DESIGN.md section 6l): EIGENSTRAT (P.geno packed or text, P.snp, P.ind) and SNP-major PLINK 1 (P.bed, P.bim,
// P.fam), read on the host into what make_tmp needs -- per --chr entry the SNPs of its contig in file order (position, the two
// allele letters), the individuals' IDs and where each SNP's row of 2-bit (or text) calls sits in the matrix file.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

namespace colate {

enum { GENO_PACKED = 0, GENO_TEXT = 1, GENO_BED = 2 };

struct GenoScan {
  int kind = GENO_PACKED;
  int64_t n_snp = 0, n_ind = 0;
  std::string matrix;                   // P.geno or P.bed
  int64_t data_off = 0, row_bytes = 0;  // SNP s's row of calls: bytes [data_off + s * row_bytes, + row_bytes)
  std::vector<std::string> ids;         // .ind column 1 / .fam IID, in file order
  // the SNPs of --chr entry e: [entry_off[e], entry_off[e + 1]) of the arrays below, in file order
  std::vector<int64_t> entry_off;
  std::vector<int64_t> snp;             // index in the .snp / .bim file
  std::vector<int32_t> pos;             // physical position (non-descending within an entry)
  std::vector<uint8_t> allele;          // 2 per SNP: the allele a homozygous call of code 0 / 1 means, the letter or 0 if not one letter
};

// Every host check of DESIGN.md section 6l: file dimensions, layout, refused variants, SNP order per entry.  0 or a negative status.
int geno_scan(const char* prefix, int format, int n_chr, const char* const* chr_names, GenoScan& g);

// The 2-bit call code of the device rule: 0 homozygous for allele[0], 1 homozygous for allele[1], 2 heterozygous, 3 missing.
#if defined(__CUDACC__)
__host__ __device__ __forceinline__
#else
inline
#endif
uint32_t geno_code(const uint8_t* row, int64_t k, int kind)
{
  if (kind == GENO_TEXT) {
    const uint32_t ch = row[k];
    return ch == '2' ? 0u : ch == '0' ? 1u : ch == '1' ? 2u : 3u;
  }
  const uint32_t b = row[k >> 2];
  if (kind == GENO_PACKED) return (0xC9u >> (2 * ((b >> (6 - 2 * (k & 3))) & 3u))) & 3u;   // 0 -> 1, 1 -> 2, 2 -> 0, 3 -> 3
  return (0x6Cu >> (2 * ((b >> (2 * (k & 3))) & 3u))) & 3u;                                 // 00 -> 0, 01 -> 3, 10 -> 2, 11 -> 1
}

}  // namespace colate
