// The make_tmp row word (colate_maketmp_word, include/colate_b200.h): what the row filters of maketmp_bam (coal.cpp:2568,
// 2584-2587) and maketmp_vcf (coal.cpp:2365, 2381-2395) need from a .mut row, computed from the mutation type exactly as
// parse_mut_line_fields leaves it in type[16] (the first 15 characters, "NN" for a longer type, "NA" without one).  Shared by
// the host reader (host_misc.cpp) and the device ingest (kernels_ingest.cu), so both paths give the same word.
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define COLATE_HD __host__ __device__ __forceinline__
#else
#define COLATE_HD inline
#endif

namespace colate {

constexpr uint32_t MKT_VCF = 1u;   // maketmp_vcf filter: type exactly "a/d", a in {A,C,G,T,0}, d in {A,C,G,T,1}
constexpr uint32_t MKT_BAM = 2u;   // maketmp_bam filter: one-letter a in {A,C,G,T,0}, '/', a non-empty derived string
constexpr uint32_t MKT_ONE = 4u;   // the derived string is one letter

// type: NUL-terminated, at most 15 characters (type[16] of parse_mut_line_fields).  Both filters also need "not flipped, one branch".
// byte 1 = ancestral letter type[0], byte 2 = first derived letter type[2]; 0 when the row passes neither filter.
COLATE_HD uint32_t maketmp_word(int flipped, int n_branch, const char* type)
{
  if (flipped != 0 || n_branch != 1) return 0;
  const char a = type[0];
  if (!(a == 'A' || a == 'C' || a == 'G' || a == 'T' || a == '0')) return 0;
  if (type[1] != '/' || type[2] == '\0') return 0;       // strchr(type, '/') - type == 1 and a non-empty derived string
  const char d = type[2];
  const bool one = type[3] == '\0';
  const bool vcf = one && (d == 'A' || d == 'C' || d == 'G' || d == 'T' || d == '1');
  return MKT_BAM | (vcf ? MKT_VCF : 0u) | (one ? MKT_ONE : 0u) | ((uint32_t)(unsigned char)a << 8) | ((uint32_t)(unsigned char)d << 16);
}

}  // namespace colate
