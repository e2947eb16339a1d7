// Genotype matrices on the host (DESIGN.md section 6l): the .snp / .bim SNP list split into --chr entries, the .ind / .fam IDs, the
// matrix layout and every refusal.  Nothing here touches a device: colate_geno_scan is this file's public face, and the device
// writer (kernels_geno.cu) starts from the same scan.
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cerrno>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "geno_reader.h"
#include "internal.h"

namespace colate {
namespace {

// contig c or chr<c>, and the numeric codes both formats use for the sex chromosomes
bool geno_contig_matches(const std::string& contig, const std::string& entry)
{
  return contig == entry || contig == "chr" + entry || (entry == "X" && contig == "23") || (entry == "Y" && contig == "24");
}

std::vector<std::string> fields(const char* b, const char* e)
{
  std::vector<std::string> f;
  while (b < e) {
    while (b < e && (*b == ' ' || *b == '\t' || *b == '\r')) b++;
    const char* s = b;
    while (b < e && !(*b == ' ' || *b == '\t' || *b == '\r')) b++;
    if (b > s) f.emplace_back(s, b - s);
  }
  return f;
}

// calls f(line number, fields) for every non-blank line; false stops
template <class F> bool each_line(const std::vector<char>& buf, F f)
{
  const char* p = buf.data();
  const char* end = p + buf.size();
  int64_t ln = 0;
  while (p < end) {
    const char* nl = (const char*)memchr(p, '\n', end - p);
    if (!nl) nl = end;
    ln++;
    std::vector<std::string> fl = fields(p, nl);
    if (!fl.empty() && !f(ln, fl)) return false;
    p = nl + 1;
  }
  return true;
}

std::string at(const std::string& path, int64_t ln) { return path + ", line " + std::to_string(ln) + ": "; }

}  // namespace

int geno_scan(const char* prefix, int format, int n_chr, const char* const* chr_names, GenoScan& g)
{
  if (!prefix || n_chr <= 0 || !chr_names || (format != COLATE_GENO_EIGENSTRAT && format != COLATE_GENO_PLINK))
    return fail(COLATE_ERR_ARG, "colate_geno_scan: bad arguments");
  std::vector<std::string> names;
  for (int c = 0; c < n_chr; c++) {
    if (!chr_names[c]) return fail(COLATE_ERR_ARG, "colate_geno_scan: bad arguments");
    names.emplace_back(chr_names[c]);
  }
  const bool eig = format == COLATE_GENO_EIGENSTRAT;
  const std::string P = prefix;
  const std::string f_snp = P + (eig ? ".snp" : ".bim"), f_ind = P + (eig ? ".ind" : ".fam");
  g = GenoScan();
  g.matrix = P + (eig ? ".geno" : ".bed");

  // individuals: .ind "ID sex population", .fam "FID IID father mother sex phenotype"
  std::vector<char> buf;
  if (!slurp(f_ind, buf)) return fail(COLATE_ERR_IO, "cannot read " + f_ind);
  std::string err;
  each_line(buf, [&](int64_t ln, const std::vector<std::string>& f) {
    if (f.size() < (eig ? 3u : 6u)) { err = at(f_ind, ln) + "expected " + (eig ? "3" : "6") + " fields, found " + std::to_string(f.size()); return false; }
    g.ids.push_back(eig ? f[0] : f[1]);
    return true;
  });
  if (!err.empty()) return fail(COLATE_ERR_IO, err);
  g.n_ind = (int64_t)g.ids.size();

  // SNPs: .snp "ID chr genetic_pos physical_pos allele_col5 allele_col6", .bim "chr ID cM position A1 A2"
  if (!slurp(f_snp, buf)) return fail(COLATE_ERR_IO, "cannot read " + f_snp);
  std::vector<std::vector<int64_t>> e_snp(n_chr);
  std::vector<std::vector<int32_t>> e_pos(n_chr);
  std::vector<std::vector<uint8_t>> e_al(n_chr);
  int err_code = COLATE_ERR_IO;
  int64_t s = 0;
  each_line(buf, [&](int64_t ln, const std::vector<std::string>& f) {
    if (f.size() < 6) {
      err = at(f_snp, ln) + (f.size() == 4 || f.size() == 5 ? "alleles missing (6 fields expected)" : "expected 6 fields, found " + std::to_string(f.size()));
      return false;
    }
    const std::string& chr = eig ? f[1] : f[0];
    errno = 0;
    char* end = nullptr;
    const long long v = strtoll(f[3].c_str(), &end, 10);
    if (*end || errno || v < 0 || v > INT_MAX) { err = at(f_snp, ln) + "physical position '" + f[3] + "' is not an integer in [0, 2^31)"; return false; }
    for (int c = 0; c < n_chr; c++) {
      if (!geno_contig_matches(chr, names[c])) continue;
      if (!e_pos[c].empty() && (int32_t)v < e_pos[c].back()) {
        err = at(f_snp, ln) + "SNP positions of --chr entry " + names[c] + " descend (" + std::to_string(e_pos[c].back()) + " then " + f[3] + ")";
        err_code = COLATE_ERR_ORDER;
        return false;
      }
      e_snp[c].push_back(s);
      e_pos[c].push_back((int32_t)v);
      // code 0 (EIGENSTRAT 2 copies of column 5, PLINK 00) and code 1 (0 copies of column 5, PLINK 11)
      e_al[c].push_back(f[4].size() == 1 ? (uint8_t)f[4][0] : 0);
      e_al[c].push_back(f[5].size() == 1 ? (uint8_t)f[5][0] : 0);
    }
    s++;
    return true;
  });
  if (!err.empty()) return fail(err_code, err);
  g.n_snp = s;
  g.entry_off.assign(1, 0);
  for (int c = 0; c < n_chr; c++) {
    g.snp.insert(g.snp.end(), e_snp[c].begin(), e_snp[c].end());
    g.pos.insert(g.pos.end(), e_pos[c].begin(), e_pos[c].end());
    g.allele.insert(g.allele.end(), e_al[c].begin(), e_al[c].end());
    g.entry_off.push_back((int64_t)g.snp.size());
  }

  // the matrix: layout from its first bytes, size from the dimensions
  const int fd = open(g.matrix.c_str(), O_RDONLY);
  if (fd < 0) return fail(COLATE_ERR_IO, "cannot read " + g.matrix);
  struct stat st;
  if (fstat(fd, &st) != 0) { close(fd); return fail(COLATE_ERR_IO, "cannot read " + g.matrix); }
  const int64_t size = (int64_t)st.st_size;
  char head[64] = {};
  const ssize_t nh = pread(fd, head, sizeof head - 1, 0);
  const int64_t packed_bytes = (g.n_ind + 3) / 4;
  int64_t want = 0;
  if (!eig) {
    if (nh < 3 || (uint8_t)head[0] != 0x6c || (uint8_t)head[1] != 0x1b) { close(fd); return fail(COLATE_ERR_IO, g.matrix + ": not a PLINK 1 .bed file (bad magic)"); }
    if ((uint8_t)head[2] == 0x00) { close(fd); return fail(COLATE_ERR_IO, g.matrix + ": individual-major .bed files are not supported (write it SNP-major: plink --make-bed)"); }
    if ((uint8_t)head[2] != 0x01) { close(fd); return fail(COLATE_ERR_IO, g.matrix + ": not a PLINK 1 .bed file (bad magic)"); }
    g.kind = GENO_BED;
    g.data_off = 3;
    g.row_bytes = packed_bytes;
    want = 3 + g.n_snp * g.row_bytes;
  } else if (nh >= 5 && memcmp(head, "TGENO", 5) == 0) {
    close(fd);
    return fail(COLATE_ERR_IO, g.matrix + ": transposed packed files (TGENO) are not supported (convert with convertf to packed EIGENSTRAT)");
  } else if (nh >= 5 && memcmp(head, "GENO ", 5) == 0) {
    // EIGENSOFT packedancestrymap: records of max(48, ceil(nind / 4)) bytes, the first one "GENO nind nsnp indhash snphash"
    long long hi = -1, hs = -1;
    if (sscanf(head + 5, "%lld %lld", &hi, &hs) != 2) { close(fd); return fail(COLATE_ERR_IO, g.matrix + ": malformed GENO header"); }
    if (hi != g.n_ind || hs != g.n_snp) {
      close(fd);
      return fail(COLATE_ERR_IO, g.matrix + ": the header counts " + std::to_string(hi) + " individuals and " + std::to_string(hs) + " SNPs, " + f_ind +
                                     " lists " + std::to_string(g.n_ind) + " and " + f_snp + " " + std::to_string(g.n_snp));
    }
    g.kind = GENO_PACKED;
    g.row_bytes = packed_bytes > 48 ? packed_bytes : 48;
    g.data_off = g.row_bytes;
    want = (g.n_snp + 1) * g.row_bytes;
  } else {
    g.kind = GENO_TEXT;
    g.row_bytes = g.n_ind + 1;
    want = g.n_snp * g.row_bytes;
  }
  if (size != want) {
    close(fd);
    return fail(COLATE_ERR_IO, g.matrix + ": " + std::to_string(size) + " bytes, but " + std::to_string(g.n_snp) + " SNPs x " + std::to_string(g.n_ind) +
                                   " individuals take " + std::to_string(want) + " in this layout");
  }
  // text: nind digits of {0, 1, 2, 9} and a newline per SNP
  if (g.kind == GENO_TEXT && size > 0) {
    void* m = mmap(nullptr, (size_t)size, PROT_READ, MAP_PRIVATE, fd, 0);
    if (m == MAP_FAILED) { close(fd); return fail(COLATE_ERR_IO, "cannot read " + g.matrix); }
    const uint8_t* p = (const uint8_t*)m;
    for (int64_t r = 0; r < g.n_snp && err.empty(); r++) {
      const uint8_t* row = p + r * g.row_bytes;
      if (row[g.n_ind] != '\n') err = at(g.matrix, r + 1) + "expected " + std::to_string(g.n_ind) + " calls and a newline";
      for (int64_t k = 0; k < g.n_ind && err.empty(); k++)
        if (!(row[k] == '0' || row[k] == '1' || row[k] == '2' || row[k] == '9'))
          err = at(g.matrix, r + 1) + "call '" + std::string(1, (char)row[k]) + "' of individual " + std::to_string(k + 1) + " is not 0, 1, 2 or 9";
    }
    munmap(m, (size_t)size);
  }
  close(fd);
  if (!err.empty()) return fail(COLATE_ERR_IO, err);
  return 0;
}

}  // namespace colate

extern "C" int colate_geno_scan(const char* prefix, int format, int n_chr, const char* const* chr_names, int64_t* n_snp, int64_t* n_ind,
                                int64_t* entry_snps, int32_t* kind)
{
  colate::GenoScan g;
  if (int rc = colate::geno_scan(prefix, format, n_chr, chr_names, g)) return rc;
  if (n_snp) *n_snp = g.n_snp;
  if (n_ind) *n_ind = g.n_ind;
  if (kind) *kind = g.kind;
  if (entry_snps)
    for (int c = 0; c < n_chr; c++) entry_snps[c] = g.entry_off[c + 1] - g.entry_off[c];
  return 0;
}
