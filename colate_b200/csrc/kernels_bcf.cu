// BCF records decoded on the device, then resolved against the .mut rows (the decoder half of parse_vcfvcf, coal.cpp:997-1137).
// The host (host_bcf.cpp) inflates the BGZF blocks of one window of the file into pinned memory and finds the record boundaries;
// k_bcf_decode reduces every record to 12 bytes (position, the codes of its first two alleles, the GT allele sum, the biallelic
// flag), which stay resident for the whole file while the raw bytes stream through (a whole-genome file: the records of every
// --chr contig, each contig's kept apart); k_bcf_rows gives every .mut row of the
// chromosome its (AAF, DAF) straight in the row-count columns of a target slot, a reference slot or both.  Window n+1 is inflated on the host while window n
// is on the device.  Bgzipped text VCF (host_vcf.cpp) takes the same path with k_vcf_decode in place of k_bcf_decode: the
// format is detected from the file's first inflated bytes (open_genotypes), as htslib's bcf_open does.
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "device.cuh"
#include "vcf_reader.h"

using namespace colate;

namespace {

// first error of a file: (inflated offset of the record << 3) | kind, atomicMin over the records
enum : unsigned { kErrNoGT = 1, kErrGTValue = 2, kErrGTLength = 3, kErrFields = 4, kErrGTType = 5 };

__device__ __forceinline__ uint32_t ld32u(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }

// typed values (VCF v4.3 6.3.3): descriptor byte = size << 4 | type, size 15 = a typed integer with the size follows.
// Element bytes by type as htslib's bcf_type_shift: 0 missing (flags: size 0), 1 int8, 2 int16, 3 int32, 5 float, 7 char.
struct Cur {
  const uint8_t* p;
  const uint8_t* e;
  bool bad;
};
__device__ __forceinline__ int type_shift(int t) { return t == 2 ? 1 : (t == 3 || t == 5) ? 2 : (t == 4 || t == 6) ? 3 : t <= 7 ? 0 : -1; }
__device__ __forceinline__ bool rd_int(Cur& c, int t, int64_t* v)
{
  const int nb = t == 1 ? 1 : t == 2 ? 2 : t == 3 ? 4 : 0;
  if (!nb || c.e - c.p < nb) return c.bad = true, false;
  *v = nb == 1 ? (int64_t)(int8_t)c.p[0] : nb == 2 ? (int64_t)(int16_t)(c.p[0] | c.p[1] << 8) : (int64_t)(int32_t)ld32u(c.p);
  c.p += nb;
  return true;
}
__device__ __forceinline__ bool descr(Cur& c, int* type, int64_t* size)
{
  if (c.p >= c.e) return c.bad = true, false;
  const uint8_t b = *c.p++;
  *type = b & 15;
  *size = b >> 4;
  if (type_shift(*type) < 0) return c.bad = true, false;
  if (*size == 15) {
    if (c.p >= c.e) return c.bad = true, false;
    const uint8_t b2 = *c.p++;
    if ((b2 >> 4) != 1 || !rd_int(c, b2 & 15, size) || *size < 0) return c.bad = true, false;
  }
  return true;
}
__device__ __forceinline__ bool skip_typed(Cur& c)
{
  int t;
  int64_t n;
  if (!descr(c, &t, &n)) return false;
  const int64_t nb = n << type_shift(t);
  if (c.e - c.p < nb) return c.bad = true, false;
  c.p += nb;
  return true;
}
__device__ __forceinline__ bool typed_int(Cur& c, int64_t* v)
{
  int t;
  int64_t n;
  if (!descr(c, &t, &n)) return false;
  if (n != 1) return c.bad = true, false;
  return rd_int(c, t, v);
}

// one GT byte (int8): allele index (b >> 1) - 1; b < 2 (missing allele '.'), 0x80 (missing), 0x81 (vector end) or any other
// negative value is refused
__device__ __forceinline__ void gt_byte(uint32_t b, uint32_t& sum, uint32_t& mx, bool& bad)
{
  bad |= b >= 0x80u || b < 2u;
  const uint32_t u = b >> 1;
  sum += u;
  mx = max(mx, u);
}
// four GT bytes at once: the phased bit of each byte must not reach the byte below it
__device__ __forceinline__ void gt_word(uint32_t w, uint32_t& sum, uint32_t& mx4, bool& bad)
{
  bad |= (w & 0x80808080u) != 0;
  const uint32_t u = (w >> 1) & 0x7f7f7f7fu;
  bad |= __vcmpeq4(u, 0u) != 0;
  sum = __dp4a(u, 0x01010101u, sum);
  mx4 = __vmaxu4(mx4, u);
}

// warp = record.  raw + rec_off[k]: l_shared, l_indiv, then the shared part (CHROM, POS, rlen, QUAL, n_allele << 16 | n_info,
// n_fmt << 24 | n_sample, ID, the alleles, FILTER, the INFO pairs) and the per-sample part (n_fmt fields: key, typed type, the
// values of all samples).  The shared part is walked by every lane alike; the lanes split the GT values.  The GT field's
// vector length must be the same in every record of the file (*nhap_state: the first record's n_hap, -1 before it).
__global__ void k_bcf_decode(int64_t n, const uint8_t* __restrict__ raw, const int64_t* __restrict__ rec_off, uint64_t ustart, int gt_key,
                             BcfCol* __restrict__ cols, int32_t* __restrict__ nhap_state, unsigned long long* __restrict__ err)
{
  const int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (k >= n) return;
  const uint8_t* r = raw + rec_off[k];
  const uint32_t l_shared = ld32u(r), l_indiv = ld32u(r + 4);
  const uint8_t* s = r + 8;
  const int32_t pos = (int32_t)ld32u(s + 4);
  const uint32_t n_allele = ld32u(s + 16) >> 16, n_info = ld32u(s + 16) & 0xffffu;
  const uint32_t n_fmt = ld32u(s + 20) >> 24, n_sample = ld32u(s + 20) & 0xffffffu;
  unsigned kind = 0;
  Cur c{s + 24, s + l_shared, false};
  uint32_t code0 = 0, code1 = 0;
  skip_typed(c);                                                   // ID
  for (uint32_t i = 0; i < n_allele && !c.bad; i++) {
    int t;
    int64_t len;
    if (!descr(c, &t, &len)) break;
    const int64_t nb = len << type_shift(t);
    if (c.e - c.p < nb) { c.bad = true; break; }
    const uint32_t cd = len == 0 ? 0u : len == 1 ? c.p[0] : 0xffu;
    if (i == 0) code0 = cd;
    if (i == 1) code1 = cd;
    c.p += nb;
  }
  if (!c.bad) skip_typed(c);                                       // FILTER
  for (uint32_t i = 0; i < n_info && !c.bad; i++) {
    int64_t key;
    if (typed_int(c, &key)) skip_typed(c);
  }
  // FORMAT fields: the GT one
  const uint8_t* gp = nullptr;
  int gt_type = 0;
  int64_t gt_len = 0;
  Cur f{s + l_shared, s + l_shared + l_indiv, c.bad};
  for (uint32_t i = 0; i < n_fmt && !f.bad; i++) {
    int64_t key, size;
    int t;
    if (!typed_int(f, &key) || !descr(f, &t, &size)) break;
    const int64_t nb = ((int64_t)n_sample * size) << type_shift(t);
    if (f.e - f.p < nb) { f.bad = true; break; }
    if (key == gt_key && !gp) { gp = f.p; gt_type = t; gt_len = size; }
    f.p += nb;
  }
  const int64_t n_hap = (int64_t)n_sample * gt_len;
  if (f.bad) kind = kErrFields;
  else if (!gp || n_hap == 0) kind = kErrNoGT;
  else if (gt_type < 1 || gt_type > 3) kind = kErrGTType;
  uint32_t sum = 0, mx = 0;
  bool bad = false;
  if (!kind) {
    if (gt_type == 1) {
      // 16-byte aligned body in uint4 loads, head and tail bytes one per lane
      const uint8_t* end = gp + n_hap;
      const uint8_t* body = (const uint8_t*)(((uintptr_t)gp + 15) & ~(uintptr_t)15);
      if (body > end) body = end;
      const uint8_t* bend = body + ((end - body) & ~(int64_t)15);
      for (int64_t i = lane; i < body - gp; i += 32) gt_byte(gp[i], sum, mx, bad);
      for (int64_t i = lane; i < end - bend; i += 32) gt_byte(bend[i], sum, mx, bad);
      uint32_t mx4 = 0;
      const uint4* v = (const uint4*)body;
      const int64_t nv = (bend - body) >> 4;
      for (int64_t j = lane; j < nv; j += 32) {
        const uint4 x = v[j];
        gt_word(x.x, sum, mx4, bad); gt_word(x.y, sum, mx4, bad); gt_word(x.z, sum, mx4, bad); gt_word(x.w, sum, mx4, bad);
      }
      mx = max(mx, max(max(mx4 & 0xffu, (mx4 >> 8) & 0xffu), max((mx4 >> 16) & 0xffu, mx4 >> 24)));
    } else {
      // int16 / int32: missing (INT_MIN), vector end (INT_MIN + 1) and '.' (0 / 1) are all below 2
      for (int64_t i = lane; i < n_hap; i += 32) {
        const uint8_t* q = gp + (i << (gt_type - 1));
        const int32_t x = gt_type == 2 ? (int32_t)(int16_t)(q[0] | q[1] << 8) : (int32_t)ld32u(q);
        bad |= x < 2;
        const uint32_t u = (uint32_t)(x >> 1);
        sum += u;
        mx = max(mx, u);
      }
    }
  }
  sum = __reduce_add_sync(0xffffffffu, sum);
  mx = __reduce_max_sync(0xffffffffu, mx);
  bad = __any_sync(0xffffffffu, bad);
  if (lane != 0) return;
  if (!kind && bad) kind = kErrGTValue;
  if (!kind) {
    const int32_t old = atomicCAS(nhap_state, -1, (int32_t)n_hap);
    if (old != -1 && old != (int32_t)n_hap) kind = kErrGTLength;
  }
  if (kind) atomicMin(err, (unsigned long long)(ustart + rec_off[k]) << 3 | kind);
  BcfCol o;
  o.pos = pos + 1;
  o.alt_sum = (int32_t)(sum - (uint32_t)n_hap);
  o.a0 = (uint8_t)code0;
  o.a1 = (uint8_t)code1;
  o.biallelic = mx <= 2u;
  o.pad = 0;
  cols[k] = o;
}

// ---- text VCF ------------------------------------------------------------------------------------------------------------
// k_vcf_decode reduces a VCF line to the BcfCol that k_bcf_decode makes from the BCF of the same record, with the semantics of
// htslib's vcf_parse:
//   pos = the text POS (the host checked it: a plain decimal);
//   a0  = REF coded as k_bcf_decode codes allele 0 (0 empty, the letter, 0xff longer);
//   a1  = the first ALT allele (up to ',' or the tab) coded so; an ALT of exactly "." is n_allele = 1, so a1 = 0;
//   GT  = the subfield of each sample column at GT's index among FORMAT's ':'-separated keys (GT need not be first);
//         its syntax is allele([/|]allele)*, an allele is decimal digits or '.';
//   alt_sum = the sum of the allele indices mod 2^32, biallelic = every index <= 1.
// Refused, as the BCF path refuses what htslib would hand it: '.' in a GT (bcf_gt_missing); samples of one line with different
// ploidies (htslib pads the shorter ones with vector-end); a line whose n_hap = samples x ploidy is not the file's first line's;
// no FORMAT column, no GT key in FORMAT, or a sample column that stops before GT's subfield (no GT value).  Refused as new cases:
// fewer than 8 fixed fields, a sample-column count other than the header's, a GT off the syntax, an allele index over 2^29.
// Kinds (the BCF numbers where the meaning is the same); when a line has several, the first in this order is reported:
// fewer than 8 fields, no FORMAT or no GT key in it, the sample count, a sample without GT, syntax, missing, ploidy, n_hap.
enum : unsigned { kVcfNoGT = 1, kVcfMissing = 2, kVcfHapCount = 3, kVcfFixed = 4, kVcfSyntax = 5, kVcfSamples = 6, kVcfPloidy = 7 };
constexpr uint64_t kVcfMaxAllele = 1u << 29;

// 4-bit mask of the bytes of w equal to c4's (c4: the byte repeated)
__device__ __forceinline__ unsigned byte_bits(uint32_t w, uint32_t c4)
{
  const uint32_t m = (__vcmpeq4(w, c4) >> 7) & 0x01010101u;
  return (m | m >> 7 | m >> 14 | m >> 21) & 15u;
}
// 16-bit mask of the tabs in the 16 bytes at c (16-aligned) that lie in [lo, hi)
__device__ __forceinline__ unsigned tab_mask(const uint8_t* raw, int64_t c, int64_t lo, int64_t hi)
{
  if (c >= hi || c + 16 <= lo) return 0;
  const uint4 x = *(const uint4*)(raw + c);
  unsigned m = byte_bits(x.x, 0x09090909u) | byte_bits(x.y, 0x09090909u) << 4 | byte_bits(x.z, 0x09090909u) << 8 | byte_bits(x.w, 0x09090909u) << 12;
  const int j0 = lo > c ? (int)(lo - c) : 0, j1 = hi - c < 16 ? (int)(hi - c) : 16;
  return m & (((1u << j1) - 1u) & ~((1u << j0) - 1u));
}
__device__ __forceinline__ int warp_excl_sum(int x, int lane)
{
  int s = x;
  for (int d = 1; d < 32; d <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, s, d);
    if (lane >= d) s += y;
  }
  return s - x;
}
// 4 bytes at any address (the window buffer is padded past its end)
__device__ __forceinline__ uint32_t ld4_any(const uint8_t* p)
{
  const uint32_t* q = (const uint32_t*)((uintptr_t)p & ~(uintptr_t)3);
  return __funnelshift_r(q[0], q[1], ((uint32_t)(uintptr_t)p & 3u) * 8u);
}
// Fast path: a sample column at p whose GT is d|d or d/d followed by a tab, ':' or the line's end (GT first in FORMAT).  The
// two digits go into sum / mx4 byte-wise.
__device__ __forceinline__ bool gt_fast(const uint8_t* raw, int64_t p, int64_t e, uint32_t& sum, uint32_t& mx4)
{
  if (p + 3 > e) return false;
  const uint32_t w = ld4_any(raw + p);
  const uint32_t d = __vsub4(w, 0x30303030u) & 0x00ff00ffu;                          // the digits, as byte lanes 0 and 2
  const bool digits = (__vcmpleu4(__vsub4(w, 0x30303030u), 0x09090909u) & 0x00ff00ffu) == 0x00ff00ffu;
  const bool sep = ((__vcmpeq4(w, 0x7c7c7c7cu) | __vcmpeq4(w, 0x2f2f2f2fu)) & 0x0000ff00u) != 0;
  const bool term = p + 3 == e || ((__vcmpeq4(w, 0x09090909u) | __vcmpeq4(w, 0x3a3a3a3au)) & 0xff000000u) != 0;
  sum = __dp4a(d, 0x01010101u, sum);
  mx4 = __vmaxu4(mx4, d);
  return digits && sep && term;
}
// General path: one sample column at p (up to the next tab or e), GT at subfield gt_idx.  flags |= 1 << kind.
__device__ __forceinline__ void gt_general(const uint8_t* raw, int64_t p, int64_t e, int gt_idx, uint32_t& sum, uint32_t& mx, int& pmin,
                                           int& pmax, unsigned& flags)
{
  for (int i = 0; i < gt_idx; i++) {
    while (p < e && raw[p] != ':' && raw[p] != '\t') p++;
    if (p >= e || raw[p] == '\t') { flags |= 1u << kVcfNoGT; return; }
    p++;
  }
  int ploidy = 0;
  for (;;) {
    uint32_t c = p < e ? raw[p] : '\t';
    if (c == '.') {
      flags |= 1u << kVcfMissing;
      p++;
    } else if (c - '0' <= 9u) {
      uint64_t v = 0;
      do {
        v = v * 10 + (c - '0');
        if (v > kVcfMaxAllele) { flags |= 1u << kVcfSyntax; return; }
        p++;
        c = p < e ? raw[p] : '\t';
      } while (c - '0' <= 9u);
      sum += (uint32_t)v;
      mx = max(mx, (uint32_t)v);
    } else {
      flags |= 1u << kVcfSyntax;
      return;
    }
    ploidy++;
    c = p < e ? raw[p] : '\t';
    if (c == '/' || c == '|') { p++; continue; }
    if (c == ':' || c == '\t') break;
    flags |= 1u << kVcfSyntax;
    return;
  }
  pmin = min(pmin, ploidy);
  pmax = max(pmax, ploidy);
}

// warp = line k0 + warp of the window: [rec_off[k], rec_off[k + 1] or text_end), its newline dropped.  Pass 1 finds the tabs
// that end the first nine columns (INFO may be tens of KB: 512 bytes a step, a tab ballot and a warp prefix sum); lane 0 codes
// REF / ALT and finds GT in FORMAT.  Pass 2 walks the sample columns 512 bytes a step: a step whose sample columns all start
// with a single-digit diploid GT (and GT is FORMAT's first key) is summed byte-wise (gt_fast), any other step parses each
// sample on the lane holding the tab before it (gt_general).  Both give the same bits.  paths (the vcf_paths test option,
// else null): [0] / [1] count the lines decoded on the fast path only / with a general step.
__global__ void __launch_bounds__(256) k_vcf_decode(int64_t k0, int64_t k1, int64_t n_win, const uint8_t* __restrict__ raw,
                                                    const int64_t* __restrict__ rec_off, int64_t text_end, uint64_t ustart, int n_sample,
                                                    BcfCol* __restrict__ cols, int32_t* __restrict__ nhap_state,
                                                    unsigned long long* __restrict__ err, unsigned long long* __restrict__ paths)
{
  __shared__ int64_t tabs_s[8][10];
  const int lane = threadIdx.x & 31;
  const int64_t k = k0 + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (k >= k1) return;
  int64_t* tp = tabs_s[threadIdx.x >> 5];
  const int64_t b = rec_off[k];
  int64_t e = k + 1 < n_win ? rec_off[k + 1] : text_end;
  if (e > b && raw[e - 1] == '\n') e--;
  // pass 1: tp[1..9] = the tabs that end columns 1..9
  int ntab = 0;
  for (int64_t c0 = b & ~(int64_t)15; c0 < e && ntab < 9; c0 += 512) {
    const int64_t c = c0 + 16 * lane;
    unsigned m = tab_mask(raw, c, b, e);
    const int cnt = __popc(m);
    int g = ntab + warp_excl_sum(cnt, lane);
    for (; m && g < 9; m &= m - 1) tp[++g] = c + __ffs(m) - 1;
    ntab += __reduce_add_sync(0xffffffffu, cnt);
  }
  __syncwarp();
  ntab = min(ntab, 9);
  unsigned flags = 0;
  int gt_idx = -1;
  uint32_t code0 = 0, code1 = 0;
  int32_t pos = 0;
  if (ntab < 7) flags |= 1u << kVcfFixed;
  else if (lane == 0) {
    for (int64_t q = tp[1] + 1; q < tp[2]; q++) pos = pos * 10 + (raw[q] - '0');
    const int64_t r0 = tp[3] + 1, rl = tp[4] - r0, al0 = tp[4] + 1, al = tp[5] - al0;
    code0 = rl == 0 ? 0u : rl == 1 ? raw[r0] : 0xffu;
    if (al == 0 || raw[al0] == ',' || (al == 1 && raw[al0] == '.')) code1 = 0;
    else code1 = al == 1 || raw[al0 + 1] == ',' ? raw[al0] : 0xffu;
    if (ntab >= 8) {                                        // FORMAT: [tp[8] + 1, tp[9] or e)
      const int64_t f1 = ntab >= 9 ? tp[9] : e;
      int key = 0;
      for (int64_t q = tp[8] + 1; q <= f1 && gt_idx < 0;) {
        int64_t qe = q;
        while (qe < f1 && raw[qe] != ':') qe++;
        if (qe - q == 2 && raw[q] == 'G' && raw[q + 1] == 'T') gt_idx = key;
        key++;
        q = qe + 1;
      }
    }
  }
  gt_idx = __shfl_sync(0xffffffffu, gt_idx, 0);
  // pass 2: the sample columns, each starting after a tab from tp[9] on
  int n_col = 0;
  uint32_t sum = 0, mx = 0;
  int pmin = 1 << 30, pmax = 0;
  bool all_fast = true;
  if (ntab == 9 && gt_idx >= 0) {
    const int64_t s0 = tp[9];
    for (int64_t c0 = s0 & ~(int64_t)15; c0 < e; c0 += 512) {
      const int64_t c = c0 + 16 * lane;
      const unsigned m = tab_mask(raw, c, s0, e);
      n_col += __reduce_add_sync(0xffffffffu, __popc(m));
      uint32_t fsum = 0, fmx4 = 0;
      bool fast = gt_idx == 0;
      for (unsigned mm = m; mm && fast; mm &= mm - 1) fast = gt_fast(raw, c + __ffs(mm), e, fsum, fmx4);
      if (__all_sync(0xffffffffu, fast)) {
        sum += fsum;
        mx = max(mx, max(fmx4 & 0xffu, fmx4 >> 16));
        if (m) pmin = min(pmin, 2), pmax = max(pmax, 2);
      } else {
        all_fast = false;
        for (unsigned mm = m; mm; mm &= mm - 1) gt_general(raw, c + __ffs(mm), e, gt_idx, sum, mx, pmin, pmax, flags);
      }
    }
  }
  sum = __reduce_add_sync(0xffffffffu, sum);
  mx = __reduce_max_sync(0xffffffffu, mx);
  pmin = __reduce_min_sync(0xffffffffu, pmin);
  pmax = __reduce_max_sync(0xffffffffu, pmax);
  flags = __reduce_or_sync(0xffffffffu, flags);
  if (lane != 0) return;
  const int64_t n_hap = (int64_t)n_col * pmax;
  unsigned kind = 0;
  if (flags >> kVcfFixed & 1u) kind = kVcfFixed;
  else if (ntab == 7 || gt_idx < 0) kind = kVcfNoGT;
  else if (n_col != n_sample) kind = kVcfSamples;
  else if (flags >> kVcfNoGT & 1u) kind = kVcfNoGT;
  else if (flags >> kVcfSyntax & 1u) kind = kVcfSyntax;
  else if (flags >> kVcfMissing & 1u) kind = kVcfMissing;
  else if (pmin != pmax) kind = kVcfPloidy;
  else {
    const int32_t old = atomicCAS(nhap_state, -1, (int32_t)n_hap);
    if (old != -1 && old != (int32_t)n_hap) kind = kVcfHapCount;
  }
  if (kind) atomicMin(err, (unsigned long long)(ustart + b) << 3 | kind);
  if (paths) atomicAdd(paths + (all_fast ? 0 : 1), 1ull);
  BcfCol o;
  o.pos = pos;
  o.alt_sum = (int32_t)sum;
  o.a0 = (uint8_t)code0;
  o.a1 = (uint8_t)code1;
  o.biallelic = mx <= 1u;
  o.pad = 0;
  cols[k - k0] = o;
}

__device__ __forceinline__ bool letter(uint32_t x) { return x != 0u && x != 0xffu; }

// thread = .mut row of the chromosome: the record at the row is the first one at or after its position (both cursors of
// parse_vcfvcf, coal.cpp:1001-1006 / 1074-1079, reduce to this lower bound: rows and records ascend).  Reference rules
// (coal.cpp:1008-1062): the record's two alleles are the row's in either order (flipped: DAF = N - allele sum) and it is
// biallelic; no record: DAF = N if --ref_genome shows the derived allele; DAF = 0 drops the row.  Target rules (1081-1131): as
// the reference, or the record reports one allele (second empty or absent), one of the row's, with allele sum 0 (DAF = N if it
// is the derived one); no record: --ref_genome gives N for the derived base, 0 for the ancestral one.  One lower bound and one
// genome read serve both roles: pile_t gets the target's row counts, pile_r the reference's (a null array is skipped), each as
// (AAF, DAF) = (N - DAF, DAF), zeros where the row is not usable for that role (as k_pack_row_counts packs them).
__global__ void k_bcf_rows(int64_t row0, int64_t n_rows, const int32_t* __restrict__ site_pos, const uint32_t* __restrict__ meta,
                           const BcfCol* __restrict__ cols, int64_t n_rec, int32_t N, const uint8_t* __restrict__ ref, int64_t ref_len,
                           int4* __restrict__ pile_t, int4* __restrict__ pile_r)
{
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n_rows) return;
  const int64_t row = row0 + m;
  const uint32_t mt = meta[row];
  const uint32_t anc = (mt >> 8) & 0xffu, der = (mt >> 16) & 0xffu;
  int32_t daf_t = -1, daf_r = -1;                             // -1: not usable
  if ((mt & 1u) && anc != der) {                              // coal.cpp:966-995: the lookups only happen for these rows
    const int32_t bp = site_pos[row];
    int64_t lo = 0, hi = n_rec;
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (cols[mid].pos < bp) lo = mid + 1; else hi = mid; }
    if (lo < n_rec && cols[lo].pos == bp) {
      const BcfCol c = cols[lo];
      const bool two = letter(c.a0) && letter(c.a1);
      const bool same = two && c.a0 == anc && c.a1 == der, flip = two && c.a0 == der && c.a1 == anc;
      if (same || flip) {
        if (c.biallelic) daf_t = daf_r = flip ? N - c.alt_sum : c.alt_sum;
      } else if (c.a0 != 0 && c.a1 == 0) {
        if (letter(c.a0) && (c.a0 == anc || c.a0 == der) && c.biallelic && c.alt_sum == 0) daf_t = c.a0 == der ? N : 0;
      }
    } else if (ref && bp >= 1 && (int64_t)bp - 1 < ref_len) {
      uint32_t b = ref[bp - 1];
      if (b >= 'a' && b <= 'z') b -= 32;                      // fasta::Read upper-cases (data.cpp:213-237)
      if (b == der) daf_t = daf_r = N;
      else if (b == anc) daf_t = 0;
    }
    if (daf_r == 0) daf_r = -1;
  }
  if (pile_t) pile_t[row] = daf_t >= 0 ? make_int4(N - daf_t, daf_t, 0, -1) : make_int4(0, 0, 0, -1);
  if (pile_r) pile_r[row] = daf_r >= 0 ? make_int4(N - daf_r, daf_r, 0, -1) : make_int4(0, 0, 0, -1);
}

inline int grid_for(int64_t n, int threads) { return (int)((n + threads - 1) / threads); }
inline size_t up(size_t x) { return (x + 255) & ~(size_t)255; }

int bcf_threads()
{
  if (const char* e = getenv("COLATE_BCF_THREADS")) return std::max(1, atoi(e));
  return (int)std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
}

// grows h->bcf_cols to hold n records, keeping the first `keep`
int ensure_cols(colate_handle* h, int64_t n, int64_t keep)
{
  const size_t bytes = (size_t)n * sizeof(BcfCol) + 16;
  if (bytes <= h->bcf_cols.cap) return 0;
  DevBuf nb;
  CK(nb.ensure(std::max(bytes, 2 * h->bcf_cols.cap)));
  if (keep) CK(cudaMemcpyAsync(nb.p, h->bcf_cols.p, (size_t)keep * sizeof(BcfCol), cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->bcf_cols.release();
  h->bcf_cols = nb;
  return 0;
}

// One BCF or bgzipped text VCF file -> h->bcf_cols.  A per-chromosome file (gr null): h->bcf_n_rec records of h->bcf_n_hap
// haplotypes.  A whole-genome file (gr: n_chr --chr entries chr_names, GenotypeReader::set_listed): the records of every listed
// contig in file order, entry c's at [gr->first[c], gr->first[c] + gr->n[c]) with GT length gr->n_hap[c]; contigs outside the
// list are not copied to the device.  Each contig has its own state (GT length, first error: 16 bytes in h->bcf_state), and its
// first record is decoded alone: its GT length is the one every later record of the contig must have.  t[]: timing
// accumulators as colate_last_bcf_timing
int decode_file(colate_handle* h, const char* path, int n_chr, const char* const* chr_names, int64_t chunk_bytes, double* t, GenomeRecs* gr)
{
  std::unique_ptr<GenotypeReader> rdp;
  if (int rc = open_genotypes(path, bcf_threads(), &rdp)) return rc;
  GenotypeReader& rd = *rdp;
  if (gr) rd.set_listed(n_chr, chr_names);
  const int n_state = gr ? n_chr : 1;
  const int gt_key = rd.text ? -1 : static_cast<BcfReader&>(rd).gt_key;
  cudaStream_t s = h->stream;
  CK(h->bcf_state.ensure((size_t)n_state * 16 + 16));
  CK(cudaMemsetAsync(h->bcf_state.p, 0xff, (size_t)n_state * 16, s));               // per contig: GT length -1, no error (~0)
  char* const paths = h->bcf_state.as<char>() + (size_t)n_state * 16;               // text VCF, vcf_paths option: lines on the fast / the general path
  CK(cudaMemsetAsync(paths, 0, 16, s));
  const size_t target = chunk_bytes > 0 ? (size_t)chunk_bytes : (size_t)64 << 20;
  Pinned raw[2], offs[2];
  cudaEvent_t done[2];
  bool pending[2] = {false, false};
  for (auto& e : done) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  struct Ev { cudaEvent_t* e; ~Ev() { cudaEventDestroy(e[0]); cudaEventDestroy(e[1]); } } ev_guard{done};
  // bcf_timing option: events around the copies and the decode of every window, and a wait after each (the host and the
  // device no longer overlap: the phases are for a breakdown, the wall time is measured without it)
  cudaEvent_t tev[3] = {};
  if (h->opt_bcf_timing)
    for (auto& e : tev) CK(cudaEventCreate(&e));
  struct TEv { cudaEvent_t* e; ~TEv() { for (int i = 0; i < 3; i++) if (e[i]) cudaEventDestroy(e[i]); } } tev_guard{tev};
  int64_t n_rec = 0, n_inflated = 0;
  std::vector<int64_t> first(n_state, -1), seen(n_state, 0);
  BcfWindow w;
  auto drain = [&]() { cudaStreamSynchronize(s); };
  for (int wi = 0;; wi++) {
    const int b = wi & 1;
    const size_t need = rd.next_window_bytes(target);
    if (need == 0) break;
    if (pending[b]) { CK(cudaEventSynchronize(done[b])); pending[b] = false; }   // window wi - 2 has left this buffer
    CK(raw[b].ensure(need));
    if (int rc = rd.fill((uint8_t*)raw[b].p, target, w)) { drain(); return rc; }
    n_inflated += (int64_t)w.n_bytes;
    const int64_t n = (int64_t)w.rec_off.size();
    if (n == 0) continue;
    CK(offs[b].ensure((size_t)n * 8));
    memcpy(offs[b].p, w.rec_off.data(), (size_t)n * 8);
    if (int rc = ensure_cols(h, n_rec + n, n_rec)) return rc;
    const size_t o_off = up(w.n_bytes), total = o_off + (size_t)n * 8;
    CK(h->bcf_buf.ensure(total + 16));   // (a reallocation waits for the device: cudaFree synchronises; k_vcf_decode reads past the end)
    char* d = h->bcf_buf.as<char>();
    const int64_t* d_off = (const int64_t*)(d + o_off);
    if (tev[0]) CK(cudaEventRecord(tev[0], s));
    // the bytes of the runs only, each at its window offset
    for (const BcfRun& r : w.runs) {
      const int64_t b0 = w.rec_off[r.first];
      CK(cudaMemcpyAsync(d + b0, (const char*)raw[b].p + b0, (size_t)(r.end - b0), cudaMemcpyHostToDevice, s));
    }
    CK(cudaMemcpyAsync(d + o_off, offs[b].p, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    if (tev[0]) CK(cudaEventRecord(tev[1], s));
    for (const BcfRun& r : w.runs) {
      const int si = gr ? r.c : 0;
      int32_t* nhap_state = (int32_t*)(h->bcf_state.as<char>() + (size_t)si * 16);
      unsigned long long* err = (unsigned long long*)(h->bcf_state.as<char>() + (size_t)si * 16 + 8);
      BcfCol* cols = h->bcf_cols.as<BcfCol>() + n_rec + r.first;
      if (seen[si] == 0) first[si] = n_rec + r.first;
      for (int64_t k0 = 0; k0 < r.n;) {
        const int64_t k1 = seen[si] == 0 && k0 == 0 ? 1 : r.n;
        if (rd.text)
          k_vcf_decode<<<grid_for((k1 - k0) * 32, 256), 256, 0, s>>>(k0, k1, r.n, (const uint8_t*)d, d_off + r.first, r.end, w.ustart, rd.n_sample,
                                                                     cols + k0, nhap_state, err,
                                                                     h->opt_vcf_paths ? (unsigned long long*)paths : nullptr);
        else
          k_bcf_decode<<<grid_for((k1 - k0) * 32, 256), 256, 0, s>>>(k1 - k0, (const uint8_t*)d, d_off + r.first + k0, w.ustart, gt_key, cols + k0,
                                                                     nhap_state, err);
        h->launches += 1;
        CK(cudaGetLastError());
        k0 = k1;
      }
      seen[si] += r.n;
    }
    if (tev[0]) {
      CK(cudaEventRecord(tev[2], s));
      CK(cudaEventSynchronize(tev[2]));
      float ms = 0;
      CK(cudaEventElapsedTime(&ms, tev[0], tev[1]));
      t[3] += ms;
      CK(cudaEventElapsedTime(&ms, tev[1], tev[2]));
      t[4] += ms;
    }
    n_rec += n;
    CK(cudaEventRecord(done[b], s));
    pending[b] = true;
  }
  CK(cudaStreamSynchronize(s));
  if (gr) {
    if (int rc = rd.listed_complete()) return rc;
  } else if (n_rec == 0) {
    return rd.err(std::string(rd.text ? "VCF" : "BCF") + " file without records (the reference reads a first record unconditionally)", 0, false);
  }
  struct St { int32_t nhap, pad; unsigned long long err; };
  std::vector<St> st((size_t)n_state + 1);
  CK(cudaMemcpy(st.data(), h->bcf_state.p, (size_t)n_state * 16 + 16, cudaMemcpyDeviceToHost));
  const unsigned long long* np = (const unsigned long long*)&st[n_state];
  h->vcf_paths[0] = rd.text ? (int64_t)np[0] : 0;
  h->vcf_paths[1] = rd.text ? (int64_t)np[1] : 0;
  t[0] += rd.index_s;
  t[1] += rd.inflate_s;
  t[2] += rd.walk_s;
  t[7] = rd.n_threads;
  t[8] += (double)n_inflated;
  t[9] += (double)n_rec;
  static const char* what[] = {"", "BCF record without a GT field", "BCF record with a missing or vector-end genotype (or an allele index below 0)",
                               "BCF record whose GT length differs from the file's first record's", "BCF record whose typed fields run past its l_shared / l_indiv",
                               "BCF record whose GT is not an integer vector"};
  static const char* what_vcf[] = {"", "VCF line without a GT value (no FORMAT column, no GT key in FORMAT, or a sample column that stops before GT)",
                                   "VCF line with a missing allele ('.') in a GT", "VCF line whose samples x ploidy differs from the file's first line's",
                                   "VCF line with fewer than 8 fixed fields", "VCF line with a GT that is not allele([/|]allele)* (allele: digits up to 2^29)",
                                   "VCF line whose sample-column count differs from the header's",
                                   "VCF line whose samples have different ploidies"};
  for (int si = 0; si < n_state; si++) {
    if (st[si].err == ~0ull) continue;
    const int rc = rd.err((rd.text ? what_vcf : what)[st[si].err & 7], st[si].err >> 3, false);
    return gr ? fail(rc, std::string("chromosome ") + chr_names[si] + ": " + colate_last_error()) : rc;
  }
  h->bcf_n_rec = n_rec;
  h->bcf_n_hap = st[0].nhap;
  if (gr) {
    gr->first = first;
    gr->n = seen;
    gr->n_hap.resize(n_chr);
    for (int c = 0; c < n_chr; c++) gr->n_hap[c] = st[c].nhap;
  }
  return 0;
}

// the row counts of the target slot t_slot and / or the reference slot r_slot (-1: that role is skipped) from one decode of every
// chromosome's file (bcf_paths), or of one whole-genome file (genome_path).  Genome: host contigs (ref_seqs / ref_lens, uploaded
// per chromosome), the handle's resident genome (resident), or none.
int rows_from_bcf(colate_handle* h, int t_slot, int r_slot, int n_chr, const char* const* chr_names, const char* const* bcf_paths,
                  const char* genome_path, const uint8_t* const* ref_seqs, const int64_t* ref_lens, bool resident, int64_t chunk_bytes)
{
  CK(cudaSetDevice(h->device));
  const auto t_start = std::chrono::steady_clock::now();
  double t[10] = {};
  cudaStream_t s = h->stream;
  const size_t n_site = (size_t)h->n_site;
  const int slots[2] = {t_slot, r_slot};
  for (int sl : slots)
    if (sl >= 0) CK(h->genomes[sl].pile.ensure(n_site * 16 + 16));
  int4* pile_t = t_slot >= 0 ? h->genomes[t_slot].pile.as<int4>() : nullptr;
  int4* pile_r = r_slot >= 0 ? h->genomes[r_slot].pile.as<int4>() : nullptr;
  cudaEvent_t tev[2] = {};
  if (h->opt_bcf_timing)
    for (auto& e : tev) CK(cudaEventCreate(&e));
  struct TEv { cudaEvent_t* e; ~TEv() { for (int i = 0; i < 2; i++) if (e[i]) cudaEventDestroy(e[i]); } } tev_guard{tev};
  GenomeRecs gr;
  if (genome_path)
    if (int rc = decode_file(h, genome_path, n_chr, chr_names, chunk_bytes, t, &gr)) return rc;
  for (int c = 0; c < n_chr; c++) {
    if (!genome_path)
      if (int rc = decode_file(h, bcf_paths[c], 0, nullptr, chunk_bytes, t, nullptr))
        return fail(rc, std::string("chromosome ") + chr_names[c] + ": " + colate_last_error());
    const uint8_t* ref = nullptr;
    int64_t L = 0;
    if (resident) {
      L = h->refg_off[c + 1] - h->refg_off[c];
      ref = L ? h->refg.as<uint8_t>() + h->refg_off[c] : nullptr;
    } else if (ref_seqs && ref_seqs[c] && ref_lens[c]) {
      L = ref_lens[c];
      CK(h->bcf_ref.ensure((size_t)L + 16));
      CK(cudaMemcpyAsync(h->bcf_ref.p, ref_seqs[c], (size_t)L, cudaMemcpyHostToDevice, s));
      h->ref_h2d_bytes += L;
      ref = h->bcf_ref.as<uint8_t>();
    }
    const int64_t r0 = h->h_site_off[c], nr = h->h_site_off[c + 1] - r0;
    if (nr == 0) continue;
    // a whole-genome file: chromosome c's records alone, so the lower bound stays inside them as in its own file
    const BcfCol* cols = h->bcf_cols.as<BcfCol>() + (genome_path ? gr.first[c] : 0);
    const int64_t n_c = genome_path ? gr.n[c] : h->bcf_n_rec;
    const int32_t N = genome_path ? gr.n_hap[c] : h->bcf_n_hap;
    if (tev[0]) CK(cudaEventRecord(tev[0], s));
    k_bcf_rows<<<grid_for(nr, 256), 256, 0, s>>>(r0, nr, h->pos.as<int32_t>(), h->meta.as<uint32_t>(), cols, n_c, N, ref, L, pile_t, pile_r);
    h->launches += 1;
    CK(cudaGetLastError());
    if (tev[0]) {
      CK(cudaEventRecord(tev[1], s));
      CK(cudaEventSynchronize(tev[1]));
      float ms = 0;
      CK(cudaEventElapsedTime(&ms, tev[0], tev[1]));
      t[5] += ms;
    }
  }
  // the slots are row-count genomes, as colate_set_row_counts leaves them
  for (int sl : slots) {
    if (sl < 0) continue;
    GenomeDev& g = h->genomes[sl];
    g.n_rec = 0;
    g.pileup = true;
    g.acgt = false;
    g.set = true;
    g.joined = false;
    CK(cudaMemsetAsync(h->order_flag.as<int>() + 1 + sl, 0, 4, s));
  }
  h->flags_done = false;
  CK(cudaStreamSynchronize(s));
  t[6] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
  memcpy(h->bcf_timing, t, sizeof t);
  return 0;
}

}  // namespace

namespace colate {
int decode_genotype_file(colate_handle* h, const char* path, int64_t chunk_bytes, double* t) { return decode_file(h, path, 0, nullptr, chunk_bytes, t, nullptr); }
int decode_genotype_genome(colate_handle* h, const char* path, int n_chr, const char* const* chr_names, int64_t chunk_bytes, double* t, GenomeRecs* gr)
{
  return decode_file(h, path, n_chr, chr_names, chunk_bytes, t, gr);
}
}

extern "C" {

int colate_rows_from_bcf(colate_handle* h, int slot, int role, int n_chr, const char* const* chr_names, const char* const* bcf_paths,
                         const uint8_t* const* ref_seqs, const int64_t* ref_lens, int64_t chunk_bytes, int32_t* aaf_out, int32_t* daf_out)
{
  if (!h || slot < 0 || slot >= COLATE_MAX_GENOMES || (role != 0 && role != 1) || n_chr <= 0 || !chr_names || !bcf_paths || chunk_bytes < 0 ||
      (ref_seqs && !ref_lens))
    return fail(COLATE_ERR_ARG, "colate_rows_from_bcf: bad arguments");
  if (!h->sites_set || n_chr != h->n_chr) return fail(COLATE_ERR_ARG, "colate_rows_from_bcf: one file per chromosome of the site set");
  for (int c = 0; c < n_chr; c++)
    if (!bcf_paths[c] || (ref_seqs && (ref_lens[c] < 0 || (ref_lens[c] > 0 && !ref_seqs[c])))) return fail(COLATE_ERR_ARG, "colate_rows_from_bcf: bad arguments");
  if (int rc = rows_from_bcf(h, role == 0 ? slot : -1, role == 1 ? slot : -1, n_chr, chr_names, bcf_paths, nullptr, ref_seqs, ref_lens, false, chunk_bytes))
    return rc;
  if (aaf_out || daf_out) {
    const size_t n_site = (size_t)h->n_site;
    std::vector<int32_t> p4(n_site * 4);
    if (n_site) CK(cudaMemcpyAsync(p4.data(), h->genomes[slot].pile.p, n_site * 16, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (size_t m = 0; m < n_site; m++) {
      if (aaf_out) aaf_out[m] = p4[4 * m];
      if (daf_out) daf_out[m] = p4[4 * m + 1];
    }
  }
  return 0;
}

int colate_rows_from_bcf_roles(colate_handle* h, int target_slot, int reference_slot, int n_chr, const char* const* chr_names,
                               const char* const* bcf_paths, int genome, int64_t chunk_bytes)
{
  if (!h || target_slot < -1 || target_slot >= COLATE_MAX_GENOMES || reference_slot < -1 || reference_slot >= COLATE_MAX_GENOMES ||
      (target_slot < 0 && reference_slot < 0) || target_slot == reference_slot || (genome != 0 && genome != 1) || n_chr <= 0 || !chr_names ||
      !bcf_paths || chunk_bytes < 0)
    return fail(COLATE_ERR_ARG, "colate_rows_from_bcf_roles: bad arguments");
  if (!h->sites_set || n_chr != h->n_chr) return fail(COLATE_ERR_ARG, "colate_rows_from_bcf_roles: one file per chromosome of the site set");
  for (int c = 0; c < n_chr; c++)
    if (!bcf_paths[c]) return fail(COLATE_ERR_ARG, "colate_rows_from_bcf_roles: bad arguments");
  if (genome == 1 && (int)h->refg_off.size() != n_chr + 1)
    return fail(COLATE_ERR_STATE, "colate_rows_from_bcf_roles: genome = 1 needs colate_set_ref_genome with one contig per chromosome");
  return rows_from_bcf(h, target_slot, reference_slot, n_chr, chr_names, bcf_paths, nullptr, nullptr, nullptr, genome == 1, chunk_bytes);
}

int colate_rows_from_bcf_genome(colate_handle* h, int target_slot, int reference_slot, int n_chr, const char* const* chr_names, const char* path,
                                int genome, int64_t chunk_bytes)
{
  if (!h || target_slot < -1 || target_slot >= COLATE_MAX_GENOMES || reference_slot < -1 || reference_slot >= COLATE_MAX_GENOMES ||
      (target_slot < 0 && reference_slot < 0) || target_slot == reference_slot || (genome != 0 && genome != 1) || n_chr <= 0 || !chr_names ||
      !path || chunk_bytes < 0)
    return fail(COLATE_ERR_ARG, "colate_rows_from_bcf_genome: bad arguments");
  if (!h->sites_set || n_chr != h->n_chr) return fail(COLATE_ERR_ARG, "colate_rows_from_bcf_genome: one --chr entry per chromosome of the site set");
  for (int c = 0; c < n_chr; c++)
    if (!chr_names[c]) return fail(COLATE_ERR_ARG, "colate_rows_from_bcf_genome: bad arguments");
  if (genome == 1 && (int)h->refg_off.size() != n_chr + 1)
    return fail(COLATE_ERR_STATE, "colate_rows_from_bcf_genome: genome = 1 needs colate_set_ref_genome with one contig per chromosome");
  return rows_from_bcf(h, target_slot, reference_slot, n_chr, chr_names, nullptr, path, nullptr, nullptr, genome == 1, chunk_bytes);
}

int colate_decode_bcf_genome(colate_handle* h, const char* path, int n_chr, const char* const* chr_names, int64_t chunk_bytes, int64_t* rec_first,
                             int64_t* n_records, int32_t* n_hap)
{
  if (!h || !path || n_chr <= 0 || !chr_names || chunk_bytes < 0) return fail(COLATE_ERR_ARG, "colate_decode_bcf_genome: bad arguments");
  for (int c = 0; c < n_chr; c++)
    if (!chr_names[c]) return fail(COLATE_ERR_ARG, "colate_decode_bcf_genome: bad arguments");
  CK(cudaSetDevice(h->device));
  const auto t_start = std::chrono::steady_clock::now();
  double t[10] = {};
  h->bcf_n_rec = 0;
  GenomeRecs gr;
  if (int rc = decode_file(h, path, n_chr, chr_names, chunk_bytes, t, &gr)) return rc;
  t[6] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
  memcpy(h->bcf_timing, t, sizeof t);
  for (int c = 0; c < n_chr; c++) {
    if (rec_first) rec_first[c] = gr.first[c];
    if (n_records) n_records[c] = gr.n[c];
    if (n_hap) n_hap[c] = gr.n_hap[c];
  }
  return 0;
}

int colate_decode_bcf(colate_handle* h, const char* bcf_path, int64_t chunk_bytes, int64_t* n_records, int32_t* n_hap)
{
  if (!h || !bcf_path || chunk_bytes < 0) return fail(COLATE_ERR_ARG, "colate_decode_bcf: bad arguments");
  CK(cudaSetDevice(h->device));
  const auto t_start = std::chrono::steady_clock::now();
  double t[10] = {};
  h->bcf_n_rec = 0;
  if (int rc = decode_file(h, bcf_path, 0, nullptr, chunk_bytes, t, nullptr)) return rc;
  t[6] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
  memcpy(h->bcf_timing, t, sizeof t);
  if (n_records) *n_records = h->bcf_n_rec;
  if (n_hap) *n_hap = h->bcf_n_hap;
  return 0;
}

int colate_bcf_records(colate_handle* h, int64_t r0, int64_t n, int32_t* rec_pos, uint8_t* rec_a0, uint8_t* rec_a1, int32_t* rec_alt_sum,
                       uint8_t* rec_biallelic)
{
  if (!h || r0 < 0 || n < 0 || r0 + n > h->bcf_n_rec) return fail(COLATE_ERR_ARG, "colate_bcf_records: bad record range");
  CK(cudaSetDevice(h->device));
  std::vector<BcfCol> c((size_t)n);
  if (n) CK(cudaMemcpyAsync(c.data(), h->bcf_cols.as<BcfCol>() + r0, (size_t)n * sizeof(BcfCol), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  for (int64_t k = 0; k < n; k++) {
    if (rec_pos) rec_pos[k] = c[k].pos;
    if (rec_a0) rec_a0[k] = c[k].a0;
    if (rec_a1) rec_a1[k] = c[k].a1;
    if (rec_alt_sum) rec_alt_sum[k] = c[k].alt_sum;
    if (rec_biallelic) rec_biallelic[k] = c[k].biallelic;
  }
  return 0;
}

int colate_test_last_vcf_paths(colate_handle* h, int64_t* fast, int64_t* general)
{
  if (!h || !fast || !general) return fail(COLATE_ERR_ARG, "colate_test_last_vcf_paths: bad arguments");
  *fast = h->vcf_paths[0];
  *general = h->vcf_paths[1];
  return 0;
}

int colate_last_bcf_timing(colate_handle* h, double* out)
{
  if (!h || !out) return fail(COLATE_ERR_ARG, "colate_last_bcf_timing: bad arguments");
  memcpy(out, h->bcf_timing, sizeof h->bcf_timing);
  return 0;
}

}  // extern "C"
