// GPU-side ingest of Relate .mut text (SURVEY.md 8f, row N1): replaces Mutations::Read
// (include/src/mutations.cpp:56-283) for the columns the tmp/tmp path uses.
//
// The file's bytes go to the device once; three kernels find the line starts (newline count per
// tile -> scan -> positions) and one thread per data line splits the ';'-separated fields exactly
// as the reference's character loops do and converts them:
//   pos, is_flipped     std::stoi    -> decimal integer (strtol semantics)
//   branch_indices      counted (the path only needs "exactly one branch")
//   age_begin, age_end  std::stof    -> CORRECTLY ROUNDED decimal -> float: the digits are taken as an
//                                       exact integer M < 2^53 and a power of ten 10^k, |k| <= 22, both
//                                       exact doubles, so M * 10^k (or M / 10^-k) is one correctly
//                                       rounded fp64 operation; rounding that double to float equals
//                                       rounding the exact value unless the double sits exactly on a
//                                       float midpoint, which is detected
//   mutation type       -> allele codes
// into the packed site word of colate_site_meta().  Rows the device cannot convert with that
// guarantee (more than 15 significant digits, huge exponents, inf / nan / hex floats, a midpoint)
// are re-parsed on the host with strtof -- the result is identical to colate_read_mut() row for row
// (tests/test_gpu_ingest.py).
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "device.cuh"
#include "maketmp_word.h"

namespace colate {

constexpr int ING_THREADS = 256;
constexpr int ING_BYTES = 32;                       // bytes per thread
constexpr int ING_TILE = ING_THREADS * ING_BYTES;   // bytes per CTA

__device__ __forceinline__ int count_nl32(const char* text, int64_t n, int64_t base, uint32_t& mask)
{
  mask = 0;
  if (base + ING_BYTES <= n && ((uintptr_t)(text + base) & 15) == 0) {
    const uint4 a = *(const uint4*)(text + base), b = *(const uint4*)(text + base + 16);
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int k = 0; k < 8; k++)
#pragma unroll
      for (int j = 0; j < 4; j++)
        if (((w[k] >> (8 * j)) & 0xff) == '\n') mask |= 1u << (4 * k + j);
  } else {
    for (int j = 0; j < ING_BYTES; j++)
      if (base + j < n && text[base + j] == '\n') mask |= 1u << j;
  }
  return __popc(mask);
}

__global__ void __launch_bounds__(ING_THREADS)
k_nl_count(const char* __restrict__ text, int64_t n, int32_t* __restrict__ tile_cnt)
{
  __shared__ int ws[ING_THREADS / 32];
  uint32_t m;
  int c = count_nl32(text, n, (int64_t)blockIdx.x * ING_TILE + (int64_t)threadIdx.x * ING_BYTES, m);
  for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int i = 0; i < ING_THREADS / 32; i++) t += ws[i];
    tile_cnt[blockIdx.x] = t;
  }
}

// exclusive scan of the tile counts (one CTA, chunks of 1024)
__global__ void __launch_bounds__(1024)
k_tile_scan(const int32_t* __restrict__ tile_cnt, int64_t n_tiles, int64_t* __restrict__ tile_off)
{
  __shared__ int64_t ws[32];
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t b = 0; b < n_tiles; b += 1024) {
    const int64_t i = b + threadIdx.x;
    int64_t v = i < n_tiles ? tile_cnt[i] : 0, x = v;
    for (int o = 1; o < 32; o <<= 1) { int64_t y = __shfl_up_sync(0xffffffffu, x, o); if ((threadIdx.x & 31) >= o) x += y; }
    if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = x;
    __syncthreads();
    if (threadIdx.x < 32) {
      int64_t w = ws[threadIdx.x], z = w;
      for (int o = 1; o < 32; o <<= 1) { int64_t y = __shfl_up_sync(0xffffffffu, z, o); if (threadIdx.x >= o) z += y; }
      ws[threadIdx.x] = z - w;
    }
    __syncthreads();
    const int64_t excl = carry + ws[threadIdx.x >> 5] + x - v;
    if (i < n_tiles) tile_off[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) tile_off[n_tiles] = carry;
}

__global__ void __launch_bounds__(ING_THREADS)
k_nl_index(const char* __restrict__ text, int64_t n, const int64_t* __restrict__ tile_off, int64_t* __restrict__ nl_pos)
{
  __shared__ int ws[ING_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * ING_TILE + (int64_t)threadIdx.x * ING_BYTES;
  uint32_t m;
  const int c = count_nl32(text, n, base, m);
  int x = c;
  for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if ((threadIdx.x & 31) >= o) x += y; }
  if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = x;
  __syncthreads();
  int before = 0;
  for (int w = 0; w < (int)(threadIdx.x >> 5); w++) before += ws[w];
  int64_t o = tile_off[blockIdx.x] + before + x - c;
  while (m) { const int j = __ffs(m) - 1; m &= m - 1; nl_pos[o++] = base + j; }
}

// ---- field conversions ------------------------------------------------------------------------
__constant__ double c_p10[23] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15,
                                 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};

__device__ __forceinline__ bool is_space(char ch) { return ch == ' ' || (ch >= '\t' && ch <= '\r'); }

// std::stoi on [s, e) (strtol base 10 + range check); false: the host decides -- no digits (the reference's std::stoi
// throws and the run ends, mutations.cpp:84-88) or more than 9 digits (may leave the int range)
__device__ bool dev_strtol(const char* s, const char* e, long long& v)
{
  while (s < e && is_space(*s)) s++;
  bool neg = false;
  if (s < e && (*s == '+' || *s == '-')) { neg = *s == '-'; s++; }
  long long x = 0;
  int nd = 0;
  while (s < e && *s >= '0' && *s <= '9') { x = x * 10 + (*s - '0'); s++; if (++nd > 9) return false; }
  v = neg ? -x : x;
  return nd > 0;
}

// strtof(s, 0) on [s, e); false: not convertible here with a correct-rounding guarantee -> host
__device__ bool dev_strtof(const char* s, const char* e, float& out)
{
  while (s < e && is_space(*s)) s++;
  bool neg = false;
  if (s < e && (*s == '+' || *s == '-')) { neg = *s == '-'; s++; }
  if (s < e && (*s == 'i' || *s == 'I' || *s == 'n' || *s == 'N')) return false;             // inf / nan spellings
  if (s + 1 < e && *s == '0' && (s[1] == 'x' || s[1] == 'X')) return false;                  // hex float
  unsigned long long M = 0;
  int nsig = 0, ndig = 0, frac = 0, dropped = 0;
  bool seen_point = false;
  for (; s < e; s++) {
    const char ch = *s;
    if (ch >= '0' && ch <= '9') {
      ndig++;
      if (M == 0 && ch == '0') { if (seen_point) frac++; continue; }      // leading zeros
      if (nsig < 15) { M = M * 10 + (unsigned)(ch - '0'); nsig++; if (seen_point) frac++; }
      else { if (ch != '0') return false; if (!seen_point) dropped++; }      // trailing zeros beyond 15 digits only
    } else if (ch == '.' && !seen_point) seen_point = true;
    else break;
  }
  if (ndig == 0) return false;                                               // no conversion: std::stof throws, the host reports the line
  int ex = 0;
  if (s < e && (*s == 'e' || *s == 'E')) {
    const char* q = s + 1;
    bool eneg = false;
    if (q < e && (*q == '+' || *q == '-')) { eneg = *q == '-'; q++; }
    if (q < e && *q >= '0' && *q <= '9') {
      int v = 0;
      while (q < e && *q >= '0' && *q <= '9') { if (v < 100000) v = v * 10 + (*q - '0'); q++; }
      ex = eneg ? -v : v;
    }
  }
  if (M == 0) { out = neg ? -0.0f : 0.0f; return true; }
  const int k = ex - frac + dropped;
  if (k > 22 || k < -22) return false;
  const double d = k >= 0 ? __dmul_rn((double)M, c_p10[k]) : __ddiv_rn((double)M, c_p10[-k]);
  if (((unsigned long long)__double_as_longlong(d) & 0x1fffffffull) == 0x10000000ull) return false;   // float midpoint
  if (d < 1.1754943508222875e-38) return false;                                                         // subnormal float: other midpoints
  const float f = __double2float_rn(d);
  out = neg ? -f : f;
  return true;
}

// one data line; status[0] = 1 + first bad row (empty line / too few fields), status[1] = rows for the host.
// mkt: the make_tmp row word (maketmp_word.h) next to meta
__global__ void __launch_bounds__(256)
k_parse_mut(const char* __restrict__ text, int64_t n_bytes, const int64_t* __restrict__ nl_pos, int64_t n_nl, int64_t n_rows,
            int32_t* __restrict__ pos, float* __restrict__ age_begin, float* __restrict__ age_end, uint32_t* __restrict__ meta,
            uint32_t* __restrict__ mkt, unsigned long long* status, int64_t* __restrict__ fb_rows, int64_t fb_cap)
{
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  const int64_t li = row + 1;                                     // line 0 is the header
  const char* p = text + nl_pos[li - 1] + 1;
  const char* nl = text + (li < n_nl ? nl_pos[li] : n_bytes);     // the last line may lack its newline
  if (nl == p) { atomicMin(status, (unsigned long long)row + 1); return; }
  // snp;pos;dist;rs-id;tree;branches;is_not_mapping;is_flipped;age_begin;age_end;type;...
  const char* f[11];
  int nf = 0;
  f[nf++] = p;
  for (const char* q = p; q < nl && nf < 11; q++) if (*q == ';') f[nf++] = q + 1;
  if (nf < 10) { atomicMin(status, (unsigned long long)row + 1); return; }
  bool ok = true;
  long long v = 0;
  // every field Mutations::Read converts with std::stoi must convert (snp, pos, dist, tree, branch indices, is_flipped,
  // frequency columns): anything doubtful goes to the host, which applies std::stoi's rules to the letter
  ok &= dev_strtol(f[0], f[1] - 1, v);
  ok &= dev_strtol(f[2], f[3] - 1, v);
  ok &= dev_strtol(f[4], f[5] - 1, v);
  ok &= dev_strtol(f[1], f[2] - 1, v);
  const int32_t ps = (int32_t)v;
  int nb = 0;
  for (const char* b = f[5]; b < f[6] - 1;) {
    while (b < f[6] - 1 && *b == ' ') b++;
    if (b < f[6] - 1) {
      const char* te = b;
      while (te < f[6] - 1 && *te != ' ') te++;
      long long bv;
      ok &= dev_strtol(b, te, bv);
      nb++;
      b = te;
    }
  }
  ok &= dev_strtol(f[7], f[8] - 1, v);
  const int flipped = v != 0;
  float ab = 0.0f, ae = 0.0f;
  ok &= dev_strtof(f[8], f[9] - 1, ab);
  ok &= dev_strtof(f[9], nf >= 11 ? f[10] - 1 : nl, ae);
  ok &= nf >= 11;                                                  // age_end without its ';': the reference reads past the line
  // mutation type runs to the next ';' or the end of the line (mutations.cpp:216-223); "NA" if absent
  uint32_t m = 0;
  if (flipped == 0 && nb == 1 && ab < ae && ae >= 0 && nf >= 11) {
    const char* t = f[10];
    const char* te = t;
    while (te < nl && *te != ';') te++;
    if (te - t == 3 && t[1] == '/') {
      const char a = t[0], d = t[2];
      const bool oka = a == 'A' || a == 'C' || a == 'G' || a == 'T' || a == '0';
      const bool okd = d == 'A' || d == 'C' || d == 'G' || d == 'T' || d == '1';
      if (oka && okd) m = 1u | ((uint32_t)(unsigned char)a << 8) | ((uint32_t)(unsigned char)d << 16);
    }
  }
  // the make_tmp word reads the first four bytes of type[16] as parse_mut_line_fields fills it: the field's first 15 bytes, "NN"
  // (no code) for a longer field.  Rows with fewer than 11 fields go to the host (ok is false), which applies its "NA".
  uint32_t w = 0;
  if (nf >= 11) {
    const char* t = f[10];
    const char* te = t;
    while (te < nl && *te != ';') te++;
    const int64_t L = te - t;
    if (L <= 15) {
      const char t4[4] = {L > 0 ? t[0] : '\0', L > 1 ? t[1] : '\0', L > 2 ? t[2] : '\0', L > 3 ? t[3] : '\0'};
      w = maketmp_word(flipped, nb, t4);
    }
  }
  if (nf >= 11) {   // upstream; downstream; frequency columns (std::stoi each, mutations.cpp:224-250)
    const char* g = f[10];
    while (g < nl && *g != ';') g++;
    if (g < nl && g + 1 < nl) {
      g++;
      int semis = 0;
      while (g < nl && semis < 2) { if (*g == ';') semis++; g++; }
      if (semis < 2) ok = false;
      while (g < nl) {
        const char* fe = g;
        while (fe < nl && *fe != ';') fe++;
        long long fv;
        ok &= dev_strtol(g, fe, fv);
        g = fe < nl ? fe + 1 : nl;
      }
    }
  }
  pos[row] = ps; age_begin[row] = ab; age_end[row] = ae; meta[row] = m; mkt[row] = w;
  if (!ok) {
    const unsigned long long k = atomicAdd(status + 1, 1ull);
    if ((int64_t)k < fb_cap) fb_rows[k] = row;
  }
}

// ---- .colate.in records (coal.cpp:2505-2514) decoded on the device ----------------------------------
// The host has cut the image into runs of equal-width records by galloping (host_misc.cpp: colate_in_runs);
// thread = record: locate its run, CHECK that its {lchrom, chrom} header equals the run's (all records passing
// this check is what makes the host's segmentation the sequential reader's, see colate_in_runs) and split the
// 14 payload bytes into the genome's structure of arrays.  Records sit at arbitrary byte offsets: byte loads.
struct DevRun { long long byte_off; int width; int chr_id; long long n_rec; long long rec_base; };

__device__ __forceinline__ uint32_t ld_u32_unaligned(const unsigned char* p)
{
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

__global__ void __launch_bounds__(256)
k_decode_colate_in(const unsigned char* __restrict__ img, const DevRun* __restrict__ runs, int n_runs, int64_t n_rec,
                   int32_t* __restrict__ bp, int32_t* __restrict__ aaf, int32_t* __restrict__ daf, uint16_t* __restrict__ alleles,
                   int* __restrict__ bad)
{
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_rec) return;
  int lo = 0, hi = n_runs;                      // last run with rec_base <= k
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (runs[mid].rec_base <= k) lo = mid; else hi = mid; }
  const DevRun r = runs[lo];
  const unsigned char* first = img + r.byte_off;
  const unsigned char* rec = first + (k - r.rec_base) * r.width;
  const int hl = r.width - 14;                  // 4 + lchrom
  bool same = true;
  for (int i = 0; i < hl; i++) same &= rec[i] == first[i];
  if (!same) *bad = 1;
  const unsigned char* q = rec + hl;
  bp[k] = (int32_t)ld_u32_unaligned(q);
  alleles[k] = (uint16_t)(q[4] | (q[5] << 8));
  aaf[k] = (int32_t)ld_u32_unaligned(q + 6);
  daf[k] = (int32_t)ld_u32_unaligned(q + 10);
}

// rows re-parsed on the host (strtof) -> their places in the site arrays
__global__ void k_patch_rows(int64_t n, const int64_t* __restrict__ idx, const int32_t* __restrict__ ps, const float* __restrict__ a,
                             const float* __restrict__ e, const uint32_t* __restrict__ m, const uint32_t* __restrict__ w,
                             int32_t* __restrict__ pos, float* __restrict__ ab, float* __restrict__ ae, uint32_t* __restrict__ meta,
                             uint32_t* __restrict__ mkt)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t r = idx[i];
  pos[r] = ps[i]; ab[r] = a[i]; ae[r] = e[i]; meta[r] = m[i]; mkt[r] = w[i];
}

}  // namespace colate

using namespace colate;


extern "C" {

int colate_ingest_begin(colate_handle* h, int n_chr, int64_t row_capacity)
{
  if (!h || n_chr <= 0 || row_capacity < 0 || row_capacity >= (int64_t(1) << 31))
    return fail(COLATE_ERR_ARG, "colate_ingest_begin: bad arguments");
  CK(cudaSetDevice(h->device));
  CK(h->pos.ensure(row_capacity * 4 + 4)); CK(h->ab.ensure(row_capacity * 4 + 4));
  CK(h->ae.ensure(row_capacity * 4 + 4)); CK(h->meta.ensure(row_capacity * 4 + 4)); CK(h->mkt.ensure(row_capacity * 4 + 4));
  h->sites_set = false;
  h->mkt_valid = false;
  h->flags_done = false;
  h->ing_active = true;
  h->ing_cap = row_capacity;
  h->ing_nchr = n_chr;
  h->ing_off.assign(1, 0);
  h->ing_ms = 0.0;
  h->ing_fallback_rows = 0;
  return 0;
}

// One .mut text already on its way to the device (d_text, ordered before h->stream's next work): line index,
// one thread per row, host re-parse of the rows the device flags.  host_text: the same bytes on the host (or
// nullptr: fetched back from the device if a row needs the host).  Returns the data rows.
static int64_t ingest_one(colate_handle* h, const char* d_text, int64_t n_bytes, const char* host_text)
{
  cudaStream_t s = h->stream;
  const int64_t row0 = h->ing_off.back();
  const char* text = host_text;
  const int location = host_text ? 0 : 1;
  const int64_t n_tiles = (n_bytes + ING_TILE - 1) / ING_TILE;
  CK(h->ing_tile_cnt.ensure(n_tiles * 4)); CK(h->ing_tile_off.ensure((n_tiles + 1) * 8)); CK(h->ing_status.ensure(64));
  CK(cudaEventRecord(h->ev[0], s));
  k_nl_count<<<(unsigned)n_tiles, ING_THREADS, 0, s>>>(d_text, n_bytes, h->ing_tile_cnt.as<int32_t>());
  k_tile_scan<<<1, 1024, 0, s>>>(h->ing_tile_cnt.as<int32_t>(), n_tiles, h->ing_tile_off.as<int64_t>());
  int64_t n_nl = 0;
  char last = 0;
  CK(cudaMemcpyAsync(&n_nl, h->ing_tile_off.as<int64_t>() + n_tiles, 8, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(&last, d_text + n_bytes - 1, 1, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  const int64_t n_lines = n_nl + (last != '\n' ? 1 : 0);
  const int64_t n_rows = n_lines > 0 ? n_lines - 1 : 0;          // minus the header line
  if (row0 + n_rows > h->ing_cap) return fail(COLATE_ERR_ARG, "colate_ingest_mut_text: row capacity of colate_ingest_begin exceeded");
  if (n_rows > 0) {
    const int64_t fb_cap = 1 << 16;
    CK(h->ing_nl.ensure((n_nl + 1) * 8)); CK(h->ing_fb.ensure(fb_cap * 8));
    const unsigned long long st0[2] = {~0ull, 0ull};
    CK(cudaMemcpyAsync(h->ing_status.p, st0, 16, cudaMemcpyHostToDevice, s));
    k_nl_index<<<(unsigned)n_tiles, ING_THREADS, 0, s>>>(d_text, n_bytes, h->ing_tile_off.as<int64_t>(), h->ing_nl.as<int64_t>());
    k_parse_mut<<<(unsigned)((n_rows + 255) / 256), 256, 0, s>>>(d_text, n_bytes, h->ing_nl.as<int64_t>(), n_nl, n_rows,
                                                                 h->pos.as<int32_t>() + row0, h->ab.as<float>() + row0,
                                                                 h->ae.as<float>() + row0, h->meta.as<uint32_t>() + row0,
                                                                 h->mkt.as<uint32_t>() + row0, h->ing_status.as<unsigned long long>(), h->ing_fb.as<int64_t>(), fb_cap);
    CK(cudaEventRecord(h->ev[1], s));
    unsigned long long st[2];
    CK(cudaMemcpyAsync(st, h->ing_status.p, 16, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    h->launches += 4;
    h->mut_texts_parsed += 1;
    float ms = 0;
    cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]);
    h->ing_ms += ms;
    if (st[0] != ~0ull) return fail(COLATE_ERR_IO, "Error reading a line in mut file (empty line or fewer than 10 fields), data row " + std::to_string(st[0] - 1));
    // rows the device could not convert with a correct-rounding guarantee: host strtof
    int64_t nfb = (int64_t)st[1];
    std::vector<int64_t> rows;
    if (nfb > fb_cap) { rows.resize(n_rows); for (int64_t i = 0; i < n_rows; i++) rows[i] = i; nfb = n_rows; }   // pathological file: everything
    else if (nfb > 0) { rows.resize(nfb); CK(cudaMemcpy(rows.data(), h->ing_fb.p, nfb * 8, cudaMemcpyDeviceToHost)); }
    if (nfb > 0) {
      std::vector<int64_t> nlp(n_nl);
      std::vector<char> htext;
      const char* ht = text;
      if (location) { htext.resize(n_bytes); CK(cudaMemcpy(htext.data(), d_text, n_bytes, cudaMemcpyDeviceToHost)); ht = htext.data(); }
      CK(cudaMemcpy(nlp.data(), h->ing_nl.p, n_nl * 8, cudaMemcpyDeviceToHost));
      // re-parsed rows are collected and scattered by one small kernel on the handle's stream (ordered against the
      // parse kernel before it and every consumer after it)
      std::vector<int64_t> pidx; std::vector<int32_t> ppos; std::vector<float> pab, pae; std::vector<uint32_t> pmeta, pw;
      pidx.reserve(rows.size()); ppos.reserve(rows.size()); pab.reserve(rows.size()); pae.reserve(rows.size()); pmeta.reserve(rows.size());
      pw.reserve(rows.size());
      for (int64_t r : rows) {
        const char* p = ht + nlp[r] + 1;
        const char* nl = ht + (r + 1 < n_nl ? nlp[r + 1] : n_bytes);
        std::string line(p, nl);                                  // NUL-terminated copy: strtof / strtol stop at the field's ';'
        line.push_back('\n');
        int32_t ps; float a, e; uint32_t m; int fl, nb; char type[16];
        if (!parse_mut_line_fields(line.data(), line.data() + line.size() - 1, &ps, &a, &e, &m, &fl, &nb, type))
          return fail(COLATE_ERR_IO, "Error reading following line in mut file: " + std::string(p, nl));
        pidx.push_back(row0 + r); ppos.push_back(ps); pab.push_back(a); pae.push_back(e); pmeta.push_back(m); pw.push_back(maketmp_word(fl, nb, type));
      }
      const size_t np = pidx.size();
      CK(h->d_tmp.ensure(np * 28 + 64));
      char* base = h->d_tmp.as<char>();
      int64_t* d_idx = (int64_t*)base;
      int32_t* d_pos = (int32_t*)(base + np * 8);
      float* d_ab = (float*)(base + np * 12);
      float* d_ae = (float*)(base + np * 16);
      uint32_t* d_meta = (uint32_t*)(base + np * 20);
      uint32_t* d_w = (uint32_t*)(base + np * 24);
      CK(cudaMemcpyAsync(d_idx, pidx.data(), np * 8, cudaMemcpyHostToDevice, s));
      CK(cudaMemcpyAsync(d_pos, ppos.data(), np * 4, cudaMemcpyHostToDevice, s));
      CK(cudaMemcpyAsync(d_ab, pab.data(), np * 4, cudaMemcpyHostToDevice, s));
      CK(cudaMemcpyAsync(d_ae, pae.data(), np * 4, cudaMemcpyHostToDevice, s));
      CK(cudaMemcpyAsync(d_meta, pmeta.data(), np * 4, cudaMemcpyHostToDevice, s));
      CK(cudaMemcpyAsync(d_w, pw.data(), np * 4, cudaMemcpyHostToDevice, s));
      k_patch_rows<<<(unsigned)((np + 255) / 256), 256, 0, s>>>((int64_t)np, d_idx, d_pos, d_ab, d_ae, d_meta, d_w, h->pos.as<int32_t>(),
                                                                h->ab.as<float>(), h->ae.as<float>(), h->meta.as<uint32_t>(),
                                                                h->mkt.as<uint32_t>());
      h->launches += 1;
      CK(cudaGetLastError());
      CK(cudaStreamSynchronize(s));   // the host vectors are locals
    }
    h->ing_fallback_rows += nfb;
  }
  h->ing_off.push_back(row0 + n_rows);
  return n_rows;
}


int64_t colate_ingest_mut_text(colate_handle* h, const char* text, int64_t n_bytes, int location)
{
  if (!h || !text || n_bytes < 0) return fail(COLATE_ERR_ARG, "colate_ingest_mut_text: bad arguments");
  if (!h->ing_active) return fail(COLATE_ERR_STATE, "colate_ingest_mut_text: call colate_ingest_begin first");
  if ((int)h->ing_off.size() > h->ing_nchr) return fail(COLATE_ERR_STATE, "colate_ingest_mut_text: more chromosomes than announced");
  CK(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const int64_t row0 = h->ing_off.back();
  if (n_bytes == 0) { h->ing_off.push_back(row0); return 0; }
  const char* d_text = text;
  if (!location) {
    CK(h->ing_text.ensure((size_t)n_bytes + 64));
    d_text = h->ing_text.as<char>();
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, text) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    if (pinned) {
      CK(cudaMemcpyAsync(h->ing_text.p, text, (size_t)n_bytes, cudaMemcpyHostToDevice, s));
    } else {
      // pageable caller memory: stage through two pinned bounce buffers so the copies run at PCIe speed
      // while the host fills the other buffer
      const size_t CH = (size_t)32 << 20;
      for (int k = 0; k < 2; k++)
        if (!h->ing_bounce[k]) { CK(cudaHostAlloc(&h->ing_bounce[k], CH, cudaHostAllocDefault)); CK(cudaEventCreateWithFlags(&h->ing_bounce_ev[k], cudaEventDisableTiming)); }
      int k = 0;
      for (size_t o = 0; o < (size_t)n_bytes; o += CH, k ^= 1) {
        const size_t m = std::min(CH, (size_t)n_bytes - o);
        CK(cudaEventSynchronize(h->ing_bounce_ev[k]));
        memcpy(h->ing_bounce[k], text + o, m);
        CK(cudaMemcpyAsync(h->ing_text.as<char>() + o, h->ing_bounce[k], m, cudaMemcpyHostToDevice, s));
        CK(cudaEventRecord(h->ing_bounce_ev[k], s));
      }
    }
  }
  return ingest_one(h, d_text, n_bytes, location ? nullptr : text);
}

// All chromosomes of a job in one call (texts[c] / n_bytes[c] in --chr order, pinned host memory or device memory):
// every text is copied on the handle's copy stream, and chromosome c is parsed on the compute stream as soon as
// its bytes have landed -- the parse kernels and the host's per-chromosome bookkeeping run under the copies of the
// following chromosomes.  rows_out[c] = data rows of chromosome c.  Equivalent to n calls of colate_ingest_mut_text.
int colate_ingest_mut_texts(colate_handle* h, int n_texts, const char* const* texts, const int64_t* n_bytes, int location,
                            int64_t* rows_out)
{
  if (!h || n_texts < 0 || (n_texts > 0 && (!texts || !n_bytes))) return fail(COLATE_ERR_ARG, "colate_ingest_mut_texts: bad arguments");
  if (!h->ing_active) return fail(COLATE_ERR_STATE, "colate_ingest_mut_texts: call colate_ingest_begin first");
  if ((int)h->ing_off.size() - 1 + n_texts > h->ing_nchr) return fail(COLATE_ERR_STATE, "colate_ingest_mut_texts: more chromosomes than announced");
  CK(cudaSetDevice(h->device));
  bool direct = location != 0;
  if (!direct) {   // pinned host memory copies asynchronously; anything else takes the bounce path text by text
    direct = true;
    for (int c = 0; c < n_texts && direct; c++) {
      if (n_bytes[c] <= 0) continue;
      cudaPointerAttributes attr;
      direct = cudaPointerGetAttributes(&attr, texts[c]) == cudaSuccess && attr.type == cudaMemoryTypeHost;
      cudaGetLastError();
    }
  }
  if (!direct || location != 0) {
    for (int c = 0; c < n_texts; c++) {
      const int64_t n = colate_ingest_mut_text(h, texts[c], n_bytes[c], location);
      if (n < 0) return (int)n;
      if (rows_out) rows_out[c] = n;
    }
    return 0;
  }
  std::vector<size_t> off(n_texts + 1, 0);
  for (int c = 0; c < n_texts; c++) {
    if (n_bytes[c] < 0 || (n_bytes[c] > 0 && !texts[c])) return fail(COLATE_ERR_ARG, "colate_ingest_mut_texts: bad text");
    off[c + 1] = off[c] + (((size_t)n_bytes[c] + 255) & ~(size_t)255);
  }
  CK(cudaStreamSynchronize(h->stream));                       // nothing may still read the text buffer this call replaces
  CK(h->ing_text.ensure(off[n_texts] + 64));
  while ((int)h->ing_evs.size() < n_texts) {
    cudaEvent_t e;
    CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    h->ing_evs.push_back(e);
  }
  for (int c = 0; c < n_texts; c++) {
    if (n_bytes[c] > 0) CK(cudaMemcpyAsync(h->ing_text.as<char>() + off[c], texts[c], (size_t)n_bytes[c], cudaMemcpyHostToDevice, h->copy_stream));
    CK(cudaEventRecord(h->ing_evs[c], h->copy_stream));
  }
  for (int c = 0; c < n_texts; c++) {
    int64_t n = 0;
    if (n_bytes[c] == 0) h->ing_off.push_back(h->ing_off.back());
    else {
      CK(cudaStreamWaitEvent(h->stream, h->ing_evs[c], 0));
      n = ingest_one(h, h->ing_text.as<char>() + off[c], n_bytes[c], texts[c]);
      if (n < 0) { cudaStreamSynchronize(h->copy_stream); return (int)n; }
    }
    if (rows_out) rows_out[c] = n;
  }
  return 0;
}

int colate_ingest_end(colate_handle* h)
{
  if (!h) return fail(COLATE_ERR_ARG, "colate_ingest_end: bad arguments");
  if (!h->ing_active || (int)h->ing_off.size() != h->ing_nchr + 1)
    return fail(COLATE_ERR_STATE, "colate_ingest_end: not every announced chromosome was ingested");
  CK(cudaSetDevice(h->device));
  CK(h->site_off.ensure((h->ing_nchr + 1) * 8));
  CK(cudaMemcpyAsync(h->site_off.p, h->ing_off.data(), (h->ing_nchr + 1) * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->n_chr = h->ing_nchr;
  h->n_site = h->ing_off.back();
  h->h_site_off = h->ing_off;
  h->ing_active = false;
  h->mut_rows_parsed += h->n_site;
  const int rc = sites_replaced_ext(h);
  h->mkt_valid = rc == 0;
  return rc;
}

int colate_ingest_fetch(colate_handle* h, int64_t row0, int64_t n_rows, int32_t* pos, float* age_begin, float* age_end, uint32_t* meta)
{
  if (!h || row0 < 0 || n_rows < 0) return fail(COLATE_ERR_ARG, "colate_ingest_fetch: bad arguments");
  const int64_t have = h->ing_active ? h->ing_off.back() : (h->sites_set ? h->n_site : 0);
  if (row0 + n_rows > have) return fail(COLATE_ERR_ARG, "colate_ingest_fetch: rows out of range");
  CK(cudaSetDevice(h->device));
  if (pos) CK(cudaMemcpy(pos, h->pos.as<int32_t>() + row0, n_rows * 4, cudaMemcpyDeviceToHost));
  if (age_begin) CK(cudaMemcpy(age_begin, h->ab.as<float>() + row0, n_rows * 4, cudaMemcpyDeviceToHost));
  if (age_end) CK(cudaMemcpy(age_end, h->ae.as<float>() + row0, n_rows * 4, cudaMemcpyDeviceToHost));
  if (meta) {
    CK(cudaMemcpy(meta, h->meta.as<uint32_t>() + row0, n_rows * 4, cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < n_rows; i++) meta[i] &= ~6u;   // bits 1-2 are the handle's own age-range marks (k_check_sites), not part of colate_site_meta()
  }
  return 0;
}

int colate_ingest_stats(colate_handle* h, double* kernel_ms, int64_t* host_fallback_rows)
{
  if (!h) return fail(COLATE_ERR_ARG, "colate_ingest_stats: bad arguments");
  if (kernel_ms) *kernel_ms = h->ing_ms;
  if (host_fallback_rows) *host_fallback_rows = h->ing_fallback_rows;
  return 0;
}

// .colate.in image -> genome slot, decoded on the device (replaces colate_read_colate_in + colate_chr_ranges +
// colate_set_genome; reader being replaced: coal.cpp:2126-2133, 2185-2192, 2205-2212).
int64_t colate_ingest_colate_in(colate_handle* h, int slot, const char* bytes, int64_t n_bytes, int n_chr,
                                const char* const* chr_names, int location)
{
  if (!h || slot < 0 || slot >= COLATE_MAX_GENOMES || n_bytes < 0 || (n_bytes > 0 && !bytes) || n_chr < 0 || (n_chr > 0 && !chr_names))
    return fail(COLATE_ERR_ARG, "colate_ingest_colate_in: bad arguments");
  if (!h->sites_set) return fail(COLATE_ERR_STATE, "colate_ingest_colate_in: call colate_set_sites / colate_ingest_end first");
  if (n_chr != h->n_chr) return fail(COLATE_ERR_ARG, "colate_ingest_colate_in: n_chr differs from the site set's");
  CK(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  std::vector<std::string> names(chr_names, chr_names + n_chr);
  std::vector<char> pulled;
  const char* host = bytes;
  if (location) {   // the run finder probes the image on the host
    pulled.resize((size_t)n_bytes);
    if (n_bytes) CK(cudaMemcpy(pulled.data(), bytes, (size_t)n_bytes, cudaMemcpyDeviceToHost));
    host = pulled.data();
  }
  GenomeDev& g = h->genomes[slot];
  const unsigned char* d_img = (const unsigned char*)bytes;
  if (!location && n_bytes > 0) {
    CK(h->ing_raw.ensure((size_t)n_bytes + 64));
    CK(cudaMemcpyAsync(h->ing_raw.p, bytes, (size_t)n_bytes, cudaMemcpyHostToDevice, s));   // under way while the host finds the runs
    d_img = h->ing_raw.as<unsigned char>();
  }
  std::vector<ColateInRun> runs;
  int64_t n_rec = colate_in_runs(host, n_bytes, names, runs);
  CK(g.bp.ensure(n_rec * 4 + 4)); CK(g.aaf.ensure(n_rec * 4 + 4)); CK(g.daf.ensure(n_rec * 4 + 4)); CK(g.alleles.ensure(n_rec * 2 + 4));
  CK(g.chr_first.ensure(n_chr * 8 + 8)); CK(g.chr_end.ensure(n_chr * 8 + 8));
  bool device_ok = true;
  if (n_rec > 0) {
    static_assert(sizeof(DevRun) == sizeof(ColateInRun), "run records are copied as they are");
    CK(h->d_tmp.ensure(runs.size() * sizeof(DevRun) + 64));
    int* d_bad = (int*)(h->d_tmp.as<char>() + runs.size() * sizeof(DevRun));
    CK(cudaMemcpyAsync(h->d_tmp.p, runs.data(), runs.size() * sizeof(DevRun), cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(d_bad, 0, 4, s));
    k_decode_colate_in<<<(unsigned)((n_rec + 255) / 256), 256, 0, s>>>(d_img, h->d_tmp.as<DevRun>(), (int)runs.size(), n_rec,
                                                                       g.bp.as<int32_t>(), g.aaf.as<int32_t>(), g.daf.as<int32_t>(),
                                                                       g.alleles.as<uint16_t>(), d_bad);
    h->launches += 1;
    CK(cudaGetLastError());
    int bad = 0;
    CK(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    device_ok = bad == 0;
  }
  std::vector<int64_t> first(n_chr + 1), end(n_chr + 1);
  if (device_ok) {
    chr_ranges_runs(n_chr, runs, first.data(), end.data());
  } else {
    // a record inside a run carries another header: interleaved chromosomes or mixed name lengths.  The
    // sequential decode is the definition; take it.
    const int64_t cap = n_bytes / 18 + 1;
    std::vector<int32_t> rc(cap), bp(cap), aaf(cap), daf(cap);
    std::vector<uint16_t> al(cap);
    n_rec = decode_colate_in_host(host, n_bytes, names, cap, rc.data(), bp.data(), aaf.data(), daf.data(), al.data());
    if (n_rec < 0) return n_rec;
    colate_chr_ranges(n_chr, n_rec, rc.data(), first.data(), end.data());
    CK(g.bp.ensure(n_rec * 4 + 4)); CK(g.aaf.ensure(n_rec * 4 + 4)); CK(g.daf.ensure(n_rec * 4 + 4)); CK(g.alleles.ensure(n_rec * 2 + 4));
    CK(cudaMemcpyAsync(g.bp.p, bp.data(), n_rec * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(g.aaf.p, aaf.data(), n_rec * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(g.daf.p, daf.data(), n_rec * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(g.alleles.p, al.data(), n_rec * 2, cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s));
    h->ing_genome_fallbacks += 1;
  }
  CK(cudaMemcpyAsync(g.chr_first.p, first.data(), n_chr * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(g.chr_end.p, end.data(), n_chr * 8, cudaMemcpyHostToDevice, s));
  g.n_rec = n_rec;
  const int rc2 = genome_replaced_ext(h, slot);
  if (rc2) return rc2;
  CK(cudaStreamSynchronize(s));   // first / end are locals
  return n_rec;
}

}  // extern "C"
