// Stage i kernels (parse_tmptmp, coal.cpp:2071-2321) on structure-of-arrays in HBM:
//   k_join      per genome: merge-join of the .colate.in records onto the site axis
//   k_cand/k_ok per pair: row filter + the two stream lookups incl. the sequential reader's
//               look-ahead rule (SURVEY.md A.3) as bitmap passes
//   k_*rank*    used-row rank = offset into the reference's generator stream
//   k_compact   used rows -> dense records in rank order, genomic block index
//   k_sample    THE per-mutation kernel: 100 Monte-Carlo age draws per used row from the
//               uniform stream in HBM (tile-ordered by k_gen, bulk-copied into per-warp rings),
//               exact bin index, per-lane byte counters in shared memory -> [slot][row] count tiles
//   k_replay    exact fp64 histograms: the reference's rounded additions replayed in row order
//               per genomic block, plus the "emp" slice

#include "device.cuh"
#include "exact_sum.cuh"

namespace colate {

constexpr int SCAN_ITEMS = 8;     // bitmap words per thread in the rank scan
constexpr int TS_ROWS_C = 32;      // used rows per count tile (== TS_ROWS below)
constexpr int ROW_BYTES_C = 192;
constexpr int SCAN_THREADS = 256;

// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int chr_of(const int64_t* __restrict__ site_off, int n_chr, int64_t m)
{
  int lo = 0, hi = n_chr;  // largest c with site_off[c] <= m
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (site_off[mid] <= m) lo = mid; else hi = mid;
  }
  return lo;
}

// largest p in [lo, m) whose bit is set, else -1
__device__ __forceinline__ int64_t prev_set(const uint32_t* __restrict__ bits, int64_t m, int64_t lo)
{
  int64_t w = m >> 5;
  uint32_t x = (m & 31) ? (bits[w] & ((1u << (m & 31)) - 1u)) : 0u;
  for (;;) {
    if (x) {
      int64_t p = (w << 5) + 31 - __clz(x);
      return p >= lo ? p : -1;
    }
    if ((w << 5) <= lo) return -1;
    w--;
    x = bits[w];
  }
}

__device__ __forceinline__ int64_t rank_of(const uint32_t* __restrict__ use, const uint32_t* __restrict__ word_rank, int64_t m)
{
  int64_t w = m >> 5;
  uint32_t r = word_rank[w];
  if (m & 31) r += __popc(use[w] & ((1u << (m & 31)) - 1u));
  return r;
}

// ------------------------------------------------------------------------------------------
// Record -> row join of one genome (coal.cpp:2181-2219 looks the row's position up in the record stream): sites and
// records are both ascending inside a chromosome, so a TILE of 256 consecutive sites of one chromosome only ever meets
// the records between the tile's first and last position.  k_join_bounds finds, per tile, the first record at or
// behind the tile's first position (one global binary search per 256 sites instead of one per site); k_join stages the
// tile's record positions in shared memory (coalesced), every site searches there, and a hit fetches the record's counts
// and alleles from a window of a few hundred records.  Tiles whose window does not fit (records much denser than sites)
// search in global memory as before.
constexpr int JOIN_TILE = 256;
constexpr int JOIN_CAP = 1024;     // record positions staged per tile

__device__ __forceinline__ void join_tile_of(int n_chr, const int32_t* __restrict__ tile_start, int t, const int64_t* __restrict__ site_off,
                                             int& c, int64_t& m0, int64_t& m1)
{
  int lo = 0, hi = n_chr;            // largest c with tile_start[c] <= t
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (tile_start[mid] <= t) lo = mid; else hi = mid; }
  c = lo;
  m0 = site_off[c] + (int64_t)(t - tile_start[c]) * JOIN_TILE;
  m1 = min(m0 + JOIN_TILE, site_off[c + 1]);
}

// everything k_join needs to know about a tile, found once per tile by k_join_bounds (k_join read it through a chain of four
// dependent lookups per thread before: tile -> chromosome -> rows -> record range -> window)
struct __align__(16) JoinTileInfo { int64_t m0, first, w0, w1; int32_t n_rows, pad_[3]; };

__global__ void k_join_bounds(int n_tiles, int n_chr, const int32_t* __restrict__ tile_start, const int64_t* __restrict__ site_off,
                              const int32_t* __restrict__ pos, const int64_t* __restrict__ chr_first, const int64_t* __restrict__ chr_end,
                              const int32_t* __restrict__ bp, JoinTileInfo* __restrict__ tile_info)
{
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  int c; int64_t m0, m1;
  join_tile_of(n_chr, tile_start, t, site_off, c, m0, m1);
  const int64_t first = chr_first[c], end = chr_end[c];
  int64_t lo = first, hi = end, lo2 = first, hi2 = end;
  if (first >= 0) {
    const int32_t p = pos[m0], q = pos[m1 - 1];      // first record at or behind the first position; first record behind the last one
    while (lo < hi || lo2 < hi2) {                   // (the two searches side by side: their loads overlap)
      if (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (bp[mid] < p) lo = mid + 1; else hi = mid; }
      if (lo2 < hi2) { const int64_t mid = (lo2 + hi2) >> 1; if (bp[mid] <= q) lo2 = mid + 1; else hi2 = mid; }
    }
  }
  JoinTileInfo ti;
  ti.m0 = m0; ti.first = first; ti.w0 = lo; ti.w1 = lo2; ti.n_rows = (int32_t)(m1 - m0); ti.pad_[0] = ti.pad_[1] = ti.pad_[2] = 0;
  tile_info[t] = ti;
}

__global__ void __launch_bounds__(JOIN_TILE)
k_join(const JoinTileInfo* __restrict__ tile_info,
       const int32_t* __restrict__ pos, const uint32_t* __restrict__ meta,
       const int32_t* __restrict__ bp, const int32_t* __restrict__ aaf,
       const int32_t* __restrict__ daf, const uint16_t* __restrict__ alleles,
       int32_t* __restrict__ j_aaf, int32_t* __restrict__ j_daf,
       int32_t* __restrict__ j_prevbp, uint8_t* __restrict__ j_flag)
{
  __shared__ int32_t sbp[JOIN_CAP + 1];     // bp[w0 - 1 .. w1): the window and the record in front of it
  const JoinTileInfo ti = tile_info[blockIdx.x];
  const int64_t m0 = ti.m0, m1 = ti.m0 + ti.n_rows, first = ti.first;
  const int64_t m = m0 + threadIdx.x;
  if (first < 0) {                           // the reader never reaches this chromosome in this file
    if (m < m1) { j_aaf[m] = 0; j_daf[m] = 0; j_prevbp[m] = -1; j_flag[m] = 0; }
    return;
  }
  const int64_t w0 = ti.w0, w1 = ti.w1;      // records with a position inside [first, last position of the tile]
  // (the row's own word and position are requested before the window is staged: their latency runs under the staging loads)
  const uint32_t mt = m < m1 ? meta[m] : 0u;
  const int32_t p = m < m1 ? pos[m] : 0;
  const int64_t base = w0 > first ? w0 - 1 : w0;                       // also the record in front of the window (for j_prevbp)
  const int n_w = (int)(w1 - base);
  const bool staged = n_w <= JOIN_CAP + 1;
  if (staged) for (int i = threadIdx.x; i < n_w; i += JOIN_TILE) sbp[i] = bp[base + i];
  __syncthreads();
  if (m >= m1) return;
  int32_t a = 0, d = 0, pb = -1;
  uint8_t fl = 0;
  if (mt & 1u) {
    int64_t k;
    int32_t hit_bp, prev_bp = -1;
    if (staged) {
      int lo = (int)(w0 - base), hi = n_w;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (sbp[mid] < p) lo = mid + 1; else hi = mid; }
      k = base + lo;
      hit_bp = lo < n_w ? sbp[lo] : -1;
      if (lo > 0) prev_bp = sbp[lo - 1];
    } else {
      int64_t lo = w0, hi = w1;
      while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (bp[mid] < p) lo = mid + 1; else hi = mid; }
      k = lo;
      hit_bp = lo < w1 ? bp[lo] : -1;
      if (lo > first) prev_bp = bp[lo - 1];
    }
    if (k < w1 && hit_bp == p) {
      fl = 1;
      a = aaf[k];
      d = daf[k];
      pb = k > first ? prev_bp : -1;
      const uint32_t al = alleles[k];
      if ((al & 0xffu) == ((mt >> 8) & 0xffu) && (al >> 8) == ((mt >> 16) & 0xffu)) fl |= 2;
    }
  }
  j_aaf[m] = a; j_daf[m] = d; j_prevbp[m] = pb; j_flag[m] = fl;
}

// Pileup genome (SURVEY.md 8f N3: the bam front-ends, coal.cpp:1884-1929 reference / 1935-1980 target): the decoder hands
// over, per .mut row, the reads showing A, C, G, T at the row's position (bam_parser::count_alleles at bp_mut - 1; all zero =
// not covered).  The row's own alleles pick AAF / DAF out of the four counts ('0' / '1' pick nothing: 0); the row is usable iff
// reads > 0, (AAF > 0 || DAF > 0) and at most two alleles were seen (coal.cpp:1916-1917, 1967-1968).  The pileup ring is
// random access, so there is no look-ahead rule: j_prevbp = INT_MAX lets every candidate pass k_ok's stream test.
__device__ __forceinline__ int acgt_index(uint32_t c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1; }
__global__ void k_pileup_join(int64_t n_site, const uint32_t* __restrict__ meta, const int4* __restrict__ counts,
                              int32_t* __restrict__ j_aaf, int32_t* __restrict__ j_daf, int32_t* __restrict__ j_prevbp, uint8_t* __restrict__ j_flag)
{
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n_site) return;
  const uint32_t mt = meta[m];
  int32_t a = 0, d = 0;
  uint8_t fl = 0;
  if (mt & 1u) {
    const int4 c = counts[m];
    if (c.w < 0) {                                 // colate_set_row_counts: (AAF, DAF) already resolved by a bcf decoder
      a = c.x; d = c.y;
      if (a > 0 || d > 0) fl = 3;
      j_aaf[m] = a; j_daf[m] = d; j_prevbp[m] = 0x7fffffff; j_flag[m] = fl;
      return;
    }
    const int cc[4] = {c.x, c.y, c.z, c.w};
    const int reads = c.x + c.y + c.z + c.w;
    const int n_alleles = (c.x > 0) + (c.y > 0) + (c.z > 0) + (c.w > 0);
    const int ia = acgt_index((mt >> 8) & 0xffu), id = acgt_index((mt >> 16) & 0xffu);
    if (reads > 0) {                               // (the counts stay 0 otherwise: coal.cpp:1879-1882)
      if (ia >= 0) a = cc[ia];
      if (id >= 0) d = cc[id];
      if ((a > 0 || d > 0) && n_alleles <= 2) fl = 3;
    }
  }
  j_aaf[m] = a; j_daf[m] = d; j_prevbp[m] = 0x7fffffff; j_flag[m] = fl;
}

// ---- pileup of decoded alignment records (SURVEY.md 8f N3, the decoder's counting loop) ----------------------------------------
// bam_parser (include/vcf/htslib.cpp) keeps, for the positions around the one parse_onebambam / maketmp_bam look up, how many
// reads show A, C, G, T: count_alleles_for_read (htslib.cpp:60-168) per read, read_to_pos (426-437) to stay ahead of the
// lookups.  At lookup time a position's counts are those of ALL reads of the contig that cover it (reads are sorted by start
// and far shorter than half the ring), so the ring reduces to a function of the reads:
//   a read counts iff mapq >= mapq_th, len >= len_th and, over its bases i in [3, len - 3) with quality >= 30 that lie inside the
//   reference genome, total > 0 and total - matching <= mismatch_th (htslib.cpp:63-99, 143);
//   it then adds one to column A/C/G/T of every position pos + i, i in [3, len - 3), whose base quality is >= 30 (145-161).
// k_read_filter: thread = read -> pass flag.  k_pileup_rows: thread = .mut row of the contig: the reads that can cover its
// position start in (p - max_len, p]: binary search in the sorted starts, then a short scan.  No atomics, no ring.
// One quirk of the reference is reproduced: the FIRST read of every contig is counted by assign_contig (htslib.cpp:535-566), which
// leaves `q` pointing at the record's packed 4-bit sequence (bam_get_seq, line 549) instead of its qualities (read_entry
// re-points it, line 406).  For that one read "quality i" is byte i of {packed sequence, then the qualities}: found by the
// golden test (one row of the fixture differed), pinned by it.
__device__ __forceinline__ int nt16_code(uint8_t c)
{
  const char* t = "=ACMGRSVTWYHKDBN";          // seq_nt16_str: bam_parser::seq holds these letters
  int k = 15;
#pragma unroll
  for (int i = 0; i < 16; i++) k = (c == (uint8_t)t[i]) ? i : k;
  return k;
}
// k_quirk: index of the contig's first record in the arrays (0), or -1 when they do not start the contig (a later BAM chunk)
__device__ __forceinline__ int read_base_quality(int64_t k, int64_t k_quirk, int64_t i, int l, int64_t o, const uint8_t* __restrict__ seq,
                                                 const uint8_t* __restrict__ qual)
{
  if (k != k_quirk) return qual[o + i];
  const int64_t nb = ((int64_t)l + 1) >> 1;
  if (i >= nb) return qual[o + i - nb];
  const int hi = nt16_code(seq[o + 2 * i]), lo = 2 * i + 1 < l ? nt16_code(seq[o + 2 * i + 1]) : 0;
  return (hi << 4) | lo;
}
__global__ void k_read_filter(int64_t n_reads, const int32_t* __restrict__ pos, const uint8_t* __restrict__ mapq, const int32_t* __restrict__ len,
                              const int64_t* __restrict__ off, const uint8_t* __restrict__ seq, const uint8_t* __restrict__ qual,
                              const uint8_t* __restrict__ ref, int64_t ref_len, int mapq_th, int len_th, int mismatch_th, int64_t k_quirk,
                              uint8_t* __restrict__ pass)
{
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_reads) return;
  const int l = len[k];
  bool ok = false;
  if ((int)mapq[k] >= mapq_th && l >= len_th) {
    const int64_t p = pos[k], o = off[k];
    int total = 0, matching = 0;
    for (int i = 3; i < l - 3; i++) {
      if (p + i >= ref_len) break;
      if (read_base_quality(k, k_quirk, i, l, o, seq, qual) >= 30) { total++; matching += ref[p + i] == seq[o + i]; }
    }
    ok = total > 0 && total - matching <= mismatch_th;
  }
  pass[k] = ok ? 1 : 0;
}

__global__ void k_pileup_rows(int64_t row0, int64_t n_rows, const int32_t* __restrict__ site_pos, int64_t n_reads, const int32_t* __restrict__ pos,
                              const int32_t* __restrict__ len, const int64_t* __restrict__ off, const uint8_t* __restrict__ seq,
                              const uint8_t* __restrict__ qual, const uint8_t* __restrict__ pass, int max_len, int64_t k_quirk,
                              int4* __restrict__ pile)
{
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n_rows) return;
  const int64_t p = (int64_t)site_pos[row0 + m] - 1;          // 0-based position of the row (coal.cpp:1885)
  int64_t lo = 0, hi = n_reads;                                // first read with start > p - max_len
  while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if ((int64_t)pos[mid] <= p - max_len) lo = mid + 1; else hi = mid; }
  int4 c = pile[row0 + m];
  for (int64_t k = lo; k < n_reads && (int64_t)pos[k] <= p; k++) {
    if (!pass[k]) continue;
    const int64_t i = p - pos[k];
    if (i < 3 || i >= (int64_t)len[k] - 3) continue;
    if (read_base_quality(k, k_quirk, i, len[k], off[k], seq, qual) < 30) continue;
    const uint8_t b = seq[off[k] + i];
    c.x += b == 'A'; c.y += b == 'C'; c.z += b == 'G'; c.w += b == 'T';
  }
  pile[row0 + m] = c;
}

__global__ void k_pack_row_counts(int64_t n_site, const int32_t* __restrict__ aaf, const int32_t* __restrict__ daf, int4* __restrict__ pile)
{
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m < n_site) pile[m] = make_int4(aaf[m], daf[m], 0, -1);       // .w = -1: "counts of the row's two alleles", not an A/C/G/T pileup
}

// ---- input order (COLATE_ERR_ORDER) ---------------------------------------------------------
// k_join's binary search and the find-previous-candidate rule of k_ok equal the reference's sequential reader
// (coal.cpp:2184-2217) only on ascending positions: .mut rows ascending within a chromosome, .colate.in records
// ascending within the record range the reader can reach on a chromosome.  One pass each; equal neighbours are fine.
__global__ void k_check_sites(int64_t n_site, int n_chr, const int64_t* __restrict__ site_off, const int32_t* __restrict__ pos,
                              const float* __restrict__ ab, const float* __restrict__ ae, uint32_t* __restrict__ meta, double thr185,
                              int* __restrict__ flag)
{
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n_site) return;
  if (m > 0 && pos[m] < pos[m - 1] && site_off[chr_of(site_off, n_chr, m)] != m) *flag = 1;   // a descent is legal only at a chromosome start
  // Age interval against the end of the age grid (bin 185 starts where 10 * age reaches thr185), from the row alone:
  //   bit 1  age_begin > 0 and the interval reaches past the grid: the reference redraws every sample beyond it
  //          (coal.cpp:2279-2294) -- the row takes the rejection-sampling path (abi.cu: sample_segmented)
  //   bit 2  the reference cannot process the row: age_begin <= 0 with the interval past the grid (it writes past the
  //          end of the histogram, coal.cpp:2269) or age_begin itself past the grid (its loop never ends)
  uint32_t mt = meta[m] & ~6u;
  if (mt & 1u) {
    const double b = fmax((double)ab[m], 0.0), e = (double)ae[m];   // coal.cpp:2225 with ref_age == 0 (coal.cpp:2075)
    const bool past = __dmul_rn(10.0, e) >= thr185;
    if (b > 0.0) {
      if (__dmul_rn(10.0, b) >= thr185) mt |= 4u; else if (past) mt |= 2u;
    } else if (past) mt |= 4u;
  }
  meta[m] = mt;
}
__global__ void k_check_genome(int64_t n_rec, int n_chr, const int64_t* __restrict__ chr_first, const int64_t* __restrict__ chr_end,
                               const int32_t* __restrict__ bp, int* __restrict__ flag)
{
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k == 0 || k >= n_rec) return;
  if (bp[k] < bp[k - 1])
    for (int c = 0; c < n_chr; c++)
      if (chr_first[c] >= 0 && k > chr_first[c] && k < chr_end[c]) *flag = 1;
}

// one stream lookup for every candidate row (coal.cpp:2181-2199 / 2201-2219): the row keeps
// `use` iff a record sits at its position with the same alleles, that record had not already
// been pulled in by the look-ahead of an earlier candidate (or by the chromosome seek), and
// DAF_ref != 0 (reference stream) / AAF+DAF != 0 (target stream).
// candidate for the reference stream = row filter x masks (coal.cpp:2150-2181), straight from the site word and the mask bits
__device__ __forceinline__ bool is_cand(int64_t m, const uint32_t* __restrict__ meta, const uint32_t* __restrict__ tmask,
                                        const uint32_t* __restrict__ rmask)
{
  bool c = meta[m] & 1u;
  if (tmask) c = c && ((tmask[m >> 5] >> (m & 31)) & 1u);
  if (rmask) c = c && ((rmask[m >> 5] >> (m & 31)) & 1u);
  return c;
}

template <bool IS_REF>
__global__ void k_ok(int64_t n_site, int n_chr, const int64_t* __restrict__ site_off, const int32_t* __restrict__ pos,
                     const uint32_t* __restrict__ in_bits, const uint32_t* __restrict__ tmask, const uint32_t* __restrict__ rmask,
                     const int32_t* __restrict__ j_aaf,
                     const int32_t* __restrict__ j_daf, const int32_t* __restrict__ j_prevbp,
                     const uint8_t* __restrict__ j_flag, uint32_t* __restrict__ out_bits, const uint32_t* __restrict__ meta,
                     int64_t* __restrict__ misc)
{
  int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool ok = false;
  if (m < n_site) {
    // Every load the common case needs is issued up front (coalesced streams, none depends on another): the kernel was a chain
    // of five dependent global loads per row (flag -> counts -> chromosome -> previous candidate -> its position) and spent 70 %
    // of its time waiting for them.  The previous candidate is row m - 1 for 93 % of the rows; the walk back is the rare case.
    const uint32_t mt = meta[m];
    const uint8_t fl = j_flag[m];
    const int32_t daf = j_daf[m], aaf = IS_REF ? 0 : j_aaf[m], prevbp = j_prevbp[m];
    const int64_t p1 = m > 0 ? m - 1 : 0;
    const int32_t pos_p1 = pos[p1];
    // the reference stream's candidates come straight from the site words (no bitmap pass in front of this kernel), the
    // target stream's from the bitmap the reference pass wrote
    bool cand, cand_p1;
    if (IS_REF) {
      cand = mt & 1u;
      cand_p1 = meta[p1] & 1u;
      if (tmask) { cand = cand && ((tmask[m >> 5] >> (m & 31)) & 1u); cand_p1 = cand_p1 && ((tmask[p1 >> 5] >> (p1 & 31)) & 1u); }
      if (rmask) { cand = cand && ((rmask[m >> 5] >> (m & 31)) & 1u); cand_p1 = cand_p1 && ((rmask[p1 >> 5] >> (p1 & 31)) & 1u); }
    } else {
      cand = ((in_bits[m >> 5] >> (m & 31)) & 1u) != 0;
      cand_p1 = ((in_bits[p1 >> 5] >> (p1 & 31)) & 1u) != 0;
    }
    if (cand && (fl & 3) == 3 && (IS_REF ? (daf != 0) : ((aaf + daf) != 0))) {
      const int64_t lo = site_off[chr_of(site_off, n_chr, m)];
      int32_t prev_cand_pos;
      if (m - 1 < lo) prev_cand_pos = 0;                       // first row of the chromosome: no earlier candidate
      else if (cand_p1) prev_cand_pos = pos_p1;
      else {
        int64_t p;
        if (IS_REF) { p = m - 2; while (p >= lo && !is_cand(p, meta, tmask, rmask)) p--; if (p < lo) p = -1; }
        else p = prev_set(in_bits, m - 1, lo);
        prev_cand_pos = p >= 0 ? pos[p] : 0;
      }
      ok = prev_cand_pos <= prevbp;
    }
    if (!IS_REF && ok) {   // a USED row: does it need the rejection path, or is it one the reference cannot process?
      if (mt & 4u) misc[3] = 1;
      if (mt & 2u) atomicAdd((unsigned long long*)&misc[4], 1ull);
    }
  }
  uint32_t b = __ballot_sync(0xffffffffu, ok);
  if ((threadIdx.x & 31) == 0 && m < n_site) out_bits[m >> 5] = b;
}

// ---- rank of every bitmap word (exclusive prefix popcount) --------------------------------
__global__ void k_popc_blocksum(const uint32_t* __restrict__ words, int64_t n_words, uint32_t* __restrict__ sums)
{
  __shared__ uint32_t s[SCAN_THREADS / 32];
  int64_t base = ((int64_t)blockIdx.x * SCAN_THREADS + threadIdx.x) * SCAN_ITEMS;
  uint32_t v = 0;
  for (int i = 0; i < SCAN_ITEMS; i++) if (base + i < n_words) v += __popc(words[base + i]);
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (int i = 0; i < SCAN_THREADS / 32; i++) t += s[i];
    sums[blockIdx.x] = t;
  }
}

__global__ void k_scan_sums(uint32_t* __restrict__ sums, int n, uint32_t* __restrict__ total)
{
  if (threadIdx.x == 0 && blockIdx.x == 0) {  // n is a few hundred
    uint32_t run = 0;
    for (int i = 0; i < n; i++) { uint32_t v = sums[i]; sums[i] = run; run += v; }
    *total = run;
  }
}

__global__ void k_word_rank(const uint32_t* __restrict__ words, int64_t n_words, const uint32_t* __restrict__ block_off,
                            const uint32_t* __restrict__ total, uint32_t* __restrict__ word_rank, int32_t* __restrict__ row_of_rank)
{
  __shared__ uint32_t s[SCAN_THREADS / 32];
  int64_t base = ((int64_t)blockIdx.x * SCAN_THREADS + threadIdx.x) * SCAN_ITEMS;
  uint32_t loc[SCAN_ITEMS];
  uint32_t v = 0;
  for (int i = 0; i < SCAN_ITEMS; i++) { loc[i] = v; if (base + i < n_words) v += __popc(words[base + i]); }
  uint32_t incl = v;
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  if (lane == 31) s[wid] = incl;
  __syncthreads();
  uint32_t woff = 0;
  for (int i = 0; i < wid; i++) woff += s[i];
  uint32_t excl = block_off[blockIdx.x] + woff + incl - v;
  for (int i = 0; i < SCAN_ITEMS; i++)
    if (base + i < n_words) {
      word_rank[base + i] = excl + loc[i];
      // the inverse map for k_compact (thread = used row): which site has rank r (it searched word_rank for it before: 18 dependent loads)
      uint32_t w = words[base + i], r = excl + loc[i];
      while (w) { const int b = __ffs(w) - 1; w &= w - 1; row_of_rank[r++] = (int32_t)(((base + i) << 5) + b); }
    }
  if (blockIdx.x == 0 && threadIdx.x == 0) word_rank[n_words] = *total;
}

// per chromosome: used rows, genomic blocks (coal.cpp:2227-2234, 2306-2310), block base
__global__ void k_chr(int n_chr, const int64_t* __restrict__ site_off, const int32_t* __restrict__ pos,
                      const uint32_t* __restrict__ use, const uint32_t* __restrict__ word_rank,
                      int64_t* __restrict__ chr_used, int32_t* __restrict__ chr_blocks, int32_t* __restrict__ chr_block_base,
                      int64_t* __restrict__ misc)
{
  // thread = chromosome for the lookups (dependent loads), then one thread strings the block bases together
  __shared__ int s_nb[1024];
  __shared__ long long s_used[1024];
  for (int c0 = 0; c0 < n_chr; c0 += 1024) {                  // (more than 1024 chromosomes: in rounds; the running sums live in misc)
    const int c = c0 + threadIdx.x;
    if (c < n_chr) {
      const int64_t lo = site_off[c], hi = site_off[c + 1];
      const int64_t used = rank_of(use, word_rank, hi) - rank_of(use, word_rank, lo);
      const int64_t p = hi > lo ? prev_set(use, hi, lo) : -1;
      s_nb[threadIdx.x] = p >= 0 ? (pos[p] - 1) / COLATE_BLOCK_BASES + 1 : 1;
      s_used[threadIdx.x] = used;
      chr_used[c] = used;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int base = c0 ? (int)misc[1] : 0;
      int64_t tot = c0 ? misc[0] : 0;
      for (int i = 0; i < min(1024, n_chr - c0); i++) {
        chr_blocks[c0 + i] = s_nb[i];
        chr_block_base[c0 + i] = base;
        base += s_nb[i];
        tot += s_used[i];
      }
      misc[0] = tot;
      misc[1] = base;
    }
    __syncthreads();
  }
  if (n_chr == 0 && threadIdx.x == 0) { misc[0] = 0; misc[1] = 0; }
}

// used rows -> dense records in rank order:
//   hdr[r]  = {(age_end - age_begin) * 2^-64, age_begin, weight into shared, weight into notshared} (fp64 x4); rows with
//             age_begin <= 0 add nothing to shared (k_replay tests .y, not the weight: raw count weights may be negative)
//   e_b2/e_ws/e_wn[r] = bin and weights of the row's single "emp" contribution (255 = none)
//   u_blk[r] = genomic block (index local to this handle)
__global__ void k_compact(int64_t n_site, int n_chr, const int64_t* __restrict__ site_off, const int32_t* __restrict__ pos,
                          const float* __restrict__ ab, const float* __restrict__ ae,
                          const int32_t* __restrict__ row_of_rank,
                          const int32_t* __restrict__ chr_block_base,
                          const int32_t* __restrict__ t_aaf, const int32_t* __restrict__ t_daf,
                          const int32_t* __restrict__ r_aaf, const int32_t* __restrict__ r_daf,
                          const double* __restrict__ thr10,
                          double4* __restrict__ hdr, uint8_t* __restrict__ e_b2, double* __restrict__ e_ws,
                          double* __restrict__ e_wn, int32_t* __restrict__ u_blk, int64_t* __restrict__ misc,
                          const uint32_t* __restrict__ meta, int64_t* __restrict__ deep_rows, int64_t deep_cap, int raw_weights)
{
  // thread = used row (rank r): one row in eight is used, so a thread per site would leave the warps of the
  // division-heavy part below nearly empty.  Site of rank r: row_of_rank, written by the rank scan (k_word_rank).
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= misc[0]) return;
  const int64_t m = row_of_rank[r];
  int c = chr_of(site_off, n_chr, m);
  // pseudo-genotype, coal.cpp:2236-2242: float /= double, then round half away
  const int32_t dt = t_daf[m], at = t_aaf[m];
  const double half_n = (double)(dt + at) / 2.0;
  float fd = __double2float_rn(__ddiv_rn((double)(float)dt, half_n));
  float fa = __double2float_rn(__ddiv_rn((double)(float)at, half_n));
  fd = roundf(fd);
  fa = roundf(fa);
  float b = ab[m];
  if (b < 0.0f) b = 0.0f;  // coal.cpp:2225 with ref_age == 0 (coal.cpp:2075)
  const float e = ae[m];
  const int32_t dafr = r_daf[m], nr = r_daf[m] + r_aaf[m];
  const double abd = (double)b;
  // float * int -> float, then / double (coal.cpp:2255-2256, 2269, 2291-2292)
  // raw_weights (the bcf / bam front-ends, SURVEY.md 8f N3): the counts themselves, int * int -> double
  // (coal.cpp:2005-2006, 2019, 2038-2039; 1164-1165, 1179, 1196-1197 with AAF_target = N_target - DAF_target).  The
  // reference multiplies in int: a product past 2^31 (depths above ~46 k on both sides) wraps to a negative weight, and the
  // reference adds that.  The wrap is spelled out in unsigned arithmetic here (signed overflow is undefined in C++).
  const double num_s = raw_weights ? (double)(int32_t)((uint32_t)dt * (uint32_t)dafr) : (double)__fmul_rn(fd, __int2float_rn(dafr));
  const double num_n = raw_weights ? (double)(int32_t)((uint32_t)at * (uint32_t)dafr) : (double)__fmul_rn(fa, __int2float_rn(dafr));
  const double den = __dmul_rn((double)nr, 100.0);
  // .x = (age_end - age_begin) * 2^-64: the sampling kernel multiplies it with the 64-bit integer
  // x2:x1 converted once (exact power-of-two scaling, same rounding as U * (age_end - age_begin))
  // .y = age_begin: rows with .y <= 0 add nothing to the shared histogram (coal.cpp:2259)
  hdr[r] = make_double4(__dmul_rn(__dsub_rn((double)e, abd), 0x1p-64), abd, __ddiv_rn(num_s, den), __ddiv_rn(num_n, den));
  uint8_t b2 = 255;
  double ws = 0.0, wn = 0.0;
  if (abd <= 0.0) {  // coal.cpp:2247-2256 with age == 0
    const double x10 = (double)__fmul_rn(10.0f, e);
    int lo = 0, hi = NBINS;  // number of thresholds <= x10
    while (lo < hi) { int mid = (lo + hi + 1) >> 1; if (x10 >= thr10[mid]) lo = mid; else hi = mid - 1; }
    if (lo < NBINS) { b2 = (uint8_t)lo; ws = __ddiv_rn(num_s, (double)nr); wn = __ddiv_rn(num_n, (double)nr); }
  }
  e_b2[r] = b2; e_ws[r] = ws; e_wn[r] = wn;
  u_blk[r] = chr_block_base[c] + (pos[m] - 1) / COLATE_BLOCK_BASES;
  // rows whose samples the reference redraws when they fall past the age grid (meta bit 1, k_check_sites): listed
  // (in any order; the host sorts the few of them) for the rejection-sampling path
  if (meta[m] & 2u) {
    const unsigned long long k = atomicAdd((unsigned long long*)&misc[5], 1ull);
    if ((int64_t)k < deep_cap) deep_rows[k] = r;
  }
}

// rejection-sampling path: the count rows of a segment sampled into scratch tiles -> their places in the tile array of all
// used rows ([tile][slot][row % 32] bytes); and one count row computed on the host
__global__ void k_scatter_count_rows(const uint8_t* __restrict__ seg_tiles, int64_t n_rows, int64_t row0, uint8_t* __restrict__ cnt_tiles)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // (row of the segment, slot)
  if (i >= n_rows * ROW_BYTES_C) return;
  const int64_t j = i / ROW_BYTES_C, r = row0 + j;
  const int slot = (int)(i - j * ROW_BYTES_C);
  cnt_tiles[(r / TS_ROWS_C) * (ROW_BYTES_C * TS_ROWS_C) + slot * TS_ROWS_C + (r % TS_ROWS_C)] =
      seg_tiles[(j / TS_ROWS_C) * (ROW_BYTES_C * TS_ROWS_C) + slot * TS_ROWS_C + (j % TS_ROWS_C)];
}
__global__ void k_put_count_row(const uint8_t* __restrict__ row_cnt /*[192]*/, int64_t r, uint8_t* __restrict__ cnt_tiles)
{
  const int slot = threadIdx.x;
  if (slot < ROW_BYTES_C) cnt_tiles[(r / TS_ROWS_C) * (ROW_BYTES_C * TS_ROWS_C) + slot * TS_ROWS_C + (r % TS_ROWS_C)] = row_cnt[slot];
}

// rank range of every genomic block
__global__ void k_block_ranges(const int32_t* __restrict__ u_blk, const int64_t* __restrict__ misc, int64_t* __restrict__ blk_rank_start)
{
  const int64_t n_used = misc[0];
  const int n_blocks = (int)misc[1];
  for (int b = threadIdx.x; b <= n_blocks; b += blockDim.x) {
    int64_t lo = 0, hi = n_used;  // first rank with u_blk >= b
    while (lo < hi) {
      int64_t mid = (lo + hi) >> 1;
      if (u_blk[mid] < b) lo = mid + 1; else hi = mid;
    }
    blk_rank_start[b] = lo;
  }
}

// ---- mbarrier / bulk-copy (TMA) helpers ------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// one lane waits (suspended by the hardware, woken by the phase change), the warp follows: keeps
// 20-odd idle warps from hammering the barrier unit while a few warps work
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity, int lane)
{
  if (lane == 0) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity), "r"(100000u) : "memory");
  }
  __syncwarp();
}
// global -> shared bulk async copy (TMA engine, SASS UBLKCP), completion counted on `bar`
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------------------------------
// uniform_real_distribution<double>(0,1) from two engine words, bit-exact with libstdc++'s
// generate_canonical<double,53>: (x1 + x2*2^32) / 2^64 rounded once and clamped below 1.  Here the
// 64-bit integer x2:x1 is converted with one round-to-nearest I2F (the same single rounding), the
// clamp becomes a min with 2^64 - 2^11, and the factor 2^-64 is folded into the row's length.
__device__ __forceinline__ double u64_scaled(uint32_t x1, uint32_t x2)
{
  const double v = __ull2double_rn(((unsigned long long)x2 << 32) | x1);
  // v == 2^64 (x2:x1 >= 2^64 - 2^10) -> the double just below: bit pattern minus one
  const int hi = __double2hiint(v);
  const bool top = hi == 0x43f00000;
  return __hiloint2double(top ? 0x43efffff : hi, top ? -1 : __double2loint(v));
}

// max(0,(int)round(log(10*a)*10)+1) (coal.cpp:2265/2284) without evaluating log: the top 17 bits
// of a select a cell of width 2^-6 in log2 (narrower than an age bin, e^0.1), a table gives the
// bin at the cell's lower edge and one exact threshold (host-computed against libm) settles it.
// Returns the count slot (internal.h: slot_of_bin) of the sample's age bin.
__device__ __forceinline__ int slot_of_age(double a, const uint16_t* lut, const double* thrP)
{
  int cell = (__double2hiint(a) >> LUT_SHIFT) - LUT_BASE;
  cell = max(0, min(cell, LUT_N - 1));
  int p = lut[cell];           // bit 15: an age-bin threshold lies inside this cell (about 1 cell in 5)
  if (p & 0x8000) {
    p &= 0xff;
    if (a >= thrP[p]) p += 1;   // slot of the next bin
  }
  return p;
}

constexpr int TS_ROWS = 32;            // used rows per tile: one per lane
constexpr int CH_WORDS = SAMPLE_CHUNK_WORDS;  // engine words per chunk and row: a ring slot holds 32 rows x CH_WORDS, one contiguous block of the stream
constexpr int SUB_WORDS = 20;                 // words per unrolled step = 10 samples
constexpr int N_CHUNK = 200 / CH_WORDS;
constexpr int ROW_BYTES = 192;         // per-row sample counts, one byte per count slot (188 used)
constexpr int TILE_BYTES = ROW_BYTES * TS_ROWS;   // count tile of 32 rows: [slot][row] bytes
static_assert(TS_ROWS == TS_ROWS_C && ROW_BYTES == ROW_BYTES_C, "count-tile geometry");
#ifndef S2_WARPS_
#define S2_WARPS_ 4
#endif
#ifndef S2_RING_
#define S2_RING_ 2
#endif
constexpr int S2_WARPS = S2_WARPS_;    // warps per CTA, each with its own tile, ring and counters
constexpr int S2_RING = S2_RING_;      // ring slots per warp (one being read, the others in flight)
constexpr int N_STEP = N_CHUNK;
struct __align__(128) SampleWarp {
  uint32_t chunk[S2_RING][TS_ROWS][CH_WORDS];   // one block of the stream per slot: 32 rows x CH_WORDS (row stride of 20 words: conflict-free LDS.128)
  uint32_t cnt[ROW_WORDS][TS_ROWS];             // this tile's counts: word w of lane L = slots 4w..4w+3 of row L (bank = lane)
  uint64_t full[S2_RING];
};

// THE per-mutation kernel.  Thread = used row: a warp owns a tile of 32 consecutive used rows and streams
// their 100 x 2 generator words (800 B per row) from HBM.  k_gen has laid the stream out in exactly this
// order (internal.h: stream_phys): tile t / chunk c is ONE contiguous block of 32 rows x 20 words, fetched
// with one 1-D bulk copy (cp.async.bulk + mbarrier) into a per-warp ring, S2_RING - 1 blocks in flight per
// warp.  (Measured, memory pipeline alone: 2-D TMA boxes of 32 x 80 B over the row-major stream 0.223 ms,
// 32 x 160 B 0.201 ms, 32 x 400 B 0.195 ms, contiguous blocks 0.181 ms: the TMA unit pays per box row.)
// Each lane turns its row's word pairs into uniform ages -> exact bin index -> its own column of the tile's
// count bytes in shared memory: no conflicts, no idle lanes, every instruction serves 32 samples.  The tile
// [188 slots][32 rows] leaves as 6 KB of coalesced stores; k_replay reads it back the same way.
//
// Bin index (coal.cpp:2265/2284: max(0,(int)round(log(10 a)*10)+1)) in the common case WITHOUT a table:
//   r = fmaf(lg2.approx(float(a)), 10 ln 2, 10 ln 10 + 1.5 + 320)
// is t + 320 with t = 10 ln(10 a) + 1.5, and the reference's bin is floor(t) wherever t is not within the
// error of r of an integer.  For t in [-64, 192) r lies in the binade [256, 512): its float bit pattern IS a
// fixed-point number with 15 fraction bits (bin = (bits >> 15) - KB, fraction = bits & 0x7fff), values
// outside the binade compare below / above as integers and clamp to bin 0 / bin 185.  Error of r against
// the reference's own boundary: lg2.approx 2 ulp at |lg| < 32 (2.6e-5 after the factor 6.93; swept over
// every float by tests/test_gpu_stage1.py::test_lg2_error_bound), one rounding of the FMA to 2^-15
// (1.5e-5), the rounded constants (2.5e-6 + 4.4e-7), float(a) and the reference's two float roundings
// (coal.cpp:2253; 2e-6): < 4.7e-5.  A sample whose fraction is within [-4, +3] units of 2^-15 (1.2e-4 /
// 9.2e-5) of an integer -- 1 in 4096 -- takes the exact threshold table (slot_of_age) instead, as does the
// one generator pair in 2^32 whose uniform needs the "< 1" clamp of generate_canonical.
// (History: MATCH.ANY aggregation 33 cycles per warp instruction on the ADU pipe -> 12 % of HBM peak;
// warp-per-row with shared-memory atomics -> 47 %; lane-per-row with 64-bit chunk indexing and the LUT in
// the main path -> 58 %, 470 instructions per 10 samples; table-free index, 270 instructions -> 70 %, then
// bound by the TMA unit's per-row cost until the stream was re-laid in tile order.)
constexpr float S2_C1 = 6.931471805599453f;        // 10 ln 2
constexpr float S2_C0 = 344.5258509299405f;        // 10 ln 10 + 1.5 + 320
constexpr int S2_KB = (0x43800000 >> 15) + 64;     // (bits(r) >> 15) of t = 0
static_assert(S2_KB % 4 == 0, "count words are addressed from the raw bits");
__device__ __forceinline__ bool s2_unsure(uint32_t rbits) { return ((rbits + 4u) & 0x7ff8u) == 0u; }
__device__ __forceinline__ uint32_t s2_rbits(double a)
{
  float lg;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(__double2float_rn(a)));
  return __float_as_uint(__fmaf_rn(lg, S2_C1, S2_C0));
}
// raw bits (clamped as signed integers into the binade of bins 0 .. 185) -> bin
__device__ __forceinline__ int s2_clamp(uint32_t rbits) { return min(max((int)rbits, S2_KB << 15), ((S2_KB + NBINS) << 15) | 0x7fff); }

// test hooks: the table-free bin index against the exact one (threshold table), on given ages and swept
// over every float in a range of bit patterns
__global__ void k_test_bin_fast(int n, const double* __restrict__ a, const double* __restrict__ thrA, const uint16_t* __restrict__ lut,
                                int32_t* __restrict__ fast, int32_t* __restrict__ exact)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t rb = s2_rbits(a[i]);
  fast[i] = s2_unsure(rb) ? -1 : (s2_clamp(rb) >> 15) - S2_KB;
  exact[i] = slot_of_age(a[i], lut, thrA);
}
__global__ void k_test_bin_sweep(uint32_t lo, uint32_t hi, const double* __restrict__ thrA, const uint16_t* __restrict__ lut,
                                 unsigned long long* __restrict__ out /* flagged, unflagged mismatches, max |t_fast - t| * 1e9 */)
{
  unsigned long long flagged = 0, bad = 0, worst = 0;
  for (uint64_t b = (uint64_t)lo + blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; b < hi; b += (uint64_t)gridDim.x * blockDim.x) {
    const double a = (double)__uint_as_float((uint32_t)b);
    const uint32_t rb = s2_rbits(a);
    const int ex = slot_of_age(a, lut, thrA);
    if (s2_unsure(rb)) flagged++;
    else if ((s2_clamp(rb) >> 15) - S2_KB != ex) bad++;
    const double t = 10.0 * log(10.0 * a) + 1.5 + 320.0;
    if (t >= 256.0 && t < 512.0) {
      const double e = fabs((double)__uint_as_float(rb) - t) * 1e9;
      worst = max(worst, (unsigned long long)e);
    }
  }
  for (int o = 16; o; o >>= 1) {
    flagged += __shfl_xor_sync(0xffffffffu, flagged, o);
    bad += __shfl_xor_sync(0xffffffffu, bad, o);
    worst = max(worst, __shfl_xor_sync(0xffffffffu, worst, o));
  }
  if ((threadIdx.x & 31) == 0) { atomicAdd(&out[0], flagged); atomicAdd(&out[1], bad); atomicMax(&out[2], worst); }
}

__global__ void __launch_bounds__(S2_WARPS * 32)
k_sample(const uint32_t* __restrict__ stream, int64_t n_used, const double4* __restrict__ hdr_g,
         const double* __restrict__ thrA_g, const uint16_t* __restrict__ lut_g, uint8_t* __restrict__ cnt_tiles)
{
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  SampleWarp& sw = ((SampleWarp*)smem_raw)[warp];
  for (int w = 0; w < ROW_WORDS; w++) sw.cnt[w][lane] = 0;
  if (lane == 0) {
    for (int i = 0; i < S2_RING; i++) mbar_init(&sw.full[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();

  // 32-bit bookkeeping throughout (800 B of generator stream per used row keep n_used far below 2^36): tiles, chunk counters, ring phases
  const uint32_t n_tile = (uint32_t)((n_used + TS_ROWS - 1) / TS_ROWS);
  const uint32_t w0 = blockIdx.x * S2_WARPS + warp, nw = gridDim.x * S2_WARPS;
  if (w0 >= n_tile) return;
  const uint32_t my_tiles = (n_tile - w0 + nw - 1) / nw;
  // producer side (lane 0): next block to request = chunk pch of tile ptile, CH_BYTES contiguous bytes of the stream
  constexpr uint32_t CH_BYTES = TS_ROWS * CH_WORDS * 4;
  const uint32_t* pblk = stream + (size_t)w0 * SAMPLE_TILE_WORDS;
  uint32_t pch = 0, pslot = 0, pleft = my_tiles * N_STEP;
  auto issue = [&]() {
    mbar_expect_tx(&sw.full[pslot], CH_BYTES);
    bulk_g2s(&sw.chunk[pslot][0][0], pblk, CH_BYTES, &sw.full[pslot]);
    pslot = pslot + 1 == S2_RING ? 0 : pslot + 1;
    pblk += TS_ROWS * CH_WORDS;
    if (++pch == N_CHUNK) { pch = 0; pblk += (size_t)(nw - 1) * SAMPLE_TILE_WORDS; }
    pleft--;
  };
  if (lane == 0)
    for (int i = 0; i < S2_RING - 1 && pleft; i++) issue();

  // rows past the end of the last tile: length 0 at age 1 (a valid bin), increment 0
  auto header = [&](uint32_t tile, double& lenp, double& abd, uint32_t& one) {
    const int64_t r = (int64_t)tile * TS_ROWS + lane;
    lenp = 0.0; abd = 1.0; one = 0;
    if (r < n_used) { const double2 h = *(const double2*)&hdr_g[r]; lenp = h.x; abd = h.y; one = 1; }
  };
  double lenp_n, abd_n;
  uint32_t one_n;
  header(w0, lenp_n, abd_n, one_n);
  uint32_t cslot = 0, cphase = 0;
  const uint32_t cnt_base = smem_u32(&sw.cnt[0][lane]) - (uint32_t)(S2_KB >> 2) * (TS_ROWS * 4);
  constexpr int NS = SUB_WORDS / 2;                      // samples per loop iteration and lane

  for (uint32_t ti = 0, tile = w0; ti < my_tiles; ti++, tile += nw) {
    const double lenp = lenp_n, abd = abd_n;
    const uint32_t one = one_n;
    if (ti + 1 < my_tiles) header(tile + nw, lenp_n, abd_n, one_n);   // next tile's header: in flight during this tile
#pragma unroll 1
    for (int st = 0; st < N_STEP; st++) {
      __syncwarp();                                              // every lane is done with the slot of the previous step
      if (lane == 0 && pleft) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic reads of that slot before the async write
        issue();
      }
      mbar_wait(&sw.full[cslot], cphase);
      const uint32_t* wslot = &sw.chunk[cslot][lane][0];
      cslot = cslot + 1 == S2_RING ? 0 : cslot + 1;
      cphase ^= cslot == 0;
#pragma unroll 1
      for (int sub = 0; sub < CH_WORDS / SUB_WORDS; sub++) {
      const uint32_t* wbase = wslot + sub * SUB_WORDS;
      auto words = [&](int i) { return *(const uint2*)(wbase + 2 * i); };
      // NS samples as straight-line code (the steps of different samples interleave)
      uint32_t rb[NS];
      bool rare = false;
#ifdef S2_EXP_NOCOMPUTE
      if (lenp != 12345.0) continue;                             // experiment: memory pipeline only
#endif
#pragma unroll
      for (int i = 0; i < NS; i++) {
        const uint2 w = words(i);
        // generate_canonical: (x1 + x2 2^32) / 2^64 with one rounding (I2F.F64.U64, the 2^-64 sits in lenp);
        // sampled_age = U * (age_end - age_begin) + age_begin, product and sum rounded separately
        const double v = __ull2double_rn(((unsigned long long)w.y << 32) | w.x);
        rare |= w.y == 0xffffffffu;                              // v may round to 2^64: needs the clamp below 1
        const double a = __dadd_rn(__dmul_rn(v, lenp), abd);
        rb[i] = s2_rbits(a);
        rare |= s2_unsure(rb[i]);
      }
      if (__any_sync(0xffffffffu, rare)) {
        // exact path for the flagged samples: clamped uniform, threshold table (global memory, L1-resident)
#pragma unroll
        for (int i = 0; i < NS; i++) {
          const uint2 w = words(i);
          if (w.y == 0xffffffffu || s2_unsure(rb[i])) {
            const double ax = __dadd_rn(__dmul_rn(u64_scaled(w.x, w.y), lenp), abd);
            rb[i] = (uint32_t)(slot_of_age(ax, lut_g, thrA_g) + S2_KB) << 15;
          }
        }
      }
#pragma unroll
      for (int i = 0; i < NS; i++) {
        // bin = clamp((bits >> 15) - KB, 0, 185) (as signed integers: r below the binade or negative -> 0,
        // above -> 185 = age out of range, reported by k_replay); count byte bin & 3 of the lane's word bin >> 2
        const int B = s2_clamp(rb[i]);
        const uint32_t addr = cnt_base + ((uint32_t)B >> 17) * (TS_ROWS * 4);
        const uint32_t inc = __funnelshift_l(0u, one, ((uint32_t)B >> 12) & 0x18u);   // 1 << 8 (bin & 3); KB % 4 == 0
        asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(inc) : "memory");   // own word, own bank: never a conflict, never waited for
      }
      }
    }
    {
      // Tile done.  Lane L holds row L as 47 words of 4 slots; the tile leaves as [slot][row] bytes, so
      // every quad of lanes transposes its 4 x 4 bytes (two shuffles + two byte permutes per word) and
      // each lane stores "one slot, four rows": 32-byte runs per slot, full sectors.  Counters back to 0.
      __syncwarp();
      uint32_t* gt = (uint32_t*)(cnt_tiles + (size_t)tile * TILE_BYTES);
      const uint32_t sel1 = (lane & 1) ? 0x3715u : 0x6240u, sel2 = (lane & 2) ? 0x3276u : 0x5410u;
      const int j = lane & 3, rg = lane >> 2;
#pragma unroll 4
      for (int w = 0; w < ROW_WORDS; w++) {
        const uint32_t x = sw.cnt[w][lane];
        sw.cnt[w][lane] = 0;
        const uint32_t t = __byte_perm(x, __shfl_xor_sync(0xffffffffu, x, 1), sel1);
        const uint32_t z = __byte_perm(t, __shfl_xor_sync(0xffffffffu, t, 2), sel2);
        gt[(4 * w + j) * (TS_ROWS / 4) + rg] = z;
      }
      gt[ROW_SLOTS * (TS_ROWS / 4) + lane] = 0;                 // slots 188..191 do not exist
    }
  }
}

constexpr int RP_SITES = 32;    // rows per replay stage
#ifndef RP_STAGES_
#define RP_STAGES_ 4
#endif
constexpr int RP_STAGES = RP_STAGES_;
#ifndef RP_ROWS_
#define RP_ROWS_ 32
#endif
constexpr int RP_ROWS = RP_ROWS_;   // rows collapsed into one exact update
constexpr int RP_CW = RP_ROWS / 4;  // count words of a run (4 rows per word)
static_assert(RP_ROWS == 8 || RP_ROWS == 16 || RP_ROWS == 32, "run width");
#ifndef RP_Q_
#define RP_Q_ 2
#endif
constexpr int RP_Q = RP_Q_;               // lanes per bin: each takes RP_ROWS / RP_Q consecutive rows of a run
constexpr int RP_BPW = 32 / RP_Q;         // bins per warp
constexpr int RP_RPL = RP_ROWS / RP_Q;    // rows per lane and run
constexpr int RP_CWL = RP_RPL / 4;        // count words per lane and run
static_assert(RP_Q == 1 || RP_Q == 2 || RP_Q == 4 || RP_Q == 8, "lanes per bin");
static_assert(RP_RPL >= 4 && RP_RPL % 4 == 0, "a lane takes whole count words");
#ifndef RP_WARPS_
#define RP_WARPS_ 3
#endif
constexpr int RP_WARPS = RP_WARPS_;       // consumer warps per CTA
constexpr int RP_BINS_CTA = RP_WARPS * RP_BPW;
constexpr int RP_GROUPS = 192 / RP_BINS_CTA;   // CTAs that cover a block's 192 >= 185 bins
static_assert(RP_GROUPS * RP_BINS_CTA == 192, "the bin ranges of the CTAs must tile 192 slots");
constexpr int RP_THREADS = (RP_WARPS + 1) * 32;   // + 1 producer warp
struct __align__(16) ReplayStage {
  uint8_t cnt[RP_BINS_CTA][RP_SITES];   // this CTA's slots of one count tile of k_sample: [slot][row]
  double4 hdr[RP_SITES];
};

// one collapsed step of the slow path: acc + c * d(w) when that is what c rounded additions give.  A negative w (a wrapped
// raw-count product) compares as a huge unsigned high word and takes the plain additions of add_repeated.
__device__ __forceinline__ double replay_row(double acc, double w, int c)
{
  const int E = __double2hiint(acc) >> 20;
  const double M = __hiloint2double((E << 20) | 0x80000, 0);
  const double d = __dsub_rn(__dadd_rn(w, M), M);
  const double err = __dsub_rn(w, d);
  const double t = __fma_rn((double)c, d, acc);
  const bool ok = (E > 54) & (E < 0x7fe) & (fabs(err) != __hiloint2double((E - 53) << 20, 0)) &
                  ((uint32_t)__double2hiint(w) < (uint32_t)((E - 1) << 20)) & ((__double2hiint(t) >> 20) == E);
  return ok ? t : exsum::add_repeated(acc, w, c);
}

// bit i of m -> byte i all ones
__device__ __forceinline__ uint32_t rp_byte_mask(uint32_t m) { return (((m & 0xfu) * 0x00204081u) & 0x01010101u) * 0xffu; }

// Exact replay: for every genomic block and both histograms, every age bin walks the block's
// used rows IN ORDER and adds the row's weight once per sample that fell into the bin, with the
// reference's rounding, so age_shared_count / age_notshared_count come out bit for bit as the
// sequential loop of coal.cpp:2259-2295 leaves them.
//
// While the sum stays inside one binade [2^E, 2^(E+1)) every rounded addition of w moves it by
// d(w) = w rounded to a multiple of ulp(acc) -- a function of w and E only -- and all these moves
// are exact, so a run of RP_ROWS rows collapses to acc += sum(count * d(w)): no serial dependency
// per row, and the sum may be taken in any order (every partial sum is a multiple of ulp(acc) below
// 2^(E+1), hence exact; a partial sum at or above 2^(E+1) can only round to something that still
// takes the total out of the binade, which is detected).  So a bin is given to RP_Q lanes, each with
// RP_ROWS / RP_Q rows of the run, whose partial sums meet in a shuffle butterfly: the walk is a
// latency chain per tile (the kernel ran at 16 % active warps with one lane per bin), and the chain
// of a lane is RP_Q times shorter this way while RP_Q times as many warps share the SMs.  Measured on
// B200 (10 M rows, bit-identical throughout): 1 lane per bin 0.64 ms, 4 lanes 0.58 - 0.60 (the fixed cost per
// tile is paid by four times as many warps: issue-bound at 3.45e8 warp instructions), 2 lanes 0.50; and CTAs of
// 3 bin-warps (48 bins, four CTAs per block and histogram) beat 6 / 12 bin-warps (0.54 / 0.61): the warps of a
// CTA share the count-tile ring and move at the pace of the slowest.  A run that
// leaves the binade, meets a rounding tie or a weight too large for the shortcut is redone row by
// row (replay_row / exact_sum.cuh) by all RP_Q lanes of the bin alike, over the rows with a count.  The collapse assumes
// moves that never go down; a negative weight (the raw count weights of the bcf / bam front-ends wrap past 2^31 in the
// reference's int product) counts as too large, and its run is redone row by row.
// blockIdx.y: 2 * group + (0 shared, 1 not shared).  Rows with hdr.y = age_begin <= 0 add nothing to shared.
template <int WHICH>
__device__ __forceinline__ void replay_body(int group, ReplayStage* st, uint64_t* full, uint64_t* empty,
                                            const int64_t* __restrict__ blk_rank_start, const uint8_t* __restrict__ cnt,
                                            const double4* __restrict__ hdr_g, double* __restrict__ out_f,
                                            int64_t* __restrict__ out_n, int64_t* misc)
{
  const int blk = blockIdx.x;
  const int64_t r0 = blk_rank_start[blk], r1 = blk_rank_start[blk + 1];
  const int64_t t0 = r0 / RP_SITES;                               // the block's rows live in count tiles t0 .. t1
  const int n_stage = r1 > r0 ? (int)((r1 - 1) / RP_SITES - t0 + 1) : 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < RP_STAGES; i++) { mbar_init(&full[i], 1); mbar_init(&empty[i], RP_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp == RP_WARPS) {
    if (lane == 0) {
      for (int it = 0; it < n_stage; it++) {
        const int slot = it % RP_STAGES;
        mbar_wait(&empty[slot], ((it / RP_STAGES) & 1) ^ 1);
        const int64_t t = t0 + it;
        constexpr uint32_t CNT_BYTES = RP_BINS_CTA * RP_SITES;        // the CTA's slots: contiguous in the [slot][row] tile
        mbar_expect_tx(&full[slot], (uint32_t)(CNT_BYTES + RP_SITES * 32));
        bulk_g2s(&st[slot].cnt[0][0], cnt + (size_t)t * TILE_BYTES + (size_t)group * CNT_BYTES, CNT_BYTES, &full[slot]);
        bulk_g2s(&st[slot].hdr[0], hdr_g + t * RP_SITES, RP_SITES * 32, &full[slot]);
      }
    }
    return;
  }
  const int q = lane & (RP_Q - 1);                                // which part of a run's rows
  const int cslot = warp * RP_BPW + lane / RP_Q;                  // slot inside the CTA's part of the tile (slot == bin; bytes 188..191 stay 0)
  const int bin = group * RP_BINS_CTA + cslot;                    // 0..191
  const unsigned gsh = lane & ~(RP_Q - 1);                        // first lane of this bin
  constexpr unsigned GMASK = RP_Q == 32 ? 0xffffffffu : (1u << RP_Q) - 1u;
  double acc = 0.0;
  uint32_t tally = 0;
  bool overflow = false;
#ifdef REPLAY_PROF
  long long pf_t0 = clock64(), pf_wait = 0, pf_slow = 0;
  int pf_runs = 0, pf_skipped = 0, pf_slowruns = 0, pf_lanes = 0, pf_tie = 0, pf_big = 0, pf_e54 = 0, pf_exp = 0, pf_rows = 0, pf_csum = 0, pf_cmax = 0;
#endif
  for (int it = 0; it < n_stage; it++) {
    const int slot = it % RP_STAGES;
#ifdef REPLAY_PROF
    long long pf_a = clock64();
#endif
    mbar_wait(&full[slot], (it / RP_STAGES) & 1);
#ifdef REPLAY_PROF
    pf_wait += clock64() - pf_a;
#endif
    // rows of this tile that belong to the block ...
    const int64_t g0r = (t0 + it) * RP_SITES;
    const int lo = (int)max((int64_t)0, r0 - g0r), hi = (int)min((int64_t)RP_SITES, r1 - g0r);
    uint32_t live = (hi >= 32 ? 0xffffffffu : (1u << hi) - 1u) & ~((1u << lo) - 1u);
    const uint32_t* cwp = (const uint32_t*)&st[slot].cnt[cslot][0];   // this bin's counts in the tile's 32 rows, 4 rows per word
    const double* hp = (const double*)&st[slot].hdr[0] + 2 + WHICH;
    // ... and add to this histogram (shared: rows with age_begin > 0), one bit per row
    if (WHICH == 0) live &= __ballot_sync(0xffffffffu, st[slot].hdr[lane].y > 0.0);
#pragma unroll
    for (int run = 0; run < RP_SITES / RP_ROWS; run++) {
      const int g0 = run * RP_ROWS;
      const int gl = g0 + q * RP_RPL;                                  // this lane's rows of the run: gl .. gl + RP_RPL
      // this bin's counts in those rows, one byte each (<= 100)
      uint32_t cs[RP_CWL];
      uint32_t cs_or = 0, cs_sum = 0;
#pragma unroll
      for (int k = 0; k < RP_CWL; k++) {
        cs[k] = cwp[(gl >> 2) + k] & rp_byte_mask(live >> (gl + 4 * k));
        cs_or |= cs[k];
        cs_sum = __dp4a(cs[k], 0x01010101u, cs_sum);
      }
      if (WHICH == 1) overflow |= (bin == NBINS) & (cs_or != 0);   // a sample in bin 185: out of bounds in the reference
      tally += cs_sum;
      const unsigned anyb = __ballot_sync(0xffffffffu, cs_or != 0);
#ifdef REPLAY_PROF
      pf_runs++;
      if (anyb == 0) { pf_skipped++; continue; }
#else
      if (anyb == 0) continue;
#endif
      const bool any = ((anyb >> gsh) & GMASK) != 0;                   // some row of the run counts for this bin
      const int E = __double2hiint(acc) >> 20;                         // biased exponent (acc < 0: E < 0, row by row)
      const double M = __hiloint2double((E << 20) | 0x80000, 0);       // 1.5 * 2^E: ulp(M) == ulp(acc)
      const int hu_hi = (E - 53) << 20;                                // high word of ulp(acc) / 2 (the low word is 0)
      const uint32_t wmax_hi = (uint32_t)((E - 1) << 20);              // w must stay below 2^(E-1) and not be negative
      bool badl = (E <= 54) | (E >= 0x7fe);
      constexpr int NTS = RP_RPL >= 8 ? 4 : 2;
      double ts[4] = {0.0, 0.0, 0.0, 0.0};                             // exact sums: any order
#ifdef REPLAY_PROF
      bool pf_c_tie = false, pf_c_big = false;
#endif
#pragma unroll
      for (int i = 0; i < RP_RPL; i++) {
        const int c = (cs[i >> 2] >> (8 * (i & 3))) & 0xff;
        const double w = hp[4 * (gl + i)];                             // (rows of other blocks carry count 0 here; the padding rows are zeroed)
        const double d = __dsub_rn(__dadd_rn(w, M), M);
        const double err = __dsub_rn(w, d);
        // |err| <= ulp / 2, and ulp / 2 itself is the only such value with its exponent field: a tie shows in the exponent alone
        badl |= (c != 0) & ((((__double2hiint(err) ^ hu_hi) & 0x7ff00000) == 0) | ((uint32_t)__double2hiint(w) >= wmax_hi));
        // (double)c without the quarter-rate I2F.F64: 2^52 + c is a register pair, one DADD takes the 2^52 off
        ts[i & (NTS - 1)] = __fma_rn(__dsub_rn(__hiloint2double(0x43300000, c), 0x1p52), d, ts[i & (NTS - 1)]);
#ifdef REPLAY_PROF
        pf_c_tie |= (c != 0) & (((__double2hiint(err) ^ hu_hi) & 0x7ff00000) == 0);
        pf_c_big |= (c != 0) & ((uint32_t)__double2hiint(w) >= wmax_hi);
#endif
      }
      double t = NTS == 4 ? __dadd_rn(__dadd_rn(ts[0], ts[1]), __dadd_rn(ts[2], ts[3])) : __dadd_rn(ts[0], ts[1]);
#pragma unroll
      for (int o = 1; o < RP_Q; o <<= 1) t = __dadd_rn(t, __shfl_xor_sync(0xffffffffu, t, o));   // the same bits in every lane of the bin
      const double accn = __dadd_rn(acc, t);
      badl |= (__double2hiint(accn) >> 20) != E;
      const unsigned badb = __ballot_sync(0xffffffffu, badl);
      const bool bad = any & (((badb >> gsh) & GMASK) != 0);
      if (__any_sync(0xffffffffu, bad)) {
#ifdef REPLAY_PROF
        pf_slowruns++;
        pf_lanes += __popc(__ballot_sync(0xffffffffu, bad));
        pf_tie += __popc(__ballot_sync(0xffffffffu, bad && pf_c_tie));
        pf_big += __popc(__ballot_sync(0xffffffffu, bad && pf_c_big));
        pf_e54 += __popc(__ballot_sync(0xffffffffu, bad && ((E <= 54) | (E >= 0x7fe))));
        pf_exp += __popc(__ballot_sync(0xffffffffu, bad && (__double2hiint(accn) >> 20) != E));
        {
          int rows = 0, csum = 0, cmax = 0;
          for (int r = g0; r < g0 + RP_ROWS; r++) {
            const int c = ((live >> r) & 1u) ? st[slot].cnt[cslot][r] : 0;
            if (bad && c) { rows++; csum += c; cmax = max(cmax, c); }
          }
          pf_rows += __reduce_add_sync(0xffffffffu, rows);
          pf_csum += __reduce_add_sync(0xffffffffu, csum);
          pf_cmax = max(pf_cmax, __reduce_max_sync(0xffffffffu, cmax));
        }
        long long pf_b = clock64();
#endif
#ifdef RP_EXP_NOSLOW
        if (false) {   // experiment: what the kernel costs without its serial path (wrong sums)
#else
        if (bad) {
#endif
          // Row by row, but only the rows of the run in which THIS bin has a count (zero in ~85 % of the rows; the counts of dead
          // rows are masked).  (A variant that located the crossing row from prefix sums of collapsed steps and committed the
          // rows on either side at once was measured SLOWER, 1.36 ms against 0.76: its passes touch every row.)
          uint32_t nzr = 0;
#pragma unroll
          for (int k = 0; k < RP_CW; k++) {
            const uint32_t cwk = cwp[(g0 >> 2) + k] & rp_byte_mask(live >> (g0 + 4 * k));
            const uint32_t nz = (cwk | ((cwk & 0x7f7f7f7fu) + 0x7f7f7f7fu)) & 0x80808080u;   // high bit of every non-zero byte
            nzr |= ((nz * 0x00204081u) >> 28) << (4 * k);                                    // -> one bit per row
          }
#pragma unroll 1
          while (nzr) {
            const int r = g0 + __ffs(nzr) - 1;
            nzr &= nzr - 1;
            const double w = hp[4 * r];
            const int c = st[slot].cnt[cslot][r];
            if ((__double_as_longlong(w) << 1) != 0) {   // x + (+-0.0) == x (acc is never -0.0)
              // a handful of samples (the usual case: 100 samples of a row spread over its bins): the reference's own additions
              if (c <= 4) { for (int j = 0; j < c; j++) acc = __dadd_rn(acc, w); }
              else acc = replay_row(acc, w, c);
            }
          }
        } else if (any) acc = accn;
#ifdef REPLAY_PROF
        __syncwarp();
        pf_slow += clock64() - pf_b;
#endif
      } else if (any) acc = accn;
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[slot]);
  }
#ifdef REPLAY_PROF
  if (lane == 0 && (blk == 3 || blk == 50))
    printf("[replay prof] blk %d which %d warp %d stages %d: cycles %lld wait %lld slow %lld | runs %d skipped %d slow %d | bad lanes %d: tie %d big %d e54 %d exp %d | rows walked %d counts %d max %d\n",
           blk, WHICH, warp, n_stage, clock64() - pf_t0, pf_wait, pf_slow, pf_runs, pf_skipped, pf_slowruns, pf_lanes, pf_tie, pf_big, pf_e54, pf_exp,
           pf_rows, pf_csum, pf_cmax);
#endif
  if (overflow) misc[3] = 1;
#pragma unroll
  for (int o = 1; o < RP_Q; o <<= 1) tally += __shfl_xor_sync(0xffffffffu, tally, o);
  if (bin < NBINS && q == 0) {
    out_f[((size_t)blk * 4 + WHICH) * NBINS + bin] = acc;
    out_n[((size_t)blk * 3 + WHICH) * NBINS + bin] = tally;
  }
}

#ifndef RP_MINB_
#define RP_MINB_ (RP_WARPS_ <= 3 ? 6 : RP_WARPS_ <= 6 ? 3 : RP_WARPS_ <= 12 ? 2 : 1)   // small CTAs (a CTA moves at the pace of its slowest bin-warp); 6 x 148 slots hold a 107-block genome's 856 CTAs in one wave
#endif
__global__ void __launch_bounds__(RP_THREADS, RP_MINB_)
k_replay(const int64_t* __restrict__ blk_rank_start, const uint8_t* __restrict__ cnt, const double4* __restrict__ hdr_g,
         double* __restrict__ out_f, int64_t* __restrict__ out_n, int64_t* misc)
{
  __shared__ ReplayStage st[RP_STAGES];
  __shared__ __align__(8) uint64_t full[RP_STAGES], empty[RP_STAGES];
  if (blockIdx.y & 1) replay_body<1>(blockIdx.y >> 1, st, full, empty, blk_rank_start, cnt, hdr_g, out_f, out_n, misc);
  else replay_body<0>(blockIdx.y >> 1, st, full, empty, blk_rank_start, cnt, hdr_g, out_f, out_n, misc);
}

// age_shared_emp / age_notshared_emp row 0 (coal.cpp:2250-2256): one addition per row with age_begin <= 0 into the bin of its
// age_end, in row order.  ONE warp per block: lane = row of a group of 32 consecutive used rows; MATCH.ANY groups the rows by
// bin, the lowest lane of every group adds its members' weights in lane (= row) order to the bin's running sums in shared
// memory -- different bins in parallel, one bin in order.  Needs only k_compact's output: launched on the side stream right
// behind the compaction, under the sampler.  (The first version gave every bin a thread that scanned ALL rows of the block:
// 192 x the work, 0.67 ms when run alone.)
__global__ void __launch_bounds__(32)
k_emp(const int64_t* __restrict__ blk_rank_start, const uint8_t* __restrict__ e_b2, const double* __restrict__ e_ws,
      const double* __restrict__ e_wn, double* __restrict__ out_f, int64_t* __restrict__ out_n)
{
  __shared__ double as[192], an[192];
  __shared__ int cn[192];
  const int lane = threadIdx.x;
  for (int i = lane; i < 192; i += 32) { as[i] = 0.0; an[i] = 0.0; cn[i] = 0; }
  __syncwarp();
  const int blk = blockIdx.x;
  const int64_t r0 = blk_rank_start[blk], r1 = blk_rank_start[blk + 1];
  // (the loads of the next group are issued before this group is worked on: the walk is a chain of dependent additions,
  // the memory latency must not be part of it)
  auto fetch = [&](int64_t base, int& b, double& ws, double& wn) {
    const int64_t r = base + lane;
    b = r < r1 ? (int)e_b2[r] : 255;                            // 255: the row adds nothing here
    ws = b != 255 ? e_ws[r] : 0.0;
    wn = b != 255 ? e_wn[r] : 0.0;
  };
  int b_n; double ws_n, wn_n;
  fetch(r0, b_n, ws_n, wn_n);
  for (int64_t base = r0; base < r1; base += 32) {
    const int b = b_n;
    const double ws = ws_n, wn = wn_n;
    fetch(base + 32, b_n, ws_n, wn_n);
    const unsigned grp = __match_any_sync(0xffffffffu, b);       // the rows of this group with my bin
    const bool leader = b != 255 && lane == __ffs(grp) - 1;
    unsigned m = leader ? grp : 0u;
    double a_s = 0.0, a_n = 0.0;
    if (leader) { a_s = as[b]; a_n = an[b]; }
    while (__any_sync(0xffffffffu, m != 0)) {
      const int src = m ? __ffs(m) - 1 : 0;
      const double vs = __shfl_sync(0xffffffffu, ws, src), vn = __shfl_sync(0xffffffffu, wn, src);
      if (m) { a_s = __dadd_rn(a_s, vs); a_n = __dadd_rn(a_n, vn); m &= m - 1; }
    }
    if (leader) { as[b] = a_s; an[b] = a_n; cn[b] += __popc(grp); }
    __syncwarp();
  }
  for (int bin = lane; bin < NBINS; bin += 32) {
    out_f[((size_t)blk * 4 + 2) * NBINS + bin] = as[bin];
    out_f[((size_t)blk * 4 + 3) * NBINS + bin] = an[bin];
    out_n[((size_t)blk * 3 + 2) * NBINS + bin] = cn[bin];
  }
}

// ------------------------------------------------------------------------------------------
static inline int grid_for(int64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// The two launches of the exact histograms, shared by stage i (run_compact / run_replay) and the test hook
// colate_test_replay: n_blocks genomic blocks, rows [blk_rank_start[b], blk_rank_start[b + 1]) of block b.
// k_replay: count tiles [tile][slot][row % 32] and double4 headers of whole tiles -> out_f[b][0..1], out_n[b][0..1], misc[3]
static void launch_replay(cudaStream_t s, int n_blocks, const int64_t* blk_rank_start, const uint8_t* cnt_tiles, const double4* hdr,
                          double* out_f, int64_t* out_n, int64_t* misc)
{
  k_replay<<<dim3(n_blocks, 2 * RP_GROUPS), RP_THREADS, 0, s>>>(blk_rank_start, cnt_tiles, hdr, out_f, out_n, misc);
}
// k_emp: the rows' single emp contributions (bin 255: none) -> out_f[b][2..3], out_n[b][2]
static void launch_emp(cudaStream_t s, int n_blocks, const int64_t* blk_rank_start, const uint8_t* e_b2, const double* e_ws,
                       const double* e_wn, double* out_f, int64_t* out_n)
{
  k_emp<<<n_blocks, 32, 0, s>>>(blk_rank_start, e_b2, e_ws, e_wn, out_f, out_n);
}

int run_join(colate_handle* h, int slot)
{
  GenomeDev& g = h->genomes[slot];
  if (g.joined) return 0;
  const int64_t n = h->n_site;
  CK(g.j_aaf.ensure(n * 4 + 4)); CK(g.j_daf.ensure(n * 4 + 4)); CK(g.j_prevbp.ensure(n * 4 + 4)); CK(g.j_flag.ensure(n + 4));
  if (g.pileup) {                            // the decoder's per-row counts: no record stream to search
    if (n > 0) {
      k_pileup_join<<<grid_for(n, 256), 256, 0, h->stream>>>(n, h->meta.as<uint32_t>(), g.pile.as<int4>(), g.j_aaf.as<int32_t>(), g.j_daf.as<int32_t>(),
                                                             g.j_prevbp.as<int32_t>(), g.j_flag.as<uint8_t>());
      CK(cudaGetLastError());
      h->launches += 1;
    }
    g.joined = true;
    return 0;
  }
  if (n > 0) {
    // tiles of JOIN_TILE sites, never across a chromosome boundary
    if ((int)h->h_tile_start.size() != h->n_chr + 1 || !h->tiles_valid) {
      h->h_tile_start.assign(h->n_chr + 1, 0);
      for (int c = 0; c < h->n_chr; c++)
        h->h_tile_start[c + 1] = h->h_tile_start[c] + (int32_t)((h->h_site_off[c + 1] - h->h_site_off[c] + JOIN_TILE - 1) / JOIN_TILE);
      CK(h->tile_start.ensure((h->n_chr + 1) * 4));
      CK(cudaMemcpyAsync(h->tile_start.p, h->h_tile_start.data(), (h->n_chr + 1) * 4, cudaMemcpyHostToDevice, h->stream));
      h->tiles_valid = true;
    }
    const int n_tiles = h->h_tile_start[h->n_chr];
    CK(h->tile_rlo.ensure((size_t)(n_tiles + 1) * sizeof(JoinTileInfo)));
    k_join_bounds<<<grid_for(n_tiles, 256), 256, 0, h->stream>>>(n_tiles, h->n_chr, h->tile_start.as<int32_t>(), h->site_off.as<int64_t>(),
                                                                h->pos.as<int32_t>(), g.chr_first.as<int64_t>(), g.chr_end.as<int64_t>(),
                                                                g.bp.as<int32_t>(), h->tile_rlo.as<JoinTileInfo>());
    k_join<<<n_tiles, JOIN_TILE, 0, h->stream>>>(h->tile_rlo.as<JoinTileInfo>(), h->pos.as<int32_t>(), h->meta.as<uint32_t>(),
                                                 g.bp.as<int32_t>(), g.aaf.as<int32_t>(), g.daf.as<int32_t>(), g.alleles.as<uint16_t>(),
                                                 g.j_aaf.as<int32_t>(), g.j_daf.as<int32_t>(), g.j_prevbp.as<int32_t>(), g.j_flag.as<uint8_t>());
    CK(cudaGetLastError());
    h->launches += 2;
  }
  g.joined = true;
  return 0;
}

int run_check_sites(colate_handle* h)
{
  if (h->n_site > 0) {
    k_check_sites<<<grid_for(h->n_site, 256), 256, 0, h->stream>>>(h->n_site, h->n_chr, h->site_off.as<int64_t>(), h->pos.as<int32_t>(),
                                                                   h->ab.as<float>(), h->ae.as<float>(), h->meta.as<uint32_t>(), h->thr185,
                                                                   h->order_flag.as<int>());
    h->launches += 1;
    CK(cudaGetLastError());
  }
  return 0;
}

int run_check_genome(colate_handle* h, int slot)
{
  GenomeDev& g = h->genomes[slot];
  if (g.n_rec > 1 && h->n_chr > 0) {
    k_check_genome<<<grid_for(g.n_rec, 256), 256, 0, h->stream>>>(g.n_rec, h->n_chr, g.chr_first.as<int64_t>(), g.chr_end.as<int64_t>(),
                                                                  g.bp.as<int32_t>(), h->order_flag.as<int>() + 1 + slot);
    h->launches += 1;
    CK(cudaGetLastError());
  }
  return 0;
}

int run_flags(colate_handle* h, int tslot, int rslot)
{
  const int64_t n = h->n_site;
  const int64_t nw = (n + 31) / 32;
  GenomeDev& T = h->genomes[tslot];
  GenomeDev& R = h->genomes[rslot];
  CK(h->candR.ensure(nw * 4 + 8)); CK(h->candT.ensure(nw * 4 + 8)); CK(h->use.ensure(nw * 4 + 8));
  CK(h->word_rank.ensure((nw + 1) * 4 + 8));
  CK(h->row_of_rank.ensure((size_t)n * 4 + 8));
  const int nsb = std::max(1, grid_for(nw, SCAN_THREADS * SCAN_ITEMS));
  CK(h->scan_tmp.ensure((size_t)nsb * 4 + 16));
  CK(h->chr_used.ensure(h->n_chr * 8 + 8)); CK(h->chr_blocks.ensure(h->n_chr * 4 + 8)); CK(h->chr_block_base.ensure(h->n_chr * 4 + 8));
  CK(h->misc.ensure(64));
  CK(cudaMemsetAsync(h->misc.p, 0, 64, h->stream));
  cudaStream_t s = h->stream;
  uint32_t* total = (uint32_t*)((char*)h->misc.p + 56);
  if (n > 0) {
    int grid = grid_for(n, 256);
    k_ok<true><<<grid, 256, 0, s>>>(n, h->n_chr, h->site_off.as<int64_t>(), h->pos.as<int32_t>(), nullptr,
                                    T.has_mask ? T.mask_bits.as<uint32_t>() : nullptr, R.has_mask ? R.mask_bits.as<uint32_t>() : nullptr,
                                    R.j_aaf.as<int32_t>(), R.j_daf.as<int32_t>(), R.j_prevbp.as<int32_t>(), R.j_flag.as<uint8_t>(),
                                    h->candT.as<uint32_t>(), h->meta.as<uint32_t>(), h->misc.as<int64_t>());
    k_ok<false><<<grid, 256, 0, s>>>(n, h->n_chr, h->site_off.as<int64_t>(), h->pos.as<int32_t>(), h->candT.as<uint32_t>(), nullptr, nullptr,
                                     T.j_aaf.as<int32_t>(), T.j_daf.as<int32_t>(), T.j_prevbp.as<int32_t>(), T.j_flag.as<uint8_t>(),
                                     h->use.as<uint32_t>(), h->meta.as<uint32_t>(), h->misc.as<int64_t>());
    k_popc_blocksum<<<nsb, SCAN_THREADS, 0, s>>>(h->use.as<uint32_t>(), nw, h->scan_tmp.as<uint32_t>());
    k_scan_sums<<<1, 32, 0, s>>>(h->scan_tmp.as<uint32_t>(), nsb, total);
    k_word_rank<<<nsb, SCAN_THREADS, 0, s>>>(h->use.as<uint32_t>(), nw, h->scan_tmp.as<uint32_t>(), total, h->word_rank.as<uint32_t>(),
                                             h->row_of_rank.as<int32_t>());
    h->launches += 5;
  } else {
    CK(cudaMemsetAsync(h->word_rank.p, 0, 8, s));
  }
  k_chr<<<1, 1024, 0, s>>>(h->n_chr, h->site_off.as<int64_t>(), h->pos.as<int32_t>(), h->use.as<uint32_t>(), h->word_rank.as<uint32_t>(),
                         h->chr_used.as<int64_t>(), h->chr_blocks.as<int32_t>(), h->chr_block_base.as<int32_t>(), h->misc.as<int64_t>());
  h->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

// used rows -> dense records in rank order, block ranges; needs h->n_used / n_blocks_local
int run_compact(colate_handle* h)
{
  const int64_t n = h->n_site, nu = h->n_used;
  GenomeDev& T = h->genomes[h->tgt_slot];
  GenomeDev& R = h->genomes[h->ref_slot];
  cudaStream_t s = h->stream;
  const size_t un = (size_t)std::max<int64_t>(nu, 1);
  const size_t un32 = (un + TS_ROWS - 1) / TS_ROWS * TS_ROWS;   // headers and counts are read / written in tiles of 32 rows
  CK(h->u_hdr.ensure(un32 * 32 + 64)); CK(h->u_eb2.ensure(un + 64)); CK(h->u_ews.ensure(un * 8 + 64)); CK(h->u_ewn.ensure(un * 8 + 64));
  CK(h->u_blk.ensure(un * 4 + 64)); CK(h->u_cnt.ensure(un32 * ROW_BYTES + 64));
  CK(h->blk_rank_start.ensure((MAX_BLOCKS + 2) * 8));
  CK(h->out_f.ensure((size_t)MAX_BLOCKS * 4 * NBINS * 8)); CK(h->out_n.ensure((size_t)MAX_BLOCKS * 3 * NBINS * 8));
  CK(h->deep_rows.ensure((size_t)std::max<int64_t>(h->n_deep, 1) * 8));
  if (un32 > (size_t)nu)   // header rows between the last used row and the end of its tile: read by k_replay, never written
    CK(cudaMemsetAsync(h->u_hdr.as<double4>() + nu, 0, (un32 - (size_t)nu) * 32, s));
  CK(cudaEventRecord(h->ev[2], s));
  if (n > 0) {
    k_compact<<<grid_for(std::max<int64_t>(nu, 1), 256), 256, 0, s>>>(n, h->n_chr, h->site_off.as<int64_t>(), h->pos.as<int32_t>(), h->ab.as<float>(),
                                               h->ae.as<float>(), h->row_of_rank.as<int32_t>(),
                                               h->chr_block_base.as<int32_t>(), T.j_aaf.as<int32_t>(), T.j_daf.as<int32_t>(),
                                               R.j_aaf.as<int32_t>(), R.j_daf.as<int32_t>(), h->thr10.as<double>(),
                                               h->u_hdr.as<double4>(), h->u_eb2.as<uint8_t>(), h->u_ews.as<double>(),
                                               h->u_ewn.as<double>(), h->u_blk.as<int32_t>(), h->misc.as<int64_t>(),
                                               h->meta.as<uint32_t>(), h->deep_rows.as<int64_t>(), h->n_deep, h->opt_raw_weights ? 1 : 0);
    h->launches += 1;
  }
  k_block_ranges<<<1, 512, 0, s>>>(h->u_blk.as<int32_t>(), h->misc.as<int64_t>(), h->blk_rank_start.as<int64_t>());
  h->launches += 1;
  CK(cudaEventRecord(h->ev[3], s));
  if (h->n_blocks_local > 0) {
    // the emp histograms need nothing but the compacted rows: on the side stream, under the sampler; run_replay joins it
    CK(cudaStreamWaitEvent(h->side_stream, h->ev[3], 0));
    launch_emp(h->side_stream, h->n_blocks_local, h->blk_rank_start.as<int64_t>(), h->u_eb2.as<uint8_t>(), h->u_ews.as<double>(),
               h->u_ewn.as<double>(), h->out_f.as<double>(), h->out_n.as<int64_t>());
    h->launches += 1;
    CK(cudaEventRecord(h->side_done, h->side_stream));
  }
  CK(cudaGetLastError());
  return 0;
}

// k_sample over used rows [row0, row0 + n_rows) whose generator words start at `stream_local` (tile order relative to
// row0).  row0 == 0 and n_rows == n_used: straight into the count tiles; otherwise (rejection-sampling path) into scratch
// tiles and from there to the rows' places.
int run_sample_rows(colate_handle* h, const uint32_t* stream_local, int64_t row0, int64_t n_rows)
{
  cudaStream_t s = h->stream;
  if (n_rows <= 0) return 0;
  const bool whole = row0 == 0 && n_rows == h->n_used;
  uint8_t* tiles = h->u_cnt.as<uint8_t>();
  if (!whole) {
    CK(h->d_tmp.ensure((size_t)((n_rows + TS_ROWS - 1) / TS_ROWS) * TILE_BYTES + 64));
    tiles = h->d_tmp.as<uint8_t>();
  }
  const size_t smem = sizeof(SampleWarp) * S2_WARPS;
  // all of the SM's 228 KB as shared memory (the kernel's only L1 traffic is one 16 B header per row): the
  // resident warps, and with them the bytes in flight, are bounded by the rings and count tiles
  CK(cudaFuncSetAttribute(k_sample, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CK(cudaFuncSetAttribute(k_sample, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  const int64_t n_tile = (n_rows + TS_ROWS - 1) / TS_ROWS;
  int per_sm = 1;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sample, S2_WARPS * 32, smem));
  per_sm = std::max(1, per_sm);
  if (const char* e = getenv("COLATE_SAMPLE_CTAS_PER_SM")) per_sm = std::max(1, atoi(e));
  const int grid = (int)std::min<int64_t>((n_tile + S2_WARPS - 1) / S2_WARPS, (int64_t)h->sm_count * per_sm);
  k_sample<<<grid, S2_WARPS * 32, smem, s>>>(stream_local, n_rows, h->u_hdr.as<double4>() + row0, h->thrA.as<double>(), h->lut.as<uint16_t>(), tiles);
  h->launches += 1;
  if (!whole) {
    k_scatter_count_rows<<<grid_for(n_rows * ROW_BYTES, 256), 256, 0, s>>>(tiles, n_rows, row0, h->u_cnt.as<uint8_t>());
    h->launches += 1;
  }
  CK(cudaGetLastError());
  return 0;
}

// one count row computed on the host (a rejection-sampled row) -> its place in the count tiles
int run_put_count_row(colate_handle* h, int64_t row, const uint8_t* cnt192_host)
{
  cudaStream_t s = h->stream;
  CK(h->d_scratch.ensure(256));
  CK(cudaMemcpyAsync(h->d_scratch.p, cnt192_host, ROW_BYTES, cudaMemcpyHostToDevice, s));
  k_put_count_row<<<1, ROW_BYTES, 0, s>>>(h->d_scratch.as<uint8_t>(), row, h->u_cnt.as<uint8_t>());
  h->launches += 1;
  CK(cudaStreamSynchronize(s));   // the host row buffer is the caller's local; d_scratch is reused by the next row
  CK(cudaGetLastError());
  return 0;
}

// exact per-block replay of the count rows
int run_replay(colate_handle* h)
{
  cudaStream_t s = h->stream;
  const int nb = h->n_blocks_local;
  CK(cudaEventRecord(h->ev[4], s));
  if (nb > 0) {
    launch_replay(s, nb, h->blk_rank_start.as<int64_t>(), h->u_cnt.as<uint8_t>(), h->u_hdr.as<double4>(), h->out_f.as<double>(),
                  h->out_n.as<int64_t>(), h->misc.as<int64_t>());
    h->launches += 1;
    CK(cudaStreamWaitEvent(s, h->side_done, 0));   // k_emp's slices of out_f / out_n (run_compact launched it on the side stream)
  }
  CK(cudaEventRecord(h->ev[5], s));
  CK(cudaGetLastError());
  return 0;
}

int run_pack_row_counts(colate_handle* h, int slot, const int32_t* aaf_dev, const int32_t* daf_dev)
{
  GenomeDev& g = h->genomes[slot];
  if (h->n_site > 0) {
    k_pack_row_counts<<<grid_for(h->n_site, 256), 256, 0, h->stream>>>(h->n_site, aaf_dev, daf_dev, g.pile.as<int4>());
    h->launches += 1;
    CK(cudaGetLastError());
  }
  return 0;
}

// pileup of one contig's decoded reads at the rows of chromosome chr (device pointers throughout).  starts_contig: reads[0] is the
// contig's first record (the assign_contig quirk applies to it); only rows [row_lo, row_hi) of the contig are searched (rows the
// reads cannot cover are left as they are; row_hi < 0: all rows).
int run_pileup_reads(colate_handle* h, int slot, int chr, int64_t n_reads, const int32_t* pos, const uint8_t* mapq, const int32_t* len,
                     const int64_t* off, const uint8_t* seq, const uint8_t* qual, const uint8_t* ref, int64_t ref_len, int max_len,
                     int mapq_th, int len_th, int mismatch_th, uint8_t* pass_scratch, bool starts_contig, int64_t row_lo, int64_t row_hi)
{
  GenomeDev& g = h->genomes[slot];
  const int64_t n_chr_rows = h->h_site_off[chr + 1] - h->h_site_off[chr];
  if (row_hi < 0) { row_lo = 0; row_hi = n_chr_rows; }
  const int64_t row0 = h->h_site_off[chr] + row_lo, n_rows = row_hi - row_lo;
  if (n_reads <= 0 || n_rows <= 0) return 0;
  const int64_t k_quirk = starts_contig ? 0 : -1;
  cudaStream_t s = h->stream;
  k_read_filter<<<grid_for(n_reads, 256), 256, 0, s>>>(n_reads, pos, mapq, len, off, seq, qual, ref, ref_len, mapq_th, len_th, mismatch_th, k_quirk,
                                                       pass_scratch);
  k_pileup_rows<<<grid_for(n_rows, 128), 128, 0, s>>>(row0, n_rows, h->pos.as<int32_t>(), n_reads, pos, len, off, seq, qual, pass_scratch, max_len,
                                                     k_quirk, g.pile.as<int4>());
  h->launches += 2;
  CK(cudaGetLastError());
  return 0;
}

int run_test_bin_fast(colate_handle* h, int n, const double* a_host, int32_t* fast_host, int32_t* exact_host)
{
  cudaStream_t s = h->stream;
  CK(h->d_scratch.ensure((size_t)n * 16));
  double* a = h->d_scratch.as<double>();
  int32_t* f = (int32_t*)(a + n);
  CK(cudaMemcpyAsync(a, a_host, (size_t)n * 8, cudaMemcpyHostToDevice, s));
  k_test_bin_fast<<<(n + 255) / 256, 256, 0, s>>>(n, a, h->thrA.as<double>(), h->lut.as<uint16_t>(), f, f + n);
  CK(cudaMemcpyAsync(fast_host, f, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(exact_host, f + n, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  return 0;
}
int run_test_bin_sweep(colate_handle* h, uint32_t lo_bits, uint32_t hi_bits, uint64_t* out3_host)
{
  cudaStream_t s = h->stream;
  CK(h->d_scratch.ensure(64));
  CK(cudaMemsetAsync(h->d_scratch.p, 0, 24, s));
  k_test_bin_sweep<<<h->sm_count * 8, 256, 0, s>>>(lo_bits, hi_bits, h->thrA.as<double>(), h->lut.as<uint16_t>(),
                                                   h->d_scratch.as<unsigned long long>());
  CK(cudaMemcpyAsync(out3_host, h->d_scratch.p, 24, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  return 0;
}

// test hooks of the exact replay: k_replay and k_emp on given rows through the launches stage i uses, and the device's
// replay_row / exsum::add_repeated element by element
__global__ void k_test_replay_row(int which, int n, const double* __restrict__ acc, const double* __restrict__ w, const int32_t* __restrict__ c,
                                  double* __restrict__ out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = which == 0 ? replay_row(acc[i], w[i], c[i]) : exsum::add_repeated(acc[i], w[i], c[i]);
}

int run_test_replay_row(colate_handle* h, int which, int n, const double* acc, const double* w, const int32_t* c, double* out)
{
  cudaStream_t s = h->stream;
  CK(h->d_scratch.ensure((size_t)n * 28 + 64));
  double* d_acc = h->d_scratch.as<double>();
  double* d_w = d_acc + n;
  double* d_out = d_w + n;
  int32_t* d_c = (int32_t*)(d_out + n);
  CK(cudaMemcpyAsync(d_acc, acc, (size_t)n * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_w, w, (size_t)n * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_c, c, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  k_test_replay_row<<<grid_for(n, 256), 256, 0, s>>>(which, n, d_acc, d_w, d_c, d_out);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, d_out, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return 0;
}

// The rows are laid out as k_compact and k_sample leave them: count tiles [tile][slot][row % 32], double4 headers
// {0, age_begin, w_shared, w_notshared}, the rows of the last tile past n_rows zeroed.
int run_test_replay(colate_handle* h, int n_blocks, const int64_t* blk_rank_start, int64_t n_rows, const uint8_t* counts,
                    const double* age_begin, const double* w_shared, const double* w_notshared, const uint8_t* emp_bin,
                    const double* emp_ws, const double* emp_wn, double* out_f, int64_t* out_n, int* out_of_range)
{
  cudaStream_t s = h->stream;
  const int64_t n_tiles = std::max<int64_t>((n_rows + TS_ROWS - 1) / TS_ROWS, 1), n32 = n_tiles * TS_ROWS;
  std::vector<uint8_t> tiles((size_t)n_tiles * TILE_BYTES, 0);
  std::vector<double4> hdr((size_t)n32, make_double4(0.0, 0.0, 0.0, 0.0));
  for (int64_t r = 0; r < n_rows; r++) {
    for (int slot = 0; slot < ROW_BYTES; slot++)
      tiles[(size_t)(r / TS_ROWS) * TILE_BYTES + slot * TS_ROWS + r % TS_ROWS] = counts[(size_t)r * ROW_BYTES + slot];
    hdr[(size_t)r] = make_double4(0.0, age_begin[r], w_shared[r], w_notshared[r]);
  }
  const size_t off_cnt = 0, off_hdr = off_cnt + tiles.size(), off_brs = off_hdr + hdr.size() * sizeof(double4),
               off_eb = off_brs + (size_t)(n_blocks + 1) * 8, off_ews = (off_eb + (size_t)n32 + 7) / 8 * 8, off_ewn = off_ews + (size_t)n32 * 8,
               off_f = off_ewn + (size_t)n32 * 8, off_n = off_f + (size_t)n_blocks * 4 * NBINS * 8, off_misc = off_n + (size_t)n_blocks * 3 * NBINS * 8,
               total = off_misc + 64;
  CK(h->d_tmp.ensure(total));
  char* d = h->d_tmp.as<char>();
  CK(cudaMemsetAsync(d, 0, total, s));
  CK(cudaMemcpyAsync(d + off_cnt, tiles.data(), tiles.size(), cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d + off_hdr, hdr.data(), hdr.size() * sizeof(double4), cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d + off_brs, blk_rank_start, (size_t)(n_blocks + 1) * 8, cudaMemcpyHostToDevice, s));
  if (n_rows > 0) {
    CK(cudaMemcpyAsync(d + off_eb, emp_bin, (size_t)n_rows, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d + off_ews, emp_ws, (size_t)n_rows * 8, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d + off_ewn, emp_wn, (size_t)n_rows * 8, cudaMemcpyHostToDevice, s));
  }
  const int64_t* brs = (const int64_t*)(d + off_brs);
  double* f = (double*)(d + off_f);
  int64_t* nn = (int64_t*)(d + off_n);
  int64_t* misc = (int64_t*)(d + off_misc);
  if (n_blocks > 0) {
    launch_emp(s, n_blocks, brs, (const uint8_t*)(d + off_eb), (const double*)(d + off_ews), (const double*)(d + off_ewn), f, nn);
    launch_replay(s, n_blocks, brs, (const uint8_t*)(d + off_cnt), (const double4*)(d + off_hdr), f, nn, misc);
    CK(cudaGetLastError());
  }
  int64_t m[8];
  CK(cudaMemcpyAsync(out_f, f, (size_t)n_blocks * 4 * NBINS * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(out_n, nn, (size_t)n_blocks * 3 * NBINS * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(m, misc, 64, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  *out_of_range = m[3] != 0;
  return 0;
}

}  // namespace colate
