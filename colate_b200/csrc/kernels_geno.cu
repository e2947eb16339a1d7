// make_tmp from a genotype matrix on the device (DESIGN.md section 6l): the .colate.in of many individuals of one EIGENSTRAT or
// PLINK dataset, each byte for byte what colate_maketmp_table writes from the (chromosome, position, allele) table of that
// individual's homozygous calls.  Once per job:
//   the matrix rows of the SNPs on listed contigs, uploaded from pinned windows
//   k_geno_join     one thread per .mut row: the row's SNPs (those at exactly its position) as a range of the uploaded rows
//   k_geno_called   per individual and --chr entry: a homozygous call there at all (the table cursor's cut-off), heterozygous calls
// Per batch of individuals and chromosome:
//   k_geno_rows     CTA = 256 rows x one individual of the batch: row filter, mask, cut-off, the first homozygous call among the
//                   row's SNPs -> (AAF, DAF), emit ballots, a count per CTA -- the layout k_maketmp_rows leaves
//   k_maketmp_scan, k_maketmp_scatter (kernels_maketmp.cu, unchanged) per individual into its own record buffer
// Then per individual one copy of its bytes to pinned host memory and the file.
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <map>

#include "device.cuh"
#include "geno_reader.h"
#include "maketmp_word.h"

using namespace colate;

namespace {

constexpr int GN_THREADS = 256;       // = the CTA of k_maketmp_scan / k_maketmp_scatter: one emit word per warp, one count per CTA
constexpr int GN_CALLED_SNPS = 512;   // SNPs per CTA of k_geno_called
constexpr size_t GN_WINDOW = 64u << 20;   // pinned upload window (two of them)
constexpr size_t GN_BATCH_BYTES = 2ull << 30;   // device bytes a batch of individuals may hold in per-row and record buffers

__device__ __forceinline__ int chr_of_row(const int64_t* __restrict__ site_off, int n_chr, int64_t row)
{
  int lo = 0, hi = n_chr - 1;
  while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (site_off[mid] <= row) lo = mid; else hi = mid - 1; }
  return lo;
}

// thread = row of the site set.  A row passing the table variant's filter (word bit 0) gets the uploaded rows [x, y) of the SNPs of
// its --chr entry at exactly its position (SNP positions do not descend within an entry); everything else gets an empty range.
// cand[c] counts chromosome c's rows with a non-empty range (their records bound a file's bytes).
__global__ void __launch_bounds__(GN_THREADS)
k_geno_join(int64_t n_site, const int32_t* __restrict__ pos, const uint32_t* __restrict__ mkt, const int64_t* __restrict__ site_off, int n_chr,
            const int64_t* __restrict__ entry_off, const int32_t* __restrict__ snp_pos, int2* __restrict__ join,
            unsigned long long* __restrict__ cand)
{
  const int64_t row = (int64_t)blockIdx.x * GN_THREADS + threadIdx.x;
  int key = -1;
  if (row < n_site) {
    int2 r = make_int2(0, 0);
    if (mkt[row] & MKT_VCF) {
      const int c = chr_of_row(site_off, n_chr, row);
      const int32_t bp = pos[row];
      int64_t lo = entry_off[c], hi = entry_off[c + 1];
      while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (snp_pos[mid] < bp) lo = mid + 1; else hi = mid; }
      int64_t e = lo;
      hi = entry_off[c + 1];
      while (e < hi) { const int64_t mid = (e + hi) >> 1; if (snp_pos[mid] <= bp) e = mid + 1; else hi = mid; }
      r = make_int2((int)lo, (int)e);
      if (e > lo) key = c;
    }
    join[row] = r;
  }
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  if (key >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&cand[key], (unsigned long long)__popc(peers));
}

// thread = individual i (column col[i]), CTA = GN_CALLED_SNPS uploaded rows: called[i * n_chr + e] |= a homozygous call on entry e,
// het[i] += heterozygous calls
__global__ void __launch_bounds__(GN_THREADS)
k_geno_called(int64_t n_snp, const uint8_t* __restrict__ mat, int64_t row_bytes, int kind, const int32_t* __restrict__ col, int n_ind,
              const int64_t* __restrict__ entry_off, int n_chr, unsigned* __restrict__ called, unsigned long long* __restrict__ het)
{
  const int i = blockIdx.y * GN_THREADS + threadIdx.x;
  if (i >= n_ind) return;
  const int64_t s0 = (int64_t)blockIdx.x * GN_CALLED_SNPS, s1 = min(s0 + GN_CALLED_SNPS, n_snp);
  const int64_t k = col[i];
  int e = 0;
  while (entry_off[e + 1] <= s0) e++;
  bool hom = false;
  unsigned long long nh = 0;
  for (int64_t s = s0; s < s1; s++) {
    while (s >= entry_off[e + 1]) {
      if (hom) atomicOr(&called[(int64_t)i * n_chr + e], 1u);
      hom = false;
      e++;
    }
    const uint32_t code = geno_code(mat + s * row_bytes, k, kind);
    hom |= code < 2;
    nh += code == 2;
  }
  if (hom) atomicOr(&called[(int64_t)i * n_chr + e], 1u);
  if (nh) atomicAdd(&het[i], nh);
}

// CTA = 256 rows of chromosome c x individual b of the batch (blockIdx.y).  The table cursor of colate_maketmp_table, for ascending
// rows and non-descending SNPs: a row passing word bit 0 and the individual's mask, on an entry before the individual's cut-off,
// takes the first SNP at exactly its position with a homozygous call; its allele must be the row's ancestral (DAF 0) or derived
// (DAF 1) letter.  AAF = 1 - DAF.  Output per individual as k_maketmp_rows leaves it: ad[m], a ballot per warp, a count per CTA.
__global__ void __launch_bounds__(GN_THREADS)
k_geno_rows(int64_t row0, int64_t n_rows, int c, const uint32_t* __restrict__ mkt, const int2* __restrict__ join, const uint8_t* __restrict__ mat,
            int64_t row_bytes, int kind, const uint8_t* __restrict__ allele, const int32_t* __restrict__ col, const int32_t* __restrict__ cut,
            const int32_t* __restrict__ mask_of, const uint32_t* __restrict__ masks, int64_t mask_words, int2* __restrict__ ad, int64_t ad_stride,
            uint32_t* __restrict__ emit, int64_t emit_stride, int32_t* __restrict__ blk_cnt, int64_t blk_stride)
{
  const int b = blockIdx.y;
  const int64_t m = (int64_t)blockIdx.x * GN_THREADS + threadIdx.x;
  bool out = false;
  if (m < n_rows && c < cut[b]) {
    const int64_t row = row0 + m;
    const int2 j = join[row];
    const int mid = mask_of[b];
    if (j.x < j.y && (mid < 0 || ((masks[mid * mask_words + (row >> 5)] >> (row & 31)) & 1u))) {
      const uint32_t w = mkt[row], a = (w >> 8) & 0xffu, d = (w >> 16) & 0xffu;
      const int64_t k = col[b];
      for (int s = j.x; s < j.y; s++) {
        const uint32_t code = geno_code(mat + (int64_t)s * row_bytes, k, kind);
        if (code >= 2) continue;
        const uint32_t al = allele[2 * (int64_t)s + code];
        if (al == a || al == d) {
          const int daf = al == d;
          ad[b * ad_stride + m] = make_int2(1 - daf, daf);
          out = true;
        }
        break;
      }
    }
  }
  const uint32_t bits = __ballot_sync(0xffffffffu, out);
  if ((threadIdx.x & 31) == 0 && m < n_rows) emit[b * emit_stride + (m >> 5)] = bits;
  const int n = __syncthreads_count(out);
  if (threadIdx.x == 0) blk_cnt[b * blk_stride + blockIdx.x] = n;
}

inline int64_t blocks_for(int64_t n) { return (n + GN_THREADS - 1) / GN_THREADS; }
inline double secs(std::chrono::steady_clock::time_point a) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - a).count(); }

template <class T> int upload(colate_handle* h, DevBuf& d, const std::vector<T>& v)
{
  CK(d.ensure(v.size() * sizeof(T) + 16));
  if (!v.empty()) CK(cudaMemcpyAsync(d.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream));
  return 0;
}

// the matrix rows of the listed SNPs (g.snp, in entry order) -> h->gn_mat, through two pinned windows
int upload_matrix(colate_handle* h, const GenoScan& g)
{
  const int64_t n = (int64_t)g.snp.size(), rb = g.row_bytes;
  CK(h->gn_mat.ensure((size_t)(n * rb) + 16));
  if (n == 0) return 0;
  const int fd = open(g.matrix.c_str(), O_RDONLY);
  if (fd < 0) return fail(COLATE_ERR_IO, "cannot read " + g.matrix);
  struct stat st;
  const size_t size = fstat(fd, &st) == 0 ? (size_t)st.st_size : 0;
  void* m = size ? mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0) : MAP_FAILED;
  close(fd);
  if (m == MAP_FAILED) return fail(COLATE_ERR_IO, "cannot read " + g.matrix);
  madvise(m, size, MADV_SEQUENTIAL);
  const uint8_t* src = (const uint8_t*)m;
  const size_t win = std::max((size_t)rb, std::min(GN_WINDOW, (size_t)(n * rb)));
  int rc = 0;
  cudaEvent_t ev[2] = {};
  for (int w = 0; w < 2 && !rc; w++) {
    if (h->gn_win[w].ensure(win) != cudaSuccess || cudaEventCreateWithFlags(&ev[w], cudaEventDisableTiming) != cudaSuccess)
      rc = fail(COLATE_ERR_CUDA, "upload of " + g.matrix + ": no pinned window");
  }
  int64_t s = 0, dst = 0;
  for (int w = 0; s < n && !rc; w ^= 1) {
    if (cudaEventSynchronize(ev[w]) != cudaSuccess) { rc = fail(COLATE_ERR_CUDA, "upload of " + g.matrix); break; }
    uint8_t* p = (uint8_t*)h->gn_win[w].p;
    size_t fill = 0;
    while (s < n && fill + rb <= win) {
      int64_t e = s + 1;   // a run of consecutive file rows is one copy
      while (e < n && g.snp[e] == g.snp[e - 1] + 1 && fill + (size_t)(e - s + 1) * rb <= win) e++;
      memcpy(p + fill, src + g.data_off + g.snp[s] * rb, (size_t)(e - s) * rb);
      fill += (size_t)(e - s) * rb;
      s = e;
    }
    if (cudaMemcpyAsync(h->gn_mat.as<uint8_t>() + dst, p, fill, cudaMemcpyHostToDevice, h->stream) != cudaSuccess ||
        cudaEventRecord(ev[w], h->stream) != cudaSuccess)
      rc = fail(COLATE_ERR_CUDA, "upload of " + g.matrix);
    dst += (int64_t)fill;
  }
  if (cudaStreamSynchronize(h->stream) != cudaSuccess && !rc) rc = fail(COLATE_ERR_CUDA, "upload of " + g.matrix);
  for (auto& e : ev) if (e) cudaEventDestroy(e);
  munmap(m, size);
  if (rc) return rc;
  h->geno_uploads++;
  h->geno_h2d_bytes += dst;
  return 0;
}

}  // namespace

extern "C" {

int64_t colate_maketmp_write_geno(colate_handle* h, const char* prefix, int format, int n_ind, const char* const* ind_ids, int n_chr,
                                  const char* const* chr_names, const char* const* out_files, const int32_t* mask_ids, const uint32_t* mask_bits,
                                  int64_t* records_out, int64_t* het_skipped_out, int32_t* cutoff_out)
{
  const char* fn = "colate_maketmp_write_geno";
  if (!h || !prefix || n_ind <= 0 || !ind_ids || n_chr <= 0 || !chr_names || !out_files) return fail(COLATE_ERR_ARG, std::string(fn) + ": bad arguments");
  for (int i = 0; i < n_ind; i++)
    if (!ind_ids[i] || !out_files[i] || (mask_ids && mask_ids[i] >= 0 && !mask_bits)) return fail(COLATE_ERR_ARG, std::string(fn) + ": bad arguments");
  const auto t_start = std::chrono::steady_clock::now();
  double t[10] = {};
  GenoScan g;
  if (int rc = geno_scan(prefix, format, n_chr, chr_names, g)) return rc;
  std::map<std::string, int64_t> where;
  for (int64_t k = 0; k < g.n_ind; k++) {
    auto it = where.emplace(g.ids[k], k).first;
    if (it->second != k) it->second = -1;   // occurs twice: not an individual's unique column
  }
  const std::string f_ind = std::string(prefix) + (format == COLATE_GENO_EIGENSTRAT ? ".ind" : ".fam");
  std::vector<int32_t> col(n_ind), mask_of(n_ind, -1);
  int n_mask = 0;
  for (int i = 0; i < n_ind; i++) {
    auto it = where.find(ind_ids[i]);
    if (it == where.end()) return fail(COLATE_ERR_ARG, std::string(fn) + ": individual " + ind_ids[i] + " is not in " + f_ind);
    if (it->second < 0) return fail(COLATE_ERR_ARG, std::string(fn) + ": individual " + ind_ids[i] + " occurs more than once in " + f_ind);
    col[i] = (int32_t)it->second;
    if (mask_ids && mask_ids[i] >= 0) { mask_of[i] = mask_ids[i]; n_mask = std::max(n_mask, mask_ids[i] + 1); }
  }
  t[0] = secs(t_start);

  if (!h->sites_set || n_chr != h->n_chr) return fail(COLATE_ERR_ARG, std::string(fn) + ": the --chr list must be the site set's chromosomes");
  if (!h->mkt_valid) return fail(COLATE_ERR_STATE, std::string(fn) + ": the sites have no make_tmp row words (colate_ingest_* or colate_set_maketmp_words)");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  int order = 0;
  CK(cudaMemcpyAsync(&order, h->order_flag.p, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (order) return fail(COLATE_ERR_ORDER, "positions of a .mut file are not ascending (the reference's sequential reader needs sorted input)");
  std::vector<std::string> names(chr_names, chr_names + n_chr);
  std::string all_names;
  std::vector<int64_t> name_off{0};
  for (auto& nm : names) {
    if (nm.size() > 800) return fail(COLATE_ERR_ARG, std::string(fn) + ": chromosome names longer than 800 bytes are not supported");
    all_names += nm;
    name_off.push_back((int64_t)all_names.size());
  }

  // once per job: the matrix, the SNP arrays, the join, the called flags
  auto t1 = std::chrono::steady_clock::now();
  if (int rc = upload_matrix(h, g)) return rc;
  t[1] = secs(t1);
  const int64_t n_snp = (int64_t)g.snp.size(), n_site = h->n_site, mask_words = (n_site + 31) / 32;
  std::vector<int64_t> site_off(h->h_site_off.begin(), h->h_site_off.end());
  if (int rc = upload(h, h->gn_snp_pos, g.pos)) return rc;
  if (int rc = upload(h, h->gn_allele, g.allele)) return rc;
  if (int rc = upload(h, h->gn_entry_off, g.entry_off)) return rc;
  if (int rc = upload(h, h->gn_site_off, site_off)) return rc;
  if (int rc = upload(h, h->gn_col, col)) return rc;
  if (int rc = upload(h, h->gn_mask_of, mask_of)) return rc;
  CK(h->gn_join.ensure((size_t)n_site * 8 + 16));
  CK(h->gn_called.ensure((size_t)n_ind * n_chr * 4 + (size_t)n_ind * 8 + (size_t)n_chr * 8 + 64));
  unsigned* d_called = h->gn_called.as<unsigned>();
  unsigned long long* d_het = (unsigned long long*)(h->gn_called.as<char>() + (((size_t)n_ind * n_chr * 4 + 15) & ~(size_t)15));
  unsigned long long* d_cand = d_het + n_ind;
  CK(cudaMemsetAsync(h->gn_called.p, 0, h->gn_called.cap, st));
  CK(h->gn_name.ensure(all_names.size() + 16));
  if (!all_names.empty()) CK(cudaMemcpyAsync(h->gn_name.p, all_names.data(), all_names.size(), cudaMemcpyHostToDevice, st));
  if (n_mask) {
    CK(h->gn_masks.ensure((size_t)n_mask * mask_words * 4 + 16));
    CK(cudaMemcpyAsync(h->gn_masks.p, mask_bits, (size_t)n_mask * mask_words * 4, cudaMemcpyHostToDevice, st));
  }
  cudaEvent_t ev[4] = {};
  struct Events { cudaEvent_t* e; ~Events() { for (int k = 0; k < 4; k++) if (e[k]) cudaEventDestroy(e[k]); } } ev_guard{ev};
  for (auto& e : ev) CK(cudaEventCreate(&e));
  CK(cudaEventRecord(ev[0], st));
  if (n_site)
    k_geno_join<<<(unsigned)blocks_for(n_site), GN_THREADS, 0, st>>>(n_site, h->pos.as<int32_t>(), h->mkt.as<uint32_t>(), h->gn_site_off.as<int64_t>(), n_chr,
                                                                     h->gn_entry_off.as<int64_t>(), h->gn_snp_pos.as<int32_t>(), h->gn_join.as<int2>(), d_cand);
  CK(cudaEventRecord(ev[1], st));
  if (n_snp)
    k_geno_called<<<dim3((unsigned)((n_snp + GN_CALLED_SNPS - 1) / GN_CALLED_SNPS), (unsigned)((n_ind + GN_THREADS - 1) / GN_THREADS)), GN_THREADS, 0, st>>>(
        n_snp, h->gn_mat.as<uint8_t>(), g.row_bytes, g.kind, h->gn_col.as<int32_t>(), n_ind, h->gn_entry_off.as<int64_t>(), n_chr, d_called, d_het);
  CK(cudaEventRecord(ev[2], st));
  h->launches += 2;
  CK(cudaGetLastError());
  std::vector<unsigned> called((size_t)n_ind * n_chr);
  std::vector<unsigned long long> het(n_ind), cand(n_chr);
  CK(cudaMemcpyAsync(called.data(), d_called, called.size() * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(het.data(), d_het, het.size() * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(cand.data(), d_cand, cand.size() * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, ev[0], ev[1]));
  t[2] = ms;
  CK(cudaEventElapsedTime(&ms, ev[1], ev[2]));
  t[3] = ms;
  // the cut-off: the table cursor seeks an entry without a line of the individual through the rest of the table
  std::vector<int32_t> cut(n_ind, 0);
  for (int i = 0; i < n_ind; i++) {
    while (cut[i] < n_chr && called[(size_t)i * n_chr + cut[i]]) cut[i]++;
    if (het_skipped_out) het_skipped_out[i] = (int64_t)het[i];
    if (cutoff_out) cutoff_out[i] = cut[i];
  }
  if (int rc = upload(h, h->gn_cut, cut)) return rc;

  // per batch of individuals: per-row buffers of the longest chromosome, a record buffer bounded by the rows that have SNPs
  int64_t max_rows = 0;
  size_t out_bound = 16;
  for (int c = 0; c < n_chr; c++) {
    max_rows = std::max(max_rows, site_off[c + 1] - site_off[c]);
    out_bound += (size_t)cand[c] * (size_t)(18 + name_off[c + 1] - name_off[c]);
  }
  out_bound = (out_bound + 15) & ~(size_t)15;
  const int64_t nb_max = blocks_for(max_rows), emit_stride = max_rows / 32 + 1;
  const size_t per_ind = (size_t)max_rows * 8 + (size_t)emit_stride * 4 + (size_t)nb_max * 12 + 64 + out_bound;
  const int B = (int)std::max<int64_t>(1, std::min<int64_t>({(int64_t)n_ind, 64, (int64_t)(GN_BATCH_BYTES / per_ind)}));
  CK(h->gn_ad.ensure((size_t)B * max_rows * 8 + 16));
  CK(h->gn_emit.ensure((size_t)B * emit_stride * 4 + 16));
  CK(h->gn_blk.ensure((size_t)B * nb_max * 4 + 16));
  CK(h->gn_blk_off.ensure((size_t)B * nb_max * 8 + 16));
  CK(h->gn_acc.ensure((size_t)B * 4 * 8 + 16));
  CK(h->gn_out.ensure((size_t)B * out_bound + 16));
  CK(h->mk_host.ensure(out_bound + 16));
  std::vector<long long> acc0((size_t)B * 4), acc((size_t)B * 4);
  for (int b = 0; b < B; b++) { acc0[4 * b + 3] = (long long)~0ull; }
  int64_t n_failed = 0;
  for (int i0 = 0; i0 < n_ind; i0 += B) {
    const int nbat = std::min(B, n_ind - i0);
    CK(cudaMemcpyAsync(h->gn_acc.p, acc0.data(), (size_t)nbat * 32, cudaMemcpyHostToDevice, st));
    for (int c = 0; c < n_chr; c++) {
      const int64_t r0 = site_off[c], nr = site_off[c + 1] - r0;
      if (nr == 0) continue;
      const int L = (int)(name_off[c + 1] - name_off[c]);
      const int64_t nb = blocks_for(nr);
      CK(cudaEventRecord(ev[0], st));
      k_geno_rows<<<dim3((unsigned)nb, (unsigned)nbat), GN_THREADS, 0, st>>>(
          r0, nr, c, h->mkt.as<uint32_t>(), h->gn_join.as<int2>(), h->gn_mat.as<uint8_t>(), g.row_bytes, g.kind, h->gn_allele.as<uint8_t>(),
          h->gn_col.as<int32_t>() + i0, h->gn_cut.as<int32_t>() + i0, h->gn_mask_of.as<int32_t>() + i0, h->gn_masks.as<uint32_t>(), mask_words,
          h->gn_ad.as<int2>(), max_rows, h->gn_emit.as<uint32_t>(), emit_stride, h->gn_blk.as<int32_t>(), nb_max);
      h->launches++;
      CK(cudaGetLastError());
      CK(cudaEventRecord(ev[1], st));
      for (int b = 0; b < nbat; b++)
        if (int rc = maketmp_scan_scatter(h, r0, nr, h->gn_blk.as<int32_t>() + b * nb_max, h->gn_blk_off.as<int64_t>() + b * nb_max,
                                          h->gn_acc.as<long long>() + 4 * b, h->gn_ad.as<int2>() + b * max_rows, h->gn_emit.as<uint32_t>() + b * emit_stride,
                                          h->gn_name.as<uint8_t>() + name_off[c], L, h->gn_out.as<uint8_t>() + b * out_bound))
          return rc;
      CK(cudaEventRecord(ev[2], st));
      CK(cudaEventSynchronize(ev[2]));
      CK(cudaEventElapsedTime(&ms, ev[0], ev[1]));
      t[4] += ms;
      CK(cudaEventElapsedTime(&ms, ev[1], ev[2]));
      t[5] += ms;
    }
    CK(cudaMemcpyAsync(acc.data(), h->gn_acc.p, (size_t)nbat * 32, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int b = 0; b < nbat; b++) {
      const int i = i0 + b;
      const size_t n_bytes = (size_t)acc[4 * b + 1];
      const auto ta = std::chrono::steady_clock::now();
      if (n_bytes) CK(cudaMemcpyAsync(h->mk_host.p, h->gn_out.as<uint8_t>() + b * out_bound, n_bytes, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      t[6] += secs(ta);
      const auto tb = std::chrono::steady_clock::now();
      FILE* fp = fopen(out_files[i], "wb");
      bool ok = fp != nullptr;
      if (fp) {
        ok = fwrite(h->mk_host.p, 1, n_bytes, fp) == n_bytes;
        ok = fclose(fp) == 0 && ok;
        if (!ok) remove(out_files[i]);
      }
      t[7] += secs(tb);
      t[9] += ok ? (double)n_bytes : 0.0;
      if (records_out) records_out[i] = ok ? acc[4 * b] : -1;
      if (!ok) {
        n_failed++;
        set_error(std::string("cannot write ") + out_files[i]);
      }
    }
  }
  t[8] = secs(t_start);
  memcpy(h->gn_timing, t, sizeof t);
  return n_failed;
}

int colate_last_geno_timing(colate_handle* h, double* out10)
{
  if (!h || !out10) return fail(COLATE_ERR_ARG, "colate_last_geno_timing: bad arguments");
  memcpy(out10, h->gn_timing, sizeof h->gn_timing);
  return 0;
}

int colate_geno_upload_counts(colate_handle* h, int64_t* out2)
{
  if (!h || !out2) return fail(COLATE_ERR_ARG, "colate_geno_upload_counts: bad arguments");
  out2[0] = h->geno_uploads;
  out2[1] = h->geno_h2d_bytes;
  return 0;
}

}  // extern "C"
