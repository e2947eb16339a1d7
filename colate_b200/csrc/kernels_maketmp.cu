// The .colate.in writer of make_tmp on the device (DESIGN.md section 6i): what maketmp_bam (coal.cpp:2527-2680) and maketmp_vcf
// (coal.cpp:2325-2525) write, from what is already resident -- the sites, their make_tmp row words (maketmp_word.h), and either a
// slot's pileup counts or the decoded records of one BCF / VCF file.  Per chromosome:
//   k_maketmp_rows<kind>   one thread per row: the row filter, the mask, the variant's counts -> emit ballot, (AAF, DAF), a count per CTA
//   k_maketmp_scan         one CTA: exclusive offsets of the CTAs' records, running record and byte totals of the file
//   k_maketmp_scatter      one CTA per 256 rows: its records assembled in shared memory, stored with 4-byte coalesced stores
// The host copies the bytes out once into pinned memory and writes the file.  colate_maketmp_pileup / colate_maketmp_records
// (host_misc.cpp) stay the reference the writer is tested against.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>

#include "device.cuh"
#include "maketmp_word.h"

using namespace colate;

namespace {

constexpr int MK_THREADS = 256;
constexpr int MK_MAX_NAME = 800;   // 256 records of 18 + L bytes in shared memory (227 KB per CTA)
enum { kPileup = 0, kRecords = 1 };

__device__ __forceinline__ int acgt_index(uint32_t c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1; }
__device__ __forceinline__ int32_t pick(const int4& c, int i) { return i == 0 ? c.x : i == 1 ? c.y : i == 2 ? c.z : c.w; }

// thread = row m of the chromosome (row0 + m of the site set).
//   kPileup (maketmp_bam, coal.cpp:2584-2646): passes the bam filter and the mask, reads > 0; AAF = reads of the ancestral letter,
//     DAF = reads of the derived letter if the derived string is that one letter; emitted iff AAF > 0 || DAF > 0.
//   kRecords (maketmp_vcf, coal.cpp:2381-2511): passes the vcf filter and the mask; the record is the lower bound of the row's
//     position among the file's records, the reader's cursor staying on the last one (rows and records ascend, so that is the
//     record the reference's forward-only cursor holds).  At the row's position: the derived allele alone with allele sum 0 and
//     biallelic gives DAF = N; the row's two alleles in either order, biallelic, give the allele sum (N - sum when flipped); any
//     other record drops the row.  No record there: the genome's base gives DAF = N (derived) or 0 (ancestral), else the row is
//     dropped.  AAF = N - DAF; AAF < 0 fails the file (err = the first such row).
// Output: ad[m] = (AAF, DAF), one emit ballot per warp, the CTA's emitted rows in blk_cnt.
template <int KIND>
__global__ void __launch_bounds__(MK_THREADS)
k_maketmp_rows(int64_t row0, int64_t n_rows, const int32_t* __restrict__ pos, const uint32_t* __restrict__ mkt,
               const uint32_t* __restrict__ mask_bits, const int4* __restrict__ pile, const BcfCol* __restrict__ cols, int64_t n_rec,
               int32_t N, const uint8_t* __restrict__ ref, int64_t ref_len, int2* __restrict__ ad, uint32_t* __restrict__ emit,
               int32_t* __restrict__ blk_cnt, unsigned long long* __restrict__ err)
{
  const int64_t m = (int64_t)blockIdx.x * MK_THREADS + threadIdx.x;
  bool out = false;
  if (m < n_rows) {
    const int64_t row = row0 + m;
    const uint32_t w = mkt[row];
    int32_t aaf = 0, daf = 0;
    const bool pass = (w & (KIND == kPileup ? MKT_BAM : MKT_VCF)) && (!mask_bits || ((mask_bits[row >> 5] >> (row & 31)) & 1u));
    if (pass) {
      const uint32_t a = (w >> 8) & 0xffu, d = (w >> 16) & 0xffu;
      if (KIND == kPileup) {
        const int4 c = pile[row];
        if (c.x + c.y + c.z + c.w > 0) {
          const int ia = acgt_index(a), id = acgt_index(d);
          aaf = ia >= 0 ? pick(c, ia) : 0;
          daf = (w & MKT_ONE) && id >= 0 ? pick(c, id) : 0;
          out = aaf > 0 || daf > 0;
        }
      } else {
        const int32_t bp = pos[row];
        int64_t lo = 0, hi = n_rec;
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (cols[mid].pos < bp) lo = mid + 1; else hi = mid; }
        if (lo == n_rec) lo = n_rec - 1;
        if (lo >= 0 && cols[lo].pos == bp) {
          const BcfCol c = cols[lo];
          if (c.a0 == d && c.a1 == 0) {
            if (c.biallelic && c.alt_sum == 0) { daf = N; out = true; }
          } else if ((c.a0 == a && c.a1 == d) || (c.a0 == d && c.a1 == a)) {
            if (c.biallelic) { daf = (c.a0 == d && c.a1 == a) ? N - c.alt_sum : c.alt_sum; out = true; }
          }
        } else if (ref && bp >= 1 && (int64_t)bp - 1 < ref_len) {
          const uint32_t g = ref[bp - 1];
          if (g == d) { daf = N; out = true; }
          else if (g == a) { daf = 0; out = true; }
        }
        aaf = N - daf;
        if (out && aaf < 0) atomicMin(err, (unsigned long long)row);
      }
    }
    ad[m] = make_int2(aaf, daf);
  }
  const uint32_t bits = __ballot_sync(0xffffffffu, out);
  if ((threadIdx.x & 31) == 0 && m < n_rows) emit[m >> 5] = bits;
  const int n = __syncthreads_count(out);
  if (threadIdx.x == 0) blk_cnt[blockIdx.x] = n;
}

// exclusive scan of the CTAs' record counts (one CTA, chunks of 1024).  acc[0] / acc[1]: records / bytes of the file so far;
// acc[2] = this chromosome's first byte; S = record bytes (18 + name length).
__global__ void __launch_bounds__(1024)
k_maketmp_scan(const int32_t* __restrict__ blk_cnt, int64_t n_blk, int64_t* __restrict__ blk_off, long long* __restrict__ acc, int S)
{
  __shared__ long long ws[32];
  __shared__ long long carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t b = 0; b < n_blk; b += 1024) {
    const int64_t i = b + threadIdx.x;
    const long long v = i < n_blk ? blk_cnt[i] : 0;
    long long x = v;
    for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, x, o); if ((threadIdx.x & 31) >= o) x += y; }
    if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = x;
    __syncthreads();
    if (threadIdx.x < 32) {
      const long long w = ws[threadIdx.x];
      long long z = w;
      for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, z, o); if (threadIdx.x >= o) z += y; }
      ws[threadIdx.x] = z - w;
    }
    __syncthreads();
    const long long excl = carry + ws[threadIdx.x >> 5] + x - v;
    if (i < n_blk) blk_off[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    acc[2] = acc[1];
    acc[0] += carry;
    acc[1] += carry * S;
  }
}

__device__ __forceinline__ void put32(uint8_t* q, uint32_t v) { q[0] = (uint8_t)v; q[1] = (uint8_t)(v >> 8); q[2] = (uint8_t)(v >> 16); q[3] = (uint8_t)(v >> 24); }

// CTA = the 256 rows of k_maketmp_rows' CTA.  Its records {int32 L, name, int32 bp, a, d, int32 AAF, int32 DAF} (coal.cpp:2505-2514)
// are contiguous in the file at acc[2] + blk_off * S but not aligned: each emitting thread writes its record into shared memory at
// its rank, then the CTA stores the run with byte stores up to a 4-byte boundary, 4-byte stores (128 B per warp), byte stores for
// the tail.
__global__ void __launch_bounds__(MK_THREADS)
k_maketmp_scatter(int64_t row0, int64_t n_rows, const int32_t* __restrict__ pos, const uint32_t* __restrict__ mkt, const int2* __restrict__ ad,
                  const uint32_t* __restrict__ emit, const int64_t* __restrict__ blk_off, const long long* __restrict__ acc,
                  const uint8_t* __restrict__ name, int L, uint8_t* __restrict__ out)
{
  extern __shared__ uint8_t sm[];
  __shared__ int wcnt[MK_THREADS / 32];
  const int S = 18 + L;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t m = (int64_t)blockIdx.x * MK_THREADS + threadIdx.x;
  const int64_t m_warp = m - lane;
  const uint32_t bits = m_warp < n_rows ? emit[m_warp >> 5] : 0u;
  if (lane == 0) wcnt[warp] = __popc(bits);
  __syncthreads();
  int before = 0, total = 0;
#pragma unroll
  for (int k = 0; k < MK_THREADS / 32; k++) { before += k < warp ? wcnt[k] : 0; total += wcnt[k]; }
  if ((bits >> lane) & 1u) {
    uint8_t* q = sm + (size_t)(before + __popc(bits & ((1u << lane) - 1u))) * S;
    const int2 v = ad[m];
    const uint32_t w = mkt[row0 + m];
    put32(q, (uint32_t)L);
    for (int i = 0; i < L; i++) q[4 + i] = name[i];
    put32(q + 4 + L, (uint32_t)pos[row0 + m]);
    q[8 + L] = (uint8_t)(w >> 8);
    q[9 + L] = (uint8_t)(w >> 16);
    put32(q + 10 + L, (uint32_t)v.x);
    put32(q + 14 + L, (uint32_t)v.y);
  }
  __syncthreads();
  const int64_t g0 = acc[2] + blk_off[blockIdx.x] * S;
  const int nbytes = total * S;
  const int head = min(nbytes, (int)((4 - (g0 & 3)) & 3));
  if ((int)threadIdx.x < head) out[g0 + threadIdx.x] = sm[threadIdx.x];
  const int nw = (nbytes - head) >> 2;
  uint32_t* ow = (uint32_t*)(out + g0 + head);
  for (int i = threadIdx.x; i < nw; i += MK_THREADS) {
    const uint8_t* p = sm + head + 4 * i;
    ow[i] = (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24;
  }
  const int t0 = head + 4 * nw;
  if (t0 + (int)threadIdx.x < nbytes) out[g0 + t0 + threadIdx.x] = sm[t0 + threadIdx.x];
}

inline int64_t blocks_for(int64_t n) { return (n + MK_THREADS - 1) / MK_THREADS; }

}  // namespace

// the scan and the scatter of one chromosome, after a rows kernel left ad / emit / blk_cnt for its rows [row0, row0 + n_rows)
int colate::maketmp_scan_scatter(colate_handle* h, int64_t row0, int64_t n_rows, const int32_t* blk_cnt, int64_t* blk_off, long long* acc,
                                 const int2* ad, const uint32_t* emit, const uint8_t* name, int L, uint8_t* out)
{
  const int64_t nb = blocks_for(n_rows);
  const size_t smem = (size_t)MK_THREADS * (18 + L);
  if (smem > 48 * 1024) CK(cudaFuncSetAttribute(k_maketmp_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_maketmp_scan<<<1, 1024, 0, h->stream>>>(blk_cnt, nb, blk_off, acc, 18 + L);
  k_maketmp_scatter<<<(unsigned)nb, MK_THREADS, smem, h->stream>>>(row0, n_rows, h->pos.as<int32_t>(), h->mkt.as<uint32_t>(), ad, emit, blk_off, acc,
                                                                    name, L, out);
  h->launches += 2;
  CK(cudaGetLastError());
  return 0;
}

namespace {

// One writer call: the state every chromosome of it shares.
struct Writer {
  colate_handle* h;
  const char* fn;                      // the public entry point, for messages
  std::vector<std::string> names;
  std::vector<int64_t> name_off;
  const uint32_t* d_mask = nullptr;
  cudaEvent_t ev[2] = {};
  float kernel_ms = 0;

  ~Writer() { for (auto& e : ev) if (e) cudaEventDestroy(e); }

  // arguments, the site set's state and the buffers of the call
  int begin(int n_chr, const char* const* chr_names, const uint32_t* mask_bits)
  {
    if (n_chr <= 0 || !chr_names) return fail(COLATE_ERR_ARG, std::string(fn) + ": bad arguments");
    if (!h->sites_set || n_chr != h->n_chr) return fail(COLATE_ERR_ARG, std::string(fn) + ": the --chr list must be the site set's chromosomes");
    if (!h->mkt_valid)
      return fail(COLATE_ERR_STATE, std::string(fn) + ": the sites have no make_tmp row words (colate_ingest_* or colate_set_maketmp_words)");
    CK(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    int order = 0;
    CK(cudaMemcpyAsync(&order, h->order_flag.p, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (order) return fail(COLATE_ERR_ORDER, "positions of a .mut file are not ascending (the reference's sequential reader needs sorted input)");
    name_off.assign(1, 0);
    size_t out_bytes = 0;
    int64_t max_rows = 0;
    for (int c = 0; c < n_chr; c++) {
      if (!chr_names[c]) return fail(COLATE_ERR_ARG, std::string(fn) + ": bad arguments");
      names.emplace_back(chr_names[c]);
      const int64_t L = (int64_t)names.back().size();
      if (L > MK_MAX_NAME) return fail(COLATE_ERR_ARG, std::string(fn) + ": chromosome names longer than " + std::to_string(MK_MAX_NAME) + " bytes are not supported");
      name_off.push_back(name_off.back() + L);
      const int64_t nr = h->h_site_off[c + 1] - h->h_site_off[c];
      out_bytes += (size_t)nr * (size_t)(18 + L);
      max_rows = std::max(max_rows, nr);
    }
    const int64_t nb = blocks_for(max_rows);
    CK(h->mk_ad.ensure((size_t)max_rows * 8 + 16));
    CK(h->mk_emit.ensure((size_t)(max_rows / 32 + 1) * 4 + 16));
    CK(h->mk_blk.ensure((size_t)nb * 12 + 16));
    CK(h->mk_acc.ensure(64));
    CK(h->mk_name.ensure((size_t)name_off.back() + 16));
    CK(h->mk_out.ensure(out_bytes + 16));
    std::string all;
    for (auto& n : names) all += n;
    if (!all.empty()) CK(cudaMemcpyAsync(h->mk_name.p, all.data(), all.size(), cudaMemcpyHostToDevice, s));
    const long long acc0[4] = {0, 0, 0, (long long)~0ull};
    CK(cudaMemcpyAsync(h->mk_acc.p, acc0, sizeof acc0, cudaMemcpyHostToDevice, s));
    if (mask_bits) {
      const size_t nw = (size_t)(h->n_site + 31) / 32;
      CK(h->mk_mask.ensure(nw * 4 + 16));
      CK(cudaMemcpyAsync(h->mk_mask.p, mask_bits, nw * 4, cudaMemcpyHostToDevice, s));
      d_mask = h->mk_mask.as<uint32_t>();
    }
    for (auto& e : ev) CK(cudaEventCreate(&e));
    CK(cudaStreamSynchronize(s));   // the local name string and the caller's mask are free again
    return 0;
  }

  // chromosome c's records, appended on the device
  template <int KIND>
  int chromosome(int c, const int4* pile, const BcfCol* cols, int64_t n_rec, int32_t N, const uint8_t* ref, int64_t ref_len)
  {
    const int64_t r0 = h->h_site_off[c], nr = h->h_site_off[c + 1] - r0;
    if (nr == 0) return 0;
    cudaStream_t s = h->stream;
    const int L = (int)(name_off[c + 1] - name_off[c]);
    const int64_t nb = blocks_for(nr);
    int32_t* blk_cnt = h->mk_blk.as<int32_t>();
    int64_t* blk_off = (int64_t*)(h->mk_blk.as<char>() + (((size_t)nb * 4 + 15) & ~(size_t)15));
    long long* acc = h->mk_acc.as<long long>();
    CK(cudaEventRecord(ev[0], s));
    k_maketmp_rows<KIND><<<(unsigned)nb, MK_THREADS, 0, s>>>(r0, nr, h->pos.as<int32_t>(), h->mkt.as<uint32_t>(), d_mask, pile, cols, n_rec, N, ref,
                                                              ref_len, h->mk_ad.as<int2>(), h->mk_emit.as<uint32_t>(), blk_cnt,
                                                              (unsigned long long*)(acc + 3));
    h->launches++;
    if (int rc = maketmp_scan_scatter(h, r0, nr, blk_cnt, blk_off, acc, h->mk_ad.as<int2>(), h->mk_emit.as<uint32_t>(),
                                      h->mk_name.as<uint8_t>() + name_off[c], L, h->mk_out.as<uint8_t>()))
      return rc;
    CK(cudaEventRecord(ev[1], s));
    CK(cudaEventSynchronize(ev[1]));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ev[0], ev[1]));
    kernel_ms += ms;
    return 0;
  }

  // every chromosome is in: one copy of the bytes to pinned host memory, then the file.  Nothing is written on failure.
  int64_t finish(const char* out_file, const char* what_failed)
  {
    cudaStream_t s = h->stream;
    long long acc[4];
    CK(cudaMemcpyAsync(acc, h->mk_acc.p, sizeof acc, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (acc[3] != (long long)~0ull) {
      int c = 0;
      while (c + 1 < h->n_chr && h->h_site_off[c + 1] <= acc[3]) c++;
      return fail(COLATE_ERR_ARG, "chromosome " + names[c] + ": " + what_failed);
    }
    const size_t n_bytes = (size_t)acc[1];
    CK(h->mk_host.ensure(n_bytes + 16));
    const auto t0 = std::chrono::steady_clock::now();
    if (n_bytes) CK(cudaMemcpyAsync(h->mk_host.p, h->mk_out.p, n_bytes, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const auto t1 = std::chrono::steady_clock::now();
    FILE* fp = fopen(out_file, "wb");
    if (!fp) return fail(COLATE_ERR_IO, std::string("cannot write ") + out_file);
    const bool ok = fwrite(h->mk_host.p, 1, n_bytes, fp) == n_bytes;
    if (fclose(fp) != 0 || !ok) { remove(out_file); return fail(COLATE_ERR_IO, std::string("cannot write ") + out_file); }
    const auto t2 = std::chrono::steady_clock::now();
    h->mk_timing[0] = kernel_ms;
    h->mk_timing[1] = std::chrono::duration<double, std::milli>(t1 - t0).count();
    h->mk_timing[2] = std::chrono::duration<double>(t2 - t1).count();
    h->mk_timing[3] = (double)acc[0];
    return (int64_t)acc[0];
  }
};

// colate_maketmp_write_bcf (bcf_paths, one file per chromosome) and colate_maketmp_write_bcf_genome (genome_path, one file)
int64_t write_bcf(colate_handle* h, const char* fn, int n_chr, const char* const* chr_names, const char* const* bcf_paths, const char* genome_path,
                  const uint32_t* mask_bits, int64_t chunk_bytes, const char* out_file)
{
  const bool has_refg = !h->refg_off.empty();
  if (has_refg && (int)h->refg_off.size() != n_chr + 1)
    return fail(COLATE_ERR_STATE, std::string(fn) + ": the genome of colate_set_ref_genome has another number of chromosomes");
  const auto t_start = std::chrono::steady_clock::now();
  Writer w{h, fn};
  if (int rc = w.begin(n_chr, chr_names, mask_bits)) return rc;
  double t[10] = {};
  GenomeRecs gr;
  // a whole-genome file: every chromosome's records resident from one decode
  if (genome_path)
    if (int rc = decode_genotype_genome(h, genome_path, n_chr, chr_names, chunk_bytes, t, &gr)) return rc;
  for (int c = 0; c < n_chr; c++) {
    // per-chromosome files: decoded records are resident for one file at a time, each chromosome's written right after its decode
    if (!genome_path)
      if (int rc = decode_genotype_file(h, bcf_paths[c], chunk_bytes, t)) return fail(rc, "chromosome " + w.names[c] + ": " + colate_last_error());
    const uint8_t* ref = has_refg ? h->refg.as<uint8_t>() + h->refg_off[c] : nullptr;
    const int64_t ref_len = has_refg ? h->refg_off[c + 1] - h->refg_off[c] : 0;
    const BcfCol* cols = h->bcf_cols.as<BcfCol>() + (genome_path ? gr.first[c] : 0);
    if (int rc = w.chromosome<kRecords>(c, nullptr, cols, genome_path ? gr.n[c] : h->bcf_n_rec, genome_path ? gr.n_hap[c] : h->bcf_n_hap, ref, ref_len))
      return rc;
  }
  t[5] = w.kernel_ms;
  t[6] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
  memcpy(h->bcf_timing, t, sizeof t);
  return w.finish(out_file, "allele sum above the number of haplotypes (the reference asserts, coal.cpp:2511)");
}

}  // namespace

extern "C" {

int colate_set_maketmp_words(colate_handle* h, const uint32_t* words, int location)
{
  if (!h || !words) return fail(COLATE_ERR_ARG, "colate_set_maketmp_words: bad arguments");
  if (!h->sites_set) return fail(COLATE_ERR_STATE, "colate_set_maketmp_words: call colate_set_sites first");
  CK(cudaSetDevice(h->device));
  const size_t n = (size_t)h->n_site;
  CK(h->mkt.ensure(n * 4 + 4));
  if (n) CK(cudaMemcpyAsync(h->mkt.p, words, n * 4, location ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->mkt_valid = true;
  return 0;
}

int colate_fetch_maketmp_words(colate_handle* h, int64_t row0, int64_t n_rows, uint32_t* words)
{
  if (!h || row0 < 0 || n_rows < 0 || (n_rows > 0 && !words)) return fail(COLATE_ERR_ARG, "colate_fetch_maketmp_words: bad arguments");
  if (!h->sites_set || !h->mkt_valid) return fail(COLATE_ERR_STATE, "colate_fetch_maketmp_words: the sites have no make_tmp row words");
  if (row0 + n_rows > h->n_site) return fail(COLATE_ERR_ARG, "colate_fetch_maketmp_words: rows out of range");
  CK(cudaSetDevice(h->device));
  if (n_rows) CK(cudaMemcpyAsync(words, h->mkt.as<uint32_t>() + row0, (size_t)n_rows * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int64_t colate_maketmp_write_pileup(colate_handle* h, int slot, int n_chr, const char* const* chr_names, const uint32_t* mask_bits,
                                    const char* out_file)
{
  if (!h || slot < 0 || slot >= COLATE_MAX_GENOMES || !out_file) return fail(COLATE_ERR_ARG, "colate_maketmp_write_pileup: bad arguments");
  const GenomeDev& g = h->genomes[slot];
  if (!g.set || !g.pileup || !g.acgt)
    return fail(COLATE_ERR_STATE, "colate_maketmp_write_pileup: the slot holds no pileup (colate_pileup_bam, colate_pileup_end or colate_set_pileup)");
  Writer w{h, "colate_maketmp_write_pileup"};
  if (int rc = w.begin(n_chr, chr_names, mask_bits)) return rc;
  for (int c = 0; c < n_chr; c++)
    if (int rc = w.chromosome<kPileup>(c, g.pile.as<int4>(), nullptr, 0, 0, nullptr, 0)) return rc;
  return w.finish(out_file, "");
}

int64_t colate_maketmp_write_bcf(colate_handle* h, int n_chr, const char* const* chr_names, const char* const* bcf_paths, const uint32_t* mask_bits,
                                 int64_t chunk_bytes, const char* out_file)
{
  if (!h || !bcf_paths || chunk_bytes < 0 || !out_file) return fail(COLATE_ERR_ARG, "colate_maketmp_write_bcf: bad arguments");
  for (int c = 0; c < n_chr; c++)
    if (!bcf_paths[c]) return fail(COLATE_ERR_ARG, "colate_maketmp_write_bcf: bad arguments");
  return write_bcf(h, "colate_maketmp_write_bcf", n_chr, chr_names, bcf_paths, nullptr, mask_bits, chunk_bytes, out_file);
}

int64_t colate_maketmp_write_bcf_genome(colate_handle* h, int n_chr, const char* const* chr_names, const char* path, const uint32_t* mask_bits,
                                        int64_t chunk_bytes, const char* out_file)
{
  if (!h || !path || n_chr <= 0 || !chr_names || chunk_bytes < 0 || !out_file) return fail(COLATE_ERR_ARG, "colate_maketmp_write_bcf_genome: bad arguments");
  for (int c = 0; c < n_chr; c++)
    if (!chr_names[c]) return fail(COLATE_ERR_ARG, "colate_maketmp_write_bcf_genome: bad arguments");
  return write_bcf(h, "colate_maketmp_write_bcf_genome", n_chr, chr_names, nullptr, path, mask_bits, chunk_bytes, out_file);
}

int colate_last_maketmp_timing(colate_handle* h, double* out4)
{
  if (!h || !out4) return fail(COLATE_ERR_ARG, "colate_last_maketmp_timing: bad arguments");
  memcpy(out4, h->mk_timing, sizeof h->mk_timing);
  return 0;
}

int colate_upload_counts(colate_handle* h, int64_t* out4)
{
  if (!h || !out4) return fail(COLATE_ERR_ARG, "colate_upload_counts: bad arguments");
  out4[0] = h->mut_texts_parsed;
  out4[1] = h->mut_rows_parsed;
  out4[2] = h->ref_uploads;
  out4[3] = h->ref_h2d_bytes;
  return 0;
}

}  // extern "C"
