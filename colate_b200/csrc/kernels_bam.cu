// BAM records decoded on the device, then piled up by the pinned counting loop (run_pileup_reads, kernels_sites.cu).
// The host (host_bam.cpp) inflates the BGZF blocks of one window of the file into pinned memory and finds the record
// boundaries; the device reads each record's fixed core, skips its read name, CIGAR and aux data, and writes the columns the
// counting loop consumes.  Window n+1 is inflated on the host while window n is on the device.
#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "bam_reader.h"
#include "device.cuh"

using namespace colate;

namespace {

__device__ __forceinline__ int32_t ld32(const uint8_t* p) { return (int32_t)((uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24); }
__device__ __forceinline__ uint32_t ld16(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8; }

// thread = record.  raw + rec_off[k]: the record's block_size field; its core follows (refID, pos, l_read_name, mapq, bin,
// n_cigar_op, flag, l_seq, next_refID, next_pos, tlen), then read_name, cigar, the packed sequence, the qualities, aux.
// seq_off[k]: where its l_seq letters (seq_nt16_str of the 4-bit codes, htslib.cpp:403) and qualities go.
// Order: a position below the previous record's (the previous chunk's last one of this contig for k = 0, prev[0] when
// has_prev) sets *flag (bam_parser refuses it, htslib.cpp:411-414; negative positions never get here: the host walk refuses
// them).  The last record's position goes to prev_out for the next chunk (the caller swaps the two slots).
__global__ void k_bam_decode(int64_t n, const uint8_t* __restrict__ raw, const int64_t* __restrict__ rec_off, const int64_t* __restrict__ seq_off,
                             int32_t* __restrict__ pos, uint8_t* __restrict__ mapq, int32_t* __restrict__ len, uint8_t* __restrict__ seq,
                             uint8_t* __restrict__ qual, const int32_t* __restrict__ prev_in, int32_t* __restrict__ prev_out, int has_prev,
                             int* __restrict__ flag)
{
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint8_t* r = raw + rec_off[k] + 4;
  const int32_t p = ld32(r + 4), l_seq = ld32(r + 16);
  const uint32_t l_read_name = r[8], n_cigar = ld16(r + 12);
  pos[k] = p;
  mapq[k] = r[9];
  len[k] = l_seq;
  const uint8_t* s = r + 32 + l_read_name + 4 * n_cigar;
  const uint8_t* q = s + ((l_seq + 1) >> 1);
  const char* nt16 = "=ACMGRSVTWYHKDBN";
  uint8_t* so = seq + seq_off[k];
  uint8_t* qo = qual + seq_off[k];
  for (int32_t i = 0; i < l_seq; i++) {
    so[i] = (uint8_t)nt16[(s[i >> 1] >> ((~i & 1) << 2)) & 15];
    qo[i] = q[i];
  }
  const bool bad = k > 0 ? p < ld32(raw + rec_off[k - 1] + 8) : has_prev && p < prev_in[0];
  if (bad) *flag = 1;
  if (k == n - 1) prev_out[0] = p;
}

// fasta::Read upper-cases the reference genome (data.cpp:213-237)
__global__ void k_upper(int64_t n, uint8_t* __restrict__ s)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { const uint8_t c = s[i]; if (c >= 'a' && c <= 'z') s[i] = c - 32; }
}

inline int grid_for(int64_t n, int threads) { return (int)((n + threads - 1) / threads); }
inline size_t up(size_t x) { return (x + 255) & ~(size_t)255; }

int bam_threads()
{
  if (const char* e = getenv("COLATE_BAM_THREADS")) return std::max(1, atoi(e));
  return (int)std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
}

}  // namespace

extern "C" {

int colate_pileup_bam(colate_handle* h, int slot, const char* bam_path, int n_chr, const char* const* chr_names, const uint8_t* const* ref_seqs,
                      const int64_t* ref_lens, int mapq_th, int len_th, int mismatch_th, int64_t chunk_bytes, int32_t* counts_out)
{
  if (!h || slot < 0 || slot >= COLATE_MAX_GENOMES || !bam_path || n_chr <= 0 || !chr_names || (ref_seqs && !ref_lens) || chunk_bytes < 0)
    return fail(COLATE_ERR_ARG, "colate_pileup_bam: bad arguments");
  if (!h->sites_set || n_chr != h->n_chr) return fail(COLATE_ERR_ARG, "colate_pileup_bam: the --chr list must be the site set's chromosomes");
  const bool resident = ref_seqs == nullptr;   // the genome of colate_set_ref_genome, already on the device
  if (resident && (int)h->refg_off.size() != n_chr + 1)
    return fail(COLATE_ERR_STATE, "colate_pileup_bam: ref_seqs = NULL needs colate_set_ref_genome with one contig per chromosome");
  for (int c = 0; c < n_chr && !resident; c++)
    if (ref_lens[c] < 0 || (ref_lens[c] > 0 && !ref_seqs[c])) return fail(COLATE_ERR_ARG, "colate_pileup_bam: bad reference sequence");
  auto ref_len_of = [&](int c) { return resident ? h->refg_off[c + 1] - h->refg_off[c] : ref_lens[c]; };
  const auto t_start = std::chrono::steady_clock::now();
  BamReader rd;
  if (int rc = rd.open(bam_path, n_chr, chr_names, bam_threads())) return rc;
  if (int rc = colate_pileup_begin(h, slot)) return rc;
  cudaStream_t s = h->stream;
  // the site positions on the host: a chunk searches only the rows its reads can cover
  std::vector<int32_t> site_pos((size_t)h->n_site);
  if (h->n_site) CK(cudaMemcpyAsync(site_pos.data(), h->pos.p, (size_t)h->n_site * 4, cudaMemcpyDeviceToHost, s));
  CK(h->bam_state.ensure(16));
  CK(cudaMemsetAsync(h->bam_state.p, 0, 16, s));
  CK(cudaStreamSynchronize(s));
  std::vector<char> sorted(n_chr, 1);
  for (int c = 0; c < n_chr; c++)
    for (int64_t m = h->h_site_off[c] + 1; m < h->h_site_off[c + 1]; m++)
      if (site_pos[m] < site_pos[m - 1]) { sorted[c] = 0; break; }

  const size_t target = chunk_bytes > 0 ? (size_t)chunk_bytes : (size_t)64 << 20;
  Pinned raw[2], meta[2];
  cudaEvent_t done[2];
  bool pending[2] = {false, false};
  for (auto& e : done) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  struct Ev { cudaEvent_t* e; ~Ev() { cudaEventDestroy(e[0]); cudaEventDestroy(e[1]); } } ev_guard{done};
  // bam_timing option: events around the copies, the decode and the pileup of every chunk, and a wait after each chunk
  // (so the host and the device no longer overlap: the phases are for a breakdown, the wall time is measured without it)
  cudaEvent_t tev[5] = {};
  if (h->opt_bam_timing)
    for (auto& e : tev) CK(cudaEventCreate(&e));
  struct TEv { cudaEvent_t* e; ~TEv() { for (int i = 0; i < 5; i++) if (e[i]) cudaEventDestroy(e[i]); } } tev_guard{tev};
  double h2d_ms = 0, decode_ms = 0, pileup_ms = 0;
  int64_t n_records = 0, n_inflated = 0;
  int cur = -1, parity = 0;
  BamWindow w;
  for (int wi = 0;; wi++) {
    const int b = wi & 1;
    const size_t need = rd.next_window_bytes(target);
    if (need == 0) break;
    if (pending[b]) { CK(cudaEventSynchronize(done[b])); pending[b] = false; }   // window wi - 2 has left this buffer
    CK(raw[b].ensure(need));
    if (int rc = rd.fill((uint8_t*)raw[b].p, target, w)) { cudaStreamSynchronize(s); return rc; }
    n_inflated += (int64_t)w.n_bytes;
    const int64_t n = (int64_t)w.rec_off.size();
    if (n == 0) continue;
    n_records += n;
    // record offsets and letter offsets (prefix sum of l_seq) go up next to the bytes
    CK(meta[b].ensure((size_t)n * 16));
    int64_t* h_rec = (int64_t*)meta[b].p;
    int64_t* h_seq = h_rec + n;
    int64_t n_letters = 0;
    for (int64_t k = 0; k < n; k++) { h_rec[k] = w.rec_off[k]; h_seq[k] = n_letters; n_letters += w.rec_lseq[k]; }
    const size_t o_raw = 0, o_rec = o_raw + up(w.n_bytes), o_seqo = o_rec + n * 8, o_pos = o_seqo + up(n * 8), o_len = o_pos + up(n * 4),
                 o_mq = o_len + up(n * 4), o_pass = o_mq + up(n), o_seq = o_pass + up(n), o_q = o_seq + up(n_letters), total = o_q + up(n_letters);
    CK(h->bam_buf.ensure(total));   // (a reallocation waits for the device: cudaFree synchronises)
    char* d = h->bam_buf.as<char>();
    if (tev[0]) CK(cudaEventRecord(tev[0], s));
    CK(cudaMemcpyAsync(d + o_raw, raw[b].p, w.n_bytes, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d + o_rec, h_rec, (size_t)n * 16, cudaMemcpyHostToDevice, s));
    if (tev[0]) CK(cudaEventRecord(tev[1], s));
    const int64_t* d_rec = (const int64_t*)(d + o_rec);
    const int64_t* d_seqo = (const int64_t*)(d + o_seqo);
    int32_t* d_pos = (int32_t*)(d + o_pos);
    int32_t* d_len = (int32_t*)(d + o_len);
    uint8_t* d_mq = (uint8_t*)(d + o_mq);
    // chunks: runs of one contig's records, at most `target` record bytes each (at least one record)
    for (int64_t r0 = 0; r0 < n;) {
      const int c = w.rec_chr[r0];
      int64_t r1 = r0 + 1;
      while (r1 < n && w.rec_chr[r1] == c && (size_t)((r1 + 1 < n ? w.rec_off[r1 + 1] : (int64_t)w.n_bytes) - w.rec_off[r0]) <= target) r1++;
      const bool starts = c != cur;
      if (starts && !resident) {
        // this contig's reference genome, upper-cased on the device
        const int64_t L = ref_lens[c];
        CK(h->bam_ref.ensure((size_t)L + 16));
        if (L) {
          CK(cudaMemcpyAsync(h->bam_ref.p, ref_seqs[c], (size_t)L, cudaMemcpyHostToDevice, s));
          h->ref_h2d_bytes += L;
          k_upper<<<grid_for(L, 256), 256, 0, s>>>(L, h->bam_ref.as<uint8_t>());
          h->launches += 1;
        }
      }
      cur = c;
      const uint8_t* d_ref = resident ? h->refg.as<uint8_t>() + h->refg_off[c] : h->bam_ref.as<uint8_t>();
      int32_t* st = h->bam_state.as<int32_t>();
      if (tev[0]) CK(cudaEventRecord(tev[2], s));
      k_bam_decode<<<grid_for(r1 - r0, 256), 256, 0, s>>>(r1 - r0, (const uint8_t*)(d + o_raw), d_rec + r0, d_seqo + r0, d_pos + r0, d_mq + r0,
                                                          d_len + r0, (uint8_t*)(d + o_seq), (uint8_t*)(d + o_q), st + parity, st + (parity ^ 1),
                                                          starts ? 0 : 1, (int*)(st + 2));
      h->launches += 1;
      CK(cudaGetLastError());
      parity ^= 1;
      if (tev[0]) CK(cudaEventRecord(tev[3], s));
      // rows [first pos, last pos + max_len) of the contig, 0-based positions (only where the contig's rows are sorted)
      int max_len = 0;
      for (int64_t k = r0; k < r1; k++) max_len = std::max(max_len, w.rec_lseq[k]);
      int64_t row_lo = 0, row_hi = -1;
      if (sorted[c]) {
        const int32_t* b0 = site_pos.data() + h->h_site_off[c];
        const int32_t* b1 = site_pos.data() + h->h_site_off[c + 1];
        const int64_t lo = (int64_t)w.rec_pos[r0] + 1, hi = (int64_t)w.rec_pos[r1 - 1] + max_len;   // 1-based row positions
        row_lo = std::lower_bound(b0, b1, lo, [](int32_t a, int64_t v) { return (int64_t)a < v; }) - b0;
        row_hi = std::lower_bound(b0, b1, hi + 1, [](int32_t a, int64_t v) { return (int64_t)a < v; }) - b0;
        if (w.rec_pos[r1 - 1] < w.rec_pos[r0]) { row_lo = 0; row_hi = -1; }   // refused below; the counts are not used
      }
      if (int rc = run_pileup_reads(h, slot, c, r1 - r0, d_pos + r0, d_mq + r0, d_len + r0, d_seqo + r0, (const uint8_t*)(d + o_seq),
                                    (const uint8_t*)(d + o_q), d_ref, ref_len_of(c), max_len, mapq_th, len_th, mismatch_th,
                                    (uint8_t*)(d + o_pass) + r0, starts, row_lo, row_hi)) {
        cudaStreamSynchronize(s);
        return rc;
      }
      if (tev[0]) {
        CK(cudaEventRecord(tev[4], s));
        CK(cudaEventSynchronize(tev[4]));
        float ms = 0;
        if (r0 == 0) { CK(cudaEventElapsedTime(&ms, tev[0], tev[1])); h2d_ms += ms; }
        CK(cudaEventElapsedTime(&ms, tev[2], tev[3]));
        decode_ms += ms;
        CK(cudaEventElapsedTime(&ms, tev[3], tev[4]));
        pileup_ms += ms;
      }
      r0 = r1;
    }
    CK(cudaEventRecord(done[b], s));
    pending[b] = true;
  }
  CK(cudaStreamSynchronize(s));
  int flag = 0;
  CK(cudaMemcpy(&flag, h->bam_state.as<int32_t>() + 2, 4, cudaMemcpyDeviceToHost));
  h->bam_timing[0] = rd.index_s;
  h->bam_timing[1] = rd.inflate_s;
  h->bam_timing[2] = rd.walk_s;
  h->bam_timing[3] = h2d_ms;
  h->bam_timing[4] = decode_ms;
  h->bam_timing[5] = pileup_ms;
  h->bam_timing[6] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
  h->bam_timing[7] = rd.n_threads;
  h->bam_timing[8] = (double)n_inflated;
  h->bam_timing[9] = (double)n_records;
  if (flag) return fail(COLATE_ERR_ORDER, "Error: BAM file not sorted by position.");   // htslib.cpp:411-414
  return colate_pileup_end(h, slot, counts_out);
}

int colate_set_ref_genome(colate_handle* h, int n_chr, const uint8_t* const* ref_seqs, const int64_t* ref_lens)
{
  if (!h || n_chr < 0 || (n_chr > 0 && (!ref_seqs || !ref_lens))) return fail(COLATE_ERR_ARG, "colate_set_ref_genome: bad arguments");
  std::vector<int64_t> off(1, 0);
  for (int c = 0; c < n_chr; c++) {
    if (ref_lens[c] < 0 || (ref_lens[c] > 0 && !ref_seqs[c])) return fail(COLATE_ERR_ARG, "colate_set_ref_genome: bad reference sequence");
    off.push_back(off.back() + ref_lens[c]);
  }
  CK(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  CK(cudaStreamSynchronize(s));   // nothing may still read the genome this call replaces
  h->refg_off.clear();
  if (n_chr == 0) return 0;
  CK(h->refg.ensure((size_t)off.back() + 16));
  for (int c = 0; c < n_chr; c++)
    if (ref_lens[c]) CK(cudaMemcpyAsync(h->refg.as<uint8_t>() + off[c], ref_seqs[c], (size_t)ref_lens[c], cudaMemcpyHostToDevice, s));
  if (off.back()) {
    k_upper<<<grid_for(off.back(), 256), 256, 0, s>>>(off.back(), h->refg.as<uint8_t>());
    h->launches += 1;
    CK(cudaGetLastError());
  }
  CK(cudaStreamSynchronize(s));   // the caller's sequences are free again
  h->refg_off = off;
  h->ref_uploads += 1;
  h->ref_h2d_bytes += off.back();
  return 0;
}

int colate_last_bam_timing(colate_handle* h, double* out)
{
  if (!h || !out) return fail(COLATE_ERR_ARG, "colate_last_bam_timing: bad arguments");
  memcpy(out, h->bam_timing, sizeof h->bam_timing);
  return 0;
}

}  // extern "C"
