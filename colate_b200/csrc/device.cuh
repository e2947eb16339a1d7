// Device-side shared declarations: handle layout, buffers, launch helpers.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

#include "internal.h"

namespace colate {

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess)                                                                   \
      return fail(COLATE_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));      \
  } while (0)

// growable device buffer
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes)
  {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return (T*)p; }
};

// growable pinned host buffer (the BGZF readers' windows)
struct Pinned {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes)
  {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 4 + 4096;
    cudaError_t e = cudaMallocHost(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  ~Pinned() { if (p) cudaFreeHost(p); }
};

// decoded BCF / VCF record (kernels_bcf.cu).  a0 / a1: first two alleles as colate_maketmp_records codes them (0 empty or absent,
// the letter, 0xff longer)
struct BcfCol {
  int32_t pos;        // 1-based
  int32_t alt_sum;    // sum of bcf_gt_allele over the n_hap haplotypes
  uint8_t a0, a1, biallelic, pad;
};
static_assert(sizeof(BcfCol) == 12, "BcfCol is 12 bytes");

// one .colate.in file on the device, plus its join onto the site axis
struct GenomeDev {
  bool set = false, joined = false, has_mask = false;
  bool pileup = false;        // slot filled by colate_set_pileup: `pile` = int32[n_site][4] reads showing A, C, G, T per row
  bool acgt = false;          // `pile` holds read counts per letter (set_pileup, pileup_*), not the (AAF, DAF) of set_row_counts / rows_from_bcf
  DevBuf pile;
  int64_t n_rec = 0;
  DevBuf bp, aaf, daf, alleles, chr_first, chr_end, mask_bits;
  // join (site-aligned): counts of the record at the row's position, position of the record
  // before it (-1: that record is the first one the reader holds on this chromosome),
  // flag bit0 = a record sits at the row's position, bit1 = its alleles equal the row's
  DevBuf j_aaf, j_daf, j_prevbp, j_flag;
};

struct Stage1Dims {
  int64_t n_used = 0;
  int n_blocks = 0;
};

}  // namespace colate

struct colate_handle {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;   // host -> device copies that run under the kernels of `stream`
  cudaEvent_t copy_done = nullptr;
  cudaStream_t side_stream = nullptr;   // k_emp under the sampler (run_compact forks, run_replay joins)
  cudaEvent_t side_done = nullptr;
  cudaEvent_t ev[8] = {};
  // sites
  bool sites_set = false;
  int n_chr = 0;
  int64_t n_site = 0;
  std::vector<int64_t> h_site_off;
  colate::DevBuf site_off, pos, ab, ae, meta, tile_start, tile_rlo;   // tile_*: k_join's tiles of 256 sites
  colate::DevBuf mkt;           // make_tmp row word per site (maketmp_word.h): colate_ingest_* or colate_set_maketmp_words
  bool mkt_valid = false;
  std::vector<int32_t> h_tile_start;
  bool tiles_valid = false;
  colate::GenomeDev genomes[COLATE_MAX_GENOMES];
  // stage-1 scratch
  bool flags_done = false, sampled = false;
  int tgt_slot = -1, ref_slot = -1;
  colate::DevBuf candR, candT, use, word_rank, scan_tmp, row_of_rank;
  colate::DevBuf chr_used, chr_blocks, chr_block_base, misc;  // misc: small device scalars
  colate::DevBuf u_hdr, u_eb2, u_ews, u_ewn, u_blk, u_cnt;   // compacted used rows, per-row sample counts
  colate::DevBuf blk_rank_start, out_f, out_n, deep_rows;
  int64_t n_deep = 0;           // used rows of the current pair that take the rejection-sampling path (coal.cpp:2279-2294)
  int64_t extra_words = 0;      // generator words the last stage-i call consumed beyond 200 per used row (redraws)
  double h_agebin[COLATE_NUM_AGE_BINS] = {};   // the age grid the EM evaluates (default: colate_age_bins(); colate_set_age_bins())
  double thr185 = 0.0;          // 10 * age from which the age bin is 185 (thr10[185])
  colate::DevBuf windows, rng_stream, mt_tail, poly, thr10, thrA, lut;
  int sm_count = 148;
  std::vector<int64_t> h_chr_used;
  std::vector<int32_t> h_chr_blocks;
  int64_t n_used = 0;
  int n_blocks_local = 0;
  int64_t mt_total_local = 0;
  // generator-stream cache (colate_set_stream_cache): state, offset and length of the tile-ordered stream in rng_stream
  bool stream_cache_on = false, sc_valid = false, mt_tail_gather = false;
  uint32_t sc_state[624] = {};
  int64_t sc_word0 = -1, sc_nwords = 0, sc_off = 0;
  bool thr_ready = false;
  colate_stage1_timing timing = {};
  // stage 2/3
  colate::DevBuf d_counts, d_blockstats, d_weights, d_epochs, d_rates, d_iters, d_ll, d_agebin, d_tmp, d_scratch, d_prof, libm_tab;
  int libm_exact = -1;  // host libm == glibc_math.cuh port on the self-check sample (1/0), -1 unknown
  int counts_R = 0;
  // colate_stage3_em_begin / _end: one EM in flight on its own stream while the next pair is uploaded and taken through stage i
  cudaStream_t em_stream = nullptr;
  bool em_inflight = false;
  int em_R = 0, em_E = 0;
  std::vector<double> em_host_in;   // epochs + initial rates of the EM in flight (the async copies read the handle's copy)
  colate::DevBuf d_gr_tab, d_gr_rates;   // colate_stage3_em_grids: grid_of + grid table, rates [R][E_max]
  colate::DevBuf d_em_scratch;      // the EM kernels' global scratch (apart from d_scratch: stage i of the next pair may use that)
  int em_kernel = -1, em_csize = 0;   // last EM launch: 0 k_em, 1 k_em_split, 2 k_em_cta; CTAs per replicate
  int64_t launches = 0;
  bool opt_rejoin = false, opt_async_uploads = false;
  bool opt_raw_weights = false;   // N3: weights of the bcf / bam front-ends (raw counts) instead of tmp/tmp's pseudo-genotype
  bool opt_norm_1e3 = false;      // N3: stage ii divides both count vectors by 1e3 (coal.cpp:3453-3463, every front-end but tmp/tmp)
  // GPU-side .mut ingest (kernels_ingest.cu)
  bool ing_active = false;
  int ing_nchr = 0;
  int64_t ing_cap = 0, ing_fallback_rows = 0, ing_genome_fallbacks = 0;
  double ing_ms = 0.0;
  std::vector<int64_t> ing_off;
  colate::DevBuf ing_text, ing_tile_cnt, ing_tile_off, ing_nl, ing_status, ing_fb, ing_raw;
  colate::DevBuf order_flag;   // device int[4]: unsorted input seen by the order checks (COLATE_ERR_ORDER)
  std::vector<cudaEvent_t> ing_evs;               // one per chromosome text in flight on the copy stream
  void* ing_bounce[2] = {nullptr, nullptr};       // pinned staging for pageable callers
  cudaEvent_t ing_bounce_ev[2] = {nullptr, nullptr};
  // colate_pileup_bam (kernels_bam.cu): one window's bytes and decoded columns, the current contig's reference, the order state
  colate::DevBuf bam_buf, bam_ref, bam_state;
  bool opt_bam_timing = false;
  double bam_timing[10] = {};
  // colate_rows_from_bcf / colate_decode_bcf (kernels_bcf.cu): one window's bytes and record offsets, the decoded columns of one
  // file (12 B per record, resident), the current chromosome's reference genome, the decode state (GT length, first error; per
  // contig for a whole-genome file)
  colate::DevBuf bcf_buf, bcf_cols, bcf_ref, bcf_state;
  int64_t bcf_n_rec = 0;       // records of the last decoded file in bcf_cols
  int32_t bcf_n_hap = 0;
  int64_t vcf_paths[2] = {};   // lines of the last decoded text VCF on k_vcf_decode's fast path only / with a general step
  bool opt_vcf_paths = false;  // (counted only with the vcf_paths test option: the count is an atomic per line)
  bool opt_bcf_timing = false;
  double bcf_timing[10] = {};
  // the --ref_genome resident for a job (colate_set_ref_genome): contigs concatenated, upper-cased
  colate::DevBuf refg;
  std::vector<int64_t> refg_off;   // n + 1 offsets; empty: none
  // the device .colate.in writer (kernels_maketmp.cu): per-row (AAF, DAF), emit ballots, per-block counts / offsets, the records
  colate::DevBuf mk_ad, mk_emit, mk_blk, mk_acc, mk_name, mk_out, mk_mask;
  colate::Pinned mk_host;
  double mk_timing[4] = {};
  // work counters of a job (colate_upload_counts)
  int64_t mut_texts_parsed = 0, mut_rows_parsed = 0, ref_uploads = 0, ref_h2d_bytes = 0;
};

namespace colate {
// kernels_bcf.cu: one BCF or bgzipped text VCF file -> h->bcf_cols (h->bcf_n_rec records of h->bcf_n_hap haplotypes)
int decode_genotype_file(colate_handle* h, const char* path, int64_t chunk_bytes, double* t);
// one whole-genome file: --chr entry c's records at h->bcf_cols [first[c], first[c] + n[c]), n_hap[c] haplotypes
struct GenomeRecs {
  std::vector<int64_t> first, n;
  std::vector<int32_t> n_hap;
};
int decode_genotype_genome(colate_handle* h, const char* path, int n_chr, const char* const* chr_names, int64_t chunk_bytes, double* t, GenomeRecs* gr);
// kernels_sites.cu
int run_join(colate_handle* h, int slot);
int run_flags(colate_handle* h, int tslot, int rslot);
int run_check_sites(colate_handle* h);
int run_check_genome(colate_handle* h, int slot);
// abi.cu
int sites_replaced_ext(colate_handle* h);
int genome_replaced_ext(colate_handle* h, int slot);
int run_compact(colate_handle* h);
int run_sample_rows(colate_handle* h, const uint32_t* stream_local, int64_t row0, int64_t n_rows);
int run_put_count_row(colate_handle* h, int64_t row, const uint8_t* cnt192_host);
int run_replay(colate_handle* h);
int run_pack_row_counts(colate_handle* h, int slot, const int32_t* aaf_dev, const int32_t* daf_dev);
int run_pileup_reads(colate_handle* h, int slot, int chr, int64_t n_reads, const int32_t* pos, const uint8_t* mapq, const int32_t* len,
                     const int64_t* off, const uint8_t* seq, const uint8_t* qual, const uint8_t* ref, int64_t ref_len, int max_len,
                     int mapq_th, int len_th, int mismatch_th, uint8_t* pass_scratch, bool starts_contig, int64_t row_lo, int64_t row_hi);
int run_test_bin_fast(colate_handle* h, int n, const double* a_host, int32_t* fast_host, int32_t* exact_host);
int run_test_bin_sweep(colate_handle* h, uint32_t lo_bits, uint32_t hi_bits, uint64_t* out3_host);
// kernels_mt.cu
int run_mt_stream(colate_handle* h, const uint32_t* mt_state, int64_t word0, int64_t n_words, int log2_chunk_sites,
                  uint32_t** stream_at_word0, uint32_t* window_after /* host, may be null */,
                  bool tiled /* lay the words out in k_sample's tile order (internal.h: stream_phys) */);
int mt_window_after(colate_handle* h, uint32_t* window_after);
// kernels_em.cu
int run_bootstrap(colate_handle* h, int R, int num_blocks, const double* block_stats_dev, double age);
int run_em(colate_handle* h, int R, int E, int max_iter, const double* epochs_host, cudaStream_t stream);
bool em_cta_fits(const colate_handle* h, int E, const double* epochs_host, int* n_pairs_cap, size_t* smem);
// k_em_cta_grids on R replicates: d_epochs / d_rates hold the packed grids and initial rates, d_counts the counts;
// grid_info_dev = int4 {E, offset, n_pairs_cap, 0} per grid; results -> d_gr_rates [R][E_out], d_iters, d_ll
int run_em_grids(colate_handle* h, int R, const int32_t* grid_of_dev, const int* grid_info_dev, int E_out, size_t smem, int max_iter,
                 cudaStream_t stream);
int run_estep(colate_handle* h, int shared, int E, int n_t);
int run_libm(colate_handle* h, int which, int n, const double* x_host, double* y_host);
int run_test_em_prims(colate_handle* h, int which, int n, const double* a_host, const double* b_host, double* y_host, int32_t* ok_host);
}  // namespace colate
