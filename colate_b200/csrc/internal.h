// Internal declarations shared by the host translation units and the CUDA ones.
#pragma once
#include <cstdint>
#include <cstddef>
#include <string>
#include <vector>

#include "../../include/colate_b200.h"

namespace colate {

constexpr int NBINS = COLATE_NUM_AGE_BINS;
constexpr int MAX_BLOCKS = COLATE_MAX_BLOCKS;
constexpr int NTHR = NBINS + 1;  // thr10[1..185]; index 0 unused
// age -> bin lookup: cell = (high word of the double >> LUT_SHIFT) - LUT_BASE, 32 cells per octave
// from 2^-4 to 2^24 (a row's age interval then spans at most ~32 32-bit words of the table:
// no shared-memory bank conflicts between the lanes of a warp)
constexpr int LUT_SHIFT = 15;
constexpr int LUT_BASE = 0x3FB00000 >> LUT_SHIFT;
constexpr int LUT_N = (0x41700000 >> LUT_SHIFT) - LUT_BASE;
// Per-row sample counts travel as one byte per age bin: 47 32-bit words per row, bin k in byte k & 3 of
// word k >> 2 (k_sample keeps one row per lane, so a row's samples never meet another row's in a word).
// slot = byte offset in the row.
constexpr int ROW_WORDS = 47;
constexpr int ROW_SLOTS = 4 * ROW_WORDS;  // 188 >= NBINS + 1 (bin 185 = "age out of range")
#if defined(__CUDACC__)
__host__ __device__
#endif
constexpr int slot_of_bin(int k) { return k; }

// The generator stream in HBM is laid out in the order k_sample consumes it: used rows in tiles of 32, the
// 200 words of a row cut into chunks of SAMPLE_CHUNK_WORDS, and tile t / chunk c stored as one contiguous
// [32 rows][SAMPLE_CHUNK_WORDS] block (k_gen scatters, k_sample fetches each block with one 1-D bulk copy).
#ifndef S2_CH_WORDS_
#define S2_CH_WORDS_ 20
#endif
constexpr int SAMPLE_TILE_ROWS = 32;
constexpr int SAMPLE_CHUNK_WORDS = S2_CH_WORDS_;
constexpr int SAMPLE_TILE_WORDS = SAMPLE_TILE_ROWS * 200;
static_assert(200 % SAMPLE_CHUNK_WORDS == 0 && SAMPLE_CHUNK_WORDS % 20 == 0, "chunks: whole steps of 10 samples");
// physical word index of logical word o of the stream buffer; tiling starts at word `off` (a row boundary), off < 0: linear
#if defined(__CUDACC__)
__host__ __device__
#endif
inline int64_t stream_phys(int64_t o, int64_t off)
{
  if (off < 0 || o < off) return o;
  const uint64_t q = (uint64_t)(o - off), row = q / 200u;
  const uint32_t w = (uint32_t)(q - row * 200u), c = w / SAMPLE_CHUNK_WORDS, ww = w - c * SAMPLE_CHUNK_WORDS;
  return off + (int64_t)((((row >> 5) * (200 / SAMPLE_CHUNK_WORDS) + c) * 32 + (row & 31)) * SAMPLE_CHUNK_WORDS + ww);
}
// the generator kernels (kernels_mt.cu), as colate_test_last_gen reports the last one launched: k_gen<TILED, PRE, W32>, k_gen_tma
constexpr int GEN_LINEAR = 0, GEN_TILED_W32 = 1, GEN_TILED_W64 = 2, GEN_PRE_W32 = 3, GEN_PRE_W64 = 4, GEN_TMA = 5;

// error plumbing (thread-local message behind colate_last_error())
void set_error(const std::string& msg);
int fail(int code, const std::string& msg);

// host_mt.cpp
uint32_t mt_temper(uint32_t z);
uint32_t mt_untemper(uint32_t y);
void mt_seed_window(uint32_t seed, uint32_t* w);
void mt_generate_window(uint32_t* w, int64_t n, uint32_t* out);
void draw_block_weights(uint32_t* w, int R, int num_blocks, int32_t* weights);
int64_t sample_deep_row_host(uint32_t* w, double age_begin, double len, uint8_t* cnt /*[192]*/, int64_t max_redraws);
const uint32_t* jump_poly(int q);  // t^(200*2^q) mod p(t), 624 x u32
const uint32_t* jump_poly3(int q); // t^(3*200*2^q) mod p(t)
void jump_window_host(const uint32_t* w, int q, uint32_t* out);

// host_misc.cpp
// thr10[k], k = 1..185: smallest double x with max(0,(int)round(log(x)*10)+1) >= k
// (coal.cpp:2253, 2265, 2284), found by bisection against this host's libm.
// Returns false if log() is not monotone in a +-16 ulp neighbourhood of a threshold.
bool bin_thresholds(double* thr10 /*[NTHR]*/);
// thrA[k], k = 1..185: smallest age a with bin(a) >= k where bin(a) = max(0,(int)round(log(10*a)*10)+1);
// thrA[186] = +inf.  thrP[slot_of_bin(k)] = thrA[k+1] (the threshold that ends bin k, indexed by count slot);
// lut[cell] = slot_of_bin(bin at the lower edge of the cell) | 0x8000 if a threshold lies inside the cell
bool age_thresholds(double* thrA /*[NBINS+2]*/, double* thrP /*[192]*/, uint16_t* lut /*[LUT_N]*/);
int bin_of_x10_host(double x10);
struct ColateInRun { int64_t byte_off; int32_t width; int32_t chr_id; int64_t n_rec; int64_t rec_base; };
int64_t decode_colate_in_host(const char* buf, int64_t sz, const std::vector<std::string>& names, int64_t cap,
                              int32_t* rec_chrom, int32_t* bp, int32_t* aaf, int32_t* daf, uint16_t* alleles);
int64_t colate_in_runs(const char* buf, int64_t sz, const std::vector<std::string>& names, std::vector<ColateInRun>& runs);
void chr_ranges_runs(int n_chr, const std::vector<ColateInRun>& runs, int64_t* chr_first, int64_t* chr_end);
bool slurp(const std::string& path, std::vector<char>& buf);
bool slurp_or_gz(const std::string& path, std::vector<char>& buf);
bool parse_mut_line_fields(const char* p, const char* nl, int32_t* pos, float* age_begin, float* age_end, uint32_t* meta, int* flipped_out,
                           int* n_branch_out, char* type16);
bool parse_mut_line_host(const char* p, const char* nl, int32_t* pos, float* age_begin, float* age_end, uint32_t* meta);

}  // namespace colate

extern "C" {
// test hooks, not part of the public ABI
int colate_test_charpoly_terms(int* out, int cap);
int colate_test_jump_window_host(const uint32_t* w, int q, uint32_t* out);
int colate_test_bin_thresholds(double* thr10);
double colate_test_add_repeated(double acc, double w, int c);
int64_t colate_test_stream_phys(int64_t o, int64_t off);
// host run finder of .colate.in images: runs[n][4] = {byte_off, width, chr_id, n_rec}; chr ranges from the runs
int64_t colate_test_colate_in_runs(const char* buf, int64_t sz, int n_chr, const char* const* chr_names, int cap_runs,
                                   int64_t* runs4, int64_t* chr_first, int64_t* chr_end);
int colate_test_libm(colate_handle* h, int which, int n, const double* x, double* y);
int colate_test_log1p_wide(int n, const double* x, double* y, int32_t* ok);
int colate_test_em_prims(colate_handle* h, int which, int n, const double* a, const double* b, double* y, int32_t* ok);
int colate_test_last_em(colate_handle* h, int* kernel, int* csize);
int colate_test_bin_fast(colate_handle* h, int n, const double* ages, int32_t* fast, int32_t* exact);
int colate_test_bin_sweep(colate_handle* h, uint32_t lo_bits, uint32_t hi_bits, uint64_t* out3);
int colate_test_replay(colate_handle* h, int n_blocks, const int64_t* blk_rank_start, int64_t n_rows, const uint8_t* counts,
                       const double* age_begin, const double* w_shared, const double* w_notshared, const uint8_t* emp_bin,
                       const double* emp_ws, const double* emp_wn, double* out_f, int64_t* out_n, int* out_of_range);
int colate_test_replay_row(colate_handle* h, int which, int n, const double* acc, const double* w, const int32_t* c, double* out);
int colate_test_mt_stream(colate_handle* h, const uint32_t* mt_state, int64_t word0, int64_t n_words,
                          int log2_chunk_sites, uint32_t* out);
int colate_test_mt_stream_tiled(colate_handle* h, const uint32_t* mt_state, int64_t word0, int64_t n_words, int log2_chunk_sites,
                                int64_t p0, int64_t n_phys, uint32_t* out_phys, uint32_t* out_after);
int colate_test_last_gen(colate_handle* h, int* kernel);
}
