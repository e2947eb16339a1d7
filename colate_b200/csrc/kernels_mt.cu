// The reference's std::mt19937 stream (coal.cpp:3157-3162, consumed at coal.cpp:2262, 2282)
// generated on the device, bit for bit, in parallel.
//
// The stream is cut into chunks of S = 200 * 2^k words (2^k used rows).  The 624-word state
// window in front of every chunk is reached by jump-ahead: x[J+j] = XOR_{i: g_i=1} x[i+j] with
// g = t^J mod p(t), p the characteristic polynomial of MT19937 (host_mt.cpp).  Chunk windows
// are filled by a binary tree of jumps (chunk d from chunk d - lowbit(d)), so only the
// polynomials t^(S*2^l) are needed; each chunk is then generated sequentially by one CTA
// (the recurrence exposes 227-wide parallelism per step) and written tempered to HBM.
#include "device.cuh"

#include <cuda.h>
#include <cudaTypedefs.h>

#include <cstring>
#include <map>
#include <mutex>

namespace colate {

constexpr int MT_N = 624;
constexpr int XLEN = 19937 + MT_N;       // base sequence needed by one jump
#ifndef JUMP_THREADS_
#define JUMP_THREADS_ 640
#endif
constexpr int JUMP_THREADS = JUMP_THREADS_;
#ifndef JUMP_COEF_US_
#define JUMP_COEF_US_ 35.0
#endif
constexpr double JUMP_COEF_US = JUMP_COEF_US_, JUMP_BASE_US = 10.0;   // measured on B200: coefficient work and base sequence of one jump on one SM

__device__ __forceinline__ uint32_t mt_mix_dev(uint32_t a, uint32_t b, uint32_t c)
{
  // five instructions instead of seven: the upper-bit / lower-bits merge as ONE bit-select LOP3 (two masks would need two),
  // the conditional constant as a multiply by the low bit
  uint32_t y;
  asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(y) : "r"(a), "r"(b), "r"(0x80000000u));   // (a & m) | (b & ~m)
  return c ^ (y >> 1) ^ ((b & 1u) * 0x9908b0dfu);
}

__device__ __forceinline__ uint32_t mt_temper_dev(uint32_t z)
{
  z ^= (z >> 11);
  z ^= (z << 7) & 0x9d2c5680u;
  z ^= (z << 15) & 0xefc60000u;
  z ^= (z >> 18);
  return z;
}

// windows[d] <- jump(windows[src]).  Binary level (radix 2): d = (2*j+1) << level, src = d - (1<<level).  Radix-4 level:
// d = (4*j + r) << level for r = 1, 2, 3 from src = (4*j) << level, with the polynomials t^(r * S * 2^level) (g0, g1, g2):
// two bits of the chunk index per launch, so the latency-bound top of the tree (a handful of jumps per level) is half
// as deep.  j / r from blockIdx.x / P;  level < 0: single jump windows[aux_dst] <- jump(windows[aux_src]).
//
// The jump itself: out[j] = XOR over the set coefficients i of g of X[i + j], X the base sequence from the source window.
// The polynomial is walked in blocks of 32 coefficients.  A lane owns JO = 20 consecutive outputs and loads the 51 words
// X[32 blk + 20 lane .. + 51) of a block ONCE (13 conflict-free LDS.128: the lane stride of 5 x 16 B visits all 8 bank
// groups); every set coefficient of the block is then 20 register XORs behind a warp-uniform branch.  One warp covers all
// 624 outputs (lane 31: 4), the CTA's 20 warps take every 20th block and meet in shared-memory atomics.  Shared-memory
// traffic per jump: 4 MB against 25 MB for one LDS.32 per (coefficient, output) -- the first version, which ran at the
// shared-memory bandwidth of its SM (~130 us per jump) -- and the tap lists (20 KB per polynomial) are gone: the
// coefficients travel as the 624-word bit mask.
// A jump may be split over P CTAs (P = 1, 2, 4, 8): CTA p takes the p-th part of the coefficient blocks and every CTA
// regenerates the base sequence; the partial results meet in global atomics on the destination window, which the host
// zeroes beforehand (every window of the tree is the destination of exactly one jump).  level < 0 runs with P = 1.
constexpr int JO = 20;                      // outputs per lane
constexpr int JW = 32 + JO - 1;             // words of X a lane needs for one block of 32 coefficients
constexpr int JBLK = (19937 + 31) / 32;     // 624 coefficient blocks
constexpr int XPAD = 32 * (JBLK - 1) + JO * 31 + ((JW + 3) & ~3);   // lane 31's window of the last block ends here (its outputs 624.. are discarded)
__global__ void __launch_bounds__(JUMP_THREADS, JUMP_THREADS <= 512 ? 2 : 1)
k_jump(uint32_t* __restrict__ windows, const uint32_t* __restrict__ g0, const uint32_t* __restrict__ g1, const uint32_t* __restrict__ g2,
       int level, int n_chunks, int P, int radix, int aux_src, int aux_dst)
{
  extern __shared__ __align__(16) uint32_t sm[];
  uint32_t* X = sm;                                   // XPAD words
  uint32_t* G = sm + XPAD;                            // the polynomial's 624 coefficient words
  uint32_t* out = G + MT_N;                           // 624 result words
  const int tid = threadIdx.x;
  const int jr = blockIdx.x / P, p = blockIdx.x % P;
  int d, src;
  const uint32_t* g = g0;
  if (level < 0) { d = aux_dst; src = aux_src; }
  else if (radix == 2) {
    d = (2 * jr + 1) << level;
    if (d >= n_chunks) return;
    src = d - (1 << level);
  } else {
    const int j = jr / 3, r = jr - 3 * j + 1;
    d = (4 * j + r) << level;
    if (d >= n_chunks) return;
    src = (4 * j) << level;
    if (r == 2) g = g1;
    if (r == 3) g = g2;
  }
  for (int i = tid; i < MT_N; i += blockDim.x) { X[i] = windows[(size_t)src * MT_N + i]; G[i] = g[i]; out[i] = 0; }
  for (int i = XLEN + tid; i < XPAD; i += blockDim.x) X[i] = 0;
  __syncthreads();
  // base sequence: 624 words per block barrier (a thread's second and third word of a round depend on its own first and second
  // one; the last word of a round needs the round's first word, which its thread recomputes: see k_gen)
  for (int base = MT_N; base < XLEN; base += MT_N) {
    if (tid < 227) {
      const int n0 = base + tid;
      uint32_t v0 = 0, v1 = 0;
      if (n0 < XLEN) { v0 = mt_mix_dev(X[n0 - 624], X[n0 - 623], X[n0 - 227]); X[n0] = v0; }
      const int n1 = n0 + 227;
      if (n1 < XLEN) { v1 = mt_mix_dev(X[n1 - 624], X[n1 - 623], v0); X[n1] = v1; }
      const int n2 = n0 + 454;
      if (tid < 170 && n2 < XLEN) {
        const uint32_t b = (tid == 169) ? mt_mix_dev(X[base - 624], X[base - 623], X[base - 227]) : X[n2 - 623];
        X[n2] = mt_mix_dev(X[n2 - 624], b, v1);
      }
    }
    __syncthreads();
  }
  const int warp = tid >> 5, lane = tid & 31;
  constexpr int NWARP = JUMP_THREADS / 32;
  const int b0 = (JBLK * p) / P, b1 = (JBLK * (p + 1)) / P;     // this CTA's coefficient blocks
  uint32_t acc[JO];
#pragma unroll
  for (int o = 0; o < JO; o++) acc[o] = 0;
#pragma unroll 1
  for (int blk = b0 + warp; blk < b1; blk += NWARP) {
    const uint32_t m = G[blk];                                   // the same word in every lane
    if (m == 0) continue;
    uint32_t r[(JW + 3) & ~3];
    const uint4* xs = (const uint4*)(X + 32 * blk + JO * lane);
#pragma unroll
    for (int i = 0; i < (JW + 3) / 4; i++) {
      const uint4 v = xs[i];
      r[4 * i] = v.x; r[4 * i + 1] = v.y; r[4 * i + 2] = v.z; r[4 * i + 3] = v.w;
    }
    // two coefficients per (warp-uniform) branch: a set pair is ONE three-input XOR per output
#pragma unroll
    for (int b = 0; b < 32; b += 2) {
      const uint32_t two = (m >> b) & 3u;
      if (two == 3u) {
#pragma unroll
        for (int o = 0; o < JO; o++) acc[o] ^= r[b + o] ^ r[b + 1 + o];
      } else if (two == 1u) {
#pragma unroll
        for (int o = 0; o < JO; o++) acc[o] ^= r[b + o];
      } else if (two == 2u) {
#pragma unroll
        for (int o = 0; o < JO; o++) acc[o] ^= r[b + 1 + o];
      }
    }
  }
#pragma unroll
  for (int o = 0; o < JO; o++)
    if (JO * lane + o < MT_N) atomicXor(&out[JO * lane + o], acc[o]);
  __syncthreads();
  for (int i = tid; i < MT_N; i += blockDim.x) {
    if (P == 1) windows[(size_t)d * MT_N + i] = out[i];
    else atomicXor(&windows[(size_t)d * MT_N + i], out[i]);
  }
}

// chunk c: sequential generation from its window, tempered words to the stream.  TILED: from word tile_off
// on, the words go where k_sample reads them (internal.h: stream_phys: tiles of 32 rows, a tile's chunk of
// SAMPLE_CHUNK_WORDS words per row stored as one contiguous block); each thread keeps (row, word in row) of its
// three words of a round relative to tile_off and steps them by 624 = 3 rows + 24 words per round, so the
// loop has no division and no 64-bit compare.  The CTA that produces the last word also leaves the last
// min(total, 624) words linearly in `tail` (from the two windows it holds) for the state recovery.
// PRE: the chunk range starts before tile_off (a sharded job whose first row does not sit on a chunk boundary): words in
// front of tile_off stay linear.  W32: the whole buffer is below 2^31 words, addresses as 32-bit word offsets.  (The
// address arithmetic was 14 of the 37 instructions of a step; without the linear fallback and in 32 bits it is 8.)
template <bool TILED, bool PRE, bool W32>
__global__ void __launch_bounds__(256)
k_gen(const uint32_t* __restrict__ windows, int64_t chunk_words, int64_t total_words, uint32_t* __restrict__ stream,
      int64_t tile_off, uint32_t* __restrict__ tail)
{
  __shared__ uint32_t bufA[MT_N + 1], bufB[MT_N + 1];
  const int tid = threadIdx.x;
  const int64_t start = (int64_t)blockIdx.x * chunk_words;
  if (start >= total_words) return;
  const int64_t end = min(start + chunk_words, total_words);
  for (int i = tid; i < MT_N; i += blockDim.x) bufA[i] = windows[(size_t)blockIdx.x * MT_N + i];
  __syncthreads();
  uint32_t* cur = bufA;
  uint32_t* nxt = bufB;
  int prow[3], pw[3];                                          // rows stay far below 2^31 (800 B of stream each)
  if (TILED) {
#pragma unroll
    for (int j = 0; j < 3; j++) {
      const int64_t q = start + tid + 227 * j - tile_off;
      int64_t r = q / 200;
      if (q - r * 200 < 0) r--;                                // floor: words before tile_off have row < 0 and stay linear
      prow[j] = (int)r;
      pw[j] = (int)(q - r * 200);
    }
  }
  uint32_t* const tiled_base = stream + tile_off;
  // where word k = tid + 227 j of the round at `lin` goes
  auto place = [&](int j, uint32_t* lin) -> uint32_t* {
    if (!TILED) return lin;
    const int c = (pw[j] * 3277) >> 16;                        // pw / 20 for pw < 200
    const int inner = (prow[j] & 31) * SAMPLE_CHUNK_WORDS + (c / (SAMPLE_CHUNK_WORDS / 20)) * (31 * SAMPLE_CHUNK_WORDS) + pw[j];
    uint32_t* t;
    if (W32) t = tiled_base + (uint32_t)((prow[j] >> 5) * SAMPLE_TILE_WORDS + inner);
    else t = tiled_base + ((int64_t)(prow[j] >> 5) * SAMPLE_TILE_WORDS + inner);
    if (!PRE) return t;
    return prow[j] >= 0 ? t : lin;
  };
  auto advance = [&]() {
    if (!TILED) return;
#pragma unroll
    for (int j = 0; j < 3; j++) {
      pw[j] += MT_N - 600;
      prow[j] += 3;
      if (pw[j] >= 200) { pw[j] -= 200; prow[j]++; }
    }
  };
  // one round = the next 624 words; `rem` masks the stores of the chunk's last round.  Thread tid makes words tid, tid + 227 and
  // tid + 454: the second needs the first and the third the second (x[n] = f(x[n-624], x[n-623], x[n-227])), i.e. the thread's
  // own values, and everything else comes from the previous round's window -- except word 623, whose x[n-623] is the new word 0:
  // its thread recomputes that one word.  So a round needs ONE block barrier (before the windows swap), not one per step.
  auto round = [&](int64_t o, int rem) {
    uint32_t* out = stream + o;
    if (tid < 227) {
      const uint32_t v0 = mt_mix_dev(cur[tid], cur[tid + 1], cur[tid + 397]);
      nxt[tid] = v0;
      if (tid < rem) *place(0, out + tid) = mt_temper_dev(v0);
      const int k = tid + 227;
      const uint32_t v1 = mt_mix_dev(cur[k], cur[k + 1], v0);
      nxt[k] = v1;
      if (k < rem) *place(1, out + k) = mt_temper_dev(v1);
      if (tid < 170) {
        const int k2 = tid + 454;
        const uint32_t b = (k2 == 623) ? mt_mix_dev(cur[0], cur[1], cur[397]) : cur[k2 + 1];
        const uint32_t v2 = mt_mix_dev(cur[k2], b, v1);
        nxt[k2] = v2;
        if (k2 < rem) *place(2, out + k2) = mt_temper_dev(v2);
      }
    }
    __syncthreads();
    uint32_t* t = cur; cur = nxt; nxt = t;
  };
  int64_t o = start;
  for (; o + MT_N <= end; o += MT_N) { round(o, MT_N); advance(); }
  if (o < end) { round(o, (int)(end - o)); o += MT_N; }
  if (end == total_words) {
    // cur = untempered words [o - 624, o), nxt = the 624 before them (the chunk's start window if only one round ran)
    const int n_tail = (int)min(total_words, (int64_t)MT_N);
    for (int i = tid; i < n_tail; i += blockDim.x) {
      const int64_t g = total_words - n_tail + i;               // >= o - 1248 because o - 624 < total_words
      const int rel = (int)(g - (o - 2 * MT_N));
      tail[i] = mt_temper_dev(rel >= MT_N ? cur[rel - MT_N] : nxt[rel]);
    }
  }
}

// k_gen for the common case (tile order from the first word on).  The address arithmetic of the scatter was a third of
// k_gen's instructions (49 per word, 11 + 5 of them the place() / advance() above: every thread works out where each of its
// three words of a round goes).  Here the tempered words go to a ring in shared memory in GENERATOR order and the TMA unit
// does the permutation: the tile order [tile][chunk c][row r][20 words] is described to it as a 4-d tensor with the dimensions
// in the order (word 20, chunk 10, row 32, tile) -- strides 4 B, 2560 B, 80 B, 25600 B -- so that a box of 20 x 10 x 4 x 1 is, on
// the shared-memory side, 4 consecutive rows of the stream exactly as the generator emits them (800 contiguous words), and on
// the global side their 40 pieces of 80 B.  A ninth warp that takes no part in the recurrence issues one tensor store per
// finished group of 4 rows (cp.async.bulk.tensor.4d shared -> global, under the next round's recurrence); the ring holds 5
// groups and the copy warp lets only the two latest rounds' stores be in flight before it joins the next barrier.
// (Measured before this: one plain bulk copy per 80-byte piece, 33 per round -- 2.0 ms, the copy engine pays per operation.)
// Chunks are whole multiples of 4 rows (2^k rows, k >= 2); the very last group of the stream may carry up to 3 rows of
// whatever the ring held beyond the last word: they land inside the last tile, which the buffer always holds whole and
// whose rows past n_used k_sample does not count.
constexpr int GEN_GROUP_WORDS = 800;                 // 4 rows
constexpr int GEN_RING = 5 * GEN_GROUP_WORDS;
__global__ void __launch_bounds__(288)
k_gen_tma(const uint32_t* __restrict__ windows, int64_t chunk_words, int64_t total_words, const __grid_constant__ CUtensorMap tmap,
          uint32_t* __restrict__ tail)
{
  static_assert(SAMPLE_CHUNK_WORDS == 20, "the tensor map describes 20-word chunks");
  __shared__ uint32_t bufA[MT_N + 1], bufB[MT_N + 1];
  __shared__ __align__(128) uint32_t ring[GEN_RING];
  const int tid = threadIdx.x;
  const int64_t start = (int64_t)blockIdx.x * chunk_words;
  if (start >= total_words) return;
  const int64_t end = min(start + chunk_words, total_words);
  for (int i = tid; i < MT_N; i += blockDim.x) bufA[i] = windows[(size_t)blockIdx.x * MT_N + i];
  for (int i = tid; i < GEN_RING; i += blockDim.x) ring[i] = 0;   // (the stream's last group may reach past its last word: defined bytes)
  __syncthreads();
  uint32_t* cur = bufA;
  uint32_t* nxt = bufB;
  int p0 = tid, p1 = tid + 227, p2 = tid + 454;      // ring positions of this thread's three words of the round
  const int row_base = (int)(start / 200);           // rows stay far below 2^31 (800 B of stream each); a multiple of 4
  int groups_issued = 0;
  int64_t o = start;
  for (; o < end; o += MT_N) {
    if (tid < 227) {
      // (see k_gen: a thread's three words of a round depend on its own, word 623's neighbour is recomputed: one barrier per round)
      const uint32_t v0 = mt_mix_dev(cur[tid], cur[tid + 1], cur[tid + 397]);
      nxt[tid] = v0;
      ring[p0] = mt_temper_dev(v0);
      const int k = tid + 227;
      const uint32_t v1 = mt_mix_dev(cur[k], cur[k + 1], v0);
      nxt[k] = v1;
      ring[p1] = mt_temper_dev(v1);
      if (tid < 170) {
        const int k2 = tid + 454;
        const uint32_t b = (k2 == 623) ? mt_mix_dev(cur[0], cur[1], cur[397]) : cur[k2 + 1];
        const uint32_t v2 = mt_mix_dev(cur[k2], b, v1);
        nxt[k2] = v2;
        ring[p2] = mt_temper_dev(v2);
      }
      p0 += MT_N; p1 += MT_N; p2 += MT_N;
      if (p0 >= GEN_RING) p0 -= GEN_RING;
      if (p1 >= GEN_RING) p1 -= GEN_RING;
      if (p2 >= GEN_RING) p2 -= GEN_RING;
    }
    __syncthreads();
    if (tid >= 256) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the other warps' generic writes of this round before the async reads
      const int64_t done = min(o + MT_N, end) - start;               // words of the chunk that are in the ring (or have left it)
      const int g_now = (int)(o + MT_N >= end ? (done + GEN_GROUP_WORDS - 1) / GEN_GROUP_WORDS : done / GEN_GROUP_WORDS);
      for (int g = groups_issued + (tid - 256); g < g_now; g += 32) {
        const int row = row_base + 4 * g;
        const uint32_t src = (uint32_t)__cvta_generic_to_shared(ring + (g % 5) * GEN_GROUP_WORDS);
        asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%1, %2, %3, %4}], [%5];" ::"l"(&tmap), "r"(0), "r"(0),
                     "r"(row & 31), "r"(row >> 5), "r"(src)
                     : "memory");
      }
      groups_issued = g_now;
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory");   // a group's place in the ring is written again 3.8 rounds after it left
    }
    uint32_t* t = cur; cur = nxt; nxt = t;
  }
  if (tid >= 256) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  if (end == total_words) {
    // cur = untempered words [o - 624, o), nxt = the 624 before them (the chunk's start window if only one round ran)
    const int n_tail = (int)min(total_words, (int64_t)MT_N);
    for (int i = tid; i < n_tail; i += blockDim.x) {
      const int64_t g = total_words - n_tail + i;               // >= o - 1248 because o - 624 < total_words
      const int rel = (int)(g - (o - 2 * MT_N));
      tail[i] = mt_temper_dev(rel >= MT_N ? cur[rel - MT_N] : nxt[rel]);
    }
  }
}

// the tile-ordered stream as the 4-d tensor k_gen_tma stores through (driver entry point fetched once; false: not available)
static bool encode_stream_map(uint32_t* base, int64_t total_words, CUtensorMap* out)
{
  static PFN_cuTensorMapEncodeTiled_v12000 enc = [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) fn = nullptr;
    return (PFN_cuTensorMapEncodeTiled_v12000)fn;
  }();
  if (!enc) return false;
  const cuuint64_t tiles = (cuuint64_t)((total_words + SAMPLE_TILE_WORDS - 1) / SAMPLE_TILE_WORDS);
  const cuuint64_t dims[4] = {20, 10, 32, tiles};
  const cuuint64_t strides[3] = {20 * 32 * 4, 20 * 4, (cuuint64_t)SAMPLE_TILE_WORDS * 4};
  const cuuint32_t box[4] = {20, 10, 4, 1}, estr[4] = {1, 1, 1, 1};
  return enc(out, CU_TENSOR_MAP_DATA_TYPE_UINT32, 4, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
             CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// the n words before logical position `from + n` of a tile-ordered stream, linearly (state recovery when the stream in
// HBM is longer than the caller's request: stream cache)
__global__ void k_tail_gather(const uint32_t* __restrict__ stream, int64_t tile_off, int64_t from, int n, uint32_t* __restrict__ tail)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) tail[i] = stream[stream_phys(from + i, tile_off)];
}

// ---- coefficient masks per polynomial, cached per device ---------------------------------------
static std::mutex g_mu;
static std::map<std::pair<int, int>, uint32_t*> g_polys;  // (device, q or 1000 + q for the 3x polynomial) -> 624 words on the device

static int get_poly(int device, int q, cudaStream_t s, const uint32_t** out, bool triple = false)
{
  std::lock_guard<std::mutex> lk(g_mu);
  const int key = triple ? 1000 + q : q;
  auto it = g_polys.find({device, key});
  if (it != g_polys.end()) { *out = it->second; return 0; }
  const uint32_t* g = triple ? jump_poly3(q) : jump_poly(q);
  if (!g) return fail(COLATE_ERR_ARG, "jump polynomial unavailable");
  uint32_t host[MT_N];
  memcpy(host, g, sizeof host);
  host[MT_N - 1] &= 1u;                                      // degree < 19937 = 623 * 32 + 1
  uint32_t* dev = nullptr;
  CK(cudaMalloc(&dev, sizeof host));
  CK(cudaMemcpyAsync(dev, host, sizeof host, cudaMemcpyHostToDevice, s));
  CK(cudaStreamSynchronize(s));  // host[] is a local
  g_polys[{device, key}] = dev;
  *out = dev;
  return 0;
}

static int launch_jump(colate_handle* h, int q, int level, int n_chunks, int n_jumps, int aux_src, int aux_dst, int radix = 2)
{
  const uint32_t *g0, *g1, *g2;
  int rc = get_poly(h->device, q, h->stream, &g0);
  if (rc) return rc;
  g1 = g0; g2 = g0;
  if (radix == 4) {
    if ((rc = get_poly(h->device, q + 1, h->stream, &g1))) return rc;
    if ((rc = get_poly(h->device, q, h->stream, &g2, true))) return rc;
  }
  // Split factor: one CTA per SM (the base sequence alone takes 82 KB of shared memory), so a launch runs in
  // ceil(n_jumps * P / SMs) waves of (coefficient work / P + the base sequence every CTA regenerates): take the cheapest
  int P = 1;
  if (level >= 0) {
    double best = 1e30;
    for (int cand = 1; cand <= 8; cand *= 2) {
      const double waves = (double)((n_jumps * cand + h->sm_count - 1) / h->sm_count);
      const double cost = waves * (JUMP_COEF_US / cand + JUMP_BASE_US);
      if (cost < best) { best = cost; P = cand; }
    }
    if (const char* e = getenv("COLATE_JUMP_SPLIT")) P = std::max(1, std::min(8, atoi(e)));
  }
  const size_t smem = (size_t)(XPAD + 2 * MT_N) * 4;
  CK(cudaFuncSetAttribute(k_jump, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_jump<<<n_jumps * P, JUMP_THREADS, smem, h->stream>>>(h->windows.as<uint32_t>(), g0, g1, g2, level, n_chunks, P, radix, aux_src, aux_dst);
  h->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

// Generates engine words [word0, word0+n_words) of the stream that starts at state window
// `mt_state`.  *stream_at_word0 points at word0 inside the handle's stream buffer (16-byte
// aligned when word0 is a multiple of 4).  window_after (host, optional) = state window after
// word0+n_words outputs.
int run_mt_stream(colate_handle* h, const uint32_t* mt_state, int64_t word0, int64_t n_words, int k,
                  uint32_t** stream_at_word0, uint32_t* window_after, bool tiled)
{
  if (k < 0 || k > 40) return fail(COLATE_ERR_ARG, "bad chunk size");
  // Stream cache (colate_set_stream_cache; all-pairs jobs reseed every pair with the same --seed): the words
  // from `word0` on depend only on the generator state, so a tile-ordered stream left by an earlier call with the
  // same state and offset serves every request that is not longer.  The state after THIS request's last word is
  // then gathered from the stream (mt_window_after).
  if (tiled && h->stream_cache_on && h->sc_valid && word0 == h->sc_word0 && n_words <= h->sc_nwords &&
      memcmp(mt_state, h->sc_state, sizeof h->sc_state) == 0) {
    *stream_at_word0 = h->rng_stream.as<uint32_t>() + h->sc_off;
    h->mt_total_local = h->sc_off + n_words;
    h->mt_tail_gather = true;
    if (window_after) return mt_window_after(h, window_after);
    return 0;
  }
  h->sc_valid = false;
  const int64_t n_req = n_words;
  if (tiled && h->stream_cache_on) n_words += n_words / 8 + SAMPLE_TILE_WORDS;   // headroom: the next pairs use a few more rows
  const int64_t S = (int64_t)200 << k;
  const int64_t c0 = word0 / S;
  const int64_t last = n_words > 0 ? word0 + n_words - 1 : word0;
  const int64_t M64 = last / S - c0 + 1;
  if (M64 > (1 << 24)) return fail(COLATE_ERR_ARG, "too many generator chunks");
  const int M = (int)M64;
  const int64_t total_local = word0 + n_words - c0 * S;  // words from the start of chunk c0
  cudaStream_t s = h->stream;
  CK(h->windows.ensure((size_t)(M + 1) * MT_N * 4));  // + one scratch window for the offset jumps
  const int64_t off = word0 - c0 * S;                    // the caller's first word inside chunk c0
  CK(h->rng_stream.ensure((size_t)(std::max<int64_t>(total_local, 4) + (tiled ? SAMPLE_TILE_WORDS : 0)) * 4 + 64));   // tiled: whole last tile
  CK(h->mt_tail.ensure(MT_N * 4));
  CK(cudaMemcpyAsync(h->windows.p, mt_state, MT_N * 4, cudaMemcpyHostToDevice, s));
  if (M > 1) CK(cudaMemsetAsync(h->windows.as<uint32_t>() + MT_N, 0, (size_t)(M - 1) * MT_N * 4, s));   // split jumps meet in atomics on their destination
  // reach chunk c0: one jump per set bit of c0, ping-ponging between window 0 and the scratch window
  int cur = 0;
  for (int b = 62; b >= 0; b--) {
    if (!((c0 >> b) & 1)) continue;
    if (k + b > 48) return fail(COLATE_ERR_ARG, "generator offset too large");
    const int nxt = cur == 0 ? M : 0;
    int rc = launch_jump(h, k + b, -1, 1, 1, cur, nxt);
    if (rc) return rc;
    cur = nxt;
  }
  if (cur != 0)
    CK(cudaMemcpyAsync(h->windows.p, h->windows.as<uint32_t>() + (size_t)M * MT_N, MT_N * 4, cudaMemcpyDeviceToDevice, s));
  // tree over the chunks of this call
  int K = 0;
  while ((1 << K) < M) K++;
  int l = K - 1;
  if (K & 1) {                                              // an odd number of index bits: the top one on its own
    if (M > (1 << l)) {
      int n_jumps = (M - (1 << l) + (2 << l) - 1) / (2 << l);
      int rc = launch_jump(h, k + l, l, M, n_jumps, 0, 0);
      if (rc) return rc;
    }
    l--;
  }
  for (l -= 1; l >= 0; l -= 2) {                            // then two bits per level: sources at multiples of 4 << l
    const int n_src = (M + (4 << l) - 1) / (4 << l);
    int rc = launch_jump(h, k + l, l, M, 3 * n_src, 0, 0, 4);
    if (rc) return rc;
  }
  if (total_local > 0) {
    if (tiled && off % 200 != 0) return fail(COLATE_ERR_ARG, "tiled generator stream must start at a row boundary");
    // gen_w64 / gen_path (colate_set_option): 64-bit addressing at any size; k_gen only, or TMA wherever it applies
    // whatever COLATE_GEN_NO_TMA says (the variable is read once per process, the options per handle)
    const bool w32 = !h->opt_gen_w64 && total_local + SAMPLE_TILE_WORDS < ((int64_t)1 << 31);
    uint32_t* win = h->windows.as<uint32_t>();
    uint32_t* st = h->rng_stream.as<uint32_t>();
    uint32_t* tl = h->mt_tail.as<uint32_t>();
    if (!tiled) { k_gen<false, false, false><<<M, 256, 0, s>>>(win, S, total_local, st, 0, tl); h->gen_kernel = GEN_LINEAR; }
    else if (off == 0) {
      CUtensorMap tm;
      static const bool no_tma_env = getenv("COLATE_GEN_NO_TMA") != nullptr;
      const bool no_tma = h->opt_gen_path == 1 || (h->opt_gen_path == 0 && no_tma_env);
      if (k >= 2 && !no_tma && encode_stream_map(st, total_local, &tm)) {
        k_gen_tma<<<M, 288, 0, s>>>(win, S, total_local, tm, tl);
        h->gen_kernel = GEN_TMA;
      } else if (w32) { k_gen<true, false, true><<<M, 256, 0, s>>>(win, S, total_local, st, off, tl); h->gen_kernel = GEN_TILED_W32; }
      else { k_gen<true, false, false><<<M, 256, 0, s>>>(win, S, total_local, st, off, tl); h->gen_kernel = GEN_TILED_W64; }
    }
    else if (w32) { k_gen<true, true, true><<<M, 256, 0, s>>>(win, S, total_local, st, off, tl); h->gen_kernel = GEN_PRE_W32; }
    else { k_gen<true, true, false><<<M, 256, 0, s>>>(win, S, total_local, st, off, tl); h->gen_kernel = GEN_PRE_W64; }
    h->launches += 1;
    CK(cudaGetLastError());
  }
  *stream_at_word0 = h->rng_stream.as<uint32_t>() + off;
  h->mt_total_local = off + n_req;
  h->mt_tail_gather = tiled && n_req != n_words;
  if (tiled && h->stream_cache_on) {
    memcpy(h->sc_state, mt_state, sizeof h->sc_state);
    h->sc_word0 = word0; h->sc_nwords = n_words; h->sc_off = off; h->sc_valid = true;
  }
  if (window_after) return mt_window_after(h, window_after);
  return 0;
}

// State window after the last word produced by the latest run_mt_stream() call, composed on
// the host from the chunk-0 window and the tail of the stream (kept linearly in mt_tail; tempering is invertible):
// y[i] = window(c0)[i] for i < 624, y[624+n] = untemper(stream[n]); answer = y[T .. T+624).
int mt_window_after(colate_handle* h, uint32_t* window_after)
{
  cudaStream_t s = h->stream;
  const int64_t T = h->mt_total_local;
  uint32_t w0[MT_N];
  std::vector<uint32_t> tail((size_t)std::min<int64_t>(T, MT_N));
  CK(cudaMemcpyAsync(w0, h->windows.p, MT_N * 4, cudaMemcpyDeviceToHost, s));
  if (!tail.empty()) {
    if (h->mt_tail_gather) {   // the stream in HBM runs past T: pick the words in front of T out of the tile order
      k_tail_gather<<<(int)(tail.size() + 255) / 256, 256, 0, s>>>(h->rng_stream.as<uint32_t>(), h->sc_off, T - (int64_t)tail.size(),
                                                                (int)tail.size(), h->mt_tail.as<uint32_t>());
      h->launches += 1;
      CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(tail.data(), h->mt_tail.p, tail.size() * 4, cudaMemcpyDeviceToHost, s));   // the last words, linearly (k_gen's copy or the gather)
  }
  CK(cudaStreamSynchronize(s));
  for (int j = 0; j < MT_N; j++) {
    int64_t i = T + j;  // index into y
    if (i < MT_N) window_after[j] = w0[i];
    else window_after[j] = mt_untemper(tail[(size_t)(i - MT_N - (T - (int64_t)tail.size()))]);
  }
  return 0;
}

}  // namespace colate
