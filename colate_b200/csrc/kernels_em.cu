// Stage ii (block bootstrap + F redistribution, coal.cpp:3344-3451) and stage iii (EM on the
// 185-bin age histograms: coal.cpp:3675-3827 driving coal_EM, coal_EM.cpp:5-468) kernels.
//
// Everything here is IEEE fp64 in the reference's operation order (the file is compiled with
// --fmad=false; products and sums are never contracted), exp/log/log1p are glibc's algorithms
// (glibc_math.cuh) and every sum over age bins runs in the reference's order, so both stages
// reproduce the reference bit for bit on a host whose libm selects the FMA variants.
#include <cooperative_groups.h>

#include "device.cuh"
#include "glibc_math.cuh"

#include <cstring>

namespace cg = cooperative_groups;

namespace colate {

constexpr int EM_THREADS = 416;  // 12 task warps + 1 warp for the prefix chain
constexpr int EM_TASKS = 384;  // 2 x 185 (bin, shared / not shared) padded; task = 2*bin + type

// ---- stage ii ------------------------------------------------------------------------------
// One CTA per replicate.  Block sums per bin in block order (thread = bin), then the F redistribution of
// coal.cpp:3392-3441: its two running sums (fcount, normf) are 185 dependent additions each and stay on one thread in bin
// order; the divisions and products around them are independent per bin and run one bin per thread (a serial version
// of the whole redistribution took 120 us per launch: 370 dependent fp64 divisions).
// norm_1e3: the front-ends other than tmp/tmp divide both vectors by 1e3 afterwards (coal.cpp:3453-3463, tmp_file == true).
__global__ void __launch_bounds__(256)
k_bootstrap(int num_blocks, const int32_t* __restrict__ weights, const double* __restrict__ blk,
            double age, const double* __restrict__ age_bin, double* __restrict__ counts, int norm_1e3)
{
  __shared__ double S[NBINS], N[NBINS], SE[NBINS], NE[NBINS], F[NBINS];
  __shared__ double s_fcount, s_normf;
  const int r = blockIdx.x;
  const int32_t* w = weights + (size_t)r * num_blocks;
  int bin_start = 0;
  while (bin_start < NBINS - 1 && age_bin[bin_start] <= age) bin_start++;      // coal.cpp:3394-3396
  for (int b = threadIdx.x; b < NBINS; b += blockDim.x) {
    double s = 0.0, n = 0.0, se = 0.0, ne = 0.0;
    // coal.cpp:3358-3390, block order kept.  Four blocks' values are requested before the first of them is added (the loop was a
    // chain of L2 latencies: the loads sat behind the `weight > 0` test of their own block)
    for (int j0 = 0; j0 < num_blocks; j0 += 4) {
      double bw[4], v0[4], v1[4], v2[4], v3[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int j = min(j0 + u, num_blocks - 1);
        const double* v = blk + (size_t)j * 4 * NBINS + b;
        bw[u] = j0 + u < num_blocks ? (double)w[j] : 0.0;
        v0[u] = v[0]; v1[u] = v[NBINS]; v2[u] = v[2 * NBINS]; v3[u] = v[3 * NBINS];
      }
#pragma unroll
      for (int u = 0; u < 4; u++)
        if (bw[u] > 0.0) {
          s = __dadd_rn(s, __dmul_rn(bw[u], v0[u]));
          n = __dadd_rn(n, __dmul_rn(bw[u], v1[u]));
          se = __dadd_rn(se, __dmul_rn(bw[u], v2[u]));
          ne = __dadd_rn(ne, __dmul_rn(bw[u], v3[u]));
        }
    }
    S[b] = s; N[b] = n; SE[b] = se; NE[b] = ne;
    // coal.cpp:3406-3417: F[bin] = emp share of bin, bins from bin_start on
    F[b] = (b >= bin_start && se > 0) ? __ddiv_rn(se, __dadd_rn(se, ne)) : 0.0;
  }
  __syncthreads();
  // coal.cpp:3420-3425: F[bin - 1] *= age_bin[bin] - lower_age for bin = bin_start .. 184, lower_age = age_bin[bin - 1] (the first
  // one age_bin[bin_start - 1] as well): slot k = bin - 1 is scaled by the width of the bin above it
  for (int k = threadIdx.x; k < NBINS - 1; k += blockDim.x)
    if (k >= bin_start - 1) F[k] = __dmul_rn(F[k], __dsub_rn(age_bin[k + 1], age_bin[k]));
  __syncthreads();
  if (threadIdx.x == 0) {         // the two running sums in bin order
    double fcount = 0.0;
    for (int bin = bin_start; bin < NBINS; bin++) fcount = __dadd_rn(fcount, SE[bin]);
    s_fcount = fcount;
  } else if (threadIdx.x == 32) {
    double normf = 0.0;
    for (int bin = 0; bin < NBINS; bin++) normf = __dadd_rn(normf, F[bin]);
    s_normf = normf;
  }
  __syncthreads();
  double* out = counts + (size_t)r * 2 * NBINS;
  for (int b = threadIdx.x; b < NBINS; b += blockDim.x) {
    const double f = __dmul_rn(__ddiv_rn(F[b], s_normf), s_fcount);   // coal.cpp:3435-3441
    double s = __dadd_rn(S[b], (0.0 < f) ? f : 0.0);                  // std::max(0.0, f): NaN -> 0.0
    double n = N[b];
    if (norm_1e3) { s = __ddiv_rn(s, 1e3); n = __ddiv_rn(n, 1e3); }
    out[b] = s; out[NBINS + b] = n;
  }
}

// ---- E-step pieces (coal_EM.cpp) -----------------------------------------------------------
__device__ __forceinline__ double neg_inf() { return __longlong_as_double(0xfff0000000000000ull); }
__device__ __forceinline__ bool bad(double x) { return !(fabs(x) < __longlong_as_double(0x7ff0000000000000ull)); }

// coal_EM::logsumexp, coal_EM.cpp:5-31
__device__ __noinline__ double lse_generic(double a, double b, const glm::Tables& T)
{
  if (bad(a)) return bad(b) ? neg_inf() : b;
  if (bad(b)) return a;
  const double hi = (a > b) ? a : b, lo = (a > b) ? b : a;   // same value as the two-branch form
  return hi + glm::log1p(glm::exp(lo - hi, T));
}
// The same, arranged for the sequential folds (their latency bounds an EM iteration): the common
// case -- finite operands, exp() on its main path, log1p() on its k = 0 path, i.e. terms between
// e^-20 and 0.414 of the running sum -- as straight-line code with one rare-case branch at the end.
// Same operations as the generic path takes for those operands.
__device__ __forceinline__ double lse(double a, double b, const glm::Tables& T)
{
  const double d = -fabs(a - b);                 // == lo - hi exactly (for a != b), without waiting for the select
  const double x = glm::exp_main(d, T);
  const double y = glm::log1p_k0(x);
  const double hi = (a > b) ? a : b;
  const bool ok = !bad(a) & !bad(b) & glm::exp_is_main(d) & glm::log1p_is_k0(x);
  if (ok) return hi + y;
  return lse_generic(a, b, T);
}
// The same for warps that run one fold per LANE (k_em_cta): at any step some lane's term is above 0.414 of its running
// sum (the first steps of a fold) or below e^-20 of it (the deep epochs), so a fast path that covers only the
// middle regime would send the whole warp through the generic code at almost every step.  log1p_wide() covers all
// regimes of 0 < x < 1 without a branch; what is left for lse_generic is rare for every lane at once (non-finite
// operands, equal operands, terms below e^-512 of the sum, three narrow bands of log1p).
__device__ __forceinline__ double lse_wide(double a, double b, const glm::Tables& T)
{
  const double d = -fabs(a - b);
  const double x = glm::exp_main(d, T);
  const double y = glm::log1p_wide(x);
  const double hi = (a > b) ? a : b;
  const bool ok = !bad(a) & !bad(b) & glm::exp_is_main(d) & glm::log1p_wide_ok(x);
  if (ok) return hi + y;
  return lse_generic(a, b, T);
}
// coal_EM::logminusexp, coal_EM.cpp:33-58
__device__ __noinline__ double lme_generic(double a, double b, const glm::Tables& T)
{
  if (bad(a)) return neg_inf();
  if (bad(b)) return a;
  if (a < b) return neg_inf();
  return a + glm::log1p(-glm::exp(b - a, T));
}
__device__ __forceinline__ double lme(double a, double b, const glm::Tables& T)   // straight-line common case, as lse()
{
  const double d = b - a;
  const double x = -glm::exp_main(d, T);
  const double y = glm::log1p_k0(x);
  const bool ok = !bad(a) & !bad(b) & !(a < b) & glm::exp_is_main(d) & glm::log1p_is_k0(x);
  if (ok) return a + y;
  return lme_generic(a, b, T);
}
// exp() with its main path first (one rare-case branch)
__device__ __forceinline__ double exp_fast(double x, const glm::Tables& T)
{
  const double y = glm::exp_main(x, T);
  if (glm::exp_is_main(x)) return y;
  return glm::exp(x, T);
}

struct EmCtx {
  int E;
  const double *ep, *rate, *A, *B, *Lam;
  glm::Tables T;
};

// cumulative hazard of the plain epoch grid (coal_EM.cpp:100-103); serial by construction
__device__ void em_cumhaz(int E, const double* ep, const double* rate, double* Lam)
{
  double l = 0.0;
  Lam[0] = 0.0;
  for (int i = 1; i < E; i++) { l = l + rate[i - 1] * (ep[i] - ep[i - 1]); Lam[i] = l; }
}

// coal_EM ctor -> get_AB, coal_EM.cpp:105-149, entry i
__device__ void em_AB(int E, const double* ep, const double* rate, const double* Lam, int i, double* A, double* B,
                      const glm::Tables& T)
{
  const double r = rate[i];
  if (i < E - 1) {
    const double tb = ep[i], te = ep[i + 1], inv = 1.0 / r;
    if (r > 0 && te != 0 && te - tb > 0) {
      A[i] = lme(-Lam[i], -Lam[i + 1], T);
      double b = (tb + inv) - (te + inv) * glm::exp(-Lam[i + 1] + Lam[i], T);
      B[i] = glm::log(b, T) - Lam[i];
    } else { A[i] = neg_inf(); B[i] = neg_inf(); }
  } else {
    if (r > 0) { A[i] = -Lam[i]; B[i] = glm::log(ep[i] + 1.0 / r, T) - Lam[i]; }
    else { A[i] = neg_inf(); B[i] = neg_inf(); }
  }
}

// the two halves of em_AB, for callers that need A_ep before B_ep
__device__ __forceinline__ void em_A(int E, const double* ep, const double* rate, const double* Lam, int i, double* A, const glm::Tables& T)
{
  const double r = rate[i];
  if (i < E - 1) {
    const double tb = ep[i], te = ep[i + 1];
    A[i] = (r > 0 && te != 0 && te - tb > 0) ? lme(-Lam[i], -Lam[i + 1], T) : neg_inf();
  } else A[i] = (r > 0) ? -Lam[i] : neg_inf();
}
__device__ __forceinline__ void em_B(int E, const double* ep, const double* rate, const double* Lam, int i, double* B, const glm::Tables& T)
{
  const double r = rate[i];
  if (i < E - 1) {
    const double tb = ep[i], te = ep[i + 1], inv = 1.0 / r;
    if (r > 0 && te != 0 && te - tb > 0) {
      double b = (tb + inv) - (te + inv) * glm::exp(-Lam[i + 1] + Lam[i], T);
      B[i] = glm::log(b, T) - Lam[i];
    } else B[i] = neg_inf();
  } else B[i] = (r > 0) ? glm::log(ep[i] + 1.0 / r, T) - Lam[i] : neg_inf();
}

// get_tint with age_begin == age_end (coal_EM.cpp:60-95): grid points before the copies of t
__device__ __forceinline__ int tint_k(int E, const double* ep, double t)
{
  for (int e = 0; e < E; e++) if (t < ep[e]) return e;
  return E;
}

// The epoch that contains t, EM_shared: log-domain num / denom (coal_EM.cpp:198-210)
__device__ __forceinline__ void shared_special(const EmCtx& c, double t, int et, double& num_t, double& den_t)
{
  const double r = c.rate[et];
  const double c0 = c.Lam[et];
  const double c1 = c0 + r * (t - c.ep[et]);
  if (r > 0) {
    const double inv = 1.0 / r, tb = c.ep[et];
    num_t = lme(-c0, -c1, c.T);
    den_t = glm::log((tb + inv) / inv - (t + inv) / inv * glm::exp(-c1 + c0, c.T), c.T) + glm::log(inv, c.T) - c0;
  } else { num_t = neg_inf(); den_t = neg_inf(); }
}

// EM_shared(t, t, ...) after the normaliser is known (coal_EM.cpp:263-292).  pl = state of the
// running logsumexp over A[0..et-1] (1.0 = the reference's "nothing yet" sentinel, coal_EM.cpp:254).
// emit(e, num_e, denom_e) for every epoch in order; returns the log normaliser.
template <class Emit>
__device__ double task_shared(const EmCtx& c, int et, bool active, double pl, double num_t, double den_t, Emit emit)
{
  const int E = c.E;
  double nc = 0.0;
  bool good = false;
  if (active) {
    nc = (pl == 1.0) ? num_t : lse(pl, num_t, c.T);
    good = !bad(nc);
  }
  double integ = 1.0;
  const int lim = (E - 1 < et + 1) ? E - 1 : et + 1;
  for (int e = 0; e < E; e++) {
    double ne = 0.0, de = 0.0;
    if (good) {
      if (e < lim) {
        ne = glm::exp(((e < et) ? c.A[e] : num_t) - nc, c.T);
        if (integ > 0.0) integ -= ne; else integ = 0.0;
        de = glm::exp(((e < et) ? c.B[e] : den_t) - nc, c.T);
        de += -c.ep[e] * ne + (c.ep[e + 1] - c.ep[e]) * integ;
        if (de < 0.0) de = 0.0;
      } else if (e == E - 1 && et == E - 1) {
        ne = glm::exp(num_t - nc, c.T);
        de = glm::exp(den_t - nc, c.T);
        de -= c.ep[e] * ne;
        if (de < 0.0) de = 0.0;
      }
    }
    emit(e, ne, de);
  }
  return good ? nc : 0.0;
}

// running logsumexp state after A[0..j-1] for j = 0..E (coal_EM.cpp:254-258), shared by all bins
__device__ void shared_prefix_chain(const EmCtx& c, double* PL)
{
  double nc = 1.0;
  PL[0] = nc;
  for (int e = 0; e < c.E; e++) {
    const double v = c.A[e];
    if (nc == 1.0) nc = v; else nc = lse(nc, v, c.T);
    PL[e + 1] = nc;
  }
}

// EM_notshared(t, t, ...), coal_EM.cpp:297-468 (327-357, 435-466)
template <class Emit>
__device__ double task_notshared(const EmCtx& c, double t, int k, bool active, Emit emit)
{
  const int E = c.E, et = k - 1;
  double num_t = 0, den_t = 0, nc = 0;
  bool good = false;
  if (active) {
    const double r = c.rate[et], inv = 1.0 / r;
    const double c1 = c.Lam[et] + r * (t - c.ep[et]);
    const double c2 = c1 + r * (t - t);
    if (et != E - 1) {
      const double c3 = c2 + r * (c.ep[k] - t);
      if (r > 0) {
        num_t = lme(-c2, -c3, c.T);
        den_t = glm::log((t + inv) - (c.ep[k] + inv) * glm::exp(-c3 + c2, c.T), c.T) - c2;
        nc = num_t;
      } else { num_t = neg_inf(); den_t = neg_inf(); nc = neg_inf(); }
      for (int e = et + 1; e < E; e++) nc = lse(nc, c.A[e], c.T);
    } else {
      num_t = -c2;
      den_t = glm::log(t + inv, c.T) - c2;
      nc = num_t;
    }
    good = !bad(nc);
  }
  double integ = 1.0;
  for (int e = 0; e < E; e++) {
    double ne = 0.0, de = 0.0;
    if (good) {
      if (e < et) {
        de = c.ep[e + 1] - c.ep[e];
      } else {
        const double ln = (e == et) ? num_t : c.A[e];
        const double ld = (e == et) ? den_t : c.B[e];
        ne = glm::exp(ln - nc, c.T);
        if (e < E - 1) {
          if (integ > 0.0) integ -= ne; else integ = 0.0;
          de = glm::exp(ld - nc, c.T);
          de += -c.ep[e] * ne + (c.ep[e + 1] - c.ep[e]) * integ;
        } else {
          de = glm::exp(ld - nc, c.T);
          de -= c.ep[e] * ne;
        }
        if (de < 0.0) de = 0.0;
      }
    }
    emit(e, ne, de);
  }
  return good ? nc : 0.0;
}

// ---- stage iii: EM to convergence, throughput mode --------------------------------------------
// One CTA per bootstrap replicate, 2 CTAs per SM (used when there are enough replicates to fill the
// GPU; small portable clusters of 2 / 4 CTAs per replicate in between).  Few replicates run on
// k_em_split below.  Per iteration:
//   A  cumulative hazard (every thread sums the per-epoch products in order), A_ep / B_ep
//   B  the sequential logsumexp folds: one prefix chain for all "shared" tasks (its own warp,
//      published entry by entry), one suffix chain per bin for the "not shared" tasks; shared tasks
//      start as soon as their prefix is ready
//   C  per (bin, type) task: posterior mass / exposure per epoch -> scratch M[task][column]
//      (tasks are dealt round-robin to the CTAs of the cluster)
//   D  (cluster barrier;) the CTA sums its columns of M over the tasks IN THE REFERENCE'S ORDER
//      (coal.cpp:3704-3733; chunks staged through shared memory), totals reach every CTA through
//      DSMEM, and the M-step runs redundantly.
constexpr int EM_STAGE_DOUBLES = 3328;  // per staging buffer of the column sums (26 KB)

__global__ void __launch_bounds__(EM_THREADS, 2)
k_em(int E, const double* __restrict__ epochs, const double* __restrict__ rates_init,
     const double* __restrict__ age_bin_g, const double* __restrict__ counts, int max_iter,
     const uint64_t* __restrict__ exp_tab_g, const uint64_t* __restrict__ log_tab_g, double* scratch,
     double* __restrict__ rates_out, int32_t* __restrict__ iters_out, double* __restrict__ ll_out, long long* prof_g)
{
  cg::cluster_group cluster = cg::this_cluster();
  const int crank = (int)cluster.block_rank(), csize = (int)cluster.num_blocks();
  const int rep = blockIdx.x / csize;

  extern __shared__ double sm[];
  double* ep = sm;                  // [E]
  double* rate = ep + E;            // [E]
  double* Lam = rate + E;           // [E]
  double* A = Lam + E;              // [E]
  double* B = A + E;                // [E]
  double* PL = B + E;               // [E+1]
  double* tn = PL + E + 1;          // [E]
  double* td = tn + E;              // [E]
  double* cand = td + E;            // [E]
  double* prod = cand + E;          // [E]
  double* stage = prod + E;         // [2][EM_STAGE_DOUBLES]
  uint64_t* etab = (uint64_t*)(stage + 2 * EM_STAGE_DOUBLES);  // [256]
  uint64_t* ltab = etab + 256;                                  // [256]
  __shared__ int stop_flag;
  __shared__ volatile int pl_ready;
  __shared__ double ll_s, prev_s, ll_new;

  const int tid = threadIdx.x;
  for (int e = tid; e < E; e += blockDim.x) { ep[e] = epochs[e]; rate[e] = rates_init[e]; }
  for (int i = tid; i < 256; i += blockDim.x) { etab[i] = exp_tab_g[i]; ltab[i] = log_tab_g[i]; }
  if (tid == 0) { stop_flag = 0; ll_s = neg_inf(); pl_ready = 0; PL[0] = 1.0; }
  // threads 0..191: shared task of bin tid; 192..383: not-shared task of bin tid-192;
  // warp 12: the prefix chain.  Row of a task in M (= the reference's summation order): 2*bin + type.
  const bool is_shared = tid < 192;
  const int bin = is_shared ? tid : tid - 192;
  const bool is_task = tid < 384 && bin < NBINS;
  const int task = 2 * bin + (is_shared ? 0 : 1);
  double t = 0.0, cnt = 0.0;
  if (is_task) {
    t = age_bin_g[bin];
    cnt = counts[(size_t)rep * 2 * NBINS + (is_shared ? 0 : NBINS) + bin];
  }
  const bool active = is_task && cnt > 0;  // coal.cpp:3706, 3719
  __syncthreads();
  const int k = is_task ? tint_k(E, ep, t) : 1;
  const int et = k - 1;
  const bool mine = active && ((task % csize) == crank);  // tasks dealt round-robin over the cluster
  EmCtx c{E, ep, rate, A, B, Lam, glm::Tables{etab, ltab}};
  // scratch of this replicate: [buf][task][RS], row = {count*num[e] (E), count*denom[e] (E), count*logl}
  const int RS = 2 * E + 2;
  const int TJ = max(1, EM_STAGE_DOUBLES / RS);  // tasks per staged chunk
  double* Mrep = scratch + (size_t)rep * 2 * EM_TASKS * RS;
  long long* prof = prof_g ? prof_g + (size_t)blockIdx.x * 8 : nullptr;
  long long tp[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (is_task && !active)  // rows of inactive tasks stay 0: x + 0.0 == x, so the sums need no test
    for (int b2 = 0; b2 < 2; b2++)
      for (int e = 0; e < RS; e++) Mrep[((size_t)b2 * EM_TASKS + task) * RS + e] = 0.0;

  int iter = 0;
  for (; iter < max_iter; iter++) {
    double* M = Mrep + (size_t)(iter & 1) * EM_TASKS * RS;
    double* Mt = M + (size_t)task * RS;
    long long t0 = prof ? clock64() : 0, t1;
    // cumulative hazard, coal_EM.cpp:100-103: products in parallel, then every thread that needs
    // Lam[e] adds them up in index order (same additions as the serial loop)
    for (int e = tid + 1; e < E; e += blockDim.x) prod[e] = rate[e - 1] * (ep[e] - ep[e - 1]);
    __syncthreads();
    for (int e = tid; e < E; e += blockDim.x) {
      double l = 0.0;
      for (int i = 1; i <= e; i++) l = l + prod[i];
      Lam[e] = l;
    }
    __syncthreads();
    for (int e = tid; e < E; e += blockDim.x) em_AB(E, ep, rate, Lam, e, A, B, c.T);
    __syncthreads();
    if (prof) { t1 = clock64(); tp[0] += t1 - t0; t0 = t1; }
    // folds, special epochs and per-task E-step
    double my_logl = 0.0;
    auto emit = [&](int e, double ne, double de) {
      Mt[e] = cnt * ne;
      Mt[E + e] = cnt * de;
    };
    if (tid == 384) {  // prefix chain of the shared tasks (coal_EM.cpp:254-258), published entry by entry
      double nc = 1.0;
      PL[0] = nc;
      for (int e = 0; e < E; e++) {
        const double v = A[e];
        if (nc == 1.0) nc = v; else nc = lse(nc, v, c.T);
        PL[e + 1] = nc;
        __threadfence_block();
        pl_ready = e + 1;
      }
    } else if (mine && !is_shared) {
      my_logl = cnt * task_notshared(c, t, k, true, emit);
    } else if (mine && is_shared) {
      double num_t, den_t;
      shared_special(c, t, et, num_t, den_t);
      while (pl_ready < et) { }
      const double pl = ((volatile double*)PL)[et];
      my_logl = cnt * task_shared(c, et, true, pl, num_t, den_t, emit);
    }
    if (mine) Mt[2 * E] = my_logl;
    __threadfence();
    if (prof) { t1 = clock64(); tp[1] += t1 - t0; t0 = t1; }
    cluster.sync();
    if (tid == 0) pl_ready = 0;
    if (prof) { t1 = clock64(); tp[3] += t1 - t0; t0 = t1; }
    // sums over the tasks in the reference's order (bin ascending, shared before not shared)
    const int n_task = 2 * NBINS;
    if (csize > 1) {
      // cluster: CTA r sums columns [r*CW, (r+1)*CW) of M over all tasks (one gather into shared
      // memory, thread = column) and stores the results into every CTA's tn / td / ll through
      // distributed shared memory
      const int ncol = 2 * E + 1;
      const int CW = (ncol + csize - 1) / csize;
      const int cbeg = crank * CW, cend = min(ncol, cbeg + CW);
      const int CB = (2 * EM_STAGE_DOUBLES) / n_task;   // columns that fit the staging buffer at once
      for (int c0 = cbeg; c0 < cend; c0 += CB) {
        const int cw = min(CB, cend - c0);
        for (int i = tid; i < n_task * cw; i += blockDim.x) {
          const int j = i / cw, cc = i - j * cw;
          stage[i] = __ldcg(M + (size_t)j * RS + c0 + cc);
        }
        __syncthreads();
        if (tid < cw) {
          double acc = 0.0;
#pragma unroll 10
          for (int j = 0; j < n_task; j++) acc += stage[j * cw + tid];
          const int col = c0 + tid;
          for (int r = 0; r < csize; r++) {
            if (col < E) cluster.map_shared_rank(tn, r)[col] = acc;
            else if (col < 2 * E) cluster.map_shared_rank(td, r)[col - E] = acc;
            else cluster.map_shared_rank(&ll_new, r)[0] = acc;
          }
        }
        __syncthreads();
      }
      cluster.sync();
      if (tid == 0) { prev_s = ll_s; ll_s = ll_new; }
    } else {
      // single CTA: chunks of TJ rows of M are staged through shared memory (double-buffered), thread = column.
      // 2E + 1 columns can outnumber the threads (E >= 208): thread tid also owns columns tid + EM_THREADS, ..., whose
      // running sums live in their final places (tn / td are contiguous; column 2E is ll_new), summed in the same task order
      double acc = 0.0;
      int buf = 0;
      for (int col = tid + EM_THREADS; col <= 2 * E; col += EM_THREADS) (col < 2 * E ? tn[col] : ll_new) = 0.0;
      for (int i = tid; i < min(TJ, n_task) * RS; i += blockDim.x) stage[i] = __ldcg(M + i);
      __syncthreads();
      for (int j0 = 0; j0 < n_task; j0 += TJ) {
        const int nj = min(TJ, n_task - j0);
        const int j1 = j0 + TJ, nn = (j1 < n_task) ? min(TJ, n_task - j1) : 0;
        double pre[9];
        const double* src = M + (size_t)j1 * RS;
#pragma unroll
        for (int u = 0; u < 9; u++) { const int i = tid + u * EM_THREADS; pre[u] = (i < nn * RS) ? __ldcg(src + i) : 0.0; }
        if (tid <= 2 * E) {
          const double* col = stage + (size_t)buf * EM_STAGE_DOUBLES + tid;
          for (int j = 0; j < nj; j++) acc += col[(size_t)j * RS];
        }
        for (int c2 = tid + EM_THREADS; c2 <= 2 * E; c2 += EM_THREADS) {
          const double* col = stage + (size_t)buf * EM_STAGE_DOUBLES + c2;
          double& a2 = c2 < 2 * E ? tn[c2] : ll_new;
          double s = a2;
          for (int j = 0; j < nj; j++) s += col[(size_t)j * RS];
          a2 = s;
        }
        double* dst = stage + (size_t)(buf ^ 1) * EM_STAGE_DOUBLES;
#pragma unroll
        for (int u = 0; u < 9; u++) { const int i = tid + u * EM_THREADS; if (i < nn * RS) dst[i] = pre[u]; }
        __syncthreads();
        buf ^= 1;
      }
      if (tid < E) tn[tid] = acc;
      else if (tid < 2 * E) td[tid - E] = acc;
      else if (tid == 2 * E) { prev_s = ll_s; ll_s = acc; }
      if (2 * E >= EM_THREADS && tid == 2 * E % EM_THREADS) { prev_s = ll_s; ll_s = ll_new; }
    }
    __syncthreads();
    if (prof) { t1 = clock64(); tp[4] += t1 - t0; t0 = t1; }
    // M-step, coal.cpp:3771-3815 (regularise == 2): rate[e] = num/denom floored at 5e-9; num == 0 ->
    // copy the (already updated) rate of the previous epoch, or 0 for epoch 0; denom == 0 -> keep
    for (int e = tid; e < E; e += blockDim.x) {
      const double n_ = tn[e], d_ = td[e];
      double r = rate[e];
      if (n_ != 0 && d_ != 0) { r = n_ / d_; r = (r < 5e-9) ? 5e-9 : r; }
      cand[e] = r;
    }
    __syncthreads();
    for (int e = tid; e < E; e += blockDim.x) {
      int s = e;
      while (s >= 0 && tn[s] == 0) s--;          // nearest epoch at or below e with a non-zero numerator
      rate[e] = (s >= 0) ? cand[s] : 0.0;
    }
    if (tid == 0 && (ll_s / prev_s > 1.0 - 1e-7) && (iter > 1000)) stop_flag = 1;  // coal.cpp:3822
    __syncthreads();
    if (prof) { t1 = clock64(); tp[5] += t1 - t0; t0 = t1; }
    if (stop_flag) break;
  }
  if (prof && tid == 0) for (int i = 0; i < 6; i++) prof[i] = tp[i];
  if (prof && tid == 384) prof[6] = tp[1];
  if (prof && tid == 192 + 8 * crank + 1) prof[7] = tp[1];
  if (crank == 0) {
    for (int e = tid; e < E; e += blockDim.x) rates_out[(size_t)rep * E + e] = rate[e];
    if (tid == 0) { iters_out[rep] = iter; ll_out[rep] = ll_s; }
  }
}

// ---- stage iii, latency mode: ONE replicate spread over a cluster of 8 CTAs ------------------
// Used when there are too few replicates to fill the GPU (config 2: R = 1).  The per-iteration
// latency floor is the two sequential logsumexp folds of the E-step (coal_EM.cpp:254-258 and
// 327-357: ~42 dependent exp + log1p pairs), so everything else is arranged around them:
//   * CTA r owns the age bins = r (mod csize), both task types; slot = 2 * (bin / csize) + type
//   * A_ep / B_ep and the fold-free part of every head (special epoch) run side by side
//   * folds: the not-shared tasks two per warp (adjacent bins: nearly identical branch decisions,
//     so the lanes rarely diverge), the shared tasks' common prefix chain on its own warp, which
//     afterwards finishes the 24 shared heads (one logsumexp each) on its lanes
//   * the two exp() per (task, epoch) are spread over the whole CTA, the serial `integ` recursion
//     is reduced to one subtraction per epoch, and the rows go out with coalesced stores
//   * rows are pushed with st.async into the column buffers of the CTAs that sum them (CTA r sums
//     columns [r*CW, (r+1)*CW) IN THE REFERENCE'S ORDER, coal.cpp:3704-3733) and the totals are
//     broadcast the same way; each destination counts the arriving bytes on an mbarrier
//     (complete_tx), so nobody waits on a cluster-wide barrier; redundant M-step.
// Same operations and operand order as task_shared / task_notshared.
constexpr int EMS_THREADS = 640;
constexpr int EMS_FOLD_WARPS = 12;
constexpr int EMS_TLMAX = 96;

// distributed-shared-memory plumbing of k_em_split: remote stores that count their bytes on an mbarrier of
// the destination CTA (st.async ... complete_tx), so a consumer waits for exactly the data it needs
// instead of a cluster-wide barrier
__device__ __forceinline__ uint32_t em_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t em_mapa(uint32_t saddr, int rank)
{
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void em_st_async(uint32_t raddr, double v, uint32_t rbar)
{
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];" ::"r"(raddr),
               "l"(__double_as_longlong(v)), "r"(rbar) : "memory");
}
__device__ __forceinline__ void em_mbar_init(uint64_t* bar, int count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(em_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void em_mbar_arm(uint64_t* bar, uint32_t bytes)   // this phase completes once `bytes` have landed
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(em_smem_u32(bar)), "r"(bytes) : "memory");
}
// false: the bytes did not arrive within ~2 s (a peer is gone or the byte accounting is off): the caller gives up
// instead of hanging the GPU
__device__ __forceinline__ bool em_mbar_wait(uint64_t* bar, uint32_t parity)
{
  const long long t0 = clock64();
  for (;;) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(em_smem_u32(bar)), "r"(parity) : "memory");
    if (done) return true;
    if (clock64() - t0 > 4000000000ll) return false;
  }
}
__device__ __forceinline__ void named_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

__global__ void __launch_bounds__(EMS_THREADS, 1)
k_em_split(int E, const double* __restrict__ epochs, const double* __restrict__ rates_init,
           const double* __restrict__ age_bin_g, const double* __restrict__ counts, int max_iter,
           const uint64_t* __restrict__ exp_tab_g, const uint64_t* __restrict__ log_tab_g, double* scratch,
           double* __restrict__ rates_out, int32_t* __restrict__ iters_out, double* __restrict__ ll_out, long long* prof_g)
{
  cg::cluster_group cluster = cg::this_cluster();
  const int crank = (int)cluster.block_rank(), csize = (int)cluster.num_blocks();
  const int rep = blockIdx.x / csize;
  const int n_task = 2 * NBINS, ncol = 2 * E + 1, RS = 2 * E + 2;
  const int CW = (ncol + csize - 1) / csize;               // columns summed by one CTA
  const int nbl = (NBINS + csize - 1) / csize;             // bins of one CTA
  const int ntl = 2 * nbl;                                 // its task slots

  extern __shared__ double sm[];
  double* ep = sm;                  // [E]
  double* rate = ep + E;            // [E]
  double* Lam = rate + E;           // [E]
  double* A = Lam + E;              // [E]
  double* B = A + E;                // [E]
  double* PL = B + E;               // [E+1]
  double* tn = PL + E + 1;          // [E]
  double* td = tn + E;              // [E]
  double* cand = td + E;            // [E]
  double* prod = cand + E;          // [E]
  double* raw = prod + E;           // [ntl][E][2]  exp() of the two log-domain terms
  double* integ_s = raw + (size_t)ntl * E * 2;             // [ntl][E]     integ after epoch e
  double* colbuf = integ_s + (size_t)ntl * E;              // [n_task][CW] columns [crank*CW, ..) of every task's row, pushed by the owners
  uint64_t* etab = (uint64_t*)(colbuf + (size_t)n_task * CW);  // [256]
  uint64_t* ltab = etab + 256;                                  // [256]
  __shared__ int stop_flag;
  __shared__ double ll_s, prev_s, ll_new;
  __shared__ __align__(8) uint64_t bar_rows, bar_tot;      // bytes of pushed rows / of broadcast totals that have landed here
  __shared__ double h_t[EMS_TLMAX], h_cnt[EMS_TLMAX], h_nc[EMS_TLMAX], h_numt[EMS_TLMAX], h_dent[EMS_TLMAX], h_logl[EMS_TLMAX];
  __shared__ int h_et[EMS_TLMAX], h_good[EMS_TLMAX];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // exact i / E and c / CW for the small indices used below (i < 2^15): one multiply-high instead of a division
  const uint32_t magicE = E > 1 ? 0xffffffffu / (uint32_t)E + 1u : 0u, magicCW = CW > 1 ? 0xffffffffu / (uint32_t)CW + 1u : 0u;
  auto divE = [&](int i) { return magicE ? (int)__umulhi((uint32_t)i, magicE) : i; };
  auto divCW = [&](int c) { return magicCW ? (int)__umulhi((uint32_t)c, magicCW) : c; };
  for (int e = tid; e < E; e += blockDim.x) { ep[e] = epochs[e]; rate[e] = rates_init[e]; }
  for (int i = tid; i < 256; i += blockDim.x) { etab[i] = exp_tab_g[i]; ltab[i] = log_tab_g[i]; }
  if (tid == 0) {
    stop_flag = 0; ll_s = neg_inf();
    em_mbar_init(&bar_rows, 1); em_mbar_init(&bar_tot, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // tasks with a positive count anywhere in the cluster: each pushes one value per column
  const int n_active = __syncthreads_count(tid < n_task && counts[(size_t)rep * 2 * NBINS + tid] > 0);
  const int my_cw = max(0, min(ncol, crank * CW + CW) - crank * CW);
  const uint32_t bytes_rows = (uint32_t)n_active * my_cw * 8, bytes_tot = (uint32_t)ncol * 8;
  const uint32_t colbuf_s = em_smem_u32(colbuf), tn_s = em_smem_u32(tn), td_s = em_smem_u32(td), ll_sa = em_smem_u32(&ll_new);
  const uint32_t bar_rows_s = em_smem_u32(&bar_rows), bar_tot_s = em_smem_u32(&bar_tot);
  if (tid < ntl) {
    const int b = (tid >> 1) * csize + crank, type = tid & 1;
    double t = 0.0, cnt = 0.0;
    if (b < NBINS) { t = age_bin_g[b]; cnt = counts[(size_t)rep * 2 * NBINS + (type ? NBINS : 0) + b]; }
    h_t[tid] = t;
    h_cnt[tid] = cnt > 0 ? cnt : 0.0;                      // coal.cpp:3706, 3719: only bins with a positive count
    h_et[tid] = tint_k(E, ep, t) - 1;
    h_good[tid] = 0; h_nc[tid] = 0.0; h_numt[tid] = 0.0; h_dent[tid] = 0.0; h_logl[tid] = 0.0;
  }
  for (int i = tid; i < n_task * CW; i += blockDim.x) colbuf[i] = 0.0;   // rows of inactive tasks stay 0: x + 0.0 == x
  EmCtx c{E, ep, rate, A, B, Lam, glm::Tables{etab, ltab}};
  long long* prof = prof_g ? prof_g + (size_t)blockIdx.x * 16 : nullptr;
  long long tp[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  cluster.sync();   // every column buffer is zeroed and every mbarrier initialised before the first remote row arrives

  int iter = 0;
  for (; iter < max_iter; iter++) {
    long long t0 = prof ? clock64() : 0, t1;
    if (tid == 0) { em_mbar_arm(&bar_rows, bytes_rows); em_mbar_arm(&bar_tot, bytes_tot); }   // this iteration's phases
    // cumulative hazard, coal_EM.cpp:100-103: products in parallel, then every thread that needs
    // Lam[e] adds them up in index order (same additions as the serial loop)
    for (int e = tid + 1; e < E; e += blockDim.x) prod[e] = rate[e - 1] * (ep[e] - ep[e - 1]);
    __syncthreads();
    for (int e = tid; e < E; e += blockDim.x) {
      double l = 0.0;
      for (int i = 1; i <= e; i++) l = l + prod[i];
      Lam[e] = l;
    }
    __syncthreads();
    // what the folds need: A_ep (threads 0..E-1) and the not-shared tasks' own first term (one thread per bin,
    // on the warps after those)
    const int ft0 = (E + 31) & ~31;
    if (tid < E) em_A(E, ep, rate, Lam, tid, A, c.T);
    else if (tid >= ft0 && tid < ft0 + nbl && h_cnt[2 * (tid - ft0) + 1] > 0) {   // EM_notshared, coal_EM.cpp:327-357, num part
      const int l = 2 * (tid - ft0) + 1, et = h_et[l], k = et + 1;
      const double t = h_t[l], r = rate[et];
      const double c1 = Lam[et] + r * (t - ep[et]);
      const double c2 = c1 + r * (t - t);
      double num_t;
      if (et != E - 1) {
        const double c3 = c2 + r * (ep[k] - t);
        num_t = (r > 0) ? lme(-c2, -c3, c.T) : neg_inf();
      } else num_t = -c2;
      h_numt[l] = num_t;
    }
    __syncthreads();
    if (prof) { t1 = clock64(); tp[0] += t1 - t0; t0 = t1; }
    // the folds; the warps without one fill in what only the later phases need (B_ep, the denominator
    // terms of the not-shared heads, the special epoch of the shared heads)
    if (warp < EMS_FOLD_WARPS) {
      const int fpw = (nbl + EMS_FOLD_WARPS - 1) / EMS_FOLD_WARPS;   // not-shared folds per warp, adjacent bins together
      const int f = warp * fpw + lane, l = 2 * f + 1;
      if (lane < fpw && f < nbl && h_cnt[l] > 0) {
        double nc = h_numt[l];
        const int et = h_et[l];
        if (et != E - 1) {
          double v = A[et + 1];
          for (int e = et + 1; e < E; e++) {               // next term loaded before the step that hides its latency
            const double vn = A[min(e + 1, E - 1)];
            nc = lse(nc, v, c.T);
            v = vn;
          }
        }
        const bool good = !bad(nc);
        h_nc[l] = nc; h_good[l] = good ? 1 : 0; h_logl[l] = h_cnt[l] * (good ? nc : 0.0);
      }
    } else if (warp == EMS_FOLD_WARPS) {
      if (lane == 0) {                                     // shared_prefix_chain with the next term prefetched
        double nc = A[0], v = A[min(1, E - 1)];
        PL[0] = 1.0;
        PL[1] = nc;
        for (int e = 1; e < E; e++) {
          const double vn = A[min(e + 1, E - 1)];
          if (nc == 1.0) nc = v; else nc = lse(nc, v, c.T);
          PL[e + 1] = nc;
          v = vn;
        }
      }
      named_bar_sync(1, EMS_THREADS - EMS_FOLD_WARPS * 32);           // the shared heads' special epochs are in
      for (int j = lane; j < nbl; j += 32) {
        const int l = 2 * j;
        if (h_cnt[l] > 0) {
          const double pl = PL[h_et[l]], num_t = h_numt[l];
          const double nc = (pl == 1.0) ? num_t : lse(pl, num_t, c.T);
          const bool good = !bad(nc);
          h_nc[l] = nc; h_good[l] = good ? 1 : 0; h_logl[l] = h_cnt[l] * (good ? nc : 0.0);
        }
      }
    } else {
      const int q = tid - (EMS_FOLD_WARPS + 1) * 32;
      if (q < E) em_B(E, ep, rate, Lam, q, B, c.T);
      else if (q < E + nbl) {                                        // EM_notshared, coal_EM.cpp:327-357, denom part
        const int l = 2 * (q - E) + 1;
        if (h_cnt[l] > 0) {
          const int et = h_et[l], k = et + 1;
          const double t = h_t[l], r = rate[et], inv = 1.0 / r;
          const double c1 = Lam[et] + r * (t - ep[et]);
          const double c2 = c1 + r * (t - t);
          double den_t;
          if (et != E - 1) {
            const double c3 = c2 + r * (ep[k] - t);
            den_t = (r > 0) ? glm::log((t + inv) - (ep[k] + inv) * glm::exp(-c3 + c2, c.T), c.T) - c2 : neg_inf();
          } else den_t = glm::log(t + inv, c.T) - c2;
          h_dent[l] = den_t;
        }
      } else if (q < E + 2 * nbl) {
        const int l = 2 * (q - E - nbl);
        if (h_cnt[l] > 0) {
          double num_t, den_t;
          shared_special(c, h_t[l], h_et[l], num_t, den_t);
          h_numt[l] = num_t; h_dent[l] = den_t;
        }
      }
      named_bar_arrive(1, EMS_THREADS - EMS_FOLD_WARPS * 32);
    }
    __syncthreads();
    if (prof) { t1 = clock64(); tp[1] += t1 - t0; t0 = t1; }
    // exp() of the two log-domain terms of every (slot, epoch) pair: first the numerator terms (the
    // integ recursion needs them), then the denominator terms while the first warp(s) run the recursion
    auto raw_term = [&](int i, int which) {
      const int l = divE(i), e = i - l * E, et = h_et[l];
      const bool sh = (l & 1) == 0;
      const int lim = (E - 1 < et + 1) ? E - 1 : et + 1;
      const bool need = h_good[l] && (sh ? (e < lim || (e == E - 1 && et == E - 1)) : (e >= et));
      const bool own = sh ? !(e < et) : (e == et);           // the task's own special-epoch terms instead of A_ep / B_ep
      if (need) {
        const double x = (which == 0 ? (own ? h_numt[l] : A[e]) : (own ? h_dent[l] : B[e])) - h_nc[l];
        raw[2 * i + which] = exp_fast(x, c.T);
      }
    };
    for (int i = tid; i < ntl * E; i += blockDim.x) raw_term(i, 0);
    __syncthreads();
    if (prof) { t1 = clock64(); tp[2] += t1 - t0; t0 = t1; }
    const int iw = ((ntl + 31) >> 5) * 32;                   // threads reserved for the recursion (one per slot)
    if (tid >= iw) {
      for (int i = tid - iw; i < ntl * E; i += blockDim.x - iw) raw_term(i, 1);
    } else if (tid < ntl && h_good[tid]) {
      // the serial part of a task: integ after epoch e (coal_EM.cpp:266-271, 437-446)
      const int et = h_et[tid];
      const int lo = (tid & 1) ? et : 0;
      const int hi = (tid & 1) ? E - 1 : ((E - 1 < et + 1) ? E - 1 : et + 1);
      double integ = 1.0;
      const double* __restrict__ rw = raw + (size_t)tid * E * 2;
      double* __restrict__ out = integ_s + tid * E;
      // Branch-free steps, loads of a chunk first.  Outside [lo, hi) the step subtracts 0.0: before lo
      // integ is still 1.0, and from hi on the value is not used.
      for (int e0 = 0; e0 < E; e0 += 8) {
        double nb[8];
#pragma unroll
        for (int u = 0; u < 8; u++) nb[u] = (e0 + u >= lo && e0 + u < hi) ? rw[2 * (e0 + u)] : 0.0;
#pragma unroll
        for (int u = 0; u < 8; u++) {
          integ = (integ > 0.0) ? integ - nb[u] : 0.0;
          if (e0 + u < E) out[e0 + u] = integ;
        }
      }
    }
    __syncthreads();
    if (prof) { t1 = clock64(); tp[8] += t1 - t0; t0 = t1; }
    // rows {count*num[e] (E), count*denom[e] (E), count*logl} -> pushed through distributed shared
    // memory into the column buffers of the CTAs that sum them
    for (int i = tid; i < ntl * E; i += blockDim.x) {
      const int l = divE(i), e = i - l * E;
      const double cnt = h_cnt[l];
      if (cnt > 0) {
        const int et = h_et[l];
        double ne = 0.0, de = 0.0;
        if (h_good[l]) {
          const double integ = integ_s[i];
          if ((l & 1) == 0) {
            const int lim = (E - 1 < et + 1) ? E - 1 : et + 1;
            if (e < lim) {
              ne = raw[2 * i];
              de = raw[2 * i + 1];
              de += -ep[e] * ne + (ep[e + 1] - ep[e]) * integ;
              if (de < 0.0) de = 0.0;
            } else if (e == E - 1 && et == E - 1) {
              ne = raw[2 * i];
              de = raw[2 * i + 1];
              de -= ep[e] * ne;
              if (de < 0.0) de = 0.0;
            }
          } else {
            if (e < et) {
              de = ep[e + 1] - ep[e];
            } else {
              ne = raw[2 * i];
              if (e < E - 1) {
                de = raw[2 * i + 1];
                de += -ep[e] * ne + (ep[e + 1] - ep[e]) * integ;
              } else {
                de = raw[2 * i + 1];
                de -= ep[e] * ne;
              }
              if (de < 0.0) de = 0.0;
            }
          }
        }
        const int tk = 2 * ((l >> 1) * csize + crank) + (l & 1);   // row of the task
        const int r1 = divCW(e), r2 = divCW(E + e);
        em_st_async(em_mapa(colbuf_s, r1) + 8u * (tk * CW + (e - r1 * CW)), cnt * ne, em_mapa(bar_rows_s, r1));
        em_st_async(em_mapa(colbuf_s, r2) + 8u * (tk * CW + (E + e - r2 * CW)), cnt * de, em_mapa(bar_rows_s, r2));
      }
    }
    if (tid < ntl && h_cnt[tid] > 0) {
      const int tk = 2 * ((tid >> 1) * csize + crank) + (tid & 1), r = (2 * E) / CW;
      em_st_async(em_mapa(colbuf_s, r) + 8u * (tk * CW + (2 * E - r * CW)), h_logl[tid], em_mapa(bar_rows_s, r));
    }
    if (prof) { t1 = clock64(); tp[6] += t1 - t0; t0 = t1; }
    if (warp == 0 && !em_mbar_wait(&bar_rows, iter & 1)) stop_flag = 2;   // all rows of this iteration have landed in colbuf
    __syncthreads();
    if (prof) { t1 = clock64(); tp[3] += t1 - t0; t0 = t1; }
    // sums over the tasks in the reference's order (bin ascending, shared before not shared)
    {
      const int cbeg = crank * CW, cw = max(0, min(ncol, cbeg + CW) - cbeg);
      if (prof) { t1 = clock64(); tp[7] += t1 - t0; t0 = t1; }
      if (tid < cw) {
        double acc = 0.0;
#pragma unroll 10
        for (int j = 0; j < n_task; j++) acc += colbuf[j * CW + tid];
        prod[tid] = acc;                                   // prod[] is free until the next iteration
      }
      __syncthreads();
      for (int i = tid; i < cw * csize; i += blockDim.x) { // totals -> every CTA's tn / td / ll (DSMEM)
        const int r = i / cw, cc = i - r * cw, col = cbeg + cc;
        const double acc = prod[cc];
        const uint32_t dst = col < E ? tn_s + 8u * col : col < 2 * E ? td_s + 8u * (col - E) : ll_sa;
        em_st_async(em_mapa(dst, r), acc, em_mapa(bar_tot_s, r));
      }
      if (warp == 0 && !em_mbar_wait(&bar_tot, iter & 1)) stop_flag = 2;    // the totals of all columns have landed here
      __syncthreads();
      if (tid == 0) { prev_s = ll_s; ll_s = ll_new; }
    }
    __syncthreads();
    if (prof) { t1 = clock64(); tp[4] += t1 - t0; t0 = t1; }
    // M-step, coal.cpp:3771-3815 (regularise == 2): rate[e] = num/denom floored at 5e-9; num == 0 ->
    // copy the (already updated) rate of the previous epoch, or 0 for epoch 0; denom == 0 -> keep
    for (int e = tid; e < E; e += blockDim.x) {
      const double n_ = tn[e], d_ = td[e];
      double r = rate[e];
      if (n_ != 0 && d_ != 0) { r = n_ / d_; r = (r < 5e-9) ? 5e-9 : r; }
      cand[e] = r;
    }
    __syncthreads();
    for (int e = tid; e < E; e += blockDim.x) {
      int s = e;
      while (s >= 0 && tn[s] == 0) s--;          // nearest epoch at or below e with a non-zero numerator
      rate[e] = (s >= 0) ? cand[s] : 0.0;
    }
    if (tid == 0 && stop_flag == 0 && (ll_s / prev_s > 1.0 - 1e-7) && (iter > 1000)) stop_flag = 1;  // coal.cpp:3822
    __syncthreads();
    if (prof) { t1 = clock64(); tp[5] += t1 - t0; t0 = t1; }
    if (stop_flag) break;
  }
  if (prof && tid == 0) for (int i = 0; i < 16; i++) prof[i] = tp[i];
  cluster.sync();   // nobody leaves while a peer may still address its shared memory
  if (crank == 0) {
    for (int e = tid; e < E; e += blockDim.x) rates_out[(size_t)rep * E + e] = rate[e];
    if (tid == 0) { iters_out[rep] = iter; ll_out[rep] = ll_s; }
  }
  if (stop_flag == 2 && tid == 0) iters_out[rep] = -1;   // handshake timed out: reported as an error by the host
}

// ---- stage iii, throughput mode: ONE replicate per CTA, work spread over the whole CTA --------------
// Used when there are enough replicates to give every SM a CTA (config 3).  Same arithmetic as k_em /
// k_em_split (same operations in the same order: rates, log-likelihood and iteration counts are bit-identical),
// organised like k_em_split inside one CTA: the sequential logsumexp folds run one per lane, everything
// else is spread over all threads, and nothing leaves shared memory.
//   P0  cumulative hazard, A_ep, the not-shared tasks' own first term
//   P1  folds: one not-shared fold per lane (warps 0..5), the shared tasks' prefix chain on its own thread,
//       followed by the 185 shared heads; the other warps fill in B_ep, the denominator terms and the shared
//       tasks' special epoch meanwhile
//   P2  exp() of the two log-domain terms of every NEEDED (task, epoch) pair -- a shared task needs epochs
//       [0, et], a not-shared task [et, E): 185 x (E + 1) pairs instead of 370 x E -- from a static pair
//       table, written to a compact store (valN / valD, a task's entries contiguous, odd-length blocks)
//   P3  thread = task: the serial `integ` recursion and the epoch's exposure, in place, times the count
//   P4  thread = column: the sums over the 370 tasks in the reference's order (coal.cpp:3704-3733) straight
//       from the compact store; M-step and stop rule.
constexpr int EMC_THREADS = 640;
constexpr int EMC_FOLD_WARPS = 6;     // 185 not-shared folds, one per lane
constexpr int EMC_NT = 384;           // task slots (370 used): slot = 2 * bin + type

struct EmcTask { int lo, hi, off, et; };   // needed epochs [lo, hi), first entry in the compact store, epoch that holds t

// entries task `l` occupies in the compact store: its needed epochs, padded to an odd count for a shared task and to
// an even count for a not-shared one: the distance between the blocks of two neighbouring bins' tasks of the same
// type is then odd, and a half-warp of P3 threads (one task each) walks 16 different 8-byte banks
__host__ __device__ inline int emc_block(int type, int et, int E)
{
  const int n = type ? E - et : ((E - 1 < et + 1 ? E - 1 : et + 1) + (et == E - 1 ? 1 : 0));
  return type ? (n + 1) & ~1 : n | 1;
}

// The body of k_em_cta and of k_em_cta_grids.  kGrids: every CTA reads its own epoch grid -- grid_of[rep] indexes
// grid_info = {E, offset into the packed epochs / rates_init, n_pairs_cap} -- and writes its row of rates_out with stride
// E_out (zeros past its E).  Everything that depends on E (the shared-memory carve-up, emc_block, the task table, wz) is
// derived from the CTA's own E below, so a replicate's arithmetic is that of a uniform launch on its grid.
template <bool kGrids>
__device__ __forceinline__ void em_cta_body(int E, int n_pairs_cap, const double* __restrict__ epochs, const double* __restrict__ rates_init,
                                            const double* __restrict__ age_bin_g, const double* __restrict__ counts, int max_iter,
                                            const uint64_t* __restrict__ exp_tab_g, const uint64_t* __restrict__ log_tab_g,
                                            double* __restrict__ rates_out, int32_t* __restrict__ iters_out, double* __restrict__ ll_out,
                                            long long* prof_g, const int32_t* __restrict__ grid_of, const int4* __restrict__ grid_info,
                                            int E_out)
{
  const int rep = blockIdx.x;
  if (kGrids) {
    const int4 g = grid_info[grid_of[rep]];
    E = g.x; n_pairs_cap = g.z;
    epochs += g.y; rates_init += g.y;
  }
  extern __shared__ double sm[];
  double* ep = sm;                  // [E]
  double* rate = ep + E;            // [E]
  double* Lam = rate + E;           // [E]
  double* A = Lam + E;              // [E]
  double* B = A + E;                // [E]
  double* PL = B + E;               // [E+1]
  double* tn = PL + E + 1;          // [E]
  double* td = tn + E;              // [E]
  double* cand = td + E;            // [E]
  double* prod = cand + E;          // [E]
  double* wz = prod + E;            // [E+1]  wz[0] = 0.0, wz[1 + e] = width of epoch e: what a task adds outside its block
  double* h_t = sm + ((11 * E + 2 + 1) & ~1);   // [192]  age of the bin (even offset: h_cg and binrec are read as 16-byte words)
  double* h_cnt = h_t + 192;        // [EMC_NT] count of the task (0: inactive, coal.cpp:3706 / 3719)
  double* h_cg = h_cnt + EMC_NT;    // count while the task's normaliser is finite, else 0.0 (set every iteration)
  double* h_nc = h_cg + EMC_NT;     // log normaliser
  double* h_numt = h_nc + EMC_NT;   // the task's own log-domain terms (epoch that holds t)
  double* h_dent = h_numt + EMC_NT;
  double* h_logl = h_dent + EMC_NT; // count * log normaliser
  double* valN = h_logl + EMC_NT;   // [n_pairs_cap] compact store: num[e] of every needed (task, epoch) pair
  double* valD = valN + n_pairs_cap;  // [n_pairs_cap]                exp(den term), then denom[e]
  uint64_t* etab = (uint64_t*)(valD + n_pairs_cap);  // [256]
  uint64_t* ltab = etab + 256;                        // [256]
  EmcTask* task = (EmcTask*)(ltab + 256);             // [EMC_NT]
  int4* binrec = (int4*)(task + EMC_NT);              // [192] column sums: {off_s, hi_s, off_n - lo_n, lo_n} of the bin's two tasks
  int* h_good = (int*)(binrec + 192);                 // [EMC_NT]
  uint16_t* pair_task = (uint16_t*)(h_good + EMC_NT); // [n_pairs_cap] task of every store entry (0xffff: padding)
  __shared__ int stop_flag, n_pairs_s;
  __shared__ double ll_s, prev_s;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_task = 2 * NBINS;
  for (int e = tid; e < E; e += blockDim.x) { ep[e] = epochs[e]; rate[e] = rates_init[e]; }
  for (int i = tid; i < 256; i += blockDim.x) { etab[i] = exp_tab_g[i]; ltab[i] = log_tab_g[i]; }
  if (tid == 0) { stop_flag = 0; ll_s = neg_inf(); }
  __syncthreads();
  for (int e = tid; e <= E; e += blockDim.x) wz[e] = (e >= 1 && e < E) ? ep[e] - ep[e - 1] : 0.0;   // wz[1 + e] = ep[e + 1] - ep[e]
  if (tid < EMC_NT) {
    const int b = tid >> 1, type = tid & 1;
    double t = 0.0, cnt = 0.0;
    int et = 0;
    if (b < NBINS) {
      t = age_bin_g[b];
      cnt = counts[(size_t)rep * 2 * NBINS + (type ? NBINS : 0) + b];
      et = tint_k(E, ep, t) - 1;
      if (type == 0) h_t[b] = t;
    }
    h_cnt[tid] = cnt > 0 ? cnt : 0.0;
    h_cg[tid] = 0.0;
    h_good[tid] = 0; h_nc[tid] = 0.0; h_numt[tid] = 0.0; h_dent[tid] = 0.0; h_logl[tid] = 0.0;
    EmcTask k;
    k.et = et;
    k.lo = type ? et : 0;
    k.hi = type ? E : ((E - 1 < et + 1 ? E - 1 : et + 1) + (et == E - 1 ? 1 : 0));
    if (b >= NBINS || !(cnt > 0)) { k.lo = 0; k.hi = 0; }     // inactive task (coal.cpp:3706, 3719): no entries, its block stays unused
    k.off = 0;
    task[tid] = k;
  }
  __syncthreads();
  if (tid == 0) {   // offsets of the tasks' blocks (static for the whole run)
    int o = 0;
    for (int l = 0; l < n_task; l++) { task[l].off = o; o += emc_block(l & 1, task[l].et, E); }
    n_pairs_s = o;
  }
  __syncthreads();
  const int n_pairs = n_pairs_s;     // <= n_pairs_cap (the host computed the same sum)
  for (int i = tid; i < n_pairs; i += blockDim.x) pair_task[i] = 0xffff;
  if (tid < 192) {
    int4 r = make_int4(0, 0, 0, E + 1);                       // no shared entries; not-shared: never in range (its count is 0.0)
    if (tid < NBINS) {
      const EmcTask ks = task[2 * tid], kn = task[2 * tid + 1];
      r.x = ks.off; r.y = ks.hi;
      if (kn.hi > kn.lo) { r.z = kn.off - kn.lo; r.w = kn.lo; }
    }
    binrec[tid] = r;
  }
  __syncthreads();
  if (tid < n_task) {
    const EmcTask k = task[tid];
    for (int j = 0; j < k.hi - k.lo; j++) pair_task[k.off + j] = (uint16_t)tid;
  }
  EmCtx c{E, ep, rate, A, B, Lam, glm::Tables{etab, ltab}};
  long long* prof = prof_g ? prof_g + (size_t)blockIdx.x * 40 : nullptr;
  long long tp[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  __syncthreads();

  int iter = 0;
  for (; iter < max_iter; iter++) {
    long long t0 = prof ? clock64() : 0, t1;
    // P0: cumulative hazard, coal_EM.cpp:100-103 (products in parallel, then every thread that needs Lam[e] adds
    // them up in index order: the same additions as the serial loop), A_ep, first terms of the not-shared heads
    for (int e = tid + 1; e < E; e += blockDim.x) prod[e] = rate[e - 1] * (ep[e] - ep[e - 1]);
    __syncthreads();
    for (int e = tid; e < E; e += blockDim.x) {
      double l = 0.0;
      for (int i = 1; i <= e; i++) l = l + prod[i];
      Lam[e] = l;
    }
    __syncthreads();
    const int ft0 = (E + 31) & ~31;
    if (tid < E) em_A(E, ep, rate, Lam, tid, A, c.T);
    else if (tid >= ft0 && tid < ft0 + NBINS && h_cnt[2 * (tid - ft0) + 1] > 0) {   // EM_notshared, coal_EM.cpp:327-357, num part
      const int l = 2 * (tid - ft0) + 1, et = task[l].et, k = et + 1;
      const double t = h_t[l >> 1], r = rate[et];
      const double c1 = Lam[et] + r * (t - ep[et]);
      const double c2 = c1 + r * (t - t);
      double num_t;
      if (et != E - 1) {
        const double c3 = c2 + r * (ep[k] - t);
        num_t = (r > 0) ? lme(-c2, -c3, c.T) : neg_inf();
      } else num_t = -c2;
      h_numt[l] = num_t;
    }
    __syncthreads();
    if (prof) { t1 = clock64(); tp[0] += t1 - t0; t0 = t1; }
    // P1: the folds; the warps without one fill in what only the later phases need
    if (warp < EMC_FOLD_WARPS) {
      const int b = tid, l = 2 * b + 1;                        // not-shared fold of bin b
      if (b < NBINS && h_cnt[l] > 0) {
        double nc = h_numt[l];
        const int et = task[l].et;
        if (et != E - 1) {
          double v = A[et + 1];
          for (int e = et + 1; e < E; e++) {                   // next term loaded before the step that hides its latency
            const double vn = A[min(e + 1, E - 1)];
            nc = lse_wide(nc, v, c.T);
            v = vn;
          }
        }
        const bool good = !bad(nc);
        h_nc[l] = nc; h_good[l] = good ? 1 : 0; h_cg[l] = good ? h_cnt[l] : 0.0; h_logl[l] = h_cnt[l] * (good ? nc : 0.0);
      }
    } else if (warp == EMC_FOLD_WARPS) {
      if (lane == 0) {                                         // shared_prefix_chain with the next term prefetched
        double nc = A[0], v = A[min(1, E - 1)];
        PL[0] = 1.0;
        PL[1] = nc;
        for (int e = 1; e < E; e++) {
          const double vn = A[min(e + 1, E - 1)];
          if (nc == 1.0) nc = v; else nc = lse(nc, v, c.T);
          PL[e + 1] = nc;
          v = vn;
        }
      }
    } else {
      const int nh = EMC_THREADS - (EMC_FOLD_WARPS + 1) * 32;
      for (int q = tid - (EMC_FOLD_WARPS + 1) * 32; q < E + 2 * NBINS; q += nh) {
        if (q < E) em_B(E, ep, rate, Lam, q, B, c.T);
        else if (q < E + NBINS) {                              // EM_notshared, coal_EM.cpp:327-357, denom part
          const int l = 2 * (q - E) + 1;
          if (h_cnt[l] > 0) {
            const int et = task[l].et, k = et + 1;
            const double t = h_t[l >> 1], r = rate[et], inv = 1.0 / r;
            const double c1 = Lam[et] + r * (t - ep[et]);
            const double c2 = c1 + r * (t - t);
            double den_t;
            if (et != E - 1) {
              const double c3 = c2 + r * (ep[k] - t);
              den_t = (r > 0) ? glm::log((t + inv) - (ep[k] + inv) * glm::exp(-c3 + c2, c.T), c.T) - c2 : neg_inf();
            } else den_t = glm::log(t + inv, c.T) - c2;
            h_dent[l] = den_t;
          }
        } else {
          const int l = 2 * (q - E - NBINS);
          if (h_cnt[l] > 0) {
            double num_t, den_t;
            shared_special(c, h_t[l >> 1], task[l].et, num_t, den_t);
            h_numt[l] = num_t; h_dent[l] = den_t;
          }
        }
      }
    }
    __syncthreads();
    if (prof) { t1 = clock64(); tp[1] += t1 - t0; t0 = t1; }
    // the shared heads: one logsumexp each (coal_EM.cpp:254-258 ends at the epoch that holds t)
    if (tid < NBINS) {
      const int l = 2 * tid;
      if (h_cnt[l] > 0) {
        const double pl = PL[task[l].et], num_t = h_numt[l];
        const double nc = (pl == 1.0) ? num_t : lse_wide(pl, num_t, c.T);
        const bool good = !bad(nc);
        h_nc[l] = nc; h_good[l] = good ? 1 : 0; h_cg[l] = good ? h_cnt[l] : 0.0; h_logl[l] = h_cnt[l] * (good ? nc : 0.0);
      }
    }
    __syncthreads();
    if (prof) { t1 = clock64(); tp[2] += t1 - t0; t0 = t1; }
    // P2: exp() of the two log-domain terms of every needed (task, epoch) pair (zeros while the task's normaliser is not finite)
    for (int i = tid; i < n_pairs; i += blockDim.x) {
      const int l = pair_task[i];
      if (l == 0xffff) continue;
      const EmcTask k = task[l];
      const int e = k.lo + (i - k.off);
      const bool own = (l & 1) ? (e == k.et) : !(e < k.et);      // the task's own special-epoch terms instead of A_ep / B_ep
      const double nc = h_nc[l];
      const double xn = (own ? h_numt[l] : A[e]) - nc, xd = (own ? h_dent[l] : B[e]) - nc;
      const bool good = h_good[l] != 0;
      valN[i] = good ? exp_fast(xn, c.T) : 0.0;
      valD[i] = good ? exp_fast(xd, c.T) : 0.0;
    }
    __syncthreads();
    if (prof) { t1 = clock64(); tp[3] += t1 - t0; t0 = t1; }
    // P3: thread = task: the serial `integ` recursion (coal_EM.cpp:266-271, 437-446) and the exposure of every needed
    // epoch, in place.  Four epochs at a time (groups aligned to multiples of four for every lane, so the epoch
    // bounds and widths are warp-uniform loads): the loads first, then the four dependent recursion steps, then the
    // four independent exposure chains -- an in-order pipeline overlaps those, not a step-by-step loop.  Same
    // operations as task_shared / task_notshared; the multiplication with the count happens in the column sums.
    // Shared tasks on warps 0..5, not-shared tasks on warps 6..11: neighbouring lanes have similar ranges.
    if (tid < 12 * 32) {
      const int type = tid >= 192, bin = type ? tid - 192 : tid;
      EmcTask k = task[2 * min(bin, NBINS - 1) + type];
      if (bin >= NBINS || !h_good[2 * bin + type]) k.hi = k.lo = 0;
      const int w_lo = __reduce_min_sync(0xffffffffu, k.hi > k.lo ? k.lo : E) & ~3, w_hi = __reduce_max_sync(0xffffffffu, k.hi);
      const double* vn = valN + k.off - k.lo;
      double* vd = valD + k.off - k.lo;
      double integ = 1.0;
      const int n_int = type ? E - 1 : (E - 1 < k.et + 1 ? E - 1 : k.et + 1);   // epochs [lo, n_int) take part in the recursion
      for (int e0 = w_lo; e0 < w_hi; e0 += 4) {
        double ne[4], de[4], el[4], ew[4], ig[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int e = e0 + u, ec = min(max(e, k.lo), max(k.hi - 1, k.lo));   // (outside [lo, hi): some entry of the block, not used)
          ne[u] = vn[ec]; de[u] = vd[ec]; el[u] = ep[min(e, E - 1)]; ew[u] = wz[1 + min(e, E - 1)];
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int e = e0 + u;
          if (e >= k.lo && e < n_int) { if (integ > 0.0) integ -= ne[u]; else integ = 0.0; }
          ig[u] = integ;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int e = e0 + u;
          double d_ = de[u];
          if (e < n_int) d_ += -el[u] * ne[u] + ew[u] * ig[u];
          else d_ -= el[u] * ne[u];                              // the last epoch (coal_EM.cpp:273-287, 455-460)
          if (d_ < 0.0) d_ = 0.0;
          if (e >= k.lo && e < k.hi) vd[e] = d_;
        }
      }
    }
    __syncthreads();
    if (prof) { t1 = clock64(); tp[4] += t1 - t0; t0 = t1; }
    // P4: sums over the tasks in the reference's order (bin ascending, shared before not shared), thread = column;
    // every term is count * value as the reference forms it (coal.cpp:3709-3731).  Outside a task's block its
    // entries are exact zeros -- read from wz[0] -- except the not-shared tasks' epochs before the one that holds
    // t, whose exposure is the whole epoch (coal_EM.cpp:437-441) -- read from wz[1 + e].  (Adding count * 0.0 = +0.0
    // changes nothing: the sums are >= +0.0, or negative in the log-likelihood column.)  Branch-free body: one
    // address select per task, loads and products issued ahead of the addition chain.
    if (tid <= 2 * E) {
      double acc = 0.0;
      if (tid == 2 * E) {
#pragma unroll 8
        for (int l = 0; l < n_task; l++) acc += h_logl[l];       // (0.0 for inactive tasks)
      } else {
        const bool den = tid >= E;
        const int e = den ? tid - E : tid;
        const double* val = (den ? valD : valN) + e;
        const double* before = den ? wz + 1 + e : wz;
        const double2* cg2 = (const double2*)h_cg;
        // groups of four bins, software-pipelined by hand: the records, addresses and values of the NEXT group are
        // loaded before the eight dependent additions of the current one
        constexpr int G = 4;
        double vs[G], vn_[G], cs[G], cn[G];
        auto fetch = [&](int g, double* ps, double* pn, double* qs, double* qn) {
#pragma unroll
          for (int j = 0; j < G; j++) {
            const int bin = min(g * G + j, NBINS);               // bin NBINS: a record without entries and counts of 0.0
            const int4 r = binrec[bin];
            const double2 cg = cg2[bin];
            ps[j] = *(e < r.y ? val + r.x : wz);
            pn[j] = *(e >= r.w ? val + r.z : before);
            qs[j] = cg.x; qn[j] = cg.y;
          }
        };
        fetch(0, vs, vn_, cs, cn);
        for (int g = 0; g < (NBINS + G - 1) / G; g++) {
          double nvs[G], nvn[G], ncs[G], ncn[G];
          fetch(g + 1, nvs, nvn, ncs, ncn);
#pragma unroll
          for (int j = 0; j < G; j++) {
            acc += cs[j] * vs[j];
            acc += cn[j] * vn_[j];
          }
#pragma unroll
          for (int j = 0; j < G; j++) { vs[j] = nvs[j]; vn_[j] = nvn[j]; cs[j] = ncs[j]; cn[j] = ncn[j]; }
        }
      }
      if (tid < E) tn[tid] = acc;
      else if (tid < 2 * E) td[tid - E] = acc;
      else { prev_s = ll_s; ll_s = acc; }
    }
    __syncthreads();
    if (prof) { t1 = clock64(); tp[5] += t1 - t0; t0 = t1; }
    // M-step, coal.cpp:3771-3815 (regularise == 2): rate[e] = num/denom floored at 5e-9; num == 0 ->
    // copy the (already updated) rate of the previous epoch, or 0 for epoch 0; denom == 0 -> keep
    for (int e = tid; e < E; e += blockDim.x) {
      const double n_ = tn[e], d_ = td[e];
      double r = rate[e];
      if (n_ != 0 && d_ != 0) { r = n_ / d_; r = (r < 5e-9) ? 5e-9 : r; }
      cand[e] = r;
    }
    __syncthreads();
    for (int e = tid; e < E; e += blockDim.x) {
      int s = e;
      while (s >= 0 && tn[s] == 0) s--;          // nearest epoch at or below e with a non-zero numerator
      rate[e] = (s >= 0) ? cand[s] : 0.0;
    }
    if (tid == 0 && (ll_s / prev_s > 1.0 - 1e-7) && (iter > 1000)) stop_flag = 1;  // coal.cpp:3822
    __syncthreads();
    if (prof) { t1 = clock64(); tp[6] += t1 - t0; t0 = t1; }
    if (stop_flag) break;
  }
  // (the clock is read when the thread ARRIVES at a barrier: a thread without work in a phase shows the phase's length
  // in the NEXT slot; thread 639 has no work in heads / P3 / P4)
  if (prof && (tid == 0 || tid == 639)) for (int i = 0; i < 8; i++) prof[(tid ? 8 : 0) + i] = tp[i];
  if (kGrids) {
    for (int e = tid; e < E_out; e += blockDim.x) rates_out[(size_t)rep * E_out + e] = e < E ? rate[e] : 0.0;
  } else {
    for (int e = tid; e < E; e += blockDim.x) rates_out[(size_t)rep * E + e] = rate[e];
  }
  if (tid == 0) { iters_out[rep] = iter; ll_out[rep] = ll_s; }
}

__global__ void __launch_bounds__(EMC_THREADS, 1)
k_em_cta(int E, int n_pairs_cap, const double* __restrict__ epochs, const double* __restrict__ rates_init,
         const double* __restrict__ age_bin_g, const double* __restrict__ counts, int max_iter,
         const uint64_t* __restrict__ exp_tab_g, const uint64_t* __restrict__ log_tab_g,
         double* __restrict__ rates_out, int32_t* __restrict__ iters_out, double* __restrict__ ll_out, long long* prof_g)
{
  em_cta_body<false>(E, n_pairs_cap, epochs, rates_init, age_bin_g, counts, max_iter, exp_tab_g, log_tab_g, rates_out, iters_out, ll_out,
                     prof_g, nullptr, nullptr, 0);
}

// k_em_cta over mixed epoch grids (cohorts: every pair's age moves its grid).  Launched with the shared memory of the
// largest grid; no profiling counters.
__global__ void __launch_bounds__(EMC_THREADS, 1)
k_em_cta_grids(const int32_t* __restrict__ grid_of, const int4* __restrict__ grid_info, const double* __restrict__ epochs,
               const double* __restrict__ rates_init, const double* __restrict__ age_bin_g, const double* __restrict__ counts, int max_iter,
               const uint64_t* __restrict__ exp_tab_g, const uint64_t* __restrict__ log_tab_g, int E_out,
               double* __restrict__ rates_out, int32_t* __restrict__ iters_out, double* __restrict__ ll_out)
{
  em_cta_body<true>(0, 0, epochs, rates_init, age_bin_g, counts, max_iter, exp_tab_g, log_tab_g, rates_out, iters_out, ll_out,
                    nullptr, grid_of, grid_info, E_out);
}

// E-step probe: one thread per age, plain stores
__global__ void k_estep(int shared, int E, const double* __restrict__ epochs, const double* __restrict__ rates,
                        int n_t, const double* __restrict__ tt, const uint64_t* __restrict__ exp_tab_g,
                        const uint64_t* __restrict__ log_tab_g, double* __restrict__ num, double* __restrict__ denom,
                        double* __restrict__ logl)
{
  extern __shared__ double sm[];
  double* ep = sm; double* rate = ep + E; double* Lam = rate + E; double* A = Lam + E; double* B = A + E; double* PL = B + E;
  EmCtx c{E, ep, rate, A, B, Lam, glm::Tables{exp_tab_g, log_tab_g}};
  for (int e = threadIdx.x; e < E; e += blockDim.x) { ep[e] = epochs[e]; rate[e] = rates[e]; }
  __syncthreads();
  if (threadIdx.x == 0) em_cumhaz(E, ep, rate, Lam);
  __syncthreads();
  for (int e = threadIdx.x; e < E; e += blockDim.x) em_AB(E, ep, rate, Lam, e, A, B, c.T);
  __syncthreads();
  if (threadIdx.x == 0) shared_prefix_chain(c, PL);
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_t; i += gridDim.x * blockDim.x) {
    const double t = tt[i];
    const int k = tint_k(E, ep, t);
    double* n = num + (size_t)i * E;
    double* d = denom + (size_t)i * E;
    auto emit = [&](int e, double ne, double de) { n[e] = ne; d[e] = de; };
    if (shared) {
      double num_t, den_t;
      shared_special(c, t, k - 1, num_t, den_t);
      logl[i] = task_shared(c, k - 1, true, PL[k - 1], num_t, den_t, emit);
    } else {
      logl[i] = task_notshared(c, t, k, true, emit);
    }
  }
}

// test hook: which = 0 exp, 1 log, 2 log1p
__global__ void k_libm(int which, int n, const double* __restrict__ x, const uint64_t* __restrict__ exp_tab_g,
                       const uint64_t* __restrict__ log_tab_g, double* __restrict__ y)
{
  glm::Tables T{exp_tab_g, log_tab_g};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    y[i] = which == 0 ? glm::exp(x[i], T) : which == 1 ? glm::log(x[i], T) : glm::log1p(x[i]);
}

// test hook: the straight-line pieces of the EM folds, element by element.  which = 0 exp_main, 1 log1p_k0, 2 log1p_wide,
// 3 div_midrange(a, b), 4 lse(a, b), 5 lse_wide(a, b), 6 lme(a, b); ok[i] = the piece's validity predicate (0..2), 1 (3), or
// whether the fold step took its straight-line path (4..6: the predicates inside lse / lse_wide / lme)
__global__ void k_test_em_prims(int which, int n, const double* __restrict__ a, const double* __restrict__ b,
                                const uint64_t* __restrict__ exp_tab_g, const uint64_t* __restrict__ log_tab_g, double* __restrict__ y,
                                int32_t* __restrict__ ok)
{
  glm::Tables T{exp_tab_g, log_tab_g};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double x = a[i], x2 = b[i];
    double r = 0.0;
    bool k = true;
    if (which == 0) { r = glm::exp_main(x, T); k = glm::exp_is_main(x); }
    else if (which == 1) { r = glm::log1p_k0(x); k = glm::log1p_is_k0(x); }
    else if (which == 2) { r = glm::log1p_wide(x); k = glm::log1p_wide_ok(x); }
    else if (which == 3) r = glm::div_midrange(x, x2);
    else if (which == 4 || which == 5) {
      const double d = -fabs(x - x2), e = glm::exp_main(d, T);
      r = which == 4 ? lse(x, x2, T) : lse_wide(x, x2, T);
      k = !bad(x) & !bad(x2) & glm::exp_is_main(d) & (which == 4 ? glm::log1p_is_k0(e) : glm::log1p_wide_ok(e));
    } else {
      const double d = x2 - x, e = -glm::exp_main(d, T);
      r = lme(x, x2, T);
      k = !bad(x) & !bad(x2) & !(x < x2) & glm::exp_is_main(d) & glm::log1p_is_k0(e);
    }
    y[i] = r;
    ok[i] = k ? 1 : 0;
  }
}

// ---- launchers -------------------------------------------------------------------------------
int ensure_libm_tables(colate_handle* h)
{
  if (h->libm_tab.p) return 0;
  CK(h->libm_tab.ensure(512 * 8));
  CK(cudaMemcpyAsync(h->libm_tab.p, glm::hEXP_TAB, 256 * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->libm_tab.as<uint64_t>() + 256, glm::hLOG_TAB, 256 * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int run_bootstrap(colate_handle* h, int R, int num_blocks, const double* block_stats_dev, double age)
{
  k_bootstrap<<<R, 256, 0, h->stream>>>(num_blocks, h->d_weights.as<int32_t>(), block_stats_dev, age,
                                        h->d_agebin.as<double>(), h->d_counts.as<double>(), h->opt_norm_1e3 ? 1 : 0);
  h->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

// k_em_cta's compact-store size and shared memory for the grid epochs_host[E] under the handle's age grid; true if the
// kernel fits (shared memory, and the threads of its first phase)
bool em_cta_fits(const colate_handle* h, int E, const double* epochs_host, int* n_pairs_cap, size_t* smem)
{
  const double* ab = h->h_agebin;
  int cap = 0;
  for (int b = 0; b < NBINS; b++) {
    int k = E;
    for (int e = 0; e < E; e++) if (ab[b] < epochs_host[e]) { k = e; break; }
    cap += emc_block(0, k - 1, E) + emc_block(1, k - 1, E);
  }
  *n_pairs_cap = cap;
  *smem = sizeof(double) * ((size_t)11 * E + 4 + 192 + 6 * EMC_NT + 2 * (size_t)cap) + 512 * 8 + EMC_NT * (sizeof(EmcTask) + 4) + 192 * 16 +
          (size_t)cap * 2 + 32;
  return *smem <= 225 * 1024 && ((E + 31) & ~31) + NBINS <= EMC_THREADS;
}

int run_em(colate_handle* h, int R, int E, int max_iter, const double* epochs_host, cudaStream_t stream)
{
  int rc = ensure_libm_tables(h);
  if (rc) return rc;
  int csize = 1;
  if (const char* e = getenv("COLATE_EM_CLUSTER")) csize = atoi(e);
  else {
    const int sms = h->sm_count;
    while (csize < 8 && R * csize * 2 <= sms) csize *= 2;
    if (csize == 8 && R * 16 * 2 <= sms) csize = 16;   // non-portable cluster size: one GPC (16-20 SMs) per replicate
    // up to SMs/32 replicates (4 on 148 SMs): one GPC each (20.5 ms for 1001 iterations at E = 43); up to SMs/8 (18):
    // clusters of 8, one CTA per SM (23 ms); beyond that one CTA per replicate (k_em_cta: 31 ms for any count up to the
    // number of SMs, against 59 ms for 30 replicates on clusters of 8 at two CTAs per SM; profiles/r02_em_throughput.md)
    if (csize < 8) csize = 1;
  }
  if (csize != 1 && csize != 2 && csize != 4 && csize != 8 && csize != 16) csize = 1;
  // latency mode: one replicate over a cluster of 8 or 16 (k_em_split) when its per-CTA tables fit
  auto split_fits = [&](int cs, size_t* bytes) {
    const int nbl = (NBINS + cs - 1) / cs, ntl = 2 * nbl, CW = (2 * E + 1 + cs - 1) / cs;
    *bytes = sizeof(double) * ((size_t)10 * E + 1 + (size_t)ntl * E * 3 + (size_t)2 * NBINS * CW) + 512 * 8;
    return cs >= 8 && ntl <= EMS_TLMAX && *bytes <= 200 * 1024 && !getenv("COLATE_EM_NOSPLIT") &&
           E + 2 * nbl <= EMS_THREADS - (EMS_FOLD_WARPS + 1) * 32 && ((E + 31) & ~31) + nbl <= EMS_THREADS;
  };
  size_t smem_split = 0;
  bool split = split_fits(csize, &smem_split);
  if (!split && csize > 8) { csize = 8; split = split_fits(csize, &smem_split); }   // k_em itself runs on portable cluster sizes only
  // throughput mode: one replicate per CTA with the work spread over the CTA (k_em_cta) whenever its compact store
  // fits shared memory; the thread-per-task k_em remains for very fine epoch grids
  bool cta = false;
  size_t smem_cta = 0;
  int n_pairs_cap = 0;
  const char* force = getenv("COLATE_EM_KERNEL");   // "cta", "task" (k_em), "split": tests and tuning
  if ((!split && csize == 1 && !(force && !strcmp(force, "task"))) || (force && !strcmp(force, "cta"))) {
    cta = em_cta_fits(h, E, epochs_host, &n_pairs_cap, &smem_cta);
    if (cta) { split = false; csize = 1; }
  }
  const size_t smem = cta ? smem_cta : split ? smem_split : sizeof(double) * ((size_t)10 * E + 1 + 2 * EM_STAGE_DOUBLES) + 512 * 8;
  if (cta) CK(cudaFuncSetAttribute(k_em_cta, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  else if (split) {
    CK(cudaFuncSetAttribute(k_em_split, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (csize > 8) CK(cudaFuncSetAttribute(k_em_split, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  }
  else CK(cudaFuncSetAttribute(k_em, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
  if (!cta) CK(h->d_em_scratch.ensure((size_t)R * 2 * (2 * E + 2) * EM_TASKS * 8 + 1024));
  long long* prof = nullptr;
  if (getenv("COLATE_EM_PROF")) {
    CK(h->d_prof.ensure((size_t)R * csize * 40 * 8));
    CK(cudaMemsetAsync(h->d_prof.p, 0, (size_t)R * csize * 40 * 8, stream));
    prof = h->d_prof.as<long long>();
  }
  h->em_kernel = cta ? 2 : split ? 1 : 0;
  h->em_csize = csize;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(R * csize);
  cfg.blockDim = dim3(cta ? EMC_THREADS : split ? EMS_THREADS : EM_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = csize; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  const uint64_t* tabs = h->libm_tab.as<uint64_t>();
  if (cta)
    CK(cudaLaunchKernelEx(&cfg, k_em_cta, E, n_pairs_cap, (const double*)h->d_epochs.as<double>(), (const double*)h->d_rates.as<double>(),
                          (const double*)h->d_agebin.as<double>(), (const double*)h->d_counts.as<double>(), max_iter, tabs, tabs + 256,
                          h->d_rates.as<double>() + E, h->d_iters.as<int32_t>(), h->d_ll.as<double>(), prof));
  else
  CK(cudaLaunchKernelEx(&cfg, split ? k_em_split : k_em, E, (const double*)h->d_epochs.as<double>(), (const double*)h->d_rates.as<double>(),
                        (const double*)h->d_agebin.as<double>(), (const double*)h->d_counts.as<double>(), max_iter, tabs, tabs + 256,
                        h->d_em_scratch.as<double>(), h->d_rates.as<double>() + E, h->d_iters.as<int32_t>(), h->d_ll.as<double>(), prof));
  h->launches += 1;
  CK(cudaGetLastError());
  if (prof) {
    if (cta) {
      long long q[16];
      CK(cudaMemcpyAsync(q, prof, 128, cudaMemcpyDeviceToHost, stream));
      CK(cudaStreamSynchronize(stream));
      for (int w = 0; w < 2; w++)
        fprintf(stderr, "[k_em_cta prof, replicate 0 thread %d, cycles between its arrivals at the phase barriers] P0 %lld | P1 folds %lld | heads %lld | P2 exps %lld | P3 integ %lld | P4 column sums %lld | M-step %lld\n",
                w ? 639 : 0, q[8 * w], q[8 * w + 1], q[8 * w + 2], q[8 * w + 3], q[8 * w + 4], q[8 * w + 5], q[8 * w + 6]);
      return 0;
    }
    const int ps = split ? 16 : 8;
    std::vector<long long> hp((size_t)ps * csize);
    CK(cudaMemcpyAsync(hp.data(), prof, (size_t)ps * 8 * csize, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    for (int r = 0; r < csize; r++) {
      const long long* q = hp.data() + (size_t)ps * r;
      if (split)
        fprintf(stderr, "[k_em_split prof, replicate 0 CTA %d thread 0, cycles] A + first terms %lld | folds %lld | raw exps %lld | integ %lld | rows out %lld | cluster.sync %lld | gather %lld | sums + broadcast + sync %lld | M-step %lld\n",
                r, q[0], q[1], q[2], q[8], q[6], q[3], q[7], q[4] - q[7], q[5]);
      else
        fprintf(stderr, "[k_em prof, replicate 0 CTA %d thread 0, cycles] AB %lld | folds + tasks %lld (prefix-chain thread %lld, a not-shared task %lld) | cluster.sync %lld | column sums %lld | M-step %lld (csize %d)\n",
                r, q[0], q[1], q[6], q[7], q[3], q[4], q[5], csize);
    }
  }
  return 0;
}

int run_em_grids(colate_handle* h, int R, const int32_t* grid_of_dev, const int* grid_info_dev, int E_out, size_t smem, int max_iter,
                 cudaStream_t stream)
{
  int rc = ensure_libm_tables(h);
  if (rc) return rc;
  CK(cudaFuncSetAttribute(k_em_cta_grids, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const uint64_t* tabs = h->libm_tab.as<uint64_t>();
  k_em_cta_grids<<<R, EMC_THREADS, smem, stream>>>(grid_of_dev, (const int4*)grid_info_dev, h->d_epochs.as<double>(), h->d_rates.as<double>(),
                                                   h->d_agebin.as<double>(), h->d_counts.as<double>(), max_iter, tabs, tabs + 256, E_out,
                                                   h->d_gr_rates.as<double>(), h->d_iters.as<int32_t>(), h->d_ll.as<double>());
  h->launches += 1;
  h->em_kernel = 2;
  h->em_csize = 1;
  CK(cudaGetLastError());
  return 0;
}

int run_estep(colate_handle* h, int shared, int E, int n_t)
{
  int rc = ensure_libm_tables(h);
  if (rc) return rc;
  const size_t smem = sizeof(double) * (6 * E + 1);   // above the default 48 KB from E = 1024 on
  CK(cudaFuncSetAttribute(k_estep, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  double* base = h->d_tmp.as<double>();  // [t: n_t][num: n_t*E][denom: n_t*E][logl: n_t]
  const uint64_t* tabs = h->libm_tab.as<uint64_t>();
  k_estep<<<1, 256, smem, h->stream>>>(shared, E, h->d_epochs.as<double>(), h->d_rates.as<double>(), n_t, base, tabs, tabs + 256,
                                       base + n_t, base + n_t + (size_t)n_t * E, base + n_t + 2 * (size_t)n_t * E);
  CK(cudaGetLastError());
  return 0;
}

int run_libm(colate_handle* h, int which, int n, const double* x_host, double* y_host)
{
  int rc = ensure_libm_tables(h);
  if (rc) return rc;
  CK(h->d_tmp.ensure((size_t)n * 16));
  double* d = h->d_tmp.as<double>();
  const uint64_t* tabs = h->libm_tab.as<uint64_t>();
  CK(cudaMemcpyAsync(d, x_host, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
  k_libm<<<296, 256, 0, h->stream>>>(which, n, d, tabs, tabs + 256, d + n);
  CK(cudaMemcpyAsync(y_host, d + n, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int run_test_em_prims(colate_handle* h, int which, int n, const double* a_host, const double* b_host, double* y_host, int32_t* ok_host)
{
  int rc = ensure_libm_tables(h);
  if (rc) return rc;
  CK(h->d_tmp.ensure((size_t)n * 28));
  double* d = h->d_tmp.as<double>();   // [a: n][b: n][y: n][ok: n int32]
  int32_t* dok = (int32_t*)(d + 3 * (size_t)n);
  const uint64_t* tabs = h->libm_tab.as<uint64_t>();
  CK(cudaMemcpyAsync(d, a_host, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
  if (b_host) CK(cudaMemcpyAsync(d + n, b_host, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
  else CK(cudaMemsetAsync(d + n, 0, (size_t)n * 8, h->stream));
  k_test_em_prims<<<296, 256, 0, h->stream>>>(which, n, d, d + n, tabs, tabs + 256, d + 2 * (size_t)n, dok);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(y_host, d + 2 * (size_t)n, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(ok_host, dok, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

}  // namespace colate
