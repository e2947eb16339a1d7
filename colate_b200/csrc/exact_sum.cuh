// acc (+)= w, c times, each addition rounded to nearest-even exactly as the reference's loop
// `hist[bin] += weight` does for the c samples of one row that fall into the same age bin
// (coal.cpp:2269, 2291-2292) -- but in O(1) instead of c dependent additions.
//
// Inside one binade every rounded addition of the same w moves acc by the same amount
// d = RN(acc + w) - acc (acc is a multiple of its ulp U, w = qU + r, and unless r == U/2 the
// rounding of r does not depend on acc), so acc + k*w "as the reference rounds it" is
// s + (k-1)*d with s = RN(acc + w), provided all partial sums stay in acc's binade, acc >= w
// (so that d and the rounding error are exact) and the sum is not a tie.  The steps that fit
// below the next power of two are taken at once, the step across it is a single rounded
// addition, and the rest continues in the new binade.  Validated against the plain loop by
// tests/test_host.py (host, colate_test_add_repeated) and tests/test_gpu_replay.py (device,
// colate_test_replay_row).
#pragma once
#include <cstdint>
#include <cstring>

#if defined(__CUDACC__)
#define ES_HD __host__ __device__ __forceinline__
#else
#define ES_HD inline
#endif

namespace exsum {

#if defined(__CUDA_ARCH__)
ES_HD double add_(double a, double b) { return __dadd_rn(a, b); }
ES_HD double sub_(double a, double b) { return __dsub_rn(a, b); }
ES_HD double fma_(double a, double b, double c) { return __fma_rn(a, b, c); }
ES_HD double div_(double a, double b) { return __ddiv_rn(a, b); }
ES_HD int hi32(double x) { return __double2hiint(x); }
ES_HD double from_hi(int hi) { return __hiloint2double(hi, 0); }
#else
}  // namespace exsum
#include <cmath>
namespace exsum {
ES_HD double add_(double a, double b) { volatile double r = a + b; return r; }
ES_HD double sub_(double a, double b) { volatile double r = a - b; return r; }
ES_HD double fma_(double a, double b, double c) { return std::fma(a, b, c); }
ES_HD double div_(double a, double b) { volatile double r = a / b; return r; }
ES_HD int hi32(double x) { uint64_t u; memcpy(&u, &x, 8); return (int)(u >> 32); }
ES_HD double from_hi(int hi) { uint64_t u = (uint64_t)(uint32_t)hi << 32; double x; memcpy(&x, &u, 8); return x; }
#endif

ES_HD double add_repeated(double acc, double w, int c)
{
  while (c > 0) {
    const double s = add_(acc, w);
    if (c == 1) return s;
    const int ea = (hi32(acc) >> 20) & 0x7ff;  // biased exponent of acc (acc >= 0 on this path)
    const int es = (hi32(s) >> 20) & 0x7ff;
    if (acc >= w && w > 0.0 && ea > 54 && ea < 0x7fe && es == ea) {
      const double d = sub_(s, acc);                  // exact (Fast2Sum, |acc| >= |w|)
      if (d == 0.0) return s;                         // w below half an ulp: every addition is a no-op
      const double err = sub_(w, d);                  // exact rounding error of acc + w
      const double half_ulp = from_hi((ea - 53) << 20);
      if (err != half_ulp && err != -half_ulp) {      // a tie's rounding depends on acc's last bit
        // k more steps of exactly d keep the sum inside acc's binade; landing on the next power of
        // two is still rounded with this binade's spacing.  Both room and d are multiples of
        // ulp(acc), and the sign of fma(k, d, -room) is exact.
        const double room = sub_(from_hi((ea + 1) << 20), s);
        int k = c - 1;
        if (fma_((double)k, d, -room) > 0.0) {
          k = (int)div_(room, d);
          if (k > c - 1) k = c - 1;
          while (k > 0 && fma_((double)k, d, -room) > 0.0) k--;
          while (k < c - 1 && fma_((double)(k + 1), d, -room) <= 0.0) k++;
        }
        acc = fma_((double)k, d, s);                  // exact: a multiple of ulp(acc) not above 2^(ea+1)
        c -= k + 1;
        continue;                                     // anything left steps over the binade boundary
      }
    }
    acc = s;
    c--;
  }
  return acc;
}

}  // namespace exsum
