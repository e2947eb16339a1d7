/* TEST INFRASTRUCTURE ONLY -- NOT PART OF THE PRODUCT.
 *
 * CPU restatement (plain C, fp64, sequential) of the reference's `Colate --mode mut`
 * tmp/tmp hot path, written from the behaviour of /root/reference (file:line cited on
 * every function).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may load this library, and only as the checker / reported CPU
 * baseline.  The product (colate_b200/) never links, imports or falls back to it.
 *
 * Pinning: the reference ships no golden vectors for this path (SURVEY.md 4); this
 * restatement is pinned against the UNMODIFIED reference compiled from source
 * (oracle/_ref/libcolate_ref.so, oracle/_ref/Colate; see oracle/Makefile) by
 * tests/test_oracle_vs_reference.py, and against fixtures generated from that reference
 * (tests/golden/, script tests/golden/make_golden.py).  Numerics depend on this image's
 * glibc libm (log/exp/log1p/round), the same libm the compiled reference uses.
 *
 * Build: gcc -O2 -std=c11 -fPIC -shared -ffp-contract=off (no FMA contraction: the
 * reference is built for baseline x86-64, which has no FMA).
 */
#define _GNU_SOURCE
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <limits.h>

#define NBINS 185          /* (int)(log(1e8)*10)+1, coal.cpp:3126-3127 */
#define MAX_BLOCKS 500     /* coal.cpp:3140 */
#define BLOCK_BASES 30000000 /* coal.cpp:3139 */
#define NSAMPLES 100       /* coal.cpp:2085 */

/* ------------------------------------------------------------------------------------
 * std::mt19937 and the two libstdc++ distributions the path uses (SURVEY.md App. C).
 * ---------------------------------------------------------------------------------- */
typedef struct { uint32_t mt[624]; uint32_t pos; } oracle_mt;

/* std::mt19937::seed(value): linear_congruential init, libstdc++ <bits/random.tcc>;
 * call site coal.cpp:3162 */
void oracle_mt_seed(oracle_mt* g, uint32_t seed)
{
  g->mt[0] = seed;
  for (uint32_t i = 1; i < 624; i++)
    g->mt[i] = 1812433253u * (g->mt[i - 1] ^ (g->mt[i - 1] >> 30)) + i;
  g->pos = 624;
}

static void mt_twist(oracle_mt* g)
{
  uint32_t* x = g->mt;
  for (int k = 0; k < 624; k++) {
    uint32_t y = (x[k] & 0x80000000u) | (x[(k + 1) % 624] & 0x7fffffffu);
    x[k] = x[(k + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
  }
  g->pos = 0;
}

uint32_t oracle_mt_next(oracle_mt* g)
{
  if (g->pos >= 624) mt_twist(g);
  uint32_t z = g->mt[g->pos++];
  z ^= (z >> 11);
  z ^= (z << 7) & 0x9d2c5680u;
  z ^= (z << 15) & 0xefc60000u;
  z ^= (z >> 18);
  return z;
}

/* std::uniform_real_distribution<double>(0,1)(rng) -> generate_canonical<double,53>:
 * two words, low word first; call sites coal.cpp:2262, 2282 */
double oracle_uniform_real(oracle_mt* g)
{
  double x1 = (double)oracle_mt_next(g);
  double x2 = (double)oracle_mt_next(g);
  double sum = x1 + x2 * 4294967296.0;
  double r = sum / 18446744073709551616.0;
  if (r >= 1.0) r = nextafter(1.0, 0.0);
  return r;
}

/* std::uniform_int_distribution<int>(0,n-1)(rng) for a 32-bit engine, libstdc++ 13
 * (Lemire's nearly-divisionless method); call sites coal.cpp:3330, 3355 */
int oracle_uniform_int(oracle_mt* g, int n)
{
  uint32_t range = (uint32_t)n;           /* urange + 1 */
  uint64_t prod = (uint64_t)oracle_mt_next(g) * range;
  uint32_t low = (uint32_t)prod;
  if (low < range) {
    uint32_t th = (uint32_t)(-range) % range;
    while (low < th) {
      prod = (uint64_t)oracle_mt_next(g) * range;
      low = (uint32_t)prod;
    }
  }
  return (int)(prod >> 32);
}

void oracle_mt_words(uint32_t seed, long discard, int n, uint32_t* out)
{
  oracle_mt g; oracle_mt_seed(&g, seed);
  for (long i = 0; i < discard; i++) oracle_mt_next(&g);
  for (int i = 0; i < n; i++) out[i] = oracle_mt_next(&g);
}
void oracle_uniform_real_n(uint32_t seed, long discard, int n, double* out)
{
  oracle_mt g; oracle_mt_seed(&g, seed);
  for (long i = 0; i < discard; i++) oracle_mt_next(&g);
  for (int i = 0; i < n; i++) out[i] = oracle_uniform_real(&g);
}
void oracle_uniform_int_n(uint32_t seed, long discard, int num_blocks, int n, int* out)
{
  oracle_mt g; oracle_mt_seed(&g, seed);
  for (long i = 0; i < discard; i++) oracle_mt_next(&g);
  for (int i = 0; i < n; i++) out[i] = oracle_uniform_int(&g, num_blocks);
}

/* ------------------------------------------------------------------------------------
 * Age grid and bin index.
 * ---------------------------------------------------------------------------------- */
/* age_bin[0]=0, age_bin[b]=exp((b-1)/10)/10; coal.cpp:3129-3137 */
void oracle_age_bins(double* age_bin /*[185]*/)
{
  double C = 10;
  age_bin[0] = 0.0;
  for (int bin = 0; bin < NBINS - 1; bin++) age_bin[bin + 1] = exp(bin / C) / 10.0;
}

/* (int) of a double as x86-64 cvttsd2si does it (out of range / NaN -> INT_MIN);
 * the reference relies on this for log(0) at coal.cpp:2252 */
static int cast_int_x86(double r)
{
  if (!(r > -2147483649.0 && r < 2147483648.0)) return INT_MIN;
  return (int)r;
}

/* std::max(0,(int)std::round(log(x10)*C)+1) where x10 is the already-multiplied
 * argument; coal.cpp:2253 (x10 = float product 10*age_end, promoted), 2265/2284
 * (x10 = double product 10*sampled_age) */
static int bin_of_x10(double x10)
{
  double C = 10;
  int v = cast_int_x86(round(log(x10) * C));
  v = (int)((unsigned)v + 1u);            /* INT_MIN+1 stays negative */
  return v > 0 ? v : 0;
}
int oracle_bin_of_double_age(double a) { return bin_of_x10(10 * a); }
int oracle_bin_of_float_age(float age_end) { float p = 10 * age_end; return bin_of_x10((double)p); }

/* ------------------------------------------------------------------------------------
 * Row filter (A.2), everything that does not depend on masks or genomes.
 * Returns the packed site meta word the product uses:
 *   bit0 = row passes coal.cpp:2150 + 2166 + 2175-2176, byte1 = ancestral char,
 *   byte2 = derived char (chars only meaningful when bit0 is set).
 * ---------------------------------------------------------------------------------- */
uint32_t oracle_site_meta(int flipped, int n_branch, float age_begin, float age_end,
                          const char* mutation_type)
{
  /* coal.cpp:2150 (age==0 inside parse_tmptmp, coal.cpp:2074) */
  if (!(flipped == 0 && n_branch == 1 && age_begin < age_end && age_end >= 0)) return 0;
  /* split at first '/', coal.cpp:2152-2163 */
  size_t n = strlen(mutation_type), i = 0;
  while (i < n && mutation_type[i] != '/') i++;
  size_t la = i;
  size_t ld = (i + 1 <= n) ? n - (i + 1) : 0;
  if (!(la > 0 && ld > 0)) return 0;      /* coal.cpp:2166 */
  /* coal.cpp:2175-2176: exactly one of ACGT0 / ACGT1 */
  if (la != 1 || ld != 1) return 0;
  char a = mutation_type[0], d = mutation_type[la + 1];
  if (!(a == 'A' || a == 'C' || a == 'G' || a == 'T' || a == '0')) return 0;
  if (!(d == 'A' || d == 'C' || d == 'G' || d == 'T' || d == '1')) return 0;
  return 1u | ((uint32_t)(unsigned char)a << 8) | ((uint32_t)(unsigned char)d << 16);
}

/* ------------------------------------------------------------------------------------
 * Stage i: parse_tmptmp, coal.cpp:2071-2321, on parsed arrays.
 * ---------------------------------------------------------------------------------- */
typedef struct {
  int64_t n;                 /* records in the .colate.in file, in file order          */
  const int32_t* chrom;      /* id of the record's chromosome string: index into the   */
                             /* --chr list, or any value >= n_chr if not listed        */
  const int32_t* bp;
  const uint8_t* anc;
  const uint8_t* der;
  const int32_t* aaf;
  const int32_t* daf;
} oracle_genome;

typedef struct {
  int64_t next;              /* next record to fread                                   */
  int loaded;                /* 0 until the first successful fread (chrom_* garbage)   */
  int32_t chrom, bp, aaf, daf;
  uint8_t anc, der;
} stream_state;

static int stream_read(const oracle_genome* g, stream_state* s)
{
  if (s->next >= g->n) return 0;        /* fread(&lchrom) != 1 -> break, state kept    */
  int64_t k = s->next++;
  s->loaded = 1;
  s->chrom = g->chrom[k]; s->bp = g->bp[k]; s->anc = g->anc[k]; s->der = g->der[k];
  s->aaf = g->aaf[k]; s->daf = g->daf[k];
  return 1;
}
static int stream_on_chr(const stream_state* s, int chr) { return s->loaded && s->chrom == chr; }

/* Outputs (all caller-allocated, zeroed here):
 *   shared, notshared, shared_emp, notshared_emp : [500][185] fp64 (emp = row 0 of the
 *       reference's 185x185 matrix, the only row it writes: coal.cpp:2252-2256)
 *   n_shared, n_notshared, n_emp : [500][185] int64 sample / site tallies
 *   n_used : [500] int64 used rows per block
 * Returns num_blocks (coal.cpp:2319), or a negative error:
 *   -2 a used row with age_begin <= 0 has bin(age_end) >= 185 (the reference writes out of bounds,
 *      coal.cpp:2269) or a used row has bin(age_begin) >= 185 (the rejection loop of coal.cpp:2279-2294
 *      never ends) -- rejected, see DESIGN.md.  Rows with age_begin > 0 and bin(age_end) >= 185 are
 *      rejection-sampled exactly as the reference does.
 *   -3 more than 500 blocks (reference overruns its 500 vectors, coal.cpp:3140)
 */
int oracle_stage1(int n_chr, const int64_t* site_off /*[n_chr+1]*/,
                  const int32_t* pos, const float* age_begin, const float* age_end,
                  const uint32_t* meta,
                  const char* const* tmask_seq, const int64_t* tmask_len, /* NULL = no mask */
                  const char* const* rmask_seq, const int64_t* rmask_len,
                  const oracle_genome* target, const oracle_genome* reference,
                  oracle_mt* rng,
                  double* shared, double* notshared, double* shared_emp, double* notshared_emp,
                  int64_t* n_shared, int64_t* n_notshared, int64_t* n_emp, int64_t* n_used,
                  int64_t* n_used_total)
{
  const double age = 0, ref_age = 0;      /* coal.cpp:2074-2075 */
  const float num_samples = NSAMPLES;
  memset(shared, 0, sizeof(double) * MAX_BLOCKS * NBINS);
  memset(notshared, 0, sizeof(double) * MAX_BLOCKS * NBINS);
  memset(shared_emp, 0, sizeof(double) * MAX_BLOCKS * NBINS);
  memset(notshared_emp, 0, sizeof(double) * MAX_BLOCKS * NBINS);
  memset(n_shared, 0, sizeof(int64_t) * MAX_BLOCKS * NBINS);
  memset(n_notshared, 0, sizeof(int64_t) * MAX_BLOCKS * NBINS);
  memset(n_emp, 0, sizeof(int64_t) * MAX_BLOCKS * NBINS);
  memset(n_used, 0, sizeof(int64_t) * MAX_BLOCKS);
  *n_used_total = 0;

  stream_state st = {0}, sr = {0};
  int num_blocks = 0;                     /* doubles as the block iterator position */

  for (int chr = 0; chr < n_chr; chr++) {
    int current_block_base = 0;           /* coal.cpp:2122 */
    /* chromosome seek, coal.cpp:2125-2145 */
    while (!stream_on_chr(&sr, chr)) { if (!stream_read(reference, &sr)) break; }
    while (!stream_on_chr(&st, chr)) { if (!stream_read(target, &st)) break; }

    for (int64_t m = site_off[chr]; m < site_off[chr + 1]; m++) {
      if (!(meta[m] & 1u)) continue;      /* coal.cpp:2150, 2166 (+2175-2176, which only */
                                          /* clear `use`; nothing else happens for them) */
      int bp_mut = pos[m];
      uint8_t anc = (uint8_t)(meta[m] >> 8), der = (uint8_t)(meta[m] >> 16);
      int use = 1;
      /* masks, coal.cpp:2169-2174; bp_mut is int, seq.size() unsigned long: the
       * comparison promotes bp_mut to unsigned long */
      if (tmask_seq && (uint64_t)(int64_t)bp_mut < (uint64_t)tmask_len[chr]) {
        if (tmask_seq[chr][bp_mut - 1] != 'P') use = 0;
      }
      if (rmask_seq && (uint64_t)(int64_t)bp_mut < (uint64_t)rmask_len[chr]) {
        if (rmask_seq[chr][bp_mut - 1] != 'P') use = 0;
      }
      /* reference stream, coal.cpp:2181-2199 */
      if (use) {
        sr.daf = 0; sr.aaf = 0;
        while (stream_on_chr(&sr, chr) && sr.bp < bp_mut) { if (!stream_read(reference, &sr)) break; }
        if (!stream_on_chr(&sr, chr) || sr.bp != bp_mut || sr.anc != anc || sr.der != der) use = 0;
      }
      if (sr.daf == 0) use = 0;
      int N_ref = sr.daf + sr.aaf;
      /* target stream, coal.cpp:2201-2219 */
      if (use) {
        st.daf = 0; st.aaf = 0;
        while (stream_on_chr(&st, chr) && st.bp < bp_mut) { if (!stream_read(target, &st)) break; }
        if (!stream_on_chr(&st, chr) || st.bp != bp_mut || st.anc != anc || st.der != der) use = 0;
      }
      int N_target = st.daf + st.aaf;
      if (N_target == 0) use = 0;
      if (!use) continue;

      /* coal.cpp:2224-2225 */
      double ab = age_begin[m];
      if (ab < ref_age) ab = ref_age;
      /* block advance, coal.cpp:2227-2234 */
      while (current_block_base + BLOCK_BASES < bp_mut) { current_block_base += BLOCK_BASES; num_blocks++; }
      if (num_blocks >= MAX_BLOCKS) return -3;
      int blk = num_blocks;
      /* pseudo-genotype, coal.cpp:2236-2242 */
      float fD = st.daf, fA = st.aaf;
      fD /= N_target / 2.0;
      fA /= N_target / 2.0;
      fD = roundf(fD);
      fA = roundf(fA);
      /* Rows the reference cannot process: with age_begin <= 0 a draw whose bin reaches 185 is written past the end of
       * the 185-long histogram (coal.cpp:2269: undefined behaviour), and with age_begin itself in bin >= 185 the
       * rejection loop of coal.cpp:2279-2294 never accepts a draw (the reference does not terminate). */
      if (ab <= age && oracle_bin_of_double_age((double)age_end[m]) >= NBINS) return -2;
      if (ab > age && oracle_bin_of_double_age(ab) >= NBINS) return -2;
      n_used[blk]++; (*n_used_total)++;

      if (ab <= age) {
        /* coal.cpp:2250-2256 */
        int b2 = oracle_bin_of_float_age(age_end[m]);
        if (b2 < NBINS) {
          shared_emp[blk * NBINS + b2] += fD * sr.daf / ((double)N_ref);
          notshared_emp[blk * NBINS + b2] += fA * sr.daf / ((double)N_ref);
          n_emp[blk * NBINS + b2]++;
        }
        /* coal.cpp:2259-2273 */
        for (int j = 0; j < NSAMPLES; j++) {
          double a = oracle_uniform_real(rng) * (age_end[m] - ab) + ab;
          if (a < age) a = age;
          int b = oracle_bin_of_double_age(a);
          if (b >= NBINS) return -2;
          notshared[blk * NBINS + b] += fA * sr.daf / ((double)N_ref * num_samples);
          n_notshared[blk * NBINS + b]++;
        }
      } else {
        /* coal.cpp:2279-2295: a draw whose bin reaches 185 (or that falls below `age`) is REDRAWN: it consumes its
         * uniform (two engine words) and does not count towards the 100 samples */
        int j = 0;
        while (j < NSAMPLES) {
          double a = oracle_uniform_real(rng) * (age_end[m] - ab) + ab;
          int skip = a < age;
          int b = oracle_bin_of_double_age(a);
          if (b >= NBINS) skip = 1;
          if (!skip) {
            shared[blk * NBINS + b] += fD * sr.daf / ((double)N_ref * num_samples);
            notshared[blk * NBINS + b] += fA * sr.daf / ((double)N_ref * num_samples);
            n_shared[blk * NBINS + b]++;
            n_notshared[blk * NBINS + b]++;
            j++;
          }
        }
      }
    }
    num_blocks++;                         /* coal.cpp:2306-2310 */
    if (num_blocks > MAX_BLOCKS) return -3;
  }
  return num_blocks;
}

/* ------------------------------------------------------------------------------------
 * SURVEY.md 8(f) N3: the bam/bam front-end parse_onebambam (coal.cpp:1799-2069) on pre-decoded pileups.
 * t_counts / r_counts: [n_site][4] reads showing A, C, G, T at each row's position, i.e. what
 * bam_parser::count_alleles holds at bp_mut - 1 when coal.cpp:1888 / 1939 look (all zero: ring entry absent or empty).
 * Pinned against the reference's own parse_onebambam run on synthetic reads through oracle/hts_stubs.c
 * (tests/golden/stage1_bambam.npz).  Outputs and error codes as oracle_stage1; -2 also for a row with age_begin > 0
 * whose draw reaches bin 185: this front-end has no bound check there (coal.cpp:2034-2039).
 * ---------------------------------------------------------------------------------- */
static int acgt_index(uint8_t c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1; }

/* width 4: [n_site][4] A, C, G, T pileups (the bam front-ends); width 2: [n_site][2] = (AAF, DAF) of the row's two alleles as a bcf
 * decoder resolved them (parse_vcfvcf, coal.cpp:997-1137: N_ref = AAF + DAF, AAF_target = N_target - DAF_target) */
int oracle_stage1_counts(int width, int n_chr, const int64_t* site_off, const int32_t* pos, const float* age_begin, const float* age_end,
                         const uint32_t* meta,
                         const char* const* tmask_seq, const int64_t* tmask_len,
                         const char* const* rmask_seq, const int64_t* rmask_len,
                         const int32_t* t_counts, const int32_t* r_counts, oracle_mt* rng,
                         double* shared, double* notshared, double* shared_emp, double* notshared_emp,
                         int64_t* n_shared, int64_t* n_notshared, int64_t* n_emp, int64_t* n_used, int64_t* n_used_total)
{
  const double age = 0, ref_age = 0;      /* coal.cpp:1801-1802 */
  const float num_samples = NSAMPLES;     /* coal.cpp:1811 */
  memset(shared, 0, sizeof(double) * MAX_BLOCKS * NBINS);
  memset(notshared, 0, sizeof(double) * MAX_BLOCKS * NBINS);
  memset(shared_emp, 0, sizeof(double) * MAX_BLOCKS * NBINS);
  memset(notshared_emp, 0, sizeof(double) * MAX_BLOCKS * NBINS);
  memset(n_shared, 0, sizeof(int64_t) * MAX_BLOCKS * NBINS);
  memset(n_notshared, 0, sizeof(int64_t) * MAX_BLOCKS * NBINS);
  memset(n_emp, 0, sizeof(int64_t) * MAX_BLOCKS * NBINS);
  memset(n_used, 0, sizeof(int64_t) * MAX_BLOCKS);
  *n_used_total = 0;
  int num_blocks = 0;
  for (int chr = 0; chr < n_chr; chr++) {
    int current_block_base = 0;           /* coal.cpp:1845 */
    for (int64_t m = site_off[chr]; m < site_off[chr + 1]; m++) {
      if (!(meta[m] & 1u)) continue;      /* coal.cpp:1849, 1865, 1874-1875: the same row filter as parse_tmptmp */
      int bp_mut = pos[m];
      uint8_t anc = (uint8_t)(meta[m] >> 8), der = (uint8_t)(meta[m] >> 16);
      int use = 1;
      if (tmask_seq && (uint64_t)(int64_t)bp_mut < (uint64_t)tmask_len[chr]) {   /* coal.cpp:1868-1873 */
        if (tmask_seq[chr][bp_mut - 1] != 'P') use = 0;
      }
      if (rmask_seq && (uint64_t)(int64_t)bp_mut < (uint64_t)rmask_len[chr]) {
        if (rmask_seq[chr][bp_mut - 1] != 'P') use = 0;
      }
      int DAF_ref = 0, AAF_ref = 0, DAF_target = 0, AAF_target = 0;
      const int ia = acgt_index(anc), id = acgt_index(der);
      for (int side = 0; side < 2 && use; side++) {      /* coal.cpp:1884-1929 (reference), then 1930-1931, then 1935-1980 (target) */
        const int32_t* c = (side == 0 ? r_counts : t_counts) + width * m;
        int A = 0, D = 0;
        if (width == 2) {
          A = c[0]; D = c[1];
          if (!(A > 0 || D > 0)) use = 0;
        } else {
          int num_reads = 0, num_alleles = 0;
          for (int i = 0; i < 4; i++) { num_reads += c[i]; num_alleles += (c[i] > 0); }
          if (num_reads > 0) {
            if (ia >= 0) A = c[ia];
            if (id >= 0) D = c[id];
            if (A > 0 || D > 0) { if (!(num_alleles <= 2)) use = 0; }
            else use = 0;
          } else use = 0;
        }
        if (side == 0) { AAF_ref = A; DAF_ref = D; if (DAF_ref == 0) use = 0; }
        else { AAF_target = A; DAF_target = D; }
      }
      if (!use) continue;
      int N_ref = DAF_ref + AAF_ref;
      double ab = age_begin[m];
      if (ab < ref_age) ab = ref_age;
      while (current_block_base + BLOCK_BASES < bp_mut) { current_block_base += BLOCK_BASES; num_blocks++; }   /* coal.cpp:1987-1994 */
      if (num_blocks >= MAX_BLOCKS) return -3;
      int blk = num_blocks;
      if (ab <= age && oracle_bin_of_double_age((double)age_end[m]) >= NBINS) return -2;
      if (ab > age && oracle_bin_of_double_age((double)age_end[m]) >= NBINS) return -2;   /* no bound check at coal.cpp:2034-2039 */
      n_used[blk]++; (*n_used_total)++;
      if (ab <= age) {
        int b2 = oracle_bin_of_float_age(age_end[m]);      /* coal.cpp:2002-2006: int * int / double */
        if (b2 < NBINS) {
          shared_emp[blk * NBINS + b2] += DAF_target * DAF_ref / ((double)N_ref);
          notshared_emp[blk * NBINS + b2] += AAF_target * DAF_ref / ((double)N_ref);
          n_emp[blk * NBINS + b2]++;
        }
        for (int j = 0; j < NSAMPLES; j++) {               /* coal.cpp:2009-2023 */
          double a = oracle_uniform_real(rng) * (age_end[m] - ab) + ab;
          if (a < age) a = age;
          int b = oracle_bin_of_double_age(a);
          if (b >= NBINS) return -2;
          notshared[blk * NBINS + b] += AAF_target * DAF_ref / ((double)N_ref * num_samples);
          n_notshared[blk * NBINS + b]++;
        }
      } else {
        int j = 0;                                         /* coal.cpp:2029-2042 */
        while (j < NSAMPLES) {
          double a = oracle_uniform_real(rng) * (age_end[m] - ab) + ab;
          int skip = a < age;
          int b = oracle_bin_of_double_age(a);
          if (!skip) {
            if (b >= NBINS) return -2;
            shared[blk * NBINS + b] += DAF_target * DAF_ref / ((double)N_ref * num_samples);
            notshared[blk * NBINS + b] += AAF_target * DAF_ref / ((double)N_ref * num_samples);
            n_shared[blk * NBINS + b]++;
            n_notshared[blk * NBINS + b]++;
            j++;
          }
        }
      }
    }
    num_blocks++;                         /* coal.cpp:2053-2057 */
    if (num_blocks > MAX_BLOCKS) return -3;
  }
  return num_blocks;
}

int oracle_stage1_pileup(int n_chr, const int64_t* site_off, const int32_t* pos, const float* age_begin, const float* age_end,
                         const uint32_t* meta,
                         const char* const* tmask_seq, const int64_t* tmask_len,
                         const char* const* rmask_seq, const int64_t* rmask_len,
                         const int32_t* t_counts, const int32_t* r_counts, oracle_mt* rng,
                         double* shared, double* notshared, double* shared_emp, double* notshared_emp,
                         int64_t* n_shared, int64_t* n_notshared, int64_t* n_emp, int64_t* n_used, int64_t* n_used_total)
{
  return oracle_stage1_counts(4, n_chr, site_off, pos, age_begin, age_end, meta, tmask_seq, tmask_len, rmask_seq, rmask_len, t_counts, r_counts, rng,
                              shared, notshared, shared_emp, notshared_emp, n_shared, n_notshared, n_emp, n_used, n_used_total);
}

/* ------------------------------------------------------------------------------------
 * Stage ii: block bootstrap + F-redistribution, coal.cpp:3344-3451 (tmp inputs: no /1e3)
 * ---------------------------------------------------------------------------------- */
/* Block multiplicities for all replicates, drawn exactly as coal.cpp:3350-3357.
 * weights: [R][num_blocks] int32 */
void oracle_draw_block_weights(oracle_mt* rng, int R, int num_blocks, int32_t* weights)
{
  for (int i = 0; i < R; i++) {
    int32_t* w = weights + (size_t)i * num_blocks;
    if (R == 1) { for (int j = 0; j < num_blocks; j++) w[j] = 1; }
    else {
      for (int j = 0; j < num_blocks; j++) w[j] = 0;
      for (int j = 0; j < num_blocks; j++) w[oracle_uniform_int(rng, num_blocks)] += 1;
    }
  }
}

/* counts: [R][2][185] (shared, notshared) */
void oracle_stage2(int R, int num_blocks, const int32_t* weights,
                   const double* blk_shared, const double* blk_notshared,
                   const double* blk_shared_emp, const double* blk_notshared_emp,
                   double age, const double* age_bin, double* counts)
{
  for (int i = 0; i < R; i++) {
    double* S = counts + (size_t)i * 2 * NBINS;
    double* N = S + NBINS;
    double semp[NBINS], nemp[NBINS], F[NBINS];
    for (int b = 0; b < NBINS; b++) { S[b] = N[b] = semp[b] = nemp[b] = F[b] = 0.0; }
    const int32_t* w = weights + (size_t)i * num_blocks;
    for (int j = 0; j < num_blocks; j++) {          /* coal.cpp:3358-3390 */
      double bw = (double)w[j];
      if (bw > 0.0) {
        for (int b = 0; b < NBINS; b++) S[b] += bw * blk_shared[j * NBINS + b];
        for (int b = 0; b < NBINS; b++) N[b] += bw * blk_notshared[j * NBINS + b];
        for (int b = 0; b < NBINS; b++) semp[b] += bw * blk_shared_emp[j * NBINS + b];
        for (int b = 0; b < NBINS; b++) nemp[b] += bw * blk_notshared_emp[j * NBINS + b];
      }
    }
    int bin = 0;                                    /* coal.cpp:3394-3396 */
    while (age_bin[bin] <= age) bin++;
    int bin_start = bin;
    double lower_age = age_bin[bin_start - 1];      /* coal.cpp:3399-3400 */
    double fcount = 0.0;
    for (bin = bin_start; bin < NBINS; bin++) {     /* coal.cpp:3406-3417 */
      fcount += semp[bin];
      if (semp[bin] > 0) F[bin] = semp[bin] / (semp[bin] + nemp[bin]);
    }
    for (bin = bin_start; bin < NBINS; bin++) {     /* coal.cpp:3420-3425 */
      F[bin - 1] *= (age_bin[bin] - lower_age);
      lower_age = age_bin[bin];
    }
    double normf = 0.0;                             /* coal.cpp:3428-3432 */
    for (bin = 0; bin < NBINS; bin++) normf += F[bin];
    for (bin = 0; bin < NBINS; bin++) {             /* coal.cpp:3435-3441 */
      F[bin] /= normf;
      F[bin] *= fcount;
      /* std::max(0.0, x): (0.0 < x) ? x : 0.0 -> NaN gives 0.0 */
      S[bin] += (0.0 < F[bin]) ? F[bin] : 0.0;
    }
  }
}

/* every front-end but tmp/tmp: both vectors divided by 1e3 afterwards (coal.cpp:3453-3463, tmp_file == true) */
void oracle_stage2_norm(int R, double* counts)
{
  const double norm = 1e3;
  for (size_t i = 0; i < (size_t)R * 2 * NBINS; i++) counts[i] /= norm;
}

/* ------------------------------------------------------------------------------------
 * Epoch grid, coal.cpp:3503-3632.  Returns num_epochs; *ep_null as at coal.cpp:3505/3622.
 * ---------------------------------------------------------------------------------- */
/* ages from the CLI strings, coal.cpp:3105-3120 */
double oracle_age_generations(const char* target_age, const char* reference_age, float years_per_gen_flag,
                              int has_ypg, double* years_per_gen_out)
{
  double ta = 0, ra = 0;
  if (target_age) ta = strtof(target_age, NULL);
  if (reference_age) ra = strtof(reference_age, NULL);
  double ypg = 28.0;
  if (has_ypg) ypg = years_per_gen_flag;
  *years_per_gen_out = ypg;
  return (ta > ra ? ta : ra) / ypg;
}

int oracle_epochs_from_bins(const char* bins, double age, double years_per_gen,
                            double* epochs /*[cap]*/, int cap, int* ep_null)
{
  double log_10 = log(10);
  double log_age = log(age * years_per_gen) / log_10;
  /* three comma-separated stof tokens, coal.cpp:3557-3590 */
  char buf[256]; double v[3]; size_t i = 0, n = strlen(bins);
  for (int t = 0; t < 3; t++) {
    size_t k = 0;
    if (t > 0 && i >= n) return -1;
    while (i < n && bins[i] != ',' && k + 1 < sizeof buf) buf[k++] = bins[i++];
    buf[k] = 0; i++;
    v[t] = strtof(buf, NULL);
  }
  double epoch_lower = v[0], epoch_upper = v[1], epoch_step = v[2];
  int ne = 0; *ep_null = 0;
  epochs[ne++] = 0.0;
  if (log_age < epoch_lower && age != 0.0) { epochs[ne++] = age; log_age = -1; }
  double epoch_boundary = epoch_lower;
  while (epoch_boundary < epoch_upper) {            /* coal.cpp:3603-3627 */
    if (ne + 3 > cap) return -1;
    if (epoch_boundary > log_age && log_age != -1) {
      epochs[ne++] = age;
      if (epoch_boundary - log_age < 0.25 * epoch_step) epoch_boundary += epoch_step;
      log_age = -1;
    } else {
      if (log_age != -1) (*ep_null)++;
      epochs[ne++] = exp(log_10 * epoch_boundary) / years_per_gen;
    }
    epoch_boundary += epoch_step;
  }
  epochs[ne++] = exp(log_10 * epoch_upper) / years_per_gen;
  { double last = 10 * epochs[ne - 1]; epochs[ne] = (1e8 < last ? last : 1e8) / years_per_gen; ne++; }
  return ne;
}

/* epoch line of a --coal file (its 2nd line), coal.cpp:3513-3544 */
int oracle_epochs_from_coal_line(const char* line, double age, double* epochs, int cap)
{
  int ne = 0, ep = 0; char tmp[128]; size_t k = 0, n = strlen(line);
  for (size_t i = 0; i <= n; i++) {
    int sep = (i == n) || line[i] == ' ' || line[i] == '\t';
    if (!sep) { if (k + 1 < sizeof tmp) tmp[k++] = line[i]; continue; }
    if (i == n && k == 0) break;                    /* trailing `if(tmp != "")` */
    tmp[k] = 0;
    if (k == 0 && i < n) return -1;                 /* stof("") throws in the reference */
    float f = strtof(tmp, NULL);
    if (ne + 2 > cap) return -1;
    if (ep == 1 && age < f && age != 0.0) { epochs[ne++] = age; ep++; }
    if (ep != 1 || age == 0.0) { epochs[ne++] = f; ep++; }
    k = 0;
  }
  return ne;
}

/* ------------------------------------------------------------------------------------
 * Stage iii: E-step (coal_EM.cpp) for age_begin == age_end == t, and the EM driver.
 * ---------------------------------------------------------------------------------- */
static int bad(double x) { return isinf(x) || isnan(x); }

/* the largest epoch grid the C ABI accepts (colate_stage3_em, colate_estep) */
#define ORACLE_MAX_E 1024

/* coal_EM::logsumexp, coal_EM.cpp:5-31 */
static double lse(double a, double b)
{
  if (bad(a)) return bad(b) ? log(0.0) : b;
  if (bad(b)) return a;
  if (a > b) return a + log1p(exp(b - a));
  return b + log1p(exp(a - b));
}
/* coal_EM::logminusexp, coal_EM.cpp:33-58 */
static double lme(double a, double b)
{
  if (bad(a)) return log(0.0);
  if (bad(b)) return a;
  if (a < b) return log(0.0);
  return a + log1p(-exp(b - a));
}

/* coal_EM ctor -> get_AB on the plain epoch grid, coal_EM.hpp:38-50, coal_EM.cpp:97-151.
 * Lam[E] = cumulative hazard at the epoch boundaries. */
void oracle_get_AB(int E, const double* ep, const double* rate, double* A, double* B, double* Lam)
{
  Lam[0] = 0.0;
  for (int i = 1; i < E; i++) Lam[i] = Lam[i - 1] + rate[i - 1] * (ep[i] - ep[i - 1]);
  for (int i = 0; i < E - 1; i++) {
    double tb = ep[i], te = ep[i + 1], r = rate[i], inv = 1.0 / rate[i];
    if (r > 0 && te != 0 && te - tb > 0) {
      A[i] = lme(-Lam[i], -Lam[i + 1]);
      double b = (tb + inv) - (te + inv) * exp(-Lam[i + 1] + Lam[i]);
      B[i] = log(b) - Lam[i];
    } else { A[i] = log(0.0); B[i] = log(0.0); }
  }
  int i = E - 1;
  if (rate[i] > 0) { A[i] = -Lam[i]; B[i] = log(ep[i] + 1.0 / rate[i]) - Lam[i]; }
  else { A[i] = log(0.0); B[i] = log(0.0); }
}

/* get_tint with age_begin==age_end, coal_EM.cpp:60-95: k = number of grid points
 * before the two copies of t (t is inserted at positions k and k+1; epoch of t = k-1) */
static int tint_k(int E, const double* ep, double t)
{
  for (int e = 0; e < E; e++) if (t < ep[e]) return e;
  return E;
}

/* cumulative hazard at the four grid points around t that the identical-times paths
 * read: cs[k-1], cs[k], cs[k+1], cs[k+2]; coal_EM.cpp:176-179 / 314-317 */
static void cs_around(int E, const double* ep, const double* rate, const double* Lam, double t, int k,
                      double* c_km1, double* c_k, double* c_k1, double* c_k2)
{
  double r = rate[k - 1];
  *c_km1 = Lam[k - 1];
  *c_k = *c_km1 + r * (t - ep[k - 1]);
  *c_k1 = *c_k + r * (t - t);
  *c_k2 = (k < E) ? *c_k1 + r * (ep[k] - t) : 0.0;
}

/* coal_EM::EM_shared with age_begin==age_end==t, coal_EM.cpp:153-295 (lines 212-242 skipped) */
double oracle_em_shared(int E, const double* ep, const double* rate, const double* A, const double* B,
                        const double* Lam, double t, double* num, double* denom)
{
  const double log_0 = log(0.0);
  for (int e = 0; e < E; e++) { num[e] = 0; denom[e] = 0; }
  int k = tint_k(E, ep, t), et = k - 1;
  double c0, c1, c2, c3; cs_around(E, ep, rate, Lam, t, k, &c0, &c1, &c2, &c3);
  double nc = 1.0;
  for (int e = 0; e <= et; e++) {
    if (e < et) { num[e] = A[e]; denom[e] = B[e]; }
    else {
      double inv = 1.0 / rate[e], tb = ep[k - 1], te = t;
      if (rate[e] > 0) {
        num[e] = lme(-c0, -c1);
        denom[e] = log((tb + inv) / inv - (te + inv) / inv * exp(-c1 + c0)) + log(inv) - c0;
      } else { num[e] = log_0; denom[e] = log_0; }
    }
    if (nc == 1.0) nc = num[e]; else nc = lse(nc, num[e]);
  }
  if (!bad(nc)) {
    double integ = 1.0;
    int lim = (E - 1 < et + 1) ? E - 1 : et + 1;
    for (int e = 0; e < lim; e++) {
      num[e] -= nc; denom[e] -= nc;
      num[e] = exp(num[e]);
      if (integ > 0.0) integ -= num[e]; else integ = 0.0;
      denom[e] = exp(denom[e]);
      denom[e] += -ep[e] * num[e] + (ep[e + 1] - ep[e]) * integ;
      if (denom[e] < 0.0) denom[e] = 0.0;
    }
    if (et == E - 1) {
      int e = E - 1;
      num[e] -= nc; denom[e] -= nc;
      num[e] = exp(num[e]); denom[e] = exp(denom[e]);
      denom[e] -= ep[e] * num[e];
      if (denom[e] < 0.0) denom[e] = 0.0;
    }
  } else {
    nc = 0.0;
    for (int e = 0; e < E; e++) { num[e] = 0; denom[e] = 0; }
  }
  return nc;
}

/* coal_EM::EM_notshared with age_begin==age_end==t, coal_EM.cpp:297-468 (327-357, 435-466).
 * num/denom are overwritten for every index, as in the reference. */
double oracle_em_notshared(int E, const double* ep, const double* rate, const double* A, const double* B,
                           const double* Lam, double t, double* num, double* denom)
{
  const double log_0 = log(0.0);
  int k = tint_k(E, ep, t), et = k - 1;
  double c0, c1, c2, c3; cs_around(E, ep, rate, Lam, t, k, &c0, &c1, &c2, &c3);
  double r = rate[et], inv = 1.0 / rate[et], nc;
  if (et != E - 1) {
    double tb = t, te = ep[k];
    if (r > 0) {
      num[et] = lme(-c2, -c3);
      denom[et] = log((tb + inv) - (te + inv) * exp(-c3 + c2)) - c2;
      nc = num[et];
    } else { num[et] = log_0; denom[et] = log_0; nc = log_0; }
    for (int e = et + 1; e < E; e++) { num[e] = A[e]; denom[e] = B[e]; nc = lse(nc, num[e]); }
  } else {
    num[et] = -c2;
    denom[et] = log(t + inv) - c2;
    nc = num[et];
  }
  if (!bad(nc)) {
    double integ = 1.0;
    int e;
    for (e = 0; e < et; e++) { num[e] = 0.0; denom[e] = ep[e + 1] - ep[e]; }
    for (; e < E - 1; e++) {
      num[e] -= nc; denom[e] -= nc;
      num[e] = exp(num[e]);
      if (integ > 0.0) integ -= num[e]; else integ = 0.0;
      denom[e] = exp(denom[e]);
      denom[e] += -ep[e] * num[e] + (ep[e + 1] - ep[e]) * integ;
      if (denom[e] < 0.0) denom[e] = 0.0;
    }
    e = E - 1;
    num[e] -= nc; denom[e] -= nc;
    num[e] = exp(num[e]); denom[e] = exp(denom[e]);
    denom[e] -= ep[e] * num[e];
    if (denom[e] < 0.0) denom[e] = 0.0;
  } else {
    nc = 0.0;
    for (int e = 0; e < E; e++) { num[e] = 0; denom[e] = 0; }
  }
  return nc;
}

/* convenience for E-step parity tests: builds A/B like the coal_EM ctor, then one call */
double oracle_estep(int shared, int E, const double* ep, const double* rate, double t, double* num, double* denom)
{
  double A[ORACLE_MAX_E], B[ORACLE_MAX_E], Lam[ORACLE_MAX_E];
  if (E > ORACLE_MAX_E) return NAN;
  oracle_get_AB(E, ep, rate, A, B, Lam);
  return shared ? oracle_em_shared(E, ep, rate, A, B, Lam, t, num, denom)
                : oracle_em_notshared(E, ep, rate, A, B, Lam, t, num, denom);
}

/* EM driver for one replicate, coal.cpp:3675-3827 with regularise==2.
 * counts: [2][185]; rates_out[E]; returns the `iter` printed at coal.cpp:3823 (the index
 * of the last iteration), or max_iter if the cap is hit.  *final_ll = last log-likelihood. */
int oracle_em_run(int E, const double* ep, const double* rates_init, const double* age_bin,
                  const double* counts, int max_iter, double* rates_out, double* final_ll)
{
  double rate[ORACLE_MAX_E], num[ORACLE_MAX_E], denom[ORACLE_MAX_E], tn[ORACLE_MAX_E], td[ORACLE_MAX_E], A[ORACLE_MAX_E], B[ORACLE_MAX_E],
      Lam[ORACLE_MAX_E];
  if (E > ORACLE_MAX_E) return -1;
  const double* S = counts; const double* N = counts + NBINS;
  for (int e = 0; e < E; e++) { rate[e] = rates_init[e]; tn[e] = 0; td[e] = 0; num[e] = 0; denom[e] = 0; }
  double ll = log(0.0), prev;
  int iter;
  for (iter = 0; iter < max_iter; iter++) {
    oracle_get_AB(E, ep, rate, A, B, Lam);          /* coal.cpp:3698 */
    prev = ll; ll = 0.0;
    for (int bin = 0; bin < NBINS; bin++) {         /* coal.cpp:3704-3733 */
      if (S[bin] > 0) {
        double c = S[bin];
        double logl = oracle_em_shared(E, ep, rate, A, B, Lam, age_bin[bin], num, denom);
        ll += c * logl;
        for (int e = 0; e < E; e++) { tn[e] += c * num[e]; td[e] += c * denom[e]; }
      }
      if (N[bin] > 0) {
        double c = N[bin];
        double logl = oracle_em_notshared(E, ep, rate, A, B, Lam, age_bin[bin], num, denom);
        ll += c * logl;
        for (int e = 0; e < E; e++) { tn[e] += c * num[e]; td[e] += c * denom[e]; }
      }
    }
    for (int e = 0; e < E; e++) {                   /* M-step, coal.cpp:3771-3815 */
      if (tn[e] == 0) rate[e] = (e > 0) ? rate[e - 1] : 0;
      else if (td[e] == 0) { }
      else { rate[e] = tn[e] / td[e]; if (rate[e] < 5e-9) rate[e] = 5e-9; }
    }
    for (int e = 0; e < E; e++) { tn[e] = 0; td[e] = 0; }
    if ((ll / prev > 1.0 - 1e-7) & (iter > 1e3)) break;   /* coal.cpp:3822 */
  }
  for (int e = 0; e < E; e++) rates_out[e] = rate[e];
  *final_ll = ll;
  return iter;
}

/* ------------------------------------------------------------------------------------
 * .coal text, coal.cpp:3660-3672 + 3830-3844.  ostream default formatting of a double
 * (precision 6, no flags) is printf("%g").  rates: [R][E] (modified copy is not made:
 * for ancient samples the caller's rates[0..ep_null] are zeroed, as coal.cpp:3832-3834).
 * ---------------------------------------------------------------------------------- */
int oracle_write_coal(const char* path, int R, int E, const double* epochs, double* rates,
                      int is_ancient, int ep_null)
{
  FILE* f = fopen(path, "w");
  if (!f) return -1;
  fprintf(f, "0\n");
  if (is_ancient) { fprintf(f, "0 "); for (int e = ep_null + 1; e < E; e++) fprintf(f, "%g ", epochs[e]); }
  else { for (int e = 0; e < E; e++) fprintf(f, "%g ", epochs[e]); }
  fprintf(f, "\n");
  for (int i = 0; i < R; i++) {
    double* r = rates + (size_t)i * E;
    fprintf(f, "0 %d ", i);
    if (is_ancient) {
      for (int j = 0; j <= ep_null; j++) r[j] = 0;
      for (int e = ep_null; e < E; e++) fprintf(f, "%g ", r[e]);
    } else {
      for (int e = 0; e < E; e++) fprintf(f, "%g ", r[e]);
    }
    fprintf(f, "\n");
  }
  fclose(f);
  return 0;
}

/* the host libm itself, for pinning the device's glibc-exact exp/log/log1p (which = 0,1,2) */
void oracle_libm(int which, int n, const double* x, double* y)
{
  for (int i = 0; i < n; i++) y[i] = which == 0 ? exp(x[i]) : which == 1 ? log(x[i]) : log1p(x[i]);
}
