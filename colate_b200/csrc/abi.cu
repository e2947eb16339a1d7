// C-ABI glue (include/colate_b200.h): handle management, uploads, stage drivers.
#include "device.cuh"
#include "glibc_math.cuh"

#include <algorithm>
#include <random>
#include <cmath>
#include <cstdlib>
#include <cstring>

using namespace colate;

namespace {

int copy_in(void* dst, const void* src, size_t bytes, int location, cudaStream_t s)
{
  if (bytes == 0) return 0;
  CK(cudaMemcpyAsync(dst, src, bytes, location ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
  return 0;
}

int ensure_tables(colate_handle* h)
{
  if (h->thr_ready) return 0;
  double thr[NTHR], ab[NBINS];
  if (!bin_thresholds(thr)) return fail(COLATE_ERR_ARG, "host libm log() is not monotone around an age-bin threshold");
  colate_age_bins(ab);
  CK(h->thr10.ensure(sizeof thr));
  CK(h->d_agebin.ensure(sizeof ab));
  static double thrA[NBINS + 2], thrP[192];
  static uint16_t lut[LUT_N];
  if (!age_thresholds(thrA, thrP, lut)) return fail(COLATE_ERR_ARG, "host libm log() is not monotone around an age-bin threshold");
  CK(h->thrA.ensure(sizeof thrP));
  CK(h->lut.ensure(sizeof lut + 16));
  CK(cudaMemcpyAsync(h->thrA.p, thrP, sizeof thrP, cudaMemcpyHostToDevice, h->stream));  // slot-indexed thresholds
  CK(cudaMemcpyAsync(h->lut.p, lut, sizeof lut, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->thr10.p, thr, sizeof thr, cudaMemcpyHostToDevice, h->stream));
  h->thr185 = thr[NBINS];
  CK(cudaMemcpyAsync(h->d_agebin.p, ab, sizeof ab, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  memcpy(h->h_agebin, ab, sizeof ab);
  h->thr_ready = true;
  return 0;
}

// Does this host's libm compute exp/log/log1p exactly like the glibc_math.cuh port (i.e. is it
// glibc 2.39 with the FMA variants selected)?  If so the device EM is bit-identical to the
// reference run on this host; if not it is bit-identical to the reference on a glibc-2.39/FMA host.
int libm_self_check()
{
  static int cached = -1;
  if (cached >= 0) return cached;
  glm::Tables T{glm::hEXP_TAB, glm::hLOG_TAB};
  std::mt19937_64 g(12345);
  std::uniform_real_distribution<double> U(0, 1);
  auto same = [](double a, double b) { return (std::isnan(a) && std::isnan(b)) || !memcmp(&a, &b, 8); };
  int ok = 1;
  for (int i = 0; i < 200000 && ok; i++) {
    double x = (i & 1) ? -U(g) * 760 : (U(g) - 0.5) * 40;
    double y = std::exp((U(g) - 0.5) * ((i & 2) ? 1400 : 1));
    double z = (i & 1) ? -std::exp(-U(g) * 700) : std::exp(-U(g) * 700);
    if (!same(std::exp(x), glm::exp(x, T)) || !same(std::log(y), glm::log(y, T)) || !same(std::log1p(z), glm::log1p(z))) ok = 0;
  }
  cached = ok;
  return ok;
}

// New site arrays are in place (colate_set_sites / colate_ingest_end): every genome's chromosome ranges, join and mask
// refer to the previous site axis and --chr list, so all slots go back to "not set"; the order check of the
// sites is queued (its verdict is read by colate_stage1_flags: COLATE_ERR_ORDER).
int sites_replaced(colate_handle* h)
{
  int rc0 = ensure_tables(h);
  if (rc0) return rc0;
  h->sites_set = true;
  h->flags_done = false;
  h->tiles_valid = false;
  for (auto& g : h->genomes) { g.set = false; g.joined = false; g.has_mask = false; }
  CK(h->order_flag.ensure((1 + COLATE_MAX_GENOMES) * 4));
  CK(cudaMemsetAsync(h->order_flag.p, 0, (1 + COLATE_MAX_GENOMES) * 4, h->stream));
  return run_check_sites(h);
}
int genome_replaced(colate_handle* h, int slot)
{
  GenomeDev& g = h->genomes[slot];
  g.set = true;
  g.joined = false;
  h->flags_done = false;
  CK(cudaMemsetAsync(h->order_flag.as<int>() + 1 + slot, 0, 4, h->stream));
  return run_check_genome(h, slot);
}

int pick_chunk_log2(int64_t n_used)
{
  if (const char* e = getenv("COLATE_CHUNK_LOG2")) return std::max(0, std::min(30, atoi(e)));
  // ~2 generator chunks per SM: a jump costs as much shared-memory traffic as generating ~1 M words,
  // while fewer than ~300 sequential chunks leave the generator latency-bound (measured optimum on B200)
  int64_t per = (n_used + 295) / 296;   // (296 = 2 x 148 SMs; the optimum is flat around it)
  int k = 0;
  while ((int64_t(1) << k) < per) k++;
  return std::max(3, std::min(k, 24));
}

}  // namespace

namespace colate {
int sites_replaced_ext(colate_handle* h) { return sites_replaced(h); }
int genome_replaced_ext(colate_handle* h, int slot) { return genome_replaced(h, slot); }
}

extern "C" {

int colate_create(int device, colate_handle** out)
{
  if (!out) return fail(COLATE_ERR_ARG, "out is null");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(COLATE_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) + " (there is no CPU fallback)");
  if (device < 0 || device >= ndev) return fail(COLATE_ERR_ARG, "device index out of range");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(COLATE_ERR_CUDA, "device is not sm_100 (kernels are built for sm_100a only)");
  colate_handle* h = new colate_handle();
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  cudaError_t ce = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking);
  if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking);
  for (auto& ev : h->ev) if (ce == cudaSuccess) ce = cudaEventCreate(&ev);
  if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&h->copy_done, cudaEventDisableTiming);
  if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&h->side_done, cudaEventDisableTiming);
  if (ce != cudaSuccess) {   // nothing half-built leaves this function
    colate_destroy(h);
    return fail(COLATE_ERR_CUDA, std::string("colate_create: ") + cudaGetErrorString(ce));
  }
  *out = h;
  return 0;
}

void colate_destroy(colate_handle* h)
{
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
  if (h->side_stream) cudaStreamSynchronize(h->side_stream);
  if (h->em_stream) { cudaStreamSynchronize(h->em_stream); cudaStreamDestroy(h->em_stream); }
  DevBuf* bufs[] = {&h->site_off, &h->pos, &h->ab, &h->ae, &h->meta, &h->candR, &h->candT, &h->use, &h->word_rank, &h->scan_tmp, &h->row_of_rank,
                    &h->chr_used, &h->chr_blocks, &h->chr_block_base, &h->misc, &h->u_hdr, &h->u_eb2, &h->u_ews, &h->u_ewn, &h->u_cnt,
                    &h->u_blk, &h->blk_rank_start, &h->out_f, &h->out_n, &h->thrA, &h->lut, &h->d_scratch, &h->d_prof, &h->libm_tab, &h->ing_text, &h->ing_tile_cnt, &h->ing_tile_off, &h->ing_nl, &h->ing_status, &h->ing_fb,
                    &h->windows, &h->rng_stream, &h->mt_tail, &h->poly, &h->thr10, &h->d_counts, &h->d_blockstats, &h->d_weights, &h->d_epochs,
                    &h->d_rates, &h->d_iters, &h->d_ll, &h->d_agebin, &h->d_tmp, &h->d_em_scratch, &h->d_gr_tab, &h->d_gr_rates, &h->order_flag, &h->ing_raw, &h->deep_rows, &h->tile_start, &h->tile_rlo};
  for (DevBuf* b : bufs) b->release();
  for (auto& g : h->genomes) {
    DevBuf* gb[] = {&g.bp, &g.aaf, &g.daf, &g.alleles, &g.chr_first, &g.chr_end, &g.mask_bits, &g.j_aaf, &g.j_daf, &g.j_prevbp, &g.j_flag, &g.pile};
    for (DevBuf* b : gb) b->release();
  }
  for (int k = 0; k < 2; k++) if (h->ing_bounce[k]) { cudaFreeHost(h->ing_bounce[k]); cudaEventDestroy(h->ing_bounce_ev[k]); }
  for (auto& ev : h->ev) if (ev) cudaEventDestroy(ev);
  for (auto& ev : h->ing_evs) cudaEventDestroy(ev);
  if (h->copy_done) cudaEventDestroy(h->copy_done);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->side_done) cudaEventDestroy(h->side_done);
  if (h->side_stream) cudaStreamDestroy(h->side_stream);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

void* colate_stream(colate_handle* h) { return h ? (void*)h->stream : nullptr; }

int colate_set_stream_cache(colate_handle* h, int enable)
{
  if (!h) return fail(COLATE_ERR_ARG, "colate_set_stream_cache: null handle");
  h->stream_cache_on = enable != 0;
  h->sc_valid = false;
  return 0;
}

int colate_set_sites(colate_handle* h, int n_chr, const int64_t* site_off, const int32_t* pos, const float* age_begin,
                     const float* age_end, const uint32_t* meta, int location)
{
  // n_chr == 0 (site_off = {0}) is legal: a rank of a chromosome-sharded job that owns no chromosome still takes
  // part in every exchange with zero used rows and zero blocks
  if (!h || n_chr < 0 || !site_off) return fail(COLATE_ERR_ARG, "colate_set_sites: bad arguments");
  CK(cudaSetDevice(h->device));
  std::vector<int64_t> off(n_chr + 1);
  if (location) CK(cudaMemcpy(off.data(), site_off, (n_chr + 1) * 8, cudaMemcpyDeviceToHost));
  else memcpy(off.data(), site_off, (n_chr + 1) * 8);
  if (off[0] != 0) return fail(COLATE_ERR_ARG, "site_off[0] must be 0");
  for (int c = 0; c < n_chr; c++) if (off[c + 1] < off[c]) return fail(COLATE_ERR_ARG, "site_off must be non-decreasing");
  const int64_t n = off[n_chr];
  if (n >= (int64_t(1) << 31)) return fail(COLATE_ERR_ARG, "more than 2^31 rows per handle");
  CK(h->site_off.ensure((n_chr + 1) * 8)); CK(h->pos.ensure(n * 4 + 4)); CK(h->ab.ensure(n * 4 + 4));
  CK(h->ae.ensure(n * 4 + 4)); CK(h->meta.ensure(n * 4 + 4));
  h->h_site_off = off;   // (the async copy below reads the handle's copy, not the local)
  CK(cudaMemcpyAsync(h->site_off.p, h->h_site_off.data(), (n_chr + 1) * 8, cudaMemcpyHostToDevice, h->stream));
  int rc;
  if ((rc = copy_in(h->pos.p, pos, n * 4, location, h->stream))) return rc;
  if ((rc = copy_in(h->ab.p, age_begin, n * 4, location, h->stream))) return rc;
  if ((rc = copy_in(h->ae.p, age_end, n * 4, location, h->stream))) return rc;
  if ((rc = copy_in(h->meta.p, meta, n * 4, location, h->stream))) return rc;
  h->n_chr = n_chr;
  h->n_site = n;
  if ((rc = sites_replaced(h))) return rc;
  if (!h->opt_async_uploads) CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int colate_set_genome(colate_handle* h, int slot, int64_t n_rec, const int64_t* chr_first, const int64_t* chr_end,
                      const int32_t* bp, const int32_t* aaf, const int32_t* daf, const uint16_t* alleles, int location)
{
  if (!h || slot < 0 || slot >= COLATE_MAX_GENOMES || n_rec < 0) return fail(COLATE_ERR_ARG, "colate_set_genome: bad arguments");
  if (!h->sites_set) return fail(COLATE_ERR_STATE, "colate_set_genome: call colate_set_sites first");
  CK(cudaSetDevice(h->device));
  GenomeDev& g = h->genomes[slot];
  const int nc = h->n_chr;
  CK(g.bp.ensure(n_rec * 4 + 4)); CK(g.aaf.ensure(n_rec * 4 + 4)); CK(g.daf.ensure(n_rec * 4 + 4)); CK(g.alleles.ensure(n_rec * 2 + 4));
  CK(g.chr_first.ensure(nc * 8)); CK(g.chr_end.ensure(nc * 8));
  int rc;
  if ((rc = copy_in(g.chr_first.p, chr_first, nc * 8, location, h->stream))) return rc;
  if ((rc = copy_in(g.chr_end.p, chr_end, nc * 8, location, h->stream))) return rc;
  if ((rc = copy_in(g.bp.p, bp, n_rec * 4, location, h->stream))) return rc;
  if ((rc = copy_in(g.aaf.p, aaf, n_rec * 4, location, h->stream))) return rc;
  if ((rc = copy_in(g.daf.p, daf, n_rec * 4, location, h->stream))) return rc;
  if ((rc = copy_in(g.alleles.p, alleles, n_rec * 2, location, h->stream))) return rc;
  g.n_rec = n_rec;
  g.pileup = false;
  if ((rc = genome_replaced(h, slot))) return rc;
  if (!h->opt_async_uploads) CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int colate_set_pileup(colate_handle* h, int slot, const int32_t* counts, int location)
{
  if (!h || slot < 0 || slot >= COLATE_MAX_GENOMES || !counts) return fail(COLATE_ERR_ARG, "colate_set_pileup: bad arguments");
  if (!h->sites_set) return fail(COLATE_ERR_STATE, "colate_set_pileup: call colate_set_sites first");
  CK(cudaSetDevice(h->device));
  GenomeDev& g = h->genomes[slot];
  CK(g.pile.ensure((size_t)h->n_site * 16 + 16));
  int rc;
  if ((rc = copy_in(g.pile.p, counts, (size_t)h->n_site * 16, location, h->stream))) return rc;
  g.n_rec = 0;
  g.pileup = true;
  g.set = true;
  g.joined = false;
  h->flags_done = false;
  CK(cudaMemsetAsync(h->order_flag.as<int>() + 1 + slot, 0, 4, h->stream));   // no record stream, nothing to be out of order
  if (!h->opt_async_uploads) CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int colate_set_row_counts(colate_handle* h, int slot, const int32_t* aaf, const int32_t* daf, int location)
{
  if (!h || slot < 0 || slot >= COLATE_MAX_GENOMES || !aaf || !daf) return fail(COLATE_ERR_ARG, "colate_set_row_counts: bad arguments");
  if (!h->sites_set) return fail(COLATE_ERR_STATE, "colate_set_row_counts: call colate_set_sites first");
  CK(cudaSetDevice(h->device));
  GenomeDev& g = h->genomes[slot];
  const size_t n = (size_t)h->n_site;
  CK(g.pile.ensure(n * 16 + 16));
  const int32_t *da = aaf, *dd = daf;
  if (!location) {
    CK(h->d_tmp.ensure(n * 8 + 16));
    CK(cudaMemcpyAsync(h->d_tmp.p, aaf, n * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_tmp.as<int32_t>() + n, daf, n * 4, cudaMemcpyHostToDevice, h->stream));
    da = h->d_tmp.as<int32_t>();
    dd = da + n;
  }
  int rc = run_pack_row_counts(h, slot, da, dd);
  if (rc) return rc;
  g.n_rec = 0;
  g.pileup = true;
  g.set = true;
  g.joined = false;
  h->flags_done = false;
  CK(cudaMemsetAsync(h->order_flag.as<int>() + 1 + slot, 0, 4, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

// ---- pileup from decoded reads (the counting loop of bam_parser, include/vcf/htslib.cpp:60-168, on the device) -----------------
int colate_pileup_begin(colate_handle* h, int slot)
{
  if (!h || slot < 0 || slot >= COLATE_MAX_GENOMES) return fail(COLATE_ERR_ARG, "colate_pileup_begin: bad arguments");
  if (!h->sites_set) return fail(COLATE_ERR_STATE, "colate_pileup_begin: call colate_set_sites first");
  CK(cudaSetDevice(h->device));
  GenomeDev& g = h->genomes[slot];
  CK(g.pile.ensure((size_t)h->n_site * 16 + 16));
  CK(cudaMemsetAsync(g.pile.p, 0, (size_t)h->n_site * 16, h->stream));
  g.set = false;
  g.pileup = false;
  g.joined = false;
  h->flags_done = false;
  return 0;
}

int colate_pileup_reads(colate_handle* h, int slot, int chr_index, int64_t n_reads, const int32_t* pos, const uint8_t* mapq, const int32_t* len,
                        const int64_t* seq_off, const uint8_t* seq, const uint8_t* qual, const uint8_t* ref_seq, int64_t ref_len,
                        int mapq_th, int len_th, int mismatch_th)
{
  if (!h || slot < 0 || slot >= COLATE_MAX_GENOMES || n_reads < 0 || (n_reads > 0 && (!pos || !mapq || !len || !seq_off || !seq || !qual || !ref_seq)))
    return fail(COLATE_ERR_ARG, "colate_pileup_reads: bad arguments");
  if (!h->sites_set || chr_index < 0 || chr_index >= h->n_chr) return fail(COLATE_ERR_ARG, "colate_pileup_reads: no such chromosome in the site set");
  if (h->genomes[slot].pile.cap < (size_t)h->n_site * 16) return fail(COLATE_ERR_STATE, "colate_pileup_reads: call colate_pileup_begin first");
  if (n_reads == 0) return 0;
  CK(cudaSetDevice(h->device));
  int max_len = 0;
  int64_t n_bytes = 0;
  for (int64_t k = 0; k < n_reads; k++) {
    if (len[k] < 0 || seq_off[k] < 0) return fail(COLATE_ERR_ARG, "colate_pileup_reads: negative read length / offset");
    if (k > 0 && pos[k] < pos[k - 1]) return fail(COLATE_ERR_ORDER, "Error: BAM file not sorted by position.");   // htslib.cpp:411-414
    max_len = std::max(max_len, len[k]);
    n_bytes = std::max<int64_t>(n_bytes, seq_off[k] + len[k]);
  }
  cudaStream_t s = h->stream;
  // one staging buffer: pos | len | off | mapq | seq | qual | ref | pass
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t o_pos = 0, o_len = o_pos + up(n_reads * 4), o_off = o_len + up(n_reads * 4), o_mq = o_off + up(n_reads * 8),
               o_seq = o_mq + up(n_reads), o_q = o_seq + up(n_bytes), o_ref = o_q + up(n_bytes), o_pass = o_ref + up(ref_len),
               total = o_pass + up(n_reads);
  CK(h->d_tmp.ensure(total));
  char* d = h->d_tmp.as<char>();
  CK(cudaMemcpyAsync(d + o_pos, pos, n_reads * 4, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d + o_len, len, n_reads * 4, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d + o_off, seq_off, n_reads * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d + o_mq, mapq, n_reads, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d + o_seq, seq, n_bytes, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d + o_q, qual, n_bytes, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d + o_ref, ref_seq, ref_len, cudaMemcpyHostToDevice, s));
  int rc = run_pileup_reads(h, slot, chr_index, n_reads, (const int32_t*)(d + o_pos), (const uint8_t*)(d + o_mq), (const int32_t*)(d + o_len),
                            (const int64_t*)(d + o_off), (const uint8_t*)(d + o_seq), (const uint8_t*)(d + o_q), (const uint8_t*)(d + o_ref), ref_len,
                            max_len, mapq_th, len_th, mismatch_th, (uint8_t*)(d + o_pass));
  if (rc) return rc;
  CK(cudaStreamSynchronize(s));      // the caller's buffers and the staging buffer are free again
  return 0;
}

int colate_pileup_end(colate_handle* h, int slot, int32_t* counts_out)
{
  if (!h || slot < 0 || slot >= COLATE_MAX_GENOMES) return fail(COLATE_ERR_ARG, "colate_pileup_end: bad arguments");
  GenomeDev& g = h->genomes[slot];
  if (!h->sites_set || g.pile.cap < (size_t)h->n_site * 16) return fail(COLATE_ERR_STATE, "colate_pileup_end: call colate_pileup_begin first");
  CK(cudaSetDevice(h->device));
  if (counts_out) CK(cudaMemcpyAsync(counts_out, g.pile.p, (size_t)h->n_site * 16, cudaMemcpyDeviceToHost, h->stream));
  g.n_rec = 0;
  g.pileup = true;
  g.set = true;
  g.joined = false;
  h->flags_done = false;
  CK(cudaMemsetAsync(h->order_flag.as<int>() + 1 + slot, 0, 4, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int colate_set_mask(colate_handle* h, int slot, const uint32_t* pass_bits, int location)
{
  if (!h || slot < 0 || slot >= COLATE_MAX_GENOMES) return fail(COLATE_ERR_ARG, "colate_set_mask: bad arguments");
  if (!h->sites_set) return fail(COLATE_ERR_STATE, "colate_set_mask: call colate_set_sites first");
  CK(cudaSetDevice(h->device));
  GenomeDev& g = h->genomes[slot];
  h->flags_done = false;
  if (!pass_bits) { g.has_mask = false; return 0; }
  const int64_t nw = (h->n_site + 31) / 32;
  CK(g.mask_bits.ensure(nw * 4 + 4));
  int rc;
  if ((rc = copy_in(g.mask_bits.p, pass_bits, nw * 4, location, h->stream))) return rc;
  if (!h->opt_async_uploads) CK(cudaStreamSynchronize(h->stream));
  g.has_mask = true;
  return 0;
}

int colate_stage1_flags(colate_handle* h, int target_slot, int reference_slot, int64_t* n_used_chr, int32_t* n_blocks_chr)
{
  if (!h || target_slot < 0 || target_slot >= COLATE_MAX_GENOMES || reference_slot < 0 || reference_slot >= COLATE_MAX_GENOMES)
    return fail(COLATE_ERR_ARG, "colate_stage1_flags: bad arguments");
  if (!h->sites_set || !h->genomes[target_slot].set || !h->genomes[reference_slot].set)
    return fail(COLATE_ERR_STATE, "colate_stage1_flags: sites / genomes not set");
  CK(cudaSetDevice(h->device));
  int rc = ensure_tables(h);
  if (rc) return rc;
  cudaStream_t s = h->stream;
  if (h->opt_rejoin) for (auto& g : h->genomes) g.joined = false;
  CK(cudaEventRecord(h->ev[0], s));
  if ((rc = run_join(h, reference_slot))) return rc;
  if ((rc = run_join(h, target_slot))) return rc;
  CK(cudaEventRecord(h->ev[1], s));
  if ((rc = run_flags(h, target_slot, reference_slot))) return rc;
  CK(cudaEventRecord(h->ev[3], s));
  h->h_chr_used.resize(h->n_chr);
  h->h_chr_blocks.resize(h->n_chr);
  int64_t misc[8];
  int order[1 + COLATE_MAX_GENOMES];
  if (h->n_chr > 0) {
    CK(cudaMemcpyAsync(h->h_chr_used.data(), h->chr_used.p, h->n_chr * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(h->h_chr_blocks.data(), h->chr_blocks.p, h->n_chr * 4, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaMemcpyAsync(misc, h->misc.p, 64, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(order, h->order_flag.p, sizeof order, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (order[0]) return fail(COLATE_ERR_ORDER, "positions of a .mut file are not ascending (the reference's sequential reader needs sorted input)");
  if (order[1 + target_slot] || order[1 + reference_slot])
    return fail(COLATE_ERR_ORDER, "positions of a .colate.in file are not ascending within a chromosome");
  h->n_used = misc[0];
  h->n_blocks_local = (int)misc[1];
  h->n_deep = misc[4];
  if (h->opt_raw_weights && h->n_deep > 0)
    return fail(COLATE_ERR_AGE_RANGE, "a used row with age_begin > 0 has an age interval beyond the age grid: the bcf / bam front-ends write past the end "
                                      "of the histogram there (coal.cpp:2034-2039 has no bound check, unlike the tmp/tmp path's coal.cpp:2289)");
  if (misc[3])
    return fail(COLATE_ERR_AGE_RANGE, "a used row cannot be processed by the reference either: age_begin <= 0 with an age interval beyond "
                                      "the age grid (~9.3e6 generations; out-of-bounds write at coal.cpp:2269), or age_begin itself beyond it "
                                      "(the rejection loop of coal.cpp:2279-2294 never ends)");
  h->tgt_slot = target_slot;
  h->ref_slot = reference_slot;
  h->flags_done = true;
  h->sampled = false;
  if (n_used_chr) memcpy(n_used_chr, h->h_chr_used.data(), h->n_chr * 8);
  if (n_blocks_chr) memcpy(n_blocks_chr, h->h_chr_blocks.data(), h->n_chr * 4);
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]); h->timing.join_ms = ms;
  cudaEventElapsedTime(&ms, h->ev[1], h->ev[3]); h->timing.flags_ms = ms;
  h->timing.n_site = h->n_site;
  h->timing.n_used = h->n_used;
  return 0;
}

// Rows with age_begin > 0 whose age interval reaches past the age grid (h->n_deep of them, coal.cpp:2279-2294): every draw
// whose bin reaches 185 is redrawn, so such a row consumes 200 + 2 * redraws engine words and every later row starts that
// much later in the stream.  The redraw count depends on the stream itself, hence strictly in row order: the used rows are
// cut into the runs BETWEEN deep rows; a run is sampled by the normal kernels from the generator state in front of it (no
// long jump: the state is carried along), the deep row in between is walked on the host (it is one row: ~100 + redraws draws).
// The exact replay then sees ordinary count rows.  win: state window in front of the first row, advanced to behind the last.
static int sample_segmented(colate_handle* h, uint32_t* win)
{
  cudaStream_t s = h->stream;
  const int64_t nu = h->n_used, nd = h->n_deep;
  std::vector<int64_t> deep((size_t)nd);
  int64_t misc[8];
  CK(cudaMemcpyAsync(misc, h->misc.p, 64, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(deep.data(), h->deep_rows.p, (size_t)nd * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (misc[5] != nd) return fail(COLATE_ERR_STATE, "rejection-sampling rows: the flag pass and the compaction disagree");
  std::sort(deep.begin(), deep.end());
  CK(cudaMemsetAsync(h->u_cnt.p, 0, (size_t)((nu + 31) / 32) * 32 * 192, s));
  h->extra_words = 0;
  int64_t r = 0;
  for (int64_t k = 0; k <= nd; k++) {
    const int64_t f = k < nd ? deep[(size_t)k] : nu;
    const int64_t len = f - r;
    if (len > 0) {
      uint32_t* stream_local = nullptr;
      uint32_t after[COLATE_MT_WORDS];
      int rc = run_mt_stream(h, win, 0, 200 * len, pick_chunk_log2(len), &stream_local, after, true);
      if (rc) return rc;
      if ((rc = run_sample_rows(h, stream_local, r, len))) return rc;
      CK(cudaStreamSynchronize(s));     // the stream buffer and the scratch tiles are reused by the next run
      memcpy(win, after, sizeof after);
    }
    if (f < nu) {
      double hdr[4];
      CK(cudaMemcpy(hdr, h->u_hdr.as<double>() + 4 * f, 32, cudaMemcpyDeviceToHost));
      uint8_t cnt[192];
      const int64_t redraws = sample_deep_row_host(win, hdr[1], hdr[0] * 0x1p64, cnt, (int64_t)1 << 26);
      if (redraws < 0)
        return fail(COLATE_ERR_AGE_RANGE, "a row's age interval lies almost entirely beyond the age grid: more than 2^26 redraws (coal.cpp:2279-2294)");
      h->extra_words += 2 * redraws;
      int rc = run_put_count_row(h, f, cnt);
      if (rc) return rc;
    }
    r = f + 1;
  }
  return 0;
}

int colate_stage1_sample(colate_handle* h, const uint32_t* mt_state, int64_t used_rank_base, int block_base,
                         double* block_stats, int64_t* block_tallies, uint32_t* mt_state_out)
{
  if (!h || !mt_state || used_rank_base < 0 || block_base < 0) return fail(COLATE_ERR_ARG, "colate_stage1_sample: bad arguments");
  if (!h->flags_done) return fail(COLATE_ERR_STATE, "colate_stage1_sample: call colate_stage1_flags first");
  if (block_base + h->n_blocks_local > MAX_BLOCKS) return fail(COLATE_ERR_BLOCKS, "more than 500 genomic blocks");
  CK(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const int64_t nu = h->n_used;
  const int nb = h->n_blocks_local;
  uint32_t win_after[COLATE_MT_WORDS];
  int rc;
  h->extra_words = 0;
  if (h->n_deep == 0) {
    uint32_t* stream_local = nullptr;
    CK(cudaEventRecord(h->ev[6], s));
    if ((rc = run_mt_stream(h, mt_state, 200 * used_rank_base, 200 * nu, pick_chunk_log2(nu), &stream_local, nullptr, true))) return rc;
    CK(cudaEventRecord(h->ev[7], s));
    if ((rc = run_compact(h))) return rc;
    if ((rc = run_sample_rows(h, stream_local, 0, nu))) return rc;
  } else {
    // rejection-sampling rows present: runs between them in row order (sample_segmented)
    CK(cudaEventRecord(h->ev[6], s));
    uint32_t* dummy = nullptr;
    if ((rc = run_mt_stream(h, mt_state, 200 * used_rank_base, 0, 3, &dummy, win_after, true))) return rc;   // state in front of this handle's rows
    CK(cudaEventRecord(h->ev[7], s));
    if ((rc = run_compact(h))) return rc;
    if ((rc = sample_segmented(h, win_after))) return rc;
  }
  if ((rc = run_replay(h))) return rc;
  int64_t misc[8];
  CK(cudaMemcpyAsync(misc, h->misc.p, 64, cudaMemcpyDeviceToHost, s));
  // (host or device destinations: unified addressing resolves the direction)
  if (block_stats && nb > 0) CK(cudaMemcpyAsync(block_stats, h->out_f.p, (size_t)nb * 4 * NBINS * 8, cudaMemcpyDefault, s));
  if (block_tallies && nb > 0) CK(cudaMemcpyAsync(block_tallies, h->out_n.p, (size_t)nb * 3 * NBINS * 8, cudaMemcpyDefault, s));
  CK(cudaStreamSynchronize(s));
  h->sampled = true;
  if (misc[3]) return fail(COLATE_ERR_AGE_RANGE, "a used row has an age bin >= 185 (age_end beyond ~9.3e6 generations)");
  if (mt_state_out) {
    if (h->n_deep == 0) { if ((rc = mt_window_after(h, win_after))) return rc; }
    memcpy(mt_state_out, win_after, sizeof win_after);
  }
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev[6], h->ev[7]); h->timing.rng_ms = ms;
  cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]); h->timing.compact_ms = ms;
  cudaEventElapsedTime(&ms, h->ev[3], h->ev[4]); h->timing.sample_ms = ms;   // k_sample alone (with rejection-sampling rows: all the runs)
  cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]); h->timing.replay_ms = ms;
  h->timing.rng_words = 200 * nu + h->extra_words;
  h->timing.total_ms = h->timing.join_ms + h->timing.flags_ms + h->timing.rng_ms + h->timing.compact_ms + h->timing.sample_ms +
                       h->timing.replay_ms;
  return 0;
}


int colate_stage1(colate_handle* h, int target_slot, int reference_slot, const uint32_t* mt_state, int* num_blocks,
                  double* block_stats, int64_t* block_tallies, int64_t* n_used_total, uint32_t* mt_state_out)
{
  int rc = colate_stage1_flags(h, target_slot, reference_slot, nullptr, nullptr);
  if (rc) return rc;
  if (h->n_blocks_local > MAX_BLOCKS) return fail(COLATE_ERR_BLOCKS, "more than 500 genomic blocks");
  rc = colate_stage1_sample(h, mt_state, 0, 0, block_stats, block_tallies, mt_state_out);
  if (rc) return rc;
  if (num_blocks) *num_blocks = h->n_blocks_local;
  if (n_used_total) *n_used_total = h->n_used;
  return 0;
}

int colate_set_option(colate_handle* h, const char* key, int64_t value)
{
  if (!h || !key) return fail(COLATE_ERR_ARG, "null");
  if (!strcmp(key, "rejoin")) { h->opt_rejoin = value != 0; return 0; }
  // async_uploads = 1: colate_set_sites / colate_set_genome / colate_set_mask queue their copies and return; the
  // caller keeps the (pinned) host buffers unchanged until the next colate_stage1_flags() has returned
  if (!strcmp(key, "async_uploads")) { h->opt_async_uploads = value != 0; return 0; }
  // front_end: which of mut()'s input branches the handle reproduces (coal.cpp:3175-3319).  0 = tmp/tmp (parse_tmptmp: pseudo-
  // genotype weights, no normalisation).  1 = the bcf / bam front-ends fed from pre-decoded per-row counts (SURVEY.md 8f N3):
  // raw count weights (coal.cpp:2005-2039, 1164-1197) and both count vectors of stage ii divided by 1e3 (coal.cpp:3453-3463).
  if (!strcmp(key, "front_end")) {
    if (value != 0 && value != 1) return fail(COLATE_ERR_ARG, "front_end: 0 (tmp/tmp) or 1 (pre-decoded bcf / bam counts)");
    h->opt_raw_weights = h->opt_norm_1e3 = value == 1;
    h->flags_done = false;
    return 0;
  }
  return fail(COLATE_ERR_ARG, std::string("unknown option ") + key);
}

int64_t colate_launch_count(colate_handle* h) { return h ? h->launches : 0; }

int64_t colate_last_stage1_extra_words(colate_handle* h) { return h ? h->extra_words : 0; }

int colate_last_stage1_timing(colate_handle* h, colate_stage1_timing* out)
{
  if (!h || !out) return fail(COLATE_ERR_ARG, "null");
  *out = h->timing;
  return 0;
}

int colate_stage2_bootstrap(colate_handle* h, int R, int num_blocks, const int32_t* block_weights,
                            const double* block_stats, double age, double* counts)
{
  if (!h || R <= 0 || num_blocks <= 0 || num_blocks > MAX_BLOCKS || !block_weights)
    return fail(COLATE_ERR_ARG, "colate_stage2_bootstrap: bad arguments");
  if (h->em_inflight) return fail(COLATE_ERR_STATE, "colate_stage2_bootstrap: an EM is in flight on the counts (call colate_stage3_em_end first)");
  if (!block_stats && (!h->flags_done || !h->sampled || num_blocks != h->n_blocks_local))
    return fail(COLATE_ERR_STATE, "colate_stage2_bootstrap: no device-resident block histograms of this size (run colate_stage1 first)");
  CK(cudaSetDevice(h->device));
  int rc = ensure_tables(h);
  if (rc) return rc;
  double ab[NBINS];
  colate_age_bins(ab);
  if (!(age >= 0) || !(age < ab[NBINS - 1])) return fail(COLATE_ERR_ARG, "age outside the age grid");
  cudaStream_t s = h->stream;
  CK(h->d_weights.ensure((size_t)R * num_blocks * 4));
  CK(h->d_blockstats.ensure((size_t)num_blocks * 4 * NBINS * 8));
  CK(h->d_counts.ensure((size_t)R * 2 * NBINS * 8));
  CK(cudaMemcpyAsync(h->d_weights.p, block_weights, (size_t)R * num_blocks * 4, cudaMemcpyDefault, s));
  const double* blk = h->out_f.as<double>();   // NULL: what the last colate_stage1_sample left on the device (no bounce through the host)
  if (block_stats) {
    CK(cudaMemcpyAsync(h->d_blockstats.p, block_stats, (size_t)num_blocks * 4 * NBINS * 8, cudaMemcpyDefault, s));
    blk = h->d_blockstats.as<double>();
  }
  if ((rc = run_bootstrap(h, R, num_blocks, blk, age))) return rc;
  if (counts) CK(cudaMemcpyAsync(counts, h->d_counts.p, (size_t)R * 2 * NBINS * 8, cudaMemcpyDefault, s));
  CK(cudaStreamSynchronize(s));
  h->counts_R = R;
  return 0;
}

int colate_stage3_em(colate_handle* h, int R, int E, const double* epochs, const double* rates_init, const double* counts,
                     int max_iter, double* rates, int32_t* iters, double* final_ll)
{
  if (!h || R <= 0 || E < 2 || E > 1024 || !epochs || !rates_init || max_iter < 0)
    return fail(COLATE_ERR_ARG, "colate_stage3_em: bad arguments");
  if (!counts && h->counts_R != R) return fail(COLATE_ERR_STATE, "colate_stage3_em: no device-resident counts for this R");
  if (h->em_inflight) return fail(COLATE_ERR_STATE, "colate_stage3_em: an EM is in flight (colate_stage3_em_begin): call colate_stage3_em_end first");
  CK(cudaSetDevice(h->device));
  int rc = ensure_tables(h);
  if (rc) return rc;
  cudaStream_t s = h->stream;
  CK(h->d_epochs.ensure((size_t)E * 8));
  CK(h->d_rates.ensure((size_t)(R + 1) * E * 8));
  CK(h->d_iters.ensure((size_t)R * 4));
  CK(h->d_ll.ensure((size_t)R * 8));
  CK(cudaMemcpyAsync(h->d_epochs.p, epochs, (size_t)E * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_rates.p, rates_init, (size_t)E * 8, cudaMemcpyHostToDevice, s));
  if (counts) {
    CK(h->d_counts.ensure((size_t)R * 2 * NBINS * 8));
    CK(cudaMemcpyAsync(h->d_counts.p, counts, (size_t)R * 2 * NBINS * 8, cudaMemcpyDefault, s));
    h->counts_R = R;
  }
  if ((rc = run_em(h, R, E, max_iter, epochs, s))) return rc;
  if (rates) CK(cudaMemcpyAsync(rates, h->d_rates.as<double>() + E, (size_t)R * E * 8, cudaMemcpyDefault, s));
  std::vector<int32_t> it_host((size_t)R);
  CK(cudaMemcpyAsync(it_host.data(), h->d_iters.p, (size_t)R * 4, cudaMemcpyDeviceToHost, s));
  if (iters) CK(cudaMemcpyAsync(iters, h->d_iters.p, (size_t)R * 4, cudaMemcpyDefault, s));
  if (final_ll) CK(cudaMemcpyAsync(final_ll, h->d_ll.p, (size_t)R * 8, cudaMemcpyDefault, s));
  CK(cudaStreamSynchronize(s));
  for (int r = 0; r < R; r++)
    if (it_host[r] < 0) return fail(COLATE_ERR_CUDA, "EM kernel: the cluster handshake timed out (replicate " + std::to_string(r) + ")");
  return 0;
}

// ---- asynchronous form: one EM in flight per handle ---------------------------------------------------------------------
int colate_stage3_em_begin(colate_handle* h, int R, int E, const double* epochs, const double* rates_init, int max_iter)
{
  if (!h || R <= 0 || E < 2 || E > 1024 || !epochs || !rates_init || max_iter < 0)
    return fail(COLATE_ERR_ARG, "colate_stage3_em_begin: bad arguments");
  if (h->counts_R != R) return fail(COLATE_ERR_STATE, "colate_stage3_em_begin: no device-resident counts for this R (run colate_stage2_bootstrap first)");
  if (h->em_inflight) return fail(COLATE_ERR_STATE, "colate_stage3_em_begin: an EM is already in flight on this handle");
  CK(cudaSetDevice(h->device));
  int rc = ensure_tables(h);
  if (rc) return rc;
  if (!h->em_stream) CK(cudaStreamCreateWithFlags(&h->em_stream, cudaStreamNonBlocking));
  cudaStream_t s = h->em_stream;
  CK(h->d_epochs.ensure((size_t)E * 8));
  CK(h->d_rates.ensure((size_t)(R + 1) * E * 8));
  CK(h->d_iters.ensure((size_t)R * 4));
  CK(h->d_ll.ensure((size_t)R * 8));
  h->em_host_in.assign(epochs, epochs + E);
  h->em_host_in.insert(h->em_host_in.end(), rates_init, rates_init + E);
  CK(cudaMemcpyAsync(h->d_epochs.p, h->em_host_in.data(), (size_t)E * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_rates.p, h->em_host_in.data() + E, (size_t)E * 8, cudaMemcpyHostToDevice, s));
  // (the counts were left by colate_stage2_bootstrap, which returns only after its stream has drained)
  if ((rc = run_em(h, R, E, max_iter, epochs, s))) return rc;
  h->em_inflight = true;
  h->em_R = R;
  h->em_E = E;
  return 0;
}

int colate_stage3_em_end(colate_handle* h, double* rates, int32_t* iters, double* final_ll)
{
  if (!h) return fail(COLATE_ERR_ARG, "colate_stage3_em_end: null handle");
  if (!h->em_inflight) return fail(COLATE_ERR_STATE, "colate_stage3_em_end: no EM in flight");
  CK(cudaSetDevice(h->device));
  cudaStream_t s = h->em_stream;
  const int R = h->em_R, E = h->em_E;
  h->em_inflight = false;
  std::vector<int32_t> it_host((size_t)R);
  if (rates) CK(cudaMemcpyAsync(rates, h->d_rates.as<double>() + E, (size_t)R * E * 8, cudaMemcpyDefault, s));
  CK(cudaMemcpyAsync(it_host.data(), h->d_iters.p, (size_t)R * 4, cudaMemcpyDeviceToHost, s));
  if (iters) CK(cudaMemcpyAsync(iters, h->d_iters.p, (size_t)R * 4, cudaMemcpyDefault, s));
  if (final_ll) CK(cudaMemcpyAsync(final_ll, h->d_ll.p, (size_t)R * 8, cudaMemcpyDefault, s));
  CK(cudaStreamSynchronize(s));
  for (int r = 0; r < R; r++)
    if (it_host[r] < 0) return fail(COLATE_ERR_CUDA, "EM kernel: the cluster handshake timed out (replicate " + std::to_string(r) + ")");
  return 0;
}

// ---- mixed epoch grids: one k_em_cta_grids launch for every replicate whose grid fits it --------------------------------
int colate_stage3_em_grids(colate_handle* h, int R, const int32_t* grid_of, int n_grids, const int32_t* grid_E, const int64_t* grid_off,
                           const double* epochs, const double* rates_init, const double* counts, int max_iter, double* rates, int32_t* iters,
                           double* final_ll)
{
  if (!h || R <= 0 || n_grids <= 0 || !grid_of || !grid_E || !grid_off || !epochs || !rates_init || !counts || max_iter < 0 || !rates ||
      !iters || !final_ll)
    return fail(COLATE_ERR_ARG, "colate_stage3_em_grids: bad arguments");
  int E_max = 0;
  for (int g = 0; g < n_grids; g++) {
    if (grid_E[g] < 2 || grid_E[g] > 1024 || grid_off[g] < 0) return fail(COLATE_ERR_ARG, "colate_stage3_em_grids: bad grid " + std::to_string(g));
    E_max = std::max(E_max, (int)grid_E[g]);
  }
  for (int r = 0; r < R; r++)
    if (grid_of[r] < 0 || grid_of[r] >= n_grids) return fail(COLATE_ERR_ARG, "colate_stage3_em_grids: grid_of[" + std::to_string(r) + "] out of range");
  if (h->em_inflight) return fail(COLATE_ERR_STATE, "colate_stage3_em_grids: an EM is in flight (colate_stage3_em_begin): call colate_stage3_em_end first");
  CK(cudaSetDevice(h->device));
  int rc = ensure_tables(h);
  if (rc) return rc;
  constexpr int C2 = 2 * NBINS;
  std::vector<int> cap(n_grids, 0), fits(n_grids, 0);
  size_t smem = 0;
  int64_t ep_len = 0;
  for (int g = 0; g < n_grids; g++) {
    size_t sm = 0;
    fits[g] = em_cta_fits(h, grid_E[g], epochs + grid_off[g], &cap[g], &sm) ? 1 : 0;
    if (fits[g]) { smem = std::max(smem, sm); ep_len = std::max(ep_len, grid_off[g] + grid_E[g]); }
  }
  memset(rates, 0, (size_t)R * E_max * 8);
  auto put = [&](int r, const double* row, int E, int32_t it, double l) {
    memcpy(rates + (size_t)r * E_max, row, (size_t)E * 8);
    iters[r] = it;
    final_ll[r] = l;
  };
  // grids the throughput kernel does not fit (shared memory or thread bound): colate_stage3_em on each of them alone
  for (int g = 0; g < n_grids; g++) {
    if (fits[g]) continue;
    std::vector<int> reps;
    for (int r = 0; r < R; r++) if (grid_of[r] == g) reps.push_back(r);
    if (reps.empty()) continue;
    const int n = (int)reps.size(), E = grid_E[g];
    std::vector<double> cn((size_t)n * C2), rt((size_t)n * E), l2(n);
    std::vector<int32_t> it(n);
    for (int k = 0; k < n; k++) memcpy(cn.data() + (size_t)k * C2, counts + (size_t)reps[k] * C2, C2 * 8);
    if ((rc = colate_stage3_em(h, n, E, epochs + grid_off[g], rates_init + grid_off[g], cn.data(), max_iter, rt.data(), it.data(), l2.data())))
      return rc;
    for (int k = 0; k < n; k++) put(reps[k], rt.data() + (size_t)k * E, E, it[k], l2[k]);
  }
  std::vector<int> reps;
  for (int r = 0; r < R; r++) if (fits[grid_of[r]]) reps.push_back(r);
  h->counts_R = 0;   // d_counts no longer holds the last colate_stage2_bootstrap's counts
  if (reps.empty()) return 0;
  const int n = (int)reps.size();
  cudaStream_t s = h->stream;
  std::vector<int32_t> tab((size_t)n + 4 * (size_t)n_grids, 0);   // grid_of of the launch's replicates, then int4 {E, offset, n_pairs_cap, 0}
  std::vector<double> cn((size_t)n * C2);
  for (int k = 0; k < n; k++) {
    tab[k] = grid_of[reps[k]];
    memcpy(cn.data() + (size_t)k * C2, counts + (size_t)reps[k] * C2, C2 * 8);
  }
  const size_t info0 = ((size_t)n + 3) & ~(size_t)3;   // int4-aligned
  tab.resize(info0 + 4 * (size_t)n_grids, 0);
  for (int g = 0; g < n_grids; g++)
    if (fits[g]) { tab[info0 + 4 * g] = grid_E[g]; tab[info0 + 4 * g + 1] = (int32_t)grid_off[g]; tab[info0 + 4 * g + 2] = cap[g]; }
  CK(h->d_gr_tab.ensure(tab.size() * 4));
  CK(h->d_epochs.ensure((size_t)ep_len * 8));
  CK(h->d_rates.ensure((size_t)ep_len * 8));
  CK(h->d_counts.ensure((size_t)n * C2 * 8));
  CK(h->d_gr_rates.ensure((size_t)n * E_max * 8));
  CK(h->d_iters.ensure((size_t)n * 4));
  CK(h->d_ll.ensure((size_t)n * 8));
  CK(cudaMemcpyAsync(h->d_gr_tab.p, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_epochs.p, epochs, (size_t)ep_len * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_rates.p, rates_init, (size_t)ep_len * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_counts.p, cn.data(), (size_t)n * C2 * 8, cudaMemcpyHostToDevice, s));
  const int32_t* d_tab = h->d_gr_tab.as<int32_t>();
  if ((rc = run_em_grids(h, n, d_tab, d_tab + info0, E_max, smem, max_iter, s))) return rc;
  std::vector<double> rt((size_t)n * E_max), l2(n);
  std::vector<int32_t> it(n);
  CK(cudaMemcpyAsync(rt.data(), h->d_gr_rates.p, (size_t)n * E_max * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(it.data(), h->d_iters.p, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(l2.data(), h->d_ll.p, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  for (int k = 0; k < n; k++) put(reps[k], rt.data() + (size_t)k * E_max, E_max, it[k], l2[k]);
  return 0;
}

int colate_estep(colate_handle* h, int shared, int E, const double* epochs, const double* rates, int n_t, const double* t,
                 double* num, double* denom, double* logl)
{
  if (!h || E < 2 || E > 1024 || n_t <= 0 || !epochs || !rates || !t) return fail(COLATE_ERR_ARG, "colate_estep: bad arguments");
  CK(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  CK(h->d_epochs.ensure((size_t)E * 8));
  CK(h->d_rates.ensure((size_t)E * 8));
  const size_t tot = (size_t)n_t * (2 + 2 * (size_t)E);
  CK(h->d_tmp.ensure(tot * 8));
  CK(cudaMemcpyAsync(h->d_epochs.p, epochs, (size_t)E * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_rates.p, rates, (size_t)E * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_tmp.p, t, (size_t)n_t * 8, cudaMemcpyHostToDevice, s));
  int rc = run_estep(h, shared, E, n_t);
  if (rc) return rc;
  double* base = h->d_tmp.as<double>();
  if (num) CK(cudaMemcpyAsync(num, base + n_t, (size_t)n_t * E * 8, cudaMemcpyDeviceToHost, s));
  if (denom) CK(cudaMemcpyAsync(denom, base + n_t + (size_t)n_t * E, (size_t)n_t * E * 8, cudaMemcpyDeviceToHost, s));
  if (logl) CK(cudaMemcpyAsync(logl, base + n_t + 2 * (size_t)n_t * E, (size_t)n_t * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return 0;
}

int colate_set_age_bins(colate_handle* h, const double* age_bin)
{
  if (!h) return fail(COLATE_ERR_ARG, "colate_set_age_bins: null handle");
  CK(cudaSetDevice(h->device));
  int rc = ensure_tables(h);
  if (rc) return rc;
  double ab[NBINS];
  if (age_bin) memcpy(ab, age_bin, sizeof ab); else colate_age_bins(ab);
  for (int b = 0; b < NBINS; b++) if (!(ab[b] >= 0) || (b > 0 && !(ab[b] >= ab[b - 1]))) return fail(COLATE_ERR_ARG, "colate_set_age_bins: the grid must be non-negative and ascending");
  memcpy(h->h_agebin, ab, sizeof ab);
  CK(cudaMemcpyAsync(h->d_agebin.p, h->h_agebin, sizeof ab, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int colate_libm_exact(void) { return libm_self_check(); }

// test hook (host): the straight-line log1p of the throughput-mode EM folds and its validity predicate
int colate_test_log1p_wide(int n, const double* x, double* y, int32_t* ok)
{
  for (int i = 0; i < n; i++) { y[i] = glm::log1p_wide(x[i]); ok[i] = glm::log1p_wide_ok(x[i]) ? 1 : 0; }
  return 0;
}

int colate_test_libm(colate_handle* h, int which, int n, const double* x, double* y)
{
  if (!h || n <= 0 || !x || !y) return fail(COLATE_ERR_ARG, "colate_test_libm: bad arguments");
  CK(cudaSetDevice(h->device));
  return run_libm(h, which, n, x, y);
}

// test hook: the straight-line fold pieces of the EM kernels on the device (which: see k_test_em_prims); b may be NULL
// for the one-operand pieces
int colate_test_em_prims(colate_handle* h, int which, int n, const double* a, const double* b, double* y, int32_t* ok)
{
  if (!h || which < 0 || which > 6 || n <= 0 || !a || !y || !ok || (which >= 3 && !b))
    return fail(COLATE_ERR_ARG, "colate_test_em_prims: bad arguments");
  CK(cudaSetDevice(h->device));
  return run_test_em_prims(h, which, n, a, b, y, ok);
}

// test hook: the kernel of the handle's last EM launch (0 k_em, 1 k_em_split, 2 k_em_cta / k_em_cta_grids, -1 none yet) and
// its CTAs per replicate
int colate_test_last_em(colate_handle* h, int* kernel, int* csize)
{
  if (!h || !kernel || !csize) return fail(COLATE_ERR_ARG, "colate_test_last_em: bad arguments");
  *kernel = h->em_kernel;
  *csize = h->em_csize;
  return 0;
}

// test hooks: k_sample's table-free age-bin index (fast[i] = -1 where the kernel would consult the exact
// table) next to the exact index, on given ages / swept over all floats with bit patterns in [lo, hi)
int colate_test_bin_fast(colate_handle* h, int n, const double* ages, int32_t* fast, int32_t* exact)
{
  if (!h || n <= 0 || !ages || !fast || !exact) return fail(COLATE_ERR_ARG, "colate_test_bin_fast: bad arguments");
  CK(cudaSetDevice(h->device));
  return run_test_bin_fast(h, n, ages, fast, exact);
}
int colate_test_bin_sweep(colate_handle* h, uint32_t lo_bits, uint32_t hi_bits, uint64_t* out3)
{
  if (!h || !out3 || hi_bits < lo_bits || hi_bits > 0x7f800000u) return fail(COLATE_ERR_ARG, "colate_test_bin_sweep: bad arguments");
  CK(cudaSetDevice(h->device));
  return run_test_bin_sweep(h, lo_bits, hi_bits, out3);
}

// test hook: raw engine words [word0, word0+n) of the stream behind `mt_state`, via the device path
int colate_test_mt_stream(colate_handle* h, const uint32_t* mt_state, int64_t word0, int64_t n_words, int log2_chunk_sites,
                          uint32_t* out)
{
  if (!h || !mt_state || word0 < 0 || n_words < 0) return fail(COLATE_ERR_ARG, "colate_test_mt_stream: bad arguments");
  CK(cudaSetDevice(h->device));
  uint32_t* p = nullptr;
  int rc = run_mt_stream(h, mt_state, word0, n_words, log2_chunk_sites, &p, out ? out + n_words : nullptr, false);
  if (rc) return rc;
  if (n_words > 0) CK(cudaMemcpyAsync(out, p, (size_t)n_words * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

}  // extern "C"
