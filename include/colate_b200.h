/* colate_b200.h -- C ABI of the B200-native `Colate --mode mut` (tmp/tmp) hot path.
 *
 * The reference (leospeidel/Colate) has no FFI: mut() calls plain C++ functions of the
 * same translation unit.  This header defines the seam between them; every entry point
 * cites the reference interface it replaces (paths relative to /root/reference/).
 * INTEGRATION.md shows the reference-side binding.
 *
 * Conventions: extern "C", plain pointers and sizes.  All functions return 0 on success
 * and a negative colate_status on error (message: colate_last_error()).  Host buffers are
 * caller-owned; device buffers are owned by the handle.  Calls are synchronous from the
 * caller's view and not re-entrant on one handle.  One handle = one GPU (one process per
 * GPU under torch.distributed / NCCL, or one host thread per handle).
 * There is no CPU fallback: every compute entry point fails with COLATE_ERR_CUDA when no
 * sm_100 device is usable.
 */
#ifndef COLATE_B200_H
#define COLATE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COLATE_NUM_AGE_BINS 185      /* (int)(log(1e8)*10)+1, coal.cpp:3126-3127 */
#define COLATE_MAX_BLOCKS 500        /* coal.cpp:3140 */
#define COLATE_BLOCK_BASES 30000000  /* coal.cpp:3139 */
#define COLATE_NUM_SAMPLES 100       /* coal.cpp:2085 */
#define COLATE_MT_WORDS 624

typedef enum {
  COLATE_OK = 0,
  COLATE_ERR_ARG = -1,        /* bad argument / inconsistent sizes                        */
  COLATE_ERR_AGE_RANGE = -2,  /* a used row the reference cannot process: age_begin <= 0 and  */
                              /* age bin >= 185 (it writes out of bounds, coal.cpp:2269), or */
                              /* age_begin itself in bin >= 185 (its loop 2279-2294 never ends) */
  COLATE_ERR_BLOCKS = -3,     /* more than 500 genomic blocks (reference overruns, 3140)   */
  COLATE_ERR_CUDA = -4,       /* CUDA runtime error or no usable device                    */
  COLATE_ERR_IO = -5,         /* unreadable / malformed input file                         */
  COLATE_ERR_ORDER = -6,      /* positions not ascending / duplicate chromosome names      */
  COLATE_ERR_STATE = -7       /* call sequence violated (e.g. stage1 before set_sites)     */
} colate_status;

typedef struct colate_handle colate_handle;

const char* colate_last_error(void);
const char* colate_version(void);

/* ---- handle -------------------------------------------------------------------------- */
int colate_create(int device, colate_handle** out);
void colate_destroy(colate_handle* h);
/* cudaStream_t the handle launches on (as void*), for event timing by the caller. */
void* colate_stream(colate_handle* h);
/* Keep the generator stream (the std::mt19937 words parse_tmptmp consumes, coal.cpp:2262/2282) in device memory
 * between colate_stage1* calls and reuse it whenever a call starts from the same generator state at the same
 * offset and needs no more words than are there.  Off by default.  For all-pairs jobs: the reference is run
 * once per pair with the same --seed (mut(), coal.cpp:3157-3162), so every pair consumes a prefix of one and the
 * same stream; results are unchanged (the stream is a function of the state alone). */
int colate_set_stream_cache(colate_handle* h, int enable);

/* ---- inputs: what parse_tmptmp (coal.cpp:2072) obtains from its readers -------------- */

/* Rows of the per-chromosome .mut files in --chr order (Mutations::Read,
 * include/src/mutations.cpp:56-283; consumed at coal.cpp:2148-2176).
 *   site_off[n_chr+1]  row range of each chromosome
 *   pos, age_begin, age_end   SNPInfo::pos / age_begin / age_end (float32 as in mutations.hpp:21)
 *   meta  bit0 = row passes coal.cpp:2150 + 2166 + 2175-2176 (everything that depends on the
 *         row alone), byte1 = ancestral char, byte2 = derived char  (colate_site_meta())
 * location: 0 = host pointers (copied host->device), 1 = device pointers (copied d2d). */
int colate_set_sites(colate_handle* h, int n_chr, const int64_t* site_off, const int32_t* pos,
                     const float* age_begin, const float* age_end, const uint32_t* meta, int location);

/* Records of one .colate.in file in file order (record layout coal.cpp:2505-2514; read at
 * coal.cpp:2126-2133, 2185-2192, 2205-2212) into genome slot `slot` (0..COLATE_MAX_GENOMES-1).
 *   chr_first[c], chr_end[c]  record range the reference's sequential reader can reach while
 *       it is on chromosome c (chr_first = the record pre-loaded by the chromosome seek,
 *       coal.cpp:2125-2145; -1/-1 if the chromosome is never reached): colate_chr_ranges()
 *   alleles = ancestral | derived << 8 */
#define COLATE_MAX_GENOMES 64
int colate_set_genome(colate_handle* h, int slot, int64_t n_rec, const int64_t* chr_first,
                      const int64_t* chr_end, const int32_t* bp, const int32_t* aaf, const int32_t* daf,
                      const uint16_t* alleles, int location);

/* SURVEY.md 8(f) N3 -- the bam front-ends' inputs, pre-decoded: the pileup of genome `slot` at the .mut rows, i.e. what
 * bam_parser::count_alleles (include/vcf/htslib.cpp:60-168) holds at bp_mut - 1 when parse_onebambam looks it up
 * (coal.cpp:1885-1929 reference, 1936-1980 target): counts[n_site][4] = reads showing A, C, G, T, all zero where the position is
 * not covered.  Replaces colate_set_genome for that slot: AAF / DAF are picked by the row's own alleles, a row is usable iff
 * reads > 0, (AAF > 0 || DAF > 0) and at most two alleles were seen (coal.cpp:1916-1917, 1967-1968); the pileup ring is random
 * access, so the look-ahead rule of the .colate.in reader does not apply.  A bcf genome resolved by its decoder (parse_vcfvcf,
 * coal.cpp:1000-1137) fits the same call: counts of the row's ancestral / derived allele in their A/C/G/T columns
 * (AAF = N - DAF), zeros for rows the decoder rejects.  Use with colate_set_option(h, "front_end", 1): raw count weights
 * (coal.cpp:2005-2039) and the 1e3 normalisation of stage ii (coal.cpp:3453-3463). */
int colate_set_pileup(colate_handle* h, int slot, const int32_t* counts, int location);

/* The bcf front-ends' inputs, pre-decoded (parse_vcfvcf, coal.cpp:997-1137; parse_vcf, parse_bamvcf, parse_onebamvcf alike): per .mut
 * row the counts of the row's ancestral / derived allele among the genome's haplotypes as the decoder resolved them -- allele match and
 * flip, biallelic test, "alt not reported" records, the --ref_genome fall-back; AAF = N - DAF -- zeros where the row is not usable for
 * this genome.  Like colate_set_pileup without the A/C/G/T detour (rows with the allele codes 0 / 1 fit too).  Use with front_end = 1. */
int colate_set_row_counts(colate_handle* h, int slot, const int32_t* aaf, const int32_t* daf, int location);

/* The decoder's counting loop on the device: the pileup of genome `slot` from DECODED alignment records instead of finished counts.
 * Replaces bam_parser::count_alleles_for_read / read_to_pos (include/vcf/htslib.cpp:60-168, 426-437) for the positions the bam
 * front-ends look up; what stays with the caller is BAM decompression (sam_read1).  Per contig of the --chr list, its reads in file
 * order (sorted by start, as the reference requires: htslib.cpp:411-414):
 *   pos[k] 0-based leftmost position, mapq[k], len[k] (l_qseq), seq_off[k] offset of the read's bases / qualities in seq / qual,
 *   seq: one ASCII letter per base (seq_nt16_str of the 4-bit code, htslib.cpp:403), qual: phred bytes;
 *   ref_seq / ref_len: the contig of --ref_genome as fasta::Read leaves it (upper-cased, data.cpp:213-237);
 *   mapq_th, len_th, mismatch_th: --filters (default "20,30,10", coal.cpp:3096); the base-quality threshold is 30 (htslib.hpp:66).
 * One call takes ALL reads of a contig: its first record is the one the reference counts from assign_contig with the record's packed
 * sequence bytes in place of its qualities (htslib.cpp:549 against 406) -- reproduced.
 * colate_pileup_begin zeroes the slot's counts, colate_pileup_reads adds one contig, colate_pileup_end makes the slot a pileup
 * genome (as colate_set_pileup would) and optionally returns counts[n_site][4] (e.g. for colate_maketmp_pileup).  Host pointers. */
int colate_pileup_begin(colate_handle* h, int slot);
int colate_pileup_reads(colate_handle* h, int slot, int chr_index, int64_t n_reads, const int32_t* pos, const uint8_t* mapq, const int32_t* len,
                        const int64_t* seq_off, const uint8_t* seq, const uint8_t* qual, const uint8_t* ref_seq, int64_t ref_len,
                        int mapq_th, int len_th, int mismatch_th);
int colate_pileup_end(colate_handle* h, int slot, int32_t* counts_out);

/* The same pileup straight from a BAM file: replaces colate_pileup_begin / _reads / _end for `slot` and leaves it a pileup genome
 * (counts_out, optional: counts[n_site][4]).  What htslib's sam_read1 and bam_parser::read_entry / assign_contig do for the bam
 * front-ends (include/vcf/htslib.cpp:379-437, 490-573) is done here: BGZF blocks are inflated in parallel on the host (CRC32 and
 * ISIZE checked), the header's contigs are matched to the --chr list (`<name>` or `chr<name>`, htslib.cpp:388), the records are
 * decoded on the device (pos, mapq, l_seq, packed sequence, qualities; read name, CIGAR, flag and aux data are not looked at)
 * and counted by the same kernels as colate_pileup_reads, in chunks of at most chunk_bytes record bytes (0: 64 MiB) while the
 * host inflates the next one.  The assign_contig quirk applies to the first record of every contig.
 *   chr_names[n_chr]: the site set's --chr list; ref_seqs[c] / ref_lens[c]: contig c of --ref_genome (host memory; upper-cased
 *   on the device as fasta::Read does, data.cpp:213-237); mapq_th, len_th, mismatch_th: --filters.
 * Refused: COLATE_ERR_IO for a file that is not BGZF (plain gzip included), truncated blocks, CRC / ISIZE mismatches, a wrong
 * magic, a header or record that runs past the data, a listed contig absent from the header or present under both spellings,
 * listed contigs whose records are not contiguous or not in --chr order (message: file and byte offset); COLATE_ERR_ORDER for
 * descending positions within a contig ("BAM file not sorted by position.", htslib.cpp:411-414, checked on the device across
 * chunks) or a record of a listed contig with a negative position (checked on the host before anything is launched).
 * Records of unlisted contigs and unmapped records without a contig (refID -1) are skipped.  A missing EOF block is accepted. */
int colate_pileup_bam(colate_handle* h, int slot, const char* bam_path, int n_chr, const char* const* chr_names, const uint8_t* const* ref_seqs,
                      const int64_t* ref_lens, int mapq_th, int len_th, int mismatch_th, int64_t chunk_bytes, int32_t* counts_out);
/* ref_seqs = NULL (ref_lens unused): the contigs come from the handle's resident genome (colate_set_ref_genome, one contig per --chr
 * entry), which stays on the device -- nothing is copied per call (COLATE_ERR_STATE without one). */
/* Phases of the last colate_pileup_bam: [0] BGZF index s, [1] inflate s (wall, summed over windows), [2] record walk s, [3] host-to-device
 * copies ms, [4] device decode ms, [5] filter + pileup ms ([3]-[5] only with colate_set_option(h, "bam_timing", 1)), [6] whole call s,
 * [7] inflate threads, [8] inflated bytes, [9] records of listed contigs. */
int colate_last_bam_timing(colate_handle* h, double* out10);

/* The row counts of genome `slot` straight from BCF files: replaces colate_set_row_counts for that slot (use with front_end = 1).
 * What htslib and parse_vcfvcf's decoder half do for the bcf/bcf front-end (coal.cpp:997-1137) is done here: per --chr entry c
 * the file bcf_paths[c] (the reference's <prefix>_chr<c>.bcf) is inflated on the host (BGZF, CRC32 and ISIZE checked) in windows
 * of about chunk_bytes inflated bytes (0: 64 MiB) while the device decodes the previous one: every record is reduced to its
 * position, the codes of its first two alleles, the sum of its GT allele indices and whether all of them are <= 1.  Those 12 bytes
 * per record stay on the device for the file; then one thread per .mut row of the chromosome finds the first record at or after
 * the row's position and applies the rules of `role`:
 *   role 1 (reference, COLATE_BCF_REFERENCE): the record's two alleles are the row's, in either order (flipped: DAF = N - sum),
 *     and it is biallelic; without a record there, DAF = N if ref_seqs shows the derived allele; DAF = 0 makes the row unusable;
 *   role 0 (target, COLATE_BCF_TARGET): as the reference, or the record reports one allele (second allele empty or absent) that is
 *     one of the row's and its allele sum is 0 (DAF = N when that allele is the derived one); without a record there, ref_seqs
 *     gives DAF = N for the derived base and 0 for the ancestral base, any other base makes the row unusable.
 * N = samples x GT length.  Only rows with meta bit 0 set and ancestral != derived are resolved (coal.cpp:966-995).  The cursors of
 * the reference need no state here: rows and records ascend, so its record for a row is that lower bound, and the target cursor
 * moving only for rows the reference kept changes nothing; k_pileup_join / k_ok then keep a row iff both slots are usable.
 *   chr_names: the site set's --chr list (messages); ref_seqs / ref_lens: contig c of --ref_genome (host memory, read upper-cased
 *   as fasta::Read leaves it), or ref_seqs = NULL for no --ref_genome; aaf_out / daf_out (optional, host): the counts per row.
 * Each file is BCF or bgzipped text VCF, told apart by its first inflated bytes as htslib's bcf_open does (BCF\2\1 / BCF\2\2 or
 * ##fileformat=VCF); a VCF line decodes to the record the BCF of the same record gives (k_vcf_decode, DESIGN.md section 6h).
 * Refused, with the file and the (inflated) byte offset: COLATE_ERR_IO for a file that is not BGZF (plain gzip, uncompressed BCF
 * or VCF), a truncated block, a CRC or ISIZE mismatch, a wrong magic (BCF\2\1 or BCF\2\2, or ##fileformat=VCF), a header or record
 * that runs past the data, a header without ##FORMAT=<ID=GT, records on more than one contig, a record whose sample count is not
 * the header's, a file without records (all on the host, before the file's records are launched); a record without GT, with a
 * missing ('.') or vector-end GT value, whose GT length differs from the file's first record's or whose typed fields run past it
 * (on the device: the first such record of the file is reported).  COLATE_ERR_ORDER for a POS below the previous record's (equal
 * ones are fine).  Text VCF, on the host: a header without a #CHROM line, a #CHROM line whose first eight columns are not CHROM POS
 * ID REF ALT QUAL FILTER INFO or that has no sample column, an empty line, a line ending in \r\n, a POS that is not a plain decimal
 * in [0, 2^31 - 2]; on the device: fewer than 8 fixed fields, a sample-column count other than the header's, no FORMAT column or no
 * GT key in FORMAT, a sample column that stops before its GT, a GT that is not allele([/|]allele)* with alleles of digits up to
 * 2^29, a '.' allele, samples of one line with different ploidies, samples x ploidy other than the first line's. */
#define COLATE_BCF_TARGET 0
#define COLATE_BCF_REFERENCE 1
int colate_rows_from_bcf(colate_handle* h, int slot, int role, int n_chr, const char* const* chr_names, const char* const* bcf_paths,
                         const uint8_t* const* ref_seqs, const int64_t* ref_lens, int64_t chunk_bytes, int32_t* aaf_out, int32_t* daf_out);
/* Both roles from one decode (DESIGN.md section 6j): every chromosome's file is decoded once and k_bcf_rows resolves each row under
 * the target rules into slot target_slot and under the reference rules into slot reference_slot, each exactly as colate_rows_from_bcf
 * with that role leaves it.  Either slot may be -1 (that role is skipped), not both; they differ.  genome = 0: no --ref_genome;
 * genome = 1: the handle's resident genome (colate_set_ref_genome, one contig per chromosome), read in place (COLATE_ERR_STATE
 * without one). */
int colate_rows_from_bcf_roles(colate_handle* h, int target_slot, int reference_slot, int n_chr, const char* const* chr_names,
                               const char* const* bcf_paths, int genome, int64_t chunk_bytes);
/* A whole-genome BCF or bgzipped text VCF file (DESIGN.md section 6k): --chr entry c (chr_names[c], one per chromosome of the site
 * set) reads the records of the contig named c or chr<c> (BCF: CHROM indexes the header's ##contig lines, IDX= honoured; VCF: the
 * CHROM text), which are exactly the records of that chromosome's own file.  The file is decoded once; the listed contigs' records
 * stay resident, each contig with its own GT length, and every chromosome's rows are resolved against its contig's records alone.
 * The result is colate_rows_from_bcf_roles' on the per-chromosome files, bit for bit; roles, slots and genome as there.  Refused as
 * there, errors on the device prefixed "chromosome <c>: ", and on the host: a listed contig whose records are not one contiguous run
 * (COLATE_ERR_ORDER), a listed contig without records, a contig matching two entries, an entry matched by two contigs with records,
 * a BCF record whose CHROM no ##contig line defines.  Records of other contigs are inflated and walked past unchecked. */
int colate_rows_from_bcf_genome(colate_handle* h, int target_slot, int reference_slot, int n_chr, const char* const* chr_names, const char* path,
                                int genome, int64_t chunk_bytes);
/* Decode only: one BCF or bgzipped text VCF file's records reduced on the device as colate_rows_from_bcf does (same checks), kept on the device;
 * colate_bcf_records copies records [r0, r0 + n) out in the arrays colate_maketmp_records takes (position 1-based, allele codes,
 * allele sum, biallelic flag).  *n_hap = samples x GT length. */
int colate_decode_bcf(colate_handle* h, const char* bcf_path, int64_t chunk_bytes, int64_t* n_records, int32_t* n_hap);
int colate_bcf_records(colate_handle* h, int64_t r0, int64_t n, int32_t* rec_pos, uint8_t* rec_a0, uint8_t* rec_a1, int32_t* rec_alt_sum,
                       uint8_t* rec_biallelic);
/* Decode only, a whole-genome file (as colate_rows_from_bcf_genome): --chr entry c's records are colate_bcf_records [rec_first[c],
 * rec_first[c] + n_records[c]), of n_hap[c] haplotypes. */
int colate_decode_bcf_genome(colate_handle* h, const char* path, int n_chr, const char* const* chr_names, int64_t chunk_bytes, int64_t* rec_first,
                             int64_t* n_records, int32_t* n_hap);
/* Phases of the last colate_rows_from_bcf / colate_decode_bcf (and their whole-genome twins), summed over its files: [0] BGZF index s, [1] inflate s, [2] record
 * walk s, [3] host-to-device copies ms, [4] k_bcf_decode ms, [5] k_bcf_rows ms ([3]-[5] only with colate_set_option(h, "bcf_timing",
 * 1)), [6] whole call s, [7] inflate threads, [8] inflated bytes, [9] records. */
int colate_last_bcf_timing(colate_handle* h, double* out10);

/* ---- make_tmp for many targets on one handle (DESIGN.md section 6i) ------------------------------------------------------ */
/* The --ref_genome of a job, read once (colate_read_fasta per --chr entry) and kept on the device, upper-cased as fasta::Read leaves
 * it: colate_pileup_bam with ref_seqs = NULL and colate_maketmp_write_bcf read their contigs from it.  n_chr = 0 drops it. */
int colate_set_ref_genome(colate_handle* h, int n_chr, const uint8_t* const* ref_seqs, const int64_t* ref_lens);
/* The make_tmp row word: what the row filters of maketmp_bam (coal.cpp:2568, 2584-2587) and maketmp_vcf (2365, 2381-2395) read from
 * a .mut row, from its mutation type as the .mut reader keeps it (the first 15 characters; a longer type is no code):
 *   bit 0  COLATE_MKT_VCF  not flipped, one branch, type exactly a/d with a in {A,C,G,T,0} and d in {A,C,G,T,1}
 *   bit 1  COLATE_MKT_BAM  not flipped, one branch, one-letter a in {A,C,G,T,0}, '/', a non-empty derived string
 *   bit 2  COLATE_MKT_ONE  the derived string is one letter
 *   byte 1 the ancestral letter, byte 2 the first derived letter (0 when the row passes neither filter).
 * colate_ingest_* builds it next to meta on the device; colate_read_mut_words is the host reader's (.mut or .mut.gz), for sites set
 * with colate_set_sites + colate_set_maketmp_words.  colate_set_sites clears the words. */
#define COLATE_MKT_VCF 1u
#define COLATE_MKT_BAM 2u
#define COLATE_MKT_ONE 4u
uint32_t colate_maketmp_word(int flipped, int n_branch, const char* mutation_type);
int64_t colate_read_mut_words(const char* path, int64_t cap, uint32_t* words);
int colate_set_maketmp_words(colate_handle* h, const uint32_t* words, int location);
int colate_fetch_maketmp_words(colate_handle* h, int64_t row0, int64_t n_rows, uint32_t* words);
/* The make_tmp mask rule (NOT the mode-mut rule of colate_mask_bits_from_fasta): a row at or beyond the mask's end is dropped, bp = 0
 * is kept, bp >= 1 is kept iff mask[bp - 1] == 'P'.  Pass bits of rows [row0, row0 + n), as colate_mask_bits_from_fasta. */
int colate_maketmp_mask_bits(const char* path, int64_t n, const int32_t* pos, int64_t row0, uint32_t* pass_bits);
/* The .colate.in of make_tmp written on the device (k_maketmp_rows, a scan, k_maketmp_scatter; one copy of the bytes to pinned host
 * memory, then the file).  Byte for byte what colate_maketmp_pileup / colate_maketmp_records write from the same arrays, for .mut
 * positions that ascend within each chromosome (COLATE_ERR_ORDER otherwise, checked before anything is written).  mask_bits: make_tmp
 * pass bits per row (colate_maketmp_mask_bits) or NULL.  Nothing is written on failure.  Return the records written or < 0.
 *   _pileup: the A/C/G/T counts of pileup slot `slot` (colate_pileup_bam, colate_pileup_end or colate_set_pileup), maketmp_bam's rules.
 *   _bcf:    per --chr entry c the BCF or bgzipped VCF bcf_paths[c], decoded as colate_decode_bcf does and written right after its
 *            decode, maketmp_vcf's rules; rows without a record read the genome of colate_set_ref_genome (none: such rows are
 *            dropped).  COLATE_ERR_ARG "allele sum above the number of haplotypes" as colate_maketmp_records.  Leaves the last
 *            file's records decoded (colate_bcf_records) and its phases in colate_last_bcf_timing ([5]: the writer's kernels). */
int64_t colate_maketmp_write_pileup(colate_handle* h, int slot, int n_chr, const char* const* chr_names, const uint32_t* mask_bits,
                                    const char* out_file);
int64_t colate_maketmp_write_bcf(colate_handle* h, int n_chr, const char* const* chr_names, const char* const* bcf_paths, const uint32_t* mask_bits,
                                 int64_t chunk_bytes, const char* out_file);
/*   _bcf_genome: one whole-genome BCF or bgzipped VCF (as colate_rows_from_bcf_genome), decoded once, then written as _bcf. */
int64_t colate_maketmp_write_bcf_genome(colate_handle* h, int n_chr, const char* const* chr_names, const char* path, const uint32_t* mask_bits,
                                        int64_t chunk_bytes, const char* out_file);
/* The last writer call: [0] writer kernels ms (CUDA events), [1] device-to-host copy ms, [2] file write s, [3] records. */
int colate_last_maketmp_timing(colate_handle* h, double* out4);
/* Work done on this handle since creation: [0] .mut texts parsed on the device, [1] .mut rows parsed (colate_ingest_end), [2] calls of
 * colate_set_ref_genome, [3] reference-genome bytes copied host-to-device (colate_set_ref_genome, colate_pileup_bam, colate_rows_from_bcf). */
int colate_upload_counts(colate_handle* h, int64_t* out4);

/* ---- make_tmp from a genotype matrix (DESIGN.md section 6l) ------------------------------------------------------------ */
/* format: COLATE_GENO_EIGENSTRAT reads <prefix>.geno (packed "GENO" or text), .snp and .ind; COLATE_GENO_PLINK reads the SNP-major
 * <prefix>.bed, .bim and .fam.  --chr entry c holds the SNPs whose contig is c or chr<c> (23 for X, 24 for Y), in file order. */
#define COLATE_GENO_EIGENSTRAT 0
#define COLATE_GENO_PLINK 1
/* Host only (no GPU): the SNP and individual counts, the SNPs per --chr entry and the matrix kind (0 packed EIGENSTRAT, 1 text
 * EIGENSTRAT, 2 PLINK .bed), with every host refusal of colate_maketmp_write_geno: COLATE_ERR_IO for an unreadable file, a line
 * with too few fields, alleles missing from .snp / .bim, a position that is not an integer in [0, 2^31), a bad .bed magic, an
 * individual-major .bed, a TGENO file, GENO header counts or a file size that disagree with the .snp / .ind (.bim / .fam) lines,
 * a text call other than 0 1 2 9; COLATE_ERR_ORDER for SNP positions that descend within an entry.  Messages name file and line. */
int colate_geno_scan(const char* prefix, int format, int n_chr, const char* const* chr_names, int64_t* n_snp, int64_t* n_ind,
                     int64_t* entry_snps, int32_t* kind);
/* The .colate.in of n_ind individuals (ind_ids: .ind column 1 / .fam IID, each present exactly once) written on the device into
 * out_files[i], each byte for byte what colate_maketmp_table(chr_names, the .mut files, T_i, masks_i, has_ref_genome = 1, ...) writes
 * for the table T_i of "c position allele" lines of the individual's homozygous calls, per --chr entry c in order (heterozygous and
 * missing calls write no line).  The handle holds the ingested .mut rows of the same --chr list (ascending positions per chromosome,
 * COLATE_ERR_ORDER otherwise).  mask_ids[i]: -1 or the index of the individual's make_tmp pass bits (colate_maketmp_mask_bits) in
 * mask_bits, (n_site + 31) / 32 words per mask; mask_ids may be NULL.  The matrix is uploaded once per call.
 * Optional outputs per individual: records_out (-1: its file could not be written, and is removed), het_skipped_out (heterozygous
 * calls on the listed entries), cutoff_out (the first entry without a homozygous call: the table cursor then consumes the rest of
 * the table, so that entry and every later one write nothing; n_chr if none).  Returns the number of files that could not be
 * written (the others are complete), or < 0 for a failure of the whole call, which writes nothing. */
int64_t colate_maketmp_write_geno(colate_handle* h, const char* prefix, int format, int n_ind, const char* const* ind_ids, int n_chr,
                                  const char* const* chr_names, const char* const* out_files, const int32_t* mask_ids, const uint32_t* mask_bits,
                                  int64_t* records_out, int64_t* het_skipped_out, int32_t* cutoff_out);
/* The last colate_maketmp_write_geno: [0] host scan s, [1] matrix upload s, [2] k_geno_join ms, [3] k_geno_called ms, [4] k_geno_rows
 * ms, [5] scans and scatters ms, [6] device-to-host copies s, [7] file writes s, [8] whole call s, [9] bytes written. */
int colate_last_geno_timing(colate_handle* h, double* out10);
/* Matrix uploads on this handle since creation: [0] uploads, [1] bytes copied host-to-device. */
int colate_geno_upload_counts(colate_handle* h, int64_t* out2);

/* P/N mask of genome `slot` evaluated at the site positions (fasta::Read,
 * include/src/data.cpp:213-237; test at coal.cpp:2169-2174): bit m of pass_bits = row m is
 * NOT rejected by the mask (positions at or beyond the mask end pass).  NULL clears it. */
int colate_set_mask(colate_handle* h, int slot, const uint32_t* pass_bits, int location);
/* Genome `src`'s per-row counts (a pileup or row-count slot: colate_pileup_bam, colate_set_pileup, colate_set_row_counts,
 * colate_rows_from_bcf[_roles], ...) copied into slot `dst` on the device, so one decoded file can sit under several masks
 * without being decoded again.  dst's mask and join state are cleared.  COLATE_ERR_STATE for a .colate.in record slot or an
 * unset one. */
int colate_copy_genome(colate_handle* h, int dst, int src);

/* ---- stage i: parse_tmptmp, coal.cpp:2071-2321 (called at coal.cpp:3317) ------------- */

/* Stage i, part A: per-row use flags (A.2 filter, both stream lookups with the sequential
 * reader's look-ahead rule, coal.cpp:2181-2219).  Outputs (host):
 *   n_used_chr[n_chr]    rows reaching coal.cpp:2222 per chromosome
 *   n_blocks_chr[n_chr]  genomic blocks the chromosome occupies (coal.cpp:2227-2234, 2306-2310) */
int colate_stage1_flags(colate_handle* h, int target_slot, int reference_slot,
                        int64_t* n_used_chr, int32_t* n_blocks_chr);

/* Stage i, part B: Monte-Carlo age binning (coal.cpp:2236-2297) of the rows flagged by part A.
 *   mt_state[624]   std::mt19937 state window: the 624 untempered words preceding the next
 *                   output (for a freshly seeded engine: its seed array; colate_mt_seed()).
 *   used_rank_base  used rows that precede this handle's first row in the global row order
 *                   (0 on one GPU; multi-GPU: exclusive sum of the other ranks' n_used) --
 *                   row r of this handle consumes generator words [200*(base+r), +200)
 *   block_base      global index of this handle's first genomic block
 * Outputs (host, caller-allocated):
 *   block_stats[n_blocks][4][185] fp64: age_shared_count, age_notshared_count, and row 0 of
 *       age_shared_emp / age_notshared_emp, for blocks block_base .. block_base+n_blocks-1
 *   block_tallies[n_blocks][3][185] int64: samples added to shared / notshared, rows added to emp
 *   mt_state_out[624]  state window after 200*(used_rank_base+n_used) words (may alias mt_state)
 * Rows with age_begin > 0 whose age interval reaches past the age grid are rejection-sampled as the reference does
 * (coal.cpp:2279-2294: 200 + 2 * redraws engine words), in row order with the redraws walked on the host. */
int colate_stage1_sample(colate_handle* h, const uint32_t* mt_state, int64_t used_rank_base,
                         int block_base, double* block_stats, int64_t* block_tallies,
                         uint32_t* mt_state_out);

/* Convenience: parts A+B on one GPU.  *num_blocks = return value of parse_tmptmp. */
int colate_stage1(colate_handle* h, int target_slot, int reference_slot, const uint32_t* mt_state,
                  int* num_blocks, double* block_stats, int64_t* block_tallies,
                  int64_t* n_used_total, uint32_t* mt_state_out);

/* ---- stage ii: block bootstrap + F redistribution, coal.cpp:3344-3451 ---------------- */
/* block_weights[R][num_blocks]: multiplicity of each block per replicate, drawn by the host
 * with the reference's generator (colate_draw_block_weights(), coal.cpp:3350-3357).
 * counts[R][2][185]: age_shared_count / age_notshared_count per replicate (optional). The
 * counts also stay resident on the device for colate_stage3_em().
 * block_stats == NULL: the histograms the last colate_stage1 / colate_stage1_sample call left on the device
 * (num_blocks must be that call's block count).
 * Data pointers of stages i-iii outputs and of block_weights / block_stats / counts may be host or device
 * pointers (unified addressing): a multi-GPU driver all-reduces the histograms on the device. */
int colate_stage2_bootstrap(colate_handle* h, int R, int num_blocks, const int32_t* block_weights,
                            const double* block_stats, double age, double* counts);

/* ---- stage iii: EM, coal.cpp:3675-3827 + coal_EM (coal_EM.hpp:38-58, coal_EM.cpp:5-468) - */
/* counts: [R][2][185] host pointer, or NULL to use the device-resident result of the last
 * colate_stage2_bootstrap().  rates[R][E], iters[R] (the `iter` printed at coal.cpp:3823),
 * final_ll[R]. */
int colate_stage3_em(colate_handle* h, int R, int E, const double* epochs, const double* rates_init,
                     const double* counts, int max_iter, double* rates, int32_t* iters, double* final_ll);

/* Asynchronous form for drivers that run many pairs through one handle (the reference is started once per pair): _begin
 * queues the EM of the device-resident counts of the last colate_stage2_bootstrap() on the handle's EM stream and returns;
 * _end waits for it and fetches the results.  In between the caller may upload the NEXT pair and take it through stage i
 * (colate_ingest_*, colate_set_*, colate_stage1*): the latency-mode EM keeps one GPC busy, stage i runs on the rest of the
 * device.  colate_stage2_bootstrap / colate_stage3_em are refused with COLATE_ERR_STATE while an EM is in flight (they
 * would overwrite its counts).  Results are those of colate_stage3_em. */
int colate_stage3_em_begin(colate_handle* h, int R, int E, const double* epochs, const double* rates_init, int max_iter);
int colate_stage3_em_end(colate_handle* h, double* rates, int32_t* iters, double* final_ll);

/* The EM of R replicates that do not share one epoch grid (a cohort: every pair's age moves its grid, coal.cpp:3553-3630).
 * Grid g has grid_E[g] epochs at epochs[grid_off[g] ..] with initial rates at rates_init[grid_off[g] ..]; replicate r runs on
 * grid grid_of[r] with counts[r][2][185] (host).  Outputs (host): rates[R][E_max] (E_max = max grid_E; entries past the row's own E
 * are 0), iters[R], final_ll[R].  Row r equals colate_stage3_em(h, 1, grid_E[g], epochs + grid_off[g], rates_init + grid_off[g],
 * counts[r], ...) bit for bit: the replicates of every grid the throughput kernel fits run in ONE launch, each CTA on its own grid;
 * a grid it does not fit (shared memory or threads) runs through colate_stage3_em alone.  The EM uses the age grid of
 * colate_set_age_bins() for all rows.  Afterwards no device-resident counts remain for colate_stage3_em(counts = NULL). */
int colate_stage3_em_grids(colate_handle* h, int R, const int32_t* grid_of, int n_grids, const int32_t* grid_E, const int64_t* grid_off,
                           const double* epochs, const double* rates_init, const double* counts, int max_iter, double* rates,
                           int32_t* iters, double* final_ll);

/* The age grid colate_stage3_em() evaluates (the point ages t = age_bin[b], coal.cpp:3708, 3721).  Default: colate_age_bins().
 * mut() started from a <out>.colate_mat cache reads the grid back from that file's first line, i.e. rounded to six
 * significant digits (coal.cpp:3481-3483), and runs the EM on THOSE ages: the host passes them here.  NULL restores the
 * default.  (Stage ii keeps the exact grid: the cache path never runs it.) */
int colate_set_age_bins(colate_handle* h, const double* age_bin);

/* One E-step call: coal_EM(epochs, rates).EM_shared / EM_notshared(t, t, num, denom)
 * (coal_EM.cpp:153, 297) evaluated on the device for n_t ages.  num/denom: [n_t][E]. */
int colate_estep(colate_handle* h, int shared, int E, const double* epochs, const double* rates,
                 int n_t, const double* t, double* num, double* denom, double* logl);

/* 1 if this host's libm evaluates exp/log/log1p bit-identically to the device implementation
 * (glibc 2.39, FMA variants): then colate_stage3_em() reproduces the reference run on this host
 * bit for bit.  0: the device still follows glibc 2.39/FMA; the host's libm differs. */
int colate_libm_exact(void);

/* ---- timing of the last stage-1 call (CUDA events on the handle's stream), ms -------- */
typedef struct {
  float join_ms;     /* k_join x2 (skipped when the join of a genome is still cached)            */
  float flags_ms;    /* row filter, both stream lookups, used-row ranks                        */
  float rng_ms;      /* MT19937 jump-ahead tree + stream generation                            */
  float compact_ms;  /* used rows -> dense records, tile table                                 */
  float sample_ms;   /* k_sample alone: the per-mutation Monte-Carlo binning kernel            */
  float replay_ms;   /* k_replay + k_emp: exact per-block histograms in the reference's addition order */
  float total_ms;
  int64_t n_site, n_used, rng_words;
} colate_stage1_timing;
int colate_last_stage1_timing(colate_handle* h, colate_stage1_timing* out);

/* Options: "rejoin" = 1 drops the cached record->row join of every genome before each
 * colate_stage1_flags() (benchmarks time the join as part of the pass). */
int colate_set_option(colate_handle* h, const char* key, int64_t value);
/* Kernels launched on this handle since creation (for launch accounting). */
int64_t colate_launch_count(colate_handle* h);
/* Generator words the last colate_stage1 / colate_stage1_sample call consumed beyond 200 per used row: the redraws of
 * the reference's rejection sampling (coal.cpp:2279-2294; rows with age_begin > 0 whose interval reaches past the age
 * grid).  A chromosome-sharded job must see 0 on every rank (a later rank's stream offset would depend on it). */
int64_t colate_last_stage1_extra_words(colate_handle* h);

/* ---- host-side pieces of the path (no GPU needed) ------------------------------------ */
/* std::mt19937::seed(seed) -> state window (coal.cpp:3157-3162). */
void colate_mt_seed(uint32_t seed, uint32_t* mt_state);
/* Next n raw engine outputs from a state window; advances the window. */
void colate_mt_generate(uint32_t* mt_state, int64_t n, uint32_t* out);
/* Block multiplicities for R replicates (coal.cpp:3350-3357; std::uniform_int_distribution
 * <int>(0,num_blocks-1) of libstdc++); advances the state window. */
void colate_draw_block_weights(uint32_t* mt_state, int R, int num_blocks, int32_t* block_weights);
/* age grid, coal.cpp:3129-3137 */
void colate_age_bins(double* age_bin);
/* packed site word from a parsed .mut row (coal.cpp:2150-2176 minus the masks). */
uint32_t colate_site_meta(int flipped, int n_branch, float age_begin, float age_end, const char* mutation_type);
/* record ranges per --chr entry, emulating the chromosome seek of coal.cpp:2125-2145.
 * rec_chrom[k] = index of record k's chromosome name in the --chr list (or >= n_chr). */
int colate_chr_ranges(int n_chr, int64_t n_rec, const int32_t* rec_chrom, int64_t* chr_first, int64_t* chr_end);
/* ages and epoch grid, coal.cpp:3105-3120, 3503-3632.  Returns num_epochs or <0. */
double colate_age_generations(const char* target_age, const char* reference_age, int has_years_per_gen,
                              float years_per_gen, double* years_per_gen_out);
int colate_epochs_from_bins(const char* bins, double age, double years_per_gen, double* epochs, int cap, int* ep_null);
int colate_epochs_from_coal_file(const char* path, double age, double* epochs, double* rates_init, int cap);

/* ---- GPU-side ingest of Relate .mut text (SURVEY.md 8f, N1) --------------------------------
 * Replaces Mutations::Read (include/src/mutations.cpp:56-283) + colate_set_sites for plain-text input:
 * the file's bytes (host or device, `location` as above) are split into lines and parsed on the
 * device, one thread per row, straight into the handle's site arrays.  Integers as std::stoi, ages
 * as std::stof (correctly rounded decimal -> float; the rare rows the device cannot convert with
 * that guarantee are re-parsed on the host with strtof).  Result == colate_read_mut() row for row.
 *   colate_ingest_begin(h, n_chr, row_capacity)     row_capacity >= total data rows of all files (any upper bound,
 *                                                   e.g. total bytes / 20: a data row has at least 10 fields)
 *   colate_ingest_mut_text(h, text, n_bytes, loc)   once per --chr entry, in order; returns its rows
 *   colate_ingest_end(h)                            == colate_set_sites() on what was ingested
 *   colate_ingest_fetch(...)                        host copies of ingested rows (masks, tests)
 *   colate_ingest_stats(...)                        device time of the parse kernels, host-parsed rows */
int colate_ingest_begin(colate_handle* h, int n_chr, int64_t row_capacity);
int64_t colate_ingest_mut_text(colate_handle* h, const char* text, int64_t n_bytes, int location);
/* All chromosomes at once: texts[c] / n_bytes[c] in --chr order.  From pinned host memory every text is copied on
 * the handle's copy stream and parsed as soon as it has landed, under the copies of the following chromosomes.
 * rows_out[c] (optional) = data rows of chromosome c.  Same result as n_texts calls of colate_ingest_mut_text. */
int colate_ingest_mut_texts(colate_handle* h, int n_texts, const char* const* texts, const int64_t* n_bytes, int location,
                            int64_t* rows_out);
int colate_ingest_end(colate_handle* h);
int colate_ingest_fetch(colate_handle* h, int64_t row0, int64_t n_rows, int32_t* pos, float* age_begin, float* age_end,
                        uint32_t* meta);
int colate_ingest_stats(colate_handle* h, double* kernel_ms, int64_t* host_fallback_rows);

/* .colate.in image (the file's bytes, host or device) -> genome slot, decoded on the device: replaces
 * colate_read_colate_in + colate_chr_ranges + colate_set_genome (the reference's inline reader: coal.cpp:2126-2133,
 * 2185-2192, 2205-2212; record layout coal.cpp:2505-2514).  The host locates the runs of equal-width records
 * ({lchrom, chrom} headers) by galloping, the device checks every record's header against its run and splits the
 * payload into the slot's arrays; an image whose runs do not verify (interleaved chromosomes) is decoded
 * sequentially on the host instead -- the result is the sequential reader's in every case.  chr_names = the --chr
 * list of the site set in the handle.  Returns the number of records (>= 0) or a negative status. */
int64_t colate_ingest_colate_in(colate_handle* h, int slot, const char* bytes, int64_t n_bytes, int n_chr,
                                const char* const* chr_names, int location);

/* ---- readers / writers (host) --------------------------------------------------------- */
/* Relate .mut[.gz] (mutations.cpp:56-283).  Two-call pattern: n = colate_read_mut(path, 0, ...NULL)
 * returns the row count; then call again with arrays of that capacity. */
int64_t colate_read_mut(const char* path, int64_t cap, int32_t* pos, float* age_begin, float* age_end, uint32_t* meta);
/* .colate.in (coal.cpp:2505-2514).  rec_chrom[k] = index of the record's name in chr_names. */
int64_t colate_read_colate_in(const char* path, int n_chr, const char* const* chr_names, int64_t cap,
                              int32_t* rec_chrom, int32_t* bp, int32_t* aaf, int32_t* daf, uint16_t* alleles);
/* BAM file, host only (no GPU): per --chr entry the number of records, the first and the last record's position and the index of
 * the header contig it matched, with every check of colate_pileup_bam but the order of positions.  window_bytes: inflated bytes per
 * window (0: 64 MiB).  0 or a negative status. */
int colate_bam_scan(const char* path, int n_chr, const char* const* chr_names, int64_t window_bytes, int64_t* n_records, int32_t* first_pos,
                    int32_t* last_pos, int32_t* ref_id);
/* BCF file, host only (no GPU): the record count, the first and last POS (0-based), the records' contig (CHROM), the header's sample
 * count and the dictionary index of GT, with every host check of colate_rows_from_bcf.  window_bytes: inflated bytes per window
 * (0: 64 MiB).  0 or a negative status. */
int colate_bcf_scan(const char* path, int64_t window_bytes, int64_t* n_records, int32_t* first_pos, int32_t* last_pos, int32_t* contig,
                    int32_t* n_sample, int32_t* gt_key);
/* Bgzipped text VCF file, host only (no GPU): the record count, the first and last POS (0-based, as htslib's bcf1_t.pos), the header's
 * sample count and the records' CHROM (NUL-terminated, cut to chrom_cap - 1 bytes), with every host check of colate_rows_from_bcf
 * on such a file.  A BCF file is refused (colate_bcf_scan reads it).  0 or a negative status. */
int colate_vcf_scan(const char* path, int64_t window_bytes, int64_t* n_records, int32_t* first_pos, int32_t* last_pos, int32_t* n_sample,
                    char* chrom, int64_t chrom_cap);
/* Whole-genome BCF or bgzipped text VCF file, host only (no GPU): per --chr entry the records of its contig, their first and last POS
 * (0-based), and the header's sample count, with every host check of colate_rows_from_bcf_genome.  0 or a negative status. */
int colate_bcf_genome_scan(const char* path, int n_chr, const char* const* chr_names, int64_t window_bytes, int64_t* n_records, int32_t* first_pos,
                           int32_t* last_pos, int32_t* n_sample);
/* fasta::Read (data.cpp:213-237): header line dropped, upper-cased, concatenated; <path> or <path>.gz.  *seq_out: malloc'd,
 * release with colate_free.  Returns the length or < 0. */
int64_t colate_read_fasta(const char* path, uint8_t** seq_out);
void colate_free(void* p);
/* fasta mask (data.cpp:213-237) evaluated at positions -> pass bits for rows [row0, row0+n). */
int colate_mask_bits_from_fasta(const char* path, int64_t n, const int32_t* pos, int64_t row0, uint32_t* pass_bits);
/* make_tmp from a table (maketmp_table, coal.cpp:2682-2808; README.md:86-127): writes the .colate.in record stream of a
 * haploid target given as whitespace-separated (chromosome, position, allele) triples in --chr order, for the rows of the
 * per-chromosome .mut files.  target_masks may be NULL (or hold NULL entries).  Returns the records written or < 0. */
int64_t colate_maketmp_table(int n_chr, const char* const* chr_names, const char* const* mut_files, const char* table_file,
                             const char* const* target_masks, int has_ref_genome, const char* out_file);
/* make_tmp from a BAM pileup (maketmp_bam, coal.cpp:2527-2680) on pre-decoded arrays: counts[n_rows][4] = reads showing A, C, G, T
 * at the position of every data row of the .mut files in --chr order (what bam_parser::count_alleles holds at bp_mut - 1; the BAM
 * decoding stays with the caller).  Returns the records written or < 0. */
int64_t colate_maketmp_pileup(int n_chr, const char* const* chr_names, const char* const* mut_files, const int32_t* counts,
                              int64_t n_rows, const char* const* target_masks, const char* out_file);
/* make_tmp from genotype records (maketmp_vcf, coal.cpp:2325-2525) on pre-decoded arrays: the records of chromosome c are
 * [rec_off[c], rec_off[c+1]) in file order, each with its 1-based position, its first two alleles (the letter if the allele is one
 * character, 0 if it is the empty string, 0xff otherwise), the sum of bcf_gt_allele over the n_hap[c] haplotypes and whether every
 * allele index is <= 1 (the BCF decoding stays with the caller).  ref_genomes / target_masks: fasta paths per chromosome, may be
 * NULL.  Returns the records written or < 0. */
int64_t colate_maketmp_records(int n_chr, const char* const* chr_names, const char* const* mut_files, const int64_t* rec_off,
                               const int32_t* rec_pos, const uint8_t* rec_a0, const uint8_t* rec_a1, const int32_t* rec_alt_sum,
                               const uint8_t* rec_biallelic, const int32_t* n_hap, const char* const* ref_genomes,
                               const char* const* target_masks, const char* out_file);
/* <out>.colate_mat as mut() writes it for every front-end but tmp/tmp (coal.cpp:3336-3343, 3453-3465): the age grid, then per
 * replicate the shared and the not-shared count vector (already divided by 1e3), default ostream formatting.  R = 0 writes the
 * grid line alone (counts may be NULL). */
int colate_write_colate_mat(const char* path, int R, const double* age_bin, const double* counts);
/* <out>.coal (coal.cpp:3660-3672, 3830-3844) and the raw fp64 side output <out>.bin. */
int colate_write_coal(const char* path, int R, int E, const double* epochs, double* rates, int is_ancient, int ep_null);
int colate_write_bin(const char* path, int R, int E, const double* epochs, const double* rates, const int32_t* iters);

#ifdef __cplusplus
}
#endif
#endif /* COLATE_B200_H */
