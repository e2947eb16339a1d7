"""Host-side mirror of the reference's `mut()` driver (include/coal/coal.cpp:3071-3863) on top
of the C-ABI.  Names follow the reference: sites = rows of the .mut files, genomes = .colate.in
record streams, blocks = 30 Mb genomic blocks, replicates = block-bootstrap replicates.

Everything that computes goes through libcolate_b200.so (CUDA); this module only marshals
arrays and mirrors the control flow of mut().
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import MAX_BLOCKS, MT_WORDS, NBINS, check, lib, ptr


def libm_exact() -> bool:
    """True if the host libm matches the device exp/log/log1p bit for bit (glibc 2.39, FMA variants)."""
    return bool(lib().colate_libm_exact())


def age_bins() -> np.ndarray:
    """age_bin[], coal.cpp:3129-3137."""
    out = np.zeros(NBINS)
    lib().colate_age_bins(out)
    return out


def mt_seed(seed: int) -> np.ndarray:
    """std::mt19937::seed(seed) as a 624-word state window (coal.cpp:3157-3162)."""
    w = np.zeros(MT_WORDS, dtype=np.uint32)
    lib().colate_mt_seed(seed & 0xFFFFFFFF, w)
    return w


def draw_block_weights(mt_state: np.ndarray, R: int, num_blocks: int) -> np.ndarray:
    """Block multiplicities per replicate (coal.cpp:3350-3357); advances mt_state in place."""
    w = np.zeros((R, num_blocks), dtype=np.int32)
    lib().colate_draw_block_weights(mt_state, R, num_blocks, w)
    return w


def ages(target_age: str | None = None, reference_age: str | None = None, years_per_gen: float | None = None):
    """(age in generations, years_per_gen), coal.cpp:3105-3118."""
    ypg = C.c_double(0)
    a = lib().colate_age_generations(target_age.encode() if target_age is not None else None,
                                     reference_age.encode() if reference_age is not None else None,
                                     0 if years_per_gen is None else 1, 0.0 if years_per_gen is None else years_per_gen,
                                     C.byref(ypg))
    return a, ypg.value


def epochs_from_bins(bins: str, age: float = 0.0, years_per_gen: float = 28.0):
    """Epoch grid of --bins x,y,step (coal.cpp:3553-3630) -> (epochs, ep_null)."""
    ep = np.zeros(4096)
    null = C.c_int(0)
    n = check(lib().colate_epochs_from_bins(bins.encode(), age, years_per_gen, ep, 4096, C.byref(null)))
    return ep[:n].copy(), null.value


def epochs_from_coal_file(path: str, age: float = 0.0):
    ep, r = np.zeros(4096), np.zeros(4096)
    n = check(lib().colate_epochs_from_coal_file(path.encode(), age, ep, r, 4096))
    return ep[:n].copy(), r[:n].copy()


def chr_ranges(n_chr: int, rec_chrom: np.ndarray):
    """Record range per --chr entry, emulating the chromosome seek (coal.cpp:2125-2145)."""
    rec_chrom = np.ascontiguousarray(rec_chrom, dtype=np.int32)
    first = np.zeros(n_chr, dtype=np.int64)
    end = np.zeros(n_chr, dtype=np.int64)
    check(lib().colate_chr_ranges(n_chr, rec_chrom.shape[0], rec_chrom, first, end))
    return first, end


def colate_in_runs(image: bytes, chr_names, cap_runs=4096):
    """Test hook: the host run finder of .colate.in images -> (n_rec, runs[n,4] = byte_off/width/chr_id/n_rec, first, end)."""
    buf = np.frombuffer(image, dtype=np.uint8) if len(image) else np.zeros(1, np.uint8)
    names = (C.c_char_p * len(chr_names))(*[s.encode() for s in chr_names])
    runs = np.zeros((cap_runs, 4), dtype=np.int64)
    first = np.zeros(max(1, len(chr_names)), dtype=np.int64); end = np.zeros(max(1, len(chr_names)), dtype=np.int64)
    r = check(lib().colate_test_colate_in_runs(C.c_void_p(buf.ctypes.data), len(image), len(chr_names), names, cap_runs, runs, first, end))
    n_rec, n_runs = r & ((1 << 40) - 1), r >> 40
    return n_rec, runs[:n_runs].copy(), first[:len(chr_names)], end[:len(chr_names)]


def read_mut(path: str):
    """Relate .mut[.gz] -> (pos, age_begin, age_end, meta) (mutations.cpp:56-283)."""
    n = check(lib().colate_read_mut(path.encode(), 0, None, None, None, None))
    pos = np.zeros(n, np.int32); ab = np.zeros(n, np.float32); ae = np.zeros(n, np.float32); meta = np.zeros(n, np.uint32)
    check(lib().colate_read_mut(path.encode(), n, ptr(pos), ptr(ab), ptr(ae), ptr(meta)))
    return pos, ab, ae, meta


def read_colate_in(path: str, chr_names):
    """.colate.in -> (rec_chrom, bp, aaf, daf, alleles) (coal.cpp:2505-2514)."""
    names = (C.c_char_p * len(chr_names))(*[s.encode() for s in chr_names])
    n = check(lib().colate_read_colate_in(path.encode(), len(chr_names), names, 0, None, None, None, None, None))
    rc = np.zeros(n, np.int32); bp = np.zeros(n, np.int32); aaf = np.zeros(n, np.int32); daf = np.zeros(n, np.int32)
    al = np.zeros(n, np.uint16)
    check(lib().colate_read_colate_in(path.encode(), len(chr_names), names, n, ptr(rc), ptr(bp), ptr(aaf), ptr(daf), ptr(al)))
    return rc, bp, aaf, daf, al


def mask_bits_from_fasta(path: str, pos: np.ndarray, row0: int, bits: np.ndarray):
    """fasta mask at the site positions -> pass bits of rows [row0, row0+len(pos)) (data.cpp:213-237, coal.cpp:2169-2174)."""
    pos = np.ascontiguousarray(pos, dtype=np.int32)
    check(lib().colate_mask_bits_from_fasta(path.encode(), pos.shape[0], ptr(pos), row0, ptr(bits)))


def mask_bits_from_seq(seqs, site_off, pos) -> np.ndarray:
    """Same as mask_bits_from_fasta for in-memory (already upper-cased) per-chromosome sequences."""
    n = int(site_off[-1])
    ok = np.ones(n, dtype=bool)
    for c, s in enumerate(seqs):
        lo, hi = int(site_off[c]), int(site_off[c + 1])
        p = pos[lo:hi].astype(np.int64)
        arr = np.frombuffer(s, dtype=np.uint8)
        inside = (p >= 0) & (p < arr.shape[0])
        okc = np.ones(hi - lo, dtype=bool)
        okc[inside] = arr[p[inside] - 1] == ord("P")
        ok[lo:hi] = okc
    pad = (-n) % 32
    by = np.packbits(np.concatenate([ok, np.zeros(pad, dtype=bool)]), bitorder="little")
    return np.ascontiguousarray(by).view("<u4").astype(np.uint32).reshape(-1)


def bam_scan(path: str, chr_names, window_bytes: int = 0) -> dict:
    """Host-only walk of a BAM file (no GPU): per --chr entry the record count, the first / last position and the index of the
    header contig it matched (colate_bam_scan).  Raises ColateError for the files colate_pileup_bam refuses."""
    n = len(chr_names)
    names = (C.c_char_p * n)(*[s.encode() for s in chr_names])
    cnt = np.zeros(n, np.int64); first = np.zeros(n, np.int32); last = np.zeros(n, np.int32); rid = np.zeros(n, np.int32)
    check(lib().colate_bam_scan(str(path).encode(), n, names, window_bytes, cnt, first, last, rid))
    return {"n_records": cnt, "first_pos": first, "last_pos": last, "ref_id": rid}


def bcf_scan(path: str, window_bytes: int = 0) -> dict:
    """Host-only walk of a BCF file (no GPU): the record count, the first / last POS (0-based), the records' contig, the header's
    sample count and the dictionary index of GT (colate_bcf_scan).  Raises ColateError for the files colate_rows_from_bcf refuses
    on the host."""
    v = [np.zeros(1, t) for t in (np.int64, np.int32, np.int32, np.int32, np.int32, np.int32)]
    check(lib().colate_bcf_scan(str(path).encode(), window_bytes, *[ptr(x) for x in v]))
    keys = ("n_records", "first_pos", "last_pos", "contig", "n_sample", "gt_key")
    return {k: int(x[0]) for k, x in zip(keys, v)}


def bcf_genome_scan(path: str, chr_names, window_bytes: int = 0) -> dict:
    """Host-only walk of a whole-genome BCF or bgzipped text VCF (no GPU): per --chr entry the records of its contig (<name> or
    chr<name>) and their first / last POS (0-based), and the header's sample count (colate_bcf_genome_scan).  Raises ColateError for
    the files colate_rows_from_bcf_genome refuses on the host."""
    n = len(chr_names)
    names = (C.c_char_p * n)(*[str(s).encode() for s in chr_names])
    cnt = np.zeros(n, np.int64); first = np.zeros(n, np.int32); last = np.zeros(n, np.int32); ns = np.zeros(1, np.int32)
    check(lib().colate_bcf_genome_scan(str(path).encode(), n, names, window_bytes, ptr(cnt), ptr(first), ptr(last), ptr(ns)))
    return {"n_records": cnt, "first_pos": first, "last_pos": last, "n_sample": int(ns[0])}


def vcf_scan(path: str, window_bytes: int = 0) -> dict:
    """Host-only walk of a bgzipped text VCF (no GPU): the record count, the first / last POS (0-based, as htslib's bcf1_t.pos), the
    header's sample count and the records' CHROM (colate_vcf_scan).  Raises ColateError for the files colate_rows_from_bcf refuses
    on the host, and for a BCF file (bcf_scan reads it)."""
    v = [np.zeros(1, t) for t in (np.int64, np.int32, np.int32, np.int32)]
    chrom = C.create_string_buffer(1 << 16)
    check(lib().colate_vcf_scan(str(path).encode(), window_bytes, *[ptr(x) for x in v], chrom, len(chrom)))
    out = {k: int(x[0]) for k, x in zip(("n_records", "first_pos", "last_pos", "n_sample"), v)}
    out["chrom"] = chrom.value.decode(errors="surrogateescape")
    return out


def read_fasta(path: str) -> np.ndarray:
    """fasta::Read (data.cpp:213-237): header line dropped, upper-cased, concatenated; <path> or <path>.gz."""
    p = C.POINTER(C.c_uint8)()
    n = check(lib().colate_read_fasta(str(path).encode(), C.byref(p)))
    try:
        return np.ctypeslib.as_array(p, shape=(n,)).copy() if n else np.zeros(0, np.uint8)
    finally:
        lib().colate_free(C.cast(p, C.c_void_p))


def maketmp_word(flipped: int, n_branch: int, mutation_type: bytes) -> int:
    """The make_tmp row word of a .mut row (colate_maketmp_word): bit 0 vcf filter, bit 1 bam filter, bit 2 one-letter derived string,
    byte 1 ancestral letter, byte 2 first derived letter."""
    return int(lib().colate_maketmp_word(flipped, n_branch, mutation_type))


def read_mut_words(path: str) -> np.ndarray:
    """The make_tmp row words of a .mut[.gz] file on the host (colate_read_mut_words), row for row as read_mut."""
    n = check(lib().colate_read_mut_words(str(path).encode(), 0, None))
    w = np.zeros(n, np.uint32)
    check(lib().colate_read_mut_words(str(path).encode(), n, ptr(w)))
    return w


def maketmp_mask_bits(path: str, pos: np.ndarray, row0: int, bits: np.ndarray):
    """The make_tmp mask rule at the site positions -> pass bits of rows [row0, row0+len(pos)) (colate_maketmp_mask_bits): rows at or
    beyond the mask's end are dropped, unlike mask_bits_from_fasta."""
    pos = np.ascontiguousarray(pos, dtype=np.int32)
    check(lib().colate_maketmp_mask_bits(str(path).encode(), pos.shape[0], ptr(pos), row0, ptr(bits)))


@dataclass
class Stage1Result:
    num_blocks: int
    block_stats: np.ndarray     # [num_blocks, 4, 185] fp64: shared, notshared, shared_emp, notshared_emp
    block_tallies: np.ndarray   # [num_blocks, 3, 185] int64: samples->shared, samples->notshared, rows->emp
    n_used: int
    mt_state: np.ndarray        # state window after the stage


class Handle:
    """One GPU.  Mirrors the data flow of mut(): readers -> parse_tmptmp -> bootstrap -> EM."""

    def __init__(self, device: int = 0):
        h = C.c_void_p()
        check(lib().colate_create(device, C.byref(h)))
        self._h = h
        self.n_chr = 0
        self.n_site = 0

    def close(self):
        if self._h:
            lib().colate_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self) -> int:
        return lib().colate_stream(self._h)

    # ---- inputs
    def set_sites(self, site_off, pos, age_begin, age_end, meta):
        site_off = np.ascontiguousarray(site_off, dtype=np.int64)
        self.n_chr = site_off.shape[0] - 1
        self.n_site = int(site_off[-1])
        a = [np.ascontiguousarray(x, dtype=dt) for x, dt in ((pos, np.int32), (age_begin, np.float32), (age_end, np.float32), (meta, np.uint32))]
        check(lib().colate_set_sites(self._h, self.n_chr, ptr(site_off), *[ptr(x) for x in a], 0))

    def set_sites_device(self, n_chr, n_site, site_off_ptr, pos_ptr, ab_ptr, ae_ptr, meta_ptr):
        """Device pointers (e.g. torch tensors' data_ptr()); site_off_ptr is a device pointer too."""
        self.n_chr, self.n_site = n_chr, n_site
        check(lib().colate_set_sites(self._h, n_chr, C.c_void_p(site_off_ptr), C.c_void_p(pos_ptr), C.c_void_p(ab_ptr),
                                     C.c_void_p(ae_ptr), C.c_void_p(meta_ptr), 1))

    def set_genome(self, slot, rec_chrom, bp, aaf, daf, alleles):
        first, end = chr_ranges(self.n_chr, rec_chrom)
        a = [np.ascontiguousarray(x, dtype=dt) for x, dt in ((bp, np.int32), (aaf, np.int32), (daf, np.int32), (alleles, np.uint16))]
        check(lib().colate_set_genome(self._h, slot, a[0].shape[0], ptr(first), ptr(end), *[ptr(x) for x in a], 0))
        return first, end

    def set_genome_device(self, slot, n_rec, first_ptr, end_ptr, bp_ptr, aaf_ptr, daf_ptr, alleles_ptr):
        check(lib().colate_set_genome(self._h, slot, n_rec, C.c_void_p(first_ptr), C.c_void_p(end_ptr), C.c_void_p(bp_ptr),
                                      C.c_void_p(aaf_ptr), C.c_void_p(daf_ptr), C.c_void_p(alleles_ptr), 1))

    def set_pileup(self, slot, counts):
        """N3 (bam / bcf front-ends from pre-decoded arrays): counts[n_site][4] = reads showing A, C, G, T at every .mut row's
        position (zeros: not covered) instead of a .colate.in record stream.  Use with set_option("front_end", 1)."""
        counts = np.ascontiguousarray(counts, dtype=np.int32)
        assert counts.shape == (self.n_site, 4)
        check(lib().colate_set_pileup(self._h, slot, ptr(counts), 0))

    def set_row_counts(self, slot, aaf, daf):
        """N3, bcf front-ends: per-row counts of the row's ancestral / derived allele as a bcf decoder resolved them (zeros: row
        not usable for this genome).  Use with set_option("front_end", 1)."""
        a = np.ascontiguousarray(aaf, dtype=np.int32); d = np.ascontiguousarray(daf, dtype=np.int32)
        assert a.shape == (self.n_site,) and d.shape == (self.n_site,)
        check(lib().colate_set_row_counts(self._h, slot, ptr(a), ptr(d), 0))

    def pileup_from_reads(self, slot, per_chr_reads, ref_genomes, filters=(20, 30, 10), fetch=False):
        """N3, the decoder's counting loop on the device: per_chr_reads[c] = (pos int32[n], mapq uint8[n], len int32[n],
        seq_off int64[n], seq uint8[bytes], qual uint8[bytes]) of contig c (or None), ref_genomes[c] = uint8 sequence of the
        contig.  Makes `slot` a pileup genome; fetch=True returns counts[n_site][4]."""
        check(lib().colate_pileup_begin(self._h, slot))
        for c, rd in enumerate(per_chr_reads):
            if rd is None or len(rd[0]) == 0:
                continue
            pos, mapq, ln, off, seq, qual = [np.ascontiguousarray(a, dtype=dt) for a, dt in zip(rd, (np.int32, np.uint8, np.int32, np.int64, np.uint8, np.uint8))]
            ref = np.ascontiguousarray(ref_genomes[c], dtype=np.uint8)
            check(lib().colate_pileup_reads(self._h, slot, c, pos.shape[0], ptr(pos), ptr(mapq), ptr(ln), ptr(off), ptr(seq), ptr(qual), ptr(ref),
                                            ref.shape[0], *filters))
        out = np.zeros((self.n_site, 4), dtype=np.int32) if fetch else None
        check(lib().colate_pileup_end(self._h, slot, ptr(out) if fetch else None))
        return out

    def pileup_from_bam(self, slot, path, chr_names, ref_genomes, filters=(20, 30, 10), chunk_bytes=0, fetch=False):
        """The same pileup straight from a BAM file (colate_pileup_bam): chr_names = the site set's --chr list (header contig <name> or
        chr<name>), ref_genomes[c] = uint8 / bytes sequence of contig c (upper-cased on the device as fasta::Read does), or None for
        the genome of set_ref_genome.  BGZF is
        inflated on the host, the records are decoded and counted on the device in chunks of at most chunk_bytes record bytes (0:
        64 MiB).  Makes `slot` a pileup genome; fetch=True returns counts[n_site][4]."""
        n = len(chr_names)
        names = (C.c_char_p * n)(*[s.encode() for s in chr_names])
        seqs = lens = None                       # ref_genomes None: the resident genome of set_ref_genome
        if ref_genomes is not None:
            refs = [np.ascontiguousarray(np.frombuffer(g, np.uint8) if isinstance(g, (bytes, bytearray)) else g, dtype=np.uint8) for g in ref_genomes]
            seqs = (C.c_void_p * n)(*[r.ctypes.data if r.shape[0] else None for r in refs])
            lens = np.array([r.shape[0] for r in refs], dtype=np.int64)
        out = np.zeros((self.n_site, 4), dtype=np.int32) if fetch else None
        check(lib().colate_pileup_bam(self._h, slot, str(path).encode(), n, names, seqs, ptr(lens), *filters, chunk_bytes, ptr(out) if fetch else None))
        return out

    # ---- make_tmp for many targets (DESIGN.md section 6i)
    def set_ref_genome(self, ref_genomes):
        """Upload --ref_genome once (colate_set_ref_genome): ref_genomes[c] = uint8 / bytes contig per --chr entry.  pileup_from_bam
        with ref_genomes=None and maketmp_write_bcf read it on the device."""
        n = len(ref_genomes)
        refs = [np.ascontiguousarray(np.frombuffer(g, np.uint8) if isinstance(g, (bytes, bytearray)) else g, dtype=np.uint8) for g in ref_genomes]
        seqs = (C.c_void_p * n)(*[r.ctypes.data if r.shape[0] else None for r in refs])
        lens = np.array([r.shape[0] for r in refs], dtype=np.int64)
        check(lib().colate_set_ref_genome(self._h, n, seqs, ptr(lens)))

    def set_maketmp_words(self, words):
        """make_tmp row words for sites given with set_sites (read_mut_words); ingest_mut* builds them itself."""
        w = np.ascontiguousarray(words, dtype=np.uint32)
        assert w.shape == (self.n_site,)
        check(lib().colate_set_maketmp_words(self._h, ptr(w), 0))

    def maketmp_words(self, row0=0, n_rows=None):
        n = self.n_site - row0 if n_rows is None else n_rows
        w = np.zeros(n, np.uint32)
        check(lib().colate_fetch_maketmp_words(self._h, row0, n, ptr(w)))
        return w

    def maketmp_write_pileup(self, slot, chr_names, out_file, mask_bits=None) -> int:
        """The .colate.in of pileup slot `slot` written on the device (colate_maketmp_write_pileup); returns the records written."""
        names = (C.c_char_p * len(chr_names))(*[s.encode() for s in chr_names])
        mb = None if mask_bits is None else np.ascontiguousarray(mask_bits, dtype=np.uint32)
        return check(lib().colate_maketmp_write_pileup(self._h, slot, len(chr_names), names, ptr(mb), str(out_file).encode()))

    def maketmp_write_bcf(self, paths, chr_names, out_file, mask_bits=None, chunk_bytes=0) -> int:
        """The .colate.in of one BCF / VCF target (paths[c] per --chr entry) written on the device (colate_maketmp_write_bcf)."""
        n = len(paths)
        names = (C.c_char_p * n)(*[s.encode() for s in chr_names])
        files = (C.c_char_p * n)(*[str(p).encode() for p in paths])
        mb = None if mask_bits is None else np.ascontiguousarray(mask_bits, dtype=np.uint32)
        return check(lib().colate_maketmp_write_bcf(self._h, n, names, files, ptr(mb), chunk_bytes, str(out_file).encode()))

    def maketmp_write_bcf_genome(self, path, chr_names, out_file, mask_bits=None, chunk_bytes=0) -> int:
        """maketmp_write_bcf from one whole-genome BCF / VCF file (colate_maketmp_write_bcf_genome): chromosome c reads the contig
        chr_names[c] or chr<chr_names[c]>."""
        n = len(chr_names)
        names = (C.c_char_p * n)(*[str(s).encode() for s in chr_names])
        mb = None if mask_bits is None else np.ascontiguousarray(mask_bits, dtype=np.uint32)
        return check(lib().colate_maketmp_write_bcf_genome(self._h, n, names, str(path).encode(), ptr(mb), chunk_bytes, str(out_file).encode()))

    def last_maketmp_timing(self) -> dict:
        t = np.zeros(4)
        check(lib().colate_last_maketmp_timing(self._h, t))
        return dict(zip(("kernel_ms", "d2h_ms", "write_s", "records"), t.tolist()))

    def upload_counts(self) -> dict:
        c = np.zeros(4, np.int64)
        check(lib().colate_upload_counts(self._h, c))
        return dict(zip(("mut_texts_parsed", "mut_rows_parsed", "ref_uploads", "ref_h2d_bytes"), c.tolist()))

    def last_bam_timing(self) -> dict:
        """Phases of the last pileup_from_bam (colate_last_bam_timing; copy / decode / pileup need set_option("bam_timing", 1))."""
        t = np.zeros(10)
        check(lib().colate_last_bam_timing(self._h, t))
        keys = ("index_s", "inflate_s", "walk_s", "h2d_ms", "decode_ms", "pileup_ms", "total_s", "threads", "inflated_bytes", "records")
        return dict(zip(keys, t.tolist()))

    def rows_from_bcf(self, slot, paths, role, ref_genomes=None, chunk_bytes=0, fetch=False):
        """The row counts of genome `slot` straight from BCF or bgzipped text VCF files (colate_rows_from_bcf): paths[c] = the file
        of chromosome c of the site set (the reference's <prefix>_chr<c>.bcf, either format, as htslib reads it), role "target" / "reference" (or 0 / 1), ref_genomes[c] = uint8 / bytes
        sequence of contig c of --ref_genome or None.  BGZF is inflated on the host, the records are decoded and resolved on the
        device.  Makes `slot` a row-count genome (use with front_end = 1); fetch=True returns (aaf, daf) per row."""
        role = {"target": 0, "reference": 1}.get(role, role)
        n = len(paths)
        names = (C.c_char_p * n)(*[str(c).encode() for c in range(n)])
        files = (C.c_char_p * n)(*[str(p).encode() for p in paths])
        seqs = lens = None
        if ref_genomes is not None:
            refs = [np.ascontiguousarray(np.frombuffer(g, np.uint8) if isinstance(g, (bytes, bytearray)) else g, dtype=np.uint8) for g in ref_genomes]
            seqs = (C.c_void_p * n)(*[r.ctypes.data if r.shape[0] else None for r in refs])
            lens = np.array([r.shape[0] for r in refs], dtype=np.int64)
        aaf = np.zeros(self.n_site, np.int32) if fetch else None
        daf = np.zeros(self.n_site, np.int32) if fetch else None
        check(lib().colate_rows_from_bcf(self._h, slot, role, n, names, files, C.cast(seqs, C.c_void_p) if seqs is not None else None,
                                         ptr(lens) if lens is not None else None, chunk_bytes, ptr(aaf) if fetch else None,
                                         ptr(daf) if fetch else None))
        return (aaf, daf) if fetch else None

    def rows_from_bcf_roles(self, target_slot, reference_slot, paths, genome=0, chunk_bytes=0):
        """Both roles' row counts from one decode of the files (colate_rows_from_bcf_roles): slot target_slot gets what
        rows_from_bcf(target_slot, paths, "target") gives, reference_slot what rows_from_bcf(reference_slot, paths, "reference")
        gives; either may be -1 to skip that role.  genome 0: no --ref_genome, 1: the genome of set_ref_genome, read on the device."""
        n = len(paths)
        names = (C.c_char_p * n)(*[str(c).encode() for c in range(n)])
        files = (C.c_char_p * n)(*[str(p).encode() for p in paths])
        check(lib().colate_rows_from_bcf_roles(self._h, int(target_slot), int(reference_slot), n, names, files, int(genome), chunk_bytes))

    def rows_from_bcf_genome(self, target_slot, reference_slot, path, chr_names, genome=0, chunk_bytes=0):
        """rows_from_bcf_roles from one whole-genome BCF / VCF file (colate_rows_from_bcf_genome): chromosome c of the site set reads
        the records of the contig chr_names[c] or chr<chr_names[c]>, as its own file would hold them.  The file is decoded once."""
        n = len(chr_names)
        names = (C.c_char_p * n)(*[str(s).encode() for s in chr_names])
        check(lib().colate_rows_from_bcf_genome(self._h, int(target_slot), int(reference_slot), n, names, str(path).encode(), int(genome),
                                                chunk_bytes))

    def decode_bcf_genome(self, path, chr_names, chunk_bytes=0) -> list:
        """decode_bcf of a whole-genome file (colate_decode_bcf_genome): per --chr entry the dict decode_bcf gives for its contig."""
        n = len(chr_names)
        names = (C.c_char_p * n)(*[str(s).encode() for s in chr_names])
        first = np.zeros(n, np.int64); cnt = np.zeros(n, np.int64); nh = np.zeros(n, np.int32)
        check(lib().colate_decode_bcf_genome(self._h, str(path).encode(), n, names, chunk_bytes, ptr(first), ptr(cnt), ptr(nh)))
        out = []
        for c in range(n):
            k = int(cnt[c])
            d = {"pos": np.zeros(k, np.int32), "a0": np.zeros(k, np.uint8), "a1": np.zeros(k, np.uint8), "alt_sum": np.zeros(k, np.int32),
                 "biallelic": np.zeros(k, np.uint8)}
            check(lib().colate_bcf_records(self._h, int(first[c]), k, *[ptr(d[x]) for x in ("pos", "a0", "a1", "alt_sum", "biallelic")]))
            d["n_hap"] = int(nh[c])
            out.append(d)
        return out

    def copy_genome(self, dst, src):
        """Slot src's per-row counts (a pileup or row-count genome) copied into slot dst on the device, dst's mask and join state
        cleared (colate_copy_genome): one decoded file under several masks."""
        check(lib().colate_copy_genome(self._h, int(dst), int(src)))

    def decode_bcf(self, path, chunk_bytes=0) -> dict:
        """One BCF or bgzipped text VCF file's records as the device reduces them (colate_decode_bcf + colate_bcf_records): pos (1-based), a0 / a1 (first
        two alleles: 0 empty or absent, the letter, 0xff longer), alt_sum (sum of the GT allele indices), biallelic, and n_hap."""
        n = np.zeros(1, np.int64)
        nh = np.zeros(1, np.int32)
        check(lib().colate_decode_bcf(self._h, str(path).encode(), chunk_bytes, ptr(n), ptr(nh)))
        k = int(n[0])
        out = {"pos": np.zeros(k, np.int32), "a0": np.zeros(k, np.uint8), "a1": np.zeros(k, np.uint8), "alt_sum": np.zeros(k, np.int32),
               "biallelic": np.zeros(k, np.uint8)}
        check(lib().colate_bcf_records(self._h, 0, k, *[ptr(out[x]) for x in ("pos", "a0", "a1", "alt_sum", "biallelic")]))
        out["n_hap"] = int(nh[0])
        return out

    def last_bcf_timing(self) -> dict:
        """Phases of the last rows_from_bcf / decode_bcf (colate_last_bcf_timing; copy / decode / rows need set_option("bcf_timing", 1))."""
        t = np.zeros(10)
        check(lib().colate_last_bcf_timing(self._h, t))
        keys = ("index_s", "inflate_s", "walk_s", "h2d_ms", "decode_ms", "rows_ms", "total_s", "threads", "inflated_bytes", "records")
        return dict(zip(keys, t.tolist()))

    def set_mask(self, slot, pass_bits):
        if pass_bits is None:
            check(lib().colate_set_mask(self._h, slot, None, 0))
        else:
            pass_bits = np.ascontiguousarray(pass_bits, dtype=np.uint32)
            assert pass_bits.shape[0] == (self.n_site + 31) // 32
            check(lib().colate_set_mask(self._h, slot, ptr(pass_bits), 0))

    def ingest_mut(self, texts, row_capacity=None):
        """GPU-side ingest of Relate .mut text (one bytes object per --chr entry, in order) straight into the
        handle's site arrays: replaces read_mut() + set_sites().  Returns rows per chromosome."""
        if row_capacity is None:
            row_capacity = sum(t.count(b"\n") + 1 for t in texts)
        check(lib().colate_ingest_begin(self._h, len(texts), row_capacity))
        rows = []
        for t in texts:
            buf = np.frombuffer(t, dtype=np.uint8) if len(t) else np.zeros(1, np.uint8)
            rows.append(check(lib().colate_ingest_mut_text(self._h, C.c_void_p(buf.ctypes.data), len(t), 0)))
        check(lib().colate_ingest_end(self._h))
        self.n_chr = len(texts)
        self.n_site = int(sum(rows))
        return rows

    def ingest_mut_bytes(self, bufs, row_capacity=None):
        """Same as ingest_mut for uint8 arrays (pinned host memory: torch.Tensor.pin_memory().numpy()): ONE call for all
        chromosomes, the copies run on the handle's copy stream under the parse kernels of the chromosomes before."""
        n = len(bufs)
        if row_capacity is None:
            row_capacity = sum(int(b.shape[0]) for b in bufs) // 20 + n     # a data row has at least 10 fields
        check(lib().colate_ingest_begin(self._h, n, row_capacity))
        ptrs = (C.c_void_p * n)(*[b.ctypes.data for b in bufs])
        sizes = np.array([b.shape[0] for b in bufs], dtype=np.int64)
        rows = np.zeros(n, dtype=np.int64)
        check(lib().colate_ingest_mut_texts(self._h, n, ptrs, sizes, 0, ptr(rows)))
        check(lib().colate_ingest_end(self._h))
        self.n_chr = n
        self.n_site = int(rows.sum())
        return rows

    def ingest_mut_device(self, ptr_sizes, row_capacity=None):
        """ingest_mut for texts that already sit in device memory: [(device pointer, bytes)] per --chr entry."""
        n = len(ptr_sizes)
        if row_capacity is None:
            row_capacity = sum(int(b) for _, b in ptr_sizes) // 20 + n
        check(lib().colate_ingest_begin(self._h, n, row_capacity))
        ptrs = (C.c_void_p * n)(*[int(p) for p, _ in ptr_sizes])
        sizes = np.array([int(b) for _, b in ptr_sizes], dtype=np.int64)
        rows = np.zeros(n, dtype=np.int64)
        check(lib().colate_ingest_mut_texts(self._h, n, ptrs, sizes, 1, ptr(rows)))
        check(lib().colate_ingest_end(self._h))
        self.n_chr = n
        self.n_site = int(rows.sum())
        return rows

    def ingest_colate_in(self, slot, image, chr_names):
        """.colate.in image (bytes or a uint8 array, e.g. pinned) -> genome slot, decoded on the device.
        Replaces read_colate_in() + set_genome().  Returns the number of records."""
        buf = np.frombuffer(image, dtype=np.uint8) if isinstance(image, (bytes, bytearray, memoryview)) else image
        names = (C.c_char_p * len(chr_names))(*[s.encode() for s in chr_names])
        return check(lib().colate_ingest_colate_in(self._h, slot, C.c_void_p(buf.ctypes.data if buf.shape[0] else None), int(buf.shape[0]),
                                                   len(chr_names), names, 0))

    def ingest_fetch(self, row0=0, n_rows=None):
        n = self.n_site - row0 if n_rows is None else n_rows
        pos = np.zeros(n, np.int32); ab = np.zeros(n, np.float32); ae = np.zeros(n, np.float32); meta = np.zeros(n, np.uint32)
        check(lib().colate_ingest_fetch(self._h, row0, n, ptr(pos), ptr(ab), ptr(ae), ptr(meta)))
        return pos, ab, ae, meta

    def ingest_stats(self):
        ms, fb = C.c_double(0), C.c_int64(0)
        check(lib().colate_ingest_stats(self._h, C.byref(ms), C.byref(fb)))
        return dict(kernel_ms=ms.value, host_fallback_rows=fb.value)

    def set_stream_cache(self, enable: bool):
        """Reuse the generator stream across stage-i calls that start from the same state (all-pairs jobs)."""
        check(lib().colate_set_stream_cache(self._h, 1 if enable else 0))

    # ---- stage i
    def stage1_flags(self, target_slot=0, reference_slot=1):
        used = np.zeros(self.n_chr, dtype=np.int64)
        blocks = np.zeros(self.n_chr, dtype=np.int32)
        check(lib().colate_stage1_flags(self._h, target_slot, reference_slot, ptr(used), ptr(blocks)))
        return used, blocks

    def stage1_sample(self, mt_state, used_rank_base=0, block_base=0, n_blocks=None, want_state=True):
        nb = MAX_BLOCKS if n_blocks is None else n_blocks
        stats = np.zeros((nb, 4, NBINS))
        tallies = np.zeros((nb, 3, NBINS), dtype=np.int64)
        mt_state = np.ascontiguousarray(mt_state, dtype=np.uint32)
        out_state = np.zeros(MT_WORDS, dtype=np.uint32) if want_state else None
        check(lib().colate_stage1_sample(self._h, ptr(mt_state), used_rank_base, block_base, ptr(stats), ptr(tallies),
                                         ptr(out_state)))
        return stats, tallies, out_state

    def stage1_sample_dev(self, mt_state, used_rank_base, block_base, stats_ptr, tallies_ptr, want_state=True):
        """stage1_sample with DEVICE destinations (e.g. rows of a torch tensor: tensor.data_ptr() + offset)."""
        mt_state = np.ascontiguousarray(mt_state, dtype=np.uint32)
        out_state = np.zeros(MT_WORDS, dtype=np.uint32) if want_state else None
        check(lib().colate_stage1_sample(self._h, ptr(mt_state), used_rank_base, block_base,
                                         C.c_void_p(stats_ptr) if stats_ptr else None, C.c_void_p(tallies_ptr) if tallies_ptr else None,
                                         ptr(out_state)))
        return out_state

    def stage2_bootstrap_dev(self, block_weights, stats_ptr, num_blocks, age=0.0, fetch=False):
        """stage2_bootstrap on block histograms that already sit on the device: stats_ptr = device pointer to
        [num_blocks][4][185] fp64, or None for what the last stage1 call left in the handle.  Counts stay on the device
        (fetch=True: also returned, [R][2][185])."""
        w = np.ascontiguousarray(block_weights, dtype=np.int32)
        assert w.shape[1] == num_blocks
        counts = np.zeros((w.shape[0], 2, NBINS)) if fetch else None
        check(lib().colate_stage2_bootstrap(self._h, w.shape[0], num_blocks, ptr(w), C.c_void_p(stats_ptr) if stats_ptr else None, age, ptr(counts)))
        return counts

    def stage1(self, mt_state, target_slot=0, reference_slot=1, fetch=True) -> Stage1Result:
        """parse_tmptmp (coal.cpp:2072) on one GPU.  fetch=False: the histograms stay on the device
        (stage2_bootstrap_dev(w, None, num_blocks)); block_stats / block_tallies of the result are None."""
        if not fetch:
            nb, nu = C.c_int(0), C.c_int64(0)
            mt_state = np.ascontiguousarray(mt_state, dtype=np.uint32)
            out_state = np.zeros(MT_WORDS, dtype=np.uint32)
            check(lib().colate_stage1(self._h, target_slot, reference_slot, ptr(mt_state), C.byref(nb), None, None, C.byref(nu), ptr(out_state)))
            return Stage1Result(nb.value, None, None, nu.value, out_state)
        stats = np.zeros((MAX_BLOCKS, 4, NBINS))
        tallies = np.zeros((MAX_BLOCKS, 3, NBINS), dtype=np.int64)
        nb, nu = C.c_int(0), C.c_int64(0)
        mt_state = np.ascontiguousarray(mt_state, dtype=np.uint32)
        out_state = np.zeros(MT_WORDS, dtype=np.uint32)
        check(lib().colate_stage1(self._h, target_slot, reference_slot, ptr(mt_state), C.byref(nb), ptr(stats), ptr(tallies),
                                  C.byref(nu), ptr(out_state)))
        return Stage1Result(nb.value, stats[:nb.value].copy(), tallies[:nb.value].copy(), nu.value, out_state)

    def set_option(self, key: str, value: int):
        check(lib().colate_set_option(self._h, key.encode(), value))

    def extra_words(self) -> int:
        """Generator words the last stage-i call consumed beyond 200 per used row (redraws, coal.cpp:2279-2294)."""
        return lib().colate_last_stage1_extra_words(self._h)

    def launch_count(self) -> int:
        return lib().colate_launch_count(self._h)

    def stage1_timing(self) -> dict:
        t = _lib.Stage1Timing()
        check(lib().colate_last_stage1_timing(self._h, C.byref(t)))
        return {k: getattr(t, k) for k, _ in t._fields_}

    # ---- stage ii / iii
    def stage2_bootstrap(self, block_weights, block_stats, age=0.0, fetch=True):
        w = np.ascontiguousarray(block_weights, dtype=np.int32)
        R, nb = w.shape
        bs = np.ascontiguousarray(block_stats, dtype=np.float64)
        assert bs.shape == (nb, 4, NBINS)
        counts = np.zeros((R, 2, NBINS)) if fetch else None
        check(lib().colate_stage2_bootstrap(self._h, R, nb, ptr(w), ptr(bs), age, ptr(counts)))
        return counts

    def stage3_em(self, R, epochs, rates_init, counts=None, max_iter=100000):
        ep = np.ascontiguousarray(epochs, dtype=np.float64)
        ri = np.ascontiguousarray(rates_init, dtype=np.float64)
        E = ep.shape[0]
        cn = None if counts is None else np.ascontiguousarray(counts, dtype=np.float64)
        rates = np.zeros((R, E)); iters = np.zeros(R, dtype=np.int32); ll = np.zeros(R)
        check(lib().colate_stage3_em(self._h, R, E, ptr(ep), ptr(ri), ptr(cn), max_iter, ptr(rates), ptr(iters), ptr(ll)))
        return rates, iters, ll

    def stage3_em_begin(self, R, epochs, rates_init, max_iter=100000):
        """Queue the EM of the device-resident counts on the handle's EM stream and return (colate_stage3_em_begin): the next
        pair can be uploaded and taken through stage i meanwhile.  stage3_em_end() fetches the results."""
        ep = np.ascontiguousarray(epochs, dtype=np.float64)
        ri = np.ascontiguousarray(rates_init, dtype=np.float64)
        self._em_shape = (R, ep.shape[0])
        check(lib().colate_stage3_em_begin(self._h, R, ep.shape[0], ptr(ep), ptr(ri), max_iter))

    def stage3_em_end(self):
        R, E = self._em_shape
        rates = np.zeros((R, E)); iters = np.zeros(R, dtype=np.int32); ll = np.zeros(R)
        check(lib().colate_stage3_em_end(self._h, ptr(rates), ptr(iters), ptr(ll)))
        return rates, iters, ll

    def stage3_em_grids(self, grid_of, grids, counts, max_iter=100000):
        """EM of R replicates on mixed epoch grids (colate_stage3_em_grids): grids = [(epochs, rates_init)], replicate r runs on
        grids[grid_of[r]] with counts[r] ([R][2][185]).  Returns (rates[R][E_max] zero-padded, iters[R], ll[R]); row r equals
        stage3_em(1, *grids[grid_of[r]], counts[r:r+1]) bit for bit."""
        go = np.ascontiguousarray(grid_of, dtype=np.int32)
        R = go.shape[0]
        eps = [np.ascontiguousarray(e, dtype=np.float64) for e, _ in grids]
        ris = [np.ascontiguousarray(r, dtype=np.float64) for _, r in grids]
        gE = np.array([e.shape[0] for e in eps], dtype=np.int32)
        assert all(r.shape == e.shape for e, r in zip(eps, ris))
        goff = np.concatenate([[0], np.cumsum(gE)[:-1]]).astype(np.int64)
        cn = np.ascontiguousarray(counts, dtype=np.float64)
        assert cn.shape == (R, 2, NBINS)
        E_max = int(gE.max())
        rates = np.zeros((R, E_max)); iters = np.zeros(R, dtype=np.int32); ll = np.zeros(R)
        check(lib().colate_stage3_em_grids(self._h, R, go, len(eps), gE, goff, np.concatenate(eps), np.concatenate(ris),
                                           cn.reshape(-1), max_iter, rates.reshape(-1), iters, ll))
        return rates, iters, ll

    def estep(self, shared: bool, epochs, rates, t):
        ep = np.ascontiguousarray(epochs, dtype=np.float64)
        r = np.ascontiguousarray(rates, dtype=np.float64)
        t = np.ascontiguousarray(t, dtype=np.float64)
        E, n = ep.shape[0], t.shape[0]
        num, den, ll = np.zeros((n, E)), np.zeros((n, E)), np.zeros(n)
        check(lib().colate_estep(self._h, 1 if shared else 0, E, ptr(ep), ptr(r), n, ptr(t), ptr(num), ptr(den), ptr(ll)))
        return ll, num, den

    def libm(self, which: str, x):
        """Test hook: the device's glibc-exact exp / log / log1p on an array."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.zeros_like(x)
        check(lib().colate_test_libm(self._h, {"exp": 0, "log": 1, "log1p": 2}[which], x.shape[0], x, y))
        return y

    EM_PRIMS = ("exp_main", "log1p_k0", "log1p_wide", "div_midrange", "lse", "lse_wide", "lme")

    def em_prims(self, which: str, a, b=None):
        """Test hook: one straight-line piece of the EM folds on the device, element by element -> (y, ok).  ok: the piece's
        validity predicate (exp_is_main, log1p_is_k0, log1p_wide_ok; always 1 for div_midrange), or for lse / lse_wide / lme
        whether the straight-line path was taken.  b: second operand of div_midrange / lse / lse_wide / lme."""
        a = np.ascontiguousarray(a, dtype=np.float64)
        bb = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
        assert bb is None or bb.shape == a.shape
        y, ok = np.zeros_like(a), np.zeros(a.shape[0], dtype=np.int32)
        check(lib().colate_test_em_prims(self._h, self.EM_PRIMS.index(which), a.shape[0], a, ptr(bb), y, ok))
        return y, ok

    def last_vcf_paths(self):
        """Test hook: (lines on k_vcf_decode's fast path only, lines with a general-path step) of the last decode_bcf /
        rows_from_bcf file; counted only with set_option("vcf_paths", 1), else (0, 0), as after a BCF file."""
        f, g = C.c_int64(0), C.c_int64(0)
        check(lib().colate_test_last_vcf_paths(self._h, C.byref(f), C.byref(g)))
        return f.value, g.value

    def last_em(self):
        """Test hook: (kernel, CTAs per replicate) of the last EM launch; kernel is "task" (k_em), "split" (k_em_split),
        "cta" (k_em_cta / k_em_cta_grids) or None."""
        k, c = C.c_int(0), C.c_int(0)
        check(lib().colate_test_last_em(self._h, C.byref(k), C.byref(c)))
        return {0: "task", 1: "split", 2: "cta"}.get(k.value), c.value

    def bin_fast(self, ages):
        """Test hook: k_sample's table-free age-bin index (-1 = sample flagged for the exact table) and the exact one."""
        a = np.ascontiguousarray(ages, dtype=np.float64)
        fast, exact = np.zeros(a.shape[0], dtype=np.int32), np.zeros(a.shape[0], dtype=np.int32)
        check(lib().colate_test_bin_fast(self._h, a.shape[0], a, fast, exact))
        return fast, exact

    def bin_sweep(self, lo_bits, hi_bits):
        """Test hook: every float with bit pattern in [lo, hi) through both bin indices on the device:
        (flagged, unflagged mismatches, max |t_fast - t| in 1e-9)."""
        out = np.zeros(3, dtype=np.uint64)
        check(lib().colate_test_bin_sweep(self._h, lo_bits, hi_bits, out))
        return int(out[0]), int(out[1]), int(out[2]) * 1e-9

    def mt_stream(self, mt_state, word0, n_words, log2_chunk_sites=3):
        """Test hook: engine words [word0, word0+n) generated by the device path (+ window after)."""
        out = np.zeros(n_words + MT_WORDS, dtype=np.uint32)
        check(lib().colate_test_mt_stream(self._h, np.ascontiguousarray(mt_state, dtype=np.uint32), word0, n_words,
                                          log2_chunk_sites, out))
        return out[:n_words], out[n_words:]

    # ---- convenience: load a synth.Sites / synth.Genome pair
    def load(self, sites, target, reference, tmask=None, rmask=None):
        self.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
        for slot, g in ((0, target), (1, reference)):
            self.set_genome(slot, g.chrom, g.bp, g.aaf, g.daf, g.anc.astype(np.uint16) | (g.der.astype(np.uint16) << 8))
        self.set_mask(0, None if tmask is None else mask_bits_from_seq(tmask, sites.site_off, sites.pos))
        self.set_mask(1, None if rmask is None else mask_bits_from_seq(rmask, sites.site_off, sites.pos))


def mut(handle: Handle, seed: int, bins: str | None = "3,7,0.2", num_bootstraps: int = 1, target_age=None,
        reference_age=None, years_per_gen=None, coal_file: str | None = None, max_iter: int = 100000):
    """mut() (coal.cpp:3071-3863) after the readers: stage i -> ii -> iii on one GPU.
    Returns dict(epochs, rates[R,E], iters[R], ep_null, is_ancient, num_blocks, stage1=Stage1Result, counts)."""
    age, ypg = ages(target_age, reference_age, years_per_gen)
    state = mt_seed(seed)
    s1 = handle.stage1(state)
    w = draw_block_weights(s1.mt_state, num_bootstraps, s1.num_blocks)
    counts = handle.stage2_bootstrap(w, s1.block_stats, age)
    if coal_file is not None:
        epochs, rates_init = epochs_from_coal_file(coal_file, age)
        ep_null = 0
    else:
        epochs, ep_null = epochs_from_bins(bins, age, ypg)
        rates_init = np.full(epochs.shape[0], 1.0 / 20000.0)
    rates, iters, ll = handle.stage3_em(num_bootstraps, epochs, rates_init, None, max_iter)
    return dict(epochs=epochs, rates=rates, iters=iters, ll=ll, ep_null=ep_null, is_ancient=age > 0.0,
                num_blocks=s1.num_blocks, stage1=s1, counts=counts, weights=w)


def write_coal(path: str, epochs, rates, is_ancient=False, ep_null=0):
    r = np.ascontiguousarray(rates, dtype=np.float64).copy()
    check(lib().colate_write_coal(path.encode(), r.shape[0], r.shape[1], np.ascontiguousarray(epochs, dtype=np.float64), r,
                                  1 if is_ancient else 0, ep_null))
    return r


def write_bin(path: str, epochs, rates, iters):
    r = np.ascontiguousarray(rates, dtype=np.float64)
    check(lib().colate_write_bin(path.encode(), r.shape[0], r.shape[1], np.ascontiguousarray(epochs, dtype=np.float64), r,
                                 np.ascontiguousarray(iters, dtype=np.int32)))


def write_colate_mat(path: str, counts, age_bin=None):
    """<out>.colate_mat (coal.cpp:3336-3343, 3453-3465): counts[R][2][185], already normalised."""
    c = np.ascontiguousarray(counts, dtype=np.float64)
    ab = age_bins() if age_bin is None else np.ascontiguousarray(age_bin, dtype=np.float64)
    check(lib().colate_write_colate_mat(path.encode(), c.shape[0], ab, c))
