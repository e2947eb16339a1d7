"""Seeded synthetic inputs of the shapes BASELINE.json names (SURVEY.md 8d).

Produces the parsed structure-of-arrays the C-ABI consumes and, for file-level tests and
the reference arm, the same data as the reference's on-disk formats (SURVEY.md App. B):
Relate ``.mut`` text, ``.colate.in`` binary records, P/N fasta masks and a ``--chr`` list.

Generator: numpy ``default_rng(seed)`` (PCG64).  Ages are generated as float32 and written
with their shortest round-trip repr, so ``strtof`` of the file gives the array bit for bit.
"""
from __future__ import annotations

import os
from dataclasses import dataclass, field

import numpy as np

# GRCh37-like autosome lengths (bp), used for the whole-genome shapes
AUTOSOME_LEN = [249250621, 243199373, 198022430, 191154276, 180915260, 171115067, 159138663,
                146364022, 141213431, 135534747, 135006516, 133851895, 115169878, 107349540,
                102531392, 90354753, 81195210, 78077248, 59128983, 63025520, 48129895, 51304566]

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


@dataclass
class Sites:
    """Rows of the per-chromosome .mut files, concatenated in --chr order."""
    chr_names: list
    site_off: np.ndarray      # int64 [n_chr+1]
    pos: np.ndarray           # int32
    age_begin: np.ndarray     # float32
    age_end: np.ndarray       # float32
    flipped: np.ndarray       # uint8
    n_branch: np.ndarray      # int32
    anc: np.ndarray           # uint8 first char of the ancestral allele string
    der: np.ndarray           # uint8 first char of the derived allele string
    odd: np.ndarray           # uint8: 0 normal "X/Y"; 1 multi-base ancestral; 2 no '/' ("NA")
    chrom_len: list = field(default_factory=list)

    @property
    def n(self):
        return int(self.pos.shape[0])

    def meta(self) -> np.ndarray:
        """Packed site word (bit0 = row passes coal.cpp:2150/2166/2175-2176, byte1 anc, byte2 der)."""
        ok = (self.flipped == 0) & (self.n_branch == 1) & (self.age_begin < self.age_end) & (self.age_end >= 0)
        ok &= self.odd == 0
        ok &= np.isin(self.anc, np.frombuffer(b"ACGT0", dtype=np.uint8))
        ok &= np.isin(self.der, np.frombuffer(b"ACGT1", dtype=np.uint8))
        m = ok.astype(np.uint32) | (self.anc.astype(np.uint32) << 8) | (self.der.astype(np.uint32) << 16)
        return np.where(ok, m, 0).astype(np.uint32)


@dataclass
class Genome:
    """Records of one .colate.in file in file order."""
    chrom: np.ndarray   # int32 index into chr_names (>= n_chr: a name not in the list)
    bp: np.ndarray      # int32
    anc: np.ndarray     # uint8
    der: np.ndarray     # uint8
    aaf: np.ndarray     # int32
    daf: np.ndarray     # int32

    @property
    def n(self):
        return int(self.bp.shape[0])


def _loguniform(rng, lo, hi, n):
    return np.exp(rng.uniform(np.log(lo), np.log(hi), n))


def make_sites(seed: int, rows_per_chr, chrom_len, chr_names=None, weird: float = 0.0) -> Sites:
    """SURVEY.md 8d config-1 distributions.  ``weird`` adds a fraction of rows that exercise
    the filter edge cases (multi-base alleles, missing '/', age_begin >= age_end, negative
    age_begin, 0/1 allele codes)."""
    rng = np.random.default_rng(seed)
    n_chr = len(rows_per_chr)
    chr_names = chr_names or [str(i + 1) for i in range(n_chr)]
    off = np.zeros(n_chr + 1, dtype=np.int64)
    off[1:] = np.cumsum(rows_per_chr)
    n = int(off[-1])
    pos = np.empty(n, dtype=np.int32)
    for c in range(n_chr):
        k = int(rows_per_chr[c])
        L = int(chrom_len[c])
        if k > L - 1:
            raise ValueError("more rows than positions")
        if k * 4 < L:
            p = np.unique(rng.integers(1, L, size=int(k * 1.05) + 16))
            while p.shape[0] < k:
                p = np.unique(np.concatenate([p, rng.integers(1, L, size=k)]))
            p = np.sort(rng.choice(p, size=k, replace=False)) if p.shape[0] > k else p
        else:
            p = np.sort(rng.choice(np.arange(1, L), size=k, replace=False))
        pos[off[c]:off[c + 1]] = p
    ab = np.where(rng.random(n) < 0.3, 0.0, _loguniform(rng, 10.0, 2e4, n)).astype(np.float32)
    ae = (ab.astype(np.float64) + _loguniform(rng, 50.0, 5e4, n)).astype(np.float32)
    flipped = (rng.random(n) < 0.02).astype(np.uint8)
    n_branch = np.where(rng.random(n) < 0.03, 2, 1).astype(np.int32)
    a = rng.integers(0, 4, n)
    d = (a + rng.integers(1, 4, n)) % 4
    anc, der = ACGT[a].copy(), ACGT[d].copy()
    odd = np.zeros(n, dtype=np.uint8)
    if weird > 0:
        w = rng.random(n)
        odd[w < weird * 0.2] = 1
        odd[(w >= weird * 0.2) & (w < weird * 0.3)] = 2
        sw = (w >= weird * 0.3) & (w < weird * 0.5)          # age_begin >= age_end
        ae[sw] = ab[sw]
        ng = (w >= weird * 0.5) & (w < weird * 0.7)          # negative age_begin (clamped to 0)
        ab[ng] = -np.abs(ab[ng]) - np.float32(1.5)
        zo = (w >= weird * 0.7) & (w < weird * 0.85)         # '0'/'1' allele codes
        anc[zo], der[zo] = ord("0"), ord("1")
        bad = (w >= weird * 0.85) & (w < weird)              # allele outside ACGT
        anc[bad] = ord("N")
    return Sites(chr_names, off, pos, ab, ae, flipped, n_branch, anc, der, odd, list(chrom_len))


def add_deep_rows(sites: Sites, seed: int, frac: float = 0.02) -> np.ndarray:
    """Gives a fraction of the rows age intervals that reach past the age grid (bin 185 starts at ~9.3e6 generations)
    with age_begin > 0: for such rows the reference redraws every sample that falls beyond the grid (coal.cpp:2279-2294),
    consuming two more engine words per redraw.  Returns the indices of the modified rows."""
    rng = np.random.default_rng(seed)
    idx = np.nonzero(rng.random(sites.n) < frac)[0]
    ab = rng.uniform(2e6, 8.5e6, idx.shape[0])
    sites.age_begin[idx] = ab.astype(np.float32)
    sites.age_end[idx] = (ab + _loguniform(rng, 5e5, 4e7, idx.shape[0])).astype(np.float32)
    return idx


def make_genome(seed: int, sites: Sites, p_present: float = 0.7, mean_extra_reads: float = 1.0,
                p_derived: float = 0.3, weird: float = 0.0) -> Genome:
    """Record present w.p. ``p_present``; N = 1 + floor(Exp(mean_extra_reads)) reads, each derived
    w.p. ``p_derived``.  ``weird`` adds allele-swapped records, records at positions absent from
    the .mut file and zero-count records."""
    rng = np.random.default_rng(seed)
    n = sites.n
    keep = rng.random(n) < p_present
    idx = np.nonzero(keep)[0]
    k = idx.shape[0]
    chrom = (np.searchsorted(sites.site_off, idx, side="right") - 1).astype(np.int32)
    bp = sites.pos[idx].copy()
    anc = sites.anc[idx].copy()
    der = sites.der[idx].copy()
    N = 1 + np.floor(rng.exponential(mean_extra_reads, k)).astype(np.int64) if mean_extra_reads > 0 \
        else np.ones(k, dtype=np.int64)
    daf = rng.binomial(N, p_derived).astype(np.int32)
    aaf = (N - daf).astype(np.int32)
    if weird > 0:
        w = rng.random(k)
        sw = w < weird * 0.3
        anc[sw], der[sw] = der[sw].copy(), anc[sw].copy()
        z = (w >= weird * 0.3) & (w < weird * 0.5)
        daf[z] = 0
        aaf[(w >= weird * 0.4) & (w < weird * 0.5)] = 0
        # extra records at positions that are not rows of the .mut file
        ex = np.nonzero((w >= weird * 0.5) & (w < weird))[0]
        ebp = bp[ex] + 1
        ok = ~np.isin(ebp.astype(np.int64) + (chrom[ex].astype(np.int64) << 32),
                      sites.pos.astype(np.int64) + ((np.searchsorted(sites.site_off, np.arange(n), side="right") - 1).astype(np.int64) << 32))
        ex, ebp = ex[ok], ebp[ok]
        chrom = np.concatenate([chrom, chrom[ex]])
        bp = np.concatenate([bp, ebp])
        anc = np.concatenate([anc, anc[ex]])
        der = np.concatenate([der, der[ex]])
        aaf = np.concatenate([aaf, aaf[ex]])
        daf = np.concatenate([daf, daf[ex]])
        order = np.lexsort((bp, chrom))
        chrom, bp, anc, der, aaf, daf = (x[order] for x in (chrom, bp, anc, der, aaf, daf))
    return Genome(chrom.astype(np.int32), bp.astype(np.int32), anc.astype(np.uint8), der.astype(np.uint8),
                  aaf.astype(np.int32), daf.astype(np.int32))


def make_mask(seed: int, length: int, frac_n: float, run_lo=1000, run_hi=50000, lower=False) -> bytes:
    """P/N mask with ``frac_n`` of the bases 'N' in runs of run_lo..run_hi bp (config 4)."""
    rng = np.random.default_rng(seed)
    m = np.full(length, ord("P"), dtype=np.uint8)
    target = int(frac_n * length)
    done = 0
    while done < target:
        L = int(rng.integers(run_lo, run_hi + 1))
        s = int(rng.integers(0, max(1, length - L)))
        m[s:s + L] = ord("N")
        done += L
    if lower:
        m = np.where(m == ord("P"), ord("p"), ord("n")).astype(np.uint8)
    return m.tobytes()


def rows_for_genome(total_rows: int, lengths=AUTOSOME_LEN):
    tot = float(sum(lengths))
    rows = [int(total_rows * L / tot) for L in lengths]
    rows[0] += total_rows - sum(rows)
    return rows


# ------------------------------------------------------------------ file writers
def _fmt_f32(x) -> str:
    return np.format_float_positional(np.float32(x), unique=True, trim="-")


def write_mut(path: str, sites: Sites, c: int):
    """Relate .mut text for chromosome index c (mutations.cpp:56-257; writer 298-328)."""
    lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
    with open(path, "w") as f:
        f.write("snp;pos_of_snp;dist;rs-id;tree_index;branch_indices;is_not_mapping;is_flipped;age_begin;age_end;ancestral_allele/alternative_allele;upstream_allele;downstream_allele;\n")
        for i in range(lo, hi):
            k = i - lo
            br = "17" if sites.n_branch[i] == 1 else "17 23"
            if sites.odd[i] == 1:
                mt = chr(sites.anc[i]) + "T/" + chr(sites.der[i])
            elif sites.odd[i] == 2:
                mt = "NA"
            else:
                mt = chr(sites.anc[i]) + "/" + chr(sites.der[i])
            dist = int(sites.pos[i + 1] - sites.pos[i]) if i + 1 < hi else 1
            f.write(f"{k};{int(sites.pos[i])};{dist};rs{k};{k // 3};{br};{int(sites.n_branch[i] > 1)};"
                    f"{int(sites.flipped[i])};{_fmt_f32(sites.age_begin[i])};{_fmt_f32(sites.age_end[i])};{mt};A;C;\n")


_synthio = None


def mut_text_fast(sites: Sites, c: int) -> np.ndarray:
    """The bytes write_mut() writes for chromosome index c, as a uint8 array, produced by the C writer
    (colate_b200/csrc/synth_io.c -> libsynthio.so): 10 M rows in a few seconds instead of minutes."""
    global _synthio
    import ctypes as C
    if _synthio is None:
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libsynthio.so")
        L = C.CDLL(path)
        L.synth_mut_text.restype = C.c_longlong
        L.synth_mut_text.argtypes = [C.c_longlong, C.c_longlong] + [C.c_void_p] * 9 + [C.c_longlong]
        _synthio = L
    lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
    cap = 256 + 200 * (hi - lo + 1)
    out = np.empty(cap, dtype=np.uint8)
    a = [np.ascontiguousarray(x, dtype=dt) for x, dt in ((sites.pos, np.int32), (sites.age_begin, np.float32), (sites.age_end, np.float32),
                                                          (sites.flipped, np.uint8), (sites.n_branch, np.int32), (sites.anc, np.uint8),
                                                          (sites.der, np.uint8), (sites.odd, np.uint8))]
    n = _synthio.synth_mut_text(lo, hi, *[x.ctypes.data for x in a], out.ctypes.data, cap)
    if n < 0:
        raise RuntimeError("synth_mut_text: buffer too small")
    return out[:n]


def mut_texts_fast(sites: Sites, threads: int | None = None):
    """mut_text_fast for every chromosome, on a thread pool (the C writer runs without the GIL)."""
    from concurrent.futures import ThreadPoolExecutor
    n = len(sites.chr_names)
    with ThreadPoolExecutor(max_workers=threads or min(n, os.cpu_count() or 1)) as ex:
        return list(ex.map(lambda c: mut_text_fast(sites, c), range(n)))


def colate_in_image(g: Genome, chr_names) -> np.ndarray:
    """The bytes write_colate_in_fast() writes, as a uint8 array."""
    parts = []
    for c, nm in enumerate(chr_names):
        sel = np.nonzero(g.chrom == c)[0]
        if sel.shape[0] == 0:
            continue
        nb = nm.encode()
        rec = np.dtype([("l", "<i4"), ("nm", f"S{len(nb)}"), ("bp", "<i4"), ("a", "u1"), ("d", "u1"), ("aaf", "<i4"), ("daf", "<i4")])
        arr = np.empty(sel.shape[0], dtype=rec)
        arr["l"], arr["nm"], arr["bp"] = len(nb), nb, g.bp[sel]
        arr["a"], arr["d"], arr["aaf"], arr["daf"] = g.anc[sel], g.der[sel], g.aaf[sel], g.daf[sel]
        parts.append(np.frombuffer(arr.tobytes(), dtype=np.uint8))
    return np.concatenate(parts) if parts else np.zeros(0, np.uint8)


def write_colate_in(path: str, g: Genome, chr_names, extra_names=None):
    """.colate.in record stream (coal.cpp:2505-2514): {i32 lchrom, chrom, i32 bp, anc, der, i32 AAF, i32 DAF}."""
    names = list(chr_names) + list(extra_names or [])
    enc = [nm.encode() for nm in names]
    out = bytearray()
    i32 = np.dtype("<i4")
    for k in range(g.n):
        nm = enc[int(g.chrom[k])]
        out += np.array([len(nm)], dtype=i32).tobytes() + nm
        out += np.array([g.bp[k]], dtype=i32).tobytes()
        out += bytes([int(g.anc[k]), int(g.der[k])])
        out += np.array([g.aaf[k], g.daf[k]], dtype=i32).tobytes()
    with open(path, "wb") as f:
        f.write(bytes(out))


def write_colate_in_fast(path: str, g: Genome, chr_names):
    """Vectorised writer for large genomes (all names must have the same byte length per chromosome)."""
    with open(path, "wb") as f:
        for c, nm in enumerate(chr_names):
            sel = np.nonzero(g.chrom == c)[0]
            if sel.shape[0] == 0:
                continue
            nb = nm.encode()
            rec = np.dtype([("l", "<i4"), ("nm", f"S{len(nb)}"), ("bp", "<i4"), ("a", "u1"), ("d", "u1"),
                            ("aaf", "<i4"), ("daf", "<i4")])
            arr = np.empty(sel.shape[0], dtype=rec)
            arr["l"], arr["nm"], arr["bp"] = len(nb), nb, g.bp[sel]
            arr["a"], arr["d"], arr["aaf"], arr["daf"] = g.anc[sel], g.der[sel], g.aaf[sel], g.daf[sel]
            f.write(arr.tobytes())


def write_mask(path: str, seq: bytes, width: int = 60000):
    with open(path, "wb") as f:
        f.write(b">mask\n")
        for i in range(0, len(seq), width):
            f.write(seq[i:i + width] + b"\n")


def write_dataset(dirname: str, sites: Sites, genomes: dict, masks: dict | None = None, prefix="syn"):
    """Writes <prefix>_chr<name>.mut, chr.txt, <gname>.colate.in and <mname>_chr<name>.fa."""
    os.makedirs(dirname, exist_ok=True)
    with open(os.path.join(dirname, "chr.txt"), "w") as f:
        for nm in sites.chr_names:
            f.write(nm + "\n")
    for c, nm in enumerate(sites.chr_names):
        write_mut(os.path.join(dirname, f"{prefix}_chr{nm}.mut"), sites, c)
    for gname, g in genomes.items():
        write_colate_in(os.path.join(dirname, f"{gname}.colate.in"), g, sites.chr_names)
    for mname, per_chr in (masks or {}).items():
        for c, nm in enumerate(sites.chr_names):
            write_mask(os.path.join(dirname, f"{mname}_chr{nm}.fa"), per_chr[c])
    return dirname


# ---- BAM files (SAM/BAM format specification 4.1-4.2): BGZF blocks around the binary records, written with zlib ----------------
NT16 = b"=ACMGRSVTWYHKDBN"
_NT16_CODE = np.full(256, 15, dtype=np.uint8)
_NT16_CODE[np.frombuffer(NT16, np.uint8)] = np.arange(16, dtype=np.uint8)
CIGAR_OPS = "MIDNSHP=X"


def bam_record(tid, pos0, mapq, flag, seq, qual, name=b"r", cigar=None, aux=b"", next_tid=-1, next_pos=-1, tlen=0) -> bytes:
    """One BAM record (block_size included).  seq: letters of seq_nt16_str (others become N); qual: phred bytes (len(seq) of them);
    cigar: [(length, op letter)] (default: one <len>M op, none for an empty sequence); aux: raw aux bytes."""
    import struct
    seq = bytes(seq)
    l = len(seq)
    if cigar is None:
        cigar = [(l, "M")] if l else []
    nm = bytes(name) + b"\0"
    codes = _NT16_CODE[np.frombuffer(seq, np.uint8)] if l else np.zeros(0, np.uint8)
    if l & 1:
        codes = np.concatenate([codes, np.zeros(1, np.uint8)])
    packed = (codes[0::2] << 4 | codes[1::2]).astype(np.uint8).tobytes()
    q = bytes(bytearray(qual))
    assert len(q) == l and len(nm) <= 255
    cig = b"".join(struct.pack("<I", n << 4 | CIGAR_OPS.index(op)) for n, op in cigar)
    core = struct.pack("<iiBBHHHiiii", tid, pos0, len(nm), mapq, 4680, len(cigar), flag, l, next_tid, next_pos, tlen)
    body = core + nm + cig + packed + q + bytes(aux)
    return struct.pack("<i", len(body)) + body


def bam_header(contig_names, contig_lens=None, text=b"") -> bytes:
    import struct
    lens = contig_lens if contig_lens is not None else [1 << 29] * len(contig_names)
    out = [b"BAM\1", struct.pack("<i", len(text)), bytes(text), struct.pack("<i", len(contig_names))]
    for nm, L in zip(contig_names, lens):
        b = nm.encode() + b"\0"
        out += [struct.pack("<i", len(b)), b, struct.pack("<i", int(L))]
    return b"".join(out)


def bgzf_block(data: bytes, level=6) -> bytes:
    """One BGZF block: a gzip member with the 'BC' extra subfield holding the block size - 1."""
    import struct
    import zlib
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    body = c.compress(data) + c.flush()
    hdr = struct.pack("<BBBBIBBH", 31, 139, 8, 4, 0, 0, 255, 6) + b"BC" + struct.pack("<HH", 2, 18 + len(body) + 8 - 1)
    return hdr + body + struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data))


BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_compress(data: bytes, block_size=65280, empty_blocks=(), eof=True, level=6, threads=1) -> bytes:
    """`data` cut into BGZF blocks of block_size inflated bytes (1..65536; records straddle blocks wherever the cut falls),
    an empty block inserted before block k for every k in empty_blocks, the EOF block at the end if eof."""
    assert 1 <= block_size <= 65536
    pieces = [data[i:i + block_size] for i in range(0, len(data), block_size)]
    if threads > 1:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(threads) as ex:
            blocks = list(ex.map(lambda p: bgzf_block(p, level), pieces, chunksize=256))
    else:
        blocks = [bgzf_block(p, level) for p in pieces]
    empty = bgzf_block(b"", level)
    out = []
    for k, b in enumerate(blocks):
        out += [empty] * sum(1 for e in empty_blocks if e == k)
        out.append(b)
    out += [empty] * sum(1 for e in empty_blocks if e >= len(blocks))
    if eof:
        out.append(BGZF_EOF)
    return b"".join(out)


def write_bam(path, contig_names, reads, contig_lens=None, text=b"", block_size=65280, empty_blocks=(), eof=True, level=6, threads=1):
    """A BAM file: header (contig_names, optional lengths and SAM text) and `reads`, each either a record from bam_record() or the
    tuple of its arguments (tid, pos0, mapq, flag, seq, qual[, name, cigar, aux]); records are written in the order given."""
    recs = [r if isinstance(r, (bytes, bytearray)) else bam_record(*r) for r in reads]
    data = bam_header(contig_names, contig_lens, text) + b"".join(recs)
    with open(path, "wb") as f:
        f.write(bgzf_compress(data, block_size, empty_blocks, eof, level, threads))


def bam_records_np(tid, pos0, mapq, lens, seq, qual, flag=None):
    """Many records at once (benchmarks): arrays tid/pos0/mapq/lens [n], seq letters and qual phred bytes concatenated in read order;
    name "r", one <len>M CIGAR op, no aux.  Returns the records as one uint8 array."""
    n = len(pos0)
    lens = np.asarray(lens, np.int64)
    nb = (lens + 1) // 2
    size = 36 + 2 + 4 + nb + lens                    # block_size field + core + name + cigar + packed + qual
    off = np.zeros(n + 1, np.int64)
    np.cumsum(size, out=off[1:])
    buf = np.zeros(int(off[-1]), np.uint8)
    o = off[:-1]

    def put(at, v, nbytes):
        v = np.asarray(v, np.int64) & ((1 << (8 * nbytes)) - 1)
        for b in range(nbytes):
            buf[at + b] = (v >> (8 * b)) & 0xFF
    put(o, size - 4, 4)
    put(o + 4, tid, 4)
    put(o + 8, pos0, 4)
    buf[o + 12] = 2
    buf[o + 13] = np.asarray(mapq, np.uint8)
    put(o + 14, 4680, 2)
    put(o + 16, 1, 2)
    put(o + 18, 0 if flag is None else flag, 2)
    put(o + 20, lens, 4)
    put(o + 24, -1, 4)
    put(o + 28, -1, 4)
    buf[o + 36] = ord("r")
    put(o + 38, lens << 4, 4)
    # packed sequence: read r's byte j = code(2j) << 4 | code(2j + 1)
    codes = _NT16_CODE[np.frombuffer(bytes(seq), np.uint8) if not isinstance(seq, np.ndarray) else seq]
    sstart = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=sstart[1:])
    rid = np.repeat(np.arange(n), nb)
    j = np.arange(int(nb.sum())) - np.repeat(np.cumsum(nb) - nb, nb)
    hi_i = sstart[rid] + 2 * j
    lo_i = hi_i + 1
    lo_ok = 2 * j + 1 < lens[rid]
    packed = (codes[hi_i] << 4) | np.where(lo_ok, codes[np.minimum(lo_i, len(codes) - 1)], 0)
    buf[np.repeat(o + 42, nb) + j] = packed.astype(np.uint8)
    qi = np.arange(int(lens.sum())) - np.repeat(sstart[:-1], lens)
    buf[np.repeat(o + 42 + nb, lens) + qi] = np.asarray(qual, np.uint8)
    return buf


# ---- BCF files (VCF specification v4.3, 6.3 "BCF2"): BGZF blocks around the header text and the binary records ------------------
BCF_INT8, BCF_INT16, BCF_INT32, BCF_FLOAT, BCF_CHAR = 1, 2, 3, 5, 7
_BCF_FMT = {BCF_INT8: "b", BCF_INT16: "h", BCF_INT32: "i", BCF_FLOAT: "f"}
GT_MISSING = {BCF_INT8: -128, BCF_INT16: -32768, BCF_INT32: -2 ** 31}
GT_VECTOR_END = {BCF_INT8: -127, BCF_INT16: -32767, BCF_INT32: -2 ** 31 + 1}


def _bcf_int_type(values):
    lo, hi = (min(values), max(values)) if len(values) else (0, 0)
    return BCF_INT8 if -120 <= lo and hi <= 127 else BCF_INT16 if -32760 <= lo and hi <= 32767 else BCF_INT32


def bcf_descr(t, n) -> bytes:
    """Typed-value descriptor: size << 4 | type, sizes from 15 up as the overflow form (15 << 4 | type, then a typed integer)."""
    return bytes([n << 4 | t]) if n < 15 else bytes([0xF0 | t]) + bcf_typed_ints([n])


def bcf_typed_ints(values, t=None) -> bytes:
    import struct
    t = t or _bcf_int_type(values)
    return bcf_descr(t, len(values)) + struct.pack("<%d%s" % (len(values), _BCF_FMT[t]), *values)


def bcf_typed_floats(values) -> bytes:
    import struct
    return bcf_descr(BCF_FLOAT, len(values)) + struct.pack("<%df" % len(values), *values)


def bcf_typed_str(s) -> bytes:
    return bcf_descr(BCF_CHAR, len(s)) + bytes(s)


BCF_FLAG = b"\x00"      # an INFO flag: type 0, size 0


def bcf_header(n_sample, ids=(("FORMAT", "GT"),), idx=None, contigs=("1",), minor=2, extra=b"", contig_idx=None) -> bytes:
    """Magic, l_text and header text.  ids: (kind, ID) pairs (FILTER / INFO / FORMAT) in order of appearance; PASS is implicit.
    idx: None (no IDX=, as a hand-written header) or {ID: number} (IDX= on every line, as bcftools writes; PASS gets 0).
    contig_idx: None or {contig: number}, the IDX= of the ##contig lines (which then need not follow their order)."""
    import struct
    lines = [b"##fileformat=VCFv4.3"]
    ix = (lambda i: b",IDX=%d" % idx[i]) if idx is not None else (lambda i: b"")
    lines.append(b'##FILTER=<ID=PASS,Description="All filters passed"' + (b",IDX=0" if idx is not None else b"") + b">")
    for kind, i in ids:
        typ = b"String" if i == "GT" else b"Integer"
        lines.append(b'##%s=<ID=%s,Number=1,Type=%s,Description="a \\"quoted\\", IDX=99 text"%s>' % (kind.encode(), i.encode(), typ, ix(i)))
    for k, c in enumerate(contigs):
        k = contig_idx[c] if contig_idx is not None else k
        lines.append(b"##contig=<ID=%s,length=1000000000%s>" % (c.encode(), b",IDX=%d" % k if idx is not None or contig_idx is not None else b""))
    lines.append(bytes(extra) if extra else b"##source=colate_b200.synth")
    cols = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO"
    if n_sample:
        cols += b"\tFORMAT" + b"".join(b"\ts%d" % s for s in range(n_sample))
    text = b"\n".join(lines + [cols]) + b"\n\0"
    return b"BCF\2" + bytes([minor]) + struct.pack("<I", len(text)) + text


def bcf_gt_values(gt, phased=False, t=BCF_INT8):
    """Allele indices [n_sample][ploidy] (-1: missing '.', None: vector end) -> the typed GT values ((a + 1) << 1 | phased)."""
    out = []
    for s in gt:
        for j, a in enumerate(s):
            if a is None:
                out.append(GT_VECTOR_END[t])
            else:
                ph = int(phased[j] if isinstance(phased, (list, tuple)) else phased) if j > 0 else 0
                out.append((int(a) + 1) << 1 | ph)
    return out


def bcf_record(chrom, pos0, alleles, gt, gt_key, phased=False, gt_type=BCF_INT8, rid=b".", qual=None, filters=(), info=(),
               fmt_before=(), fmt_after=(), gt_raw=None, n_sample=None) -> bytes:
    """One BCF record (l_shared and l_indiv included).  gt: allele indices [n_sample][ploidy] (bcf_gt_values); gt_raw: the typed GT
    values themselves instead (per sample a list); gt_key=None writes no GT.  info: (key, typed value bytes) pairs; filters: dictionary
    indices; fmt_before / fmt_after: FORMAT fields (key, type, values per sample) around GT."""
    import struct
    ns = len(gt) if n_sample is None else n_sample
    shared = [struct.pack("<ii", chrom, pos0), struct.pack("<i", max(1, len(alleles[0]) if alleles else 1)),
              struct.pack("<I", 0x7F800001) if qual is None else struct.pack("<f", qual)]
    fmts = list(fmt_before)
    if gt_key is not None:
        vals = gt_raw if gt_raw is not None else [bcf_gt_values([s], phased, gt_type) for s in gt]
        fmts.append((gt_key, gt_type, vals))
    fmts += list(fmt_after)
    shared.append(struct.pack("<II", len(alleles) << 16 | len(info), len(fmts) << 24 | ns))
    shared.append(bcf_typed_str(rid))
    shared += [bcf_typed_str(a) for a in alleles]
    shared.append(bcf_typed_ints(list(filters), BCF_INT8) if filters else bytes([BCF_INT8]))
    for key, val in info:
        shared += [bcf_typed_ints([key]), bytes(val)]
    indiv = []
    for key, t, vals in fmts:
        size = max(len(v) for v in vals) if vals else 0
        indiv += [bcf_typed_ints([key]), bcf_descr(t, size)]
        for v in vals:
            v = list(v) + [0] * (size - len(v)) if t != BCF_CHAR else bytes(v).ljust(size, b"\0")
            indiv.append(bytes(v) if t == BCF_CHAR else struct.pack("<%d%s" % (size, _BCF_FMT[t]), *v))
    s, i = b"".join(shared), b"".join(indiv)
    return struct.pack("<II", len(s), len(i)) + s + i


def write_bcf(path, header, records, block_size=65280, empty_blocks=(), eof=True, level=6, threads=1):
    """A BCF file: `header` (bcf_header) and the records (bytes or a uint8 array) in the order given, BGZF-compressed."""
    data = bytes(header) + (records.tobytes() if isinstance(records, np.ndarray) else b"".join(records))
    with open(path, "wb") as f:
        f.write(bgzf_compress(data, block_size, empty_blocks, eof, level, threads))


def bcf_records_np(pos0, a0, a1, gt_values, gt_key, ploidy=2, chrom=0) -> np.ndarray:
    """Many records at once (benchmarks): pos0 [n], a0 / a1 [n] one-letter alleles (uint8), gt_values [n][n_hap] the typed int8 GT
    values; ID '.', FILTER PASS, no INFO, GT the only FORMAT field.  Returns the records as one uint8 array."""
    gt_values = np.asarray(gt_values, np.int8)
    n, n_hap = gt_values.shape
    assert n_hap % ploidy == 0 and ploidy < 15 and gt_key < 120
    ns = n_hap // ploidy
    l_shared, l_indiv = 24 + 2 + 2 + 2 + 2, 2 + 1 + n_hap
    size = 8 + l_shared + l_indiv
    buf = np.zeros((n, size), np.uint8)
    head = np.array([l_shared, l_indiv, chrom, 0, 1, 0x7F800001, 2 << 16, 1 << 24 | ns], np.uint32).view(np.uint8)
    buf[:, :32] = head
    buf[:, 12:16] = np.asarray(pos0, np.int32).view(np.uint8).reshape(n, 4)
    buf[:, 32:34] = [0x17, ord(".")]
    buf[:, 34] = 0x17
    buf[:, 35] = a0
    buf[:, 36] = 0x17
    buf[:, 37] = a1
    buf[:, 38:40] = [0x11, 0x00]                     # FILTER: PASS
    buf[:, 40:43] = [0x11, gt_key, ploidy << 4 | BCF_INT8]
    buf[:, 43:] = gt_values.view(np.uint8)
    return buf.reshape(-1)


# ---- bgzipped text VCF (VCF specification v4.3, section 1): what htslib's bcf_open reads in place of BCF ------------------------
def vcf_header(n_sample, ids=(("FORMAT", "GT"),), contigs=("1",), extra=(), fileformat=b"##fileformat=VCFv4.3") -> bytes:
    """The ## lines and the #CHROM line.  ids: (kind, ID) pairs as bcf_header; contigs: ##contig lines; extra: more ## lines."""
    lines = [fileformat, b'##FILTER=<ID=PASS,Description="All filters passed">']
    for kind, i in ids:
        typ = b"String" if i == "GT" else b"Integer"
        lines.append(b'##%s=<ID=%s,Number=1,Type=%s,Description="a \\"quoted\\" text">' % (kind.encode(), i.encode(), typ))
    lines += [b"##contig=<ID=%s,length=1000000000>" % c.encode() for c in contigs]
    lines += [bytes(x) for x in extra] or [b"##source=colate_b200.synth"]
    cols = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO"
    if n_sample:
        cols += b"\tFORMAT" + b"".join(b"\ts%d" % s for s in range(n_sample))
    return b"\n".join(lines + [cols]) + b"\n"


def vcf_gt_text(alleles, phased=False) -> bytes:
    """One sample's GT: allele indices (-1 or None: '.') joined by '|' (phased) or '/'; phased may be a list per separator."""
    out = b""
    for j, a in enumerate(alleles):
        if j:
            ph = phased[j - 1] if isinstance(phased, (list, tuple)) else phased
            out += b"|" if ph else b"/"
        out += b"." if a is None or a < 0 else b"%d" % a
    return out


def vcf_line(chrom, pos0, alleles, gt, phased=False, rid=b".", qual=b".", filt=b"PASS", info=b".", fmt_before=(), fmt_after=(),
             gt_text=None, keep=None, fmt=None, newline=True) -> bytes:
    """One record line.  alleles: REF then the ALT alleles (ALT '.' when there are none); gt: allele indices [n_sample][ploidy]
    (-1: '.'), or gt_text: the GT strings themselves; fmt_before / fmt_after: (key, [value per sample]) FORMAT fields around GT;
    keep: per sample, the number of leading subfields written (trailing ones dropped); fmt: the FORMAT column itself (b"" drops
    FORMAT and the samples)."""
    keys = [k for k, _ in fmt_before] + ["GT"] + [k for k, _ in fmt_after]
    fmt = b":".join(k.encode() for k in keys) if fmt is None else fmt
    gts = gt_text if gt_text is not None else [vcf_gt_text(s, phased) for s in gt]
    cols = [chrom.encode() if isinstance(chrom, str) else bytes(chrom), b"%d" % (pos0 + 1), bytes(rid), bytes(alleles[0]),
            b",".join(bytes(a) for a in alleles[1:]) or b".", bytes(qual), bytes(filt), bytes(info)]
    if fmt != b"":
        cols.append(fmt)
        for s, g in enumerate(gts):
            sub = [bytes(v[s]) for _, v in fmt_before] + [bytes(g)] + [bytes(v[s]) for _, v in fmt_after]
            cols.append(b":".join(sub[:keep[s]] if keep is not None else sub))
    return b"\t".join(cols) + (b"\n" if newline else b"")


def write_vcf(path, header, lines, block_size=65280, empty_blocks=(), eof=True, level=6, threads=1):
    """A bgzipped VCF: `header` (vcf_header) and the lines (bytes or a uint8 array) in the order given, in BGZF blocks."""
    data = bytes(header) + (lines.tobytes() if isinstance(lines, np.ndarray) else b"".join(lines))
    with open(path, "wb") as f:
        f.write(bgzf_compress(data, block_size, empty_blocks, eof, level, threads))


def vcf_lines_np(pos0, a0, a1, alleles, phased=None, chrom=b"1") -> np.ndarray:
    """Many diploid lines at once (benchmarks): pos0 [n], a0 / a1 [n] one-letter alleles (uint8), alleles [n][2 n_sample] single-digit
    allele indices, phased [n][n_sample] (None: unphased); ID '.', QUAL '.', FILTER PASS, INFO '.', FORMAT GT.  The lines as one
    uint8 array."""
    alleles = np.asarray(alleles, np.uint8)
    n, n_hap = alleles.shape
    ns = n_hap // 2
    if n == 0:
        return np.zeros(0, np.uint8)
    pos_txt = np.char.mod(b"%d", np.asarray(pos0, np.int64) + 1).astype(bytes)
    W = pos_txt.dtype.itemsize
    head = np.frombuffer(bytes(chrom) + b"\t", np.uint8)
    rest = np.frombuffer(b"\t.\tPASS\t.\tGT", np.uint8)
    # one row per line with POS left-aligned in W columns; the padding is dropped at the end
    cols = head.size + W + 3 + 3 + rest.size + 4 * ns + 1
    buf = np.empty((n, cols), np.uint8)
    buf[:, :head.size] = head
    buf[:, head.size:head.size + W] = pos_txt.view(np.uint8).reshape(n, W)
    q = head.size + W
    buf[:, q:q + 3] = np.frombuffer(b"\t.\t", np.uint8)
    buf[:, q + 3] = a0
    buf[:, q + 4] = 9
    buf[:, q + 5] = a1
    buf[:, q + 6:q + 6 + rest.size] = rest
    smp = buf[:, q + 6 + rest.size:cols - 1].reshape(n, ns, 4)
    smp[:, :, 0] = 9
    smp[:, :, 1] = alleles[:, 0::2] + 48
    smp[:, :, 2] = ord("/") if phased is None else np.where(np.asarray(phased, bool), ord("|"), ord("/"))
    smp[:, :, 3] = alleles[:, 1::2] + 48
    buf[:, -1] = 10
    keep = np.ones((n, cols), bool)
    keep[:, head.size:head.size + W] = buf[:, head.size:head.size + W] != 0
    return buf[keep]
