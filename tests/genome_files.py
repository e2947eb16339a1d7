"""Whole-genome BCF / VCF files (one file, many contigs) and their split twins, written from the same record lists, and a
gzip + struct / text parse of such a file.  A record is (pos0, alleles, allele index per haplotype), as test_gpu_bcf.py writes them."""
import gzip
import re
import struct

import numpy as np

from colate_b200 import synth
from bcf_helpers import IDS, keys_of, py_decode

VCF_IDS = [("INFO", "DP"), ("FORMAT", "GQ"), ("FORMAT", "GT"), ("FORMAT", "AD")]


def _bcf_recs(chrom, n_sample, ploidy, recs):
    gt_key = keys_of(None)["GT"]
    return [synth.bcf_record(chrom, p0, list(al), np.asarray(gt).reshape(n_sample, ploidy).tolist(), gt_key, info=[(1, synth.bcf_typed_ints([7]))])
            for p0, al, gt in recs]


def _vcf_lines(chrom, n_sample, ploidy, recs):
    return [synth.vcf_line(chrom, p0, list(al), np.asarray(gt).reshape(n_sample, ploidy).tolist(), info=b"DP=7") for p0, al, gt in recs]


def write_genome(path, fmt, n_sample, contigs, header_contigs=None, contig_idx=None, block_size=65280):
    """One file: contigs = [(name, recs, ploidy)] in file order.  BCF: CHROM indexes the header's contig dictionary, whose ##contig
    lines are header_contigs (default: the file's contigs, reversed) numbered in order, or by contig_idx {name: IDX}.  VCF: CHROM is
    the name."""
    if fmt == "bcf":
        hc = list(header_contigs) if header_contigs is not None else list(dict.fromkeys(nm for nm, _, _ in contigs))[::-1]
        index = dict(contig_idx) if contig_idx is not None else {nm: k for k, nm in enumerate(hc)}
        out = []
        for nm, recs, pl in contigs:
            out += _bcf_recs(index[nm], n_sample, pl, recs)
        synth.write_bcf(str(path), synth.bcf_header(n_sample, IDS, contigs=hc, contig_idx=contig_idx), out, block_size=block_size)
    else:
        hc = list(header_contigs) if header_contigs is not None else list(dict.fromkeys(nm for nm, _, _ in contigs))
        out = []
        for nm, recs, pl in contigs:
            out += _vcf_lines(nm, n_sample, pl, recs)
        synth.write_vcf(str(path), synth.vcf_header(n_sample, VCF_IDS, contigs=hc), out, block_size=block_size)


def write_split(prefix, fmt, n_sample, chr_names, recs_per_chr, ploidy_per_chr=None, block_size=65280):
    """The per-chromosome twins: <prefix>_chr<c>.bcf, one contig each."""
    for c, nm in enumerate(chr_names):
        pl = ploidy_per_chr[c] if ploidy_per_chr else 2
        write_genome(f"{prefix}_chr{nm}.bcf", fmt, n_sample, [(nm, recs_per_chr[c], pl)], block_size=block_size)


def decoys(rng, n_sample, ploidy, n=30):
    """Records of an unlisted contig: unsorted positions, which only a listed contig would be refused for."""
    return [(int(p), [b"A", b"G"], [int(x) for x in rng.integers(0, 2, n_sample * ploidy)]) for p in rng.integers(0, 10 ** 6, n)]


def parse(path):
    """gzip + struct / text parse of a whole-genome file: ({contig name: [pos0, ...]} in file order, n_sample)."""
    data = gzip.decompress(open(path, "rb").read())
    out = {}
    if data[:4] == b"BCF\2":
        l_text = struct.unpack_from("<I", data, 5)[0]
        text = data[9:9 + l_text].split(b"\0")[0].decode()
        names, nxt = {}, 0
        for m in re.finditer(r"^##contig=<ID=([^,>]+)[^\n]*?(?:,IDX=(\d+))?>$", text, re.M):
            k = int(m.group(2)) if m.group(2) else nxt
            names[k] = m.group(1)
            nxt = max(nxt, k + 1)
        ns, _, recs = py_decode(data)
        for r in recs:
            out.setdefault(names[r[0]], []).append(r[1])
        return out, ns
    ns = 0
    for line in data.split(b"\n"):
        if line.startswith(b"#CHROM"):
            ns = line.count(b"\t") - 8
        elif line and not line.startswith(b"#"):
            f = line.split(b"\t", 2)
            out.setdefault(f[0].decode(), []).append(int(f[1]) - 1)
    return out, ns


def genome_layout(rng, chr_names, recs_per_chr, n_sample, ploidy_per_chr=None, prefix_chr=False, order=None):
    """The contig list of a whole-genome file: an unlisted decoy before, between and after the listed contigs, which come in
    `order` (indices into chr_names; default reversed) and are named <c> or chr<c>."""
    order = list(range(len(chr_names)))[::-1] if order is None else list(order)
    pl = ploidy_per_chr or [2] * len(chr_names)
    name = (lambda c: "chr" + chr_names[c]) if prefix_chr else (lambda c: chr_names[c])
    contigs = [("decoy_a", decoys(rng, n_sample, 2), 2)]
    for i, c in enumerate(order):
        contigs.append((name(c), recs_per_chr[c], pl[c]))
        if i == 0:
            contigs.append(("chrUn_b", decoys(rng, n_sample, 2), 2))
    contigs.append(("chrM", decoys(rng, n_sample, 1), 1))
    return contigs
