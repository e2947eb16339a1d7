"""Random genotype-matrix datasets for make_tmp (DESIGN.md section 6l) and the pin they are checked against: each individual's
(chromosome, position, allele) table of homozygous calls, written by colate_maketmp_table (host only)."""
import os

import numpy as np

from colate_b200 import _lib, synth

NAMES = ["1", "X", "5"]                       # --chr entries
CONTIGS = ["chr1", "23", "4", "5"]            # .snp / .bim contigs in file order: chr-prefixed, 23 for X, an unlisted contig
ENTRY_OF = {"chr1": 0, "23": 1, "4": None, "5": 2}


def _names(xs):
    return (_lib.C.c_char_p * len(xs))(*[str(x).encode() for x in xs])


def make_case(d, seed, n_ind=200, rows=(1500, 900, 1200)):
    """.mut files (repeated positions, rows before the first and after the last SNP), genome presence files, masks, and a matrix:
    SNPs at row positions and elsewhere, duplicate SNP positions, alleles equal to neither row letter and multi-letter alleles,
    pseudo-haploid and diploid individuals with missing calls, individual 7 without a homozygous call on entry X.
    Returns a dict: snps, ids, calls, masks (prefixes)."""
    rng = np.random.default_rng(seed)
    lens = [int(4e5 + 1e5 * k) for k in range(len(NAMES))]
    sites = synth.make_sites(seed, list(rows), lens, chr_names=list(NAMES), weird=0.1)
    for c in range(len(NAMES)):                                   # repeated .mut positions (rows stay ascending)
        lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
        for k in rng.choice(np.arange(lo + 1, hi), size=(hi - lo) // 40, replace=False):
            sites.pos[k] = sites.pos[k - 1]
    synth.write_dataset(d, sites, {})
    for nm in NAMES:
        open(os.path.join(d, f"g_chr{nm}.fa"), "w").write(">g\nACGT\n")
    snps = []
    for contig in CONTIGS:
        c = ENTRY_OF[contig]
        if c is None:
            p = np.sort(rng.integers(1, 10 ** 6, 50))
            snps += [(f"u{len(snps)}", contig, int(x), "A", "G") for x in p]
            continue
        lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
        inner = np.arange(lo + 40, hi - 40)                       # rows before the first SNP and after the last one
        at_rows = rng.choice(inner, size=len(inner) // 2, replace=False)
        p = np.concatenate([sites.pos[at_rows], rng.integers(sites.pos[lo + 40], sites.pos[hi - 41], 60)])
        p = np.sort(p)
        row_at = {int(sites.pos[k]): k for k in range(lo, hi)}
        for x in p:
            k = row_at.get(int(x))
            a, dd = (chr(sites.anc[k]), chr(sites.der[k])) if k is not None else ("C", "T")
            u = rng.random()
            if u < 0.06:
                al = (a, "N" if dd != "N" else "C")                 # the second allele is neither row letter
            elif u < 0.09:
                al = (a + "T", dd)                                  # a multi-letter allele
            elif u < 0.55:
                al = (a, dd)
            else:
                al = (dd, a)
            snps.append((f"s{len(snps)}", contig, int(x), al[0], al[1]))
            if rng.random() < 0.05:                                 # a duplicate SNP at the same position
                snps.append((f"s{len(snps)}", contig, int(x), al[1], al[0]))
    n_snp = len(snps)
    diploid = rng.random(n_ind) < 0.3
    calls = rng.integers(0, 2, (n_snp, n_ind)).astype(np.uint8)
    het = (rng.random((n_snp, n_ind)) < 0.3) & diploid[None, :]
    calls[het] = 2
    calls[rng.random((n_snp, n_ind)) < rng.uniform(0.1, 0.6, n_ind)[None, :]] = 3
    for s in range(1, n_snp):                                      # duplicates: the first one missing, the second called
        if snps[s][2] == snps[s - 1][2] and snps[s][1] == snps[s - 1][1] and rng.random() < 0.6:
            calls[s - 1, :n_ind // 2] = 3
    on_x = np.array([ENTRY_OF[x[1]] == 1 for x in snps])
    calls[on_x, 7] = np.where(rng.random(on_x.sum()) < 0.5, 3, 2) if n_ind > 7 else calls[on_x, 7]
    masks = []
    for m in range(2):
        for c, nm in enumerate(NAMES):
            L = lens[c] // 2 if (m + c) % 2 == 0 else lens[c]      # masks shorter than the positions
            synth.write_mask(os.path.join(d, f"m{m}_chr{nm}.fa"), synth.make_mask(seed * 7 + 10 * m + c, L, 0.3, run_lo=100, run_hi=5000))
        masks.append(os.path.join(d, f"m{m}"))
    ids = [f"I{seed}_{k}" for k in range(n_ind)]
    return {"snps": snps, "ids": ids, "calls": calls, "masks": masks, "sites": sites}


def table_of(case, k):
    """The table individual k's homozygous calls spell out: per --chr entry in order, its SNPs in file order."""
    lines = []
    for c, nm in enumerate(NAMES):
        for s, (_, contig, p, a1, a2) in enumerate(case["snps"]):
            if ENTRY_OF[contig] == c and case["calls"][s, k] < 2:
                lines.append(f"{nm} {p} {a1 if case['calls'][s, k] == 0 else a2}\n")
    return "".join(lines)


def pinned(d, case, k, out, mask=None):
    """colate_maketmp_table on individual k's table: the bytes its .colate.in must have."""
    tab = str(out) + ".table"
    open(tab, "w").write(table_of(case, k))
    muts = [os.path.join(d, f"syn_chr{nm}.mut") for nm in NAMES]
    masks = _names([f"{mask}_chr{nm}.fa" for nm in NAMES]) if mask else None
    _lib.check(_lib.lib().colate_maketmp_table(len(NAMES), _names(NAMES), _names(muts), tab.encode(), masks, 1, str(out).encode()))
    return open(out, "rb").read()


def write_all(d, case, tag="x"):
    """The case in all three layouts: <d>/<tag>_bed (PLINK), <tag>_pk (packed EIGENSTRAT), <tag>_tx (text EIGENSTRAT)."""
    synth.write_plink(os.path.join(d, f"{tag}_bed"), case["snps"], case["ids"], case["calls"])
    synth.write_eigenstrat(os.path.join(d, f"{tag}_pk"), case["snps"], case["ids"], case["calls"], packed=True)
    synth.write_eigenstrat(os.path.join(d, f"{tag}_tx"), case["snps"], case["ids"], case["calls"], packed=False)
    return {"plink": os.path.join(d, f"{tag}_bed"), "packed": os.path.join(d, f"{tag}_pk"), "text": os.path.join(d, f"{tag}_tx")}
