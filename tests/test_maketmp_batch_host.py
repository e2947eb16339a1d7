"""No GPU: `Colate --mode make_tmp --targets <file>` refuses malformed targets files and conflicting flags before it touches a device,
naming the offending line; the make_tmp row word of the host reader on hand-made .mut lines; the writer kernels compile for sm_100a
without spills."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from colate_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")
CSRC = os.path.join(ROOT, "colate_b200", "csrc")


@pytest.fixture()
def tdir(built, tmp_path):
    (tmp_path / "syn.mut").write_text("")
    (tmp_path / "syn_chr1.mut").write_text("")
    (tmp_path / "chr.txt").write_text("1\n")
    for i in range(3):
        (tmp_path / f"s{i}.bam").write_bytes(b"")
    (tmp_path / "c_chr1.bcf").write_bytes(b"")
    return tmp_path


def run_targets(d, lines, *flags, chr_list=True, ref=True):
    tf = d / "targets.txt"
    tf.write_text("".join(x + "\n" for x in lines))
    cmd = [CLI, "--mode", "make_tmp", "--mut", str(d / "syn"), "--targets", str(tf)]
    if chr_list:
        cmd += ["--chr", str(d / "chr.txt")]
    if ref:
        cmd += ["--ref_genome", str(d / "g")]
    return subprocess.run(cmd + list(flags), capture_output=True, text=True, timeout=60)


def refused(r, *needles):
    assert r.returncode != 0, r.stderr
    for n in needles:
        assert n in r.stderr, (n, r.stderr)
    # nothing got as far as a device (on this machine there is none: that would read "no CUDA device")
    assert "CUDA" not in r.stderr and "colate_create" not in r.stderr, r.stderr
    return r.stderr


def bam(d, i):
    return f"target_bam={d}/s{i}.bam"


def test_field_counts(tdir):
    d = tdir
    refused(run_targets(d, ["# header", f"{bam(d, 0)} {d}/o0", "", f"{bam(d, 1)}"]), "line 4", "found 1 field(s)")
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0 target_mask={d}/m x"]), "line 1", "found 4 field(s)")
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0 {d}/o1"]), "line 1", "one output prefix, found 2")


@pytest.mark.parametrize("field", ["=x", "target_mask=", "target_bam="])
def test_key_value_syntax(tdir, field):
    d = tdir
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0", f"{bam(d, 1)} {d}/o1 {field}"]), "line 2", "key=value")


def test_unknown_and_repeated_keys(tdir):
    d = tdir
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0 target_age=100"]), "line 1", "unknown key 'target_age'")
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0", f"{bam(d, 1)} {d}/o1 target_mask={d}/m", f"target_mask={d}/m {d}/o2 target_mask={d}/n"]),
            "line 3", "'target_mask' is given twice")
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0 {bam(d, 1)}"]), "line 1", "'target_bam' is given twice")


def test_one_input_per_line(tdir):
    d = tdir
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0 target_bcf={d}/c"]), "line 1", "exactly one of target_bam= and target_bcf=")
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0", f"{d}/o1 target_mask={d}/m"]), "line 2", "exactly one of target_bam= and target_bcf=")


def test_table_lines_are_out_of_scope(tdir):
    d = tdir
    err = refused(run_targets(d, [f"{bam(d, 0)} {d}/o0", f"target_table={d}/t.txt {d}/o1"]), "line 2", "target_table")
    assert "host" in err


def test_duplicate_output_prefix(tdir):
    d = tdir
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0", f"{bam(d, 1)} {d}/o1", f"target_bcf={d}/c {d}/o0"]), "line 3", "already used on line 1")


def test_unreadable_inputs(tdir):
    d = tdir
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0", f"target_bam={d}/nope.bam {d}/o1"]), "line 2", f"cannot read {d}/nope.bam")
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0", f"target_bcf={d}/nope {d}/o1"]), "line 2", f"cannot read {d}/nope_chr1.bcf")
    refused(run_targets(d, [f"{bam(d, 0)} {d}/o0", f"target_bcf={d}/c {d}/o1"], chr_list=False), "line 2", "target_bcf needs --chr")


def test_conflicting_flags(tdir):
    d = tdir
    line = [f"{bam(d, 0)} {d}/o0"]
    for flag, val in (("--target_bam", f"{d}/s0.bam"), ("--target_bcf", f"{d}/c"), ("--target_table", f"{d}/t"), ("--target_mask", f"{d}/m"),
                      ("-o", f"{d}/o")):
        refused(run_targets(d, line, flag, val), "cannot be combined with --targets")
    refused(run_targets(d, line, "--strandfilter"), "--strandfilter")
    refused(run_targets(d, line, "--filters", "20,30"), "--filters")
    refused(run_targets(d, line, "--filters", "20,x,10"), "--filters")
    refused(run_targets(d, line, ref=False), "--ref_genome")
    refused(run_targets(d, line, "--devices", "0,1"), "one device")


def test_no_target(tdir):
    refused(run_targets(tdir, ["# nothing", ""]), "lists no target")


# ---- the make_tmp row word on the host reader's path ------------------------------------------------------------------------------
MKT_VCF, MKT_BAM, MKT_ONE = 1, 2, 4


def _row(snp, pos, typ, flipped=0, branches="5", n_fields=None):
    f = [str(snp), str(pos), "1", "rs", "0", branches, "0", str(flipped), "10.5", "20.25", typ, "C", "G", "3", "4"]
    if n_fields is not None:
        f = f[:n_fields]
    return ";".join(f) + ";"


def _word(a, d, vcf, one):
    return MKT_BAM | (MKT_VCF if vcf else 0) | (MKT_ONE if one else 0) | (ord(a) << 8) | (ord(d) << 16)


# (type field, flipped, branches) -> the word, by the rules of colate_maketmp_pileup / colate_maketmp_records
CASES = [
    ("A/G", 0, "5", _word("A", "G", True, True)),
    ("0/1", 0, "5", _word("0", "1", True, True)),
    ("T/1", 0, "5", _word("T", "1", True, True)),
    ("0/A", 0, "5", _word("0", "A", True, True)),
    ("A/0", 0, "5", _word("A", "0", False, True)),        # 0 is not a derived code of the vcf variant; bam takes any string
    ("1/A", 0, "5", 0),                                    # 1 is not an ancestral code
    ("C/GT", 0, "5", _word("C", "G", False, False)),      # multi-letter derived: bam only, and only its first letter is written
    ("C/GTTACGTAAAAA", 0, "5", _word("C", "G", False, False)),   # 13 characters: kept
    ("C/GTTACGTAAAAAA", 0, "5", _word("C", "G", False, False)),  # 15: kept
    ("C/GTTACGTAAAAAAA", 0, "5", 0),                       # 16 characters: the reader keeps "NN", no code
    ("A/", 0, "5", 0),                                     # empty derived string
    ("AG/T", 0, "5", 0),
    ("/A", 0, "5", 0),
    ("NA", 0, "5", 0),
    ("a/g", 0, "5", 0),                                    # codes are upper case
    ("A/g", 0, "5", _word("A", "g", False, True)),         # bam: any derived string; the lower-case letter counts no reads
    ("A/G", 1, "5", 0),                                    # flipped
    ("A/G", 0, "5 6", 0),                                  # two branches
    ("A/G", 0, "", 0),                                     # no branch
]


def test_row_word_from_host_reader(tmp_path, built):
    lines = ["snp;pos_of_snp;dist;rs-id;tree_index;branch_indices;is_not_mapping;is_flipped;age_begin;age_end;type;ACGT;"]
    want = []
    for k, (typ, fl, br, w) in enumerate(CASES):
        lines.append(_row(k, 100 + k, typ, fl, br))
        want.append(w)
    lines.append(_row(99, 500, "A/G", n_fields=10))        # no type field: the reader's "NA"
    want.append(0)
    p = tmp_path / "x.mut"
    p.write_text("\n".join(lines) + "\n")
    got = api.read_mut_words(str(p))
    assert got.tolist() == want, [(c[0], hex(g), hex(w)) for c, g, w in zip(CASES + [("none",)], got, want) if g != w]
    # the same rows through gzip
    import gzip
    pg = tmp_path / "y.mut"
    with gzip.open(str(pg) + ".gz", "wt") as f:
        f.write("\n".join(lines) + "\n")
    assert api.read_mut_words(str(pg)).tolist() == want
    # the word is the function of (flipped, branches, type as the reader keeps it)
    for typ, fl, br, w in CASES:
        nb = len(br.split())
        t = typ.encode() if len(typ) <= 15 else b"NN"
        assert api.maketmp_word(fl, nb, t) == w, typ


def test_make_tmp_mask_rule(tmp_path, built):
    """make_tmp drops rows at or beyond the mask's end and keeps bp = 0 (not the mode-mut rule of mask_bits_from_fasta)."""
    (tmp_path / "m.fa").write_text(">m\nPPNPx\nPpP\n")           # 8 bases: PPNPXPPP (upper-cased)
    pos = np.array([0, 1, 2, 3, 4, 5, 6, 7, 8, 9, -1, 100], np.int32)
    want = [1, 1, 1, 0, 1, 0, 1, 1, 0, 0, 0, 0]
    bits = np.zeros(2, np.uint32)
    api.maketmp_mask_bits(str(tmp_path / "m.fa"), pos, 3, bits)
    got = [(int(bits[(3 + k) >> 5]) >> ((3 + k) & 31)) & 1 for k in range(len(pos))]
    assert got == want
    mb = np.zeros(2, np.uint32)
    api.mask_bits_from_fasta(str(tmp_path / "m.fa"), pos, 3, mb)
    assert [(int(mb[(3 + k) >> 5]) >> ((3 + k) & 31)) & 1 for k in range(len(pos))][9] == 1     # mode mut keeps rows past the end


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="needs nvcc")
def test_writer_kernels_compile_without_spills(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--fmad=false", "-Xptxas", "-v", "-c",
                        os.path.join(CSRC, "kernels_maketmp.cu"), "-o", str(tmp_path / "k.o")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    found = {}
    cur = None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            found[cur] = (int(m.group(1)), int(m.group(2)))
    names = [k for k in found if "k_maketmp" in k]
    assert len(names) == 4, found                      # rows<0>, rows<1>, scan, scatter
    for k in names:
        assert found[k] == (0, 0), (k, found[k])
