"""No GPU: whole-genome BCF / VCF files, host side.  bcf_genome_scan (colate_bcf_genome_scan) agrees with a gzip + struct / text
parse on BCF with and without contig IDX= and on VCF; every host refusal of the whole-genome walk; the CLI's detection rule
(per-chromosome files first, so today's messages stand) and its refusals before any device is touched; BAM's contig messages."""
import os
import subprocess
import sys

import numpy as np
import pytest

from colate_b200 import _lib, api, synth

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from genome_files import decoys, genome_layout, parse, write_genome  # noqa: E402

CLI = os.path.join(os.path.dirname(HERE), "colate_b200", "bin", "Colate")
NAMES = ["1", "2", "X"]


def _recs(rng, n, n_hap, step=(0, 4)):
    p = int(rng.integers(0, 50))
    out = []
    for _ in range(n):
        p += int(rng.integers(*step))
        out.append((p, [b"A", b"C"] if rng.random() < 0.8 else [b"T"], [int(x) for x in rng.integers(0, 2, n_hap)]))
    return out


def _layout(rng, ns=3, prefix_chr=False):
    recs = [_recs(rng, n, ns * 2) for n in (40, 25, 60)]
    return recs, genome_layout(rng, NAMES, recs, ns, prefix_chr=prefix_chr)


@pytest.mark.parametrize("fmt, idx, prefix_chr", [("bcf", False, False), ("bcf", True, True), ("vcf", False, True), ("vcf", False, False)])
def test_scan_agrees_with_a_struct_parse(built, tmp_path, fmt, idx, prefix_chr):
    rng = np.random.default_rng(3)
    recs, contigs = _layout(rng, prefix_chr=prefix_chr)
    names = [nm for nm, _, _ in contigs]
    cidx = {nm: 2 * k + 5 for k, nm in enumerate(names[::-1])} if idx else None      # IDX= overrides the line order
    f = str(tmp_path / "g.gz")
    write_genome(f, fmt, 3, contigs, contig_idx=cidx, block_size=997)
    by_contig, ns = parse(f)
    assert list(by_contig) == names
    for wb in (0, 101, 5000):
        s = api.bcf_genome_scan(f, NAMES, wb)
        assert s["n_sample"] == ns == 3
        for c, nm in enumerate(NAMES):
            pos = by_contig[("chr" if prefix_chr else "") + nm]
            assert (s["n_records"][c], s["first_pos"][c], s["last_pos"][c]) == (len(pos), pos[0], pos[-1]), (wb, nm)
            assert [p for p, _, _ in recs[c]] == pos
    # a subset of the contigs: the others are walked past
    s = api.bcf_genome_scan(f, ["X"])
    assert s["n_records"][0] == len(recs[2])


def _refused(f, names, *needles):
    with pytest.raises(_lib.ColateError) as e:
        api.bcf_genome_scan(f, names, 211)
    for n in needles:
        assert n in str(e.value), (n, str(e.value))
    return str(e.value)


@pytest.mark.parametrize("fmt", ["bcf", "vcf"])
def test_host_refusals(built, tmp_path, fmt):
    rng = np.random.default_rng(5)
    a, b = _recs(rng, 20, 4), _recs(rng, 20, 4)
    f = str(tmp_path / "g.gz")
    kind = fmt.upper()
    # a listed contig in two runs
    write_genome(f, fmt, 2, [("1", a[:10], 2), ("2", b, 2), ("1", a[10:], 2)])
    _refused(f, ["1", "2"], f, "records of contig 1 are not contiguous", "at inflated byte offset")
    # ... also when only unlisted records come between
    write_genome(f, fmt, 2, [("1", a[:10], 2), ("decoy", decoys(rng, 2, 2), 2), ("1", a[10:], 2)])
    _refused(f, ["1"], "records of contig 1 are not contiguous")
    # a listed contig without records
    write_genome(f, fmt, 2, [("1", a, 2), ("decoy", decoys(rng, 2, 2), 2)], header_contigs=["decoy", "1", "2"])
    _refused(f, ["1", "2"], f, f"{kind} file without records of contig 2 of the --chr list (neither 2 nor chr2")
    # a contig matching two entries
    write_genome(f, fmt, 2, [("chr1", a, 2)])
    _refused(f, ["1", "chr1"], f, "contig chr1 matches two --chr entries")
    # an entry matched by two contigs that both have records; with one of them empty the file is fine
    write_genome(f, fmt, 2, [("1", a, 2), ("chr1", b, 2)])
    _refused(f, ["1"], f, f"contig 1 of the --chr list appears in the {kind} file as both 1 and chr1")
    write_genome(f, fmt, 2, [("chr1", a, 2)], header_contigs=["1", "chr1"])
    assert api.bcf_genome_scan(f, ["1"])["n_records"][0] == len(a)
    # POS descending inside a listed contig: today's message; unlisted contigs are not order-checked
    bad = a[:6] + [(a[5][0] - 1,) + a[5][1:]] + a[6:]
    write_genome(f, fmt, 2, [("decoy", decoys(rng, 2, 2), 2), ("1", bad, 2)])
    _refused(f, ["1"], f"{kind} records not sorted by position (POS {a[5][0]} after {a[5][0] + 1})")


def test_bcf_chrom_outside_the_dictionary(built, tmp_path):
    rng = np.random.default_rng(6)
    f = str(tmp_path / "g.bcf")
    write_genome(f, "bcf", 2, [("1", _recs(rng, 5, 4), 2), ("2", _recs(rng, 5, 4), 2)], header_contigs=["1"], contig_idx={"1": 0, "2": 7})
    _refused(f, ["1"], "BCF record on contig 7, which no ##contig line of the header defines")


def test_per_chromosome_scans_keep_the_one_contig_rule(built, tmp_path):
    rng = np.random.default_rng(7)
    f = str(tmp_path / "g.bcf")
    write_genome(f, "bcf", 2, [("1", _recs(rng, 5, 4), 2), ("2", _recs(rng, 5, 4), 2)])
    with pytest.raises(_lib.ColateError, match="a per-chromosome file holds one contig"):
        api.bcf_scan(f)
    v = str(tmp_path / "g.vcf.gz")
    write_genome(v, "vcf", 2, [("1", _recs(rng, 5, 4), 2), ("2", _recs(rng, 5, 4), 2)])
    with pytest.raises(_lib.ColateError, match="a per-chromosome file holds one contig"):
        api.vcf_scan(v)


# ---- the CLI: detection and refusals before a device ----------------------------------------------------------------------------
@pytest.fixture()
def cdir(built, tmp_path):
    rng = np.random.default_rng(9)
    (tmp_path / "chr.txt").write_text("1\n2\n")
    for nm in ("1", "2"):
        (tmp_path / f"syn_chr{nm}.mut").write_text("")
    recs = [_recs(rng, 10, 2), _recs(rng, 10, 2)]
    write_genome(str(tmp_path / "whole.vcf.gz"), "vcf", 1, [("chr2", recs[1], 2), ("chr1", recs[0], 2)])
    return tmp_path


def _run(d, *args):
    return subprocess.run([CLI, "--mut", str(d / "syn"), "--chr", str(d / "chr.txt")] + list(args), capture_output=True, text=True, timeout=60)


def _before_device(r, *needles):
    assert r.returncode != 0, r.stderr
    for n in needles:
        assert n in r.stderr, (n, r.stderr)
    assert "CUDA" not in r.stderr and "colate_create" not in r.stderr and "handle" not in r.stderr, r.stderr


def test_per_chromosome_files_take_precedence(cdir):
    d = cdir
    # X is a regular file and X_chr1.bcf exists: per-chromosome, and the missing X_chr2.bcf is today's message
    (d / "whole.vcf.gz_chr1.bcf").write_bytes(b"")
    tg = d / "targets.txt"
    tg.write_text(f"target_bcf={d}/whole.vcf.gz {d}/o\n")
    r = _run(d, "--mode", "make_tmp", "--ref_genome", str(d / "g"), "--targets", str(tg))
    _before_device(r, "line 1", f"cannot read {d}/whole.vcf.gz_chr2.bcf")
    pf = d / "pairs.txt"
    pf.write_text(f"target_bcf={d}/whole.vcf.gz reference_bcf={d}/whole.vcf.gz {d}/p\n")
    r = _run(d, "--mode", "mut", "--pairs", str(pf), "--seed", "1", "--bins", "3,7,0.2")
    _before_device(r, "line 1", f"cannot read {d}/whole.vcf.gz_chr2.bcf")


def test_missing_inputs_keep_the_per_chromosome_message(cdir):
    d = cdir
    tg = d / "targets.txt"
    tg.write_text(f"target_bcf={d}/nothing {d}/o\n")
    _before_device(_run(d, "--mode", "make_tmp", "--ref_genome", str(d / "g"), "--targets", str(tg)), f"cannot read {d}/nothing_chr1.bcf")
    # a directory is not a whole-genome file
    os.mkdir(d / "adir")
    tg.write_text(f"target_bcf={d}/adir {d}/o\n")
    _before_device(_run(d, "--mode", "make_tmp", "--ref_genome", str(d / "g"), "--targets", str(tg)), f"cannot read {d}/adir_chr1.bcf")


def test_whole_genome_lines_keep_the_argument_refusals(cdir):
    d = cdir
    w = f"{d}/whole.vcf.gz"
    pf = d / "pairs.txt"
    pf.write_text(f"target_bcf={w} reference_bcf={w} {d}/p\n")
    r = subprocess.run([CLI, "--mode", "mut", "--mut", str(d / "syn"), "--pairs", str(pf), "--seed", "1", "--bins", "3,7,0.2"],
                       capture_output=True, text=True, timeout=60)
    _before_device(r, "line 1", "BCF inputs need --chr")
    pf.write_text(f"target_bcf={w} reference_bam={d}/x.bam {d}/p\n")
    _before_device(_run(d, "--mode", "mut", "--pairs", str(pf), "--seed", "1", "--bins", "3,7,0.2"), "line 1")
    r = subprocess.run([CLI, "--mode", "mut", "--mut", str(d / "syn"), "--target_bcf", w, "--reference_bcf", w, "--seed", "1", "--bins", "3,7,0.2",
                        "-o", str(d / "o")], capture_output=True, text=True, timeout=60)
    _before_device(r, "BCF inputs need --chr")
    r = _run(d, "--mode", "mut", "--target_bcf", w, "--reference_bcf", w, "--devices", "0,1", "--seed", "1", "--bins", "3,7,0.2", "-o", str(d / "o"))
    _before_device(r, "BCF inputs run on one device")
    tg = d / "targets.txt"
    tg.write_text(f"target_bcf={w} {d}/o\n")
    r = subprocess.run([CLI, "--mode", "make_tmp", "--mut", str(d / "syn"), "--ref_genome", str(d / "g"), "--targets", str(tg)],
                       capture_output=True, text=True, timeout=60)
    _before_device(r, "line 1", "target_bcf needs --chr")


# ---- BAM: the contig rule moved, its messages did not ---------------------------------------------------------------------------
def test_bam_contig_messages_unchanged(built, tmp_path):
    f = str(tmp_path / "a.bam")
    synth.write_bam(f, ["1", "chr1", "chr2"], [])
    with pytest.raises(_lib.ColateError) as e:
        api.bam_scan(f, ["1"])
    assert str(e.value).endswith(f"{f}: contig 1 of the --chr list appears in the BAM header as both 1 and chr1")
    with pytest.raises(_lib.ColateError) as e:
        api.bam_scan(f, ["2", "chr2"])
    assert str(e.value).endswith(f"{f}: header contig chr2 matches two --chr entries")
    with pytest.raises(_lib.ColateError) as e:
        api.bam_scan(f, ["3"])
    assert str(e.value).endswith(f"{f}: contig 3 of the --chr list is not in the BAM header (neither 3 nor chr3)")
    assert list(api.bam_scan(f, ["2"])["ref_id"]) == [2]
