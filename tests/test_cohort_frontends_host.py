"""No GPU: `Colate --mode mut --pairs <file>` with target_bam= / reference_bam= and target_bcf= / reference_bcf= lines refuses, before it
touches a device and naming the line, everything the single-pair BAM / BCF runs refuse; the slot limit counts BAM and BCF genomes
(a BCF prefix once per role); pure .colate.in pairs files keep their messages; the .colate_mat of R = 0 is the age-grid line alone; the two-role k_bcf_rows
compiles for sm_100a without spills."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")
CSRC = os.path.join(ROOT, "colate_b200", "csrc")


@pytest.fixture()
def fdir(built, tmp_path):
    (tmp_path / "syn_chr1.mut").write_text("")
    (tmp_path / "syn.mut").write_text("")
    (tmp_path / "chr.txt").write_text("1\n")
    for i in range(70):
        (tmp_path / f"s{i}.bam").write_bytes(b"")
        (tmp_path / f"v{i}_chr1.bcf").write_bytes(b"")
    for i in range(4):
        (tmp_path / f"g{i}.colate.in").write_bytes(b"")
    return tmp_path


def run_pairs(d, lines, *flags, chr_list=True, ref=True):
    pf = d / "pairs.txt"
    pf.write_text("".join(x + "\n" for x in lines))
    cmd = [CLI, "--mode", "mut", "--mut", str(d / "syn"), "--pairs", str(pf), "--seed", "1", "--bins", "3,7,0.2"]
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
    assert "CUDA" not in r.stderr and "colate_create" not in r.stderr and "handle" not in r.stderr, r.stderr
    return r.stderr


def bam(d, i, j, out=None):
    return f"target_bam={d}/s{i}.bam reference_bam={d}/s{j}.bam {d}/{out or f'o{i}_{j}'}"


def bcf(d, i, j, out=None):
    return f"target_bcf={d}/v{i} reference_bcf={d}/v{j} {d}/{out or f'p{i}_{j}'}"


def test_mixed_kinds_are_refused(fdir):
    d = fdir
    refused(run_pairs(d, [bam(d, 0, 1), f"target_bam={d}/s0.bam reference_bcf={d}/v1 {d}/x"]), "line 2", "a bam target with a bcf reference")
    refused(run_pairs(d, [f"target_bcf={d}/v0 reference_bam={d}/s1.bam {d}/x"]), "line 1", "a bcf target with a bam reference")
    refused(run_pairs(d, [f"target_bam={d}/s0.bam {d}/g1.colate.in {d}/x"]), "line 1", "a bam target with a .colate.in reference")
    refused(run_pairs(d, [bcf(d, 0, 1), f"{d}/g0.colate.in reference_bcf={d}/v1 {d}/x"]), "line 2", "a .colate.in target with a bcf reference")


def test_roles_in_the_wrong_field_are_refused(fdir):
    d = fdir
    refused(run_pairs(d, [f"reference_bam={d}/s0.bam reference_bam={d}/s1.bam {d}/x"]), "line 1", "'reference_bam=' in field 1")
    refused(run_pairs(d, [bcf(d, 0, 1), f"reference_bcf={d}/v0 target_bcf={d}/v1 {d}/x"]), "line 2", "'reference_bcf=' in field 1")
    refused(run_pairs(d, [f"target_bam={d}/s0.bam target_bam={d}/s1.bam {d}/x"]), "line 1", "'target_bam=' in field 2")
    refused(run_pairs(d, [f"{bam(d, 0, 1)} target_bcf={d}/v0"]), "line 1", "'target_bcf=' goes in field 1")
    refused(run_pairs(d, [f"target_bam= reference_bam={d}/s1.bam {d}/x"]), "line 1", "key=value")


def test_bam_lines_need_ref_genome_and_no_strandfilter(fdir):
    d = fdir
    refused(run_pairs(d, [bcf(d, 0, 1), bam(d, 0, 1)], ref=False), "line 2", "BAM inputs need --ref_genome")
    refused(run_pairs(d, [bcf(d, 0, 1), bam(d, 0, 1)], "--strandfilter"), "line 2", "--strandfilter")
    refused(run_pairs(d, [bam(d, 0, 1)], "--filters", "20,30"), "--filters")


def test_bcf_lines_need_chr(fdir):
    d = fdir
    refused(run_pairs(d, [bam(d, 0, 1), bcf(d, 0, 1)], chr_list=False), "line 2", "BCF inputs need --chr")


def test_unreadable_inputs(fdir):
    d = fdir
    refused(run_pairs(d, [bam(d, 0, 1), f"target_bam={d}/s0.bam reference_bam={d}/nope.bam {d}/x"]), "line 2", f"cannot read {d}/nope.bam")
    refused(run_pairs(d, [bcf(d, 0, 1), f"target_bcf={d}/nope reference_bcf={d}/v1 {d}/x"]), "line 2", f"cannot read {d}/nope_chr1.bcf")


def test_single_pair_input_flags_stay_refused(fdir):
    d = fdir
    for flag, val in (("--target_bam", f"{d}/s0.bam"), ("--reference_bam", f"{d}/s1.bam"), ("--target_bcf", f"{d}/v0"), ("--reference_bcf", f"{d}/v1")):
        refused(run_pairs(d, [bam(d, 0, 1)], flag, val), f"{flag} cannot be combined with --pairs")


def test_unknown_key_message_lists_the_new_keys(fdir):
    d = fdir
    err = refused(run_pairs(d, [f"{bam(d, 0, 1)} seed=3"]), "line 1", "unknown key 'seed' (known: target_age, reference_age, target_mask, reference_mask")
    assert "target_bam" in err and "reference_bcf" in err


def test_slot_limit_counts_front_end_genomes(fdir):
    d = fdir
    lines = [bam(d, 2 * k, 2 * k + 1) for k in range(16)]                      # 32 BAM genomes
    lines += [bcf(d, 2 * k, 2 * k + 1) for k in range(16)]                     # 32 BCF genomes: 64 slots, fine so far
    # a BAM already in a slot takes the reference role at no cost; the same BAM under a mask is another slot
    ok = run_pairs(d, lines + [bam(d, 1, 0, "swapped")], "--filters", "20,x,10")
    assert "more than 64" not in ok.stderr and "line 33" not in ok.stderr
    refused(run_pairs(d, lines + [f"{bam(d, 0, 1, 'm')} target_mask={d}/m"]), "line 33", "more than 64")
    # a BCF prefix is one slot per role: v1 was a reference only
    refused(run_pairs(d, lines + [bcf(d, 1, 0, "swapped")]), "line 33", "more than 64")
    refused(run_pairs(d, lines[:-1] + [bcf(d, 30, 31), bcf(d, 31, 30, "swapped")]), "line 33", "more than 64")


def test_pure_tmp_pairs_files_keep_their_messages(fdir):
    d = fdir
    g = lambda i: f"{d}/g{i}.colate.in"
    refused(run_pairs(d, [f"{g(0)} {g(1)} {d}/o0 seed=3"]), "line 1", "unknown key 'seed' (known: target_age, reference_age, target_mask, reference_mask")
    refused(run_pairs(d, [f"{g(0)} {g(1)} {d}/o0", f"{g(0)} {d}/missing.colate.in {d}/o1"]), "line 2", "cannot read", "missing.colate.in")
    refused(run_pairs(d, [f"{g(0)} {g(1)}"]), "line 1", "found 2 field(s)")
    refused(run_pairs(d, [f"{g(0)} {g(1)} {d}/same", f"{g(2)} {g(3)} {d}/same"]), "line 2", "already used on line 1")
    # the BAM-only flag checks do not apply to .colate.in lines
    r = run_pairs(d, [f"{g(0)} {g(1)} {d}/o0 bad"], "--strandfilter", ref=False)
    refused(r, "line 1", "key=value")


def test_nothing_is_written(fdir):
    d = fdir
    run_pairs(d, [bam(d, 0, 1), bcf(d, 0, 1), f"{bam(d, 2, 3)} bad"])
    assert not any(p.name.startswith(("o", "p")) and p.name != "pairs.txt" for p in d.iterdir())


def test_colate_mat_of_zero_replicates_is_the_grid_line(built, tmp_path):
    """--num_bootstraps 0 on a BAM / BCF line (alone or in a cohort): <out>.colate_mat is the age-grid line alone, as the reference
    writes it (coal.cpp:3336-3343; the per-replicate lines of 3453-3465 are a loop over no replicates)."""
    from colate_b200 import _lib, api
    api.write_colate_mat(str(tmp_path / "r0.colate_mat"), np.zeros((0, 2, api.NBINS)))
    api.write_colate_mat(str(tmp_path / "r1.colate_mat"), np.ones((1, 2, api.NBINS)))
    r0 = open(tmp_path / "r0.colate_mat").read()
    assert r0 == open(tmp_path / "r1.colate_mat").read().split("\n")[0] + "\n"
    with pytest.raises(_lib.ColateError):
        _lib.check(_lib.lib().colate_write_colate_mat(str(tmp_path / "neg.colate_mat").encode(), -1, api.age_bins(), np.zeros(2 * api.NBINS)))


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="needs nvcc")
def test_two_role_rows_kernel_compiles_without_spills(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--fmad=false", "-Xptxas", "-v", "-c",
                        os.path.join(CSRC, "kernels_bcf.cu"), "-o", str(tmp_path / "k.o")], capture_output=True, text=True, timeout=600)
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
    names = [k for k in found if "k_bcf_rows" in k]
    assert len(names) == 1, found                      # one kernel for both roles
    assert found[names[0]] == (0, 0), found[names[0]]
