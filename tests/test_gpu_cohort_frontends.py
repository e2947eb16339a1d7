"""GPU: cohorts on BAM and BCF / VCF pairs (`--pairs` lines with target_bam= / reference_bam= and target_bcf= / reference_bcf=).

* the bambam line inside a cohort reproduces the reference CLI's goldens (tests/golden/bambam_R1 / R3), next to swapped, masked,
  aged and .colate.in lines;
* every line's .coal / .bin / .colate_mat equal the single-pair run of that line byte for byte (BCF, VCF and mixed prefixes, with and
  without --ref_genome, one prefix in both roles and under two masks, R = 0), on one and on several devices;
* every input file is decoded once per device, the genome uploaded and the .mut text parsed once per device (the summary lines);
* the two-role k_bcf_rows (colate_rows_from_bcf_roles) equals colate_rows_from_bcf per role bit for bit, and colate_copy_genome +
  a mask equals a fresh decode under that mask;
* failing genomes fail only their lines; the stale-cache path; pairs.cohort(front_ends=...)."""
import ctypes as C
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from colate_b200 import _lib, api, pairs, synth

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
from bcf_helpers import IDS, random_records  # noqa: E402
from helpers import GOLDEN, bambam_masks  # noqa: E402
from test_gpu_bam import _fixture_reads, golden_dir  # noqa: E402,F401  (module fixture: the bambam fixture as BAM files)
from test_gpu_bcf import _fixture_recs, _write_records  # noqa: E402
from test_gpu_vcf import vcf_dir  # noqa: E402,F401  (module fixture: the vcfvcf fixture as BCF t / r and VCF tv / rv)

CLI = os.path.join(os.path.dirname(HERE), "colate_b200", "bin", "Colate")
pytestmark = pytest.mark.gpu
EXTS = (".coal", ".bin", ".colate_mat")
SUMMARY = re.compile(r"device (\d+) \(handle \d+ of \d+\): BAM files piled (\d+), BCF/VCF files decoded (\d+), \.mut texts parsed (\d+) "
                     r"\((\d+) rows\), reference genome uploads (\d+) \((\d+) bytes\)")


def _run(args):
    return subprocess.run([CLI] + args, capture_output=True, text=True, timeout=900)


def _files(o):
    return {e: open(o + e, "rb").read() for e in EXTS if os.path.exists(o + e)}


def _shared(d, R, refg=True):
    a = ["--mode", "mut", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--bins", "3,7,0.2", "--seed", "23",
         "--num_bootstraps", str(R)]
    return a + (["--ref_genome", os.path.join(d, "g")] if refg else [])


def _line_flags(line):
    """A pairs-file line -> (output prefix, the single-pair run's flags)."""
    f = line.split()
    flags = []
    for x, tmp_flag in zip(f[:2], ("--target_tmp", "--reference_tmp")):
        k, _, v = x.partition("=")
        flags += ["--" + k, v] if v else [tmp_flag, x]
    for x in f[3:]:
        k, _, v = x.partition("=")
        flags += ["--" + k, v]
    return f[2], flags


def _cohort_vs_single(tmp_path, shared, lines, extra=()):
    """Runs the cohort, then every line alone; returns (cohort stderr, {out: files}) after checking each line byte for byte."""
    pf = tmp_path / "pairs.txt"
    pf.write_text("".join(x + "\n" for x in lines))
    r = _run(shared + ["--pairs", str(pf)] + list(extra))
    assert r.returncode == 0, r.stderr[-3000:]
    got = {}
    for ln in lines:
        out, flags = _line_flags(ln)
        one = out + "_single"
        q = _run(shared + flags + ["-o", one])
        assert q.returncode == 0, (ln, q.stderr[-3000:])
        got[out] = _files(out)
        want = _files(one)
        assert set(got[out]) == set(want), (ln, sorted(got[out]), sorted(want))
        for e in want:
            assert got[out][e] == want[e], (ln, e)
    return r.stderr, got


def _summaries(err):
    return [tuple(int(x) for x in m.groups()) for m in SUMMARY.finditer(err)]


# ---- 1. the reference goldens inside a cohort; BAM lines equal their single runs; work counts ------------------------------------
@pytest.mark.parametrize("R", [1, 3])
def test_bambam_goldens_inside_a_cohort(golden_dir, tmp_path, R):
    d, z, sites, *_ = golden_dir
    tg = tmp_path / "targets.txt"
    tg.write_text(f"target_bam={d}/t.bam {tmp_path}/tt\ntarget_bam={d}/r.bam {tmp_path}/rt\n")
    q = _run(["--mode", "make_tmp", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--ref_genome", os.path.join(d, "g"),
              "--targets", str(tg)])
    assert q.returncode == 0, q.stderr[-3000:]
    t = tmp_path
    lines = [f"target_bam={d}/r.bam reference_bam={d}/t.bam {t}/swapped",
             f"target_bam={d}/t.bam reference_bam={d}/r.bam {t}/o",
             f"target_bam={d}/t.bam reference_bam={d}/r.bam {t}/masked target_mask={d}/tm",
             f"target_bam={d}/t.bam reference_bam={d}/r.bam {t}/aged target_age=2000",
             f"{t}/tt.colate.in {t}/rt.colate.in {t}/tmp"]
    err, got = _cohort_vs_single(tmp_path, _shared(d, R), lines)
    for e in (".coal", ".colate_mat"):
        assert got[f"{t}/o"][e] == open(os.path.join(GOLDEN, f"bambam_R{R}{e}"), "rb").read(), e
    assert ".colate_mat" not in got[f"{t}/tmp"]
    (dev, n_bam, n_bcf, n_txt, n_rows, n_up, n_bytes), = _summaries(err)
    assert (n_bam, n_bcf, n_txt, n_rows, n_up) == (2, 0, len(sites.chr_names), int(sites.site_off[-1]), 1), err
    assert n_bytes == sum(len(g) for g in golden_dir[4])


# ---- 2. BCF / VCF lines equal their single runs; work counts -----------------------------------------------------------------------
@pytest.mark.parametrize("R, refg", [(1, False), (3, True), (0, True)])
def test_bcf_vcf_lines_equal_single_runs(vcf_dir, tmp_path, R, refg):
    d, z, sites, genome = vcf_dir
    tm, rm = bambam_masks(z)
    for c, nm in enumerate(sites.chr_names):
        synth.write_mask(str(tmp_path / f"tm_chr{nm}.fa"), tm[c])
        synth.write_mask(str(tmp_path / f"rm_chr{nm}.fa"), rm[c])
    t = tmp_path
    lines = [f"target_bcf={d}/t reference_bcf={d}/r {t}/a",
             f"target_bcf={d}/tv reference_bcf={d}/rv {t}/b",
             f"target_bcf={d}/t reference_bcf={d}/rv {t}/c",
             f"target_bcf={d}/r reference_bcf={d}/t {t}/d",                       # t: target on line 1, reference here
             f"target_bcf={d}/t reference_bcf={d}/r {t}/e target_mask={t}/tm",     # t as target under a second mask
             f"target_bcf={d}/tv reference_bcf={d}/r {t}/f reference_mask={t}/rm target_age=1500"]
    err, got = _cohort_vs_single(tmp_path, _shared(d, R, refg), lines)
    for o in got:
        assert ".colate_mat" in got[o]
    (dev, n_bam, n_bcf, n_txt, n_rows, n_up, n_bytes), = _summaries(err)
    # four prefixes (t, r, tv, rv), each decoded once although t and r are used in both roles and t under two masks
    assert (n_bam, n_bcf, n_txt, n_up) == (0, 4 * len(sites.chr_names), len(sites.chr_names), 1 if refg else 0), err


# ---- 4. the two-role kernel ------------------------------------------------------------------------------------------------------
def _slot_rows(handle, slot):
    """(AAF, DAF) per row of a row-count slot (colate_pileup_end copies the slot's columns out; the slot is not used afterwards)."""
    p4 = np.zeros((handle.n_site, 4), np.int32)
    _lib.check(_lib.lib().colate_pileup_end(handle._h, slot, p4.ctypes.data_as(C.c_void_p)))
    return p4[:, 0].copy(), p4[:, 1].copy()


def _roles_equal_per_role(handle, paths, genome):
    """rows_from_bcf_roles with no genome / the resident genome vs rows_from_bcf with none / the host genome."""
    for genome_mode in (0, 1):
        host = genome if genome_mode else None
        want_t = handle.rows_from_bcf(2, paths, "target", host, fetch=True)
        want_r = handle.rows_from_bcf(3, paths, "reference", host, fetch=True)
        if genome_mode:
            handle.set_ref_genome(genome)
        handle.rows_from_bcf_roles(0, 1, paths, genome_mode)
        for slot, want in ((0, want_t), (1, want_r)):
            got = _slot_rows(handle, slot)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (genome_mode, slot)
        # one role at a time, into other slots
        handle.rows_from_bcf_roles(-1, 4, paths, genome_mode)
        handle.rows_from_bcf_roles(5, -1, paths, genome_mode)
        for slot, want in ((4, want_r), (5, want_t)):
            got = _slot_rows(handle, slot)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (genome_mode, slot)
    handle.set_ref_genome([])


def test_two_role_rows_equal_each_role_on_the_fixture(vcf_dir, handle):
    d, z, sites, genome = vcf_dir
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    for prefix in ("t", "r", "tv"):
        _roles_equal_per_role(handle, [os.path.join(d, f"{prefix}_chr{nm}.bcf") for nm in sites.chr_names], genome)


def test_two_role_rows_equal_each_role_on_random_records(handle, tmp_path):
    rng = np.random.default_rng(11)
    lens = [60000, 40000]
    sites = synth.make_sites(12, [3000, 2000], lens)
    genome = [np.frombuffer(b"ACGTacgtN", np.uint8)[rng.integers(0, 9, L)].copy() for L in lens]
    letters = [b"A", b"C", b"G", b"T"]

    def alleles(r, k):        # one-allele records (REF alone) for a third of them
        al = [letters[int(x)] for x in r.permutation(4)[:int(r.choice([1, 2, 2, 3]))]]
        return al
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    for n_sample in (1, 4):
        paths = []
        for c, L in enumerate(lens):
            out, recs = random_records(rng, 25000 if c == 0 else 15000, n_sample, pos_step=(0, 3), alleles=alleles, extras=False)
            assert any(recs[i][0] == recs[i + 1][0] for i in range(len(recs) - 1))          # repeated positions
            assert any(len(x[1]) == 1 for x in recs)                                          # one-allele records
            paths.append(str(tmp_path / f"x{n_sample}_{c}.bcf"))
            synth.write_bcf(paths[-1], synth.bcf_header(n_sample, IDS), out)
        _roles_equal_per_role(handle, paths, genome)


def test_copy_genome_then_mask_equals_a_fresh_decode(vcf_dir, handle):
    d, z, sites, genome = vcf_dir
    tm, rm = bambam_masks(z)
    bits = api.mask_bits_from_seq(tm, sites.site_off, sites.pos)
    paths = {p: [os.path.join(d, f"{p}_chr{nm}.bcf") for nm in sites.chr_names] for p in ("t", "r")}
    handle.set_option("front_end", 1)
    try:
        handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
        handle.set_ref_genome(genome)
        handle.rows_from_bcf_roles(0, 1, paths["t"], 1)
        handle.rows_from_bcf_roles(-1, 2, paths["r"], 1)
        handle.set_mask(0, bits)
        handle.copy_genome(3, 0)                    # the copy starts without the source's mask
        s_plain = handle.stage1(api.mt_seed(23), target_slot=3, reference_slot=2)
        handle.set_mask(3, bits)
        s_copy = handle.stage1(api.mt_seed(23), target_slot=3, reference_slot=2)
        handle.rows_from_bcf(4, paths["t"], "target", genome)
        handle.set_mask(4, bits)
        s_fresh = handle.stage1(api.mt_seed(23), target_slot=4, reference_slot=2)
        handle.set_mask(4, None)
        s_fresh_plain = handle.stage1(api.mt_seed(23), target_slot=4, reference_slot=2)
        for a, b in ((s_copy, s_fresh), (s_plain, s_fresh_plain)):
            assert a.num_blocks == b.num_blocks and a.n_used == b.n_used
            assert np.array_equal(a.block_stats, b.block_stats) and np.array_equal(a.block_tallies, b.block_tallies)
            assert np.array_equal(a.mt_state, b.mt_state)
        assert s_copy.n_used != s_plain.n_used
        # a .colate.in record slot is not copied; nor is a slot onto itself
        handle.set_genome(5, np.zeros(1, np.int32), np.array([int(sites.pos[0])], np.int32), np.ones(1, np.int32), np.ones(1, np.int32),
                          np.array([ord("A") | ord("C") << 8], np.uint16))
        with pytest.raises(_lib.ColateError):
            handle.copy_genome(6, 5)
        with pytest.raises(_lib.ColateError):
            handle.copy_genome(0, 0)
    finally:
        handle.set_option("front_end", 0)
        handle.set_ref_genome([])
        for s in range(5):
            handle.set_mask(s, None)


def test_resident_genome_is_required_for_genome_1(vcf_dir, handle):
    d, z, sites, genome = vcf_dir
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    handle.set_ref_genome([])
    with pytest.raises(_lib.ColateError) as e:
        handle.rows_from_bcf_roles(0, 1, [os.path.join(d, f"t_chr{nm}.bcf") for nm in sites.chr_names], 1)
    assert e.value.code == -7 and "colate_set_ref_genome" in str(e.value)


# ---- 5. devices ------------------------------------------------------------------------------------------------------------------
def test_devices_give_identical_files(golden_dir, tmp_path):
    import torch
    d, z, sites, *_ = golden_dir
    lists = ["0", "0,0"] + (["0,1"] if torch.cuda.device_count() >= 2 else [])
    outs = {}
    for dl in lists:
        t = tmp_path / dl.replace(",", "_")
        t.mkdir()
        lines = [f"target_bam={d}/t.bam reference_bam={d}/r.bam {t}/a",
                 f"target_bam={d}/r.bam reference_bam={d}/t.bam {t}/b target_mask={d}/tm",
                 f"target_bam={d}/t.bam reference_bam={d}/r.bam {t}/c reference_age=300 target_age=900"]
        (t / "pairs.txt").write_text("".join(x + "\n" for x in lines))
        r = _run(_shared(d, 2) + ["--pairs", str(t / "pairs.txt"), "--devices", dl])
        assert r.returncode == 0, r.stderr[-3000:]
        outs[dl] = {x: _files(f"{t}/{x}") for x in "abc"}
        n_dev = len(dl.split(","))
        summ = _summaries(r.stderr)
        assert len(summ) == min(n_dev, 3)
        if n_dev == 2:       # pairs a, c on the first handle; b on the second: each pile its own inputs, once
            assert sorted(s[1] for s in summ) == [2, 2] and all(s[5] == 1 for s in summ), r.stderr
    for dl in lists:
        assert outs[dl] == outs["0"], dl


# ---- 6. failing genomes ----------------------------------------------------------------------------------------------------------
def test_failing_genomes_fail_only_their_lines(golden_dir, vcf_dir, tmp_path):
    d, z, sites, lens, genome, reads_t, reads_r = golden_dir
    # an unsorted BAM: two records of the first contig swapped
    rd = _fixture_reads(reads_t, np.random.default_rng(1))
    k = next(i for i in range(len(rd) - 1) if rd[i][0] == rd[i + 1][0] and rd[i][1] < rd[i + 1][1])
    rd[k], rd[k + 1] = rd[k + 1], rd[k]
    bam_names = ["chr" + sites.chr_names[0], sites.chr_names[1]]
    synth.write_bam(str(tmp_path / "bad.bam"), bam_names, rd, contig_lens=lens)
    t = tmp_path
    lines = [f"target_bam={t}/bad.bam reference_bam={d}/r.bam {t}/x1",
             f"target_bam={d}/t.bam reference_bam={d}/r.bam {t}/ok",
             f"target_bam={d}/r.bam reference_bam={t}/bad.bam {t}/x2 target_mask={d}/tm"]
    (t / "pairs.txt").write_text("".join(x + "\n" for x in lines))
    r = _run(_shared(d, 1) + ["--pairs", str(t / "pairs.txt")])
    assert r.returncode == 1, r.stderr[-3000:]
    assert "2 of 3 pairs failed" in r.stderr and "bad.bam" in r.stderr and "not sorted" in r.stderr, r.stderr
    assert not any(os.path.exists(f"{t}/x{i}{e}") for i in (1, 2) for e in EXTS)
    q = _run(_shared(d, 1) + ["--target_bam", f"{d}/t.bam", "--reference_bam", f"{d}/r.bam", "-o", f"{t}/ok_single"])
    assert q.returncode == 0 and _files(f"{t}/ok") == _files(f"{t}/ok_single")

    # a BCF with a '.' genotype
    dv, zv, sv, gv = vcf_dir
    v = tmp_path / "v"
    v.mkdir()
    for c, nm in enumerate(sv.chr_names):
        recs = _fixture_recs(zv, "t", c)
        if c == 1:
            p0, al, gt = recs[5]
            recs[5] = (p0, al, [-1] + gt[1:])
        _write_records(str(v / f"bad_chr{nm}.bcf"), int(zv["n_hap_target"]) // 2, 2, recs)
    lines = [f"target_bcf={v}/bad reference_bcf={dv}/r {v}/x1", f"target_bcf={dv}/t reference_bcf={dv}/r {v}/ok",
             f"target_bcf={dv}/r reference_bcf={v}/bad {v}/x2"]
    (v / "pairs.txt").write_text("".join(x + "\n" for x in lines))
    r = _run(_shared(dv, 2, refg=False) + ["--pairs", str(v / "pairs.txt")])
    assert r.returncode == 1 and "2 of 3 pairs failed" in r.stderr and "bad_chr" in r.stderr and "missing" in r.stderr, r.stderr[-3000:]
    assert not any(os.path.exists(f"{v}/x{i}{e}") for i in (1, 2) for e in EXTS)
    q = _run(_shared(dv, 2, refg=False) + ["--target_bcf", f"{dv}/t", "--reference_bcf", f"{dv}/r", "-o", f"{v}/ok_single"])
    assert q.returncode == 0 and _files(f"{v}/ok") == _files(f"{v}/ok_single")


# ---- 7. the stale cache ----------------------------------------------------------------------------------------------------------
def test_stale_cache_bam_line(golden_dir, tmp_path):
    d, *_ = golden_dir
    t = tmp_path
    mat = os.path.join(GOLDEN, "bambam_R3.colate_mat")
    # the cache of age 0 on a line of target age 500: not what the inputs give, but the line must use it, as the single-pair run does
    cached = open(mat).read()
    for o in ("c", "c_single"):
        shutil.copy(mat, f"{t}/{o}.colate_mat")
        os.utime(f"{t}/{o}.colate_mat", (1e9, 1e9))
    lines = [f"target_bam={d}/t.bam reference_bam={d}/r.bam {t}/c target_age=500", f"target_bam={d}/r.bam reference_bam={d}/t.bam {t}/live"]
    (t / "pairs.txt").write_text("".join(x + "\n" for x in lines))
    r = _run(_shared(d, 3) + ["--pairs", str(t / "pairs.txt")])
    assert r.returncode == 0, r.stderr[-3000:]
    assert f"from {t}/c.colate_mat" in r.stderr
    q = _run(_shared(d, 3) + ["--target_bam", f"{d}/t.bam", "--reference_bam", f"{d}/r.bam", "--target_age", "500", "-o", f"{t}/c_single"])
    assert q.returncode == 0, q.stderr[-3000:]
    assert _files(f"{t}/c") == _files(f"{t}/c_single")
    assert open(f"{t}/c.colate_mat").read() == cached and os.path.getmtime(f"{t}/c.colate_mat") == 1e9


# ---- 8. pairs.cohort(front_ends=...) -----------------------------------------------------------------------------------------------
def test_python_cohort_front_ends_equal_api_mut(vcf_dir, handle):
    d, z, sites, genome = vcf_dir
    R = 2
    paths = {p: [os.path.join(d, f"{p}_chr{nm}.bcf") for nm in sites.chr_names] for p in ("t", "r", "tv")}
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    for s in range(8):
        handle.set_mask(s, None)
    handle.set_ref_genome(genome)
    try:
        handle.rows_from_bcf_roles(2, 3, paths["t"], 1)          # t as target (2) and as reference (3)
        handle.rows_from_bcf_roles(4, 5, paths["r"], 1)
        handle.rows_from_bcf_roles(6, -1, paths["tv"], 1)
        plist = [(2, 5, None, None), (4, 3, "1000", None), (6, 5, None, "300")]
        res = pairs.cohort(handle, plist, seed=23, bins="3,7,0.2", num_bootstraps=R, front_ends=[1, 1, 1])
        for (ts, rs, ta, ra), got in zip(plist, res["pairs"]):
            handle.copy_genome(0, ts)
            handle.copy_genome(1, rs)
            handle.set_option("front_end", 1)
            try:
                want = api.mut(handle, seed=23, bins="3,7,0.2", num_bootstraps=R, target_age=ta, reference_age=ra)
            finally:
                handle.set_option("front_end", 0)
            assert np.array_equal(got["rates"].view(np.int64), want["rates"].view(np.int64))
            assert np.array_equal(got["iters"], want["iters"]) and np.array_equal(got["counts"], want["counts"])
            assert got["num_blocks"] == want["num_blocks"]
        # without front_ends the option is left alone: front_end 0 gives other counts on the same slots
        plain = pairs.cohort(handle, plist[:1], seed=23, bins="3,7,0.2", num_bootstraps=R)
        assert not np.array_equal(plain["pairs"][0]["counts"], res["pairs"][0]["counts"])
        with pytest.raises(ValueError):
            pairs.cohort(handle, plist, seed=23, bins="3,7,0.2", front_ends=[1, 1])
    finally:
        handle.set_option("front_end", 0)
        handle.set_ref_genome([])
