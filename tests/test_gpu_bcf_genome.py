"""GPU: whole-genome BCF / VCF files (colate_rows_from_bcf_genome, colate_maketmp_write_bcf_genome, and the CLI wherever
--target_bcf / --reference_bcf are read).  Chromosome c of a whole-genome file is the per-chromosome file holding exactly contig c's
records, so every result must equal the run on the split twins written from the same record lists: rows bit for bit (per role, both
roles, chunk sizes from one record to the whole file, without a genome and with the resident one), stage i against the reference
(stage1_vcfvcf.npz), a haploid contig beside diploid ones, the CLI's files byte for byte (mode mut, make_tmp, --targets, --pairs,
each file decoded once), and refused files failing only their own lines."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from colate_b200 import _lib, api, synth

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
from bcf_helpers import random_records  # noqa: E402
from genome_files import decoys, genome_layout, write_genome, write_split  # noqa: E402
from helpers import bambam_masks, load, sites_from, vcfvcf_counts  # noqa: E402
from test_gpu_bcf import _fixture_recs  # noqa: E402

CLI = os.path.join(os.path.dirname(HERE), "colate_b200", "bin", "Colate")
pytestmark = pytest.mark.gpu
EXTS = (".coal", ".bin", ".colate_mat")
SUMMARY = re.compile(r"BCF/VCF files decoded (\d+)")


@pytest.fixture(scope="module")
def gdir(tmp_path_factory, built):
    """The vcfvcf fixture: split twins t / r (BCF), tv / rv (VCF), and whole-genome files tg.bcf (contigs chr<c>, IDX=),
    rg.bcf (contigs <c>), tvg.vcf.gz / rvg.vcf.gz (chr<c> / <c>), each with the listed contigs reversed against --chr and
    unlisted contigs before, between and after them."""
    z = load("stage1_vcfvcf.npz")
    sites = sites_from(z)
    names = list(sites.chr_names)
    d = str(tmp_path_factory.mktemp("bcf_genome"))
    synth.write_dataset(d, sites, {})
    rng = np.random.default_rng(17)
    for tag, ns in (("t", int(z["n_hap_target"]) // 2), ("r", int(z["n_hap_ref"]) // 2)):
        recs = [_fixture_recs(z, tag, c) for c in range(len(names))]
        write_split(os.path.join(d, tag), "bcf", ns, names, recs, block_size=20000)
        write_split(os.path.join(d, tag + "v"), "vcf", ns, names, recs, block_size=3001)
        chr_prefix = tag == "t"
        contigs = genome_layout(rng, names, recs, ns, prefix_chr=chr_prefix)
        cidx = {nm: 3 * k + 2 for k, (nm, _, _) in enumerate(contigs)} if tag == "t" else None
        write_genome(os.path.join(d, f"{tag}g.bcf"), "bcf", ns, contigs, contig_idx=cidx, block_size=20000)
        contigs = genome_layout(rng, names, recs, ns, prefix_chr=not chr_prefix)
        write_genome(os.path.join(d, f"{tag}vg.vcf.gz"), "vcf", ns, contigs, block_size=3001)
    genome = []
    for c, nm in enumerate(names):
        lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
        g = np.full(int(sites.pos[lo:hi].max()) + 10, ord("n"), np.uint8)
        g[sites.pos[lo:hi] - 1] = z["refg_at_rows"][lo:hi]
        g[sites.pos[lo:hi:2] - 1] += 32
        genome.append(g)
        with open(os.path.join(d, f"g_chr{nm}.fa"), "wb") as f:
            f.write(b">ref\n" + g.tobytes() + b"\n")
    return d, z, sites, genome


def _slot_rows(handle, slot):
    p4 = np.zeros((handle.n_site, 4), np.int32)
    _lib.check(_lib.lib().colate_pileup_end(handle._h, slot, p4.ctypes.data_as(C.c_void_p)))
    return p4[:, 0].copy(), p4[:, 1].copy()


def _genome_equals_split(handle, split_paths, whole, names, genome, chunks=(0,)):
    """rows_from_bcf_genome (both roles, and each alone) equals rows_from_bcf on the split files, without a genome and with the
    resident one, bit for bit."""
    for gm in (0, 1):
        host = genome if gm else None
        want = [handle.rows_from_bcf(2, split_paths, "target", host, fetch=True), handle.rows_from_bcf(3, split_paths, "reference", host, fetch=True)]
        if gm:
            handle.set_ref_genome(genome)
        for chunk in chunks:
            handle.rows_from_bcf_genome(0, 1, whole, names, gm, chunk)
            for slot in (0, 1):
                got = _slot_rows(handle, slot)
                assert np.array_equal(got[0], want[slot][0]) and np.array_equal(got[1], want[slot][1]), (whole, gm, chunk, slot)
        handle.rows_from_bcf_genome(4, -1, whole, names, gm)
        handle.rows_from_bcf_genome(-1, 5, whole, names, gm)
        for slot, w in ((4, want[0]), (5, want[1])):
            got = _slot_rows(handle, slot)
            assert np.array_equal(got[0], w[0]) and np.array_equal(got[1], w[1]), (whole, gm, slot)
    handle.set_ref_genome([])


@pytest.mark.parametrize("split, whole", [("t", "tg.bcf"), ("r", "rg.bcf"), ("tv", "tvg.vcf.gz"), ("rv", "rvg.vcf.gz")])
def test_rows_equal_the_split_files_on_the_fixture(gdir, handle, split, whole):
    d, z, sites, genome = gdir
    names = list(sites.chr_names)
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    _genome_equals_split(handle, [os.path.join(d, f"{split}_chr{nm}.bcf") for nm in names], os.path.join(d, whole), names, genome,
                         chunks=(1, 777, 65536, 0))
    assert handle.last_bcf_timing()["records"] > 0


@pytest.mark.parametrize("tag", ["plain", "refg", "refg_masked"])
def test_stage1_on_whole_genome_files_matches_reference_parse_vcfvcf(gdir, handle, tag):
    d, z, sites, genome = gdir
    names = list(sites.chr_names)
    tm, rm = bambam_masks(z) if tag == "refg_masked" else (None, None)
    handle.set_option("front_end", 1)
    try:
        handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
        gm = 0 if tag == "plain" else 1
        if gm:
            handle.set_ref_genome(genome)
        handle.rows_from_bcf_genome(0, -1, os.path.join(d, "tvg.vcf.gz"), names, gm)
        handle.rows_from_bcf_genome(-1, 1, os.path.join(d, "rg.bcf"), names, gm)
        handle.set_mask(0, None if tm is None else api.mask_bits_from_seq(tm, sites.site_off, sites.pos))
        handle.set_mask(1, None if rm is None else api.mask_bits_from_seq(rm, sites.site_off, sites.pos))
        s1 = handle.stage1(api.mt_seed(int(z["seed"])))
        assert s1.num_blocks == int(z[f"ref_{tag}_num_blocks"])
        for v, k in enumerate(("shared", "notshared", "shared_emp", "notshared_emp")):
            assert np.array_equal(s1.block_stats[:, v], z[f"ref_{tag}_{k}"]), k
        _, tc, rc = vcfvcf_counts(z, tag != "plain")
        handle.set_row_counts(0, tc[:, 0], tc[:, 1])
        handle.set_row_counts(1, rc[:, 0], rc[:, 1])
        s2 = handle.stage1(api.mt_seed(int(z["seed"])))
        assert np.array_equal(s1.mt_state, s2.mt_state) and np.array_equal(s1.block_tallies, s2.block_tallies) and s1.n_used == s2.n_used
    finally:
        handle.set_option("front_end", 0)
        handle.set_mask(0, None); handle.set_mask(1, None)
        handle.set_ref_genome([])


def test_random_streams_and_a_haploid_contig(handle, tmp_path):
    """Repeated positions and one-allele records; contig 3 haploid next to diploid autosomes (its own GT length)."""
    rng = np.random.default_rng(23)
    lens = [60000, 40000, 30000]
    names = ["1", "2", "X"]
    sites = synth.make_sites(24, [3000, 2000, 1500], lens, chr_names=names)
    genome = [np.frombuffer(b"ACGTacgtN", np.uint8)[rng.integers(0, 9, L)].copy() for L in lens]
    letters = [b"A", b"C", b"G", b"T"]

    def alleles(r, k):
        return [letters[int(x)] for x in r.permutation(4)[:int(r.choice([1, 2, 2, 3]))]]
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    ploidy = [2, 2, 1]
    for n_sample in (1, 4):
        recs = []
        for c in range(3):
            _, r = random_records(rng, 12000 if c == 0 else 6000, n_sample, ploidy=ploidy[c], pos_step=(0, 3), alleles=alleles, extras=False)
            assert any(r[i][0] == r[i + 1][0] for i in range(len(r) - 1)) and any(len(x[1]) == 1 for x in r)
            recs.append(r)
        for fmt in ("bcf", "vcf"):
            prefix = str(tmp_path / f"s{n_sample}{fmt}")
            write_split(prefix, fmt, n_sample, names, recs, ploidy_per_chr=ploidy)
            whole = str(tmp_path / f"w{n_sample}.{fmt}")
            write_genome(whole, fmt, n_sample, genome_layout(rng, names, recs, n_sample, ploidy_per_chr=ploidy, prefix_chr=fmt == "bcf",
                                                            order=[1, 2, 0]), block_size=4000)
            _genome_equals_split(handle, [f"{prefix}_chr{nm}.bcf" for nm in names], whole, names, genome, chunks=(0, 3000))
            dec = handle.decode_bcf_genome(whole, names)
            assert [x["n_hap"] for x in dec] == [n_sample * p for p in ploidy]
            for c, nm in enumerate(names):
                one = handle.decode_bcf(f"{prefix}_chr{nm}.bcf")
                for k in ("pos", "a0", "a1", "alt_sum", "biallelic", "n_hap"):
                    assert np.array_equal(dec[c][k], one[k]), (fmt, nm, k)


def _run(args):
    return subprocess.run([CLI] + args, capture_output=True, text=True, timeout=900)


def _files(o):
    return {e: open(o + e, "rb").read() for e in EXTS if os.path.exists(o + e)}


def _mut(d, t, r, o, R, refg):
    a = ["--mode", "mut", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--target_bcf", t, "--reference_bcf", r,
         "--bins", "3,7,0.2", "--seed", "23", "--num_bootstraps", str(R), "-o", o]
    return a + (["--ref_genome", os.path.join(d, "g")] if refg else [])


@pytest.mark.parametrize("R, refg", [(1, False), (3, False), (1, True), (3, True)])
def test_cli_mut_equals_the_split_run(gdir, tmp_path, R, refg):
    d, z, sites, genome = gdir
    j = lambda x: os.path.join(d, x)  # noqa: E731
    base = str(tmp_path / "split")
    p = _run(_mut(d, j("t"), j("r"), base, R, refg))
    assert p.returncode == 0, p.stderr[-3000:]
    want = _files(base)
    assert set(want) == set(EXTS)
    for k, (t, r) in enumerate(((j("tg.bcf"), j("rvg.vcf.gz")), (j("tvg.vcf.gz"), j("r")), (j("t"), j("rg.bcf")))):
        o = str(tmp_path / f"w{k}")
        p = _run(_mut(d, t, r, o, R, refg))
        assert p.returncode == 0, p.stderr[-3000:]
        assert _files(o) == want, (t, r)


@pytest.mark.parametrize("tag", ["plain", "masked"])
def test_cli_make_tmp_whole_genome_matches_reference_cli(built, tmp_path, tag):
    import make_golden
    z = load("maketmp_vcf.npz")
    d = str(tmp_path)
    sites, recs, n_hap = make_golden.maketmp_vcf_inputs(d)
    names = list(sites.chr_names)
    rng = np.random.default_rng(4)
    for fmt, f in (("bcf", "w.bcf"), ("vcf", "w.vcf.gz")):
        write_genome(os.path.join(d, f), fmt, n_hap // 2, genome_layout(rng, names, recs, n_hap // 2, prefix_chr=fmt == "vcf"), block_size=3000)
        o = str(tmp_path / f"mk_{fmt}")
        cmd = [CLI, "--mode", "make_tmp", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--target_bcf", os.path.join(d, f),
               "--ref_genome", os.path.join(d, "g"), "-o", o]
        if tag == "masked":
            cmd += ["--target_mask", os.path.join(d, "tm")]
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-3000:]
        assert open(o + ".colate.in", "rb").read() == z[tag].tobytes(), fmt


def test_targets_and_pairs_lines_equal_split_runs(gdir, tmp_path):
    d, z, sites, genome = gdir
    names = list(sites.chr_names)
    t = tmp_path
    tm, _ = bambam_masks(z)
    for c, nm in enumerate(names):
        synth.write_mask(str(t / f"tm_chr{nm}.fa"), tm[c])
    # --targets: whole-genome lines and their split twins
    tg = t / "targets.txt"
    tg.write_text(f"target_bcf={d}/tg.bcf {t}/a\ntarget_bcf={d}/t {t}/a_split\n"
                  f"target_bcf={d}/rvg.vcf.gz {t}/b target_mask={t}/tm\ntarget_bcf={d}/rv {t}/b_split target_mask={t}/tm\n")
    r = _run(["--mode", "make_tmp", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--ref_genome", os.path.join(d, "g"),
              "--targets", str(tg)])
    assert r.returncode == 0, r.stderr[-3000:]
    for o in ("a", "b"):
        assert open(t / f"{o}.colate.in", "rb").read() == open(t / f"{o}_split.colate.in", "rb").read(), o
    # --pairs: a whole-genome file in both roles and beside a split prefix, decoded once each
    lines = [f"target_bcf={d}/tg.bcf reference_bcf={d}/rvg.vcf.gz {t}/p1", f"target_bcf={d}/rvg.vcf.gz reference_bcf={d}/tg.bcf {t}/p2",
             f"target_bcf={d}/tg.bcf reference_bcf={d}/r {t}/p3 target_mask={t}/tm"]
    twins = [f"target_bcf={d}/t reference_bcf={d}/rv {t}/q1", f"target_bcf={d}/rv reference_bcf={d}/t {t}/q2",
             f"target_bcf={d}/t reference_bcf={d}/r {t}/q3 target_mask={t}/tm"]
    shared = ["--mode", "mut", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--bins", "3,7,0.2", "--seed", "23",
              "--num_bootstraps", "2", "--ref_genome", os.path.join(d, "g")]
    for tag, ls in (("whole", lines), ("split", twins)):
        pf = t / f"pairs_{tag}.txt"
        pf.write_text("".join(x + "\n" for x in ls))
        r = _run(shared + ["--pairs", str(pf)])
        assert r.returncode == 0, r.stderr[-3000:]
        n = [int(x) for x in SUMMARY.findall(r.stderr)]
        # whole: tg.bcf and rvg.vcf.gz once each, r split into its files; split: t, rv, r file by file
        assert n == ([2 + len(names)] if tag == "whole" else [3 * len(names)]), r.stderr
    for k in (1, 2, 3):
        got, want = _files(f"{t}/p{k}"), _files(f"{t}/q{k}")
        assert set(got) == set(EXTS) and got == want, k


def test_refused_files_fail_only_their_lines(gdir, tmp_path):
    d, z, sites, genome = gdir
    names = list(sites.chr_names)
    t = tmp_path
    rng = np.random.default_rng(8)
    ns = int(z["n_hap_target"]) // 2
    recs = [_fixture_recs(z, "t", c) for c in range(len(names))]
    h = len(recs[0]) // 2
    bad = {"split_run": [(names[0], recs[0][:h], 2), (names[1], recs[1], 2), (names[0], recs[0][h:], 2)],
           "missing": [(names[0], recs[0], 2), ("decoy", decoys(rng, ns, 2), 2)],
           "ambiguous": [(names[0], recs[0], 2), ("chr" + names[0], recs[0], 2), (names[1], recs[1], 2)]}
    for k, contigs in bad.items():
        write_genome(str(t / f"{k}.bcf"), "bcf", ns, contigs)
    tg = t / "targets.txt"
    tg.write_text("".join(f"target_bcf={t}/{k}.bcf {t}/x_{k}\n" for k in bad) + f"target_bcf={d}/tg.bcf {t}/ok\n")
    for k in bad:
        open(f"{t}/x_{k}.colate.in", "wb").write(b"stale")
    r = _run(["--mode", "make_tmp", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--ref_genome", os.path.join(d, "g"),
              "--targets", str(tg)])
    assert r.returncode == 1, r.stderr[-3000:]
    assert "3 of 4 targets failed" in r.stderr and "not contiguous" in r.stderr and "without records of contig" in r.stderr
    assert "appears in the BCF file as both" in r.stderr, r.stderr[-3000:]
    assert not any(os.path.exists(f"{t}/x_{k}.colate.in") for k in bad) and os.path.exists(f"{t}/ok.colate.in")
    pf = t / "pairs.txt"
    pf.write_text("".join(f"target_bcf={t}/{k}.bcf reference_bcf={d}/r {t}/y_{k}\n" for k in bad) + f"target_bcf={d}/tg.bcf reference_bcf={d}/r {t}/ok\n")
    r = _run(["--mode", "mut", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--bins", "3,7,0.2", "--seed", "23",
              "--pairs", str(pf)])
    assert r.returncode == 1 and "3 of 4 pairs failed" in r.stderr, r.stderr[-3000:]
    assert not any(os.path.exists(f"{t}/y_{k}{e}") for k in bad for e in EXTS)
    r = _run(_mut(d, f"{t}/split_run.bcf", f"{d}/r", f"{t}/z", 1, False))
    assert r.returncode != 0 and "not contiguous" in r.stderr and not any(os.path.exists(f"{t}/z{e}") for e in EXTS)


def test_device_errors_name_the_chromosome(handle, tmp_path):
    """A bad GT in the second listed contig: the message of the per-chromosome file, prefixed with its chromosome."""
    rng = np.random.default_rng(12)
    lens = [20000, 20000]
    names = ["1", "2"]
    sites = synth.make_sites(3, [500, 500], lens, chr_names=names)
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    recs = [[(p, [b"A", b"C"], [0, 1]) for p in range(10, 2000, 7)] for _ in names]
    recs[1][5] = (recs[1][5][0], [b"A", b"C"], [0, -1])
    write_genome(str(tmp_path / "w.vcf.gz"), "vcf", 1, [("1", recs[0], 2), ("2", recs[1], 2)])
    write_split(str(tmp_path / "s"), "vcf", 1, names, recs)
    with pytest.raises(_lib.ColateError) as e:
        handle.rows_from_bcf_genome(0, 1, str(tmp_path / "w.vcf.gz"), names)
    with pytest.raises(_lib.ColateError) as f:
        handle.rows_from_bcf(0, [str(tmp_path / f"s_chr{nm}.bcf") for nm in names], "target")
    msg = str(e.value).split(": ", 1)[1]
    assert msg.startswith("chromosome 2: ") and "VCF line with a missing allele ('.') in a GT" in msg, msg
    # (rows_from_bcf names the chromosomes of its files by index, so its prefix reads "chromosome 1: ")
    assert "VCF line with a missing allele ('.') in a GT" in str(f.value) and "s_chr2.bcf" in str(f.value)
