"""Bgzipped text VCF read wherever BCF is (colate_rows_from_bcf / colate_decode_bcf, `--target_bcf` / `--reference_bcf`): a VCF
line must decode to the record the BCF of the same record gives, bit for bit, so everything downstream is the pinned BCF path.
The fixtures' records written as VCF text reproduce the reference's results (stage1_vcfvcf.npz, maketmp_vcf.npz); the CLI gives
the same files for BCF, VCF and mixed inputs; decode_bcf of VCF equals decode_bcf of BCF on shapes the fixtures lack, on both of
k_vcf_decode's paths; the device refusals name the first bad line; stage i on ~2 M records equals the BCF path."""
import os
import subprocess
import sys

import numpy as np
import pytest

from colate_b200 import _lib, api, synth

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
from bcf_helpers import IDS, keys_of  # noqa: E402
from helpers import bambam_masks, load, sites_from  # noqa: E402
from test_gpu_bcf import _fixture_recs, _write_records  # noqa: E402

CLI = os.path.join(os.path.dirname(HERE), "colate_b200", "bin", "Colate")
pytestmark = pytest.mark.gpu
GT_KEY = keys_of(None)["GT"]
VCF_IDS = [("INFO", "DP"), ("FORMAT", "GQ"), ("FORMAT", "GT"), ("FORMAT", "AD")]


def _write_vcf_records(path, n_sample, ploidy, recs, block_size=65280):
    """(pos0, alleles, allele index per haplotype) records as VCF text: REF, ALT ('.' for a one-allele record), unphased GT."""
    lines = [synth.vcf_line("1", p0, list(al), np.asarray(gt).reshape(n_sample, ploidy).tolist(), info=b"DP=7") for p0, al, gt in recs]
    synth.write_vcf(str(path), synth.vcf_header(n_sample, VCF_IDS), lines, block_size=block_size)


@pytest.fixture(scope="module")
def vcf_dir(tmp_path_factory, built):
    """The layout of test_gpu_bcf.py's vcfvcf_dir with every genome written twice: t / r as BCF, tv / rv as VCF text (both named
    <prefix>_chr<c>.bcf, as the reference opens them)."""
    z = load("stage1_vcfvcf.npz")
    sites = sites_from(z)
    d = str(tmp_path_factory.mktemp("vcfvcf_text"))
    synth.write_dataset(d, sites, {})
    genome = []
    for c, nm in enumerate(sites.chr_names):
        for tag, ns in (("t", int(z["n_hap_target"]) // 2), ("r", int(z["n_hap_ref"]) // 2)):
            recs = _fixture_recs(z, tag, c)
            _write_records(os.path.join(d, f"{tag}_chr{nm}.bcf"), ns, 2, recs, block_size=20000 if tag == "t" else 65280)
            _write_vcf_records(os.path.join(d, f"{tag}v_chr{nm}.bcf"), ns, 2, recs, block_size=3001 if tag == "t" else 65280)
        lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
        g = np.full(int(sites.pos[lo:hi].max()) + 10, ord("n"), np.uint8)
        g[sites.pos[lo:hi] - 1] = z["refg_at_rows"][lo:hi]
        g[sites.pos[lo:hi:2] - 1] += 32
        genome.append(g)
        with open(os.path.join(d, f"g_chr{nm}.fa"), "wb") as f:
            f.write(b">ref\n" + g.tobytes() + b"\n")
    return d, z, sites, genome


def test_fixture_has_one_allele_records_as_alt_dot(vcf_dir):
    d, z, sites, _ = vcf_dir
    n1 = sum(int((z[f"t{c}_nal"] == 1).sum()) for c in range(len(sites.chr_names)))
    assert n1 > 0
    import gzip
    text = b"".join(gzip.decompress(open(os.path.join(d, f"tv_chr{nm}.bcf"), "rb").read()) for nm in sites.chr_names)
    assert sum(1 for ln in text.split(b"\n") if ln and not ln.startswith(b"#") and ln.split(b"\t")[4] == b".") == n1


@pytest.mark.parametrize("tag", ["plain", "refg", "refg_masked"])
def test_rows_from_vcf_then_stage1_matches_reference_parse_vcfvcf(vcf_dir, handle, tag):
    d, z, sites, genome = vcf_dir
    refg = genome if tag != "plain" else None
    tm, rm = bambam_masks(z) if tag == "refg_masked" else (None, None)
    handle.set_option("front_end", 1)
    try:
        handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
        rows = {}
        for kind in ("", "v"):
            for slot, (t, role) in enumerate((("t", "target"), ("r", "reference"))):
                rows[kind, slot] = handle.rows_from_bcf(slot, [os.path.join(d, f"{t}{kind}_chr{nm}.bcf") for nm in sites.chr_names], role, refg,
                                                        fetch=True)
        for slot in (0, 1):
            assert np.array_equal(rows["", slot][0], rows["v", slot][0]) and np.array_equal(rows["", slot][1], rows["v", slot][1])
        handle.set_mask(0, None if tm is None else api.mask_bits_from_seq(tm, sites.site_off, sites.pos))
        handle.set_mask(1, None if rm is None else api.mask_bits_from_seq(rm, sites.site_off, sites.pos))
        s1 = handle.stage1(api.mt_seed(int(z["seed"])))        # the slots hold the VCF genomes
        assert s1.num_blocks == int(z[f"ref_{tag}_num_blocks"])
        for v, k in enumerate(("shared", "notshared", "shared_emp", "notshared_emp")):
            assert np.array_equal(s1.block_stats[:, v], z[f"ref_{tag}_{k}"]), k
    finally:
        handle.set_option("front_end", 0)
        handle.set_mask(0, None); handle.set_mask(1, None)


@pytest.mark.parametrize("R, refg", [(1, False), (3, False), (1, True), (3, True)])
def test_cli_mut_same_files_for_bcf_vcf_and_mixed_inputs(vcf_dir, tmp_path, R, refg):
    d, z, sites, genome = vcf_dir
    out = {}
    for t, r in (("t", "r"), ("tv", "rv"), ("t", "rv"), ("tv", "r")):
        o = str(tmp_path / f"o_{t}_{r}")
        cmd = [CLI, "--mode", "mut", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--target_bcf", os.path.join(d, t),
               "--reference_bcf", os.path.join(d, r), "--bins", "3,7,0.2", "--seed", "23", "--num_bootstraps", str(R), "-o", o]
        if refg:
            cmd += ["--ref_genome", os.path.join(d, "g")]
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-3000:]
        out[t, r] = {ext: open(o + ext, "rb").read() for ext in (".coal", ".colate_mat", ".bin")}
    for k in out:
        assert out[k] == out["t", "r"], k


@pytest.mark.parametrize("tag", ["plain", "masked"])
def test_cli_make_tmp_vcf_matches_reference_cli(built, tmp_path, tag):
    import make_golden
    z = load("maketmp_vcf.npz")
    d = str(tmp_path)
    sites, recs, n_hap = make_golden.maketmp_vcf_inputs(d)
    for c, nm in enumerate(sites.chr_names):
        _write_vcf_records(os.path.join(d, f"tv_chr{nm}.bcf"), n_hap // 2, 2, recs[c], block_size=3000)
    o = str(tmp_path / "mk")
    cmd = [CLI, "--mode", "make_tmp", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--target_bcf", os.path.join(d, "tv"),
           "--ref_genome", os.path.join(d, "g"), "-o", o]
    if tag == "masked":
        cmd += ["--target_mask", os.path.join(d, "tm")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    assert open(o + ".colate.in", "rb").read() == z[tag].tobytes()


# ---- decode equivalence with the BCF of the same records ---------------------------------------------------------------------------
def _random_pair(rng, n, n_sample, ploidy, max_index=3, gt_first=True, seps="mixed", trim=False, extras=True, pos_step=(0, 3),
                 long_info=0):
    """The same n records as BCF records (GT only) and as VCF lines with the given shape.  seps: "phased", "unphased" or "mixed"
    (per separator); max_index: the records' largest allele index (their ALT lists grow to match); trim: samples drop the subfields
    after GT at random."""
    bcf, vcf = [], []
    p = int(rng.integers(0, 100))
    letters = [b"A", b"C", b"G", b"T"]
    for r in range(n):
        p += int(rng.integers(*pos_step))
        if max_index > 3 and rng.random() < 0.5:
            na = int(rng.integers(2, max_index + 2))
            al = [b"A"] + [b"<A%d>" % i for i in range(1, na)]
        else:
            na = int(rng.choice([1, 2, 2, 2, 3, 4]))
            al = [letters[int(x)] for x in rng.permutation(4)[:na]]
            if rng.random() < 0.15:
                al[-1] = rng.choice([b"ACGT", b"<DEL>", b"*", b"GATTACA" * 3])
            if rng.random() < 0.05:
                al[0] = b"GG"
        gt = rng.integers(0, na, (n_sample, ploidy))
        if na > 1 and rng.random() < 0.5:
            gt = np.minimum(gt, 1)
        if seps == "mixed":
            sep = rng.random((n_sample, max(ploidy - 1, 1))) < 0.5
        else:
            sep = np.full((n_sample, max(ploidy - 1, 1)), seps == "phased")
        gtxt = [b"".join((b"" if j == 0 else (b"|" if sep[s, j - 1] else b"/")) + b"%d" % gt[s, j] for j in range(ploidy)) for s in range(n_sample)]
        before = [] if gt_first else [("GQ", [b"%d" % x for x in rng.integers(0, 99, n_sample)])]
        after = [("AD", [b"%d,%d" % tuple(x) for x in rng.integers(0, 50, (n_sample, 2))])] if extras else []
        keep = None
        if trim and after:
            keep = [len(before) + 1 + int(rng.random() < 0.5) for _ in range(n_sample)]
        info = b"."
        if extras:
            info = b"DP=%d;AF=0.%d" % (r, r % 97) + (b";DB" if r % 3 == 0 else b"")
        if long_info and r % 7 == 3:
            info = b"ANN=" + b"x|y," * (long_info // 4)
        rid = b"rs%d" % r * int(rng.choice([1, 1, 5, 40])) if extras else b"."
        qual = b"%d.5" % r if extras and r % 2 else b"."
        vcf.append(synth.vcf_line("1", p, al, None, gt_text=gtxt, rid=rid, qual=qual, filt=b"PASS" if r % 4 else b"q10;s50", info=info,
                                  fmt_before=before, fmt_after=after, keep=keep))
        bcf.append(synth.bcf_record(0, p, al, gt.tolist(), GT_KEY, gt_type=1 if max_index < 60 else 2))
    return bcf, vcf


def _decode_pair(handle, tmp_path, n_sample, bcf, vcf, chunks=(0,), block_size=65280):
    pb, pv = tmp_path / "s.bcf", tmp_path / "s_vcf.bcf"
    synth.write_bcf(str(pb), synth.bcf_header(n_sample, IDS), bcf)
    synth.write_vcf(str(pv), synth.vcf_header(n_sample, VCF_IDS), vcf, block_size=block_size)
    want = handle.decode_bcf(str(pb))
    paths = [0, 0]
    handle.set_option("vcf_paths", 1)
    try:
        for chunk in chunks:
            got = handle.decode_bcf(str(pv), chunk)
            for k in ("pos", "a0", "a1", "alt_sum", "biallelic", "n_hap"):
                assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), (k, chunk)
            f, g = handle.last_vcf_paths()
            assert f + g == len(vcf)
            paths[0] += f
            paths[1] += g
        handle.decode_bcf(str(pb))
        assert handle.last_vcf_paths() == (0, 0)
    finally:
        handle.set_option("vcf_paths", 0)
    got = handle.decode_bcf(str(pv))                                         # without the test option: the same, not counted
    assert handle.last_vcf_paths() == (0, 0) and np.array_equal(got["alt_sum"], want["alt_sum"])
    return want, paths


@pytest.mark.parametrize("n_sample, ploidy, n", [(1, 2, 300), (1, 1, 300), (7, 1, 200), (7, 2, 200), (7, 3, 200), (2504, 2, 60),
                                                 (20000, 2, 12)])
@pytest.mark.parametrize("seps", ["phased", "unphased", "mixed"])
def test_decode_equals_bcf_on_record_shapes(handle, tmp_path, n_sample, ploidy, n, seps):
    rng = np.random.default_rng(n_sample * 10 + ploidy + len(seps))
    gt_first = n_sample != 7 and ploidy != 1
    bcf, vcf = _random_pair(rng, n, n_sample, ploidy, seps=seps, gt_first=gt_first, trim=n_sample < 100)
    want, paths = _decode_pair(handle, tmp_path, n_sample, bcf, vcf, chunks=(1, 777, 65536, 0) if n_sample < 100 else (0, 100000),
                               block_size=int(rng.choice([1000, 65280])))
    assert len(set(want["pos"].tolist())) < n                                  # repeated positions
    if n >= 60:
        assert (want["biallelic"] == 0).any() and (want["biallelic"] == 1).any()
        assert (want["a1"] == 0).any() and (want["a1"] == 0xFF).any()            # ALT '.', and longer ALT alleles
    if gt_first and ploidy == 2:
        assert paths[0] > 0                                                   # GT first, single digits: the fast path
    else:
        assert paths[1] > 0 and paths[0] == 0


@pytest.mark.parametrize("gt_first", [True, False])
def test_allele_indices_to_300(handle, tmp_path, gt_first):
    """Multi-digit indices (the BCF needs int16): never on the fast path, which takes single digits only."""
    rng = np.random.default_rng(300 + gt_first)
    bcf, vcf = _random_pair(rng, 120, 9, 2, max_index=300, gt_first=gt_first, seps="phased", extras=False)
    want, paths = _decode_pair(handle, tmp_path, 9, bcf, vcf, chunks=(1, 0))
    assert want["alt_sum"].max() > 300 * 3 and paths[1] > 0


def test_fast_and_general_paths_give_the_same_bits(handle, tmp_path):
    """2,504 diploid samples, GT first: plain panel lines (fast path) interleaved with lines where one sample holds a two-digit
    index (general strides), a subfield after GT or an unphased call (still the fast shape): each line's record must not depend
    on the path its strides took."""
    rng = np.random.default_rng(77)
    ns = 2504
    bcf, vcf = [], []
    for r in range(60):
        gt = (rng.random((ns, 2)) < 0.1).astype(int)
        al = [b"A", b"C"]
        kind = r % 4
        if kind == 1:
            al = [b"A"] + [b"<A%d>" % i for i in range(1, 13)]
            gt[int(rng.integers(0, ns)), 1] = 12                              # one two-digit index: general stride(s)
        gtxt = [b"%d|%d" % tuple(g) for g in gt]
        if kind == 2:
            s = int(rng.integers(0, ns))
            gtxt[s] += b":5"                                                   # a subfield after GT: still the fast shape
        if kind == 3:
            s = int(rng.integers(0, ns))
            gtxt[s] = b"%d/%d" % tuple(gt[s])
        vcf.append(synth.vcf_line("1", 100 + r, al, None, gt_text=gtxt, fmt=b"GT" if kind != 2 else b"GT:GQ"))
        bcf.append(synth.bcf_record(0, 100 + r, al, gt.tolist(), GT_KEY))
    want, paths = _decode_pair(handle, tmp_path, ns, bcf, vcf, chunks=(0, 50000))
    assert paths[0] > 0 and paths[1] > 0
    assert (want["alt_sum"] > 0).all()


def test_long_info_lines_longer_than_the_window(handle, tmp_path):
    rng = np.random.default_rng(5)
    bcf, vcf = _random_pair(rng, 50, 3, 2, long_info=90000)
    _decode_pair(handle, tmp_path, 3, bcf, vcf, chunks=(1, 777, 65536, 0))


def test_records_straddle_blocks_and_last_line_without_newline(handle, tmp_path):
    rng = np.random.default_rng(6)
    bcf, vcf = _random_pair(rng, 80, 5, 2)
    vcf[-1] = vcf[-1][:-1]
    _decode_pair(handle, tmp_path, 5, bcf, vcf, chunks=(1, 333, 0), block_size=7)


# ---- device refusals --------------------------------------------------------------------------------------------------------------
def _gline(r, gts, fmt=b"GT", cols=None):
    line = synth.vcf_line("1", 10 * r, [b"A", b"C"], None, gt_text=gts, fmt=fmt)
    if cols is not None:
        line = b"\t".join(line.rstrip(b"\n").split(b"\t")[:cols]) + b"\n"
    return line


BAD = {
    "dot": [b"0|1", b".", b"0|0"],
    "dot_dot": [b"0|1", b"./.", b"0|0"],
    "dot_allele": [b"0|1", b"0/.", b"0|0"],
    "mixed_ploidy": [b"0|1", b"1", b"0|0"],
    "ploidy_change": [b"0|1|1", b"0|1|0", b"0|0|0"],
    "few_samples": [b"0|1", b"0|0"],
    "many_samples": [b"0|1", b"0|0", b"1|1", b"1|1"],
    "not_digit": [b"0|1", b"0/a", b"0|0"],
    "double_sep": [b"0|1", b"0//1", b"0|0"],
    "empty_gt": [b"0|1", b"", b"0|0"],
    "plus": [b"0|1", b"+1/0", b"0|0"],
    "trailing_sep": [b"0|1", b"1/", b"0|0"],
    "huge_index": [b"0|1", b"536870913/0", b"0|0"],
}


@pytest.mark.parametrize("case", sorted(BAD) + ["no_gt_in_format", "no_format", "fixed_fields", "trimmed_before_gt"])
def test_device_refusals(handle, tmp_path, case):
    good = [_gline(r, [b"0|1", b"1|0", b"0|0"]) for r in range(40)]
    if case in BAD:
        bad = _gline(20, BAD[case])
    elif case == "no_gt_in_format":
        bad = _gline(20, [b"5", b"6", b"7"], fmt=b"GQ")
    elif case == "no_format":
        bad = _gline(20, [b"0|1"] * 3, cols=8)
    elif case == "fixed_fields":
        bad = _gline(20, [b"0|1"] * 3, cols=6)
    else:
        bad = synth.vcf_line("1", 200, [b"A", b"C"], None, gt_text=[b"0|1"] * 3, fmt_before=[("GQ", [b"5", b"6", b"7"])], keep=[2, 1, 2])
    lines = good[:20] + [bad] + good[20:]
    if case == "ploidy_change":
        good3 = [_gline(r, [b"0|1|1"] * 3) for r in range(40)]
        lines = [_gline(r, [b"0|1"] * 3) for r in range(20)] + good3[20:]             # diploid, then triploid from line 20
    hdr = synth.vcf_header(3, VCF_IDS)
    lines.append(_gline(45, [b".", b".", b"."]))                                        # a later bad line, in a later window
    p = tmp_path / "bad.bcf"
    synth.write_vcf(str(p), hdr, lines, block_size=300)
    at = len(hdr) + sum(len(x) for x in lines[:20])
    for chunk in (1, 0):
        with pytest.raises(_lib.ColateError) as e:
            handle.decode_bcf(str(p), chunk)
        assert e.value.code == -5 and f"inflated byte offset {at}" in str(e.value) and str(p) in str(e.value), str(e.value)


# ---- scale --------------------------------------------------------------------------------------------------------------------------
def test_random_millions_of_vcf_records_then_stage1(handle, tmp_path):
    """~2 M records over two chromosomes, 40 diploid reference samples and one target sample, written as BCF and as VCF text
    from the same arrays: the rows and stage i of the VCF genomes equal those of the BCF genomes bit for bit."""
    rng = np.random.default_rng(15)
    lens = [40_000_000, 25_000_000]
    sites = synth.make_sites(5, [120_000, 80_000], lens)
    genome = [np.frombuffer(b"ACGTacgt", np.uint8)[rng.integers(0, 8, L)].copy() for L in lens]
    paths = {}
    for tag, ns, n_per in (("t", 1, [700_000, 400_000]), ("r", 40, [550_000, 350_000])):
        for c, n in enumerate(n_per):
            lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
            at_rows = sites.pos[lo:hi][rng.random(hi - lo) < 0.8] - 1
            pos0 = np.sort(np.concatenate([at_rows, rng.integers(0, lens[c], n - at_rows.shape[0])])).astype(np.int32)
            m = np.minimum(np.searchsorted(sites.pos[lo:hi], pos0 + 1), hi - lo - 1) + lo
            sw = rng.random(n) < 0.5
            a0 = np.where(sw, sites.der[m], sites.anc[m]).astype(np.uint8)
            a1 = np.where(sw, sites.anc[m], sites.der[m]).astype(np.uint8)
            af = rng.integers(0, 256, (n, 1), dtype=np.uint8)
            allele = (rng.integers(0, 256, (n, 2 * ns), dtype=np.uint8) < af).astype(np.int8)
            allele[rng.random(n) < 0.01, 0] = 2
            phased = rng.random((n, ns)) < 0.5
            gt = ((allele + 1) << 1) | (np.repeat(phased, 2, axis=1) & np.array([False, True] * ns)).astype(np.int8)
            pb, pv = str(tmp_path / f"{tag}_{c}.bcf"), str(tmp_path / f"{tag}v_{c}.bcf")
            synth.write_bcf(pb, synth.bcf_header(ns, IDS), synth.bcf_records_np(pos0, a0, a1, gt.astype(np.int8), GT_KEY), level=1, threads=8)
            synth.write_vcf(pv, synth.vcf_header(ns, VCF_IDS), synth.vcf_lines_np(pos0, a0, a1, allele, phased), level=1, threads=8)
            paths.setdefault(tag, []).append(pb)
            paths.setdefault(tag + "v", []).append(pv)
    handle.set_option("front_end", 1)
    handle.set_option("vcf_paths", 1)
    try:
        handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
        handle.set_mask(0, None); handle.set_mask(1, None)
        s = {}
        for kind in ("", "v"):
            got = []
            for slot, (tag, role) in enumerate((("t", "target"), ("r", "reference"))):
                got.append(handle.rows_from_bcf(slot, paths[tag + kind], role, genome, chunk_bytes=(1 << 22) if kind else 0, fetch=True))
                if kind:
                    assert handle.last_vcf_paths()[0] > 0
            s[kind] = (got, handle.stage1(api.mt_seed(7)))
        (gb, sb), (gv, sv) = s[""], s["v"]
        for slot in (0, 1):
            assert np.array_equal(gb[slot][0], gv[slot][0]) and np.array_equal(gb[slot][1], gv[slot][1])
        assert ((gb[0][0] + gb[0][1] > 0) & (gb[1][1] > 0)).sum() > 50000
        assert sv.num_blocks == sb.num_blocks and sv.n_used == sb.n_used
        assert np.array_equal(sv.block_stats, sb.block_stats) and np.array_equal(sv.block_tallies, sb.block_tallies)
        assert np.array_equal(sv.mt_state, sb.mt_state)
    finally:
        handle.set_option("front_end", 0)
        handle.set_option("vcf_paths", 0)
