"""BCF files read directly (colate_rows_from_bcf / colate_decode_bcf, `--target_bcf` / `--reference_bcf`): the fixtures' genotype
records written into real BGZF BCFs must reproduce what the reference computed from them (stage1_vcfvcf.npz, maketmp_vcf.npz) bit
for bit and byte for byte; the CLI must equal the API run on pre-decoded row counts; the device decode must equal a struct parse on
record shapes the fixtures lack; the device refusals; chunking down to one record per window; stage i on ~2 M records."""
import os
import subprocess
import sys

import numpy as np
import pytest

from colate_b200 import _lib, api, synth
from oracle import pyoracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
from bcf_helpers import IDS, IDX_SHUFFLED, keys_of, py_decode, random_records, resolve_bcf_rows  # noqa: E402
from helpers import bambam_masks, load, sites_from, vcfvcf_counts  # noqa: E402

CLI = os.path.join(os.path.dirname(HERE), "colate_b200", "bin", "Colate")
pytestmark = pytest.mark.gpu


def _write_records(path, n_sample, ploidy, recs, block_size=65280):
    """(pos0, alleles, allele index per haplotype) records as a BCF of n_sample x ploidy haplotypes, GT (a + 1) << 1 (unphased)."""
    gt_key = keys_of(None)["GT"]
    out = [synth.bcf_record(0, p0, list(al), np.asarray(gt).reshape(n_sample, ploidy).tolist(), gt_key, info=[(1, synth.bcf_typed_ints([7]))])
           for p0, al, gt in recs]
    synth.write_bcf(str(path), synth.bcf_header(n_sample, IDS), out, block_size=block_size)


def _fixture_recs(z, tag, c):
    al = z[f"{tag}{c}_al"]
    return [(int(p), [bytes(a) for a in al[i][:int(n)]], [int(g) for g in gt])
            for i, (p, n, gt) in enumerate(zip(z[f"{tag}{c}_pos"], z[f"{tag}{c}_nal"], z[f"{tag}{c}_gt"]))]


@pytest.fixture(scope="module")
def vcfvcf_dir(tmp_path_factory, built):
    z = load("stage1_vcfvcf.npz")
    sites = sites_from(z)
    d = str(tmp_path_factory.mktemp("vcfvcf"))
    synth.write_dataset(d, sites, {})
    genome = []
    for c, nm in enumerate(sites.chr_names):
        for tag, ns in (("t", int(z["n_hap_target"]) // 2), ("r", int(z["n_hap_ref"]) // 2)):
            _write_records(os.path.join(d, f"{tag}_chr{nm}.bcf"), ns, 2, _fixture_recs(z, tag, c), block_size=20000 if tag == "t" else 65280)
        lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
        g = np.full(int(sites.pos[lo:hi].max()) + 10, ord("n"), np.uint8)       # the fixture keeps the reference genome at the rows
        g[sites.pos[lo:hi] - 1] = z["refg_at_rows"][lo:hi]
        g[sites.pos[lo:hi:2] - 1] += 32                                          # soft-masked half: read upper-cased
        genome.append(g)
        with open(os.path.join(d, f"g_chr{nm}.fa"), "wb") as f:
            f.write(b">ref\n" + g.tobytes() + b"\n")
    return d, z, sites, genome


@pytest.mark.parametrize("tag", ["plain", "refg", "refg_masked"])
def test_rows_from_bcf_then_stage1_matches_reference_parse_vcfvcf(vcfvcf_dir, handle, tag):
    d, z, sites, genome = vcfvcf_dir
    refg = genome if tag != "plain" else None
    tm, rm = bambam_masks(z) if tag == "refg_masked" else (None, None)
    paths = {t: [os.path.join(d, f"{t}_chr{nm}.bcf") for nm in sites.chr_names] for t in ("t", "r")}
    handle.set_option("front_end", 1)
    try:
        handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
        handle.rows_from_bcf(0, paths["t"], "target", refg)
        handle.rows_from_bcf(1, paths["r"], "reference", refg)
        handle.set_mask(0, None if tm is None else api.mask_bits_from_seq(tm, sites.site_off, sites.pos))
        handle.set_mask(1, None if rm is None else api.mask_bits_from_seq(rm, sites.site_off, sites.pos))
        s1 = handle.stage1(api.mt_seed(int(z["seed"])))
        assert s1.num_blocks == int(z[f"ref_{tag}_num_blocks"])
        for v, k in enumerate(("shared", "notshared", "shared_emp", "notshared_emp")):
            assert np.array_equal(s1.block_stats[:, v], z[f"ref_{tag}_{k}"]), k
        # generator state and tallies: those of the row-count path, which test_gpu_stage1.py pins to the reference
        _, tc, rc = vcfvcf_counts(z, tag != "plain")
        handle.set_row_counts(0, tc[:, 0], tc[:, 1])
        handle.set_row_counts(1, rc[:, 0], rc[:, 1])
        s2 = handle.stage1(api.mt_seed(int(z["seed"])))
        assert np.array_equal(s1.mt_state, s2.mt_state) and np.array_equal(s1.block_tallies, s2.block_tallies) and s1.n_used == s2.n_used
    finally:
        handle.set_option("front_end", 0)
        handle.set_mask(0, None); handle.set_mask(1, None)


@pytest.mark.parametrize("chunk", [1, 777, 65536, 0])
def test_rows_from_bcf_equal_the_per_genome_restatement(vcfvcf_dir, handle, chunk):
    """Every row's counts per genome, chunk sizes from one record per window to the whole file, with and without --ref_genome."""
    d, z, sites, genome = vcfvcf_dir
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    meta = sites.meta()
    for refg in (None, genome):
        for slot, (t, role, nh) in enumerate((("t", "target", int(z["n_hap_target"])), ("r", "reference", int(z["n_hap_ref"])))):
            aaf, daf = handle.rows_from_bcf(slot, [os.path.join(d, f"{t}_chr{nm}.bcf") for nm in sites.chr_names], role, refg,
                                            chunk_bytes=chunk, fetch=True)
            for c in range(len(sites.chr_names)):
                lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
                usable = ((meta[lo:hi] & 1) != 0) & (sites.anc[lo:hi] != sites.der[lo:hi])
                want = resolve_bcf_rows(role, sites.pos[lo:hi], sites.anc[lo:hi], sites.der[lo:hi], usable, _fixture_recs(z, t, c), nh,
                                        z["refg_at_rows"][lo:hi] if refg is not None else None)
                assert np.array_equal(aaf[lo:hi], want[:, 0]) and np.array_equal(daf[lo:hi], want[:, 1]), (role, c, chunk)
    assert handle.last_bcf_timing()["records"] == sum(len(z[f"r{c}_pos"]) for c in range(len(sites.chr_names)))


@pytest.mark.parametrize("R, refg", [(1, False), (3, False), (1, True), (3, True)])
def test_cli_mut_bcf_bcf_equals_api_on_decoded_row_counts(vcfvcf_dir, handle, tmp_path, R, refg):
    d, z, sites, genome = vcfvcf_dir
    o = str(tmp_path / "o")
    cmd = [CLI, "--mode", "mut", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--target_bcf", os.path.join(d, "t"),
           "--reference_bcf", os.path.join(d, "r"), "--bins", "3,7,0.2", "--seed", "23", "--num_bootstraps", str(R), "-o", o]
    if refg:
        cmd += ["--ref_genome", os.path.join(d, "g")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    # the same run through the API from set_row_counts(decode_vcfvcf(...))
    _, tc, rc = vcfvcf_counts(z, refg)
    handle.set_option("front_end", 1)
    try:
        handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
        handle.set_row_counts(0, tc[:, 0], tc[:, 1])
        handle.set_row_counts(1, rc[:, 0], rc[:, 1])
        handle.set_mask(0, None); handle.set_mask(1, None)
        res = api.mut(handle, seed=23, bins="3,7,0.2", num_bootstraps=R)
    finally:
        handle.set_option("front_end", 0)
    a = str(tmp_path / "a")
    rates = api.write_coal(a + ".coal", res["epochs"], res["rates"], res["is_ancient"], res["ep_null"])
    api.write_bin(a + ".bin", res["epochs"], rates, res["iters"])
    api.write_colate_mat(a + ".colate_mat", res["counts"])
    for ext in (".coal", ".colate_mat", ".bin"):
        assert open(o + ext, "rb").read() == open(a + ext, "rb").read(), ext
    if po.ref_cli():
        # live against the reference CLI, which reads the same records from the fake BCFs of oracle/hts_stubs.c
        for c, nm in enumerate(sites.chr_names):
            for tag, nh in (("t", int(z["n_hap_target"])), ("r", int(z["n_hap_ref"]))):
                po.write_fake_bcf(os.path.join(d, f"f{tag}_chr{nm}.bcf"), nh // 2, 2, _fixture_recs(z, tag, c))
        ref = str(tmp_path / "ref")
        cmd = [po.ref_cli()] + cmd[1:cmd.index("-o")] + ["-o", ref]
        cmd[cmd.index("--target_bcf") + 1] = os.path.join(d, "ft")
        cmd[cmd.index("--reference_bcf") + 1] = os.path.join(d, "fr")
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-3000:]
        for ext in (".coal", ".colate_mat"):
            assert open(o + ext, "rb").read() == open(ref + ext, "rb").read(), ext


@pytest.mark.parametrize("tag", ["plain", "masked"])
def test_cli_make_tmp_bcf_matches_reference_cli(built, tmp_path, tag):
    import make_golden
    z = load("maketmp_vcf.npz")
    d = str(tmp_path)
    sites, recs, n_hap = make_golden.maketmp_vcf_inputs(d)
    for c, nm in enumerate(sites.chr_names):
        _write_records(os.path.join(d, f"tb_chr{nm}.bcf"), n_hap // 2, 2, recs[c], block_size=3000)
    o = str(tmp_path / "mk")
    cmd = [CLI, "--mode", "make_tmp", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--target_bcf", os.path.join(d, "tb"),
           "--ref_genome", os.path.join(d, "g"), "-o", o]
    if tag == "masked":
        cmd += ["--target_mask", os.path.join(d, "tm")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    assert open(o + ".colate.in", "rb").read() == z[tag].tobytes()


def _decode_check(handle, path, chunks=(0,)):
    import gzip
    ns, gt_key, want = py_decode(gzip.decompress(open(path, "rb").read()))
    for chunk in chunks:
        got = handle.decode_bcf(str(path), chunk)
        assert got["n_hap"] == want[0][6]
        for i, k in enumerate(("pos", "a0", "a1", "alt_sum", "biallelic")):
            col = np.array([r[1] + 1 if k == "pos" else r[i + 1] for r in want])         # (chrom, pos, a0, a1, alt_sum, biallelic, n_hap)
            assert np.array_equal(got[k].astype(np.int64), col.astype(np.int64)), (k, chunk)
    return want


@pytest.mark.parametrize("gt_type", [1, 2, 3])
@pytest.mark.parametrize("n_sample, ploidy, n", [(1, 2, 300), (1, 1, 300), (7, 1, 200), (2504, 2, 60), (20000, 2, 12)])
def test_decode_equals_struct_parse_on_record_shapes(handle, tmp_path, gt_type, n_sample, ploidy, n):
    """INFO fields of every type (flags, overflow sizes), FILTER lists, long IDs, multi-letter and symbolic alleles, FORMAT fields
    before and after GT, repeated positions, phased and unphased GT of every integer width, haploid samples."""
    rng = np.random.default_rng(gt_type * 1000 + n_sample + ploidy)
    idx = IDX_SHUFFLED if n_sample % 2 else None
    out, _ = random_records(rng, n, n_sample, ploidy=ploidy, gt_type=gt_type, idx=idx, pos_step=(0, 3))
    p = tmp_path / "s.bcf"
    synth.write_bcf(str(p), synth.bcf_header(n_sample, IDS, idx=idx), out, block_size=int(rng.choice([1000, 65280])))
    want = _decode_check(handle, p, chunks=(1, 5000, 0) if n_sample < 100 else (0, 100000))
    if n >= 60:
        assert any(not r[5] for r in want) and any(r[5] for r in want)
        assert len({r[1] for r in want}) < len(want)                        # repeated positions


def test_phased_bit_is_dropped(handle, tmp_path):
    """All-phased diploid records in one 16-byte-aligned run: the phased bit of one GT byte must not leak into the next."""
    k = keys_of(None)["GT"]
    recs = [synth.bcf_record(0, 10 + r, [b"A", b"C"], [[r % 2, 1]] * 64, k, phased=True) for r in range(50)]
    p = tmp_path / "ph.bcf"
    synth.write_bcf(str(p), synth.bcf_header(64, IDS), recs)
    want = _decode_check(handle, p)
    assert [r[4] for r in want] == [64 * (1 + r % 2) for r in range(50)]


@pytest.mark.parametrize("case", ["missing", "vector_end", "no_gt", "gt_length", "missing_int16", "truncated_info"])
def test_device_refusals(handle, tmp_path, case):
    k = keys_of(None)
    good = [synth.bcf_record(0, 10 * r, [b"A", b"C"], [[0, 1]] * 3, k["GT"]) for r in range(40)]
    if case == "missing":
        bad = synth.bcf_record(0, 200, [b"A", b"C"], [[0, 1], [-1, 1], [0, 0]], k["GT"])
    elif case == "missing_int16":
        bad = synth.bcf_record(0, 200, [b"A", b"C"], [[0, 1]] * 3, k["GT"], gt_type=2, gt_raw=[[2, 4], [synth.GT_MISSING[2], 4], [2, 2]])
    elif case == "vector_end":
        bad = synth.bcf_record(0, 200, [b"A", b"C"], [[0, 1], [0, None], [0, 0]], k["GT"])
    elif case == "no_gt":
        bad = synth.bcf_record(0, 200, [b"A", b"C"], [[0, 1]] * 3, None, fmt_before=[(k["GQ"], 1, [[5]] * 3)])
    elif case == "gt_length":
        bad = synth.bcf_record(0, 200, [b"A", b"C"], [[0, 1, 1]] * 3, k["GT"])
    else:
        bad = bytearray(synth.bcf_record(0, 200, [b"A", b"C"], [[0, 1]] * 3, k["GT"], info=[(k["ANN"], synth.bcf_typed_str(b"x" * 40))]))
        import struct
        l_shared = struct.unpack_from("<I", bad, 0)[0]
        struct.pack_into("<I", bad, 0, l_shared - 20)                       # the INFO string now runs past l_shared
        struct.pack_into("<I", bad, 4, struct.unpack_from("<I", bad, 4)[0] + 20)
        bad = bytes(bad)
    hdr = synth.bcf_header(3, IDS)
    p = tmp_path / "bad.bcf"
    synth.write_bcf(str(p), hdr, good[:20] + [bad] + good[20:], block_size=300)
    at = len(hdr) + sum(len(r) for r in good[:20])
    for chunk in (1, 0):
        with pytest.raises(_lib.ColateError) as e:
            handle.decode_bcf(str(p), chunk)
        assert e.value.code == -5 and f"inflated byte offset {at}" in str(e.value) and str(p) in str(e.value), str(e.value)


def _np_rows(role, pos_rows, anc, der, usable, rpos1, a0, a1, alt, bi, N, refg_rows):
    """Vectorised resolve_bcf_rows on decoded record columns (for millions of records)."""
    n = rpos1.shape[0]
    k = np.searchsorted(rpos1, pos_rows, "left")
    kk = np.minimum(k, n - 1)
    found = (k < n) & (rpos1[kk] == pos_rows)
    A0, A1, S, B = a0[kk].astype(np.int64), a1[kk].astype(np.int64), alt[kk].astype(np.int64), bi[kk].astype(bool)
    anc, der = anc.astype(np.int64), der.astype(np.int64)
    letter = lambda x: (x != 0) & (x != 255)
    two = letter(A0) & letter(A1)
    same, flip = two & (A0 == anc) & (A1 == der), two & (A0 == der) & (A1 == anc)
    daf = np.full(pos_rows.shape[0], -1, np.int64)
    m = found & (same | flip) & B
    daf[m] = np.where(flip, N - S, S)[m]
    if role == "target":
        m = found & ~(same | flip) & (A0 != 0) & (A1 == 0) & letter(A0) & ((A0 == anc) | (A0 == der)) & B & (S == 0)
        daf[m] = np.where(A0 == der, N, 0)[m]
    if refg_rows is not None:
        b = refg_rows.astype(np.int64)
        daf[~found & (b == der)] = N
        if role == "target":
            daf[~found & (b == anc) & (b != der)] = 0
    if role == "reference":
        daf[daf == 0] = -1
    daf[~usable] = -1
    ok = daf >= 0
    return np.where(ok, N - daf, 0).astype(np.int32), np.where(ok, daf, 0).astype(np.int32)


def test_random_millions_of_records_then_stage1(handle, tmp_path):
    """~2 M records over two chromosomes, 150 diploid reference samples and one target sample: stage i on the BCF genomes equals
    stage i on set_row_counts of the same resolution bit for bit."""
    rng = np.random.default_rng(5)
    lens = [40_000_000, 25_000_000]
    sites = synth.make_sites(5, [120_000, 80_000], lens)
    meta = sites.meta()
    usable = ((meta & 1) != 0) & (sites.anc != sites.der)
    genome = [np.frombuffer(b"ACGTacgt", np.uint8)[rng.integers(0, 8, L)].copy() for L in lens]
    paths = {"t": [], "r": []}
    want = {}
    key = keys_of(None)["GT"]
    for tag, ns, n_per in (("t", 1, [700_000, 400_000]), ("r", 150, [550_000, 350_000])):
        cols = []
        for c, n in enumerate(n_per):
            lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
            at_rows = sites.pos[lo:hi][rng.random(hi - lo) < 0.8] - 1
            pos0 = np.sort(np.concatenate([at_rows, rng.integers(0, lens[c], n - at_rows.shape[0])])).astype(np.int32)
            m = np.minimum(np.searchsorted(sites.pos[lo:hi], pos0 + 1), hi - lo - 1) + lo
            sw = rng.random(n) < 0.5
            a0 = np.where(sw, sites.der[m], sites.anc[m]).astype(np.uint8)
            a1 = np.where(sw, sites.anc[m], sites.der[m]).astype(np.uint8)
            noise = rng.random(n) < 0.1
            a1[noise] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(noise.sum()))]
            af = rng.integers(0, 256, (n, 1), dtype=np.uint8)
            allele = (rng.integers(0, 256, (n, 2 * ns), dtype=np.uint8) < af).view(np.int8)
            allele[rng.random(n) < 0.01, 0] = 2
            gt = ((allele + 1) << 1) | (rng.integers(0, 2, (n, 2 * ns), dtype=np.int8) * np.array([0, 1] * ns, np.int8))
            rec = synth.bcf_records_np(pos0, a0, a1, gt.astype(np.int8), key)
            paths[tag].append(str(tmp_path / f"{tag}_{c}.bcf"))
            synth.write_bcf(paths[tag][-1], synth.bcf_header(ns, IDS), rec, level=1, threads=8)
            cols.append((pos0 + 1, a0, a1, allele.astype(np.int64).sum(1), allele.max(1) <= 1, 2 * ns))
        want[tag] = cols
    handle.set_option("front_end", 1)
    try:
        handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
        handle.set_mask(0, None); handle.set_mask(1, None)
        for slot, (tag, role) in enumerate((("t", "target"), ("r", "reference"))):
            aaf = np.zeros(sites.n, np.int32); daf = np.zeros(sites.n, np.int32)
            for c in range(2):
                lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
                rp, a0, a1, alt, bi, N = want[tag][c]
                aaf[lo:hi], daf[lo:hi] = _np_rows(role, sites.pos[lo:hi], sites.anc[lo:hi], sites.der[lo:hi], usable[lo:hi], rp, a0, a1, alt, bi,
                                                  N, genome[c][sites.pos[lo:hi] - 1] & 0xDF)
            want[slot] = (aaf, daf)
            handle.set_row_counts(slot, aaf, daf)
        assert ((want[0][0] + want[0][1] > 0) & (want[1][1] > 0)).sum() > 50000
        s_ref = handle.stage1(api.mt_seed(7))
        for slot, (tag, role) in enumerate((("t", "target"), ("r", "reference"))):
            for chunk in ((1 << 22, 0) if slot == 0 else (0,)):
                got = handle.rows_from_bcf(slot, paths[tag], role, genome, chunk_bytes=chunk, fetch=True)
                assert np.array_equal(got[0], want[slot][0]) and np.array_equal(got[1], want[slot][1]), (tag, chunk)
        s_bcf = handle.stage1(api.mt_seed(7))
        assert s_bcf.num_blocks == s_ref.num_blocks and s_bcf.n_used == s_ref.n_used
        assert np.array_equal(s_bcf.block_stats, s_ref.block_stats) and np.array_equal(s_bcf.block_tallies, s_ref.block_tallies)
        assert np.array_equal(s_bcf.mt_state, s_ref.mt_state)
    finally:
        handle.set_option("front_end", 0)
