"""make_tmp for many targets (`--mode make_tmp --targets`, colate_maketmp_write_pileup / _bcf): the device .colate.in writer must
reproduce the reference CLI's files (stage1_bambam.npz maketmp_bam_*, maketmp_vcf.npz) byte for byte, equal the host writers
(colate_maketmp_pileup / colate_maketmp_records) on the same arrays, build the make_tmp row word on the device as the host reader
does, and a mixed batch must equal single-target runs; failing lines leave no file; the job parses the .mut text and uploads the
reference genome once."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from colate_b200 import _lib, api, synth

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
from helpers import bambam_masks, load  # noqa: E402
from test_gpu_bcf import _write_records  # noqa: E402
from test_gpu_vcf import _write_vcf_records  # noqa: E402
from test_maketmp_batch_host import CASES, _row  # noqa: E402

CLI = os.path.join(os.path.dirname(HERE), "colate_b200", "bin", "Colate")
pytestmark = pytest.mark.gpu


def _cli(*args, env=None):
    return subprocess.run([CLI] + [str(a) for a in args], capture_output=True, text=True, timeout=900, env=env)


def _targets(path, lines):
    with open(path, "w") as f:
        f.write("# batch\n" + "".join(x + "\n" for x in lines))
    return path


def _names(xs):
    return (C.c_char_p * len(xs))(*[x.encode() for x in xs])


# ---- against the reference goldens -------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def bam_golden_dir(tmp_path_factory, built):
    import make_golden
    z = load("stage1_bambam.npz")
    sites, lens, genome, reads_t, _ = make_golden.bambam_inputs(int(z["seed"]))
    d = str(tmp_path_factory.mktemp("mk_bam"))
    synth.write_dataset(d, sites, {})
    for c, L in enumerate(lens):
        with open(os.path.join(d, f"g_chr{sites.chr_names[c]}.fa"), "wb") as f:
            f.write(b">ref\n")
            for i in range(0, L, 1 << 20):
                f.write(genome[c][i:i + (1 << 20)].tobytes() + b"\n")
    reads = [(c, st, mq, 16 if rev else 0, seq, qual, b"r%d" % k, [(len(seq), "M")], b"") for k, (c, st, mq, rev, seq, qual) in enumerate(reads_t)]
    synth.write_bam(os.path.join(d, "t.bam"), ["chr" + sites.chr_names[0], sites.chr_names[1]], reads, contig_lens=lens, block_size=60000)
    tm, _ = bambam_masks(z)
    for c, nm in enumerate(sites.chr_names):
        synth.write_mask(os.path.join(d, f"tm_chr{nm}.fa"), tm[c])
    return d, z


def test_batch_bam_matches_reference_cli(bam_golden_dir, tmp_path):
    d, z = bam_golden_dir
    tf = _targets(tmp_path / "t.txt", [f"target_bam={d}/t.bam {tmp_path}/plain", f"target_bam={d}/t.bam {tmp_path}/masked target_mask={d}/tm"])
    p = _cli("--mode", "make_tmp", "--mut", f"{d}/syn", "--chr", f"{d}/chr.txt", "--ref_genome", f"{d}/g", "--targets", tf)
    assert p.returncode == 0, p.stderr[-3000:]
    for tag in ("plain", "masked"):
        assert open(f"{tmp_path}/{tag}.colate.in", "rb").read() == z["maketmp_bam_" + tag].tobytes(), tag


@pytest.mark.parametrize("fmt", ["bcf", "vcf"])
def test_batch_bcf_vcf_matches_reference_cli(built, tmp_path, fmt):
    import make_golden
    z = load("maketmp_vcf.npz")
    d = str(tmp_path)
    sites, recs, n_hap = make_golden.maketmp_vcf_inputs(d)
    write = _write_records if fmt == "bcf" else _write_vcf_records
    for c, nm in enumerate(sites.chr_names):
        write(os.path.join(d, f"tb_chr{nm}.bcf"), n_hap // 2, 2, recs[c], block_size=3000)
    tf = _targets(tmp_path / "t.txt", [f"target_bcf={d}/tb {d}/plain", f"target_bcf={d}/tb {d}/masked target_mask={d}/tm"])
    p = _cli("--mode", "make_tmp", "--mut", f"{d}/syn", "--chr", f"{d}/chr.txt", "--ref_genome", f"{d}/g", "--targets", tf)
    assert p.returncode == 0, p.stderr[-3000:]
    for tag in ("plain", "masked"):
        assert open(f"{d}/{tag}.colate.in", "rb").read() == z[tag].tobytes(), tag


# ---- the device writer against the host writers --------------------------------------------------------------------------------------
def _dataset(d, seed, rows, names, empty_chr=None):
    """Random .mut files (weird types included); chromosome `empty_chr` keeps its header line only."""
    lens = [int(2e6 + 1e6 * k) for k in range(len(rows))]
    sites = synth.make_sites(seed, rows, lens, chr_names=names, weird=0.15)
    synth.write_dataset(d, sites, {})
    files = [os.path.join(d, f"syn_chr{nm}.mut") for nm in names]
    if empty_chr is not None:
        head = open(files[empty_chr], "rb").read().split(b"\n", 1)[0]
        open(files[empty_chr], "wb").write(head + b"\n")
    return sites, lens, files


def _masks(d, seed, lens, names):
    out = []
    for c, (nm, L) in enumerate(zip(names, lens)):
        m = bytearray(synth.make_mask(seed + c, L if c % 2 else L // 3, 0.3, run_lo=50, run_hi=5000))   # the first one ends early
        rng = np.random.default_rng(seed + c)
        for i in rng.integers(0, len(m), size=len(m) // 50):
            m[i] = b"pNnXA"[int(rng.integers(0, 5))]                                                       # bytes other than 'P'
        path = os.path.join(d, f"m{seed}_chr{nm}.fa")
        synth.write_mask(path, bytes(m))
        out.append(path)
    return out


def _mask_bits(handle, files, site_off):
    pos = handle.ingest_fetch()[0]
    bits = np.zeros(int(site_off[-1]) // 32 + 2, np.uint32)
    for c, f in enumerate(files):
        api.maketmp_mask_bits(f, pos[site_off[c]:site_off[c + 1]], int(site_off[c]), bits)
    return bits


def _ingest(handle, files):
    rows = handle.ingest_mut([open(f, "rb").read() for f in files])
    return np.concatenate([[0], np.cumsum(rows)]).astype(np.int64)


@pytest.mark.parametrize("seed, names, empty", [(3, ["1", "22"], None), (8, ["chrX_long_name", "2", "mt"], 1), (11, [""], None)])
def test_pileup_writer_equals_host_writer(handle, tmp_path, seed, names, empty):
    d = str(tmp_path)
    sites, lens, files = _dataset(d, seed, [3000 + 500 * k for k in range(len(names))], names, empty)
    site_off = _ingest(handle, files)
    n = int(site_off[-1])
    rng = np.random.default_rng(seed)
    counts = (rng.poisson(0.7, (n, 4)) * (rng.random((n, 1)) < 0.6)).astype(np.int32)
    if len(names) > 2:
        counts[site_off[2]:site_off[3]] = 0                              # a chromosome with nothing to write
    handle.set_pileup(0, counts)
    mask_files = _masks(d, seed, lens, names)
    for masked in (False, True):
        mb = _mask_bits(handle, mask_files, site_off) if masked else None
        dev, host = tmp_path / f"dev{masked}.colate.in", tmp_path / f"host{masked}.colate.in"
        nd = handle.maketmp_write_pileup(0, names, dev, mb)
        nh = _lib.check(_lib.lib().colate_maketmp_pileup(len(names), _names(names), _names(files), _lib.ptr(counts), n,
                                                         _names(mask_files) if masked else None, str(host).encode()))
        assert nd == nh and nd > 0
        assert dev.read_bytes() == host.read_bytes(), masked
    assert handle.last_maketmp_timing()["records"] == nd


def _bcf_case(d, seed, fmt):
    import make_golden
    sites, recs, n_hap = make_golden.maketmp_vcf_inputs(d, seed=seed, rows=(1200, 700))
    rng = np.random.default_rng(seed)
    for c, nm in enumerate(sites.chr_names):
        out = []
        for p0, al, gt in recs[c]:
            u = rng.random()
            if u < 0.05:
                al = [al[0], b"T", b"G"] if len(al) > 1 and al[1] else al             # a third allele
                gt = [min(g + (k == 0), 2) for k, g in enumerate(gt)] if len(al) > 2 else gt
            out.append((p0, al, gt))
            if u > 0.97:
                out.append((p0, list(al), gt))                                        # repeated position
        if c == 1:
            out = [r for r in out if r[0] > int(sites.pos[int(sites.site_off[1]) + 30])]   # rows before the first record
        (_write_records if fmt == "bcf" else _write_vcf_records)(os.path.join(d, f"x_chr{nm}.bcf"), n_hap // 2, 2, out, block_size=2500)
    return sites


@pytest.mark.parametrize("seed, fmt", [(5, "bcf"), (77, "vcf"), (31, "bcf")])
def test_bcf_writer_equals_host_writer(handle, tmp_path, seed, fmt):
    d = str(tmp_path)
    sites = _bcf_case(d, seed, fmt)
    names = list(sites.chr_names)
    muts = [os.path.join(d, f"syn_chr{nm}.mut") for nm in names]
    refs = [os.path.join(d, f"g_chr{nm}.fa") for nm in names]
    masks = [os.path.join(d, f"tm_chr{nm}.fa") for nm in names]
    paths = [os.path.join(d, f"x_chr{nm}.bcf") for nm in names]
    site_off = _ingest(handle, muts)
    # the host writer on the decoded arrays
    dec = [handle.decode_bcf(p) for p in paths]
    off = np.concatenate([[0], np.cumsum([len(x["pos"]) for x in dec])]).astype(np.int64)
    cat = {k: np.ascontiguousarray(np.concatenate([x[k] for x in dec])) for k in ("pos", "a0", "a1", "alt_sum", "biallelic")}
    n_hap = np.array([x["n_hap"] for x in dec], np.int32)
    for refg in (False, True):
        handle.set_ref_genome([api.read_fasta(r) for r in refs] if refg else [])
        for masked in (False, True):
            mb = _mask_bits(handle, masks, site_off) if masked else None
            dev, host = tmp_path / f"dev{refg}{masked}.colate.in", tmp_path / f"host{refg}{masked}.colate.in"
            nd = handle.maketmp_write_bcf(paths, names, dev, mb, chunk_bytes=4096)
            nh = _lib.check(_lib.lib().colate_maketmp_records(len(names), _names(names), _names(muts), _lib.ptr(off), _lib.ptr(cat["pos"]),
                                                              _lib.ptr(cat["a0"]), _lib.ptr(cat["a1"]), _lib.ptr(cat["alt_sum"]),
                                                              _lib.ptr(cat["biallelic"]), _lib.ptr(n_hap), _names(refs) if refg else None,
                                                              _names(masks) if masked else None, str(host).encode()))
            assert nd == nh and nd > 0
            assert dev.read_bytes() == host.read_bytes(), (refg, masked)


def test_device_row_word_equals_host_reader(handle, tmp_path):
    d = str(tmp_path)
    names = ["1", "2"]
    _, _, files = _dataset(d, 19, [4000, 2500], names)
    # the hand-made rows of the host test, plus rows the device hands to the host (17 significant digits in an age)
    extra = os.path.join(d, "syn_chr3.mut")
    lines = ["snp;pos;dist;rs;tree;br;nm;fl;ab;ae;type;ACGT;"] + [_row(k, 100 + k, t, fl, br) for k, (t, fl, br, _) in enumerate(CASES)]
    lines.append(_row(50, 400, "A/G").replace("10.5", "10.500000000000000001"))
    open(extra, "w").write("\n".join(lines) + "\n")
    files.append(extra)
    handle.ingest_mut([open(f, "rb").read() for f in files])
    want = np.concatenate([api.read_mut_words(f) for f in files])
    assert np.array_equal(handle.maketmp_words(), want)
    assert handle.ingest_stats()["host_fallback_rows"] >= 1


def test_descending_rows_refused(handle, tmp_path):
    d = str(tmp_path)
    lines = ["snp;pos;dist;rs;tree;br;nm;fl;ab;ae;type;ACGT;", _row(0, 200, "A/G"), _row(1, 100, "C/T")]
    handle.ingest_mut([("\n".join(lines) + "\n").encode()])
    handle.set_pileup(0, np.ones((2, 4), np.int32))
    with pytest.raises(_lib.ColateError) as e:
        handle.maketmp_write_pileup(0, ["1"], tmp_path / "o.colate.in")
    assert e.value.code == -6 and "not ascending" in str(e.value)
    assert not os.path.exists(tmp_path / "o.colate.in")


# ---- the CLI: a mixed batch against single runs, failing lines, work done once -------------------------------------------------------
@pytest.fixture(scope="module")
def mixed_dir(tmp_path_factory, built):
    import make_golden
    d = str(tmp_path_factory.mktemp("mk_mixed"))
    sites, recs, n_hap = make_golden.maketmp_vcf_inputs(d, seed=41, rows=(1500, 900))
    genome = [api.read_fasta(os.path.join(d, f"g_chr{nm}.fa")) for nm in sites.chr_names]
    lens = [g.shape[0] for g in genome]
    for k in range(2):
        reads = make_golden.bambam_reads(np.random.default_rng(100 + k), sites, genome, 0.8, 1.5)
        reads = [(c, st, mq, 16 if rev else 0, seq, qual, b"r%d" % i, [(len(seq), "M")], b"") for i, (c, st, mq, rev, seq, qual) in enumerate(reads)]
        synth.write_bam(os.path.join(d, f"s{k}.bam"), list(sites.chr_names), reads, contig_lens=lens, block_size=30000)
    for c, nm in enumerate(sites.chr_names):
        _write_records(os.path.join(d, f"b_chr{nm}.bcf"), n_hap // 2, 2, recs[c], block_size=3000)
        _write_vcf_records(os.path.join(d, f"v_chr{nm}.bcf"), n_hap // 2, 2, recs[c], block_size=3000)
        synth.write_mask(os.path.join(d, f"m2_chr{nm}.fa"), synth.make_mask(7 + c, lens[c], 0.4, run_lo=100, run_hi=3000))
    return d, sites


MIXED = [("target_bam", "s0", None), ("target_bam", "s1", "tm"), ("target_bcf", "b", None), ("target_bcf", "b", "tm"),
         ("target_bcf", "v", "m2"), ("target_bam", "s0", "m2")]


def test_mixed_batch_equals_single_runs(mixed_dir, tmp_path):
    d, _ = mixed_dir
    shared = ["--mode", "make_tmp", "--mut", f"{d}/syn", "--chr", f"{d}/chr.txt", "--ref_genome", f"{d}/g"]
    lines = []
    for k, (key, src, mask) in enumerate(MIXED):
        inp = f"{d}/{src}.bam" if key == "target_bam" else f"{d}/{src}"
        lines.append(f"{key}={inp} {tmp_path}/b{k}" + (f" target_mask={d}/{mask}" if mask else ""))
    env = dict(os.environ, COLATE_TIMING="1")
    p = _cli(*shared, "--targets", _targets(tmp_path / "t.txt", lines), env=env)
    assert p.returncode == 0, p.stderr[-3000:]
    # work done once: one .mut parse per chromosome, one genome upload and nothing else copied of the genome
    glen = sum(os.path.getsize(f"{d}/g_chr{nm}.fa") for nm in open(f"{d}/chr.txt").read().split())
    stat = [x for x in p.stderr.splitlines() if "reference genome uploads" in x][0]
    assert ".mut texts parsed 2 " in stat and "reference genome uploads 1 " in stat, stat
    up_bytes = int(stat.split("(")[-1].split()[0])
    assert 0 < up_bytes < glen
    for k, (key, src, mask) in enumerate(MIXED):
        inp = f"{d}/{src}.bam" if key == "target_bam" else f"{d}/{src}"
        o = tmp_path / f"s{k}"
        q = _cli(*shared, f"--{key}", inp, *(["--target_mask", f"{d}/{mask}"] if mask else []), "-o", o)
        assert q.returncode == 0, q.stderr[-3000:]
        assert open(f"{tmp_path}/b{k}.colate.in", "rb").read() == open(f"{o}.colate.in", "rb").read(), MIXED[k]
        assert f"target on line {k + 2} ({tmp_path}/b{k}): " in p.stderr


def test_failing_lines_leave_no_file(mixed_dir, tmp_path):
    d, sites = mixed_dir
    # a BAM that is not sorted, a BCF with a missing GT
    reads = [(0, st, 60, 0, b"ACGTACGTACGTACGTACGTACGTACGTACGTA", bytes([37]) * 33, b"r", [(33, "M")], b"") for st in (5000, 100, 9000)]
    synth.write_bam(f"{tmp_path}/uns.bam", list(sites.chr_names), reads, contig_lens=[10 ** 7] * len(sites.chr_names))
    for c, nm in enumerate(sites.chr_names):
        recs = [(1000 + 10 * i, [b"A", b"G"], [0, 1, 1, 0, 0, 0]) for i in range(20)]
        if c == 1:
            recs[7] = (1070, [b"A", b"G"], [0, -1, 1, 0, 0, 0])
        _write_records(f"{tmp_path}/bad_chr{nm}.bcf", 3, 2, recs)
    open(f"{tmp_path}/f1.colate.in", "wb").write(b"stale")
    lines = [f"target_bam={d}/s0.bam {tmp_path}/f0", f"target_bam={tmp_path}/uns.bam {tmp_path}/f1", f"target_bcf={d}/b {tmp_path}/f2",
             f"target_bcf={tmp_path}/bad {tmp_path}/f3", f"target_bcf={d}/v {tmp_path}/f4 target_mask={d}/tm"]
    p = _cli("--mode", "make_tmp", "--mut", f"{d}/syn", "--chr", f"{d}/chr.txt", "--ref_genome", f"{d}/g", "--targets",
             _targets(tmp_path / "t.txt", lines))
    assert p.returncode == 1, p.stderr[-3000:]
    assert f"target on line 3 ({tmp_path}/f1) FAILED" in p.stderr and "not sorted" in p.stderr
    assert f"target on line 5 ({tmp_path}/f3) FAILED" in p.stderr and "missing" in p.stderr
    assert "2 of 5 targets failed" in p.stderr
    for k in (1, 3):
        assert not os.path.exists(f"{tmp_path}/f{k}.colate.in")
    for k in (0, 2, 4):
        assert os.path.getsize(f"{tmp_path}/f{k}.colate.in") > 0
        assert f"target on line {k + 2} ({tmp_path}/f{k}): " in p.stderr


def test_handle_parses_and_uploads_once(mixed_dir, tmp_path):
    """Through the API: one ingest and one genome upload serve several targets; pileup_from_bam with the resident genome copies none."""
    d, sites = mixed_dir
    names = list(sites.chr_names)
    h = api.Handle(0)
    try:
        h.ingest_mut([open(f"{d}/syn_chr{nm}.mut", "rb").read() for nm in names])
        genome = [api.read_fasta(f"{d}/g_chr{nm}.fa") for nm in names]
        h.set_ref_genome(genome)
        before = h.upload_counts()
        for k in range(2):
            h.pileup_from_bam(0, f"{d}/s{k}.bam", names, None)
            h.maketmp_write_pileup(0, names, tmp_path / f"p{k}.colate.in")
            h.maketmp_write_bcf([f"{d}/b_chr{nm}.bcf" for nm in names], names, tmp_path / f"q{k}.colate.in")
        assert h.upload_counts() == before
        assert before == {"mut_texts_parsed": len(names), "mut_rows_parsed": int(sites.site_off[-1]), "ref_uploads": 1,
                          "ref_h2d_bytes": sum(g.shape[0] for g in genome)}
        # the resident genome gives the pileup the per-call upload gives
        c0 = h.pileup_from_bam(1, f"{d}/s0.bam", names, None, fetch=True)
        c1 = h.pileup_from_bam(1, f"{d}/s0.bam", names, genome, fetch=True)
        assert np.array_equal(c0, c1)
    finally:
        h.close()
