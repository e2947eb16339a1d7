"""BAM files read directly (colate_pileup_bam, `--target_bam` / `--reference_bam`): the fixture's reads written into real BGZF BAMs
must reproduce, byte for byte, what the reference CLI wrote from them (tests/golden/bambam_R1 / R3, stage1_bambam.npz
maketmp_bam_*); the device decode must equal the host-array path (pileup_from_reads) and the oracle on records the fixture never
had; the position-order refusals; chunking down to one record per chunk."""
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
from helpers import GOLDEN, bambam_masks, load  # noqa: E402

CLI = os.path.join(os.path.dirname(HERE), "colate_b200", "bin", "Colate")
pytestmark = pytest.mark.gpu


def _fixture_reads(reads, rng):
    """The fixture's reads as BAM records with extra content the reference's outputs must not depend on: read names, <len>M
    CIGARs, aux tags; flag 0x10 for reverse strand, as the reference saw."""
    out = []
    for k, (c, st, mq, rev, seq, qual) in enumerate(reads):
        name = b"read_%d" % k
        aux = b"NMC" + bytes([int(rng.integers(0, 10))]) + b"RGZgrp1\0"
        out.append((c, st, mq, 16 if rev else 0, seq, qual, name, [(len(seq), "M")], aux))
    return out


@pytest.fixture(scope="module")
def golden_dir(tmp_path_factory, built):
    import make_golden
    z = load("stage1_bambam.npz")
    sites, lens, genome, reads_t, reads_r = make_golden.bambam_inputs(int(z["seed"]))
    d = str(tmp_path_factory.mktemp("bambam"))
    synth.write_dataset(d, sites, {})
    for c, L in enumerate(lens):
        with open(os.path.join(d, f"g_chr{sites.chr_names[c]}.fa"), "wb") as f:
            f.write(b">ref\n")
            for i in range(0, L, 1 << 20):
                f.write(genome[c][i:i + (1 << 20)].tobytes() + b"\n")
    bam_names = ["chr" + sites.chr_names[0], sites.chr_names[1]]          # both spellings, as make_golden.py does
    rng = np.random.default_rng(1)
    synth.write_bam(os.path.join(d, "t.bam"), bam_names, _fixture_reads(reads_t, rng), contig_lens=lens, block_size=60000)
    synth.write_bam(os.path.join(d, "r.bam"), bam_names, _fixture_reads(reads_r, rng), contig_lens=lens, block_size=65280)
    tm, _ = bambam_masks(z)
    for c, nm in enumerate(sites.chr_names):
        synth.write_mask(os.path.join(d, f"tm_chr{nm}.fa"), tm[c])
    return d, z, sites, lens, genome, reads_t, reads_r


@pytest.mark.parametrize("R", [1, 3])
def test_cli_mut_bam_bam_matches_reference_cli(golden_dir, tmp_path, R):
    d, *_ = golden_dir
    o = str(tmp_path / "o")
    cmd = [CLI, "--mode", "mut", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--target_bam", os.path.join(d, "t.bam"),
           "--reference_bam", os.path.join(d, "r.bam"), "--ref_genome", os.path.join(d, "g"), "--bins", "3,7,0.2", "--seed", "23", "-o", o]
    if R == 3:
        cmd += ["--num_bootstraps", "3"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    for ext in (".coal", ".colate_mat"):
        assert open(o + ext).read() == open(os.path.join(GOLDEN, f"bambam_R{R}{ext}")).read(), ext
    assert os.path.exists(o + ".bin")


@pytest.mark.parametrize("tag", ["plain", "masked"])
def test_cli_make_tmp_bam_matches_reference_cli(golden_dir, tmp_path, tag):
    d, z, *_ = golden_dir
    o = str(tmp_path / "mk")
    cmd = [CLI, "--mode", "make_tmp", "--mut", os.path.join(d, "syn"), "--chr", os.path.join(d, "chr.txt"), "--target_bam", os.path.join(d, "t.bam"),
           "--ref_genome", os.path.join(d, "g"), "-o", o]
    if tag == "masked":
        cmd += ["--target_mask", os.path.join(d, "tm")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    assert open(o + ".colate.in", "rb").read() == z["maketmp_bam_" + tag].tobytes()


def _soa(reads_per_chr):
    """[(pos0, mapq, seq bytes, qual)] per contig -> the arrays pileup_from_reads takes."""
    per = []
    for rd in reads_per_chr:
        ln = np.array([len(r[2]) for r in rd], np.int32)
        off = np.concatenate([[0], np.cumsum(ln)[:-1]]).astype(np.int64) if len(rd) else np.zeros(0, np.int64)
        per.append((np.array([r[0] for r in rd], np.int32), np.array([r[1] for r in rd], np.uint8), ln, off,
                    np.frombuffer(b"".join(bytes(r[2]) for r in rd), np.uint8),
                    np.concatenate([np.asarray(r[3], np.uint8) for r in rd]) if rd else np.zeros(0, np.uint8)))
    return per


@pytest.mark.parametrize("chunk", [1, 700, 65536, 0])
def test_fixture_pileup_from_bam_equals_reference_bam_parser(golden_dir, handle, chunk):
    d, z, sites, lens, genome, reads_t, reads_r = golden_dir
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    names = list(sites.chr_names)
    for slot, (bam, key, reads) in enumerate((("t.bam", "t_counts", reads_t), ("r.bam", "r_counts", reads_r))):
        got = handle.pileup_from_bam(slot, os.path.join(d, bam), names, genome, chunk_bytes=chunk, fetch=True)
        assert np.array_equal(got, z[key]), (bam, chunk)
    if chunk == 0:
        per = [[(r[1], r[2], r[4], r[5]) for r in reads_t if r[0] == c] for c in range(len(lens))]
        assert np.array_equal(handle.pileup_from_reads(0, _soa(per), genome, fetch=True), z["t_counts"])


def _edge_case_contigs(rng, n_contigs=3, L=4000, n_reads=400):
    """Small contigs with every record shape the fixture lacks.  Returns (header names, contig genomes, per-contig reads as
    (pos0, mapq, seq, qual, flag, name, cigar, aux))."""
    genomes = [np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)].copy() for _ in range(n_contigs)]
    per = []
    letters = np.frombuffer(synth.NT16, np.uint8)
    for c in range(n_contigs):
        rd = []
        p = 0
        for k in range(n_reads):
            p += int(rng.integers(0, 12))
            ln = int(rng.choice([0, 1, 5, 31, 40, 60, 90, 120]))
            if p + ln > L:
                break
            seq = genomes[c][p:p + ln].copy()
            mm = rng.random(ln) < 0.05
            seq[mm] = letters[rng.integers(0, 16, int(mm.sum()))]           # every nt16 code, '=' included
            qual = np.where(rng.random(ln) < 0.15, rng.choice([0, 12, 29, 255], ln), rng.choice([30, 37, 41], ln)).astype(np.uint8)
            cig = [[(ln, "M")], [(2, "S"), (max(ln - 4, 0), "M"), (2, "S")], [(5, "H"), (ln, "M"), (3, "H")],
                   [(ln // 2, "M"), (3, "D"), (ln - ln // 2, "M")], [(ln // 2, "M"), (100, "N"), (max(ln - ln // 2 - 1, 0), "M"), (1, "I")]][k % 5]
            name = rng.choice(list(b"ACGTxyz:_0123456789"), int(rng.choice([1, 2, 17, 100, 254]))).astype(np.uint8).tobytes()
            aux = b"XBBc" + np.int32(7).tobytes() + bytes(range(7)) + b"YBBI" + np.int32(2).tobytes() + np.array([1, 2], np.uint32).tobytes() + b"ZZZhi\0"
            flag = int(rng.choice([0, 16, 4, 256, 1024, 2048, 4 | 16]))
            rd.append((p, int(rng.choice([0, 19, 20, 37, 60])), seq.tobytes(), qual, flag, name, cig, aux))
        per.append(rd)
    return ["chr1", "2", "chr3"][:n_contigs], genomes, per


def _write_edge_bam(path, header, per, **kw):
    recs = [(c, r[0], r[1], r[4], r[2], r[3], r[5], r[6], r[7]) for c, rd in enumerate(per) for r in rd]
    synth.write_bam(str(path), header, recs, **kw)


def test_decode_equals_host_arrays_and_oracle_on_record_shapes(handle, tmp_path):
    rng = np.random.default_rng(11)
    header, genomes, per = _edge_case_contigs(rng)
    names = ["1", "2", "3"]
    # rows: every 3rd position of each contig
    rows = [np.arange(5, len(g), 3, dtype=np.int32) for g in genomes]
    sites = synth.make_sites(2, [len(r) for r in rows], [len(g) for g in genomes])
    sites.pos = np.concatenate(rows).astype(np.int32)
    sites.chr_names = names
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    bam = tmp_path / "e.bam"
    _write_edge_bam(bam, header, per, block_size=3000, empty_blocks=(1, 4))
    want = handle.pileup_from_reads(0, _soa([[(r[0], r[1], r[2], r[3]) for r in rd] for rd in per]), genomes, fetch=True)
    oracle = np.concatenate([po.pileup_from_reads(rows[c], [(r[0], r[1], r[2], r[3]) for r in per[c]], genomes[c]) for c in range(3)])
    assert np.array_equal(want, oracle)
    assert (want.sum(1) > 0).sum() > 500
    soft = [np.where(rng.random(len(g)) < 0.5, g + 32, g).astype(np.uint8) for g in genomes]       # soft-masked (lower-case) bases
    for chunk in (1, 97, 5000, 0):
        for ref in (genomes, soft):
            got = handle.pileup_from_bam(1, str(bam), names, ref, chunk_bytes=chunk, fetch=True)
            assert np.array_equal(got, want), chunk


def test_quirk_lands_on_the_contigs_first_record_only(handle, tmp_path):
    """Records whose packed-sequence bytes are under 30 where their qualities are over it: the quirk drops the first record's
    bases, and applying it to the first record of every chunk would drop more."""
    L = 600
    g = np.frombuffer(b"AC" * (L // 2), np.uint8).copy()           # packed bytes 0x12 = 18 < 30
    reads = [(p, 60, g[p:p + 40].tobytes(), np.full(40, 40, np.uint8)) for p in range(0, 400, 10)]
    rows = np.arange(1, L, 1, dtype=np.int32)
    sites = synth.make_sites(3, [len(rows)], [L])
    sites.pos = rows
    sites.chr_names = ["1"]
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    synth.write_bam(str(tmp_path / "q.bam"), ["1"], [(0, r[0], r[1], 0, r[2], r[3]) for r in reads])
    want = po.pileup_from_reads(rows, reads, g)
    no_quirk = po.pileup_from_reads(rows, [(-1000, 0, b"ACGTACGT", np.zeros(8, np.uint8))] + reads, g)
    assert not np.array_equal(want, no_quirk)
    for chunk in (1, 60, 200, 0):
        assert np.array_equal(handle.pileup_from_bam(0, str(tmp_path / "q.bam"), ["1"], [g], chunk_bytes=chunk, fetch=True), want), chunk


def test_order_refusals(handle, tmp_path):
    L = 3000
    g = np.frombuffer(b"ACGT", np.uint8)[np.random.default_rng(2).integers(0, 4, L)].copy()
    rows = np.arange(10, L, 7, dtype=np.int32)
    sites = synth.make_sites(4, [len(rows), len(rows)], [L, L])
    sites.pos = np.concatenate([rows, rows]).astype(np.int32)
    sites.chr_names = ["1", "2"]
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    rec = lambda c, p: (c, p, 60, 0, g[max(p, 0):max(p, 0) + 50].tobytes(), np.full(50, 40, np.uint8))
    ok = [rec(0, p) for p in range(0, 2000, 20)] + [rec(1, p) for p in range(0, 100, 20)]
    synth.write_bam(str(tmp_path / "ok.bam"), ["1", "2"], ok)
    handle.pileup_from_bam(0, str(tmp_path / "ok.bam"), ["1", "2"], [g, g], chunk_bytes=1)
    # a new contig may start lower; a descent inside a chunk, across a chunk boundary, and a negative position may not
    cases = {"inside": ok[:5] + [rec(0, 30)] + ok[5:], "negative": [rec(0, -5)] + ok}
    for name, reads in cases.items():
        synth.write_bam(str(tmp_path / f"{name}.bam"), ["1", "2"], reads)
        for chunk in (1, 0):
            with pytest.raises(_lib.ColateError) as e:
                handle.pileup_from_bam(0, str(tmp_path / f"{name}.bam"), ["1", "2"], [g, g], chunk_bytes=chunk)
            assert e.value.code == -6, (name, chunk)
            if name == "inside":
                assert "not sorted by position" in str(e.value)
    # descent exactly at a chunk boundary: one record per chunk, and chunks of ~10 records with the descent at record 10
    one = len(synth.bam_record(*rec(0, 0)))
    reads = ok[:10] + [rec(0, 150)] + ok[10:]
    synth.write_bam(str(tmp_path / "edge.bam"), ["1", "2"], reads)
    for chunk in (1, 10 * one):
        with pytest.raises(_lib.ColateError) as e:
            handle.pileup_from_bam(0, str(tmp_path / "edge.bam"), ["1", "2"], [g, g], chunk_bytes=chunk)
        assert e.value.code == -6, chunk


def test_random_millions_of_reads_then_stage1(handle, tmp_path):
    """2.5 M random reads over two contigs: counts equal the host-array path for three chunk sizes, and stage i on the BAM genomes
    equals stage i on the host-array genomes bit for bit."""
    rng = np.random.default_rng(42)
    lens = [3_000_000, 2_000_000]
    genome = [np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)].copy() for L in lens]
    sites = synth.make_sites(42, [60000, 40000], lens)
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    path = {}
    arrays = {}
    for tag, n_per in (("t", [1_000_000, 500_000]), ("r", [600_000, 400_000])):
        chunks, soa = [], []
        for c, n in enumerate(n_per):
            ln = rng.integers(30, 121, n).astype(np.int32)
            pos = np.sort(rng.integers(0, lens[c] - 121, n)).astype(np.int32)
            idx = np.repeat(pos.astype(np.int64), ln) + (np.arange(int(ln.sum())) - np.repeat(np.cumsum(ln) - ln, ln))
            seq = genome[c][idx].copy()
            mm = rng.random(seq.shape[0]) < 0.02
            seq[mm] = np.frombuffer(b"ACGTN", np.uint8)[rng.integers(0, 5, int(mm.sum()))]
            qual = np.where(rng.random(seq.shape[0]) < 0.1, 15, 37).astype(np.uint8)
            mapq = rng.choice(np.array([0, 25, 60], np.uint8), n)
            chunks.append(synth.bam_records_np(np.full(n, c), pos, mapq, ln, seq, qual))
            soa.append((pos, mapq, ln, np.concatenate([[0], np.cumsum(ln)[:-1]]).astype(np.int64), seq, qual))
        data = synth.bam_header(["chr1", "chr2"], lens) + np.concatenate(chunks).tobytes()
        path[tag] = str(tmp_path / f"{tag}.bam")
        open(path[tag], "wb").write(synth.bgzf_compress(data, level=1, threads=8))
        arrays[tag] = soa
    handle.set_option("front_end", 1)
    try:
        ref_t = handle.pileup_from_reads(0, arrays["t"], genome, fetch=True)
        ref_r = handle.pileup_from_reads(1, arrays["r"], genome, fetch=True)
        assert (ref_t.sum(1) > 0).sum() > 50000
        s_ref = handle.stage1(api.mt_seed(7))
        for chunk in (1 << 16, 1 << 22, 0):
            assert np.array_equal(handle.pileup_from_bam(0, path["t"], ["1", "2"], genome, chunk_bytes=chunk, fetch=True), ref_t), chunk
        assert np.array_equal(handle.pileup_from_bam(1, path["r"], ["1", "2"], genome, fetch=True), ref_r)
        s_bam = handle.stage1(api.mt_seed(7))
        assert s_bam.num_blocks == s_ref.num_blocks and s_bam.n_used == s_ref.n_used
        assert np.array_equal(s_bam.block_stats, s_ref.block_stats) and np.array_equal(s_bam.block_tallies, s_ref.block_tallies)
        assert np.array_equal(s_bam.mt_state, s_ref.mt_state)
    finally:
        handle.set_option("front_end", 0)
