"""BCF input on the host, no GPU: BGZF blocks, the header (sample count, GT key with and without IDX=) and the record walk
(colate_bcf_scan), checked against a struct-based parse of Python's gzip.decompress output; every host refusal of
colate_rows_from_bcf; the CLI's refusals of BCF argument combinations, which come before any device is touched; and the per-genome
split of parse_vcfvcf's decoder half that the device resolves rows by."""
import gzip
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

from colate_b200 import _lib, api, synth
from oracle import pyoracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from bcf_helpers import IDS, IDX_SHUFFLED, combine, keys_of, py_decode, random_records, resolve_bcf_rows  # noqa: E402
from helpers import load, sites_from, vcfvcf_counts  # noqa: E402

ROOT = os.path.dirname(HERE)
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")


def _file(tmp_path, name, n=200, n_sample=3, idx=None, minor=2, block_size=500, eof=True, empty=(), seed=0, **kw):
    rng = np.random.default_rng(seed)
    recs, _ = random_records(rng, n, n_sample, idx=idx, **kw)
    p = tmp_path / name
    synth.write_bcf(str(p), synth.bcf_header(n_sample, IDS, idx=idx, minor=minor), recs, block_size=block_size, empty_blocks=empty, eof=eof)
    return p


def _check_scan(p, window=0):
    ns, gt_key, recs = py_decode(gzip.decompress(open(p, "rb").read()))
    got = api.bcf_scan(str(p), window)
    assert got == {"n_records": len(recs), "first_pos": recs[0][1], "last_pos": recs[-1][1], "contig": recs[0][0], "n_sample": ns,
                   "gt_key": gt_key}, (got, len(recs))
    return got


@pytest.mark.parametrize("block_size", [1, 7, 100, 4096, 65280, 65536])
@pytest.mark.parametrize("eof", [True, False])
def test_scan_equals_python_parse(built, tmp_path, block_size, eof):
    p = _file(tmp_path, "a.bcf", n=40 if block_size == 1 else 300, n_sample=int(1 + block_size % 5), block_size=block_size, eof=eof,
              empty=(0, 2, 5, 10 ** 9) if block_size != 65536 else (1,), seed=block_size)
    for window in (0, 1, 333):
        _check_scan(p, window)


@pytest.mark.parametrize("idx", [None, IDX_SHUFFLED], ids=["order_of_appearance", "IDX"])
@pytest.mark.parametrize("minor", [1, 2])
def test_scan_magics_and_gt_key(built, tmp_path, idx, minor):
    p = _file(tmp_path, "k.bcf", idx=idx, minor=minor, seed=minor)
    got = _check_scan(p)
    assert got["gt_key"] == keys_of(idx)["GT"]
    assert got["gt_key"] == (5 if idx else 7)


def test_repeated_positions_and_wide_records(built, tmp_path):
    p = _file(tmp_path, "r.bcf", n=60, n_sample=2504, pos_step=(0, 2), block_size=65280)
    got = _check_scan(p)
    assert got["n_sample"] == 2504


def refused(path, *words, code=-5):
    with pytest.raises(_lib.ColateError) as e:
        api.bcf_scan(str(path))
    msg = str(e.value)
    assert e.value.code == code, msg
    assert str(path) in msg, msg
    for w in words:
        assert w in msg, msg
    return msg


def _raw(n=50, n_sample=2, contigs=None, positions=None, ids=IDS, idx=None, n_sample_rec=None):
    k = keys_of(idx)
    hdr = synth.bcf_header(n_sample, ids, idx=idx)
    recs = []
    for r in range(n):
        c = contigs[r] if contigs else 0
        p = positions[r] if positions else 10 * r
        recs.append(synth.bcf_record(c, p, [b"A", b"G"], [[0, 1]] * n_sample, k["GT"], n_sample=n_sample_rec))
    return hdr, recs


def _write(path, data, block_size=500, eof=True):
    open(path, "wb").write(synth.bgzf_compress(data, block_size=block_size, eof=eof))
    return path


def test_refuses_malformed_bgzf_and_other_formats(built, tmp_path):
    hdr, recs = _raw()
    data = hdr + b"".join(recs)
    good = open(_write(tmp_path / "g.bcf", data), "rb").read()
    assert api.bcf_scan(str(tmp_path / "g.bcf"))["n_records"] == 50
    open(tmp_path / "plain.bcf", "wb").write(gzip.compress(data))
    refused(tmp_path / "plain.bcf", "BC", "plain gzip is not BCF", "byte offset 0")
    open(tmp_path / "u.bcf", "wb").write(data)                                    # bcftools -Ou
    refused(tmp_path / "u.bcf", "not a gzip member", "byte offset 0")
    open(tmp_path / "t.vcf", "wb").write(b"##fileformat=VCFv4.3\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n")
    refused(tmp_path / "t.vcf", "not a gzip member", "byte offset 0")
    open(tmp_path / "t1.bcf", "wb").write(good[:len(good) - 40])
    refused(tmp_path / "t1.bcf", "truncated", "byte offset")
    b2 = struct.unpack_from("<H", good, 16)[0] + 1
    b3 = b2 + struct.unpack_from("<H", good, b2 + 16)[0] + 1
    bad = bytearray(good); bad[b3 - 8] ^= 1
    open(tmp_path / "crc.bcf", "wb").write(bad)
    refused(tmp_path / "crc.bcf", "CRC", f"byte offset {b2}")
    bad = bytearray(good); bad[b3 - 4] += 1
    open(tmp_path / "isize.bcf", "wb").write(bad)
    refused(tmp_path / "isize.bcf", "ISIZE", f"byte offset {b2}")


def test_refuses_malformed_bcf(built, tmp_path):
    hdr, recs = _raw()
    data = hdr + b"".join(recs)
    refused(_write(tmp_path / "magic.bcf", b"BCF\2\3" + data[5:]), "magic", "offset 0")
    refused(_write(tmp_path / "bam.bcf", b"BAM\1" + data[4:]), "magic", "offset 0")
    refused(_write(tmp_path / "hdr.bcf", hdr[:len(hdr) - 6]), "header runs past", "offset")
    refused(_write(tmp_path / "rec.bcf", data[:len(data) - 3]), "runs past the end", "offset")
    refused(_write(tmp_path / "empty.bcf", hdr), "without records")
    # no ##FORMAT=<ID=GT line (a GT line under INFO does not count)
    h2, r2 = _raw(ids=[("INFO", "GT"), ("FORMAT", "GQ")])
    refused(_write(tmp_path / "nogt.bcf", h2 + b"".join(r2)), "##FORMAT=<ID=GT")
    # records on two contigs
    h3, r3 = _raw(n=6, contigs=[0, 0, 0, 1, 1, 1])
    msg = refused(_write(tmp_path / "two.bcf", h3 + b"".join(r3)), "contig 1", "one contig")
    assert f"inflated byte offset {len(h3) + sum(len(r) for r in r3[:3])}" in msg
    # a record whose sample count is not the header's
    h4, r4 = _raw(n=3)
    _, bad = _raw(n=1, n_sample=2, n_sample_rec=3)
    refused(_write(tmp_path / "ns.bcf", h4 + r4[0] + bad[0] + r4[2]), "3 samples", "header has 2", f"offset {len(h4) + len(r4[0])}")
    # descending POS: COLATE_ERR_ORDER; equal positions are fine
    h5, r5 = _raw(n=4, positions=[5, 9, 9, 8])
    refused(_write(tmp_path / "desc.bcf", h5 + b"".join(r5)), "not sorted", code=-6)
    h6, r6 = _raw(n=4, positions=[5, 9, 9, 9])
    assert api.bcf_scan(str(_write(tmp_path / "eq.bcf", h6 + b"".join(r6))))["n_records"] == 4


def _cli(*args):
    return subprocess.run([CLI, *args], capture_output=True, text=True, timeout=120)


@pytest.mark.parametrize("extra, words", [
    (["--target_tmp", "x.colate.in"], "--target_tmp cannot be mixed"),
    (["--reference_bam", "r.bam"], "cannot be mixed"),
    (["--target_table", "t.txt"], "--target_table cannot be mixed"),
    (["--devices", "0,1"], "one device"),
])
def test_cli_refuses_bcf_combinations(built, tmp_path, extra, words):
    base = ["--mode", "mut", "--mut", "m", "--chr", "c.txt", "--target_bcf", "t", "--reference_bcf", "r", "--bins", "3,7,0.2",
            "-o", str(tmp_path / "o")]
    p = _cli(*base, *extra)
    assert p.returncode == 1 and words in p.stderr, p.stderr
    assert "no CUDA device" not in p.stderr and "colate_create" not in p.stderr


def test_cli_refuses_single_bcf_missing_chr_and_pairs(built, tmp_path):
    base = ["--mode", "mut", "--mut", "m", "--bins", "3,7,0.2", "-o", str(tmp_path / "o")]
    for one in (["--target_bcf", "t"], ["--reference_bcf", "r"]):
        p = _cli(*base, "--chr", "c.txt", *one)
        assert p.returncode == 1 and "both --target_bcf and --reference_bcf" in p.stderr, p.stderr
    p = _cli(*base, "--target_bcf", "t", "--reference_bcf", "r")
    assert p.returncode == 1 and "--chr" in p.stderr, p.stderr
    p = _cli("--mode", "mut", "--mut", "m", "--pairs", "p.txt", "--seed", "1", "--bins", "3,7,0.2", "--target_bcf", "t")
    assert p.returncode == 1 and "--pairs" in p.stderr, p.stderr
    p = _cli("--mode", "make_tmp", "--mut", "m", "--target_bcf", "t", "--ref_genome", "g", "-o", str(tmp_path / "o"))
    assert p.returncode == 1 and "--chr" in p.stderr, p.stderr
    p = _cli("--mode", "make_tmp", "--mut", "m", "--chr", "c.txt", "--target_bcf", "t", "-o", str(tmp_path / "o"))
    assert p.returncode == 1 and "ref_genome" in p.stderr, p.stderr
    p = _cli("--mode", "make_tmp", "--mut", "m", "--chr", "c.txt", "--target_bcf", "t", "--target_bam", "t.bam", "--ref_genome", "g",
             "-o", str(tmp_path / "o"))
    assert p.returncode == 1 and "cannot be mixed" in p.stderr, p.stderr
    assert not os.path.exists(str(tmp_path / "o.colate.in"))


# ---- the per-genome split of parse_vcfvcf's decoder half -----------------------------------------------------------------------
def _split(pos, anc, der, usable, recs_t, recs_r, n_t, n_r, refg):
    tc = resolve_bcf_rows("target", pos, anc, der, usable, recs_t, n_t, refg)
    rc = resolve_bcf_rows("reference", pos, anc, der, usable, recs_r, n_r, refg)
    return combine(tc, rc)


@pytest.mark.parametrize("with_refg", [False, True])
def test_per_genome_split_equals_decode_vcfvcf_on_the_fixture(with_refg):
    z = load("stage1_vcfvcf.npz")
    sites, tc, rc = vcfvcf_counts(z, with_refg)
    meta = sites.meta()
    for c in range(len(sites.chr_names)):
        lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
        recs = {}
        for tag in ("t", "r"):
            al = z[f"{tag}{c}_al"]
            recs[tag] = [(int(p), [bytes(a) for a in al[i][:int(n)]], [int(g) for g in gt])
                         for i, (p, n, gt) in enumerate(zip(z[f"{tag}{c}_pos"], z[f"{tag}{c}_nal"], z[f"{tag}{c}_gt"]))]
        usable = ((meta[lo:hi] & 1) != 0) & (sites.anc[lo:hi] != sites.der[lo:hi])
        t2, r2 = _split(sites.pos[lo:hi], sites.anc[lo:hi], sites.der[lo:hi], usable, recs["t"], recs["r"], int(z["n_hap_target"]),
                        int(z["n_hap_ref"]), z["refg_at_rows"][lo:hi] if with_refg else None)
        assert np.array_equal(t2, tc[lo:hi]) and np.array_equal(r2, rc[lo:hi])
        assert (t2.sum(1) > 0).sum() > 100


@pytest.mark.parametrize("seed", range(6))
def test_per_genome_split_equals_decode_vcfvcf_on_random_streams(seed):
    """Record streams with repeated positions, one-allele and empty-allele records, third alleles, records between and beyond
    the rows, and a reference genome with every kind of base at the rows."""
    rng = np.random.default_rng(100 + seed)
    n_rows = 400
    pos = np.sort(rng.integers(1, 3000, n_rows)).astype(np.int32)
    bases = np.frombuffer(b"ACGT", np.uint8)
    anc = bases[rng.integers(0, 4, n_rows)]
    der = bases[rng.integers(0, 4, n_rows)]
    usable = rng.random(n_rows) < 0.9
    refg = np.frombuffer(b"ACGTN", np.uint8)[rng.integers(0, 5, n_rows)]

    def stream(n_hap):
        recs = []
        cands = np.sort(np.concatenate([pos[rng.random(n_rows) < 0.7] - 1, rng.integers(0, 3100, 100)]))
        for p0 in cands:
            for _ in range(int(rng.choice([1, 1, 1, 2, 3]))):
                m = int(np.searchsorted(pos, p0 + 1))
                a, d = (bytes([anc[m]]), bytes([der[m]])) if m < n_rows and rng.random() < 0.8 else (b"A", b"C")
                al = [[a, d], [d, a], [a], [d], [d, b""], [a, d, b"T"], [b"GG", d], [a, b"<X>"]][int(rng.integers(0, 8))]
                gt = list(rng.integers(0, len(al) if rng.random() < 0.2 else min(2, len(al)), n_hap))
                if len(al) == 1 or al[1] == b"":
                    gt = [0] * n_hap if rng.random() < 0.7 else gt
                recs.append((int(p0), al, [int(g) for g in gt]))
        return recs

    rt, rr = stream(2), stream(6)
    for refg_rows in (None, refg):
        tc, rc = po.decode_vcfvcf(pos, anc, der, usable, rt, rr, 2, 6, refg_rows)
        t2, r2 = _split(pos, anc, der, usable, rt, rr, 2, 6, refg_rows)
        assert np.array_equal(t2, tc) and np.array_equal(r2, rc)
        assert (tc.sum(1) > 0).sum() > 10
