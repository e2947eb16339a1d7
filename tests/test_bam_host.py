"""BAM input on the host, no GPU: BGZF blocks, the header, contig matching and the record walk (colate_bam_scan), checked against a
struct-based parse of Python's gzip.decompress output; every refusal of colate_pileup_bam's host side; the CLI's refusals of BAM
argument combinations, which come before any device is touched."""
import gzip
import os
import struct
import subprocess

import numpy as np
import pytest

from colate_b200 import _lib, api, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")


def py_scan(data, header_names, chr_names):
    """Reference walk of an inflated BAM stream: per --chr entry (header contig <name> or chr<name>) count, first and last pos."""
    assert data[:4] == b"BAM\1"
    l_text = struct.unpack_from("<i", data, 4)[0]
    o = 8 + l_text
    n_ref = struct.unpack_from("<i", data, o)[0]
    o += 4
    names = []
    for _ in range(n_ref):
        ln = struct.unpack_from("<i", data, o)[0]
        names.append(data[o + 4:o + 4 + ln - 1].decode())
        o += 4 + ln + 4
    assert names == header_names
    listed = {}
    for c, nm in enumerate(chr_names):
        for r, h in enumerate(names):
            if h in (nm, "chr" + nm):
                listed[r] = c
    n = np.zeros(len(chr_names), np.int64)
    first = np.full(len(chr_names), -1, np.int32)
    last = np.full(len(chr_names), -1, np.int32)
    while o < len(data):
        bs, ref, pos = struct.unpack_from("<iii", data, o)
        if ref in listed:
            c = listed[ref]
            if n[c] == 0:
                first[c] = pos
            last[c] = pos
            n[c] += 1
        o += 4 + bs
    return n, first, last


def rand_reads(rng, n, tid_choices, extras=True):
    reads = []
    pos = {t: 0 for t in tid_choices}
    tids = sorted(rng.choice(tid_choices, n))
    for t in tids:
        pos[t] += int(rng.integers(0, 50))
        ln = int(rng.integers(0, 150))
        seq = rng.choice(list(b"ACGTN"), ln).astype(np.uint8).tobytes()
        qual = rng.integers(0, 256, ln).astype(np.uint8)
        if extras:
            name = rng.choice(list(b"abcdefXYZ0123:_"), int(rng.integers(1, 255))).astype(np.uint8).tobytes()
            aux = b"NMC" + bytes([int(rng.integers(0, 9))]) + b"XBBc" + struct.pack("<i", 3) + b"\x01\x02\x03"
            reads.append((int(t), pos[t], int(rng.integers(0, 61)), int(rng.choice([0, 16, 4, 256, 1024, 2048])), seq, qual, name, None, aux))
        else:
            reads.append((int(t), pos[t], 30, 0, seq, qual))
    return reads


def scan(path, chr_names, window=0):
    return api.bam_scan(str(path), chr_names, window)


def refused(path, chr_names, *words):
    with pytest.raises(_lib.ColateError) as e:
        scan(path, chr_names)
    assert e.value.code == -5, str(e.value)
    msg = str(e.value)
    assert str(path) in msg, msg
    for w in words:
        assert w in msg, msg
    return msg


@pytest.mark.parametrize("block_size", [1, 7, 100, 4096, 65280, 65536])
@pytest.mark.parametrize("eof", [True, False])
def test_scan_equals_python_parse(built, tmp_path, block_size, eof):
    rng = np.random.default_rng(block_size)
    header = ["chr1", "2", "chrX"]
    reads = rand_reads(rng, 300 if block_size > 1 else 60, [0, 1, 2])
    empty = (0, 2, 5, 10 ** 9) if block_size != 65536 else (1,)
    p = tmp_path / "a.bam"
    synth.write_bam(str(p), header, reads, text=b"@HD\tVN:1.6\n", block_size=block_size, empty_blocks=empty, eof=eof)
    raw = open(p, "rb").read()
    data = gzip.decompress(raw)                       # the writer's output is valid gzip
    for chr_names in (["1", "2", "X"], ["2"], ["1", "X"]):
        n, first, last = py_scan(data, header, chr_names)
        for window in (0, 1, 333):
            got = scan(p, chr_names, window)
            assert np.array_equal(got["n_records"], n) and np.array_equal(got["first_pos"], first) and np.array_equal(got["last_pos"], last)
    assert list(scan(p, ["1", "2", "X"])["ref_id"]) == [0, 1, 2]


def test_name_matching_unlisted_contigs_and_unmapped_tail(built, tmp_path):
    rng = np.random.default_rng(3)
    header = ["chr1", "5", "2", "chr3", "chrUn"]
    reads = rand_reads(rng, 400, [0, 1, 2, 3, 4], extras=False)
    reads += [(-1, -1, 0, 4, b"ACGT", [30] * 4)] * 7                       # unmapped, no contig: skipped
    p = tmp_path / "m.bam"
    synth.write_bam(str(p), header, reads, block_size=999)
    got = scan(p, ["1", "2", "3"])
    n, first, last = py_scan(gzip.decompress(open(p, "rb").read()), header, ["1", "2", "3"])
    assert list(got["ref_id"]) == [0, 2, 3]
    assert np.array_equal(got["n_records"], n) and np.array_equal(got["first_pos"], first) and np.array_equal(got["last_pos"], last)
    assert n.sum() == sum(1 for r in reads if r[0] in (0, 2, 3))


def _bam_bytes(header=("chr1", "2"), reads=None, **kw):
    reads = reads if reads is not None else [(0, 10 * k, 30, 0, b"ACGTACGT", [30] * 8) for k in range(50)] + \
        [(1, 10 * k, 30, 0, b"ACGT", [30] * 4) for k in range(50)]
    data = synth.bam_header(list(header)) + b"".join(synth.bam_record(*r) for r in reads)
    return data


def _write(path, data, block_size=500, eof=True):
    open(path, "wb").write(synth.bgzf_compress(data, block_size=block_size, eof=eof))
    return path


def test_refuses_malformed_bgzf(built, tmp_path):
    data = _bam_bytes()
    good = open(_write(tmp_path / "g.bam", data), "rb").read()
    assert scan(tmp_path / "g.bam", ["1", "2"])["n_records"].tolist() == [50, 50]
    # a plain gzip file (no BC subfield)
    open(tmp_path / "plain.bam", "wb").write(gzip.compress(data))
    refused(tmp_path / "plain.bam", ["1", "2"], "BC", "byte offset 0")
    # truncated blocks: inside a block and inside a header
    open(tmp_path / "t1.bam", "wb").write(good[:len(good) - 40])
    refused(tmp_path / "t1.bam", ["1", "2"], "truncated", "byte offset")
    open(tmp_path / "t2.bam", "wb").write(good[:good.index(b"BC", 100) + 2])
    refused(tmp_path / "t2.bam", ["1", "2"], "truncated", "byte offset")
    # CRC and ISIZE of the second block
    b2 = struct.unpack_from("<H", good, 16)[0] + 1
    b3 = b2 + struct.unpack_from("<H", good, b2 + 16)[0] + 1
    bad = bytearray(good); bad[b3 - 8] ^= 1
    open(tmp_path / "crc.bam", "wb").write(bad)
    refused(tmp_path / "crc.bam", ["1", "2"], "CRC", f"byte offset {b2}")
    bad = bytearray(good); bad[b3 - 4] += 1
    open(tmp_path / "isize.bam", "wb").write(bad)
    refused(tmp_path / "isize.bam", ["1", "2"], "ISIZE", f"byte offset {b2}")
    # corrupt deflate data
    bad = bytearray(good); bad[b2 + 20] ^= 0xFF; bad[b2 + 21] ^= 0xFF
    open(tmp_path / "z.bam", "wb").write(bad)
    refused(tmp_path / "z.bam", ["1", "2"], f"byte offset {b2}")


def test_refuses_malformed_bam(built, tmp_path):
    data = _bam_bytes()
    refused(_write(tmp_path / "magic.bam", b"BAM\2" + data[4:]), ["1", "2"], "magic", "offset 0")
    hdr = synth.bam_header(["chr1", "2"])
    refused(_write(tmp_path / "hdr.bam", hdr[:len(hdr) - 6]), ["1", "2"], "header runs past", "offset")
    refused(_write(tmp_path / "rec.bam", data[:len(data) - 3]), ["1", "2"], "runs past the end", "offset")
    # a record whose fields run past its block_size: l_seq too large
    rec = bytearray(synth.bam_record(0, 5, 30, 0, b"ACGT", [30] * 4))
    struct.pack_into("<i", rec, 20, 400)
    refused(_write(tmp_path / "lseq.bam", hdr + bytes(rec)), ["1", "2"], "block_size", f"offset {len(hdr)}")
    rec = bytearray(synth.bam_record(7, 5, 30, 0, b"ACGT", [30] * 4))
    refused(_write(tmp_path / "ref.bam", hdr + bytes(rec)), ["1", "2"], "refID 7")
    # a record of a listed contig with a negative position (COLATE_ERR_ORDER); unlisted contigs may have one
    with pytest.raises(_lib.ColateError) as e:
        scan(_write(tmp_path / "neg.bam", hdr + synth.bam_record(1, -3, 30, 0, b"ACGT", [30] * 4)), ["1", "2"])
    assert e.value.code == -6 and "negative position" in str(e.value)
    assert scan(tmp_path / "neg.bam", ["1"])["n_records"].tolist() == [0]
    # the EOF block is optional
    assert scan(_write(tmp_path / "noeof.bam", data, eof=False), ["1", "2"])["n_records"].tolist() == [50, 50]


def test_refuses_contig_layouts(built, tmp_path):
    r = lambda t, p: (t, p, 30, 0, b"ACGTACGT", [30] * 8)
    refused(_write(tmp_path / "absent.bam", _bam_bytes(["chr1", "2"], [r(0, 1)])), ["1", "3"], "contig 3", "not in the BAM header")
    refused(_write(tmp_path / "both.bam", _bam_bytes(["chr1", "1", "2"], [r(0, 1)])), ["1", "2"], "both")
    refused(_write(tmp_path / "split.bam", _bam_bytes(["chr1", "2"], [r(0, 1), r(1, 1), r(0, 5)])), ["1", "2"], "not contiguous", "offset")
    refused(_write(tmp_path / "order.bam", _bam_bytes(["chr1", "2"], [r(1, 1), r(0, 5)])), ["1", "2"], "--chr order")
    # the same file is fine when the --chr list follows the file, or leaves the out-of-order contig out
    p = _write(tmp_path / "ok.bam", _bam_bytes(["chr1", "2"], [r(1, 1), r(0, 5)]))
    assert scan(p, ["2", "1"])["n_records"].tolist() == [1, 1]
    assert scan(p, ["1"])["n_records"].tolist() == [1]


def _cli(*args):
    return subprocess.run([CLI, *args], capture_output=True, text=True, timeout=120)


@pytest.mark.parametrize("extra, words", [
    (["--strandfilter"], "--strandfilter"),
    (["--target_tmp", "x.colate.in"], "--target_tmp cannot be mixed"),
    (["--devices", "0,1"], "one device"),
    (["--filters", "20,30"], "--filters"),
])
def test_cli_refuses_bam_combinations(built, tmp_path, extra, words):
    base = ["--mode", "mut", "--mut", "m", "--target_bam", "t.bam", "--reference_bam", "r.bam", "--ref_genome", "g", "--bins", "3,7,0.2",
            "-o", str(tmp_path / "o")]
    p = _cli(*base, *extra)
    assert p.returncode == 1 and words in p.stderr, p.stderr
    assert "no CUDA device" not in p.stderr and "colate_create" not in p.stderr


def test_cli_refuses_bam_without_ref_genome_or_with_pairs(built, tmp_path):
    base = ["--mode", "mut", "--mut", "m", "--target_bam", "t.bam", "--bins", "3,7,0.2", "-o", str(tmp_path / "o")]
    p = _cli(*base, "--reference_bam", "r.bam")
    assert p.returncode == 1 and "--ref_genome" in p.stderr, p.stderr
    p = _cli(*base, "--ref_genome", "g")
    assert p.returncode == 1 and "both --target_bam and --reference_bam" in p.stderr, p.stderr
    p = _cli("--mode", "mut", "--mut", "m", "--pairs", "p.txt", "--seed", "1", "--bins", "3,7,0.2", "--target_bam", "t.bam")
    assert p.returncode == 1 and "--pairs" in p.stderr, p.stderr
    p = _cli("--mode", "make_tmp", "--mut", "m", "--target_bam", "t.bam", "-o", str(tmp_path / "o"))
    assert p.returncode == 1 and "--ref_genome" in p.stderr, p.stderr
    p = _cli("--mode", "make_tmp", "--mut", "m", "--target_bam", "t.bam", "--ref_genome", "g", "--strandfilter", "-o", str(tmp_path / "o"))
    assert p.returncode == 1 and "--strandfilter" in p.stderr, p.stderr
    assert not os.path.exists(str(tmp_path / "o.colate.in"))


def test_read_fasta_upper_cases_and_reads_gz(built, tmp_path):
    open(tmp_path / "g.fa", "wb").write(b">x y\nacgtN\nACgt\n")
    assert api.read_fasta(str(tmp_path / "g.fa")).tobytes() == b"ACGTNACGT"
    open(tmp_path / "h.fa.gz", "wb").write(gzip.compress(b">x\nttAA\n"))
    assert api.read_fasta(str(tmp_path / "h.fa")).tobytes() == b"TTAA"
    with pytest.raises(_lib.ColateError):
        api.read_fasta(str(tmp_path / "missing.fa"))
