"""Bgzipped text VCF on the host, no GPU: the format detection shared with BCF, the header (##, #CHROM) and the line walk
(colate_vcf_scan), checked against a Python parse of gzip.decompress output; every host refusal of colate_rows_from_bcf on a text
VCF, with its code, the path and the inflated offset; and colate_bcf_scan still refusing a text VCF."""
import gzip

import numpy as np
import pytest

from colate_b200 import _lib, api, synth

IDS = [("INFO", "DP"), ("FORMAT", "GQ"), ("FORMAT", "GT"), ("FORMAT", "AD")]


def _lines(rng, n, n_sample, chrom="1", pos_step=(0, 40), long_every=0, long_len=70000):
    out = []
    p = int(rng.integers(0, 100))
    for r in range(n):
        p += int(rng.integers(*pos_step))
        info = b"DP=%d" % r
        rid = b"."
        if long_every and r % long_every == 1:
            info = b"ANN=" + b"x|y" * (long_len // 3)
            rid = b"rs" + b"7" * (long_len // 4)
        gt = rng.integers(0, 2, (n_sample, 2)).tolist()
        out.append(synth.vcf_line(chrom, p, [b"A", b"G"], gt, phased=bool(r % 2), rid=rid, info=info,
                                  fmt_before=[("GQ", [b"%d" % (r % 99)] * n_sample)], fmt_after=[("AD", [b"1,2"] * n_sample)]))
    return out


def _write(path, data, block_size=500, empty=(), eof=True):
    open(path, "wb").write(synth.bgzf_compress(data, block_size=block_size, empty_blocks=empty, eof=eof))
    return path


def py_scan(path):
    text = gzip.decompress(open(path, "rb").read()).decode()
    lines = text.split("\n")
    if lines[-1] == "":
        lines.pop()
    hdr = [ln for ln in lines if ln.startswith("#")]
    recs = [ln.split("\t") for ln in lines if not ln.startswith("#")]
    return {"n_records": len(recs), "first_pos": int(recs[0][1]) - 1, "last_pos": int(recs[-1][1]) - 1,
            "n_sample": hdr[-1].count("\t") - 8, "chrom": recs[0][0]}


def _check(path, windows=(0, 1, 333, 70001)):
    want = py_scan(path)
    for w in windows:
        assert api.vcf_scan(str(path), w) == want, w
    return want


@pytest.mark.parametrize("block_size", [1, 7, 100, 4096, 65280, 65536])
@pytest.mark.parametrize("eof", [True, False])
def test_scan_equals_python_parse(built, tmp_path, block_size, eof):
    rng = np.random.default_rng(block_size)
    n_sample = int(1 + block_size % 5)
    data = synth.vcf_header(n_sample, IDS) + b"".join(_lines(rng, 30 if block_size == 1 else 300, n_sample))
    p = _write(tmp_path / "a.vcf.gz", data, block_size, empty=(0, 2, 5, 10 ** 9) if block_size != 65536 else (1,), eof=eof)
    _check(p)


def test_long_info_and_id_fields_one_line_per_window(built, tmp_path):
    rng = np.random.default_rng(1)
    data = synth.vcf_header(3, IDS) + b"".join(_lines(rng, 40, 3, long_every=3, long_len=150000))
    p = _write(tmp_path / "l.vcf.gz", data, 65280)
    got = _check(p, windows=(0, 1, 1000, 65280, 200000))
    assert got["n_records"] == 40


def test_extra_header_lines_contigs_and_no_final_newline(built, tmp_path):
    rng = np.random.default_rng(2)
    extra = [b"##contig=<ID=chr%d,length=%d>" % (c, 1000 * c) for c in range(1, 30)] + [b"##source=x" * 500, b"##reference=file:///x"]
    lines = _lines(rng, 50, 4, chrom="chr7", pos_step=(0, 3))
    data = synth.vcf_header(4, IDS, contigs=("chr7", "chrX"), extra=extra) + b"".join(lines)
    got = _check(_write(tmp_path / "e.vcf.gz", data, 777))
    assert got["chrom"] == "chr7" and got["n_sample"] == 4
    assert _check(_write(tmp_path / "nn.vcf.gz", data[:-1], 333))["n_records"] == 50     # last line without its newline


def refused(path, *words, code=-5):
    with pytest.raises(_lib.ColateError) as e:
        api.vcf_scan(str(path))
    msg = str(e.value)
    assert e.value.code == code, msg
    assert str(path) in msg, msg
    for w in words:
        assert w in msg, msg
    return msg


def _rec(r, pos=None, chrom="1", n_sample=2):
    return synth.vcf_line(chrom, 10 * r if pos is None else pos, [b"A", b"G"], [[0, 1]] * n_sample)


def test_header_refusals(built, tmp_path):
    recs = b"".join(_rec(r) for r in range(5))
    hdr = synth.vcf_header(2, IDS)
    nogt = synth.vcf_header(2, [("INFO", "GT"), ("FORMAT", "GQ")])
    refused(_write(tmp_path / "nogt.vcf.gz", nogt + recs), "##FORMAT=<ID=GT", "inflated byte offset 0")
    body = hdr[:hdr.index(b"#CHROM")]
    refused(_write(tmp_path / "nochrom.vcf.gz", body + recs), "#CHROM", f"inflated byte offset {len(body)}")
    refused(_write(tmp_path / "nochrom2.vcf.gz", body), "#CHROM", f"inflated byte offset {len(body)}")
    bad = body + b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTR\tINFO\tFORMAT\ts0\ts1\n"
    refused(_write(tmp_path / "cols.vcf.gz", bad + recs), "first eight columns", f"inflated byte offset {len(body)}")
    short = body + b"#CHROM\tPOS\tID\tREF\tALT\n"
    refused(_write(tmp_path / "short.vcf.gz", short + recs), "first eight columns")
    nos = synth.vcf_header(0, IDS)
    refused(_write(tmp_path / "nos.vcf.gz", nos + recs), "without samples", f"inflated byte offset {len(body)}")
    fmt_only = body + b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\n"
    refused(_write(tmp_path / "fmt.vcf.gz", fmt_only + recs), "FORMAT but no sample", f"inflated byte offset {len(body)}")
    refused(_write(tmp_path / "empty.vcf.gz", hdr), "without records")


def test_line_refusals(built, tmp_path):
    hdr = synth.vcf_header(2, IDS)
    good = [_rec(r) for r in range(6)]

    def at(k):
        return f"inflated byte offset {len(hdr) + sum(len(x) for x in good[:k])}"

    def case(name, bad, *words, code=-5):
        for bs in (500, 7):
            refused(_write(tmp_path / f"{name}{bs}.vcf.gz", hdr + b"".join(good[:3]) + bad + b"".join(good[3:]), bs), *words, at(3), code=code)
    case("chrom", _rec(3, chrom="2") + b"".join(_rec(r, chrom="2") for r in range(4, 6)), "contig 2", "one contig")
    case("order", _rec(3, pos=5), "not sorted", code=-6)
    case("empty", b"\n", "empty VCF line")
    case("crlf", _rec(3)[:-1] + b"\r\n", "\\r\\n")
    for i, pos in enumerate([b"", b"x1", b"+5", b"-1", b"2147483647", b"99999999999", b"1e3", b" 30"]):
        line = b"1\t" + pos + b"\t.\tA\tG\t.\tPASS\t.\tGT\t0|1\t0|1\n"
        case(f"pos{i}", line, "POS")
    case("nopos", b"1\n", "POS")
    # equal positions are fine, and so is POS 0 and 2^31 - 2
    data = hdr + b"1\t0\t.\tA\tG\t.\t.\t.\tGT\t0|0\t0|0\n" + b"".join(_rec(r, pos=7) for r in range(3)) + \
        b"1\t2147483646\t.\tA\tG\t.\t.\t.\tGT\t0|0\t0|0\n"
    got = api.vcf_scan(str(_write(tmp_path / "eq.vcf.gz", data)))
    assert got["n_records"] == 5 and got["first_pos"] == -1 and got["last_pos"] == 2147483645


def test_other_formats_keep_their_refusals(built, tmp_path):
    data = synth.vcf_header(2, IDS) + b"".join(_rec(r) for r in range(5))
    open(tmp_path / "plain.vcf.gz", "wb").write(gzip.compress(data))
    refused(tmp_path / "plain.vcf.gz", "plain gzip is not BCF", "byte offset 0")
    open(tmp_path / "u.vcf", "wb").write(data)
    refused(tmp_path / "u.vcf", "not a gzip member", "byte offset 0")
    refused(_write(tmp_path / "x.vcf.gz", b"##fileformat=VCX\n" + data[17:]), "not a BCF file", "offset 0")
    refused(_write(tmp_path / "tiny.vcf.gz", b"##file"), "not a BCF file")
    # a BCF file is bcf_scan's
    hdr = synth.bcf_header(2, IDS)
    recs = [synth.bcf_record(0, 10 * r, [b"A", b"G"], [[0, 1]] * 2, 3) for r in range(5)]
    p = tmp_path / "b.bcf"
    synth.write_bcf(str(p), hdr, recs)
    refused(p, "a BCF file")
    assert api.bcf_scan(str(p))["n_records"] == 5
    # and bcf_scan still refuses text VCF by its magic
    p = _write(tmp_path / "v.vcf.gz", data)
    assert api.vcf_scan(str(p))["n_records"] == 5
    with pytest.raises(_lib.ColateError) as e:
        api.bcf_scan(str(p))
    assert e.value.code == -5 and "not a BCF file (magic" in str(e.value) and str(p) in str(e.value)
