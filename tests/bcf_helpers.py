"""The decoder half of parse_vcfvcf (coal.cpp:997-1137) split per genome, as colate_rows_from_bcf resolves it: every role looks
its record up on its own (the first record at or after the row's position) and a row is used when both roles can use it.
test_bcf_host.py pins `combine(resolve_bcf_rows("target", ...), resolve_bcf_rows("reference", ...))` to
oracle/pyoracle.py:decode_vcfvcf, which restates the reference's two sequential cursors."""
import bisect

import numpy as np


def resolve_bcf_rows(role, pos_rows, anc_rows, der_rows, usable_rows, recs, n_hap, refg_at_rows=None):
    """(AAF, DAF) per row for one genome, zeros where the row is not usable for it.  recs: [(pos0, [alleles], [allele index per
    haplotype])] ascending (equal positions allowed); role "target" or "reference"; other arguments as decode_vcfvcf."""
    out = np.zeros((len(pos_rows), 2), np.int32)
    starts = [r[0] + 1 for r in recs]
    for m in range(len(pos_rows)):
        if not usable_rows[m]:
            continue
        bp, anc, der = int(pos_rows[m]), bytes([anc_rows[m]]), bytes([der_rows[m]])
        k = bisect.bisect_left(starts, bp)
        daf = None
        if k < len(recs) and starts[k] == bp:
            al, gt = recs[k][1], recs[k][2]
            a0 = bytes(al[0]) if len(al) > 0 else b""
            a1 = bytes(al[1]) if len(al) > 1 else b""
            biallelic = all(g <= 1 for g in gt)
            if (a0 == anc and a1 == der) or (a0 == der and a1 == anc):
                if biallelic:
                    daf = n_hap - sum(gt) if a0 == der else sum(gt)
            elif role == "target" and a0 != b"" and a1 == b"":
                if a0 in (anc, der) and biallelic and sum(gt) == 0:
                    daf = n_hap if a0 == der else 0
        elif refg_at_rows is not None:
            b = bytes([refg_at_rows[m]])
            if b == der:
                daf = n_hap
            elif role == "target" and b == anc:
                daf = 0
        if role == "reference" and daf == 0:
            daf = None
        if daf is not None:
            out[m] = (n_hap - daf, daf)
    return out


def combine(tc, rc):
    """Rows both genomes can use keep their counts; k_pileup_join + k_ok decide the same on the device."""
    both = (tc.sum(1) > 0) & (rc.sum(1) > 0)
    return np.where(both[:, None], tc, 0).astype(np.int32), np.where(both[:, None], rc, 0).astype(np.int32)


# ---- a struct-based BCF reader (the device decode and colate_bcf_scan are checked against it) ----------------------------------
_SHIFT = {0: 0, 1: 0, 2: 1, 3: 2, 5: 2, 7: 0}
_FMT = {1: "b", 2: "h", 3: "i"}


def _typed(data, o):
    import struct
    b = data[o]
    t, n = b & 15, b >> 4
    o += 1
    if n == 15:
        t2 = data[o] & 15
        n = struct.unpack_from("<" + _FMT[t2], data, o + 1)[0]
        o += 1 + (1 << _SHIFT[t2])
    return t, n, o


def _int(data, o):
    import struct
    t, n, o = _typed(data, o)
    assert n == 1
    return struct.unpack_from("<" + _FMT[t], data, o)[0], o + (1 << _SHIFT[t])


def header_keys(text):
    """n_sample and the GT key of a header text, restated: PASS = 0, FILTER / INFO / FORMAT IDs numbered by first appearance
    unless IDX= is given."""
    import re
    d, nxt, gt, ns = {"PASS": 0}, 1, None, 0
    for line in text.split("\n"):
        if line.startswith("#CHROM"):
            ns = max(0, line.count("\t") - 8)
        m = re.match(r"##(FILTER|INFO|FORMAT)=<ID=([^,>]+)", line)
        if not m:
            continue
        i = m.group(2)
        if i not in d:
            mi = re.search(r",IDX=(\d+)>?$", line)
            d[i] = int(mi.group(1)) if mi else nxt
        nxt = max(nxt, d[i] + 1)
        if m.group(1) == "FORMAT" and i == "GT":
            gt = d[i]
    return ns, gt


def py_decode(data):
    """Inflated BCF bytes -> header (n_sample, gt_key) and per record (chrom, pos0, a0 code, a1 code, alt_sum, biallelic, n_hap)."""
    import struct
    assert data[:4] == b"BCF\2" and data[4] in (1, 2)
    l_text = struct.unpack_from("<I", data, 5)[0]
    ns, gt_key = header_keys(data[9:9 + l_text].split(b"\0")[0].decode())
    o = 9 + l_text
    recs = []
    code = lambda a: 0 if len(a) == 0 else a[0] if len(a) == 1 else 0xFF
    while o < len(data):
        ls, li = struct.unpack_from("<II", data, o)
        s = o + 8
        chrom, pos = struct.unpack_from("<ii", data, s)
        nai, nfs = struct.unpack_from("<II", data, s + 16)
        n_allele, n_fmt, n_sample = nai >> 16, nfs >> 24, nfs & 0xFFFFFF
        p = s + 24
        t, n, p = _typed(data, p)
        p += n << _SHIFT[t]                                                   # ID
        al = []
        for _ in range(n_allele):
            t, n, p = _typed(data, p)
            al.append(data[p:p + n])
            p += n
        f = s + ls
        gt = None
        for _ in range(n_fmt):
            key, f = _int(data, f)
            t, n, f = _typed(data, f)
            nb = (n_sample * n) << _SHIFT[t]
            if key == gt_key:
                gt = struct.unpack_from("<%d%s" % (n_sample * n, _FMT[t]), data, f)
            f += nb
        idx = [(v >> 1) - 1 for v in gt]
        recs.append((chrom, pos, code(al[0]) if al else 0, code(al[1]) if len(al) > 1 else 0, sum(idx), max(idx) <= 1, len(gt)))
        o = s + ls + li
    return ns, gt_key, recs


# ---- random records of every shape ------------------------------------------------------------------------------------------
IDS = [("INFO", "DP"), ("FILTER", "q10"), ("INFO", "AF"), ("FORMAT", "GQ"), ("INFO", "DB"), ("INFO", "ANN"), ("FORMAT", "GT"),
       ("FILTER", "s50"), ("INFO", "BIG"), ("FORMAT", "AD"), ("FORMAT", "FT")]
IDX_SHUFFLED = {"PASS": 0, "DP": 7, "q10": 3, "AF": 12, "GQ": 2, "DB": 9, "ANN": 1, "GT": 5, "s50": 4, "BIG": 11, "AD": 8, "FT": 6}


def keys_of(idx):
    if idx is not None:
        return dict(idx)
    d = {"PASS": 0}
    for _, i in IDS:
        d.setdefault(i, len(d))
    return d


def random_records(rng, n, n_sample, ploidy=2, gt_type=1, idx=None, pos_step=(0, 40), chrom=0, alleles=None, extras=True):
    """n records with rich shared parts (long IDs, FILTER lists, INFO fields of every type with overflow sizes and flags),
    FORMAT fields before and after GT, repeated positions, 1-4 alleles (multi-letter and symbolic ones among them), phased and
    unphased GT of the given type.  Returns the record bytes and, per record, (pos0, alleles, allele indices per haplotype)."""
    from colate_b200 import synth
    k = keys_of(idx)
    out, recs = [], []
    p = int(rng.integers(0, 100))
    letters = [b"A", b"C", b"G", b"T"]
    for r in range(n):
        p += int(rng.integers(*pos_step))
        if alleles is not None:
            al = alleles(rng, r)
        else:
            na = int(rng.choice([1, 2, 2, 2, 3, 4]))
            al = [letters[int(x)] for x in rng.permutation(4)[:na]]
            if rng.random() < 0.1:
                al[-1] = rng.choice([b"ACGT", b"<DEL>", b"*", b"GATTACA" * 3])
        na = max(1, len(al))
        gt = rng.integers(0, na, (n_sample, ploidy))
        if na > 1 and rng.random() < 0.5:
            gt = np.minimum(gt, 1)
        phased = bool(rng.random() < 0.5)
        info, filters, before, after = [], [], [], []
        rid = b"."
        if extras:
            rid = b"rs%d" % r * int(rng.choice([1, 1, 5, 40]))
            filters = list(rng.choice([0, k["q10"], k["s50"]], int(rng.integers(0, 3)), replace=False))
            if rng.random() < 0.7:
                info.append((k["DP"], synth.bcf_typed_ints([int(rng.choice([3, 300, 70000]))])))
            if rng.random() < 0.5:
                info.append((k["AF"], synth.bcf_typed_floats(list(rng.random(na - 1 or 1)))))
            if rng.random() < 0.3:
                info.append((k["DB"], synth.BCF_FLAG))
            if rng.random() < 0.4:
                info.append((k["ANN"], synth.bcf_typed_str(b"x|y" * int(rng.integers(1, 30)))))
            if rng.random() < 0.3:
                info.append((k["BIG"], synth.bcf_typed_ints(list(rng.integers(-5, 40000, int(rng.integers(15, 40)))))))
            before = [(k["GQ"], int(rng.choice([1, 2])), [[int(x)] for x in rng.integers(0, 99, n_sample)])]
            after = [(k["AD"], 3, [list(rng.integers(0, 1000, 2)) for _ in range(n_sample)]),
                     (k["FT"], 7, [b"PASS" if rng.random() < 0.5 else b"q10;s50" for _ in range(n_sample)])]
        out.append(synth.bcf_record(chrom, p, al, gt.tolist(), k["GT"], phased=phased, gt_type=gt_type, rid=rid, filters=filters,
                                    info=info, fmt_before=before, fmt_after=after))
        recs.append((p, al, gt.reshape(-1).tolist()))
    return out, recs
