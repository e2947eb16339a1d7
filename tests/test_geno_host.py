"""No GPU: genotype matrices for make_tmp (DESIGN.md section 6l).  colate_geno_scan agrees with a numpy parse of all three layouts
and refuses every malformed file with its message and line; `Colate --mode make_tmp --target_geno / --target_bed --individuals`
refuses malformed individuals files and conflicting flags before it touches a device; the new kernels compile without spills."""
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from colate_b200 import _lib, api

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import geno_helpers as gh  # noqa: E402

ROOT = os.path.dirname(HERE)
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")
CSRC = os.path.join(ROOT, "colate_b200", "csrc")


@pytest.fixture(scope="module")
def case(built, tmp_path_factory):
    d = str(tmp_path_factory.mktemp("geno"))
    c = gh.make_case(d, 5, n_ind=37)
    return d, c, gh.write_all(d, c)


def _numpy_parse(path, fmt, kind, n_ind, n_snp):
    """[n_snp, n_ind] codes (0 hom first, 1 hom second, 2 het, 3 missing) read back with numpy."""
    raw = np.fromfile(path, np.uint8)
    if kind == "text":
        d = raw.reshape(n_snp, n_ind + 1)[:, :n_ind]
        return np.select([d == ord("2"), d == ord("0"), d == ord("1")], [0, 1, 2], 3)
    nb = (n_ind + 3) // 4
    if kind == "bed":
        b = raw[3:].reshape(n_snp, nb)
        v = np.stack([(b >> (2 * j)) & 3 for j in range(4)], axis=2).reshape(n_snp, -1)[:, :n_ind]
        return np.array([0, 3, 2, 1])[v]
    rlen = max(48, nb)
    b = raw[rlen:].reshape(n_snp, rlen)[:, :nb]
    v = np.stack([(b >> (6 - 2 * j)) & 3 for j in range(4)], axis=2).reshape(n_snp, -1)[:, :n_ind]
    return np.array([1, 2, 0, 3])[v]


@pytest.mark.parametrize("layout", ["plink", "packed", "text"])
def test_scan_agrees_with_numpy(case, layout):
    d, c, p = case
    fmt = "plink" if layout == "plink" else "eigenstrat"
    s = api.geno_scan(p[layout], fmt, gh.NAMES)
    assert s["kind"] == {"plink": "bed", "packed": "packed", "text": "text"}[layout]
    assert s["n_snp"] == len(c["snps"]) and s["n_ind"] == len(c["ids"])
    want = [sum(1 for x in c["snps"] if gh.ENTRY_OF[x[1]] == e) for e in range(len(gh.NAMES))]
    assert list(s["entry_snps"]) == want and min(want) > 0
    mat = p[layout] + (".bed" if layout == "plink" else ".geno")
    assert np.array_equal(_numpy_parse(mat, fmt, s["kind"], s["n_ind"], s["n_snp"]), c["calls"])


def test_contig_aliases(case):
    d, c, p = case
    s = api.geno_scan(p["plink"], "plink", ["X", "4", "1", "23", "Y", "chr5"])
    n1, n23 = (sum(1 for x in c["snps"] if x[1] == k) for k in ("chr1", "23"))
    assert list(s["entry_snps"]) == [n23, 50, n1, n23, 0, 0]      # X <- 23, 1 <- chr1; entry chr5 does not read contig 5


def _copy(p, layout, dst):
    exts = (".bed", ".bim", ".fam") if layout == "plink" else (".geno", ".snp", ".ind")
    for e in exts:
        shutil.copy(p[layout] + e, dst + e)
    return dst


def _refused(prefix, fmt, code, *needles, names=None):
    with pytest.raises(_lib.ColateError) as e:
        api.geno_scan(prefix, fmt, names or gh.NAMES)
    assert e.value.code == code, str(e.value)
    for n in needles:
        assert n in str(e.value), (n, str(e.value))


def test_refusals(case, tmp_path):
    d, c, p = case
    t = str(tmp_path)
    # .bed magic, individual-major .bed
    q = _copy(p, "plink", t + "/b1")
    raw = bytearray(open(q + ".bed", "rb").read())
    open(q + ".bed", "wb").write(b"\x6c\x1c" + raw[2:])
    _refused(q, "plink", -5, "bad magic")
    open(q + ".bed", "wb").write(b"\x6c\x1b\x00" + raw[3:])
    _refused(q, "plink", -5, "individual-major")
    open(q + ".bed", "wb").write(raw[:-1])
    _refused(q, "plink", -5, "bytes, but")
    # TGENO, header counts, size
    q = _copy(p, "packed", t + "/e1")
    raw = bytearray(open(q + ".geno", "rb").read())
    open(q + ".geno", "wb").write(b"TGENO" + raw[5:])
    _refused(q, "eigenstrat", -5, "TGENO")
    open(q + ".geno", "wb").write(raw.replace(f"GENO {len(c['ids'])} ".encode(), f"GENO {len(c['ids']) + 1} ".encode(), 1))
    _refused(q, "eigenstrat", -5, "header counts")
    open(q + ".geno", "wb").write(raw + b"\0")
    _refused(q, "eigenstrat", -5, "bytes, but")
    # text: a bad call, names its line
    q = _copy(p, "text", t + "/e2")
    raw = bytearray(open(q + ".geno", "rb").read())
    raw[(len(c["ids"]) + 1) * 4 + 3] = ord("5")
    open(q + ".geno", "wb").write(raw)
    _refused(q, "eigenstrat", -5, "e2.geno, line 5", "is not 0, 1, 2 or 9")
    # .snp: alleles missing, a position that is not an integer, SNPs descending within an entry
    q = _copy(p, "packed", t + "/e3")
    lines = open(q + ".snp").read().splitlines()
    open(q + ".snp", "w").write("\n".join(lines[:3] + ["\t".join(lines[3].split()[:4])] + lines[4:]) + "\n")
    _refused(q, "eigenstrat", -5, "e3.snp, line 4", "alleles missing")
    f = lines[3].split()
    open(q + ".snp", "w").write("\n".join(lines[:3] + ["\t".join(f[:3] + ["12.5"] + f[4:])] + lines[4:]) + "\n")
    _refused(q, "eigenstrat", -5, "e3.snp, line 4", "not an integer")
    open(q + ".snp", "w").write("\n".join(lines[:3] + [lines[4], lines[3]] + lines[5:]) + "\n")
    _refused(q, "eigenstrat", -6, "e3.snp, line 5", "descend")
    # the unlisted contig may descend: it is not read
    q = _copy(p, "plink", t + "/b2")
    bl = open(q + ".bim").read().splitlines()
    k = [i for i, x in enumerate(bl) if x.split()[0] == "4"]
    bl[k[0]], bl[k[1]] = bl[k[1]], bl[k[0]]
    open(q + ".bim", "w").write("\n".join(bl) + "\n")
    api.geno_scan(q, "plink", gh.NAMES)
    _refused(q, "plink", -6, f"b2.bim, line {k[1] + 1}", names=gh.NAMES + ["4"])
    # .fam with too few fields, a missing file
    q = _copy(p, "plink", t + "/b3")
    open(q + ".fam", "a").write("f x 0\n")
    _refused(q, "plink", -5, f"b3.fam, line {len(c['ids']) + 1}", "expected 6 fields")
    q = _copy(p, "plink", t + "/b4")
    os.remove(q + ".bim")
    _refused(q, "plink", -5, "cannot read", "b4.bim")


# ---- the CLI: every refusal before a device is touched ---------------------------------------------------------------------------
def run_geno(case, lines, *flags, layout="plink"):
    d, c, p = case
    f = os.path.join(d, "ind.txt")
    open(f, "w").write("".join(x + "\n" for x in lines))
    cmd = [CLI, "--mode", "make_tmp", "--mut", f"{d}/syn", "--chr", f"{d}/chr.txt", "--ref_genome", f"{d}/g", "--individuals", f,
           "--target_bed" if layout == "plink" else "--target_geno", p[layout]]
    return subprocess.run(cmd + [str(x) for x in flags], capture_output=True, text=True, timeout=60)


def refused(r, *needles):
    assert r.returncode != 0, r.stderr
    for n in needles:
        assert n in r.stderr, (n, r.stderr)
    # nothing got as far as a device (on this machine there is none: that would read "no CUDA device")
    assert "CUDA" not in r.stderr and "colate_create" not in r.stderr, r.stderr
    return r.stderr


def test_cli_line_refusals(case):
    d, c, p = case
    ids = c["ids"]
    refused(run_geno(case, ["# header", f"{ids[0]} {d}/o0", "", f"{ids[1]}"]), "line 4", "found 1 field(s)")
    refused(run_geno(case, [f"{ids[0]} {d}/o0 target_mask={c['masks'][0]} x"]), "line 1", "found 4 field(s)")
    refused(run_geno(case, [f"{ids[0]} {d}/o0", f"{ids[1]} {d}/o1 target_mask"]), "line 2", "key=value")
    refused(run_geno(case, [f"{ids[0]} {d}/o0", f"{ids[1]} {d}/o1 target_age=10"]), "line 2", "unknown key 'target_age'")
    refused(run_geno(case, [f"{ids[0]} {d}/o0", f"nobody {d}/o1"]), "line 2", "individual nobody is not in", ".fam")
    refused(run_geno(case, [f"{ids[0]} {d}/o0", f"{ids[1]} {d}/o0"]), "line 2", "output prefix", "already used on line 1")
    refused(run_geno(case, [f"{ids[0]} {d}/o0", f"{ids[1]} {d}/o1 target_mask={d}/nomask"]), "line 2", "cannot read the mask", "nomask_chr1.fa")
    refused(run_geno(case, ["# nothing"]), "lists no individual")


def test_cli_duplicate_id(case, tmp_path):
    d, c, p = case
    q = _copy(p, "packed", str(tmp_path / "dup"))
    il = open(q + ".ind").read().splitlines()
    il[3] = il[3].replace(c["ids"][3], c["ids"][5])
    open(q + ".ind", "w").write("\n".join(il) + "\n")
    refused(run_geno((d, c, {"packed": q}), [f"{c['ids'][0]} {d}/o0", f"{c['ids'][5]} {d}/o1"], layout="packed"),
            "line 2", f"individual {c['ids'][5]} occurs 2 times")


def test_cli_file_refusals(case, tmp_path):
    d, c, p = case
    q = _copy(p, "plink", str(tmp_path / "im"))
    raw = open(q + ".bed", "rb").read()
    open(q + ".bed", "wb").write(raw[:2] + b"\x00" + raw[3:])
    refused(run_geno((d, c, {"plink": q}), [f"{c['ids'][0]} {d}/o0"]), "individual-major")
    q = _copy(p, "packed", str(tmp_path / "tg"))
    raw = open(q + ".geno", "rb").read()
    open(q + ".geno", "wb").write(b"TGENO" + raw[5:])
    refused(run_geno((d, c, {"packed": q}), [f"{c['ids'][0]} {d}/o0"], layout="packed"), "TGENO")


@pytest.mark.parametrize("extra, needle", [
    (["--targets", "t.txt"], "--targets cannot be combined with --target_bed"),
    (["--target_bam", "x.bam"], "--target_bam cannot be combined"),
    (["--target_bcf", "x"], "--target_bcf cannot be combined"),
    (["--target_table", "x"], "--target_table cannot be combined"),
    (["--target_mask", "x"], "--target_mask cannot be combined"),
    (["-o", "x"], "--output/-o cannot be combined"),
    (["--devices", "0,1"], "runs on one device"),
    (["--strandfilter"], "--strandfilter does not apply"),
    (["--filters", "20,30,10"], "--filters does not apply"),
    (["--target_geno", "x"], "give one of --target_geno and --target_bed"),
])
def test_cli_flag_refusals(case, extra, needle):
    d, c, p = case
    refused(run_geno(case, [f"{c['ids'][0]} {d}/o0"], *extra), needle)


def test_cli_required_flags(case):
    d, c, p = case
    f = os.path.join(d, "ind1.txt")
    open(f, "w").write(f"{c['ids'][0]} {d}/o0\n")
    base = {"--mut": f"{d}/syn", "--chr": f"{d}/chr.txt", "--ref_genome": f"{d}/g", "--individuals": f, "--target_bed": p["plink"]}
    for drop, needle in [("--individuals", "needs --individuals"), ("--mut", "needs --mut"), ("--ref_genome", "needs --ref_genome"),
                         ("--chr", "needs --chr"), ("--target_bed", "--individuals needs --target_geno or --target_bed")]:
        args = [x for k, v in base.items() if k != drop for x in (k, v)]
        refused(subprocess.run([CLI, "--mode", "make_tmp"] + args, capture_output=True, text=True, timeout=60), needle)
    args = [x for k, v in base.items() for x in (k, v if k != "--ref_genome" else f"{d}/nog")]
    refused(subprocess.run([CLI, "--mode", "make_tmp"] + args, capture_output=True, text=True, timeout=60), "cannot read", "nog_chr1.fa")


def test_help_has_usage():
    r = subprocess.run([CLI, "--help"], capture_output=True, text=True, timeout=60)
    assert "--target_geno <prefix> | --target_bed <prefix>" in r.stdout and "heterozygous" in r.stdout


# ---- the pin itself runs on the host: derived tables through colate_maketmp_table ---------------------------------------------------
def test_quirk_individual_writes_nothing_after_the_entry(case, tmp_path):
    """Individual 7 has no homozygous call on X: its table run writes records on entry 1 only."""
    d, c, p = case
    img = gh.pinned(d, c, 7, tmp_path / "q.colate.in")
    names = [nm for nm in gh.NAMES]
    chrom = api.read_colate_in(str(tmp_path / "q.colate.in"), names)[0]
    assert len(img) > 0 and set(np.unique(chrom).tolist()) == {0}


def test_kernels_compile_without_spills(built, tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--fmad=false", "-Xptxas", "-v", "-c",
                        os.path.join(CSRC, "kernels_geno.cu"), "-o", str(tmp_path / "k.o")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    names = re.findall(r"Compiling entry function '(\w+)'", r.stderr)
    assert sum(any(k in n for k in ("k_geno_join", "k_geno_called", "k_geno_rows")) for n in names) == 3, names
    assert re.findall(r"(\d+) bytes spill stores", r.stderr) and all(x == "0" for x in re.findall(r"(\d+) bytes spill stores", r.stderr))
    assert all(x == "0" for x in re.findall(r"(\d+) bytes spill loads", r.stderr))
