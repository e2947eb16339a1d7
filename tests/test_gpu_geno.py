"""make_tmp from genotype matrices (`--target_geno` / `--target_bed --individuals`, colate_maketmp_write_geno): every individual's
.colate.in must equal colate_maketmp_table on the table of its homozygous calls, byte for byte, for PLINK .bed, packed and text
EIGENSTRAT; a 20-line CLI job equals 20 `--target_table` runs; a failing line writes no file; the job parses the .mut text once and
uploads the matrix once."""
import os
import subprocess
import sys

import numpy as np
import pytest

from colate_b200 import api

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import geno_helpers as gh  # noqa: E402

CLI = os.path.join(os.path.dirname(HERE), "colate_b200", "bin", "Colate")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def case(built, tmp_path_factory):
    d = str(tmp_path_factory.mktemp("gpu_geno"))
    c = gh.make_case(d, 11, n_ind=200)
    return d, c, gh.write_all(d, c)


def _mask_bits(h, d, masks):
    pos = h.ingest_fetch()[0]
    off = np.concatenate([[0], np.cumsum([int(x) for x in h.rows])]).astype(np.int64)
    bits = np.zeros((len(masks), (int(off[-1]) + 31) // 32), np.uint32)
    for m, prefix in enumerate(masks):
        for c, nm in enumerate(gh.NAMES):
            api.maketmp_mask_bits(f"{prefix}_chr{nm}.fa", pos[off[c]:off[c + 1]], int(off[c]), bits[m])
    return bits


@pytest.fixture(scope="module")
def written(case, tmp_path_factory):
    """All 200 individuals written from each layout through one handle per layout; masks: none, m0 or m1 (shared by many)."""
    d, c, p = case
    out = str(tmp_path_factory.mktemp("gpu_geno_out"))
    n = len(c["ids"])
    mask_ids = np.array([k % 3 - 1 for k in range(n)], np.int32)
    res = {}
    for layout, prefix in p.items():
        h = api.Handle(0)
        try:
            h.rows = h.ingest_mut([open(f"{d}/syn_chr{nm}.mut", "rb").read() for nm in gh.NAMES])
            bits = _mask_bits(h, d, c["masks"])
            files = [f"{out}/{layout}_{k}.colate.in" for k in range(n)]
            r = h.maketmp_write_geno(prefix, "plink" if layout == "plink" else "eigenstrat", c["ids"], gh.NAMES, files, mask_ids, bits)
            r["files"] = files
            r["uploads"] = h.geno_upload_counts()
            r["counts"] = h.upload_counts()
            res[layout] = r
        finally:
            h.close()
    return out, mask_ids, res


@pytest.mark.parametrize("layout", ["plink", "packed", "text"])
def test_every_individual_equals_table_writer(case, written, layout):
    d, c, p = case
    out, mask_ids, res = written
    r = res[layout]
    assert r["failed"] == 0
    on_listed = np.array([gh.ENTRY_OF[x[1]] is not None for x in c["snps"]])
    assert np.array_equal(r["het_skipped"], (c["calls"][on_listed] == 2).sum(axis=0))
    assert r["cutoff"][7] == 1 and (r["cutoff"] == 3).sum() > 150
    n_rec = 0
    for k in range(len(c["ids"])):
        mask = c["masks"][mask_ids[k]] if mask_ids[k] >= 0 else None
        want = gh.pinned(d, c, k, f"{out}/{layout}_{k}.pinned", mask)
        got = open(r["files"][k], "rb").read()
        assert got == want, (layout, k, len(got), len(want))
        assert r["records"][k] * 19 == len(got)                     # 18 + one-letter names
        n_rec += r["records"][k]
    assert n_rec > 20000


def test_layouts_give_identical_files(case, written):
    d, c, p = case
    out, _, res = written
    for k in range(len(c["ids"])):
        a = open(res["plink"]["files"][k], "rb").read()
        assert a == open(res["packed"]["files"][k], "rb").read() == open(res["text"]["files"][k], "rb").read(), k


def test_parsed_and_uploaded_once(case, written):
    d, c, p = case
    _, _, res = written
    for layout, r in res.items():
        assert r["counts"]["mut_texts_parsed"] == len(gh.NAMES), layout
        assert r["uploads"]["matrix_uploads"] == 1, layout
        n_listed = sum(1 for x in c["snps"] if gh.ENTRY_OF[x[1]] is not None)
        row = {"plink": (200 + 3) // 4, "packed": 50, "text": 201}[layout]
        assert r["uploads"]["matrix_h2d_bytes"] == n_listed * row, layout


def _cli(*args, env=None):
    return subprocess.run([CLI] + [str(a) for a in args], capture_output=True, text=True, timeout=900, env=env)


def test_cli_job_equals_table_runs(case, tmp_path):
    d, c, p = case
    ks = list(range(0, 200, 10))
    lines = ["# id out mask"]
    for j, k in enumerate(ks):
        lines.append(f"{c['ids'][k]} {tmp_path}/g{k}" + (f" target_mask={c['masks'][j % 2]}" if j % 3 else ""))
    f = tmp_path / "ind.txt"
    f.write_text("\n".join(lines) + "\n")
    shared = ["--mode", "make_tmp", "--mut", f"{d}/syn", "--chr", f"{d}/chr.txt", "--ref_genome", f"{d}/g"]
    r = _cli(*shared, "--target_geno", p["packed"], "--individuals", f, env=dict(os.environ, COLATE_TIMING="1"))
    assert r.returncode == 0, r.stderr[-3000:]
    stat = [x for x in r.stderr.splitlines() if "matrix uploads" in x][0]
    assert f".mut texts parsed {len(gh.NAMES)} " in stat and "matrix uploads 1 " in stat, stat
    assert f"Warning: individual {c['ids'][0]}" not in r.stderr
    for j, k in enumerate(ks):
        tab = tmp_path / f"t{k}.txt"
        tab.write_text(gh.table_of(c, k))
        q = _cli(*shared, "--target_table", tab, *(["--target_mask", c["masks"][j % 2]] if j % 3 else []), "-o", tmp_path / f"t{k}")
        assert q.returncode == 0, q.stderr[-2000:]
        assert open(f"{tmp_path}/g{k}.colate.in", "rb").read() == open(f"{tmp_path}/t{k}.colate.in", "rb").read(), k
        assert f"individual on line {j + 2} ({c['ids'][k]} -> {tmp_path}/g{k}): " in r.stderr
    # individual 7's warning names the entry where its table runs dry
    f.write_text(f"{c['ids'][7]} {tmp_path}/w7\n")
    r = _cli(*shared, "--target_bed", p["plink"], "--individuals", f)
    assert r.returncode == 0 and f"Warning: individual {c['ids'][7]} (line 1) has no homozygous call on --chr entry X" in r.stderr, r.stderr


def test_failing_line_writes_no_file(case, tmp_path):
    d, c, p = case
    f = tmp_path / "ind.txt"
    f.write_text(f"{c['ids'][0]} {tmp_path}/ok0\n{c['ids'][1]} {tmp_path}/nodir/bad\n{c['ids'][2]} {tmp_path}/ok2\n")
    r = _cli("--mode", "make_tmp", "--mut", f"{d}/syn", "--chr", f"{d}/chr.txt", "--ref_genome", f"{d}/g", "--target_geno", p["text"],
             "--individuals", f)
    assert r.returncode == 1, r.stderr[-3000:]
    assert f"individual on line 2 ({c['ids'][1]} -> {tmp_path}/nodir/bad) FAILED" in r.stderr and "1 of 3 individuals failed" in r.stderr
    assert not os.path.exists(f"{tmp_path}/nodir/bad.colate.in")
    for k in (0, 2):
        assert open(f"{tmp_path}/ok{k}.colate.in", "rb").read() == gh.pinned(d, c, k, tmp_path / f"p{k}")
