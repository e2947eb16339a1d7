"""No GPU: `Colate --mode mut --pairs <file>` refuses malformed pairs files and conflicting flags before it touches a device,
naming the offending line; and the mixed-grid EM kernel left the existing throughput kernel `k_em_cta` as it was."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")
LIB = os.path.join(ROOT, "colate_b200", "libcolate_b200.so")


@pytest.fixture()
def cohort_dir(built, tmp_path):
    for i in range(70):
        (tmp_path / f"g{i}.colate.in").write_bytes(b"")
    (tmp_path / "syn.mut").write_text("")
    return tmp_path


def run_pairs(d, lines, *flags):
    pf = d / "pairs.txt"
    pf.write_text("".join(x + "\n" for x in lines))
    base = ["--mode", "mut", "--mut", str(d / "syn.mut"), "--pairs", str(pf)]
    if "--no-seed" not in flags:
        base += ["--seed", "1"]
    if not any(f in flags for f in ("--bins", "--coal")):
        base += ["--bins", "3,7,0.2"]
    r = subprocess.run([CLI] + base + [f for f in flags if f != "--no-seed"], capture_output=True, text=True, timeout=60)
    return r


def refused(r, *needles):
    assert r.returncode != 0, r.stderr
    for n in needles:
        assert n in r.stderr, (n, r.stderr)
    # nothing got as far as a device (on this machine there is none: that would read "no CUDA device")
    assert "CUDA" not in r.stderr and "device" not in r.stderr.lower().replace("--devices", ""), r.stderr
    return r.stderr


def g(d, i):
    return str(d / f"g{i}.colate.in")


def test_too_few_fields(cohort_dir):
    d = cohort_dir
    refused(run_pairs(d, ["# header", f"{g(d, 0)} {g(d, 1)} {d}/o0", "", f"{g(d, 0)} {g(d, 2)}"]), "line 4", "found 2 field(s)")


@pytest.mark.parametrize("field", ["target_age7000", "=7000", "target_age=", "7000"])
def test_key_value_syntax(cohort_dir, field):
    d = cohort_dir
    refused(run_pairs(d, [f"{g(d, 0)} {g(d, 1)} {d}/o0 target_age=100", f"{g(d, 0)} {g(d, 1)} {d}/o1 {field}"]), "line 2", "key=value")


def test_unknown_and_repeated_keys(cohort_dir):
    d = cohort_dir
    refused(run_pairs(d, [f"{g(d, 0)} {g(d, 1)} {d}/o0 seed=3"]), "line 1", "unknown key 'seed'")
    refused(run_pairs(d, [f"{g(d, 0)} {g(d, 1)} {d}/o0 target_age=1 target_age=2"]), "line 1", "given twice")


def test_duplicate_output_prefix(cohort_dir):
    d = cohort_dir
    err = refused(run_pairs(d, [f"{g(d, 0)} {g(d, 1)} {d}/same", "   # indented comment", f"{g(d, 2)} {g(d, 3)} {d}/same"]), "line 3")
    assert "line 1" in err


def test_unreadable_colate_in(cohort_dir):
    d = cohort_dir
    refused(run_pairs(d, [f"{g(d, 0)} {g(d, 1)} {d}/o0", f"{g(d, 0)} {d}/missing.colate.in {d}/o1"]), "line 2", "missing.colate.in")


def test_more_genomes_than_slots(cohort_dir):
    d = cohort_dir
    lines = [f"{g(d, 2 * k)} {g(d, 2 * k + 1)} {d}/o{k}" for k in range(32)]          # 64 genomes: fine so far
    # the same file under a mask is another genome (another slot): the 65th
    refused(run_pairs(d, lines + [f"{g(d, 0)} {g(d, 1)} {d}/o_masked target_mask={d}/m"]), "line 33", "more than 64")
    refused(run_pairs(d, lines + [f"{g(d, 64)} {g(d, 1)} {d}/o_new"]), "line 33", "more than 64")


@pytest.mark.parametrize("flag", [["--target_tmp", "x"], ["--reference_tmp", "x"], ["-o", "x"], ["--target_age", "100"],
                                  ["--reference_age", "100"], ["--target_mask", "m"], ["--reference_mask", "m"]])
def test_single_pair_flags_are_refused(cohort_dir, flag):
    d = cohort_dir
    refused(run_pairs(d, [f"{g(d, 0)} {g(d, 1)} {d}/o0"], *flag), "cannot be combined with --pairs")


def test_seed_is_required(cohort_dir):
    d = cohort_dir
    refused(run_pairs(d, [f"{g(d, 0)} {g(d, 1)} {d}/o0"], "--no-seed"), "--seed")


def test_nothing_is_written(cohort_dir):
    d = cohort_dir
    run_pairs(d, [f"{g(d, 0)} {g(d, 1)} {d}/o0", f"{g(d, 2)} {g(d, 3)} {d}/o1 bad"])
    assert not any(p.name.startswith("o") for p in d.iterdir())


# k_em_cta of the parent commit (the throughput-mode EM before the mixed-grid form shared its body): registers and SASS
# instructions of the sm_100a build (CUDA 12.9).  The uniform kernel must compile to the same code.
K_EM_CTA = "_ZN6colate8k_em_ctaEiiPKdS1_S1_S1_iPKmS3_PdPiS4_Px"
K_EM_CTA_REGS, K_EM_CTA_INSTRUCTIONS = 94, 5040


def test_k_em_cta_code_unchanged(built):
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump is not installed")
    res = subprocess.run([tool, "-res-usage", LIB], capture_output=True, text=True).stdout
    m = re.search(r"Function " + K_EM_CTA + r":\s*\n\s*REG:(\d+)", res)
    assert m, "k_em_cta not found in the library"
    assert int(m.group(1)) == K_EM_CTA_REGS
    sass = subprocess.run([tool, "-sass", LIB], capture_output=True, text=True).stdout
    body = sass.split("Function : " + K_EM_CTA + "\n", 1)[1].split("\n\t\t..........", 1)[0]
    n = sum(1 for ln in body.split("\n") if re.match(r"\s+/\*[0-9a-f]{4,}\*/\s", ln))
    assert n == K_EM_CTA_INSTRUCTIONS
