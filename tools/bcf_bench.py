"""BCF input at reference-panel size on one GPU: one chromosome with a panel BCF of ~1 M records x 1,000 diploid samples (about
2 GB inflated, mostly the GT vectors) and a one-sample target BCF at the same sites, written with synth.bcf_records_np and BGZF
level 1.  Times, in one process:
  1. the whole CLI: `Colate --mode mut --chr --target_bcf --reference_bcf` (files -> .colate_mat / .coal / .bin), twice;
  2. Handle.rows_from_bcf on the panel, wall time, for several host inflate thread counts;
  3. the same with bcf_timing on: BGZF index, inflate, record walk, host-to-device copies, k_bcf_decode (with its rate over the
     record bytes) and k_bcf_rows, for both files.
  4. the text-VCF leg: the same records as bgzipped VCF text (synth.vcf_lines_np, GT the only FORMAT field, '|' or '/' at
     random), read through the same flags: the CLI wall time, the phases with k_vcf_decode's rate over the text bytes, and a
     check that both formats gave identical row counts.
Prints the GPU's name and power limit with the numbers.
usage: bcf_bench.py [--records 1000000] [--samples 1000] [--rows 400000] [--threads 1,4,16,32] [--no-vcf] [--out DIR]"""
import argparse, json, os, shutil, subprocess, sys, tempfile, time
from concurrent.futures import ThreadPoolExecutor
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colate_b200 import api, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")
ap = argparse.ArgumentParser()
ap.add_argument("--records", type=int, default=1_000_000)
ap.add_argument("--samples", type=int, default=1000)
ap.add_argument("--rows", type=int, default=400_000)
ap.add_argument("--threads", default="1,4,16,32")
ap.add_argument("--out", default=None, help="directory for the JSON result")
ap.add_argument("--no-vcf", action="store_true", help="skip the text-VCF leg")
a = ap.parse_args()

try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
except FileNotFoundError:
    gpu = ""
gpu = gpu.splitlines()[0] if gpu else "unknown"
print("GPU:", gpu, "| host CPUs:", os.cpu_count(), flush=True)
res = {"gpu": gpu, "host_cpus": os.cpu_count()}
t0 = time.time()
L = 249_000_000
sites = synth.make_sites(1, [a.rows], [L])
d = tempfile.mkdtemp(prefix="colate_bcf_bench_")
with open(d + "/chr.txt", "w") as f:
    f.write("1\n")
synth.mut_texts_fast(sites)[0].tofile(f"{d}/syn_chr1.mut")
pool = ThreadPoolExecutor(os.cpu_count() or 8)
gt_key = 1
rng = np.random.default_rng(3)
# record positions: most rows carry a record, the rest lie between rows; alleles are the row's (either order) or others
at_rows = sites.pos[rng.random(sites.n) < 0.9] - 1
pos0 = np.sort(np.concatenate([at_rows, rng.integers(0, L, max(0, a.records - at_rows.shape[0]))]))[:a.records].astype(np.int32)
n = pos0.shape[0]
m = np.minimum(np.searchsorted(sites.pos, pos0 + 1), sites.n - 1)
sw = rng.random(n) < 0.5
a0 = np.where(sw, sites.der[m], sites.anc[m]).astype(np.uint8)
a1 = np.where(sw, sites.anc[m], sites.der[m]).astype(np.uint8)


def write_bcf(path, n_sample, seed, vcf=False):
    """Records in batches, streamed through BGZF blocks of 65280 bytes (level 1).  Allele frequencies are mostly low, as in a panel.
    vcf: the same records (same seed) as VCF text."""
    r = np.random.default_rng(seed)
    tot = 0
    with open(path, "wb") as f:
        pending = bytearray(synth.vcf_header(n_sample) if vcf else synth.bcf_header(n_sample))

        def flush(final=False):
            nonlocal pending, tot
            cut = len(pending) if final else len(pending) // 65280 * 65280
            pieces = [bytes(pending[i:i + 65280]) for i in range(0, cut, 65280)]
            for b in pool.map(lambda p: synth.bgzf_block(p, 1), pieces):
                f.write(b)
            tot += cut
            del pending[:cut]
        step = max(1, (1 << 27) // (2 * n_sample))
        for b0 in range(0, n, step):
            k = min(n, b0 + step) - b0
            af = (r.beta(0.3, 3.0, (k, 1)) * 256).astype(np.uint8)
            allele = (r.integers(0, 256, (k, 2 * n_sample), dtype=np.uint8) < af).view(np.int8)
            gt = ((allele + 1) << 1) | (np.array([0, 1] * n_sample, np.int8) & r.integers(0, 2, (1, 2 * n_sample), dtype=np.int8))
            if vcf:
                pending += synth.vcf_lines_np(pos0[b0:b0 + k], a0[b0:b0 + k], a1[b0:b0 + k], allele, (gt[:, 1::2] & 1) != 0).tobytes()
            else:
                pending += synth.bcf_records_np(pos0[b0:b0 + k], a0[b0:b0 + k], a1[b0:b0 + k], gt.astype(np.int8), gt_key).tobytes()
            flush()
        flush(final=True)
        f.write(synth.BGZF_EOF)
    return tot


sizes = {}
for tag, ns, seed in (("r", a.samples, 12), ("t", 1, 11)):
    sizes[tag] = write_bcf(f"{d}/{tag}_chr1.bcf", ns, seed)
    sizes[tag + "_file"] = os.path.getsize(f"{d}/{tag}_chr1.bcf")
res["dataset"] = {"rows": int(sites.n), "records": int(n), "panel_samples": a.samples, "panel_inflated_bytes": sizes["r"],
                  "panel_file_bytes": sizes["r_file"], "target_inflated_bytes": sizes["t"], "target_file_bytes": sizes["t_file"],
                  "written_s": round(time.time() - t0, 1)}
print("dataset:", res["dataset"], flush=True)

# 1. the whole CLI (twice: the first run also reads the files into the page cache)
cli = [CLI, "--mode", "mut", "--mut", d + "/syn", "--chr", d + "/chr.txt", "--target_bcf", d + "/t", "--reference_bcf", d + "/r",
       "--bins", "3,7,0.2", "--seed", "1", "--num_bootstraps", "10"]
walls = []
for k in range(2):
    for ext in (".colate_mat", ".coal", ".bin"):
        if os.path.exists(f"{d}/cli{ext}"):
            os.remove(f"{d}/cli{ext}")
    t = time.time()
    p = subprocess.run(cli + ["-o", d + "/cli"], capture_output=True, text=True, env=dict(os.environ, COLATE_TIMING="1"))
    walls.append(time.time() - t)
    assert p.returncode == 0, p.stderr[-3000:]
res["cli_wall_s"] = [round(x, 3) for x in walls]
res["cli_timing_lines"] = [ln for ln in p.stderr.splitlines() if ln.startswith("[timing]")]
print("CLI wall:", res["cli_wall_s"], *res["cli_timing_lines"], sep="\n  ", flush=True)

# 2. rows_from_bcf on the panel, by inflate threads
h = api.Handle(0)
h.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
h.set_option("front_end", 1)
res["rows_from_bcf"] = []
for th in [int(x) for x in a.threads.split(",")]:
    os.environ["COLATE_BCF_THREADS"] = str(th)
    t = time.time()
    h.rows_from_bcf(1, [f"{d}/r_chr1.bcf"], "reference")
    wall = time.time() - t
    row = {"threads": th, "wall_s": round(wall, 3), **{k: round(v, 4) for k, v in h.last_bcf_timing().items()}}
    res["rows_from_bcf"].append(row)
    print("rows_from_bcf (panel)", row, flush=True)
os.environ.pop("COLATE_BCF_THREADS")

# 3. phases with bcf_timing on (waits after every window: a breakdown, not a wall time)
h.set_option("bcf_timing", 1)
res["phases"] = []
for slot, tag, role in ((1, "r", "reference"), (0, "t", "target")):
    h.rows_from_bcf(slot, [f"{d}/{tag}_chr1.bcf"], role)
    tm = h.last_bcf_timing()
    rec_bytes = sizes[tag] - len(synth.bcf_header(a.samples if tag == "r" else 1))
    tm["decode_GBps"] = rec_bytes / (tm["decode_ms"] * 1e-3) / 1e9 if tm["decode_ms"] > 0 else 0.0
    tm["decode_share_of_7.7TBps"] = tm["decode_GBps"] / 7700.0
    res["phases"].append({"file": tag, **{k: round(v, 4) for k, v in tm.items()}})
    print("phases (bcf_timing on)", res["phases"][-1], flush=True)
h.set_option("bcf_timing", 0)
t = time.time()
s1 = h.stage1(api.mt_seed(1))
res["stage1_s"] = round(time.time() - t, 3)
res["used_rows"] = int(s1.n_used)
print("stage i:", res["stage1_s"], "s, used rows", s1.n_used, flush=True)

# 4. the text-VCF leg on the same records
if not a.no_vcf:
    bcf_rows = {}
    for slot, tag, role in ((1, "r", "reference"), (0, "t", "target")):
        bcf_rows[tag] = h.rows_from_bcf(slot, [f"{d}/{tag}_chr1.bcf"], role, fetch=True)
    t0 = time.time()
    for tag, ns, seed in (("r", a.samples, 12), ("t", 1, 11)):
        sizes[tag + "v"] = write_bcf(f"{d}/{tag}v_chr1.bcf", ns, seed, vcf=True)
        sizes[tag + "v_file"] = os.path.getsize(f"{d}/{tag}v_chr1.bcf")
    res["vcf_dataset"] = {"panel_inflated_bytes": sizes["rv"], "panel_file_bytes": sizes["rv_file"], "target_inflated_bytes": sizes["tv"],
                          "target_file_bytes": sizes["tv_file"], "written_s": round(time.time() - t0, 1)}
    print("vcf dataset:", res["vcf_dataset"], flush=True)
    walls = []
    for k in range(2):
        t = time.time()
        p = subprocess.run([x if x not in (d + "/t", d + "/r") else x + "v" for x in cli] + ["-o", d + "/cliv"], capture_output=True, text=True,
                           env=dict(os.environ, COLATE_TIMING="1"))
        walls.append(time.time() - t)
        assert p.returncode == 0, p.stderr[-3000:]
    res["vcf_cli_wall_s"] = [round(x, 3) for x in walls]
    res["vcf_cli_same_files"] = all(open(f"{d}/cli{e}", "rb").read() == open(f"{d}/cliv{e}", "rb").read() for e in (".colate_mat", ".coal", ".bin"))
    print("VCF CLI wall:", res["vcf_cli_wall_s"], "same .colate_mat/.coal/.bin as BCF:", res["vcf_cli_same_files"], flush=True)
    h.set_option("bcf_timing", 1)
    h.set_option("vcf_paths", 1)
    res["vcf_phases"] = []
    same = True
    for slot, tag, role in ((1, "r", "reference"), (0, "t", "target")):
        got = h.rows_from_bcf(slot, [f"{d}/{tag}v_chr1.bcf"], role, fetch=True)
        same &= all(np.array_equal(x, y) for x, y in zip(got, bcf_rows[tag]))
        tm = h.last_bcf_timing()
        text_bytes = sizes[tag + "v"] - len(synth.vcf_header(a.samples if tag == "r" else 1))
        tm["decode_GBps"] = text_bytes / (tm["decode_ms"] * 1e-3) / 1e9 if tm["decode_ms"] > 0 else 0.0
        tm["decode_share_of_7.7TBps"] = tm["decode_GBps"] / 7700.0
        tm["fast_lines"], tm["general_lines"] = h.last_vcf_paths()
        res["vcf_phases"].append({"file": tag, **{k: round(v, 4) for k, v in tm.items()}})
        print("vcf phases (bcf_timing on)", res["vcf_phases"][-1], flush=True)
    h.set_option("bcf_timing", 0)
    h.set_option("vcf_paths", 0)
    res["vcf_rows_identical"] = bool(same)
    print("row counts identical for BCF and VCF:", same, flush=True)
h.close()
if a.out:
    os.makedirs(a.out, exist_ok=True)
    json.dump(res, open(os.path.join(a.out, "bcf_bench.json"), "w"), indent=1)
shutil.rmtree(d, ignore_errors=True)
