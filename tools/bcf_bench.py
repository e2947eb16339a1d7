"""BCF input at reference-panel size on one GPU: one chromosome with a panel BCF of ~1 M records x 1,000 diploid samples (about
2 GB inflated, mostly the GT vectors) and a one-sample target BCF at the same sites, written with synth.bcf_records_np and BGZF
level 1.  Times, in one process:
  1. the whole CLI: `Colate --mode mut --chr --target_bcf --reference_bcf` (files -> .colate_mat / .coal / .bin), twice;
  2. Handle.rows_from_bcf on the panel, wall time, for several host inflate thread counts;
  3. the same with bcf_timing on: BGZF index, inflate, record walk, host-to-device copies, k_bcf_decode (with its rate over the
     record bytes) and k_bcf_rows, for both files.
Prints the GPU's name and power limit with the numbers.
usage: bcf_bench.py [--records 1000000] [--samples 1000] [--rows 400000] [--threads 1,4,16,32] [--out DIR]"""
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


def write_bcf(path, n_sample, seed):
    """Records in batches, streamed through BGZF blocks of 65280 bytes (level 1).  Allele frequencies are mostly low, as in a panel."""
    r = np.random.default_rng(seed)
    tot = 0
    with open(path, "wb") as f:
        pending = bytearray(synth.bcf_header(n_sample))

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
h.close()
if a.out:
    os.makedirs(a.out, exist_ok=True)
    json.dump(res, open(os.path.join(a.out, "bcf_bench.json"), "w"), indent=1)
shutil.rmtree(d, ignore_errors=True)
