"""A cohort at whole-genome size on one GPU: T ancient targets (ages spread over 1-10 kyr, sparse records, a mask each) against
F references, every (target, reference) pair with R bootstrap replicates.  Times, in one process:
  1. the cohort CLI end to end (`Colate --mode mut --pairs`, files -> .coal / .bin of every pair);
  2. pairs.cohort from in-memory arrays, phases split (stages i+ii of every pair; the EM of all replicates on mixed grids);
  3. the single-pair CLI, one process per pair, on the first `--loop` pairs (the loop is long: its per-pair time is
     extrapolated to the cohort and the output says so); its .coal / .bin are compared with the cohort CLI's byte for byte.
Reports pair-site evaluations/s (P x N_site / wall) and EM replicate-iterations/s beside the GPU's name and power limit.
usage: cohort_bench.py [--rows 10000000] [--targets 8] [--refs 24] [--R 10] [--loop 4]"""
import argparse, os, shutil, subprocess, sys, tempfile, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colate_b200 import api, pairs, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")
ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=10_000_000)
ap.add_argument("--targets", type=int, default=8)
ap.add_argument("--refs", type=int, default=24)
ap.add_argument("--R", type=int, default=10)
ap.add_argument("--loop", type=int, default=4)
ap.add_argument("--mask-len", type=int, default=3_000_000, help="bases masked at the start of every chromosome (beyond: callable)")
a = ap.parse_args()

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("GPU:", gpu.splitlines()[0] if gpu else "unknown", flush=True)
t0 = time.time()
sites = synth.make_sites(1, synth.rows_for_genome(a.rows), synth.AUTOSOME_LEN)
targets = [synth.make_genome(2000 + k, sites, 0.15) for k in range(a.targets)]       # ~0.5x coverage: sparse records
refs = [synth.make_genome(3000 + k, sites, 0.35) for k in range(a.refs)]
masks = [[synth.make_mask(4000 + 100 * k + c, min(a.mask_len, int(L)), 0.4) for c, L in enumerate(sites.chrom_len)] for k in range(a.targets)]
ages = [int(x) for x in np.linspace(1000, 10000, a.targets)]                         # years
d = tempfile.mkdtemp(prefix="colate_cohort_bench_")
with open(d + "/chr.txt", "w") as f:
    f.write("".join(nm + "\n" for nm in sites.chr_names))
for c, (nm, txt) in enumerate(zip(sites.chr_names, synth.mut_texts_fast(sites))):
    txt.tofile(f"{d}/syn_chr{nm}.mut")
for k, g in enumerate(targets):
    synth.write_colate_in_fast(f"{d}/t{k}.colate.in", g, sites.chr_names)
    for c, nm in enumerate(sites.chr_names):
        synth.write_mask(f"{d}/m{k}_chr{nm}.fa", masks[k][c])
for k, g in enumerate(refs):
    synth.write_colate_in_fast(f"{d}/r{k}.colate.in", g, sites.chr_names)
plist = [(t, r) for t in range(a.targets) for r in range(a.refs)]
P = len(plist)
lines = [f"{d}/t{t}.colate.in {d}/r{r}.colate.in {d}/out_{t}_{r} target_age={ages[t]} reference_age=0 target_mask={d}/m{t}" for t, r in plist]
with open(d + "/pairs.txt", "w") as f:
    f.write("\n".join(lines) + "\n")
print("dataset: %d sites, %d targets x %d references = %d pairs, R = %d, written in %.0f s" % (sites.n, a.targets, a.refs, P, a.R, time.time() - t0), flush=True)
shared = ["--mode", "mut", "--mut", d + "/syn", "--chr", d + "/chr.txt", "--seed", "1", "--bins", "3,7,0.1", "--num_bootstraps", str(a.R),
          "--years_per_gen", "28"]


def iters_of(prefix):
    raw = open(prefix + ".bin", "rb").read()
    R, E = np.frombuffer(raw[8:16], np.int32)
    return np.frombuffer(raw[16 + 8 * E + 8 * R * E:], np.int32)


# 1. the cohort CLI, twice (the first run also pays the page cache of the inputs)
walls = []
for rep in range(2):
    t0 = time.perf_counter()
    r = subprocess.run([CLI] + shared + ["--pairs", d + "/pairs.txt"], capture_output=True, text=True)
    walls.append(time.perf_counter() - t0)
    assert r.returncode == 0, r.stderr[-3000:]
t_cli = min(walls)
it_cli = sum(int(iters_of(f"{d}/out_{t}_{r}").sum()) for t, r in plist)
print("cohort CLI: %.2f s wall (runs: %s) | %.3e pair-site evaluations/s | %d EM replicate-iterations in all"
      % (t_cli, ", ".join("%.2f" % w for w in walls), P * sites.n / t_cli, it_cli), flush=True)

# 2. pairs.cohort from arrays, phases split
h = api.Handle(0)
t0 = time.perf_counter()
h.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
for k, g in enumerate(targets + refs):
    h.set_genome(k, g.chrom, g.bp, g.aaf, g.daf, g.anc.astype(np.uint16) | (g.der.astype(np.uint16) << 8))
    h.set_mask(k, api.mask_bits_from_seq(masks[k], sites.site_off, sites.pos) if k < a.targets else None)
t_load = time.perf_counter() - t0
cp = [(t, a.targets + r, str(ages[t]), "0") for t, r in plist]
for rep in range(2):                                   # the first pass also joins every genome once
    res = pairs.cohort(h, cp, seed=1, bins="3,7,0.1", num_bootstraps=a.R, years_per_gen=28.0)
sec = res["seconds"]
it_api = sum(int(p["iters"].sum()) for p in res["pairs"])
grids = len({p["epochs"].tobytes() for p in res["pairs"]})
print("pairs.cohort: load %.2f s | stage i+ii %.3f s (%.2f ms/pair) | EM of %d replicates on %d grids %.3f s: %.3e replicate-iterations/s | "
      "total %.3f s: %.3e pair-site evaluations/s"
      % (t_load, sec["stage12"], 1e3 * sec["stage12"] / P, P * a.R, grids, sec["em"], it_api / sec["em"], sec["stage12"] + sec["em"],
         P * sites.n / (sec["stage12"] + sec["em"])), flush=True)
same = all(np.array_equal(p["iters"], iters_of(f"{d}/out_{t}_{r}")) for p, (t, r) in zip(res["pairs"], plist))
print("pairs.cohort iterations == cohort CLI iterations on every pair:", same, flush=True)
h.close()

# 3. the single-pair CLI in a loop over the first pairs
n_loop = min(a.loop, P)
t0 = time.perf_counter()
identical = True
for k in range(n_loop):
    t, r = plist[k]
    out = f"{d}/single_{t}_{r}"
    q = subprocess.run([CLI] + shared + ["--target_tmp", f"{d}/t{t}.colate.in", "--reference_tmp", f"{d}/r{r}.colate.in", "--target_age", str(ages[t]),
                        "--reference_age", "0", "--target_mask", f"{d}/m{t}", "-o", out], capture_output=True, text=True)
    assert q.returncode == 0, q.stderr[-3000:]
    for ext in (".coal", ".bin"):
        identical &= open(out + ext, "rb").read() == open(f"{d}/out_{t}_{r}{ext}", "rb").read()
t_loop = time.perf_counter() - t0
per = t_loop / n_loop
print("single-pair CLI loop: %d of %d pairs in %.2f s (%.2f s/pair; extrapolated to all %d pairs: %.0f s, %.3e pair-site evaluations/s) | "
      "outputs byte-identical to the cohort CLI: %s" % (n_loop, P, t_loop, per, P, per * P, sites.n / per, identical))
print("cohort CLI speed-up over the extrapolated loop: %.1fx" % (per * P / t_cli))
shutil.rmtree(d, ignore_errors=True)
