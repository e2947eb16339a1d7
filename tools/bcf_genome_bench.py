"""Whole-genome BCF against the same records as 22 per-chromosome files, on one GPU: a synthetic 22-contig dataset
(synth.rows_for_genome rows) with a one-sample target (records at ~85% of the rows) and a --panel_samples diploid panel (records at
~50% of the rows), each written once as one whole-genome BCF (contigs in --chr order) and once as <prefix>_chr<c>.bcf.
  rows:     Handle.rows_from_bcf_genome(0, 1, whole) against Handle.rows_from_bcf_roles(0, 1, split), --reps times each, alternating;
            the two slots' rows are compared bit for bit.
  make_tmp: `Colate --mode make_tmp --targets` with the whole-genome line and with the split line; the line's decode+write time
            (COLATE_TIMING) and the .colate.in files compared byte for byte.
Prints the GPU's name and power limit, read in the same run, and one JSON line.
usage: bcf_genome_bench.py [--rows 10000000] [--panel_samples 100] [--reps 3] [--out DIR]"""
import argparse, ctypes as C, json, os, re, shutil, subprocess, sys, tempfile, time
from concurrent.futures import ThreadPoolExecutor
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colate_b200 import _lib, api, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")
ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=10_000_000)
ap.add_argument("--panel_samples", type=int, default=100)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--out", default=None, help="directory for the JSON result")
a = ap.parse_args()

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip() if shutil.which("nvidia-smi") else ""
gpu = gpu.splitlines()[0] if gpu else "unknown"
print("GPU:", gpu, "| host CPUs:", os.cpu_count(), flush=True)
res = {"gpu": gpu, "host_cpus": os.cpu_count(), "rows": a.rows}
sites = synth.make_sites(1, synth.rows_for_genome(a.rows), synth.AUTOSOME_LEN)
names = list(sites.chr_names)
d = tempfile.mkdtemp(prefix="colate_bcf_genome_bench_")
with open(d + "/chr.txt", "w") as f:
    f.write("".join(nm + "\n" for nm in names))
for nm, txt in zip(names, synth.mut_texts_fast(sites)):
    txt.tofile(f"{d}/syn_chr{nm}.mut")
rng = np.random.default_rng(7)
for c, (nm, L) in enumerate(zip(names, sites.chrom_len)):
    with open(f"{d}/g_chr{nm}.fa", "wb") as f:
        f.write(b">" + nm.encode() + b"\n" + np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(L), dtype=np.uint8)].tobytes() + b"\n")
pool = ThreadPoolExecutor(os.cpu_count() or 8)


def bgzf(path, header, parts):
    data = bytes(header) + b"".join(p.tobytes() for p in parts)
    blocks = pool.map(lambda i: synth.bgzf_block(data[i:i + 65280], 1), range(0, len(data), 65280))
    with open(path, "wb") as f:
        for b in blocks:
            f.write(b)
        f.write(synth.bgzf_compress(b"", eof=True)[-28:])


def genome_files(prefix, n_sample, frac, gt_key=1):
    """prefix.bcf (whole genome) and prefix_chr<c>.bcf, from the same records."""
    ids = [("FORMAT", "GT")]
    whole = []
    for c, nm in enumerate(names):
        lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
        keep = np.sort(rng.choice(hi - lo, int((hi - lo) * frac), replace=False))
        pos0 = sites.pos[lo:hi][keep] - 1
        anc, der = sites.anc[lo:hi][keep], sites.der[lo:hi][keep]
        gt = ((rng.random((len(keep), 2 * n_sample)) < 0.3).astype(np.int8) + 1) << 1
        whole.append(synth.bcf_records_np(pos0, anc, der, gt, gt_key, chrom=c))
        bgzf(f"{prefix}_chr{nm}.bcf", synth.bcf_header(n_sample, ids, contigs=(nm,)), [synth.bcf_records_np(pos0, anc, der, gt, gt_key, chrom=0)])
    bgzf(prefix + ".bcf", synth.bcf_header(n_sample, ids, contigs=names), whole)
    return prefix + ".bcf", [f"{prefix}_chr{nm}.bcf" for nm in names]


t0 = time.time()
inputs = {"target_1": genome_files(d + "/t", 1, 0.85), f"panel_{a.panel_samples}": genome_files(d + "/p", a.panel_samples, 0.5)}
print(f"inputs written in {time.time() - t0:.1f} s:", {k: round(os.path.getsize(v[0]) / 1e6, 1) for k, v in inputs.items()}, "MB", flush=True)

h = api.Handle(0)
h.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())


def slot_rows(slot):
    p4 = np.zeros((h.n_site, 4), np.int32)
    _lib.check(_lib.lib().colate_pileup_end(h._h, slot, p4.ctypes.data_as(C.c_void_p)))
    return p4[:, :2].copy()


for key, (whole, split) in inputs.items():
    t = {"genome": [], "split": []}
    out = {}
    for r in range(a.reps + 1):                       # the first pair of runs warms the page cache and the device buffers
        for kind in ("split", "genome"):
            s = time.perf_counter()
            if kind == "genome":
                h.rows_from_bcf_genome(0, 1, whole, names)
            else:
                h.rows_from_bcf_roles(0, 1, split)
            dt = time.perf_counter() - s
            if r:
                t[kind].append(dt)
            out[kind] = (slot_rows(0), slot_rows(1))
    same = all(np.array_equal(x, y) for x, y in zip(out["genome"], out["split"]))
    res[f"rows_{key}"] = {"genome_s": t["genome"], "split_s": t["split"], "identical": same, "records": int(h.last_bcf_timing()["records"])}
    print(f"rows {key}: whole-genome {min(t['genome']):.3f} s, 22 files {min(t['split']):.3f} s (best of {a.reps}); identical: {same}", flush=True)
h.close()

# make_tmp --targets: one line per job, whole-genome and split alternating
for key, (whole, split) in inputs.items():
    t = {"genome": [], "split": []}
    for r in range(a.reps):
        for kind, inp in (("split", split[0][:-len("_chr1.bcf")]), ("genome", whole)):
            tg = f"{d}/targets_{kind}.txt"
            with open(tg, "w") as f:
                f.write(f"target_bcf={inp} {d}/mk_{kind}\n")
            p = subprocess.run([CLI, "--mode", "make_tmp", "--mut", d + "/syn", "--chr", d + "/chr.txt", "--ref_genome", d + "/g", "--targets", tg],
                               capture_output=True, text=True, env=dict(os.environ, COLATE_TIMING="1"))
            assert p.returncode == 0, p.stderr[-3000:]
            t[kind].append(float(re.search(r"line 1 bcf: .*decode\+write ([0-9.]+) s", p.stderr).group(1)))
    same = open(f"{d}/mk_genome.colate.in", "rb").read() == open(f"{d}/mk_split.colate.in", "rb").read()
    res[f"make_tmp_{key}"] = {"genome_s": t["genome"], "split_s": t["split"], "identical": same}
    print(f"make_tmp {key}: decode+write whole-genome {min(t['genome']):.3f} s, 22 files {min(t['split']):.3f} s; identical: {same}", flush=True)

shutil.rmtree(d, ignore_errors=True)
print(json.dumps(res))
if a.out:
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bcf_genome_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
