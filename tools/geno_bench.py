"""make_tmp from a genotype matrix at AADR-like size on one GPU: a synthetic 22-contig .mut set (--rows rows), a packed EIGENSTRAT
matrix of --snps SNPs (at .mut row positions) x --ind individuals (random 2-bit calls, about 600 MB at the defaults), every
individual written.  Times, in one process:
  1. colate_maketmp_write_geno for all individuals with each file sent to /dev/null (the device path and the copies, no disk);
  2. the same call for the first --disk individuals into real files under a temporary directory (the file-write rate);
  3. the `--target_table` CLI, one process per individual, for the first --loop individuals on their derived tables, extrapolated
     to all individuals (the output says so); each table run's file is compared with the device's byte for byte.
Reports the phases of (1) and (2) (scan, upload, join, called, rows, scatter, d2h, write) and the output GB/s, with the GPU's name
and power limit read in the same run.
usage: geno_bench.py [--rows 10000000] [--snps 1200000] [--ind 2000] [--disk 100] [--loop 5] [--out DIR]"""
import argparse, json, os, shutil, subprocess, sys, tempfile, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colate_b200 import api, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")
ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=10_000_000)
ap.add_argument("--snps", type=int, default=1_200_000)
ap.add_argument("--ind", type=int, default=2000)
ap.add_argument("--disk", type=int, default=100, help="individuals written to real files")
ap.add_argument("--loop", type=int, default=5, help="--target_table CLI runs")
ap.add_argument("--out", default=None, help="directory for the JSON result")
a = ap.parse_args()

try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
except FileNotFoundError:
    gpu = ""
gpu = gpu.splitlines()[0] if gpu else "unknown"
print("GPU:", gpu, "| host CPUs:", os.cpu_count(), flush=True)
res = {"gpu": gpu, "host_cpus": os.cpu_count(), "rows": a.rows, "snps": a.snps, "individuals": a.ind}
t0 = time.time()
sites = synth.make_sites(1, synth.rows_for_genome(a.rows), synth.AUTOSOME_LEN)
names = list(sites.chr_names)
d = tempfile.mkdtemp(prefix="colate_geno_bench_")
try:
    open(d + "/chr.txt", "w").write("".join(nm + "\n" for nm in names))
    for nm, txt in zip(names, synth.mut_texts_fast(sites)):
        txt.tofile(f"{d}/syn_chr{nm}.mut")
        open(f"{d}/g_chr{nm}.fa", "w").write(">g\nACGT\n")
    rng = np.random.default_rng(3)
    rows = np.sort(rng.choice(sites.n, size=a.snps, replace=False))          # rows are sorted by contig, then position
    chrom = np.searchsorted(sites.site_off, rows, side="right") - 1
    swap = rng.random(a.snps) < 0.5
    al1 = np.where(swap, sites.der[rows], sites.anc[rows])
    al2 = np.where(swap, sites.anc[rows], sites.der[rows])
    cn = np.array(names)[chrom]
    lines = np.char.add(np.char.add(np.char.add("rs", rows.astype(str)), "\t"), cn)
    lines = np.char.add(np.char.add(lines, "\t0.0\t"), sites.pos[rows].astype(str))
    lines = np.char.add(np.char.add(np.char.add(lines, "\t"), al1.view("S1").astype(str)), "\t")
    lines = np.char.add(lines, al2.view("S1").astype(str))
    open(d + "/m.snp", "w").write("\n".join(lines.tolist()) + "\n")
    ids = [f"ind{k}" for k in range(a.ind)]
    open(d + "/m.ind", "w").write("".join(f"{x}\tU\tpop\n" for x in ids))
    rlen = max(48, (a.ind + 3) // 4)
    with open(d + "/m.geno", "wb") as f:
        f.write(f"GENO {a.ind} {a.snps} 0 0".encode().ljust(rlen, b"\0"))
        for s0 in range(0, a.snps, 100_000):
            n = min(100_000, a.snps - s0)
            f.write(rng.integers(0, 256, (n, rlen), dtype=np.uint8).tobytes())
    res["matrix_bytes"] = os.path.getsize(d + "/m.geno")
    res["setup_s"] = time.time() - t0
    print(f"inputs in {res['setup_s']:.1f} s: {a.rows} rows, matrix {res['matrix_bytes'] / 1e6:.0f} MB", flush=True)

    h = api.Handle(0)
    t1 = time.time()
    h.ingest_mut([open(f"{d}/syn_chr{nm}.mut", "rb").read() for nm in names])
    res["mut_ingest_s"] = time.time() - t1
    for tag, n, files in (("all_devnull", a.ind, ["/dev/null"] * a.ind),
                          ("disk", a.disk, [f"{d}/o{k}.colate.in" for k in range(a.disk)])):
        t1 = time.time()
        r = h.maketmp_write_geno(d + "/m", "eigenstrat", ids[:n], names, files)
        wall = time.time() - t1
        t = h.last_geno_timing()
        t["wall_s"] = wall
        t["records"] = int(r["records"].sum())
        t["output_GBps"] = t["bytes"] / wall / 1e9
        res[tag] = t
        print(tag, json.dumps({k: round(v, 4) if isinstance(v, float) else v for k, v in t.items()}), flush=True)
    h.close()

    # the table route: one --target_table process per individual
    raw = np.fromfile(d + "/m.geno", np.uint8)[rlen:].reshape(a.snps, rlen)
    table_s = []
    for k in range(a.loop):
        v = (raw[:, k >> 2] >> (6 - 2 * (k & 3))) & 3                       # copies of column 5
        hom = (v == 2) | (v == 0)
        al = np.where(v == 2, al1, al2)[hom].view("S1").astype(str)
        tl = np.char.add(np.char.add(np.char.add(np.char.add(cn[hom], " "), sites.pos[rows][hom].astype(str)), " "), al)
        open(f"{d}/t{k}.txt", "w").write("\n".join(tl.tolist()) + "\n")
        t1 = time.time()
        p = subprocess.run([CLI, "--mode", "make_tmp", "--mut", f"{d}/syn", "--chr", f"{d}/chr.txt", "--ref_genome", f"{d}/g", "--target_table",
                            f"{d}/t{k}.txt", "-o", f"{d}/t{k}"], capture_output=True, text=True)
        table_s.append(time.time() - t1)
        assert p.returncode == 0, p.stderr[-2000:]
        assert open(f"{d}/t{k}.colate.in", "rb").read() == open(f"{d}/o{k}.colate.in", "rb").read(), k
    res["table_run_s"] = table_s
    res["table_runs_extrapolated_s"] = float(np.mean(table_s)) * a.ind
    print(f"--target_table: {np.mean(table_s):.2f} s per individual (measured on {a.loop}), extrapolated to {a.ind}: "
          f"{res['table_runs_extrapolated_s']:.0f} s; outputs equal the device's", flush=True)
    d_all = res["all_devnull"]
    disk_rate = res["disk"]["bytes"] / max(res["disk"]["write_s"], 1e-9)
    res["job_extrapolated_s"] = d_all["wall_s"] - d_all["write_s"] + d_all["bytes"] / disk_rate
    print(f"job for all {a.ind}: {d_all['wall_s']:.1f} s to /dev/null; with files at the measured {disk_rate / 1e9:.2f} GB/s: "
          f"{res['job_extrapolated_s']:.1f} s (extrapolated)", flush=True)
finally:
    shutil.rmtree(d, ignore_errors=True)
print(json.dumps(res))
if a.out:
    os.makedirs(a.out, exist_ok=True)
    json.dump(res, open(os.path.join(a.out, "geno_bench.json"), "w"), indent=1)
