"""Cohorts on BAM and BCF pairs at whole-genome size on one GPU: a synthetic 22-contig dataset (synth.rows_for_genome rows, a 2.88 Gbase
reference genome) and two workloads, each one `Colate --mode mut --pairs` job:
  BAM: --bam_targets aDNA-like target BAMs (30-120 bp reads, 1% errors) x --bam_refs deeper reference BAMs, every target against every
       reference, target ages 2000 years and up, R = --R bootstrap replicates;
  BCF: --bcf_targets one-sample target BCFs x --panels panel BCFs of --panel_samples diploid samples (records at ~85% of the rows).
Per workload it times the cohort CLI end to end, twice (the first run also reads the inputs into the page cache), and the
single-pair CLI (one process per pair) on the first --loop pairs, whose per-pair time is extrapolated to all pairs -- the output
says so.  Every single-pair output is compared with the cohort's byte for byte.  Prints the GPU's name and power limit, read in the
same run.
usage: cohort_frontend_bench.py [--rows 10000000] [--bam_targets 4] [--bam_refs 3] [--target_reads 2000000] [--ref_reads 4000000]
                                [--bcf_targets 8] [--panels 2] [--panel_samples 100] [--R 10] [--loop 2] [--out DIR]"""
import argparse, json, os, shutil, subprocess, sys, tempfile, time
from concurrent.futures import ThreadPoolExecutor
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colate_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")
ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=10_000_000)
ap.add_argument("--bam_targets", type=int, default=4)
ap.add_argument("--bam_refs", type=int, default=3)
ap.add_argument("--target_reads", type=int, default=2_000_000, help="reads per target BAM")
ap.add_argument("--ref_reads", type=int, default=4_000_000, help="reads per reference BAM")
ap.add_argument("--bcf_targets", type=int, default=8)
ap.add_argument("--panels", type=int, default=2)
ap.add_argument("--panel_samples", type=int, default=100)
ap.add_argument("--R", type=int, default=10)
ap.add_argument("--loop", type=int, default=2, help="single-pair runs per workload")
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
sites = synth.make_sites(1, synth.rows_for_genome(a.rows), synth.AUTOSOME_LEN)
lens = [int(L) for L in sites.chrom_len]
names = list(sites.chr_names)
d = tempfile.mkdtemp(prefix="colate_cohort_frontend_bench_")
with open(d + "/chr.txt", "w") as f:
    f.write("".join(nm + "\n" for nm in names))
for nm, txt in zip(names, synth.mut_texts_fast(sites)):
    txt.tofile(f"{d}/syn_chr{nm}.mut")
pool = ThreadPoolExecutor(os.cpu_count() or 8)
rng = np.random.default_rng(7)
genome = []
for c, (nm, L) in enumerate(zip(names, lens)):
    g = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L, dtype=np.uint8)]
    lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
    anc = sites.anc[lo:hi]
    ok = np.isin(anc, np.frombuffer(b"ACGT", np.uint8))
    g[sites.pos[lo:hi][ok] - 1] = anc[ok]
    genome.append(g)
    with open(f"{d}/g_chr{nm}.fa", "wb") as f:
        f.write(b">" + nm.encode() + b"\n")
        g.tofile(f)
        f.write(b"\n")


def stream(path, header, batches):
    """header + record batches through BGZF blocks of 65280 bytes (level 1)."""
    with open(path, "wb") as f:
        pending = bytearray(header)

        def flush(final=False):
            nonlocal pending
            cut = len(pending) if final else len(pending) // 65280 * 65280
            for b in pool.map(lambda p: synth.bgzf_block(p, 1), [bytes(pending[i:i + 65280]) for i in range(0, cut, 65280)]):
                f.write(b)
            del pending[:cut]
        for b in batches:
            pending += b
            flush()
        flush(final=True)
        f.write(synth.BGZF_EOF)


def bam_batches(seed, n_reads):
    r = np.random.default_rng(seed)
    counts = r.multinomial(n_reads, np.array(lens, np.float64) / sum(lens))
    for c, n in enumerate(counts):
        pos_all = np.sort(r.integers(0, lens[c] - 120, int(n))).astype(np.int32)
        ln_all = r.integers(30, 121, int(n)).astype(np.int32)
        for b0 in range(0, int(n), 1_000_000):
            p, l = pos_all[b0:b0 + 1_000_000], ln_all[b0:b0 + 1_000_000]
            idx = np.repeat(p.astype(np.int64), l) + (np.arange(int(l.sum())) - np.repeat(np.cumsum(l) - l, l))
            seq = genome[c][idx]
            err = r.random(seq.shape[0]) < 0.01
            seq[err] = np.frombuffer(b"ACGT", np.uint8)[r.integers(0, 4, int(err.sum()))]
            qual = np.where(r.random(seq.shape[0]) < 0.1, 20, 37).astype(np.uint8)
            mapq = r.choice(np.array([0, 25, 37, 60, 60], np.uint8), p.shape[0])
            yield synth.bam_records_np(np.full(p.shape[0], c), p, mapq, l, seq, qual).tobytes()


def bcf_batches(seed, c, n_sample):
    """records at ~85% of the chromosome's rows, the row's alleles in either order; n_sample diploid samples"""
    r = np.random.default_rng(seed)
    lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
    m = lo + np.flatnonzero(r.random(hi - lo) < 0.85)
    pos0 = np.unique(sites.pos[m] - 1).astype(np.int32)
    m = lo + np.searchsorted(sites.pos[lo:hi], pos0 + 1)
    sw = r.random(m.shape[0]) < 0.3
    a0 = np.where(sw, sites.der[m], sites.anc[m]).astype(np.uint8)
    a1 = np.where(sw, sites.anc[m], sites.der[m]).astype(np.uint8)
    step = max(1, (1 << 22) // (2 * n_sample))
    for b0 in range(0, m.shape[0], step):
        s = slice(b0, b0 + step)
        n = pos0[s].shape[0]
        af = r.random((n, 1))
        gt = (((r.random((n, 2 * n_sample)) < af).astype(np.int8) + 1) << 1).astype(np.int8)
        yield synth.bcf_records_np(pos0[s], a0[s], a1[s], gt, 1).tobytes()


KT, KR = a.bam_targets, a.bam_refs
for k in range(KT):
    stream(f"{d}/t{k}.bam", synth.bam_header(names, lens), bam_batches(11 + k, a.target_reads))
for k in range(KR):
    stream(f"{d}/r{k}.bam", synth.bam_header(names, lens), bam_batches(31 + k, a.ref_reads))
for k in range(a.bcf_targets):
    for c, nm in enumerate(names):
        stream(f"{d}/v{k}_chr{nm}.bcf", synth.bcf_header(1), bcf_batches(50 + 100 * k + c, c, 1))
for k in range(a.panels):
    for c, nm in enumerate(names):
        stream(f"{d}/p{k}_chr{nm}.bcf", synth.bcf_header(a.panel_samples), bcf_batches(5000 + 100 * k + c, c, a.panel_samples))
res["dataset"] = {"rows": int(sites.n), "contigs": len(lens), "genome_bases": int(sum(lens)), "bam_targets": KT, "target_reads": a.target_reads,
                  "bam_refs": KR, "ref_reads": a.ref_reads, "bcf_targets": a.bcf_targets, "panels": a.panels, "panel_samples": a.panel_samples,
                  "R": a.R, "bam_file_bytes": [os.path.getsize(f"{d}/t{k}.bam") for k in range(KT)] + [os.path.getsize(f"{d}/r{k}.bam") for k in range(KR)],
                  "panel_bytes": sum(os.path.getsize(f"{d}/p{k}_chr{nm}.bcf") for k in range(a.panels) for nm in names),
                  "written_s": round(time.time() - t0, 1)}
print("dataset:", res["dataset"], flush=True)
shared = [CLI, "--mode", "mut", "--mut", d + "/syn", "--chr", d + "/chr.txt", "--ref_genome", d + "/g", "--bins", "3,7,0.2", "--seed", "23",
          "--num_bootstraps", str(a.R)]
workloads = {
    "bam": [(f"target_bam={d}/t{i}.bam", f"reference_bam={d}/r{j}.bam", f"target_age={2000 + 500 * i}") for i in range(KT) for j in range(KR)],
    "bcf": [(f"target_bcf={d}/v{i}", f"reference_bcf={d}/p{j}", f"target_age={1000 + 250 * i}") for i in range(a.bcf_targets) for j in range(a.panels)],
}
for name, lines in workloads.items():
    out = {"pairs": len(lines)}
    pf = f"{d}/pairs_{name}.txt"
    with open(pf, "w") as f:
        f.write("".join(f"{t} {r} {d}/{name}{k} {age}\n" for k, (t, r, age) in enumerate(lines)))
    walls = []
    for rep in range(2):
        for k in range(len(lines)):
            for e in (".coal", ".bin", ".colate_mat"):
                if os.path.exists(f"{d}/{name}{k}{e}"):
                    os.remove(f"{d}/{name}{k}{e}")          # a .colate_mat left behind would take the stale-cache path
        t = time.time()
        p = subprocess.run(shared + ["--pairs", pf], capture_output=True, text=True)
        walls.append(time.time() - t)
        assert p.returncode == 0, p.stderr[-3000:]
    out["cohort_wall_s"] = [round(x, 3) for x in walls]
    out["summary"] = [ln for ln in p.stderr.splitlines() if ln.startswith("device ")]
    single, identical = [], True
    for k in range(min(a.loop, len(lines))):
        t_in, r_in, age = lines[k]
        flags = []
        for x in (t_in, r_in, age):
            key, _, val = x.partition("=")
            flags += ["--" + key, val]
        t = time.time()
        q = subprocess.run(shared + flags + ["-o", f"{d}/one_{name}{k}"], capture_output=True, text=True)
        single.append(round(time.time() - t, 3))
        assert q.returncode == 0, q.stderr[-3000:]
        for e in (".coal", ".bin", ".colate_mat"):
            identical &= open(f"{d}/one_{name}{k}{e}", "rb").read() == open(f"{d}/{name}{k}{e}", "rb").read()
    out["single_pair_wall_s"] = single
    out["single_extrapolated_s"] = round(float(np.mean(single)) * len(lines), 1)
    out["identical"] = bool(identical)
    out["speedup_vs_extrapolated"] = round(out["single_extrapolated_s"] / min(walls), 2)
    res[name] = out
    print("%s: %d pairs | cohort CLI wall %s s | single-pair CLI %s s on the first %d pairs, extrapolated to all %d: %.1f s (extrapolated) | "
          "%.2fx | sampled pairs byte-identical: %s" % (name, len(lines), out["cohort_wall_s"], single, len(single), len(lines),
                                                        out["single_extrapolated_s"], out["speedup_vs_extrapolated"], identical), flush=True)
    print("  " + "\n  ".join(out["summary"]), flush=True)
if a.out:
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "cohort_frontend_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
shutil.rmtree(d, ignore_errors=True)
