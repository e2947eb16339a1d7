"""make_tmp for many targets at whole-genome size on one GPU: a synthetic 22-contig dataset (synth.rows_for_genome rows, a 2.88 Gbase
reference genome), K aDNA-like BAM targets (30-120 bp reads, 1% errors) and K one-sample BCF targets (records at most rows), one
mask shared by every target.  Times, in one process:
  1. the batch CLI (`Colate --mode make_tmp --targets`) end to end, twice (the first run also reads the inputs into the page cache),
     with its per-phase lines (COLATE_TIMING=1): .mut read / parse, genome read / upload, masks, and per target inflate, decode or
     pileup, the writer's kernels, the device-to-host copy and the file write;
  2. the single-target CLI, one process per target, on the first --loop BAM and --loop BCF targets; its per-target time is
     extrapolated to all 2K targets and the output says so.  Every single-target output is compared with the batch's byte for byte.
Prints the GPU's name and power limit, read in the same run.
usage: maketmp_bench.py [--rows 10000000] [--k 4] [--reads 4000000] [--loop 1] [--out DIR]"""
import argparse, json, os, shutil, subprocess, sys, tempfile, time
from concurrent.futures import ThreadPoolExecutor
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colate_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")
ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=10_000_000)
ap.add_argument("--k", type=int, default=4, help="BAM targets, and as many BCF targets")
ap.add_argument("--reads", type=int, default=4_000_000, help="reads per BAM target")
ap.add_argument("--loop", type=int, default=1, help="single-target runs per kind (BAM, BCF)")
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
d = tempfile.mkdtemp(prefix="colate_maketmp_bench_")
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
    synth.write_mask(f"{d}/m_chr{nm}.fa", synth.make_mask(100 + c, L, 0.3))


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


def bam_batches(seed):
    r = np.random.default_rng(seed)
    counts = r.multinomial(a.reads, np.array(lens, np.float64) / sum(lens))
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


def bcf_batches(seed, c):
    """one sample, records at ~85% of the chromosome's rows: the row's alleles in either order or the derived allele alone"""
    r = np.random.default_rng(seed)
    lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
    m = lo + np.flatnonzero(r.random(hi - lo) < 0.85)
    pos0 = np.unique(sites.pos[m] - 1).astype(np.int32)
    m = lo + np.searchsorted(sites.pos[lo:hi], pos0 + 1)
    sw = r.random(m.shape[0]) < 0.3
    a0 = np.where(sw, sites.der[m], sites.anc[m]).astype(np.uint8)
    a1 = np.where(sw, sites.anc[m], sites.der[m]).astype(np.uint8)
    allele = (r.random((m.shape[0], 2)) < 0.3).astype(np.int8)
    gt = ((allele + 1) << 1).astype(np.int8)
    for b0 in range(0, m.shape[0], 1 << 20):
        s = slice(b0, b0 + (1 << 20))
        yield synth.bcf_records_np(pos0[s], a0[s], a1[s], gt[s], 1).tobytes()


K = a.k
for k in range(K):
    stream(f"{d}/s{k}.bam", synth.bam_header(names, lens), bam_batches(11 + k))
    for c, nm in enumerate(names):
        stream(f"{d}/v{k}_chr{nm}.bcf", synth.bcf_header(1), bcf_batches(50 + 100 * k + c, c))
targets = [("target_bam", f"{d}/s{k}.bam") for k in range(K)] + [("target_bcf", f"{d}/v{k}") for k in range(K)]
with open(d + "/targets.txt", "w") as f:
    f.write("".join(f"{key}={inp} {d}/b{i} target_mask={d}/m\n" for i, (key, inp) in enumerate(targets)))
res["dataset"] = {"rows": int(sites.n), "contigs": len(lens), "genome_bases": int(sum(lens)), "bam_targets": K, "reads_per_bam": a.reads,
                  "bcf_targets": K, "bam_file_bytes": [os.path.getsize(f"{d}/s{k}.bam") for k in range(K)], "written_s": round(time.time() - t0, 1)}
print("dataset:", res["dataset"], flush=True)
shared = [CLI, "--mode", "make_tmp", "--mut", d + "/syn", "--chr", d + "/chr.txt", "--ref_genome", d + "/g"]

# 1. the batch CLI
walls = []
for rep in range(2):
    t = time.time()
    p = subprocess.run(shared + ["--targets", d + "/targets.txt"], capture_output=True, text=True, env=dict(os.environ, COLATE_TIMING="1"))
    walls.append(time.time() - t)
    assert p.returncode == 0, p.stderr[-3000:]
res["batch_wall_s"] = [round(x, 3) for x in walls]
res["batch_timing_lines"] = [ln for ln in p.stderr.splitlines() if ln.startswith("[timing]")]
print("batch CLI wall (%d targets): %s" % (2 * K, res["batch_wall_s"]), *res["batch_timing_lines"], sep="\n  ", flush=True)

# 2. single-target runs on a subset, extrapolated
single, identical = [], True
for i in list(range(min(a.loop, K))) + list(range(K, K + min(a.loop, K))):
    key, inp = targets[i]
    t = time.time()
    q = subprocess.run(shared + [f"--{key}", inp, "--target_mask", d + "/m", "-o", f"{d}/one{i}"], capture_output=True, text=True)
    single.append({"target": i, "kind": key, "wall_s": round(time.time() - t, 3)})
    assert q.returncode == 0, q.stderr[-3000:]
    identical &= open(f"{d}/one{i}.colate.in", "rb").read() == open(f"{d}/b{i}.colate.in", "rb").read()
res["single"] = single
per = {kind: np.mean([s["wall_s"] for s in single if s["kind"] == kind]) for kind in ("target_bam", "target_bcf")}
res["single_extrapolated_s"] = round(K * per["target_bam"] + K * per["target_bcf"], 1)
res["identical"] = bool(identical)
res["batch_speedup"] = round(res["single_extrapolated_s"] / min(walls), 2)
print("single-target CLI: %s | extrapolated to all %d targets: %.1f s (a subset was run) | batch %.1f s -> %.2fx | outputs byte-identical: %s"
      % (single, 2 * K, res["single_extrapolated_s"], min(walls), res["batch_speedup"], identical), flush=True)
if a.out:
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "maketmp_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
shutil.rmtree(d, ignore_errors=True)
