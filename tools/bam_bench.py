"""BAM input at whole-genome size on one GPU: a synthetic 22-contig dataset (synth.rows_for_genome rows) with two BAM files, an
aDNA-like target (30-120 bp reads) and a deeper reference (100 bp reads), both drawn from the synthetic reference genome with 1%
sequencing errors.  Times, in one process:
  1. the whole CLI: `Colate --mode mut --target_bam --reference_bam --ref_genome` (files -> .colate_mat / .coal / .bin);
  2. Handle.pileup_from_bam per file, wall time, for several host inflate thread counts;
  3. the same with bam_timing on: BGZF index, inflate, record walk, host-to-device copies, device decode, filter + pileup;
  4. stages i-iii on the two BAM genomes (API);
  5. with --python-path, the path that existed before: the target BAM decoded in Python (gzip + struct/numpy) and fed to
     pileup_from_reads; its counts must equal pileup_from_bam's.  (Off by default: at the default size the Python record walk
     alone runs for many minutes.)
Prints the GPU's name and power limit with the numbers.
usage: bam_bench.py [--rows 10000000] [--target-reads 20000000] [--ref-reads 30000000] [--out DIR]"""
import argparse, gzip, json, os, shutil, struct, subprocess, sys, tempfile, time
from concurrent.futures import ThreadPoolExecutor
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colate_b200 import api, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")
ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=10_000_000)
ap.add_argument("--target-reads", type=int, default=20_000_000)
ap.add_argument("--ref-reads", type=int, default=30_000_000)
ap.add_argument("--threads", default="1,4,16,32")
ap.add_argument("--python-path", action="store_true", help="also time the Python decode + pileup_from_reads path (slow)")
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
d = tempfile.mkdtemp(prefix="colate_bam_bench_")
with open(d + "/chr.txt", "w") as f:
    f.write("".join(nm + "\n" for nm in sites.chr_names))
for nm, txt in zip(sites.chr_names, synth.mut_texts_fast(sites)):
    txt.tofile(f"{d}/syn_chr{nm}.mut")
rng = np.random.default_rng(7)
genome = []
for c, (nm, L) in enumerate(zip(sites.chr_names, lens)):
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
pool = ThreadPoolExecutor(os.cpu_count() or 8)


def write_bam(path, n_reads, len_lo, len_hi, seed):
    """Reads spread over the contigs by length, sorted by position, streamed through BGZF blocks of 65280 bytes (level 1)."""
    r = np.random.default_rng(seed)
    per = np.array(lens, np.float64) / sum(lens)
    counts = r.multinomial(n_reads, per)
    tot_bytes = 0
    with open(path, "wb") as f:
        pending = bytearray(synth.bam_header([f"chr{nm}" for nm in sites.chr_names], lens))

        def flush(final=False):
            nonlocal pending, tot_bytes
            cut = len(pending) if final else len(pending) // 65280 * 65280
            pieces = [bytes(pending[i:i + 65280]) for i in range(0, cut, 65280)]
            for b in pool.map(lambda p: synth.bgzf_block(p, 1), pieces):
                f.write(b)
            tot_bytes += cut
            del pending[:cut]
        for c, n in enumerate(counts):
            pos_all = np.sort(r.integers(0, lens[c] - len_hi, int(n))).astype(np.int32)
            ln_all = r.integers(len_lo, len_hi + 1, int(n)).astype(np.int32)
            for b0 in range(0, int(n), 1_000_000):
                p, l = pos_all[b0:b0 + 1_000_000], ln_all[b0:b0 + 1_000_000]
                idx = np.repeat(p.astype(np.int64), l) + (np.arange(int(l.sum())) - np.repeat(np.cumsum(l) - l, l))
                seq = genome[c][idx]
                err = r.random(seq.shape[0]) < 0.01
                seq[err] = np.frombuffer(b"ACGT", np.uint8)[r.integers(0, 4, int(err.sum()))]
                qual = np.where(r.random(seq.shape[0]) < 0.1, 20, 37).astype(np.uint8)
                mapq = r.choice(np.array([0, 25, 37, 60, 60], np.uint8), p.shape[0])
                pending += synth.bam_records_np(np.full(p.shape[0], c), p, mapq, l, seq, qual).tobytes()
                flush()
        flush(final=True)
        f.write(synth.BGZF_EOF)
    return tot_bytes


sizes = {}
for tag, n, lo, hi, seed in (("t", a.target_reads, 30, 120, 11), ("r", a.ref_reads, 100, 100, 12)):
    sizes[tag] = write_bam(f"{d}/{tag}.bam", n, lo, hi, seed)
    sizes[tag + "_file"] = os.path.getsize(f"{d}/{tag}.bam")
res["dataset"] = {"rows": int(sites.n), "contigs": len(lens), "target_reads": a.target_reads, "ref_reads": a.ref_reads,
                  "target_inflated_bytes": sizes["t"], "target_file_bytes": sizes["t_file"], "ref_inflated_bytes": sizes["r"],
                  "ref_file_bytes": sizes["r_file"], "written_s": round(time.time() - t0, 1)}
print("dataset:", res["dataset"], flush=True)

# 1. the whole CLI (twice: the first run also reads the files into the page cache)
cli = [CLI, "--mode", "mut", "--mut", d + "/syn", "--chr", d + "/chr.txt", "--target_bam", d + "/t.bam", "--reference_bam", d + "/r.bam",
       "--ref_genome", d + "/g", "--bins", "3,7,0.2", "--seed", "1", "--num_bootstraps", "10"]
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

# 2.-4. the API
h = api.Handle(0)
h.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
h.set_option("front_end", 1)
names = list(sites.chr_names)
res["pileup_from_bam"] = []
counts = {}
for th in [int(x) for x in a.threads.split(",")]:
    os.environ["COLATE_BAM_THREADS"] = str(th)
    for slot, tag in ((0, "t"), (1, "r")):
        t = time.time()
        counts[tag] = h.pileup_from_bam(slot, f"{d}/{tag}.bam", names, genome, fetch=True)
        wall = time.time() - t
        tm = h.last_bam_timing()
        row = {"file": tag, "threads": th, "wall_s": round(wall, 3), **{k: round(v, 4) for k, v in tm.items()}}
        res["pileup_from_bam"].append(row)
        print("pileup_from_bam", row, flush=True)
os.environ.pop("COLATE_BAM_THREADS")
h.set_option("bam_timing", 1)
res["phases"] = []
for slot, tag in ((0, "t"), (1, "r")):
    h.pileup_from_bam(slot, f"{d}/{tag}.bam", names, genome)
    tm = h.last_bam_timing()
    res["phases"].append({"file": tag, **{k: round(v, 4) for k, v in tm.items()}})
    print("phases (bam_timing on)", res["phases"][-1], flush=True)
h.set_option("bam_timing", 0)
t = time.time()
s1 = h.stage1(api.mt_seed(1))
t1 = time.time()
w = api.draw_block_weights(s1.mt_state.copy(), 10, s1.num_blocks)
cn = h.stage2_bootstrap(w, s1.block_stats, 0.0)
t2 = time.time()
ep, _ = api.epochs_from_bins("3,7,0.2")
h.stage3_em(10, ep, np.full(len(ep), 1 / 20000.0), None, 100000)
t3 = time.time()
res["stages_s"] = {"i": round(t1 - t, 3), "ii": round(t2 - t1, 3), "iii": round(t3 - t2, 3), "used_rows": int(s1.n_used), "blocks": int(s1.num_blocks)}
print("stages:", res["stages_s"], flush=True)

# 5. the path that existed before: decode in Python, then pileup_from_reads
if a.python_path:
    t = time.time()
    data = gzip.decompress(open(f"{d}/t.bam", "rb").read())
    t_inflate = time.time() - t
    o = 8 + struct.unpack_from("<i", data, 4)[0]
    n_ref = struct.unpack_from("<i", data, o)[0]
    o += 4
    for _ in range(n_ref):
        o += 8 + struct.unpack_from("<i", data, o)[0]
    offs = []
    while o < len(data):
        offs.append(o)
        o += 4 + struct.unpack_from("<i", data, o)[0]
    offs = np.array(offs, np.int64)
    buf = np.frombuffer(data, np.uint8)
    i32 = lambda at: buf[at[:, None] + np.arange(4)].copy().view("<i4")[:, 0]
    tid, pos, lseq = i32(offs + 4), i32(offs + 8), i32(offs + 20)
    mapq = buf[offs + 13]
    lrn, ncig = buf[offs + 12].astype(np.int64), buf[offs + 16].astype(np.int64) | buf[offs + 17].astype(np.int64) << 8
    sstart = offs + 36 + lrn + 4 * ncig
    L = lseq.astype(np.int64)
    rel = np.arange(int(L.sum())) - np.repeat(np.cumsum(L) - L, L)
    byte = buf[np.repeat(sstart, L) + rel // 2]
    code = np.where(rel % 2 == 0, byte >> 4, byte & 15)
    seq = np.frombuffer(synth.NT16, np.uint8)[code]
    qual = buf[np.repeat(sstart + (L + 1) // 2, L) + rel]
    t_decode = time.time() - t - t_inflate
    per = []
    soff = np.concatenate([[0], np.cumsum(L)]).astype(np.int64)
    for c in range(len(lens)):
        k = np.nonzero(tid == c)[0]
        if k.size == 0:
            per.append(None)
            continue
        a0, a1 = soff[k[0]], soff[k[-1] + 1]
        per.append((pos[k], mapq[k], lseq[k], soff[k] - a0, seq[a0:a1], qual[a0:a1]))
    t = time.time()
    old = h.pileup_from_reads(0, per, genome, fetch=True)
    t_pile = time.time() - t
    assert np.array_equal(old, counts["t"]), "pileup_from_reads and pileup_from_bam disagree"
    res["python_decode_path"] = {"gzip_decompress_s": round(t_inflate, 3), "python_walk_and_decode_s": round(t_decode, 3),
                                 "pileup_from_reads_s": round(t_pile, 3), "total_s": round(t_inflate + t_decode + t_pile, 3), "counts_equal": True}
    print("python decode + pileup_from_reads (target):", res["python_decode_path"], flush=True)
h.close()
if a.out:
    os.makedirs(a.out, exist_ok=True)
    json.dump(res, open(os.path.join(a.out, "bam_bench.json"), "w"), indent=1)
shutil.rmtree(d, ignore_errors=True)
