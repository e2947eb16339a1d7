#!/usr/bin/env python
"""bench.py -- pair-site evaluations/s of the `Colate --mode mut` hot path on B200.

One step = one full pass of the path over one synthetic whole-genome sample pair
(BASELINE.json configs[1]: 22 autosomes, 10 M .mut rows, two ~1x .colate.in genomes,
--bins 3,7,0.1, one replicate): stage i (record->row join, row filter + stream look-ahead,
std::mt19937 stream by jump-ahead, 100 Monte-Carlo age draws per used row, per-block
histograms) -> stage ii (block bootstrap + F redistribution) -> stage iii (EM to convergence).

  value    device-resident: parsed structure-of-arrays inputs already in HBM when the timed region starts
  e2e      the same pass from the FILE BYTES the reference starts from -- the 22 `.mut` texts and the two
           `.colate.in` record streams in pinned host memory -- through the C-ABI: host->device copies, text
           parse and record decode on the GPU, stages i-iii, device->host read of the rates, all inside the
           timed region.  Consecutive passes are pipelined the way a driver over many pairs runs them
           (colate_stage3_em_begin / _end): the EM of pass i (one replicate = one GPC) runs on the handle's EM
           stream while pass i+1 is copied in, parsed and taken through stage i; every pass's EM result is
           read back inside the timed region (the last one before the closing event).  e2e.serial_ms_per_step
           is the same pass without that overlap.
  e2e_soa  round 1's leg: the pass from already parsed SoA arrays in pinned host memory
  config3  BASELINE.json configs[2]: the same dataset with 1000 block-bootstrap replicates through
           colate_b200/dist.py (chromosomes sharded for stage i, replicates for stages ii-iii) on all N
           GPUs: wall time of the whole job, a hash of the results (equal for every N) and the NCCL calls

N > 1 (torchrun, one process per GPU): `value` / `e2e` shard by sample pair (configs[4]): every rank runs its
own pair of the same shape, no data-path collective, weak scaling; the max over ranks of the device time is
taken with one NCCL all-reduce outside the timed steps.  `config3` is strong scaling.

--impl reference times the unmodified reference CLI (oracle/_ref/Colate, compiled from /root/reference by
oracle/Makefile) on ALL host cores on the same dataset from the same files: one reference process per
chromosome, longest first on a pool of `cores` workers (see reference_arm()).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "pair_site_evals_per_s"
UNIT = "pair-site evaluations/s"
BINS = "3,7,0.1"
SEED = 1


def workload_name(rows):
    return (f"synthetic whole-genome single pair: 22 autosomes, {rows} .mut rows, two ~1x .colate.in genomes "
            f"(record w.p. 0.7, N=1+floor(Exp(1)), derived w.p. 0.3), --bins {BINS}, --seed {SEED}, 1 replicate "
            f"(BASELINE.json configs[1]; per rank one such pair when --gpus > 1)")


def config_of(rows):
    """Identical in both arms (the driver compares them)."""
    return {"workload": workload_name(rows)}


# --------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(local):
    """Pin this rank's host threads (and with them its pinned staging buffers: first touch) to the NUMA node its GPU hangs
    off.  With one rank per GPU and ~1 GB of file bytes copied in per pass, buffers left on the other socket cross the
    inter-socket link and every rank's copies slow down.  No-op where the topology is not exposed."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        cpus = sorted(set(cpus) & os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": node, "cpus": len(cpus)}
    except Exception:
        pass
    return None


def make_dataset(rows, pair=0):
    """Sites are the same for every pair (one Relate .mut set); genomes differ per pair."""
    from colate_b200 import synth
    sites = synth.make_sites(SEED, synth.rows_for_genome(rows), synth.AUTOSOME_LEN)
    gt = synth.make_genome(SEED + 100 + 1000 * pair, sites, 0.7)
    gr = synth.make_genome(SEED + 200 + 1000 * pair, sites, 0.7)
    return sites, gt, gr


def scratch_dir(prefix):
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    return tempfile.mkdtemp(prefix=prefix, dir=base)


def write_dataset_files(workdir, sites, gt, gr, texts=None, split_by_chr=False):
    """The dataset in the reference's on-disk formats: <dir>/syn_chr<name>.mut, chr.txt, t.colate.in, r.colate.in
    (+ per-chromosome chr_<name>.txt, t_<name>.colate.in, r_<name>.colate.in when split_by_chr)."""
    from colate_b200 import synth
    os.makedirs(workdir, exist_ok=True)
    texts = texts if texts is not None else synth.mut_texts_fast(sites)
    with open(os.path.join(workdir, "chr.txt"), "w") as f:
        for nm in sites.chr_names:
            f.write(nm + "\n")
    for c, nm in enumerate(sites.chr_names):
        with open(os.path.join(workdir, f"syn_chr{nm}.mut"), "wb") as f:
            f.write(texts[c].tobytes())
    for tag, g in (("t", gt), ("r", gr)):
        with open(os.path.join(workdir, f"{tag}.colate.in"), "wb") as f:
            f.write(synth.colate_in_image(g, sites.chr_names).tobytes())
    if split_by_chr:
        for c, nm in enumerate(sites.chr_names):
            with open(os.path.join(workdir, f"chr_{nm}.txt"), "w") as f:
                f.write(nm + "\n")
            for tag, g in (("t", gt), ("r", gr)):
                sel = g.chrom == c
                sub = synth.Genome(g.chrom[sel], g.bp[sel], g.anc[sel], g.der[sel], g.aaf[sel], g.daf[sel])
                with open(os.path.join(workdir, f"{tag}_{nm}.colate.in"), "wb") as f:
                    f.write(synth.colate_in_image(sub, sites.chr_names).tobytes())
    return texts


def ref_cmd(cli, workdir, chr_file, t_file, r_file, out_prefix):
    return [cli, "--mode", "mut", "--mut", os.path.join(workdir, "syn"), "--chr", os.path.join(workdir, chr_file),
            "--target_tmp", os.path.join(workdir, t_file), "--reference_tmp", os.path.join(workdir, r_file),
            "--bins", BINS, "--seed", str(SEED), "-o", out_prefix]


def cpu_baseline_one_core(rows, sites, gt, gr, texts):
    """The unmodified reference CLI, ONE process (it is single-threaded) on the whole dataset from the same files."""
    from oracle import pyoracle as po
    if po.ref_cli() is None:
        return cpu_baseline_port(sites, gt, gr)
    d = scratch_dir("colate_cpu_")
    try:
        write_dataset_files(d, sites, gt, gr, texts)
        t0 = time.perf_counter()
        p = subprocess.Popen(ref_cmd(po.ref_cli(), d, "chr.txt", "t.colate.in", "r.colate.in", os.path.join(d, "ref")),
                             stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        p.wait()
        dt = time.perf_counter() - t0
        return {"value": sites.n / dt, "unit": UNIT, "cores": 1, "kind": "reference",
                "sample": f"oracle/_ref/Colate --mode mut, one process, the WHOLE dataset ({sites.n} rows in 22 .mut files, two .colate.in; "
                          f".mut text parse, site loop and EM included), {dt:.2f} s wall"}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def cpu_baseline_port(sites, gt, gr):
    """Fallback when oracle/_ref is absent: the C restatement on in-memory arrays (no text parse)."""
    from oracle import pyoracle as po
    t0 = time.perf_counter()
    o = po.stage1(sites, gt, gr, seed=SEED)
    counts = po.stage2(np.ones((1, o["num_blocks"]), np.int32), o, 0.0)
    ep, _ = po.epochs_from_bins(BINS)
    po.em_run(ep, np.full(len(ep), 1 / 20000.0), counts[0])
    dt = time.perf_counter() - t0
    return {"value": sites.n / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"oracle/liboracle.so stages i-iii on the whole dataset ({sites.n} rows, arrays in memory, no text parse), {dt:.2f} s"}


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on all host cores, same dataset, same files.

    The reference is single-threaded and consumes its generator sequentially, so the only way it can use more than
    one core on ONE pair is by chromosome: one unmodified `Colate --mode mut` process per chromosome (its own
    --chr file; the .colate.in files pre-split by chromosome outside the timed region so that no process pays the
    sequential seek through the other chromosomes' records), started longest-first on a pool of `cores` workers.
    A step = all 22 processes = every row of the dataset parsed from text, joined and sampled, and an EM per
    process (the 21 redundant EMs run concurrently with the longest chromosome's; the critical path holds one)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import pyoracle as po
    cores = os.cpu_count() or 1
    sites, gt, gr = make_dataset(args.rows)
    base_line = {"metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                 "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                 "impl": "reference", "config": config_of(args.rows)}
    if po.ref_cli() is None:
        base = cpu_baseline_port(sites, gt, gr)
        print(json.dumps({**base_line, "value": base["value"], "ms_per_step": None, "cpu_baseline": base,
                          "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0
    d = scratch_dir("colate_ref_")
    try:
        write_dataset_files(d, sites, gt, gr, split_by_chr=True)
        order = np.argsort(-np.diff(sites.site_off))          # longest chromosome first
        cli = po.ref_cli()

        def step(i):
            pending = [int(c) for c in order]
            running = []
            while pending or running:
                while pending and len(running) < cores:
                    c = pending.pop(0)
                    nm = sites.chr_names[c]
                    running.append(subprocess.Popen(ref_cmd(cli, d, f"chr_{nm}.txt", f"t_{nm}.colate.in", f"r_{nm}.colate.in",
                                                            os.path.join(d, f"out{i}_{nm}")),
                                                    stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL))
                os.wait()                                    # any child
                still = []
                for p in running:
                    rc = p.poll()
                    if rc is None:
                        still.append(p)
                    elif rc != 0:
                        raise SystemExit(f"reference process failed with exit code {rc}")
                running = still

        for i in range(args.warmup):
            step(-1 - i)
        t0 = time.perf_counter()
        for i in range(args.steps):
            step(i)
        dt = (time.perf_counter() - t0) / max(1, args.steps)
        val = sites.n / dt
        base = {"value": val, "unit": UNIT, "cores": cores, "kind": "reference",
                "sample": f"the WHOLE dataset per step ({sites.n} rows from the same 22 .mut text files and .colate.in records): one unmodified "
                          f"oracle/_ref/Colate --mode mut process per chromosome, longest first on {cores} cores (.mut parse + site loop + EM each)"}
        print(json.dumps({**base_line, "value": val, "ms_per_step": dt * 1e3, "cpu_baseline": base,
                          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0
    finally:
        shutil.rmtree(d, ignore_errors=True)


# --------------------------------------------------------------------------------------------
# DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum, `ncu --set full`) of the stage-i kernels on THIS
# workload, from the capture summarised in profiles/ (bytes per site / per used row, so that --rows scales it)
NCU_TRAFFIC = None   # filled in from profiles/r02_ncu_stage1_traffic.json when present


def load_traffic():
    p = os.path.join(ROOT, "profiles", "r02_ncu_stage1_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def dump_outputs(dirname, outputs):
    """Write each array as <dirname>/<name>.npy in float64 (exact here: integers below 2**53, 32-bit generator words)."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(dirname, name + ".npy"), np.asarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed passes per leg")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000, help="rows of the whole-genome .mut (default: configs[1])")
    ap.add_argument("--replicates", type=int, default=1000, help="bootstrap replicates of the config-3 leg")
    ap.add_argument("--config3-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config3", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs: device-resident leg only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed device-resident pass returned (rank 0's pair) as DIR/<name>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what this project's timed pass computed; --impl reference runs the reference CLI")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        return reference_arm(args)

    import torch
    import torch.distributed as dist
    from colate_b200 import api, synth
    from colate_b200 import dist as cdist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: colate_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # ---- synthetic pair of this rank (pair index = rank) in both forms: parsed SoA and the reference's file bytes
    sites, gt, gr = make_dataset(args.rows, pair=rank)
    meta = sites.meta()
    keep = []

    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        keep.append(t)
        return t.numpy()

    host = {name: pinned(arr) for name, arr in (("pos", sites.pos), ("ab", sites.age_begin), ("ae", sites.age_end), ("meta", meta))}
    genomes = []
    for g in (gt, gr):
        al = g.anc.astype(np.uint16) | (g.der.astype(np.uint16) << 8)
        first, end = api.chr_ranges(len(sites.chr_names), g.chrom)
        d = {name: pinned(arr) for name, arr in (("bp", g.bp), ("aaf", g.aaf), ("daf", g.daf), ("al", al))}
        d["first"], d["end"] = first, end
        genomes.append(d)
    soa_bytes = sum(v.nbytes for v in host.values()) + sum(sum(d[k].nbytes for k in ("bp", "aaf", "daf", "al", "first", "end")) for d in genomes)
    texts = synth.mut_texts_fast(sites)                                  # the bytes of the 22 .mut files
    text_pin = [pinned(t) for t in texts]
    img_pin = [pinned(synth.colate_in_image(g, sites.chr_names)) for g in (gt, gr)]   # the bytes of the two .colate.in files
    file_bytes = sum(t.nbytes for t in text_pin) + sum(t.nbytes for t in img_pin)

    h = api.Handle(local)
    h.set_option("rejoin", 1)  # the record->row join is part of every timed pass
    site_off = np.ascontiguousarray(sites.site_off, dtype=np.int64)
    ep, _ = api.epochs_from_bins(BINS)
    E = len(ep)
    rates_init = np.full(E, 1.0 / 20000.0)

    def upload_soa():
        h.set_sites(site_off, host["pos"], host["ab"], host["ae"], host["meta"])
        for slot, d in enumerate(genomes):
            api.check(api.lib().colate_set_genome(h._h, slot, d["bp"].shape[0], api.ptr(d["first"]), api.ptr(d["end"]),
                                                  api.ptr(d["bp"]), api.ptr(d["aaf"]), api.ptr(d["daf"]), api.ptr(d["al"]), 0))

    # N > 1: the cohort's .mut files are the same for every pair (make_dataset), i.e. for every rank: each rank copies 1/N of
    # their bytes from its pinned memory and the ranks all-gather the text over NVLink (pairs.SharedMutText) -- the bytes
    # cross PCIe once per node and pass instead of once per GPU; every rank still parses the whole text on its own GPU
    shared_text = None
    if world > 1:
        from colate_b200 import pairs as cpairs
        shared_text = cpairs.SharedMutText(text_pin, torch.device("cuda", local), world, rank)
        file_bytes = shared_text.h2d_bytes + sum(t.nbytes for t in img_pin)

    def upload_files():
        if shared_text is not None:
            h.ingest_mut_device(shared_text.exchange())                  # own slice H2D + NVLink all-gather, then text -> site arrays
        else:
            h.ingest_mut_bytes(text_pin)                                 # text -> site arrays on the GPU
        for slot, img in enumerate(img_pin):
            h.ingest_colate_in(slot, img, sites.chr_names)               # records -> genome arrays on the GPU

    acc = {}
    last = {}                           # what the last pass returned to its caller (--dump-outputs)

    def one_pass():
        s1 = h.stage1(api.mt_seed(SEED), fetch=False)                    # block histograms stay on the device
        for k, v in h.stage1_timing().items():
            acc.setdefault(k, []).append(v)
        t0 = time.perf_counter()
        w = api.draw_block_weights(s1.mt_state, 1, s1.num_blocks)
        h.stage2_bootstrap_dev(w, None, s1.num_blocks, 0.0)
        t1 = time.perf_counter()
        rates, iters, ll = h.stage3_em(1, ep, rates_init)
        t2 = time.perf_counter()
        acc.setdefault("bootstrap_wall_ms", []).append((t1 - t0) * 1e3)
        acc.setdefault("em_wall_ms", []).append((t2 - t1) * 1e3)
        last.update(num_blocks=[s1.num_blocks], n_used=[s1.n_used], mt_state=s1.mt_state, block_weights=w,
                    rates=rates, em_iterations=iters, log_likelihood=ll)
        return s1, rates, iters

    # pipelined form: the EM of the previous pass is still running (EM stream) while this pass is uploaded and taken
    # through stage i; its result is fetched before this pass's bootstrap overwrites the counts
    pend = {"s1": None, "out": None}

    host_ms = {}                        # host wall clock per phase of the pipelined pass (what the host thread waits for)

    def clk(name, t0):
        t1 = time.perf_counter()
        host_ms.setdefault(name, []).append((t1 - t0) * 1e3)
        return t1

    def one_pass_pipelined():
        t = time.perf_counter()
        s1 = h.stage1(api.mt_seed(SEED), fetch=False)
        t = clk("stage1", t)
        if pend["s1"] is not None:
            rates, iters, ll = h.stage3_em_end()
            pend["out"] = (pend["s1"], rates, iters)
        t = clk("wait_for_previous_em", t)
        w = api.draw_block_weights(s1.mt_state, 1, s1.num_blocks)
        h.stage2_bootstrap_dev(w, None, s1.num_blocks, 0.0)
        h.stage3_em_begin(1, ep, rates_init)
        clk("stage2_and_em_launch", t)
        pend["s1"] = s1
        return pend["out"]

    def drain():
        if pend["s1"] is not None:
            rates, iters, ll = h.stage3_em_end()
            pend["out"] = (pend["s1"], rates, iters)
            pend["s1"] = None
        return pend["out"]

    ext = torch.cuda.ExternalStream(h.stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, finish=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ext):
            e0.record()
        out = None
        for _ in range(steps):
            out = fn()
        if finish is not None:
            out = finish()          # the last pass's EM is waited for and read back inside the timed region
        with torch.cuda.stream(ext):
            e1.record()
        torch.cuda.synchronize()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    # ---- value: device-resident pass
    upload_soa()
    for _ in range(args.warmup):
        one_pass()
    acc.clear()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = h.launch_count()
    ms_res, (s1, rates, iters) = timed(one_pass, args.steps)
    launches = h.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"epochs": ep, **last})
    t_stage = {k: float(np.mean(v)) for k, v in acc.items() if k.endswith("_ms")}
    rates_soa = rates.copy()
    # the same device-resident passes with the EM of pass i under stage i of pass i+1 (not the headline `value`: its stage-i
    # kernel times are what `roofline` reports, so the timed passes above run one after the other)
    keep_acc = dict(acc)
    for _ in range(2):
        one_pass_pipelined()
    drain()
    ms_pipe, (_, rates_p, _) = timed(one_pass_pipelined, args.steps, finish=drain)
    if not np.array_equal(rates_p, rates_soa):
        raise SystemExit("bench.py: pipelined and serial passes disagree")
    acc.clear(); acc.update(keep_acc)

    # ---- e2e: the same pass from the file bytes
    e2e = e2e_soa = None
    if not args.no_e2e:
        def e2e_pass():
            upload_files()
            return one_pass()

        def e2e_pass_pipelined():
            t = time.perf_counter()
            upload_files()
            clk("copy_parse_decode", t)
            return one_pass_pipelined()

        for _ in range(2):
            e2e_pass()
        ms_e2e_serial, (s1f, rates_f, iters_f) = timed(e2e_pass, args.steps)
        ms_e2e_serial /= args.steps
        if not (np.array_equal(rates_f, rates_soa) and s1f.n_used == s1.n_used):
            raise SystemExit("bench.py: the pass from the file bytes and the pass from the parsed arrays disagree")
        for _ in range(2):
            e2e_pass_pipelined()
        drain()
        host_ms.clear()
        ms_e2e, (s1f, rates_f, iters_f) = timed(e2e_pass_pipelined, args.steps, finish=drain)
        e2e_host_ms = {k: float(np.mean(v)) for k, v in host_ms.items()}
        ing = h.ingest_stats()
        if not (np.array_equal(rates_f, rates_soa) and s1f.n_used == s1.n_used):
            raise SystemExit("bench.py: the pass from the file bytes and the pass from the parsed arrays disagree")
        d2h = int(rates.nbytes + iters.nbytes + 8 + 624 * 4 + 64 * (len(text_pin) + 4))
        e2e = {"value": world * sites.n / (ms_e2e / args.steps * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(file_bytes),
               "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps,
               "from": "file bytes in pinned host memory: 22 .mut texts (colate_ingest_mut_texts) + 2 .colate.in images (colate_ingest_colate_in)" +
                       ("; the .mut text is the cohort's (the same for every pair / rank): each rank copies 1/N of it and the ranks all-gather it "
                        "over NVLink (pairs.SharedMutText, one NCCL all_gather of %d bytes per pass); h2d_bytes_per_step is per rank" % (shared_text.per * world)
                        if shared_text is not None else ""),
               "mut_parse_kernel_ms": ing["kernel_ms"], "rows_reparsed_on_host": ing["host_fallback_rows"],
               "rates_equal_device_resident_pass": True, "serial_ms_per_step": ms_e2e_serial, "host_phase_ms": e2e_host_ms,
               "pipeline": "EM of pass i on the handle's EM stream (colate_stage3_em_begin/_end) under the copies, parse and stage i of pass i+1; "
                           "every pass's rates are read back inside the timed region"}
        # round 1's leg: parsed SoA in pinned host memory, uploads queued without a sync per call
        h.set_option("async_uploads", 1)

        def soa_pass():
            upload_soa()
            return one_pass()

        for _ in range(2):
            soa_pass()
        ms_soa, _ = timed(soa_pass, args.steps)
        h.set_option("async_uploads", 0)
        e2e_soa = {"value": world * sites.n / (ms_soa / args.steps * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(soa_bytes),
                   "d2h_bytes_per_step": d2h, "ms_per_step": ms_soa / args.steps, "from": "parsed SoA arrays in pinned host memory"}
    clocks = sampler.stop()

    rows = sites.n
    n_used = int(s1.n_used)
    per_step = ms_res / args.steps
    value = world * rows / (per_step * 1e-3)

    # ---- roofline: stage i as a whole (SURVEY.md 8(d)): (40 B x rows + 800 B x used rows) / time of ALL its kernels,
    # measured live with CUDA events on the handle's stream inside the library (colate_last_stage1_timing)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    stage_bytes = 40.0 * rows + 800.0 * n_used
    st_ms = t_stage["total_ms"]
    ach = stage_bytes / (st_ms * 1e-3) / 1e9
    tr = load_traffic()
    traffic = None
    if tr:
        traffic = float(tr["bytes_per_site"]) * rows + float(tr["bytes_per_used_row"]) * n_used
    sample_bytes = 800.0 * n_used
    sample_gbs = sample_bytes / (t_stage["sample_ms"] * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "stage i = parse_tmptmp (k_join x2, flag passes, rank scan, k_jump tree + k_gen, k_compact, k_sample, k_replay)",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                "traffic_source": tr.get("source") if tr else None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": stage_bytes, "launch_ms": st_ms,
                "stage1_pair_site_evals_per_s": rows / (st_ms * 1e-3),
                "formula": "(40 B x rows + 800 B x used rows) / sum of the stage's kernel times",
                "per_phase_ms": {k: t_stage[k] for k in ("join_ms", "flags_ms", "rng_ms", "compact_ms", "sample_ms", "replay_ms")},
                "k_sample": {"algorithmic_bytes_per_launch": sample_bytes, "launch_ms": t_stage["sample_ms"], "achieved": sample_gbs,
                             "frac": sample_gbs / peak,
                             "traffic": (float(tr["k_sample_bytes_per_used_row"]) * n_used) if tr and "k_sample_bytes_per_used_row" in tr else None}}
    em_iters = int(iters[0])
    em = {"R1": {"replicates": 1, "iterations": em_iters, "ms": t_stage["em_wall_ms"],
                 "replicate_iterations_per_s": em_iters / (t_stage["em_wall_ms"] * 1e-3), "kernel": "k_em_split (one replicate on a 16-CTA cluster)"}}

    # ---- config 3: whole genome + R block-bootstrap replicates over all ranks (strong scaling)
    config3 = None
    if not args.no_config3:
        h.close()
        if rank == 0:
            s3, g3t, g3r = sites, gt, gr
        else:
            s3, g3t, g3r = make_dataset(args.rows, pair=0)
        h3 = api.Handle(local)
        cdist.load_shard(h3, s3, g3t, g3r, world, rank)
        be = cdist.CudaBackend(h3)
        R = args.replicates

        def c3_pass():
            return cdist.mut_sharded(be, seed=SEED, bins=BINS, num_bootstraps=R, device="cuda" if world > 1 else "cuda")

        if world == 1 and not dist.is_initialized():
            # a one-rank process group so that N = 1 takes the same code path (NCCL on one GPU)
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("MASTER_PORT", str(29500 + (os.getpid() % 2000)))
            dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", local))
        c3_pass()                                                        # cold: allocations, NCCL connections
        cdist.CALLS.clear()
        c3_pass()
        calls = list(cdist.CALLS)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t_all = []
        em_ms = []
        for _ in range(max(1, args.config3_steps)):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            res = c3_pass()
            torch.cuda.synchronize()
            dt = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            t_all.append(float(dt.item()))
            em_ms.append(res.seconds.get("em", 0.0) * 1e3)
        stats3, _ = res.stats()
        hsh = hashlib.sha256()
        for a in (np.array([res.num_blocks, res.n_used], dtype=np.int64), stats3, res.rates, res.iters.astype(np.int64)):
            hsh.update(np.ascontiguousarray(a).tobytes())
        t3 = float(np.median(t_all))
        tot_iters = int(res.iters.sum())
        config3 = {"workload": f"BASELINE.json configs[2]: the same dataset, --num_bootstraps {R}, chromosomes -> ranks for stage i, replicates -> ranks for stages ii-iii",
                   "wg_1000_bootstrap_s": t3, "seconds_all": t_all, "replicates": R, "n_gpus": world, "scaling": "strong",
                   "timing": "host wall clock around the whole job (device synchronised before and after), max over ranks, median of the repeats; inputs device-resident",
                   "result_sha256": hsh.hexdigest(), "result_hash_covers": "num_blocks, used rows, block histograms [nb,4,185] fp64, rates [R,E] fp64, EM iterations [R] -- equal for every N",
                   "em_iterations_total": tot_iters, "em_iterations_min_max": [int(res.iters.min()), int(res.iters.max())],
                   "nccl_calls_per_job": calls}
        em["R%d" % R] = {"replicates": R, "replicates_per_gpu": (R + world - 1) // world, "iterations": tot_iters, "ms": float(np.median(em_ms)),
                         "replicate_iterations_per_s": tot_iters / (float(np.median(em_ms)) * 1e-3) if np.median(em_ms) > 0 else None,
                         "kernel": "k_em_cta / k_em (one CTA per replicate)"}
        h3.close()

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": config_of(args.rows),
                "workload_detail": {"rows_per_pair": rows, "used_rows_per_pair": n_used, "num_blocks": int(s1.num_blocks), "epochs": E,
                                    "em_iterations": em_iters,
                                    "sharding": "one sample pair per GPU, no data-path collective" if world > 1 else "single GPU",
                                    "l2": "inputs (~0.5 GB SoA + 0.2-1 GB generator stream per pass) exceed the 126 MB L2; no flush needed"},
                "value_pipelined": {"value": world * rows / (ms_pipe / args.steps * 1e-3), "ms_per_step": ms_pipe / args.steps,
                                    "what": "device-resident passes with the EM of pass i overlapped with stage i of pass i+1 (two streams of one handle)"},
                "host_binding": numa,
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "em": em,
                "stage_ms": {**t_stage, "pass_total_ms": per_step}}
        if e2e:
            line["e2e"] = e2e
            line["e2e_soa"] = e2e_soa
        if config3:
            line["config3"] = config3
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_one_core(args.rows, sites, gt, gr, texts)
        print(json.dumps(line))
    if dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()
    if args.no_config3:
        h.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
