"""All-pairs driver (BASELINE.json configs[4]: N genomes -> every ordered pair target=i, reference=j, i<j).

The reference is run once per pair (`Colate --mode mut --target_tmp i --reference_tmp j --seed S`); the
estimator is asymmetric in target / reference (coal.cpp:2198, 2236-2242).  On the device the pairs share
almost everything:
  * the mutation SoA is uploaded once, every genome is joined against it once (k_join; the joined
    columns are cached per genome slot), and because every pair reseeds with the same --seed they all
    consume prefixes of ONE generator stream, which is generated once (colate_set_stream_cache) --
    only the per-pair passes (flags, compaction, sampling, exact replay, stage ii) run per pair;
  * the EM of ALL pairs runs as one launch in throughput mode (one CTA per pair, 2 CTAs/SM), ~0.3 ms per
    pair instead of the ~21 ms the latency-mode EM needs for a single pair.
Results per pair are what `api.mut()` returns for that pair alone (same seed): bit-identical.

Across GPUs (`all_pairs_sharded`, SURVEY.md 8(e).3): pair p -> rank p mod world, every rank holds the mutation SoA and
all genomes, no collective on the data path; the result tables are combined by one all-reduce at the end.

The cohort's `.mut` files are the same for every pair, hence for every rank.  `SharedMutText` brings their bytes to all
GPUs of a node with ONE crossing of PCIe: every rank copies 1/world of the bytes from its pinned host memory and the ranks
all-gather the text over NVLink (687 MB for the whole-genome set: ~86 MB of host-to-device copy per rank at 8 GPUs instead
of 687 MB each through PCIe uplinks that pairs of GPUs share); each rank then parses the text on its own GPU
(`Handle.ingest_mut_device`).  This is the one real exchange step of the pair-sharded path.
"""
from __future__ import annotations

import itertools
import time

import numpy as np

from . import api


def all_pairs(handle: api.Handle, n_genomes: int, seed: int, bins: str = "3,7,0.1", pairs=None, target_age=None,
              reference_age=None, years_per_gen=None, max_iter: int = 100000, em_batch: int = 2048):
    """Genomes must already sit in slots 0..n_genomes-1 of `handle` (set_sites + set_genome / set_mask).
    Returns dict(pairs[P,2], epochs[E], rates[P,E], iters[P], ll[P], num_blocks[P], n_used[P], seconds=dict)."""
    if pairs is None:
        pairs = list(itertools.combinations(range(n_genomes), 2))
    pairs = [(int(i), int(j)) for i, j in pairs]
    for i, j in pairs:
        if not (0 <= i < n_genomes and 0 <= j < n_genomes and i != j):
            raise ValueError(f"bad pair ({i}, {j})")
    age, ypg = api.ages(target_age, reference_age, years_per_gen)
    epochs, ep_null = api.epochs_from_bins(bins, age, ypg)
    init = np.full(epochs.shape[0], 1.0 / 20000.0)
    P = len(pairs)
    counts = np.zeros((P, 2, api.NBINS))
    nb = np.zeros(P, dtype=np.int32)
    nu = np.zeros(P, dtype=np.int64)
    t0 = time.perf_counter()
    mt0 = api.mt_seed(seed)
    handle.set_stream_cache(True)       # every pair reseeds with the same --seed: one generator stream serves them all
    try:
        for p, (i, j) in enumerate(pairs):
            # (the block histograms stay on the device between the stages: fetching 0.6 MB per pair and handing it back cost a
            # third of a pair's time)
            s1 = handle.stage1(mt0, target_slot=i, reference_slot=j, fetch=False)      # the reference reseeds per run
            w = api.draw_block_weights(s1.mt_state, 1, s1.num_blocks)
            counts[p] = handle.stage2_bootstrap_dev(w, None, s1.num_blocks, age, fetch=True)[0]
            nb[p], nu[p] = s1.num_blocks, s1.n_used
    finally:
        handle.set_stream_cache(False)
    t1 = time.perf_counter()
    rates = np.zeros((P, epochs.shape[0]))
    iters = np.zeros(P, dtype=np.int32)
    ll = np.zeros(P)
    for b0 in range(0, P, em_batch):                        # every pair is one "replicate" of one EM launch
        b1 = min(P, b0 + em_batch)
        rates[b0:b1], iters[b0:b1], ll[b0:b1] = handle.stage3_em(b1 - b0, epochs, init, counts[b0:b1], max_iter)
    t2 = time.perf_counter()
    return dict(pairs=np.array(pairs, dtype=np.int32).reshape(P, 2), epochs=epochs, ep_null=ep_null, rates=rates, iters=iters,
                ll=ll, num_blocks=nb, n_used=nu, counts=counts, seconds=dict(stage12=t1 - t0, em=t2 - t1))


def cohort(handle: api.Handle, pairs, seed: int, bins: str | None = None, coal: str | None = None, num_bootstraps: int = 1,
           years_per_gen=None, max_iter: int = 100000, em_batch: int = 2048, front_ends=None):
    """A cohort: pairs = [(target_slot, reference_slot, target_age, reference_age)], ages in years as the CLI takes them (str,
    number or None), genomes (and their masks) already in the handle's slots.  Per pair: stage i from the --seed state (the
    generator stream is shared, colate_set_stream_cache), `num_bootstraps` block weights drawn from the pair's post-stage-i state,
    stage ii at the pair's age and the pair's epoch grid (--bins, or --coal with its initial rates).  Then the EM of all
    P x num_bootstraps replicates on their mixed grids (Handle.stage3_em_grids, em_batch replicates per call).
    Every pair's result is what `api.mut()` returns for that pair alone.
    front_ends: None leaves the handle's "front_end" option as it is.  A list of 0 / 1, one per pair, sets the option to that
    value before the pair's stage i (1 for BAM / BCF genomes: raw count weights and counts / 1e3, as `api.mut` with front_end = 1
    gives them; 0 for .colate.in genomes) and sets it back to 0 at the end.  Returns dict(pairs=[per-pair dict(epochs, ep_null,
    is_ancient, rates[R][E], iters[R], ll[R], num_blocks, n_used, counts[R][2][185])], seconds=dict(stage12, em))."""
    if (bins is None) == (coal is None):
        raise ValueError("give exactly one of bins and coal")
    R = int(num_bootstraps)
    if R < 1:
        raise ValueError("num_bootstraps must be >= 1")
    pairs = list(pairs)
    if front_ends is not None:
        front_ends = [int(f) for f in front_ends]
        if len(front_ends) != len(pairs) or any(f not in (0, 1) for f in front_ends):
            raise ValueError("front_ends: one 0 / 1 per pair")
    txt = lambda a: None if a is None else str(a)
    t0 = time.perf_counter()
    mt0 = api.mt_seed(seed)
    out, grids, grid_key = [], [], {}
    handle.set_stream_cache(True)       # every pair reseeds with the same --seed: one generator stream serves them all
    try:
        for p, (t_slot, r_slot, t_age, r_age) in enumerate(pairs):
            age, ypg = api.ages(txt(t_age), txt(r_age), years_per_gen)
            if front_ends is not None:
                handle.set_option("front_end", front_ends[p])
            s1 = handle.stage1(mt0, target_slot=int(t_slot), reference_slot=int(r_slot), fetch=False)
            w = api.draw_block_weights(s1.mt_state, R, s1.num_blocks)
            counts = handle.stage2_bootstrap_dev(w, None, s1.num_blocks, age, fetch=True)
            if coal is not None:
                epochs, init = api.epochs_from_coal_file(coal, age)
                ep_null = 0
            else:
                epochs, ep_null = api.epochs_from_bins(bins, age, ypg)
                init = np.full(epochs.shape[0], 1.0 / 20000.0)
            key = (epochs.tobytes(), init.tobytes())
            if key not in grid_key:
                grid_key[key] = len(grids)
                grids.append((epochs, init))
            out.append(dict(epochs=epochs, ep_null=ep_null, is_ancient=age > 0.0, num_blocks=s1.num_blocks, n_used=s1.n_used,
                            counts=counts, grid=grid_key[key]))
    finally:
        handle.set_stream_cache(False)
        if front_ends is not None:
            handle.set_option("front_end", 0)
    t1 = time.perf_counter()
    P = len(out)
    grid_of = np.repeat(np.array([p["grid"] for p in out], dtype=np.int32), R)
    counts = np.concatenate([p["counts"] for p in out]) if P else np.zeros((0, 2, api.NBINS))
    E_max = max((g[0].shape[0] for g in grids), default=0)
    rates, iters, ll = np.zeros((P * R, E_max)), np.zeros(P * R, dtype=np.int32), np.zeros(P * R)
    for b0 in range(0, P * R, em_batch):
        b1 = min(P * R, b0 + em_batch)
        used = sorted(set(grid_of[b0:b1].tolist()))            # the grids of this batch only: the launch is sized to its largest
        remap = {g: k for k, g in enumerate(used)}
        r_, i_, l_ = handle.stage3_em_grids([remap[g] for g in grid_of[b0:b1]], [grids[g] for g in used], counts[b0:b1], max_iter)
        rates[b0:b1, :r_.shape[1]], iters[b0:b1], ll[b0:b1] = r_, i_, l_
    t2 = time.perf_counter()
    for p, res in enumerate(out):
        E = res["epochs"].shape[0]
        res.update(rates=rates[p * R:(p + 1) * R, :E].copy(), iters=iters[p * R:(p + 1) * R].copy(), ll=ll[p * R:(p + 1) * R].copy())
        del res["grid"]
    return dict(pairs=out, seconds=dict(stage12=t1 - t0, em=t2 - t1))


def all_pairs_sharded(handle, n_genomes: int, seed: int, bins: str = "3,7,0.1", pairs=None, device="cuda", **kw):
    """`all_pairs` across the ranks of the default torch.distributed process group (NCCL on GPUs, gloo in the CPU
    tests).  Pair p of the list goes to rank p mod world; each rank runs its pairs exactly as `all_pairs` does (its own
    generator-stream cache, its own batched EM launch).  Every rank returns the full tables: the per-rank rows are
    placed into zero tables and summed as 64-bit integers (bit patterns; disjoint supports), so the combined result is
    bit-identical to a single-process run.  `seconds` holds the maximum over the ranks."""
    import torch
    import torch.distributed as dist
    world, rank = dist.get_world_size(), dist.get_rank()
    if pairs is None:
        pairs = list(itertools.combinations(range(n_genomes), 2))
    pairs = [(int(i), int(j)) for i, j in pairs]
    P = len(pairs)
    mine = np.arange(rank, P, world)
    res = all_pairs(handle, n_genomes, seed, bins, pairs=[pairs[k] for k in mine], **kw)
    E = res["epochs"].shape[0]

    def combine(rows, shape, dtype):
        full = np.zeros((P,) + shape, dtype=dtype)
        if mine.shape[0]:
            full[mine] = rows
        t = torch.from_numpy(full.view(np.int64) if dtype == np.float64 else full.astype(np.int64)).to(device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        out = t.cpu().numpy()
        return out.view(np.float64) if dtype == np.float64 else out.astype(dtype)

    out = dict(pairs=np.array(pairs, dtype=np.int32).reshape(P, 2), epochs=res["epochs"], ep_null=res["ep_null"],
               rates=combine(res["rates"], (E,), np.float64), iters=combine(res["iters"], (), np.int32),
               ll=combine(res["ll"], (), np.float64), num_blocks=combine(res["num_blocks"], (), np.int32),
               n_used=combine(res["n_used"], (), np.int64), counts=combine(res["counts"], (2, api.NBINS), np.float64))
    sec = torch.tensor([res["seconds"]["stage12"], res["seconds"]["em"]], dtype=torch.float64, device=device)
    dist.all_reduce(sec, op=dist.ReduceOp.MAX)
    out["seconds"] = dict(stage12=float(sec[0]), em=float(sec[1]))
    return out


class SharedMutText:
    """The `.mut` texts of a cohort (one uint8 array per --chr entry, the SAME bytes on every rank, in pinned host memory) on
    every GPU of the job: rank r copies byte range [r, r+1) * per of their concatenation, `dist.all_gather_into_tensor`
    completes the text on every GPU.  exchange() returns per-chromosome (device pointer, bytes) for ingest_mut_device()."""

    def __init__(self, texts, device, world: int, rank: int):
        import torch
        self.torch = torch
        self.world, self.rank = world, rank
        sizes = [int(t.shape[0]) for t in texts]
        self.sizes = sizes
        self.offs = np.concatenate([[0], np.cumsum([(n + 255) & ~255 for n in sizes])]).astype(np.int64)   # 256-byte aligned starts
        total = int(self.offs[-1])
        self.per = ((total + world - 1) // world + 255) & ~255
        host = torch.zeros(self.per, dtype=torch.uint8)                   # this rank's slice of the concatenation
        if torch.cuda.is_available():
            host = host.pin_memory()
        lo, hi = rank * self.per, (rank + 1) * self.per
        hv = host.numpy()
        for c, t in enumerate(texts):
            a, b = int(self.offs[c]), int(self.offs[c]) + sizes[c]
            x, y = max(a, lo), min(b, hi)
            if x < y:
                hv[x - lo:y - lo] = t[x - a:y - a]
        self.host = host
        self.dev = torch.empty(world * self.per, dtype=torch.uint8, device=device)
        self.h2d_bytes = self.per

    def exchange(self):
        import torch.distributed as dist
        mine = self.dev[self.rank * self.per:(self.rank + 1) * self.per]
        mine.copy_(self.host, non_blocking=True)
        if self.world > 1:
            dist.all_gather_into_tensor(self.dev, mine)
        if self.dev.is_cuda:
            self.torch.cuda.current_stream().synchronize()      # the handle parses on its own stream
        base = self.dev.data_ptr()
        return [(base + int(self.offs[c]), self.sizes[c]) for c in range(len(self.sizes))]
