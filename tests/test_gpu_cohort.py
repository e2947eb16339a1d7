"""GPU: cohorts -- many target / reference pairs with their own ages, masks and bootstrap replicates in one job.

* colate_stage3_em_grids: replicates on mixed epoch grids in one k_em_cta_grids launch equal the oracle and the EM of each
  grid alone, bit for bit;
* pairs.cohort: every pair equals api.mut() run on that pair alone;
* `Colate --mode mut --pairs`: every line's .coal / .bin equal the single-pair CLI run with the same flags byte for byte (and
  the reference CLI's own .coal files for the golden flag sets), with the stale-cache path, --coal warm starts, a failing line
  and several devices."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from colate_b200 import api, pairs, synth
from oracle import pyoracle as po
from helpers import GOLDEN, dataset_from, load

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "colate_b200", "bin", "Colate")


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _block_stats(seed=1, rows=(30000, 20000)):
    sites = synth.make_sites(seed, list(rows), [2.5e8, 1.2e8][:len(rows)])
    return po.stage1(sites, synth.make_genome(seed + 100, sites, 0.7), synth.make_genome(seed + 200, sites, 0.7), seed=seed)


# ---- 1. the mixed-grid EM ------------------------------------------------------------------------------------------------
def _grids():
    """(epochs, rates_init, age in generations): ages 0 / 100 / 250 / 1000 generations, --bins 3,7,0.1 and 3,7,0.2 (different E),
    a --coal warm start, and --bins 3,7,0.05, whose compact store does not fit k_em_cta's shared memory."""
    out = []
    for bins, age in (("3,7,0.1", 0.0), ("3,7,0.2", 100.0), ("3,7,0.1", 250.0), ("3,7,0.2", 1000.0)):
        ep, _ = po.epochs_from_bins(bins, age, 28.0)
        out.append((ep, np.full(len(ep), 1 / 20000.), age))
    ep, ri = api.epochs_from_coal_file(os.path.join(GOLDEN, "cli_ancient.coal"), 250.0)
    out.append((ep, ri, 250.0))
    ep, _ = po.epochs_from_bins("3,7,0.05", 0.0, 28.0)
    out.append((ep, np.full(len(ep), 1 / 20000.), 0.0))
    return out


@pytest.mark.parametrize("with_large", [False, True])
def test_em_grids_equal_each_grid_alone_and_the_oracle(handle, with_large):
    grids = _grids() if with_large else _grids()[:-1]
    assert len({len(g[0]) for g in grids}) >= 3
    o = _block_stats()
    R = 14
    grid_of = np.arange(R) % len(grids)                                     # interleaved
    w = api.draw_block_weights(api.mt_seed(21), R, o["num_blocks"])
    counts = np.stack([po.stage2(w[r:r + 1], o, grids[grid_of[r]][2])[0] for r in range(R)])
    mi = 1200
    n0 = handle.launch_count()
    rates, iters, ll = handle.stage3_em_grids(grid_of, [(g[0], g[1]) for g in grids], counts, max_iter=mi)
    launches = handle.launch_count() - n0
    assert launches == (2 if with_large else 1)            # every fitting grid in one launch; the large one through colate_stage3_em
    E_max = max(len(g[0]) for g in grids)
    assert rates.shape == (R, E_max)
    for r in range(R):
        ep, ri, _ = grids[grid_of[r]]
        E = len(ep)
        assert not rates[r, E:].any()
        r1, i1, l1 = handle.stage3_em(1, ep, ri, counts[r:r + 1], max_iter=mi)
        assert iters[r] == i1[0] and _same(rates[r, :E], r1[0]) and _same(ll[r], l1[0]), r
        if r < len(grids) or r == R - 1:
            ro, it, llo = po.em_run(ep, ri, counts[r], max_iter=mi)
            assert iters[r] == it and _same(rates[r, :E], ro) and _same(ll[r], llo), r
    assert iters.max() > 1000


def test_em_grids_refuses_bad_arguments(handle):
    ep, _ = po.epochs_from_bins("3,7,0.2", 0.0, 28.0)
    c = np.zeros((1, 2, api.NBINS))
    with pytest.raises(api._lib.ColateError):
        handle.stage3_em_grids([1], [(ep, np.full(len(ep), 1 / 20000.))], c)


# ---- 2. pairs.cohort -------------------------------------------------------------------------------------------------------
def test_cohort_equals_mut_on_every_pair(handle):
    sites = synth.make_sites(7, [25000, 15000], [2.4e8, 1.3e8])
    gs = [synth.make_genome(300 + k, sites, 0.6 + 0.05 * k) for k in range(5)]
    masks = {1: [synth.make_mask(91, int(sites.chrom_len[0]), 0.3), synth.make_mask(92, int(sites.chrom_len[1]), 0.2)],
             3: [synth.make_mask(93, int(sites.chrom_len[0]), 0.25), synth.make_mask(94, int(sites.chrom_len[1]) // 2, 0.1)]}
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    for k, g in enumerate(gs):
        handle.set_genome(k, g.chrom, g.bp, g.aaf, g.daf, g.anc.astype(np.uint16) | (g.der.astype(np.uint16) << 8))
        handle.set_mask(k, api.mask_bits_from_seq(masks[k], sites.site_off, sites.pos) if k in masks else None)
    plist = [(0, 1, None, None), (1, 0, "7000", "0"), (2, 3, "1500", None), (4, 2, "250", "0"), (3, 4, None, None), (0, 3, "9000", "1000")]
    R = 3
    res = pairs.cohort(handle, plist, seed=5, bins="3,7,0.2", num_bootstraps=R, years_per_gen=28.0)["pairs"]
    assert len({len(p["epochs"]) for p in res}) > 1                         # the ages really give different grids
    h2 = api.Handle(0)
    try:
        for (t, r, ta, ra), got in zip(plist, res):
            h2.load(sites, gs[t], gs[r], masks.get(t), masks.get(r))
            want = api.mut(h2, seed=5, bins="3,7,0.2", num_bootstraps=R, target_age=ta, reference_age=ra, years_per_gen=28.0)
            assert got["num_blocks"] == want["num_blocks"] and got["n_used"] == want["stage1"].n_used
            assert got["ep_null"] == want["ep_null"] and got["is_ancient"] == want["is_ancient"] and _same(got["epochs"], want["epochs"])
            assert _same(got["counts"], want["counts"])
            assert np.array_equal(got["iters"], want["iters"]) and _same(got["rates"], want["rates"]) and _same(got["ll"], want["ll"])
    finally:
        h2.close()
    # the oracle on the ancient pair with both masks
    t, r, ta, ra = plist[5]
    up = lambda ms: [bytes(m).upper() for m in ms] if ms else None
    o = po.stage1(sites, gs[t], gs[r], seed=5, tmask=up(masks.get(t)), rmask=up(masks.get(r)))
    age, ypg = po.ages(ta, ra, 28.0)
    w = po.draw_block_weights(o["rng"], R, o["num_blocks"])
    counts = po.stage2(w, o, age)
    ep, _ = po.epochs_from_bins("3,7,0.2", age, ypg)
    for i in range(R):
        ro, it, llo = po.em_run(ep, np.full(len(ep), 1 / 20000.), counts[i])
        assert res[5]["iters"][i] == it and _same(res[5]["rates"][i], ro) and _same(res[5]["ll"][i], llo)


# ---- 3.-6. the CLI -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cli_dir():
    z = load("cli_small.npz")
    sites, gt, gr = dataset_from(z)
    d = tempfile.mkdtemp(prefix="colate_cohort_")
    extra = {f"x{k}": synth.make_genome(500 + k, sites, 0.65) for k in range(2)}
    masks = {"tm": [synth.make_mask(70 + c, int(L), 0.3) for c, L in enumerate(sites.chrom_len)]}
    synth.write_dataset(d, sites, {"t": gt, "r": gr, **extra}, masks)
    yield d, z
    shutil.rmtree(d, ignore_errors=True)


def _cli(args, ok=True):
    r = subprocess.run([CLI, "--mode", "mut"] + args, capture_output=True, text=True)
    if ok:
        assert r.returncode == 0, r.stderr
    return r


def _outputs(prefix):
    return open(prefix + ".coal", "rb").read(), open(prefix + ".bin", "rb").read()


def _single(d, line, shared, out):
    """The single-pair CLI run of one pairs-file line."""
    f = line.split()
    args = shared + ["--target_tmp", f[0], "--reference_tmp", f[1], "-o", out]
    for kv in f[3:]:
        k, v = kv.split("=", 1)
        args += ["--" + k, v]
    _cli(args)
    return _outputs(out)


def _write_pairs(d, name, lines):
    p = os.path.join(d, name)
    with open(p, "w") as f:
        f.write("# target reference output [key=value ...]\n\n" + "\n".join(lines) + "\n")
    return p


@pytest.mark.parametrize("name", ["bins02_R1", "bins02_R3", "ancient", "bins01_R1"])
def test_cli_pairs_equal_reference_and_single_runs(cli_dir, name):
    d, z = cli_dir
    args = [str(x) for x in z[f"{name}_args"]]
    opt = dict(zip(args[::2], args[1::2]))
    keys = " ".join(f"{k[2:]}={opt[k]}" for k in ("--target_age", "--reference_age") if k in opt)
    shared = ["--mut", d + "/syn", "--chr", d + "/chr.txt", "--seed", str(int(z["seed"]))]
    shared += sum(([k, v] for k, v in opt.items() if k not in ("--target_age", "--reference_age")), [])
    lines = [f"{d}/x0.colate.in {d}/r.colate.in {d}/{name}_a target_age=3000 target_mask={d}/tm",
             f"{d}/t.colate.in {d}/r.colate.in {d}/{name}_golden {keys}",
             f"{d}/r.colate.in {d}/x1.colate.in {d}/{name}_b",
             f"{d}/t.colate.in {d}/x0.colate.in {d}/{name}_c reference_mask={d}/tm"]
    r = _cli(shared + ["--pairs", _write_pairs(d, f"pairs_{name}.txt", lines)])
    assert "line 4" in r.stderr and f"blocks {int(z[f'{name}_num_blocks'])}" in r.stderr
    assert open(f"{d}/{name}_golden.coal").read() == open(os.path.join(GOLDEN, f"cli_{name}.coal")).read()
    for k, line in enumerate(lines):
        out = line.split()[2]
        assert _outputs(out) == _single(d, line, shared, out + "_single"), (name, k)


def test_cli_pairs_stale_cache_and_warm_start(cli_dir):
    d, z = cli_dir
    common = ["--mut", d + "/syn", "--chr", d + "/chr.txt", "--seed", "1"]
    shutil.copy(os.path.join(GOLDEN, "n2_cache.colate_mat"), d + "/cached.colate_mat")
    lines = [f"{d}/t.colate.in {d}/r.colate.in {d}/cached", f"{d}/x0.colate.in {d}/t.colate.in {d}/fresh target_age=2000"]
    shared = common + ["--bins", "3,7,0.2", "--num_bootstraps", "3"]
    r = _cli(shared + ["--pairs", _write_pairs(d, "pairs_cache.txt", lines)])
    assert "from " + d + "/cached.colate_mat" in r.stderr
    assert open(d + "/cached.coal").read() == open(os.path.join(GOLDEN, "n2_cache.coal")).read()
    cached = _outputs(d + "/cached")
    shutil.copy(os.path.join(GOLDEN, "n2_cache.colate_mat"), d + "/cached_single.colate_mat")
    assert cached == _single(d, lines[0], shared, d + "/cached_single")
    assert _outputs(d + "/fresh") == _single(d, lines[1], shared, d + "/fresh_single")
    # --coal warm start: epochs and initial rates from a .coal file, shifted by each line's age
    lines = [f"{d}/t.colate.in {d}/r.colate.in {d}/warm target_age=7000 reference_age=0", f"{d}/t.colate.in {d}/x1.colate.in {d}/warm0 target_age=0"]
    shared = common + ["--coal", os.path.join(GOLDEN, "cli_ancient.coal"), "--years_per_gen", "28"]
    _cli(shared + ["--pairs", _write_pairs(d, "pairs_warm.txt", lines)])
    assert open(d + "/warm.coal").read() == open(os.path.join(GOLDEN, "n2_warm.coal")).read()
    assert _outputs(d + "/warm0") == _single(d, lines[1], shared, d + "/warm0_single")


def test_cli_pairs_failing_line_leaves_the_others(tmp_path):
    """One line's pair has used rows in 501 genomic blocks (COLATE_ERR_BLOCKS); its genomes' first-contig subsets make
    pairs of at most 70 blocks.  The failing line is named, writes nothing, and the others equal their single runs."""
    from test_gpu_stage1_shapes import _blocks_dataset
    sites, gt, gr = _blocks_dataset(17, bump=True)
    first = lambda g: synth.Genome(g.chrom[g.chrom == 0], g.bp[g.chrom == 0], g.anc[g.chrom == 0], g.der[g.chrom == 0],
                                   g.aaf[g.chrom == 0], g.daf[g.chrom == 0])
    d = str(tmp_path)
    synth.write_dataset(d, sites, {"t": gt, "r": gr, "a": first(gt), "b": first(gr)})
    shared = ["--mut", d + "/syn", "--chr", d + "/chr.txt", "--seed", "3", "--bins", "3,7,0.2", "--num_bootstraps", "2"]
    lines = [f"{d}/a.colate.in {d}/b.colate.in {d}/ab", f"{d}/t.colate.in {d}/r.colate.in {d}/tr", f"{d}/b.colate.in {d}/a.colate.in {d}/ba"]
    r = _cli(shared + ["--pairs", _write_pairs(d, "pairs.txt", lines)], ok=False)
    assert r.returncode != 0
    assert "line 4" in r.stderr and "FAILED" in r.stderr and "1 of 3 pairs failed" in r.stderr, r.stderr
    assert not os.path.exists(d + "/tr.coal") and not os.path.exists(d + "/tr.bin")
    for line in (lines[0], lines[2]):
        out = line.split()[2]
        assert _outputs(out) == _single(d, line, shared, out + "_single")


def test_cli_pairs_devices(cli_dir):
    """Pairs dealt round-robin to the devices, one handle and host thread each: the output does not depend on the list
    (two handles on one GPU everywhere; two GPUs where there are two)."""
    import torch
    d, z = cli_dir
    shared = ["--mut", d + "/syn", "--chr", d + "/chr.txt", "--seed", "2", "--bins", "3,7,0.2", "--num_bootstraps", "4"]
    lists = ["0", "0,0"] + (["0,1"] if torch.cuda.device_count() > 1 else [])
    res = []
    for i, devs in enumerate(lists):
        lines = [f"{d}/t.colate.in {d}/r.colate.in {d}/dv{i}_0 target_age=5000", f"{d}/x0.colate.in {d}/x1.colate.in {d}/dv{i}_1",
                 f"{d}/x1.colate.in {d}/t.colate.in {d}/dv{i}_2 target_mask={d}/tm", f"{d}/r.colate.in {d}/x0.colate.in {d}/dv{i}_3"]
        _cli(shared + ["--devices", devs, "--pairs", _write_pairs(d, f"pairs_dev{i}.txt", lines)])
        res.append([_outputs(f"{d}/dv{i}_{k}") for k in range(4)])
    for other in res[1:]:
        assert other == res[0]

