"""Stage i (parse_tmptmp, coal.cpp:2071-2321) on input shapes synth.make_sites / make_genome never produce: repeated .mut
positions and repeated record positions, record streams much denser than the rows, block edges and the 500-block limit,
deep coverage and the weight regimes it brings.  Every device result is compared with the oracle bit for bit.

The oracle-only section at the top runs without a GPU: the hand-checked repeated-position case pins the oracle's
restatement of the reference's reader independently of the device."""
import os
import tempfile

import numpy as np
import pytest

from colate_b200 import api, synth
from oracle import pyoracle as po
from test_gpu_stage1 import _compare_stage1

gpu = pytest.mark.gpu

B = 30_000_000                     # COLATE_BLOCK_BASES
JOIN_TILE, JOIN_CAP = 256, 1024    # kernels_sites.cu: rows per join tile, record positions staged per tile
ACGT = np.frombuffer(b"ACGT", np.uint8)


# ---------------------------------------------------------------------------------------------------- dataset builders
def _sites(pos_per_chr, rng, names=None, lens=None):
    """Rows at the given positions (ascending per chromosome, repeats allowed), filters passed, random alleles and ages."""
    names = names or [str(c + 1) for c in range(len(pos_per_chr))]
    off = np.concatenate([[0], np.cumsum([len(p) for p in pos_per_chr])]).astype(np.int64)
    pos = np.concatenate([np.asarray(p, np.int64) for p in pos_per_chr]).astype(np.int32)
    n = pos.shape[0]
    ab = np.where(rng.random(n) < 0.3, 0.0, np.exp(rng.uniform(np.log(10.0), np.log(2e4), n))).astype(np.float32)
    ae = (ab.astype(np.float64) + np.exp(rng.uniform(np.log(50.0), np.log(5e4), n))).astype(np.float32)
    a = rng.integers(0, 4, n)
    d = (a + rng.integers(1, 4, n)) % 4
    lens = lens or [int(p[-1]) + 1 if len(p) else 1000 for p in pos_per_chr]
    return synth.Sites(names, off, pos, ab, ae, np.zeros(n, np.uint8), np.ones(n, np.int32), ACGT[a].copy(), ACGT[d].copy(),
                       np.zeros(n, np.uint8), list(lens))


def _genome(recs):
    """recs: list of (chrom, bp, anc, der, aaf, daf) in file order."""
    if not recs:
        z = np.zeros(0, np.int32)
        return synth.Genome(z, z, z.astype(np.uint8), z.astype(np.uint8), z, z)
    c, bp, a, d, aaf, daf = zip(*recs)
    return synth.Genome(np.array(c, np.int32), np.array(bp, np.int32), np.array(a, np.uint8), np.array(d, np.uint8),
                        np.array(aaf, np.int32), np.array(daf, np.int32))


def _chr_of_rows(sites):
    return (np.searchsorted(sites.site_off, np.arange(sites.n), side="right") - 1).astype(np.int32)


def _concat(parts):
    """Datasets (sites, target, reference) side by side: the chromosomes of each part in turn."""
    names, lens, offs, fields, gts, grs = [], [], [0], [], [], []
    c0 = 0
    for s, gt, gr in parts:
        k = len(s.chr_names)
        names += [str(c0 + c + 1) for c in range(k)]
        lens += list(s.chrom_len)
        offs += list(offs[-1] + s.site_off[1:])
        fields.append((s.pos, s.age_begin, s.age_end, s.flipped, s.n_branch, s.anc, s.der, s.odd))
        gts.append((gt, c0)); grs.append((gr, c0))
        c0 += k
    cat = [np.concatenate(x) for x in zip(*fields)]
    sites = synth.Sites(names, np.array(offs, np.int64), *cat, lens)

    def g(lst):
        return synth.Genome(np.concatenate([x.chrom + c for x, c in lst]).astype(np.int32),
                            *[np.concatenate([getattr(x, f) for x, _ in lst]) for f in ("bp", "anc", "der", "aaf", "daf")])
    return sites, g(gts), g(grs)


def _pass_rows(sites, mask):
    """coal.cpp:2169-2174 per row: the mask (bytes per chromosome) says 'P', or the position lies beyond it."""
    if mask is None:
        return np.ones(sites.n, bool)
    ok = np.ones(sites.n, bool)
    for c, s in enumerate(mask):
        lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
        p = sites.pos[lo:hi].astype(np.int64)
        arr = np.frombuffer(s, np.uint8)
        inside = p < arr.shape[0]
        ok[lo:hi][inside] = arr[p[inside] - 1] == ord("P")
    return ok


def _reader(sites, gt, gr, tmask=None, rmask=None):
    """The reference's sequential reader (coal.cpp:2125-2219) restated per row, without the sampling: which rows are used
    and which record each stream had loaded for them.  Returns (used[n_site], t_rec[n_site], r_rec[n_site]) (-1: none)."""
    meta = sites.meta()
    tp, rp = _pass_rows(sites, tmask), _pass_rows(sites, rmask)
    used = np.zeros(sites.n, bool)
    hit = {0: np.full(sites.n, -1), 1: np.full(sites.n, -1)}

    class Stream:
        def __init__(self, g):
            self.g, self.next, self.k = g, 0, -1
            self.daf = self.aaf = 0

        def read(self):
            if self.next >= self.g.n:
                return False
            self.k = self.next; self.next += 1
            self.daf, self.aaf = int(self.g.daf[self.k]), int(self.g.aaf[self.k])
            return True

        def on(self, c):
            return self.k >= 0 and int(self.g.chrom[self.k]) == c

        def look(self, c, p, anc, der):
            self.daf = self.aaf = 0
            while self.on(c) and int(self.g.bp[self.k]) < p:
                if not self.read():
                    break
            return self.on(c) and int(self.g.bp[self.k]) == p and self.g.anc[self.k] == anc and self.g.der[self.k] == der

    st, sr = Stream(gt), Stream(gr)
    for c in range(len(sites.chr_names)):
        for s in (sr, st):
            while not s.on(c):
                if not s.read():
                    break
        for m in range(int(sites.site_off[c]), int(sites.site_off[c + 1])):
            if not meta[m] & 1:
                continue
            p, anc, der = int(sites.pos[m]), sites.anc[m], sites.der[m]
            use = bool(tp[m] and rp[m])
            if use and not sr.look(c, p, anc, der):
                use = False
            if sr.daf == 0:
                use = False
            if use and not st.look(c, p, anc, der):
                use = False
            if st.daf + st.aaf == 0:
                use = False
            if use:
                used[m] = True
                hit[0][m], hit[1][m] = st.k, sr.k
    return used, hit[0], hit[1]


def _blocks_of_used(sites, used):
    """Genomic block of every used row (coal.cpp:2227-2234, 2306-2310) and the number of blocks."""
    blk = np.full(sites.n, -1)
    base = 0
    for c in range(len(sites.chr_names)):
        lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
        u = np.nonzero(used[lo:hi])[0] + lo
        blk[u] = base + (sites.pos[u].astype(np.int64) - 1) // B
        base += int((int(sites.pos[u[-1]]) - 1) // B + 1) if u.shape[0] else 1
    return blk, base


def _rep_mask(chrom, pos):
    """Rows (or records) whose position equals a neighbour's on the same chromosome."""
    same = (chrom[1:] == chrom[:-1]) & (pos[1:] == pos[:-1])
    r = np.zeros(pos.shape[0], bool)
    r[1:] |= same; r[:-1] |= same
    return r


# ---- A: repeated positions -----------------------------------------------------------------------------------------
def _hand_case(swap):
    """.mut rows 100, 200, 200, 300, 400, 500 (A/C); target: one record at every row position; reference: 100, 200 A/G,
    200 A/C, 300, 350, 400, 500, 500 (A/C unless said).  Every row's age interval lies inside one age bin of its own."""
    pos = [100, 200, 200, 300, 400, 500]
    ages = [60.0, 300.0, 1500.0, 7000.0, 30000.0, 200000.0]
    n = len(pos)
    ab = np.array(ages, np.float32)
    ae = (ab * np.float32(1.0005)).astype(np.float32)
    A, Cc = ord("A"), ord("C")
    sites = synth.Sites(["1"], np.array([0, n], np.int64), np.array(pos, np.int32), ab, ae, np.zeros(n, np.uint8),
                        np.ones(n, np.int32), np.full(n, A, np.uint8), np.full(n, Cc, np.uint8), np.zeros(n, np.uint8), [1000])
    gt = _genome([(0, p, A, Cc, 1, 1) for p in (100, 200, 300, 400, 500)])
    at200 = [(0, 200, A, ord("G"), 1, 2), (0, 200, A, Cc, 1, 2)]
    if swap:
        at200 = at200[::-1]
    gr = _genome([(0, 100, A, Cc, 1, 2)] + at200 + [(0, p, A, Cc, 1, 2) for p in (300, 350, 400, 500, 500)])
    return sites, gt, gr


def _hand_case_rows(o, sites):
    """Rows whose 100 samples the oracle put into the notshared tallies (every row has a bin of its own)."""
    bins = [po.lib().oracle_bin_of_double_age(float(a)) for a in sites.age_begin]
    assert bins == [po.lib().oracle_bin_of_double_age(float(a)) for a in sites.age_end]
    assert len(set(bins)) == sites.n
    tal = o["n_notshared"].sum(0)
    assert set(np.unique(tal)) <= {0, 100}
    return [m for m in range(sites.n) if tal[bins[m]] == 100]


def _repeats_dataset(seed, n_chr=3, n_pos=1400, L=4_000_000):
    """Runs of 2-4 .mut rows at one position (same alleles, different alleles, one of the run filtered), runs of 2-3
    records at one bp in both genomes (identical, different alleles, different counts), placed at a chromosome's first row
    and first record and across the first join-tile boundaries; sparse enough that look-ahead reads pull runs' first records."""
    rng = np.random.default_rng(seed)
    pos_chr, kinds = [], []
    for c in range(n_chr):
        u = np.sort(rng.choice(np.arange(1, L, 3), n_pos, replace=False))
        mult = np.where(rng.random(n_pos) < 0.2, rng.integers(2, 5, n_pos), 1)
        mult[0] = max(mult[0], 2)                                           # the chromosome's first row
        for edge in (JOIN_TILE, 2 * JOIN_TILE):                             # a run over rows edge-1 / edge
            start = np.concatenate([[0], np.cumsum(mult)[:-1]])
            j = int(np.searchsorted(start, edge - 1, side="right") - 1)
            mult[j] = max(mult[j], edge + 1 - start[j])
        pos_chr.append(np.repeat(u, mult))
        kinds.append((u, mult))
    sites = _sites(pos_chr, rng, lens=[L] * n_chr)
    rchr = _chr_of_rows(sites)
    # alleles inside a run: same as its first row, or a different derived allele; a row of some runs filtered out
    for c in range(n_chr):
        lo = int(sites.site_off[c])
        u, mult = kinds[c]
        start = lo + np.concatenate([[0], np.cumsum(mult)[:-1]])
        for s, k in zip(start, mult):
            if k < 2:
                continue
            for i in range(s + 1, s + k):
                r = rng.random()
                if r < 0.5:
                    sites.anc[i], sites.der[i] = sites.anc[s], sites.der[s]
                elif r < 0.8:
                    sites.anc[i] = sites.anc[s]
                    sites.der[i] = ACGT[(np.searchsorted(ACGT, sites.anc[s]) + rng.integers(1, 4)) % 4]
                elif r < 0.9:
                    sites.anc[i], sites.der[i] = sites.anc[s], sites.der[s]
                    sites.flipped[i] = 1
                else:
                    sites.anc[i], sites.der[i] = sites.anc[s], sites.der[s]
                    sites.n_branch[i] = 2

    def genome(p_present, gseed):
        g = np.random.default_rng(gseed)
        recs = []
        for c in range(n_chr):
            lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
            pos = sites.pos[lo:hi]
            first_pos = True
            for p in np.unique(pos):
                rows = np.nonzero(pos == p)[0] + lo
                present = first_pos or g.random() < p_present
                if not first_pos and g.random() < 0.1:                       # a record at p - 1, which is not a row
                    N = int(g.integers(1, 6)); d = int(g.binomial(N, 0.4))
                    recs.append((c, int(p) - 1, sites.anc[rows[0]], sites.der[rows[0]], N - d, d))
                if not present:
                    continue
                k = 2 if first_pos else (int(g.integers(2, 4)) if g.random() < 0.25 else 1)
                first_pos = False
                m = rows[g.integers(0, rows.shape[0])]
                a, d_ = sites.anc[m], sites.der[m]
                N = int(g.integers(1, 7)); d = int(g.binomial(N, 0.45))
                run = [(c, int(p), a, d_, N - d, d)]
                for _ in range(k - 1):
                    r = g.random()
                    if r < 0.35:
                        run.append(run[0])                                   # identical
                    elif r < 0.7:
                        m2 = rows[g.integers(0, rows.shape[0])]
                        d2 = sites.der[m2] if sites.der[m2] != d_ else ACGT[(np.searchsorted(ACGT, a) + 2) % 4]
                        run.append((c, int(p), a, d2, 1, int(g.integers(1, 4))))   # different alleles
                    else:
                        N2 = int(g.integers(1, 7)); dd = int(g.integers(0, N2 + 1))
                        run.append((c, int(p), a, d_, N2 - dd, dd))           # same alleles, different counts
                if g.random() < 0.3:
                    g.shuffle(run)
                recs += run
        return _genome(recs)

    gt = genome(0.72, seed + 100)
    gr = genome(0.8, seed + 200)
    return sites, gt, gr, rchr


def _repeat_masks(sites, seed):
    """Masks with a few % N, cut through some runs' positions, the target's shorter than its chromosome."""
    rng = np.random.default_rng(seed)
    tm, rm = [], []
    for c, L in enumerate(sites.chrom_len):
        for out, frac, ln in ((tm, 0.05, int(L) * 3 // 4), (rm, 0.04, int(L))):
            m = np.frombuffer(synth.make_mask(int(rng.integers(1 << 30)), ln, frac, run_lo=50, run_hi=3000), np.uint8).copy()
            lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
            rep = np.unique(sites.pos[lo:hi][_rep_mask(np.zeros(hi - lo), sites.pos[lo:hi])])
            cut = rep[rng.random(rep.shape[0]) < 0.1]
            cut = cut[cut <= ln]
            m[cut - 1] = ord("N")
            out.append(m.tobytes())
    return tm, rm


def test_repeated_positions_hand_case_oracle():
    """The first record of a chromosome is counted dead by the seek, the first record of an equal-bp run is the one compared,
    and a repeated .mut row gets no counts (the reader only loads counts when it reads a new record)."""
    for swap, want in ((False, [3, 4, 5]), (True, [1, 3, 4, 5])):
        sites, gt, gr = _hand_case(swap)
        o = po.stage1(sites, gt, gr, seed=1)
        assert o["num_blocks"] == 1 and o["n_used_total"] == len(want)
        assert _hand_case_rows(o, sites) == want
        used, _, _ = _reader(sites, gt, gr)
        assert list(np.nonzero(used)[0]) == want


@pytest.mark.parametrize("seed", [3, 4])
def test_repeated_positions_reader_restatement_oracle(seed):
    """The per-row restatement (_reader) agrees with the oracle's used rows per block on the random repeat datasets, and the
    datasets contain repeated rows and repeated records that are used as well as ones that are dropped."""
    sites, gt, gr, rchr = _repeats_dataset(seed)
    for masks in (False, True):
        tm, rm = _repeat_masks(sites, seed) if masks else (None, None)
        o = po.stage1(sites, gt, gr, seed=seed, tmask=tm, rmask=rm)
        used, th, rh = _reader(sites, gt, gr, tm, rm)
        blk, nb = _blocks_of_used(sites, used)
        assert nb == o["num_blocks"]
        assert np.array_equal(np.bincount(blk[used], minlength=nb), o["n_used"])
        rep_rows = _rep_mask(rchr, sites.pos)
        cand = rep_rows & ((sites.meta() & 1) != 0) & _pass_rows(sites, tm) & _pass_rows(sites, rm)
        assert (cand & used).sum() > 20 and (cand & ~used).sum() > 20
        for g, h in ((gt, th), (gr, rh)):
            rep_rec = _rep_mask(g.chrom, g.bp)
            hit = np.zeros(g.n, bool); hit[h[used]] = True
            assert (rep_rec & hit).sum() > 10 and (rep_rec & ~hit).sum() > 10
        # a repeated row whose run's first record the seek or an earlier look-ahead had already loaded
        first_row = sites.site_off[:-1]
        assert rep_rows[first_row].all() and not used[first_row].any()


def _dense_tiles(sites, g):
    """Per join tile, mirroring k_join_bounds: (chromosome, first tile of it, last tile of it, w0 == first, n_w, w0)."""
    first, end = api.chr_ranges(len(sites.chr_names), g.chrom)
    out = []
    for c in range(len(sites.chr_names)):
        lo, hi = int(sites.site_off[c]), int(sites.site_off[c + 1])
        if first[c] < 0:
            continue
        bp = g.bp[first[c]:end[c]]
        for m0 in range(lo, hi, JOIN_TILE):
            m1 = min(m0 + JOIN_TILE, hi)
            w0 = int(first[c]) + int(np.searchsorted(bp, sites.pos[m0], "left"))
            w1 = int(first[c]) + int(np.searchsorted(bp, sites.pos[m1 - 1], "right"))
            base = w0 - 1 if w0 > first[c] else w0
            out.append((c, m0 == lo, m1 == hi, w0 == first[c], w1 - base, w0))
    return out


def _dense_dataset(seed):
    """Rows 1 kb apart; most tiles sparse (records at ~75 % of the rows), some with extra records between the rows (and a
    few repeated record positions) so that a tile's window holds exactly 1024 .. 1027 records, or 10-50 per row."""
    rng = np.random.default_rng(seed)
    # chromosome 0: tiles 1-4 -> 1024..1027, tile 6 ~50 / row, tile 7 ~10 / row, dense partial last tile
    # chromosome 1: dense first tile (w0 == first), sparse otherwise
    plan = [{1: 1024, 2: 1025, 3: 1026, 4: 1027, 6: 12800, 7: 2600, 10: 2100}, {0: 4000, 1: 1025}]
    rows = [10 * JOIN_TILE + 77, 3 * JOIN_TILE + 40]
    pos_chr = [1000 * np.arange(1, k + 1) for k in rows]
    sites = _sites(pos_chr, rng, lens=[1000 * (k + 2) for k in rows])

    def genome(gseed):
        g = np.random.default_rng(gseed)
        recs = []
        for c, k in enumerate(rows):
            lo = int(sites.site_off[c])
            has = g.random(k) < 0.75
            for t in plan[c]:                                         # a planned tile's first row and the row in front of it
                has[max(t * JOIN_TILE - 1, 0):t * JOIN_TILE + 1] = True   # have records: the window's first record is a hit
            chrom_recs = []
            for t in range((k + JOIN_TILE - 1) // JOIN_TILE):
                m0, m1 = t * JOIN_TILE, min((t + 1) * JOIN_TILE, k)
                tile = [(c, int(pos_chr[c][i]), sites.anc[lo + i], sites.der[lo + i]) for i in range(m0, m1) if has[i]]
                if t in plan[c]:
                    front = 1 if chrom_recs else 0
                    extra = plan[c][t] - front - len(tile)
                    n_dup = min(20, extra // 4)
                    dup_at = 1 + g.choice(len(tile) - 1, n_dup, replace=False)
                    cand = np.arange(pos_chr[c][m0] + 1, pos_chr[c][m1 - 1])
                    cand = cand[cand % 1000 != 0]
                    nonrow = np.sort(g.choice(cand, extra - n_dup, replace=False))
                    more = [(c, int(p), ACGT[g.integers(0, 4)], ACGT[g.integers(0, 4)]) for p in nonrow]
                    for j in dup_at:                                  # a repeated position: another allele pair in front
                        more.append((c, tile[j][1], tile[j][2], ACGT[(np.searchsorted(ACGT, tile[j][3]) + 1) % 4]))
                    tile = sorted(tile + more, key=lambda r: r[1])     # (stable: the extra record of a repeated bp ...
                    tile = _front_dups(tile)                           # ... is moved in front of the row's own)
                chrom_recs += tile
            for (cc, p, a, d) in chrom_recs:
                N = int(g.integers(1, 8)); dd = int(g.integers(1, N + 1)) if g.random() < 0.9 else 0
                recs.append((cc, p, a, d, N - dd, dd))
        return _genome(recs)

    return sites, genome(seed + 1), genome(seed + 2)


def _front_dups(tile):
    """Within runs of equal bp, put the later-added records (different alleles) first: the row's own record is shadowed."""
    out, i = [], 0
    while i < len(tile):
        j = i
        while j < len(tile) and tile[j][1] == tile[i][1]:
            j += 1
        out += tile[i:j][::-1]
        i = j
    return out


def test_dense_windows_reach_the_staging_limit():
    """The dense datasets contain tiles whose record window holds 1024, 1025 (still staged), 1026, 1027 (global search) and
    far more records, a dense first tile of a chromosome (w0 == first) and a dense last tile, with repeated positions inside."""
    sites, gt, gr = _dense_dataset(5)
    used, t_rec, r_rec = _reader(sites, gt, gr)
    for g, rec in ((gt, t_rec), (gr, r_rec)):
        tiles = _dense_tiles(sites, g)
        nw = {t[4] for t in tiles}
        assert {JOIN_CAP, JOIN_CAP + 1, JOIN_CAP + 2, JOIN_CAP + 3} <= nw and max(nw) > 10 * JOIN_TILE
        assert any(t[1] and t[3] and t[4] > JOIN_CAP + 1 for t in tiles)          # dense first tile, w0 == first
        assert any(t[2] and t[4] > JOIN_CAP + 1 for t in tiles)                   # dense last tile
        assert any(t[4] <= JOIN_CAP + 1 for t in tiles if t[0] == 0) and any(t[4] > JOIN_CAP + 1 for t in tiles if t[0] == 0)
        assert _rep_mask(g.chrom, g.bp).sum() > 40
        # used rows whose record opens a global-search window behind earlier records (k_join's `lo > first` case)
        opens = [t[5] for t in tiles if t[4] > JOIN_CAP + 1 and not t[3]]
        assert np.isin(rec[used], opens).sum() >= 2
    o = po.stage1(sites, gt, gr, seed=5)
    assert o["n_used_total"] == used.sum() > 1000


# ---- C: block edges and the 500-block limit -------------------------------------------------------------------------
def _blocks_dataset(seed, bump=False):
    """Four long contigs whose last row -- always used -- ends them at 70, 70, 51 and 30 blocks, and 279 short ones of one
    block: exactly 500 blocks.  bump=True moves the last row of the 30-block contig one base up, over its block edge: 501.
    Rows at k*30e6 - 1, k*30e6, k*30e6 + 1; blocks whose only row sits on an edge; runs of empty blocks."""
    rng = np.random.default_rng(seed)
    lasts = [2_100_000_000, 2_100_000_000, 1_500_000_001, 900_000_000 + (1 if bump else 0)]
    pos_chr, edge_only = [], []
    for last in lasts:
        nblk = (last - 1) // B + 1
        occ = np.nonzero(rng.random(nblk) < 0.5)[0]
        occ = occ[occ < nblk - 3]
        p = [rng.integers(b * B + 1, (b + 1) * B + 1, 12) for b in occ]
        for k in rng.choice(np.arange(1, nblk - 3), 8, replace=False):          # rows around block edges
            p.append(np.array([k * B - 1, k * B, k * B + 1]))
        # blocks nblk-3 / nblk-2 hold one row each, on their lower / upper edge; empty blocks in front of them
        p.append(np.array([(nblk - 3) * B + 1, (nblk - 1) * B, last]))
        edge_only += [(nblk - 3) * B + 1, (nblk - 1) * B]
        pos_chr.append(np.unique(np.concatenate(p)))
    for _ in range(279):
        pos_chr.append(np.unique(rng.integers(1, 1_000_000, int(rng.integers(1, 6)))))
    lens = [int(p[-1]) + 1 for p in pos_chr]
    sites = _sites(pos_chr, rng, lens=lens)
    chr_of = _chr_of_rows(sites)

    def genome(p, gseed):
        g = np.random.default_rng(gseed)
        keep = g.random(sites.n) < p
        keep[sites.site_off[1:] - 1] = keep[sites.site_off[1:] - 2 * (np.diff(sites.site_off) > 1)] = True
        keep[sites.site_off[:-1]] = True
        keep[np.isin(sites.pos, edge_only)] = True
        idx = np.nonzero(keep)[0]
        N = g.integers(1, 6, idx.shape[0]); d = g.integers(1, N + 1)
        return synth.Genome(chr_of[idx], sites.pos[idx].copy(), sites.anc[idx].copy(), sites.der[idx].copy(),
                            (N - d).astype(np.int32), d.astype(np.int32))

    return sites, genome(0.85, seed + 1), genome(1.0, seed + 2)


def _many_contigs_dataset(seed, n_contigs=1100):
    """More contigs than k_chr's 1024 threads; each 1-3 blocks long, every one with records in both genomes."""
    rng = np.random.default_rng(seed)
    pos_chr = [np.unique(rng.integers(1, int(rng.choice([1e6, 5e7, 9e7])), int(rng.integers(1, 8)))) for _ in range(n_contigs)]
    sites = _sites(pos_chr, rng, lens=[int(p[-1]) + 1 for p in pos_chr])
    chr_of = _chr_of_rows(sites)

    def genome(p, gseed):
        g = np.random.default_rng(gseed)
        keep = g.random(sites.n) < p
        keep[sites.site_off[:-1]] = True
        idx = np.nonzero(keep)[0]
        N = g.integers(1, 6, idx.shape[0]); d = g.integers(0, N + 1)
        return synth.Genome(chr_of[idx], sites.pos[idx].copy(), sites.anc[idx].copy(), sites.der[idx].copy(),
                            (N - d).astype(np.int32), d.astype(np.int32))

    return sites, genome(0.8, seed + 1), genome(0.9, seed + 2)


def _sub(sites, g, lo, hi):
    """Contigs [lo, hi) of a dataset as a dataset of their own (records of those contigs only, ids shifted)."""
    s0, s1 = int(sites.site_off[lo]), int(sites.site_off[hi])
    sl = slice(s0, s1)
    s = synth.Sites(sites.chr_names[lo:hi], sites.site_off[lo:hi + 1] - s0, sites.pos[sl], sites.age_begin[sl], sites.age_end[sl],
                    sites.flipped[sl], sites.n_branch[sl], sites.anc[sl], sites.der[sl], sites.odd[sl], sites.chrom_len[lo:hi])
    k = (g.chrom >= lo) & (g.chrom < hi)
    return s, synth.Genome(g.chrom[k] - lo, g.bp[k], g.anc[k], g.der[k], g.aaf[k], g.daf[k])


def test_block_limit_oracle():
    """Exactly 500 blocks pass and 501 are refused (COLATE_ERR_BLOCKS); the per-row restatement gives the same blocks."""
    sites, gt, gr = _blocks_dataset(8)
    assert sites.pos.max() <= 2_100_000_000
    o = po.stage1(sites, gt, gr, seed=8)
    used, _, _ = _reader(sites, gt, gr)
    blk, nb = _blocks_of_used(sites, used)
    assert o["num_blocks"] == nb == 500
    assert np.array_equal(np.bincount(blk[used], minlength=nb), o["n_used"])
    assert (o["n_used"] == 0).sum() > 50                                        # runs of empty blocks
    on_edge = used & (((sites.pos.astype(np.int64) - 1) % B == 0) | (sites.pos.astype(np.int64) % B == 0))
    assert on_edge.sum() > 10
    sites, gt, gr = _blocks_dataset(8, bump=True)
    assert po.stage1(sites, gt, gr, seed=8)["num_blocks"] == -3


# ---- D: deep coverage ------------------------------------------------------------------------------------------------
def _deep_dataset(seed):
    """Chromosome 1: one 30 Mb block with 60 k rows, every one with a record in both genomes (>= 50 k used rows in one
    block).  Chromosome 2: ages narrow enough for all 100 samples to share a bin, age_end on the age-bin thresholds, rows
    whose target counts make the pseudo-genotype a tie (N = 4 DAF: 0.5; N = 4/3 DAF: AAF gives 0.5).  Target N from 20 to
    ~2000, reference N from 1 to 5008."""
    rng = np.random.default_rng(seed)
    p1 = np.unique(rng.integers(1, B, 61000))[:60000]
    p2 = np.unique(rng.integers(1, 9 * 10**7, 20100))[:20000]
    sites = _sites([p1, p2], rng, lens=[B, 9 * 10**7])
    n = sites.n
    o2 = int(sites.site_off[1])
    thr = np.zeros(186)
    assert api.lib().colate_test_bin_thresholds(thr) == 0
    t = (thr[1:185] / 10.0).astype(np.float32)
    on = np.concatenate([t, np.nextafter(t, np.float32(0)), np.nextafter(t, np.float32(np.inf))])
    k = o2 + rng.choice(n - o2, 2 * on.shape[0], replace=False)
    sites.age_end[k[:on.shape[0]]] = on
    sites.age_begin[k[:on.shape[0]]] = 0.0                                       # emp slice: bin of age_end itself
    sites.age_end[k[on.shape[0]:]] = on
    sites.age_begin[k[on.shape[0]:]] = (on * np.float32(0.5)).astype(np.float32)
    narrow = o2 + rng.choice(n - o2, 6000, replace=False)
    narrow = narrow[~np.isin(narrow, k)]
    ab = np.exp(rng.uniform(np.log(5.0), np.log(4e6), narrow.shape[0])).astype(np.float32)
    sites.age_begin[narrow] = ab
    sites.age_end[narrow] = (ab.astype(np.float64) * (1 + 1e-3)).astype(np.float32)
    chr_of = _chr_of_rows(sites)
    # target counts: N 20 .. ~2000; ties on a third of chromosome 2
    Nt = np.exp(rng.uniform(np.log(20), np.log(2000), n)).astype(np.int64)
    dt = rng.binomial(Nt, rng.uniform(0.05, 0.95, n))
    tie = o2 + rng.choice(n - o2, (n - o2) // 3, replace=False)
    h = rng.integers(5, 500, tie.shape[0])
    Nt[tie] = 4 * h
    dt[tie] = np.where(rng.random(tie.shape[0]) < 0.5, h, 3 * h)                 # DAF / (N / 2) = 0.5, or 1.5 with AAF's 0.5
    Nr = np.exp(rng.uniform(0, np.log(5008), n)).astype(np.int64).clip(1, 5008)
    dr = np.maximum(rng.binomial(Nr, rng.uniform(0.05, 0.95, n)), 1)
    dr = np.minimum(dr, Nr)
    gt = synth.Genome(chr_of, sites.pos.copy(), sites.anc.copy(), sites.der.copy(), (Nt - dt).astype(np.int32), dt.astype(np.int32))
    gr = synth.Genome(chr_of, sites.pos.copy(), sites.anc.copy(), sites.der.copy(), (Nr - dr).astype(np.int32), dr.astype(np.int32))
    return sites, gt, gr


def test_deep_coverage_oracle_reaches_its_regimes():
    """The deep dataset has >= 50 k used rows in one block, pseudo-genotype ties, and bins that take all 100 samples of a row."""
    sites, gt, gr = _deep_dataset(13)
    o = po.stage1(sites, gt, gr, seed=13)
    assert o["n_used"].max() >= 50000
    assert int(o["n_notshared"].sum()) == 100 * o["n_used_total"]
    half = gt.daf.astype(np.float64) / ((gt.daf + gt.aaf) / 2.0)
    assert (half == 0.5).sum() > 1000 and (half == 1.5).sum() > 1000
    assert (gt.daf + gt.aaf).max() > 1500 and (gr.daf + gr.aaf).max() >= 4000


# ---- E: the reference itself ----------------------------------------------------------------------------------------
def _combined_small():
    s1, t1, r1, _ = _repeats_dataset(31, n_chr=2, n_pos=600)
    s2, t2, r2 = _dense_dataset(32)
    rng = np.random.default_rng(33)
    p = np.unique(np.concatenate([rng.integers(1, 12 * B, 400), [k * B + d for k in range(1, 12) for d in (-1, 0, 1)]]))
    s3 = _sites([p], rng, lens=[12 * B + 10])
    chr_of = _chr_of_rows(s3)
    keep = rng.random(s3.n) < 0.8
    g3 = lambda s: synth.Genome(chr_of[keep], s3.pos[keep].copy(), s3.anc[keep].copy(), s3.der[keep].copy(),
                                np.full(keep.sum(), s, np.int32), np.full(keep.sum(), 2, np.int32))
    return _concat([(s1, t1, r1), (s2, t2, r2), (s3, g3(1), g3(3))])


@pytest.mark.skipif(not po.ref_available(), reason="oracle/_ref not built (needs the reference's sources)")
def test_shapes_vs_live_reference():
    """Repeated positions, dense record windows and block-edge rows in one dataset: oracle == the reference's parse_tmptmp."""
    sites, gt, gr = _combined_small()
    with tempfile.TemporaryDirectory() as d:
        synth.write_dataset(d, sites, {"t": gt, "r": gr})
        r = po.ref_parse_tmptmp(d, sites.chr_names, "syn", "t", "r", seed=34)
    o = po.stage1(sites, gt, gr, seed=34)
    assert o["num_blocks"] == r["num_blocks"]
    for k in ("shared", "notshared", "shared_emp", "notshared_emp"):
        assert np.array_equal(o[k], r[k]), k
    assert np.array_equal(o["rng"].words(), r["mt"])


# ================================================================================================= GPU section
def _check(o, s1):
    """_compare_stage1 on a copy of the oracle's generator state (it draws the next words from it): one oracle run can
    be compared with several device runs."""
    _compare_stage1(dict(o, rng=po.MT.from_buffer_copy(o["rng"])), s1)


def _run(handle, sites, gt, gr, seed, tm=None, rm=None, ingest=False):
    if ingest:
        handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
        with tempfile.TemporaryDirectory() as d:
            for slot, g in ((0, gt), (1, gr)):
                p = os.path.join(d, f"{slot}.colate.in")
                synth.write_colate_in(p, g, sites.chr_names)
                assert handle.ingest_colate_in(slot, open(p, "rb").read(), sites.chr_names) == g.n
        handle.set_mask(0, None if tm is None else api.mask_bits_from_seq(tm, sites.site_off, sites.pos))
        handle.set_mask(1, None if rm is None else api.mask_bits_from_seq(rm, sites.site_off, sites.pos))
    else:
        handle.load(sites, gt, gr, tm, rm)
    return handle.stage1(api.mt_seed(seed))


@gpu
def test_repeated_positions_hand_case(handle):
    for swap, n_used in ((False, 3), (True, 4)):
        sites, gt, gr = _hand_case(swap)
        o = po.stage1(sites, gt, gr, seed=2)
        assert o["n_used_total"] == n_used
        for ingest in (False, True):
            _check(o, _run(handle, sites, gt, gr, 2, ingest=ingest))


@gpu
@pytest.mark.parametrize("seed", [3, 4])
@pytest.mark.parametrize("masks", [False, True])
def test_repeated_positions_random(handle, seed, masks):
    """Runs of repeated rows and records against the oracle, in both genome slots, with and without masks, through the
    array upload and through the device decoder of .colate.in images."""
    sites, gt, gr, _ = _repeats_dataset(seed)
    tm, rm = _repeat_masks(sites, seed) if masks else (None, None)
    o = po.stage1(sites, gt, gr, seed=seed, tmask=tm, rmask=rm)
    assert o["n_used_total"] > 500
    for ingest in (False, True):
        _check(o, _run(handle, sites, gt, gr, seed, tm, rm, ingest=ingest))
    # target and reference swapped: the other genome's runs meet the reference-stream rules
    o = po.stage1(sites, gr, gt, seed=seed, tmask=rm, rmask=tm)
    _check(o, _run(handle, sites, gr, gt, seed, rm, tm))


@gpu
def test_dense_record_windows(handle):
    """Tiles staged in shared memory and tiles that fall back to global searches on one chromosome (windows of 1024 .. 1027
    records and far more), a dense first and a dense last tile, repeated positions inside dense windows."""
    sites, gt, gr = _dense_dataset(5)
    for t, r, seed in ((gt, gr, 5), (gr, gt, 6)):
        o = po.stage1(sites, t, r, seed=seed)
        _check(o, _run(handle, sites, t, r, seed))
    s1, t1, r1, _ = _repeats_dataset(7, n_chr=2, n_pos=900)                    # dense windows with masks cutting through them
    sites2, gt2, gr2 = _concat([(sites, gt, gr), (s1, t1, r1)])
    tm = [synth.make_mask(70 + c, int(L), 0.1, run_lo=500, run_hi=20000) for c, L in enumerate(sites2.chrom_len)]
    o = po.stage1(sites2, gt2, gr2, seed=7, tmask=tm)
    _check(o, _run(handle, sites2, gt2, gr2, 7, tm=tm, ingest=True))


@gpu
def test_all_pairs_on_a_dense_genome(handle):
    """The all-pairs driver with a dense genome among sparse ones: every pair == that pair alone (oracle), counts and EM."""
    from colate_b200 import pairs as pairs_mod
    sites, gd, gd2 = _dense_dataset(9)
    rng = np.random.default_rng(9)
    keep = rng.random(sites.n) < 0.7
    chr_of = _chr_of_rows(sites)
    N = rng.integers(1, 5, keep.sum()); d = rng.integers(0, N + 1)
    gs = synth.Genome(chr_of[keep], sites.pos[keep].copy(), sites.anc[keep].copy(), sites.der[keep].copy(),
                      (N - d).astype(np.int32), d.astype(np.int32))
    genomes = [gd, gs, gd2]
    handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
    for g, G in enumerate(genomes):
        handle.set_genome(g, G.chrom, G.bp, G.aaf, G.daf, G.anc.astype(np.uint16) | (G.der.astype(np.uint16) << 8))
        handle.set_mask(g, None)
    res = pairs_mod.all_pairs(handle, 3, seed=4, bins="3,7,0.2", pairs=[(0, 1), (1, 0), (0, 2), (2, 1)], max_iter=60)
    ep, _ = po.epochs_from_bins("3,7,0.2", 0.0, 28.0)
    init = np.full(len(ep), 1 / 20000.)
    for p, (i, j) in enumerate(res["pairs"]):
        o = po.stage1(sites, genomes[i], genomes[j], seed=4)
        assert res["num_blocks"][p] == o["num_blocks"] and res["n_used"][p] == o["n_used_total"] > 100
        w = po.draw_block_weights(o["rng"], 1, o["num_blocks"])
        assert np.array_equal(res["counts"][p], po.stage2(w, o, 0.0)[0]), (i, j)
        ro, it, llo = po.em_run(ep, init, res["counts"][p], max_iter=60)
        assert res["iters"][p] == it and np.array_equal(res["rates"][p], ro) and res["ll"][p] == llo, (i, j)


def _shard_replay(handle, sites, gt, gr, seed, world):
    """test_gpu_stage1.py::test_stage1_chromosome_shards_on_one_gpu's decomposition: (stats, tallies, state, used, blocks)."""
    from colate_b200 import dist as cdist
    parts = cdist.split_chromosomes(np.diff(sites.site_off), world)
    used_base = block_base = 0
    stats, tallies, state = [], [], None
    for lo, hi in parts:
        s0, s1 = int(sites.site_off[lo]), int(sites.site_off[hi])
        handle.set_sites(sites.site_off[lo:hi + 1] - sites.site_off[lo], sites.pos[s0:s1], sites.age_begin[s0:s1],
                         sites.age_end[s0:s1], sites.meta()[s0:s1])
        for slot, g in ((0, gt), (1, gr)):
            first, end = api.chr_ranges(len(sites.chr_names), g.chrom)
            al = g.anc.astype(np.uint16) | (g.der.astype(np.uint16) << 8)
            api.check(api.lib().colate_set_genome(handle._h, slot, g.n, api.ptr(np.ascontiguousarray(first[lo:hi])),
                                                  api.ptr(np.ascontiguousarray(end[lo:hi])), api.ptr(g.bp), api.ptr(g.aaf),
                                                  api.ptr(g.daf), api.ptr(al), 0))
        handle.set_mask(0, None); handle.set_mask(1, None)
        used_chr, blocks_chr = handle.stage1_flags()
        n_local = int(np.sum(blocks_chr))
        if block_base + n_local > 500:
            n0 = handle.launch_count()
            with pytest.raises(api._lib.ColateError) as e:
                handle.stage1_sample(api.mt_seed(seed), used_base, block_base, n_local)
            assert e.value.code == -3 and handle.launch_count() == n0        # refused before any kernel
            return None
        st, tl, state = handle.stage1_sample(api.mt_seed(seed), used_base, block_base, n_local)
        stats.append(st[:n_local]); tallies.append(tl[:n_local])
        used_base += int(np.sum(used_chr)); block_base += n_local
    return np.concatenate(stats), np.concatenate(tallies), state, used_base, block_base


@gpu
def test_block_edges_and_the_500_block_limit(handle):
    """Exactly 500 blocks: stage i bit for bit, stage ii with R = 1 and R = 5, and the chromosome-shard replay whose last
    shard ends at block 500.  One row moved one base over its block edge: 501 blocks, refused by the oracle, by
    colate_stage1 and by the shard form, before any sampling kernel runs."""
    sites, gt, gr = _blocks_dataset(8)
    o = po.stage1(sites, gt, gr, seed=8)
    assert o["num_blocks"] == 500
    s1 = _run(handle, sites, gt, gr, 8)
    _check(o, s1)
    assert int(s1.block_tallies[:, 1].sum()) == 100 * s1.n_used
    for R in (1, 5):
        w = api.draw_block_weights(s1.mt_state.copy(), R, s1.num_blocks)
        assert np.array_equal(w, po.draw_block_weights(po.MT.from_buffer_copy(o["rng"]), R, 500))
        assert np.array_equal(handle.stage2_bootstrap(w, s1.block_stats, 0.0), po.stage2(w, o, 0.0)), R
    stats, tallies, state, nu, nb = _shard_replay(handle, sites, gt, gr, 8, 3)
    assert (nu, nb) == (o["n_used_total"], 500)
    assert np.array_equal(stats, s1.block_stats) and np.array_equal(tallies, s1.block_tallies)
    assert np.array_equal(state, s1.mt_state)

    sites, gt, gr = _blocks_dataset(8, bump=True)
    assert po.stage1(sites, gt, gr, seed=8)["num_blocks"] == -3
    handle.load(sites, gt, gr)
    _, blocks = handle.stage1_flags()
    assert int(blocks.sum()) == 501
    n0 = handle.launch_count()
    handle.stage1_flags()
    n1 = handle.launch_count()
    with pytest.raises(api._lib.ColateError) as e:
        handle.stage1(api.mt_seed(8))
    assert e.value.code == -3 and handle.launch_count() - n1 == n1 - n0      # the flag pass and nothing after it
    assert _shard_replay(handle, sites, gt, gr, 8, 3) is None


@gpu
def test_more_contigs_than_one_round_of_k_chr(handle):
    """1100 contigs (k_chr strings them together in rounds of 1024): used rows and blocks per contig == the oracle on
    groups of contigs below 500 blocks; the whole stage is refused with COLATE_ERR_BLOCKS, like the oracle refuses it."""
    sites, gt, gr = _many_contigs_dataset(12)
    handle.load(sites, gt, gr)
    used_chr, blocks_chr = handle.stage1_flags()
    n_c = len(sites.chr_names)
    for lo in range(0, n_c, 150):
        hi = min(lo + 150, n_c)
        s, t = _sub(sites, gt, lo, hi)
        _, r = _sub(sites, gr, lo, hi)
        o = po.stage1(s, t, r, seed=1)
        assert o["num_blocks"] == int(blocks_chr[lo:hi].sum()) < 500, lo
        assert o["n_used_total"] == int(used_chr[lo:hi].sum()), lo
        cut = np.cumsum(blocks_chr[lo:hi])[:-1]
        assert np.array_equal(np.array([x.sum() for x in np.split(o["n_used"], cut)]), used_chr[lo:hi]), lo
    assert (blocks_chr > 1).sum() > 100 and (used_chr > 0).sum() > 500
    assert po.stage1(sites, gt, gr, seed=1)["num_blocks"] == -3
    with pytest.raises(api._lib.ColateError) as e:
        handle.stage1(api.mt_seed(1))
    assert e.value.code == -3


@gpu
def test_deep_coverage_tmp_weights(handle):
    """tmp/tmp genomes with N up to ~2000: pseudo-genotype ties, 100 samples in one bin (replay_row with c > 4), age_end on
    the bin thresholds, a block of 60 k used rows."""
    sites, gt, gr = _deep_dataset(13)
    o = po.stage1(sites, gt, gr, seed=13)
    s1 = _run(handle, sites, gt, gr, 13)
    _check(o, s1)
    assert int(s1.block_tallies[:, 1].sum()) == 100 * s1.n_used


@gpu
def test_deep_coverage_row_counts_front_end(handle):
    """front_end = 1 on per-row (AAF, DAF) with N_ref up to 5008: raw count weights DAF_t * DAF_r / (N_r * 100) with full
    mantissas and magnitudes up to ~20 per sample."""
    sites, gt, gr = _deep_dataset(14)
    tc = np.stack([gt.aaf, gt.daf], 1).astype(np.int32)
    rc = np.stack([gr.aaf, gr.daf], 1).astype(np.int32)
    assert (tc[:, 1].astype(np.int64) * rc[:, 1]).max() < 2**31
    o = po.stage1_pileup(sites, tc, rc, seed=14)
    handle.set_option("front_end", 1)
    try:
        handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
        handle.set_row_counts(0, tc[:, 0], tc[:, 1])
        handle.set_row_counts(1, rc[:, 0], rc[:, 1])
        handle.set_mask(0, None); handle.set_mask(1, None)
        s1 = handle.stage1(api.mt_seed(14))
        _check(o, s1)
        assert int(s1.block_tallies[:, 1].sum()) == 100 * s1.n_used and s1.n_used == sites.n
        assert s1.block_stats[:, 1].max() > 1e3
    finally:
        handle.set_option("front_end", 0)
