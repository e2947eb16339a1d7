"""k_replay and k_emp (the exact fp64 histograms of stage i) against a plain sequential fp64 loop, at the places where the
kernel's shortcuts could go wrong: rounding ties, weights at the 2^(E-1) bound, runs that land on or cross a power of two,
absorbed additions, negative weights (raw count products past 2^31 wrap in the reference's int arithmetic), every count
byte and the block / tile geometry.  The kernels run on rows given directly (Handle.test_replay: the launches of stage i);
the device replay_row / exsum::add_repeated run element by element (Handle.test_replay_row).  End to end, row-count genomes
whose weights wrap negative or tie are compared with the oracle.

The CPU section at the top runs without a GPU: it shows, counted over the reference loop itself, that every generated case
reaches the regime it is named for, and that the oracle's raw-count sums are those of explicitly wrapped int32 products."""
from collections import Counter

import numpy as np
import pytest

from colate_b200 import api, synth
from oracle import pyoracle as po
from test_gpu_stage1 import _compare_stage1

gpu = pytest.mark.gpu

NB = 185               # age bins; count slot 185 = "age out of range", 186..191 never written by k_sample
SLOTS = 192
TILE = 32              # rows per count tile = rows per collapsed run of k_replay (RP_ROWS)
HALF = 16              # rows of a run per lane of a bin (RP_ROWS / RP_Q)
STAGES = 4             # k_replay's ring of count tiles (RP_STAGES)
B = 30_000_000         # COLATE_BLOCK_BASES


# ================================================================================================= the plain loop
def _fold(w, c):
    """acc = 0; acc += w[i], c[i] times for every row i in order, each addition rounded: np.add.accumulate is a strictly
    sequential left fold.  Returns every partial sum (partial[0] = 0)."""
    return np.add.accumulate(np.concatenate([[0.0], np.repeat(np.asarray(w, np.float64), c)]))


def _sequences(case):
    """Every (block, histogram, bin) of the reference loop: (absolute rows with a count, their weights, their counts).
    Histogram 0 (shared) takes the rows with age_begin > 0, histogram 1 (not shared) every row."""
    brs, cnt = case["brs"], case["cnt"]
    for b in range(len(brs) - 1):
        r0, r1 = int(brs[b]), int(brs[b + 1])
        C = cnt[r0:r1, :NB].astype(np.int64)
        for which, w, live in ((0, case["ws"], case["ab"] > 0), (1, case["wn"], np.ones(cnt.shape[0], bool))):
            Cw = C * live[r0:r1, None]
            for k in np.nonzero(Cw.any(0))[0]:
                rr = np.nonzero(Cw[:, k])[0]
                yield b, which, int(k), r0 + rr, w[r0 + rr], Cw[rr, k]


def replay_ref(case):
    """What k_replay + k_emp must return for the case: (out_f [nb][4][185], out_n [nb][3][185], out_of_range)."""
    brs, cnt = case["brs"], case["cnt"]
    nb = len(brs) - 1
    F = np.zeros((nb, 4, NB)); N = np.zeros((nb, 3, NB), np.int64)
    oor = False
    for b, which, k, rows, w, c in _sequences(case):
        F[b, which, k] = _fold(w, c)[-1]
        N[b, which, k] = c.sum()
    for b in range(nb):
        r0, r1 = int(brs[b]), int(brs[b + 1])
        oor |= bool(cnt[r0:r1, NB].any())
        for r in range(r0, r1):                       # emp: one addition per row, in row order
            k = int(case["eb"][r])
            if k != 255:
                F[b, 2, k] = np.float64(F[b, 2, k] + case["ews"][r])
                F[b, 3, k] = np.float64(F[b, 3, k] + case["ewn"][r])
                N[b, 2, k] += 1
    return F, N, oor


def _ties(a, x, s):
    """s = RN(a + x) was a tie: the exact error (TwoSum) is half the spacing towards the neighbour it points at."""
    bb = s - a
    err = (a - (s - bb)) + (x - bb)
    nb = np.nextafter(s, np.where(err > 0, np.inf, -np.inf))
    return (err != 0) & (2 * np.abs(err) == np.abs(nb - s))


def _binade(x):
    """(sign, exponent) of x: two partial sums share a binade iff their keys are equal."""
    return np.sign(x) * 4096 + np.frexp(x)[1]


def regimes(case):
    """Counts, over the reference loop, of the situations the kernel's shortcuts must recognise."""
    st = Counter()
    for _, _, _, rows, w, c in _sequences(case):
        part = _fold(w, c)
        a, s, x = part[:-1], part[1:], np.repeat(w, c)
        crow, rrow = np.repeat(c, c), np.repeat(rows, c)
        tie = _ties(a, x, s)
        lsb = a.view(np.uint64) & np.uint64(1)
        st["tie_acc_even"] += int((tie & (lsb == 0)).sum()); st["tie_acc_odd"] += int((tie & (lsb == 1)).sum())
        st["tie_c1"] += int((tie & (crow == 1)).sum())
        st["tie_c2_4"] += int((tie & (crow >= 2) & (crow <= 4)).sum())
        st["tie_c5_up"] += int((tie & (crow >= 5)).sum())
        st["tie_lane0"] += int((tie & (rrow % TILE < HALF)).sum()); st["tie_lane1"] += int((tie & (rrow % TILE >= HALF)).sum())
        st["absorbed"] += int(((s == a) & (x != 0) & ~tie).sum())
        st["negative"] += int((x < 0).sum())
        st["w_zero"] += int(((w == 0) & ~np.signbit(w)).sum()); st["w_negzero"] += int(((w == 0) & np.signbit(w)).sum())
        first = np.concatenate([[0], np.cumsum(c)[:-1]])          # index in `part` of the acc in front of each row
        acc = part[first]
        pos = acc > 0
        half = np.ldexp(1.0, np.frexp(acc)[1] - 2)                # 2^(E-1) for acc in [2^E, 2^(E+1))
        st["w_at_bound"] += int((pos & (w == half)).sum())
        st["w_ulp_below_bound"] += int((pos & (w == np.nextafter(half, 0))).sum())
        st["w_ulp_above_bound"] += int((pos & (w == np.nextafter(half, np.inf))).sum())
        st["w_ge_acc"] += int((pos & (w >= acc)).sum())
        hi = lambda v: np.asarray(v, np.float64).view(np.uint64) >> np.uint64(32)
        with np.errstate(invalid="ignore"):                                       # (ulp of a subnormal acc: 0)
            on_grid = (w % np.ldexp(1.0, np.frexp(acc)[1] - 53)) == 0             # a multiple of ulp(acc): no tie
        st["w_above_bound_same_hi_word"] += int((pos & (w > half) & (hi(w) == hi(half)) & on_grid).sum())
        # runs: the tile-aligned groups of 32 rows the kernel collapses
        run = rows // TILE
        brk = np.nonzero(np.diff(run))[0] + 1
        starts = np.concatenate([[0], brk]); ends = np.concatenate([brk, [len(rows)]])
        keys = _binade(part)
        for i0, i1 in zip(starts, ends):
            p0 = first[i0]
            p1 = first[i1] if i1 < len(rows) else len(part) - 1
            a0, a1 = part[p0], part[p1]
            if a0 > 0:
                top = np.ldexp(1.0, np.frexp(a0)[1])              # 2^(E+1)
                st["run_on_top"] += int(a1 == top); st["run_ulp_short"] += int(a1 == np.nextafter(top, 0))
                st["run_binades_crossed_max"] = max(st["run_binades_crossed_max"], int(np.frexp(a1)[1] - np.frexp(a0)[1]))
            inner = keys[p0:p1 + 1]
            if (inner != inner[0]).any() and inner[-1] == inner[0]:
                st["run_leaves_binade_and_returns"] += 1
    return st


# ================================================================================================= cases
class Rows:
    """Rows and blocks as colate_test_replay takes them, appended in row order."""

    def __init__(self):
        self.cnt, self.ab, self.ws, self.wn, self.eb, self.ews, self.ewn = [], [], [], [], [], [], []
        self.starts = [0]

    @property
    def n(self):
        return len(self.ab)

    def row(self, counts=None, ws=0.0, wn=None, ab=1.0, eb=255, ews=0.0, ewn=0.0):
        c = np.zeros(SLOTS, np.uint8)
        if counts is not None:
            for k, v in (counts.items() if isinstance(counts, dict) else enumerate(counts)):
                c[k] = v
        self.cnt.append(c); self.ab.append(ab); self.ws.append(ws); self.wn.append(ws if wn is None else wn)
        self.eb.append(eb); self.ews.append(ews); self.ewn.append(ewn)

    def pad(self, off=0):
        """rows without counts up to the next row index = off (mod 32)"""
        while self.n % TILE != off:
            self.row()

    def block(self):
        """close the current block: it holds the rows since the previous call"""
        self.starts.append(self.n)

    def buildup(self, w):
        """every bin of both histograms to acc = 100 w (exact for w = 3 * 2^k), finished in a tile of its own"""
        self.pad()
        self.row({k: 100 for k in range(NB)}, w)
        self.pad()

    def case(self):
        return dict(brs=np.array(self.starts, np.int64), cnt=np.array(self.cnt, np.uint8).reshape(-1, SLOTS),
                    ab=np.array(self.ab, np.float64), ws=np.array(self.ws, np.float64), wn=np.array(self.wn, np.float64),
                    eb=np.array(self.eb, np.uint8), ews=np.array(self.ews, np.float64), ewn=np.array(self.ewn, np.float64))


def _realistic(R, rng, n, p_emp=0.3, bins=None):
    """rows like k_sample leaves them: 100 samples over a window of bins, weights num / (reads * 100), a third emp rows"""
    for _ in range(n):
        lo = int(rng.integers(0, NB - 12)) if bins is None else int(rng.choice(bins))
        cnt = np.bincount(rng.integers(lo, min(lo + 12, NB), 100), minlength=SLOTS)
        emp = rng.random() < p_emp
        R.row(cnt, float(rng.integers(0, 40) / (rng.integers(1, 60) * 100.0)), float(rng.integers(0, 40) / (rng.integers(1, 60) * 100.0)),
              ab=0.0 if emp else float(rng.uniform(1, 1e4)), eb=int(rng.integers(0, NB)) if emp else 255,
              ews=float(rng.integers(0, 40) / rng.integers(1, 60)) if emp else 0.0, ewn=float(rng.integers(0, 40) / rng.integers(1, 60)) if emp else 0.0)


def case_ties(seed=1):
    """acc built up to 300 * 2^k in every bin, then rows whose w ends in exactly ulp(acc) / 2, interleaved with rows on the
    grid of ulp(acc) (odd multiples flip acc's last bit) and rows of full mantissas; c = 1, 2..4 and 5..100."""
    rng = np.random.default_rng(seed)
    R = Rows()
    for k in (-20, -7, 0, 5, 30):
        R.buildup(3.0 * 2.0 ** k)
        U = 2.0 ** (k - 44)                                       # ulp(acc): acc in [2^(k+8), 2^(k+9))
        for i in range(150):
            kind = rng.integers(0, 4)
            m = float(rng.integers(0, 1 << 20))
            w = (m + 0.5) * U if kind < 2 else (m * U if kind == 2 else float(rng.uniform(0, 2.0 ** (k - 10))))
            cls = rng.integers(0, 3)
            counts = {int(b): int(1 if cls == 0 else rng.integers(2, 5) if cls == 1 else rng.integers(5, 101))
                      for b in rng.choice(NB, int(rng.integers(1, 7)), replace=False)}
            R.row(counts, w, (float(rng.integers(0, 1 << 20)) + 0.5) * U, ab=1.0 if rng.random() < 0.8 else 0.0)
        R.block()
    return R.case()


def case_bounds():
    """w = 2^(E-1), one ulp below (a tie in these binades) and above, on the grid of ulp(acc) just above (same high word as
    2^(E-1): a bound test on the high word must include it) and just below, w >= acc, w = 0 and -0.0,
    each with c = 1, 3, 7, 50 in a bin of its own; and blocks whose first runs start from acc = 0 with tiny and
    subnormal weights (E <= 54)."""
    R = Rows()
    for k in (-40, 0, 17, 60):
        R.buildup(3.0 * 2.0 ** k)
        acc, h, U = 300.0 * 2.0 ** k, 128.0 * 2.0 ** k, 2.0 ** (k - 44)
        ws = [h, np.nextafter(h, 0), np.nextafter(h, np.inf), h + U, h + 2 * U, h - U, h - 2 * U, acc, 1.5 * acc, 2.0 ** (k + 12),
              0.0, -0.0, 2.0 ** (k - 60), U / 2]
        for i, w in enumerate(ws):
            R.row({4 * i + j: c for j, c in enumerate((1, 3, 7, 50))}, float(w))
        R.block()
    for w0 in (5e-324, 1e-310, 2.0 ** -1000, 1e-300, 1.0):
        R.pad()
        for i in range(TILE + 5):
            R.row({i % 40: 1 + i % 9, 100 + i % 3: 100}, w0 * (1 + i))
        R.block()
    return R.case()


def case_binade():
    """Runs whose collapsed total lands exactly on 2^(E+1), one ulp short of it, or short by a whole w; runs across 10+
    binades from a tiny acc; sums past 2^53 w, where additions are absorbed (and w = ulp / 2 is a tie)."""
    R = Rows()
    for k in (-30, 0, 25):
        U = 2.0 ** (k - 44)
        for short in (0.0, U):                                     # 300 + 32 * 6.625 = 512 (* 2^k)
            R.buildup(3.0 * 2.0 ** k)
            for i in range(TILE):
                R.row({0: 1, 1: 1 if i < TILE - 1 else 0, 2: 2 if i < HALF else 0}, 6.625 * 2.0 ** k - (short if i == TILE - 1 else 0.0))
            R.block()
        R.buildup(3.0 * 2.0 ** k)                                  # 300 + 4 * 53 = 512, four rows with c > 4
        for i in range(4):
            R.row({7 * i: 53, 7 * i + 1: 53, 100: 53}, 2.0 ** k)
        R.block()
    R.pad()
    R.row({k: 1 for k in range(NB)}, 1.0)                          # acc = 1 ...
    R.pad()
    R.row({k: 100 for k in range(0, NB, 2)}, 1024.0)               # ... to 102401 in one run, then small rows in the new binades
    for i in range(TILE - 1):
        R.row({k: 1 + (i + k) % 5 for k in range(NB)}, 0.37 * (i + 1))
    R.block()
    R.pad()
    R.row({k: 64 for k in range(NB)}, 2.0 ** 54)                   # acc = 2^60: ulp 2^8
    R.pad()
    for w in (1.0, 3.0, 2.0 ** 6, 2.0 ** 7 - 1, 2.0 ** 7, 2.0 ** 7 + 1, 2.0 ** 8, 5e-324):
        R.row({k: 1 + k % 100 for k in range(NB)}, w)
    R.block()
    return R.case()


def case_counts(rng_seed=4, bin185=False, bin185_outside=False):
    """Every count byte 0..100 and 255; one bin holding all 100 samples of every row; slots 186..191 nonzero (never
    written by k_sample: must not leak); bin 185 set inside a block (raises the flag) or only outside every block."""
    rng = np.random.default_rng(rng_seed)
    R = Rows()
    vals = list(range(101)) + [255]
    for j in range(3):
        for i, v in enumerate(rng.permutation(vals)):
            cnt = np.zeros(SLOTS, np.int64)
            cnt[3] = v
            cnt[5] = 100
            cnt[10 + (i % 150)] = vals[(i * 7 + j) % len(vals)]
            cnt[186:] = rng.integers(0, 256, 6) if i % 3 == 0 else 0
            if bin185 and j == 1 and i == 40:
                cnt[NB] = 1
            R.row(cnt, float(rng.integers(0, 40) / (rng.integers(1, 60) * 100.0)), float(rng.uniform(0, 3)),
                  ab=0.0 if i % 4 == 0 else 2.0)
        R.block()
    if bin185_outside:
        R.row({NB: 7, 3: 1}, 1.0)                                  # after the last block: no block reads it
    return R.case()


def case_geometry(seed=5):
    """Blocks starting at every offset 0..31 inside a tile with 0, 1, 31, 32, 33 rows; a block over 7 tiles (more than the
    4-stage ring) and one over 300; bins with counts in one lane's half of every run only; k_emp groups of 32 rows of one
    bin, of one row of a bin, of no row (255)."""
    rng = np.random.default_rng(seed)
    R = Rows()
    for off in range(TILE):
        for L in (0, 1, 31, 32, 33):
            gap = (off - R.n) % TILE
            if gap:
                _realistic(R, rng, gap); R.block()
            _realistic(R, rng, L); R.block()
    for n_tiles in (7, 300):
        R.pad(int(rng.integers(0, TILE)))
        R.block()                                                  # (the padding rows: a block of their own)
        r0 = R.n
        _realistic(R, rng, n_tiles * TILE - 3)
        for r in range(r0, R.n):
            R.cnt[r][180] = 3 if r % TILE < HALF else 0            # lane 0's rows only
            R.cnt[r][181] = 0 if r % TILE < HALF else 2            # lane 1's rows only
            R.cnt[r][182] = 100 if (r - r0) % 97 == 0 and r % TILE >= HALF else 0
            g = (r - r0) // TILE                                   # k_emp's groups start at the block's first row
            R.eb[r] = 7 if g == 0 else (9 if (r - r0) == TILE + 5 else 255) if g in (1, 2) else R.eb[r]
            if g in (0, 1):
                R.ews[r], R.ewn[r] = float(rng.uniform(0, 5)), float(rng.uniform(0, 5))
        R.block()
    return R.case()


def case_500_blocks(seed=6):
    rng = np.random.default_rng(seed)
    R = Rows()
    for b in range(500):
        _realistic(R, rng, int(rng.integers(0, 45)))
        R.block()
    return R.case()


def case_negative(seed=7):
    """Negative shared and not-shared weights (wrapped int32 products) among positive ones: runs whose partial sums leave
    acc's binade and come back, acc pushed below zero and back, negative weights on rows that add nothing to shared,
    negative emp weights."""
    rng = np.random.default_rng(seed)
    R = Rows()
    for k in (-3, 0, 9):
        s = 2.0 ** k
        R.buildup(3.0 * s)                                         # acc = 300 s in [256 s, 512 s)
        for i in range(3):
            R.row({i: 1, 50 + i: 1}, 150.0 * s + rng.uniform(0, s), -(150.0 * s + rng.uniform(0, s)))
            R.row({i: 1, 50 + i: 1}, 100.0 * s + rng.uniform(0, s), -(100.0 * s + rng.uniform(0, s)))       # above 512 s / below 256 s
            R.row({i: 1, 50 + i: 1}, -(210.0 * s + rng.uniform(0, s)), 220.0 * s + rng.uniform(0, s))       # ... and back
        R.pad(HALF)
        R.row({60: 2}, -400.0 * s)                                 # acc below zero ...
        R.pad()
        R.row({60: 3}, 250.0 * s + rng.uniform(0, s))              # ... and back above
        for i in range(3 * TILE):
            w = float(rng.uniform(0.1, 250.0) * s) * (1 if rng.random() < 0.5 else -1)
            counts = {int(b): int(rng.integers(1, 101)) for b in rng.choice(NB, int(rng.integers(1, 8)), replace=False)}
            emp = rng.random() < 0.3
            R.row(counts, w, -w * rng.uniform(0.5, 2), ab=0.0 if emp else 1.0, eb=int(rng.integers(0, NB)) if emp else 255,
                  ews=-float(rng.uniform(0, 9)) if emp else 0.0, ewn=float(rng.uniform(-9, 9)) if emp else 0.0)
        R.block()
    return R.case()


CASES = {"ties": case_ties, "bounds": case_bounds, "binade": case_binade, "counts": case_counts, "geometry": case_geometry,
         "500_blocks": case_500_blocks, "negative": case_negative}


# ================================================================================================= CPU: the cases reach their regimes
def test_ties_case_reaches_ties():
    st = regimes(case_ties())
    for key in ("tie_acc_even", "tie_acc_odd", "tie_c1", "tie_c2_4", "tie_c5_up", "tie_lane0", "tie_lane1"):
        assert st[key] > 20, (key, st)


def test_bounds_case_reaches_the_weight_bounds():
    c = case_bounds()
    st = regimes(c)
    for key in ("w_at_bound", "w_ulp_below_bound", "w_ulp_above_bound", "w_above_bound_same_hi_word", "w_ge_acc", "w_zero",
                "w_negzero", "tie_acc_even", "absorbed"):
        assert st[key] >= 4, (key, st)
    # first runs from acc = 0 with acc staying below 2^-968 (biased exponent <= 54) for a whole run
    assert any(w[0] > 0 and _fold(w, cc)[-1] < 2.0 ** -968 for _, _, _, _, w, cc in _sequences(c))


def test_binade_case_reaches_the_binade_edges():
    st = regimes(case_binade())
    assert st["run_on_top"] >= 6 and st["run_ulp_short"] >= 3, st
    assert st["run_binades_crossed_max"] >= 10, st
    assert st["absorbed"] > 100 and st["tie_acc_even"] + st["tie_acc_odd"] > 0, st


def test_counts_case_covers_every_byte():
    c = case_counts(bin185=True)
    assert set(np.unique(c["cnt"][:, 3])) == set(range(101)) | {255}
    assert (c["cnt"][:, 5] == 100).all() and c["cnt"][:, 186:].any() and c["cnt"][:, NB].sum() == 1
    assert replay_ref(c)[2] and not replay_ref(case_counts())[2]
    c = case_counts(bin185_outside=True)
    assert c["cnt"][:, NB].any() and not replay_ref(c)[2]


def test_geometry_case_covers_offsets_lengths_and_groups():
    c = case_geometry()
    brs = c["brs"]
    L = np.diff(brs)
    for off in range(TILE):
        for n in (0, 1, 31, 32, 33):
            assert ((brs[:-1] % TILE == off) & (L == n)).any(), (off, n)
    tiles = (brs[1:] - 1) // TILE - brs[:-1] // TILE + 1
    assert tiles[L > 0].max() >= 300 and ((tiles > STAGES) & (tiles < 10)).any()
    big = np.nonzero(L > 200)[0]
    for b in big:
        r0, r1 = brs[b], brs[b + 1]
        rows = np.arange(r0, r1)
        assert (c["cnt"][rows[rows % TILE < HALF], 181] == 0).all() and c["cnt"][rows, 181].any()
        assert (c["cnt"][rows[rows % TILE >= HALF], 180] == 0).all() and c["cnt"][rows, 180].any()
        groups = [c["eb"][g:g + TILE] for g in range(r0, r1, TILE)]
        assert (groups[0] == 7).all() and (groups[1] != 255).sum() == 1 and (groups[2] == 255).all()
    assert len(case_500_blocks()["brs"]) == 501


def test_negative_case_reaches_negative_moves():
    c = case_negative()
    st = regimes(c)
    assert st["negative"] > 1000 and st["run_leaves_binade_and_returns"] >= 6, st
    assert ((c["ab"] <= 0) & (c["ws"] < 0) & c["cnt"][:, :NB].any(1)).any()     # negative weights the shared histogram must not see
    assert (c["ews"] < 0).any()
    # the collapsed run total (every move in acc's binade at the run's start, added in any order) is not what the loop gives
    lost = 0
    for _, _, _, rows, w, cc in _sequences(c):
        part = _fold(w, cc)
        first = np.concatenate([[0], np.cumsum(cc)[:-1]])
        for r in np.unique(rows // TILE):
            sel = np.nonzero(rows // TILE == r)[0]
            a0 = part[first[sel[0]]]
            a1 = part[first[sel[-1]] + cc[sel[-1]]]
            if a0 > 0 and (w[sel] < 0).any():
                M = np.float64(1.5) * np.ldexp(1.0, np.frexp(a0)[1] - 1)
                d = (w[sel] + M) - M
                t = np.float64(a0 + np.sum(cc[sel] * d))
                lost += int(np.frexp(t)[1] == np.frexp(a0)[1] and t != a1)
    assert lost > 0


# ---- the device replay_row / add_repeated: the host test's cases, ties, negative weights
def _row_cases():
    rng = np.random.default_rng(5)
    cases = []
    for _ in range(4000):
        w = float(rng.integers(0, 3) * rng.integers(0, 40) / (rng.integers(1, 60) * 100.0))
        acc = float(rng.choice([0.0, w, rng.uniform(0, 1e-3), rng.uniform(0, 4), np.exp(rng.uniform(-5, 12))]))
        cases.append((acc, w, int(rng.integers(1, 101))))
    for e in range(-6, 14):
        top = 2.0 ** e
        for w in (top / 64, top / 64 * (1 + 2.0 ** -30), 0.3 * top, top / 3, top * 2.0 ** -52, top * 2.0 ** -53, top * 1.5 * 2.0 ** -53):
            for back in (1, 2, 7, 63, 64, 65):
                cases.append((float(np.float64(top) - np.float64(back) * np.float64(w)), float(w), 100))
                cases.append((float(np.nextafter(top, 0)), float(w), 37))
    for k in (-30, 0, 12, 40):                                     # ties: w ends in exactly ulp(acc) / 2, acc even and odd
        U = 2.0 ** (k - 44)
        for acc in (300.0 * 2.0 ** k, 300.0 * 2.0 ** k + U, 511.0 * 2.0 ** k, 511.0 * 2.0 ** k + U):
            for m in (0, 1, 2, 5, 1000, 123457):
                for c in (1, 2, 3, 4, 5, 17, 100, 255):
                    cases.append((acc, (m + 0.5) * U, c))
        for w in (-(2.0 ** k), -3.3 * 2.0 ** k, -(0.5 * U), -(7.5 * U)):   # negative weights (the slow path's wrapped products)
            for c in (1, 5, 100):
                cases.append((300.0 * 2.0 ** k, w, c))
    a, w, c = (np.array(x) for x in zip(*cases))
    return a.astype(np.float64), w.astype(np.float64), c.astype(np.int32)


def _plain_rows(a, w, c):
    acc = a.copy()
    for j in range(int(c.max())):
        acc = np.where(j < c, acc + w, acc)
    return acc


def test_row_cases_reach_ties_and_negative_weights():
    a, w, c = _row_cases()
    assert (w < 0).sum() >= 40
    n_tie = sum(int(_ties(np.float64(x), np.float64(y), np.float64(x + y))) for x, y in zip(a, w))
    assert n_tie > 300


# ---- raw count weights: the reference's int products wrap
def _wrap32(x):
    return ((np.asarray(x, np.int64) + 2**31) % 2**32) - 2**31


def _narrow_bin_ages(rng, n, bins):
    """(age_begin, age_end) as float32 with every age in between in bin bins[i] (10 ln(10 a) within 0.02 of the bin's centre)"""
    k = np.asarray(bins)
    a = np.exp((k - 1) / 10.0) / 10.0
    ab = (a * (1 - rng.uniform(1e-4, 1e-3, n))).astype(np.float32)
    ae = (a * (1 + rng.uniform(1e-4, 1e-3, n))).astype(np.float32)
    return ab, ae


def _rowcount_sites(pos, ab, ae, rng):
    n = pos.shape[0]
    acgt = np.frombuffer(b"ACGT", np.uint8)
    a = rng.integers(0, 4, n)
    d = (a + rng.integers(1, 4, n)) % 4
    return synth.Sites(["1"], np.array([0, n], np.int64), pos.astype(np.int32), ab, ae, np.zeros(n, np.uint8), np.ones(n, np.int32),
                       acgt[a].copy(), acgt[d].copy(), np.zeros(n, np.uint8), [int(pos[-1]) + 10])


def wrap_dataset(seed, narrow):
    """Row-count genomes (front_end = 1) with depths up to 10^5 on both sides: DAF_t * DAF_r and AAF_t * DAF_r pass 2^31 (negative
    int32) and 2^32 (positive again) on some rows.  narrow=True: every row's ages lie inside one bin (age_begin > 0) or below
    the first bin edge (age_begin = 0, emp rows), so that every addition of the reference is known without the generator."""
    rng = np.random.default_rng(seed)
    n = 1500
    pos = np.sort(rng.choice(np.arange(1, 3 * B), n, replace=False))
    if narrow:
        emp = rng.random(n) < 0.25
        ab, ae = _narrow_bin_ages(rng, n, rng.integers(20, 150, n))
        ab[emp] = 0.0
        ae[emp] = np.float32(0.05)
    else:
        ab = np.where(rng.random(n) < 0.3, 0.0, np.exp(rng.uniform(np.log(10.0), np.log(2e4), n))).astype(np.float32)
        ae = (ab.astype(np.float64) + np.exp(rng.uniform(np.log(50.0), np.log(5e4), n))).astype(np.float32)
    sites = _rowcount_sites(pos, ab, ae, rng)
    deep = rng.random(n) < 0.5
    Nt = np.where(deep, rng.integers(60_000, 200_000, n), rng.integers(1, 3000, n))
    Nr = np.where(deep, rng.integers(60_000, 200_000, n), rng.integers(1, 3000, n))
    dt = rng.binomial(Nt, rng.uniform(0.2, 0.9, n))
    dr = np.maximum(rng.binomial(Nr, rng.uniform(0.2, 0.9, n)), 1)
    tc = np.stack([Nt - dt, dt], 1).astype(np.int32)
    rc = np.stack([Nr - dr, dr], 1).astype(np.int32)
    return sites, tc, rc


def tie_dataset(seed):
    """Raw weights that tie in production: reference rows with N_ref = 2^30 and DAF_t * DAF_r (and AAF_t * DAF_r) = 25 x odd,
    so w = odd / 2^32, whose last bit is half an ulp once the bin's sum is in [2^21, 2^22); large-weight rows of the same
    bin (all 100 samples of a row in it) bring the sum there."""
    rng = np.random.default_rng(seed)
    groups = [int(b) for b in rng.choice(np.arange(30, 140), 6, replace=False)]
    rows = []                                                      # (bin, AAF_t, DAF_t, AAF_r, DAF_r)
    for g in groups:
        big = lambda: (int(rng.integers(30_000, 42_000)), int(rng.integers(30_000, 42_000)), 0, 50_000)   # w = DAF_t / 100
        for _ in range(75):
            rows.append((g,) + big())
        for i in range(50):
            if i % 5 == 4:
                rows.append((g,) + big())
            else:
                qr = 2 * int(rng.integers(100, 2000)) + 1
                dt, at = 2 * int(rng.integers(0, 40)) + 1, 2 * int(rng.integers(0, 40)) + 1
                rows.append((g, at, dt, 2**30 - 25 * qr, 25 * qr))
    n = len(rows)
    k = np.array([r[0] for r in rows])
    ab, ae = _narrow_bin_ages(rng, n, k)
    pos = np.sort(rng.choice(np.arange(1, 2 * B), n, replace=False))
    sites = _rowcount_sites(pos, ab, ae, rng)
    tc = np.array([(r[1], r[2]) for r in rows], np.int32)
    rc = np.array([(r[3], r[4]) for r in rows], np.int32)
    return sites, tc, rc


def restate_narrow(sites, tc, rc):
    """The reference's additions for a narrow dataset (every row usable, its samples in one known bin) with the int32
    products wrapped explicitly: the four histograms and the per-bin addition sequences (block, histogram, bin, w, c)."""
    at, dt = tc[:, 0].astype(np.int64), tc[:, 1].astype(np.int64)
    ar, dr = rc[:, 0].astype(np.int64), rc[:, 1].astype(np.int64)
    nr = (ar + dr).astype(np.float64)
    ps, pn = _wrap32(dt * dr).astype(np.float64), _wrap32(at * dr).astype(np.float64)
    ws, wn = ps / (nr * 100.0), pn / (nr * 100.0)
    emp = sites.age_begin <= 0
    bin_of = np.array([po.lib().oracle_bin_of_double_age(float(x)) for x in sites.age_end])
    assert np.array_equal(bin_of[~emp], [po.lib().oracle_bin_of_double_age(float(x)) for x in sites.age_begin[~emp]])
    assert (bin_of[emp] == 0).all()                                # every sample of an emp row in [0, 0.05): bin 0
    blk = (sites.pos.astype(np.int64) - 1) // B
    nb = int(blk.max()) + 1
    out = {k: np.zeros((nb, NB)) for k in ("shared", "notshared", "shared_emp", "notshared_emp")}
    seqs = []
    for b in range(nb):
        for k in range(NB):
            sel = (blk == b) & (bin_of == k)
            if sel.any():
                c = np.full(sel.sum(), 100)
                for name, w, live in (("shared", ws, ~emp), ("notshared", wn, np.ones_like(emp))):
                    cc = c * live[sel]
                    out[name][b, k] = _fold(w[sel], cc)[-1]
                    seqs.append((b, name, k, w[sel], cc))
            sel = (blk == b) & emp & (bin_of == k)
            if sel.any():
                out["shared_emp"][b, k] = _fold(ps[sel] / nr[sel], np.ones(sel.sum(), int))[-1]
                out["notshared_emp"][b, k] = _fold(pn[sel] / nr[sel], np.ones(sel.sum(), int))[-1]
    return out, seqs, dt * dr, at * dr


def test_oracle_raw_weights_are_wrapped_int32_products():
    sites, tc, rc = wrap_dataset(11, narrow=True)
    want, _, ps, pn = restate_narrow(sites, tc, rc)
    assert (ps >= 2**31).sum() > 100 and (pn >= 2**31).sum() > 50 and (ps >= 2**32).sum() > 20
    assert (_wrap32(ps) < 0).sum() > 50 and (_wrap32(pn) < 0).sum() > 20
    o = po.stage1_pileup(sites, tc, rc, seed=11)
    assert o["num_blocks"] == 3 and o["n_used_total"] == sites.n
    for k, v in want.items():
        assert np.array_equal(o[k].view(np.uint64), v.view(np.uint64)), k
    assert (o["shared"] < 0).any() and (o["notshared"] < 0).any()
    assert ((_wrap32(ps) < 0) & (sites.age_begin <= 0)).any()          # negative emp additions too


def test_tie_dataset_ties_in_the_reference_loop():
    sites, tc, rc = tie_dataset(12)
    want, seqs, ps, pn = restate_narrow(sites, tc, rc)
    assert (ps < 2**31).all() and (pn < 2**31).all()
    ties = Counter()
    for _, name, _, w, c in seqs:
        part = _fold(w, c)
        ties[name] += int(_ties(part[:-1], np.repeat(w, c), part[1:]).sum())
    assert ties["shared"] > 1000 and ties["notshared"] > 1000, ties
    o = po.stage1_pileup(sites, tc, rc, seed=12)
    for k, v in want.items():
        assert np.array_equal(o[k].view(np.uint64), v.view(np.uint64)), k


@pytest.mark.skipif(not po.ref_available(), reason="oracle/_ref not built (needs the reference's sources)")
def test_wrapped_raw_weights_vs_live_reference():
    """The reference's own parse_vcfvcf on genotype records 10^5 haplotypes deep (DAF_t * DAF_r past 2^31 and 2^32) ==
    the oracle on the same row counts: the wrapped products are the reference's, not an artefact of the restatement."""
    import os
    import tempfile
    rng = np.random.default_rng(15)
    n = 40
    pos = np.sort(rng.choice(np.arange(1, B), n, replace=False))
    ab = np.where(rng.random(n) < 0.3, 0.0, np.exp(rng.uniform(np.log(10.0), np.log(2e4), n))).astype(np.float32)
    ae = (ab.astype(np.float64) + np.exp(rng.uniform(np.log(50.0), np.log(5e4), n))).astype(np.float32)
    sites = _rowcount_sites(pos, ab, ae, rng)
    (ns_t, n_t), (ns_r, n_r) = (50_000, 100_000), (40_000, 80_000)
    dt = rng.integers(30_000, n_t, n)
    dr = rng.integers(30_000, n_r, n)
    assert (_wrap32(dt * dr) < 0).sum() > 5 and (dt * dr >= 2**32).sum() > 5
    with tempfile.TemporaryDirectory() as d:
        synth.write_dataset(d, sites, {})
        for tag, ns, N, daf in (("t", ns_t, n_t, dt), ("r", ns_r, n_r, dr)):
            recs = [(int(p) - 1, [bytes([int(a)]), bytes([int(b)])], [1] * int(k) + [0] * (N - int(k)))
                    for p, a, b, k in zip(sites.pos, sites.anc, sites.der, daf)]
            po.write_fake_bcf(os.path.join(d, f"{tag}_chr1.bcf"), ns, 2, recs)
        r = po.ref_parse_vcfvcf(d, sites.chr_names, "syn", "t", "r", seed=15)
    tc = np.stack([n_t - dt, dt], 1).astype(np.int32)
    rc = np.stack([n_r - dr, dr], 1).astype(np.int32)
    o = po.stage1_pileup(sites, tc, rc, seed=15)
    assert o["num_blocks"] == r["num_blocks"] == 1 and o["n_used_total"] == n
    for k in ("shared", "notshared", "shared_emp", "notshared_emp"):
        assert np.array_equal(o[k].view(np.uint64), r[k].view(np.uint64)), k
    assert (o["shared"] < 0).any()


# ================================================================================================= GPU
def _same(got, want, what):
    F, N, oor = got
    Fw, Nw, oorw = want
    assert F.shape == Fw.shape
    bad = np.argwhere(F.view(np.uint64) != Fw.view(np.uint64))
    assert bad.shape[0] == 0, (what, "sums", bad[:5].tolist(), [(F[tuple(i)], Fw[tuple(i)]) for i in bad[:5]])
    bad = np.argwhere(N != Nw)
    assert bad.shape[0] == 0, (what, "tallies", bad[:5].tolist())
    assert oor == oorw, (what, "bin-185 flag")


def _kernel(handle, c):
    return handle.test_replay(c["brs"], c["cnt"], c["ab"], c["ws"], c["wn"], c["eb"], c["ews"], c["ewn"])


@gpu
@pytest.mark.parametrize("name", list(CASES))
def test_replay_kernel_matches_the_plain_loop(handle, name):
    c = CASES[name]()
    _same(_kernel(handle, c), replay_ref(c), name)


@gpu
def test_replay_kernel_bin_185_flag(handle):
    for kw in (dict(bin185=True), dict(bin185_outside=True), {}):
        c = case_counts(**kw)
        _same(_kernel(handle, c), replay_ref(c), kw)


@gpu
def test_replay_kernel_rows_that_add_nothing_to_shared(handle):
    """The marker is age_begin <= 0 alone: such rows' shared weights, whatever their sign, never reach the shared histogram."""
    c = case_negative()
    for ws in (c["ws"], np.where(c["ab"] > 0, c["ws"], -0.0), np.where(c["ab"] > 0, c["ws"], 1e300)):
        d = dict(c, ws=ws)
        _same(_kernel(handle, d), replay_ref(d), "marker")
    d = dict(c, ab=np.zeros_like(c["ab"]))
    F, N, _ = _kernel(handle, d)
    assert (F[:, 0].view(np.uint64) == 0).all() and (N[:, 0] == 0).all()


@gpu
@pytest.mark.parametrize("which", ["replay_row", "add_repeated"])
def test_device_replay_row_matches_the_plain_loop(handle, which):
    a, w, c = _row_cases()
    if which == "replay_row":           # k_replay calls it for rows with acc >= 0, w != 0 and c > 4
        keep = (w != 0) & (c > 4)
        a, w, c = a[keep], w[keep], c[keep]
    got = handle.test_replay_row(which, a, w, c)
    want = _plain_rows(a, w, c)
    bad = np.nonzero(got.view(np.uint64) != want.view(np.uint64))[0]
    assert bad.shape[0] == 0, [(a[i], w[i], c[i], got[i], want[i]) for i in bad[:5]]


def _rowcount_stage1(handle, sites, tc, rc, seed):
    handle.set_option("front_end", 1)
    try:
        handle.set_sites(sites.site_off, sites.pos, sites.age_begin, sites.age_end, sites.meta())
        handle.set_row_counts(0, tc[:, 0], tc[:, 1])
        handle.set_row_counts(1, rc[:, 0], rc[:, 1])
        handle.set_mask(0, None); handle.set_mask(1, None)
        return handle.stage1(api.mt_seed(seed))
    finally:
        handle.set_option("front_end", 0)


@gpu
@pytest.mark.parametrize("narrow", [True, False])
def test_wrapped_raw_weights_end_to_end(handle, narrow):
    """Row counts whose int32 products wrap negative: stage i == the oracle bit for bit (the sums go negative)."""
    sites, tc, rc = wrap_dataset(11 if narrow else 13, narrow)
    o = po.stage1_pileup(sites, tc, rc, seed=11)
    s1 = _rowcount_stage1(handle, sites, tc, rc, 11)
    _compare_stage1(o, s1)
    assert (s1.block_stats[:, 0] < 0).any() and (s1.block_stats[:, 1] < 0).any()


@gpu
def test_raw_weight_ties_end_to_end(handle):
    sites, tc, rc = tie_dataset(12)
    o = po.stage1_pileup(sites, tc, rc, seed=12)
    _compare_stage1(o, _rowcount_stage1(handle, sites, tc, rc, 12))
