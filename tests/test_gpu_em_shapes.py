"""Stage ii and the three EM kernels against the oracle on inputs the synthetic bootstrap never produces.

Every other EM test bootstraps one dense synthetic dataset, starts from the flat rate 1/20000 and runs on `--bins` grids of
23 to 354 epochs.  There every age bin has counts, no rate reaches 0 (but the first epoch's), the 5e-9 floor or a value that
makes the deep epochs underflow, and every task's normaliser is finite.  The cases here reach the code the kernels hold for
everything else: the M-step's `num == 0` / `denom == 0` branches and its floor, the `de < 0` clamps, tasks with a non-finite
normaliser, zero-rate and zero-width epochs that hold age bins, the generic fallbacks behind the straight-line fold steps,
grids at the launcher's limits, and the iteration limits.  Every device result is compared with the oracle (or host glibc)
bit for bit.

Cases that need no device (oracle only) are not marked `gpu`.
"""
import functools
import math
import os

import numpy as np
import pytest

from colate_b200 import api, synth
from colate_b200._lib import ColateError
from oracle import pyoracle as po

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
gpu = pytest.mark.gpu
NB = 185


def bits_equal(a, b):
    """bit for bit (NaNs of any payload equal)"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(np.all((a.view(np.int64) == b.view(np.int64)) | (np.isnan(a) & np.isnan(b))))


# ---- inputs ------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _block_stats():
    sites = synth.make_sites(1, [30000, 20000], [2.5e8, 1.2e8])
    return po.stage1(sites, synth.make_genome(101, sites, 0.7), synth.make_genome(201, sites, 0.7), seed=1)


@functools.lru_cache(maxsize=None)
def _normal(age=0.0, R=10, seed=5):
    """R ordinary bootstrap replicates of the synthetic dataset at `age` (generations): [R][2][185]"""
    o = _block_stats()
    return po.stage2(api.draw_block_weights(api.mt_seed(seed), R, o["num_blocks"]), o, age)


def _grid(bins="3,7,0.2", age=0.0, ypg=28.0):
    ep, null = po.epochs_from_bins(bins, age, ypg)
    return ep, null


def _geom_grid(E):
    """an age-0 `--bins`-like grid of E epochs: [0, 0, 1e3/28 .. 1e7/28 (log-spaced), 1e8/28]"""
    return np.concatenate([[0.0, 0.0], np.geomspace(1e3 / 28, 1e7 / 28, E - 3), [1e8 / 28]])


FLAT = 1 / 20000.


def _flat(ep):
    return np.full(len(ep), FLAT)


def _epoch_of(ep, t):
    """epoch that holds age t (get_tint: grid points before t, minus one)"""
    return int(np.searchsorted(ep, t, side="right")) - 1


# ---- oracle (memoised: the same replicate is compared on every kernel) --------------------------------------------------
@functools.lru_cache(maxsize=None)
def _oracle_cached(ep_b, init_b, counts_b, max_iter):
    ep, init, c = (np.frombuffer(x, dtype=np.float64) for x in (ep_b, init_b, counts_b))
    r, it, ll = po.em_run(ep, init, c.reshape(2, NB), max_iter=max_iter)
    assert it >= 0, "the oracle refused the grid"
    return r, it, ll


def oracle(ep, init, counts_row, max_iter):
    return _oracle_cached(np.ascontiguousarray(ep, np.float64).tobytes(), np.ascontiguousarray(init, np.float64).tobytes(),
                          np.ascontiguousarray(counts_row, np.float64).tobytes(), max_iter)


def assert_rows(res, ep, init, counts, max_iter, rows=None, what=""):
    rates, iters, ll = res
    for r in (range(len(counts)) if rows is None else rows):
        ro, it, llo = oracle(ep, init, counts[r], max_iter)
        assert iters[r] == it, (what, r, iters[r], it)
        assert bits_equal(rates[r][:len(ep)], ro), (what, r, rates[r][:len(ep)], ro)
        assert bits_equal(ll[r], llo), (what, r, ll[r], llo)


# ---- which kernel runs ----------------------------------------------------------------------------------------------------
EMC_NT, EMC_THREADS, EMS_THREADS, EMS_TLMAX = 384, 640, 640, 96


def _emc_block(typ, et, E):
    n = E - et if typ else (min(E - 1, et + 1) + (1 if et == E - 1 else 0))
    return (n + 1) & ~1 if typ else n | 1


def cta_fits(ep):
    """em_cta_fits: k_em_cta's compact store and tables fit shared memory, and its first phase has threads enough"""
    E = len(ep)
    cap = sum(_emc_block(0, _epoch_of(ep, t), E) + _emc_block(1, _epoch_of(ep, t), E) for t in po.age_bins())
    smem = 8 * (11 * E + 4 + 192 + 6 * EMC_NT + 2 * cap) + 512 * 8 + EMC_NT * (16 + 4) + 192 * 16 + cap * 2 + 32
    return smem <= 225 * 1024 and ((E + 31) & ~31) + NB <= EMC_THREADS


def split_fits(E, cs):
    """run_em's split_fits: k_em_split's per-CTA tables on a cluster of cs CTAs"""
    nbl = (NB + cs - 1) // cs
    ntl, CW = 2 * nbl, (2 * E + 1 + cs - 1) // cs
    b = 8 * (10 * E + 1 + ntl * E * 3 + 2 * NB * CW) + 512 * 8
    return cs >= 8 and ntl <= EMS_TLMAX and b <= 200 * 1024 and E + 2 * nbl <= EMS_THREADS - 13 * 32 and \
        ((E + 31) & ~31) + nbl <= EMS_THREADS


def default_kernel(R, ep, sms):
    """the kernel run_em picks without COLATE_EM_* overrides: (name, CTAs per replicate)"""
    cs = 1
    while cs < 8 and R * cs * 2 <= sms:
        cs *= 2
    if cs == 8 and R * 32 <= sms:
        cs = 16
    if cs < 8:
        cs = 1
    split = split_fits(len(ep), cs)
    if not split and cs > 8:
        cs = 8
        split = split_fits(len(ep), cs)
    if not split and cs == 1 and cta_fits(ep):
        return "cta", 1
    return ("split" if split else "task"), cs


@functools.lru_cache(maxsize=None)
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


_EM_ENV = ("COLATE_EM_KERNEL", "COLATE_EM_CLUSTER", "COLATE_EM_NOSPLIT")
# route -> (environment, kernel it must reach)
ROUTES = {
    "cta": ({"COLATE_EM_KERNEL": "cta"}, ("cta", 1)),
    "task1": ({"COLATE_EM_KERNEL": "task", "COLATE_EM_CLUSTER": "1"}, ("task", 1)),          # k_em, one CTA per replicate
    "task8": ({"COLATE_EM_KERNEL": "task", "COLATE_EM_CLUSTER": "8", "COLATE_EM_NOSPLIT": "1"}, ("task", 8)),   # k_em, clusters
    "split8": ({"COLATE_EM_CLUSTER": "8"}, ("split", 8)),
    "split16": ({"COLATE_EM_CLUSTER": "16"}, ("split", 16)),
}
ALL_ROUTES = tuple(ROUTES) + ("grids",)


def em(handle, mp, route, ep, init, counts, max_iter, want=None):
    """stage3_em on one route; asserts the kernel that ran.  route None: the default launcher (want: its expected kernel)"""
    env, expect = ROUTES[route] if route else ({}, want)
    with mp.context() as m:
        for k in _EM_ENV:
            m.delenv(k, raising=False)
        for k, v in env.items():
            m.setenv(k, v)
        res = handle.stage3_em(len(counts), ep, init, counts, max_iter)
    assert handle.last_em() == expect, (route, handle.last_em(), expect)
    return res


def em_grids(handle, mp, ep, init, counts, max_iter, normal_ep, normal_counts):
    """the case's replicates interleaved with replicates on an ordinary grid, one stage3_em_grids call; returns the case's rows
    (and checks the ordinary ones against the oracle)"""
    R = len(counts)
    go = np.array([0, 1] * R, dtype=np.int32)
    cn = np.empty((2 * R, 2, NB))
    cn[0::2], cn[1::2] = counts, normal_counts[:R]
    with mp.context() as m:
        for k in _EM_ENV:
            m.delenv(k, raising=False)
        rates, iters, ll = handle.stage3_em_grids(go, [(ep, init), (normal_ep, _flat(normal_ep))], cn, max_iter)
    assert handle.last_em() == ("cta", 1)
    assert_rows((rates[1::2], iters[1::2], ll[1::2]), normal_ep, _flat(normal_ep), normal_counts[:R], max_iter, what="grids/normal")
    return rates[0::2, :len(ep)], iters[0::2], ll[0::2]


def check_case(handle, mp, ep, init, rows, max_iter, age=0.0, routes=ALL_ROUTES, mixed_to=10):
    """`rows` (<= 4 replicates) on every route against the oracle: alone, then interleaved into one launch with ordinary
    replicates of the same grid (at least `mixed_to` replicates in all)"""
    rows = np.ascontiguousarray(rows, dtype=np.float64).reshape(-1, 2, NB)
    normal = _normal(age)
    n_norm = max(len(rows), mixed_to - len(rows))
    mixed = np.concatenate([rows, normal[:n_norm]])
    order = np.argsort(np.concatenate([np.arange(len(rows)) * 2, np.arange(n_norm) * 2 + 1]), kind="stable")
    mixed = mixed[order]
    case_at = np.flatnonzero(order < len(rows))
    for route in routes:
        if route == "grids":
            nep, _ = _grid("3,7,0.2", age)
            res = em_grids(handle, mp, ep, init, rows, max_iter, nep, normal)
            assert_rows(res, ep, init, rows, max_iter, what="grids")
            continue
        assert_rows(em(handle, mp, route, ep, init, rows, max_iter), ep, init, rows, max_iter, what=route)
        rates, iters, ll = em(handle, mp, route, ep, init, mixed, max_iter)
        assert_rows((rates[case_at], iters[case_at], ll[case_at]), ep, init, rows, max_iter, what=route + "/mixed")
        others = np.setdiff1d(np.arange(len(mixed)), case_at)[:2]
        assert_rows((rates[others], iters[others], ll[others]), ep, init, mixed[others], max_iter, what=route + "/mixed normal")


# =========================================================================================================================
# 1. The fold primitives on the device
# =========================================================================================================================
def _needs_libm():
    if not api.libm_exact():
        pytest.skip("this host's libm is not glibc 2.39 / FMA")


def _hi_words(words, lows=(0, 1, 0xffffffff)):
    """doubles with the given high words and low words, and +-1 / +-2^32 ulp around each"""
    w = np.array(words, dtype=np.uint64)
    out = []
    for lo in lows:
        base = (w << np.uint64(32)) | np.uint64(lo)
        for d in (0, 1, -1, 1 << 32, -(1 << 32)):
            out.append((base.astype(np.int64) + d).view(np.float64))
    return np.concatenate(out)


# high words at which log1p_is_k0 / log1p_wide_ok / exp_is_main change their answer, and their neighbours
K0_WORDS = [0x3e1fffff, 0x3e200000, 0x3fda8279, 0x3fda827a, 0x3fd2bec3, 0x3fd2bec4]
WIDE_WORDS = [0x3c8fffff, 0x3c900000, 0x3e1fffff, 0x3e200000, 0x3fda8279, 0x3fda827a, 0x3fefffff, 0x3ff00000]
U_WORDS = [0x3ff6a09c, 0x3ff6a09d, 0x3ff6a09e, 0x3ff6a09f, 0x3ffffffb, 0x3ffffffc, 0x3ffffffd, 0x3ffffffe, 0x3fffffff]   # of u = 1 + x
EXP_WORDS = [0x3c8fffff, 0x3c900000, 0x407fffff, 0x40800000]


def _log1p_inputs(rng):
    x = [_hi_words(K0_WORDS), -_hi_words(K0_WORDS), _hi_words(WIDE_WORDS), _hi_words(U_WORDS) - 1.0,
         np.exp(-rng.uniform(0, 745, 200000)), -np.exp(-rng.uniform(0, 745, 100000)), rng.uniform(-0.3, 0.42, 100000),
         rng.uniform(0.40, 0.43, 100000), rng.uniform(0.9999, 1.0, 100000), rng.uniform(0, 1, 100000),
         # u = 1 + x with the high words where the generic code turns off (u/2 within 2^-20 of 1)
         ((np.uint64(0x3ffffffc) + rng.integers(0, 4, 100000).astype(np.uint64)) << np.uint64(32) |
          rng.integers(0, 2 ** 32, 100000, dtype=np.uint64)).view(np.float64) - 1.0,
         np.array([0.0, -0.0, 1.0, -1.0, 2.0 ** -54, 2.0 ** -29, math.sqrt(2) - 1, 5e-324, np.inf, np.nan])]
    return np.concatenate(x)


def _k0_expected(x):
    """fdlibm log1p takes its k = 0 polynomial with f = x (and nothing else) for 2^-29 <= |x|, -0.2929 < x < 0.41422"""
    hx = (x.view(np.uint64) >> np.uint64(32)).astype(np.int64)
    ax = hx & 0x7fffffff
    neg = hx >> 31 == 1
    return (ax >= 0x3e200000) & np.where(neg, ax <= 0x3fd2bec3, ax <= 0x3fda8279)


def _wide_expected(x):
    """the branches of fdlibm log1p that log1p_wide restates for 0 <= x < 1: x < 0.41422 (k = 0, any size), or u = 1 + x in
    [sqrt2, 2) with u/2 not within 2^-20 of 1 (k = 1 and the polynomial); the generic code does something else elsewhere"""
    hx = (x.view(np.uint64) >> np.uint64(32)).astype(np.int64)
    with np.errstate(invalid="ignore"):
        hu = ((x + 1.0).view(np.uint64) >> np.uint64(32)).astype(np.int64)
    band = (hu >> 20 == 0x3ff) & ((hu & 0xfffff) > 0x6a09d) & ((0x100000 - (hu & 0xfffff)) >> 2 != 0)
    return (hx >= 0) & (hx <= 0x3fefffff) & ((hx <= 0x3fda8279) | band)


def _lse_ref(a, b):
    """coal_EM::logsumexp with host libm: hi + log1p(exp(lo - hi))"""
    out = np.empty_like(a)
    fa, fb = np.isfinite(a), np.isfinite(b)
    out[~fa] = np.where(fb[~fa], b[~fa], -np.inf)
    m = fa & ~fb
    out[m] = a[m]
    m = fa & fb
    hi, lo = np.maximum(a[m], b[m]), np.minimum(a[m], b[m])
    out[m] = hi + po.libm("log1p", po.libm("exp", lo - hi))
    return out


def _lme_ref(a, b):
    """coal_EM::logminusexp with host libm: a + log1p(-exp(b - a))"""
    out = np.full_like(a, -np.inf)
    fa, fb = np.isfinite(a), np.isfinite(b)
    m = fa & ~fb
    out[m] = a[m]
    m = fa & fb & ~(a < b)
    out[m] = a[m] + po.libm("log1p", -po.libm("exp", b[m] - a[m]))
    return out


def test_fold_predicates_follow_the_generic_branches_on_the_host(built):
    """The host build of log1p_wide_ok agrees with the branch structure of fdlibm's log1p at every edge it names (and the
    values agree with libm wherever it holds)."""
    _needs_libm()
    x = _log1p_inputs(np.random.default_rng(1))
    x = x[(x >= 0) & (x <= 1)]
    y, ok = np.zeros_like(x), np.zeros(x.shape[0], np.int32)
    api.lib().colate_test_log1p_wide(x.shape[0], np.ascontiguousarray(x), y, ok)
    assert np.array_equal(ok == 1, _wide_expected(x))
    assert bits_equal(y[ok == 1], po.libm("log1p", x[ok == 1]))


@gpu
def test_exp_main_on_the_device(handle):
    _needs_libm()
    rng = np.random.default_rng(2)
    x = np.concatenate([_hi_words(EXP_WORDS), -_hi_words(EXP_WORDS), -rng.uniform(0, 745, 300000), rng.uniform(-512, 512, 200000),
                        -np.exp(rng.uniform(-40, 6.5, 100000)), [0.0, -0.0, -708.4, -745.1, 511.9, -511.9, 2.0 ** -54]])
    y, ok = handle.em_prims("exp_main", x)
    top = (x.view(np.uint64) >> np.uint64(52)).astype(np.int64) & 0x7ff
    assert np.array_equal(ok == 1, (top >= 0x3c9) & (top <= 0x407))          # 2^-54 <= |x| < 512
    assert bits_equal(y[ok == 1], po.libm("exp", x[ok == 1]))


@gpu
@pytest.mark.parametrize("which", ["log1p_k0", "log1p_wide"])
def test_log1p_straight_lines_on_the_device(handle, which):
    """The device's straight-line log1p pieces equal host log1p wherever their predicate holds, and the predicates admit
    exactly the inputs for which fdlibm's generic code takes the restated branches."""
    _needs_libm()
    x = _log1p_inputs(np.random.default_rng(3))
    y, ok = handle.em_prims(which, x)
    expected = _k0_expected(x) if which == "log1p_k0" else _wide_expected(x)
    bad = (ok == 1) != expected
    assert not bad.any(), (x[bad][:5], ok[bad][:5])
    assert bits_equal(y[ok == 1], po.libm("log1p", x[ok == 1]))
    assert (ok == 1).sum() > x.shape[0] // 10


@gpu
def test_div_midrange_on_the_device(handle):
    """rcp.approx + two Newton steps + correction == IEEE division (correctly rounded, like __ddiv_rn) on the operands the
    folds give it: (f, f + 2) for the log1p polynomials, (x - (u - 1), u) for log1p_wide's k = 1 term, and mid-range pairs."""
    rng = np.random.default_rng(4)
    f = np.concatenate([rng.uniform(-0.2929, 0.41422, 300000), np.exp(-rng.uniform(0, 45, 100000)),
                        -np.exp(-rng.uniform(1.2, 45, 100000)), rng.uniform(-0.2929, 0.0, 50000)])
    x = np.concatenate([rng.uniform(0.41421, 1.0, 200000), _hi_words(U_WORDS) - 1.0])
    u = x + 1.0
    num = x - (u - 1.0)
    a = np.concatenate([f, num, rng.uniform(1, 2, 200000) * 2.0 ** rng.integers(-500, 500, 200000),
                        -rng.uniform(1, 2, 1000) * 2.0 ** rng.integers(-500, 500, 1000)])
    b = np.concatenate([f + 2.0, u, rng.uniform(1, 2, 200000) * 2.0 ** rng.integers(-500, 500, 200000),
                        rng.uniform(1, 2, 1000) * 2.0 ** rng.integers(-500, 500, 1000)])
    y, _ = handle.em_prims("div_midrange", a, b)
    assert bits_equal(y, a / b)
    assert (num != 0).sum() > 1000                   # the k = 1 correction term is not always 0


def _fold_operands(rng):
    """pairs for the fold steps: running sums and terms at every distance, +-inf / NaN, equal operands, differences past
    -512 and -745 (exp underflows), and the log1p band edges of the terms"""
    n = 200000
    s = rng.uniform(-2000, 10, n)
    d = np.concatenate([rng.uniform(0, 1, n // 4), rng.uniform(0, 40, n // 4), rng.uniform(0, 800, n // 4),
                        np.exp(rng.uniform(-40, 0, n // 4))])
    a = np.concatenate([s, s - d])
    b = np.concatenate([s - d, s])
    t = np.log(np.concatenate([_hi_words(K0_WORDS), _hi_words(WIDE_WORDS), _hi_words(U_WORDS) - 1.0]).clip(5e-324, None))
    specials = np.array([0.0, -0.0, 1.0, -np.inf, np.inf, np.nan, -745.2, -512.0, -1e300, 3.0])
    sa, sb = np.meshgrid(specials, specials)
    a = np.concatenate([a, np.full(t.shape, -3.0), sa.ravel(), [5.0, -7.0, -1e3], np.full(3, -100.0)])
    b = np.concatenate([b, t - 3.0, sb.ravel(), [5.0, -7.0, -1e3], [-100.0 - 512.0, -100.0 - 512.5, -100.0 - 745.2]])
    return a, b


@gpu
@pytest.mark.parametrize("which", ["lse", "lse_wide", "lme"])
def test_fold_steps_equal_the_generic_formula(handle, which):
    """lse / lse_wide / lme on the device == the generic formula with host libm for every operand pair, whichever path the
    step took; both paths are taken."""
    _needs_libm()
    a, b = _fold_operands(np.random.default_rng(5))
    y, ok = handle.em_prims(which, a, b)
    want = _lme_ref(a, b) if which == "lme" else _lse_ref(a, b)
    bad = ~((y.view(np.int64) == want.view(np.int64)) | (np.isnan(y) & np.isnan(want)))
    assert not bad.any(), (a[bad][:5], b[bad][:5], y[bad][:5], want[bad][:5])
    assert 0.01 < ok.mean() < 0.999, ok.mean()        # both the straight line and the generic fallback ran


# =========================================================================================================================
# 2. Which kernel ran: the default launcher's thresholds, from the device's SM count
# =========================================================================================================================
@gpu
def test_default_launcher_thresholds(handle, monkeypatch):
    """Up to SMs/32 replicates run on 16-CTA clusters, up to SMs/8 on clusters of 8 (k_em_split), from there on one CTA
    per replicate (k_em_cta); both sides of each threshold, and 9 / 10."""
    sms = sm_count()
    ep, _ = _grid()
    init = _flat(ep)
    t16, t8 = sms // 32, sms // 8
    seen = set()
    for R in sorted({max(1, t16), t16 + 1, 9, 10, t8, t8 + 1}):
        counts = _normal(0.0, R, seed=21)
        want = default_kernel(R, ep, sms)
        seen.add(want)
        res = em(handle, monkeypatch, None, ep, init, counts, 40, want=want)
        assert_rows(res, ep, init, counts, 40, rows=(0, R - 1), what=f"R={R}")
    assert {("split", 16), ("split", 8), ("cta", 1)} <= seen


# =========================================================================================================================
# 3. Count vectors
# =========================================================================================================================
def _count_cases():
    ep, _ = _grid()
    ab = po.age_bins()
    et = np.array([_epoch_of(ep, t) for t in ab])
    first = int(np.flatnonzero(et == 1)[1])          # an age in the first epoch of non-zero width (epoch 0 is [0, 0))
    last = int(np.flatnonzero(et == len(ep) - 1)[0])  # an age in the last epoch
    base = _normal(0.0)[0]
    rng = np.random.default_rng(6)

    def one(typ, b, c=1000.0):
        v = np.zeros((2, NB))
        v[typ, b] = c
        return v

    def scattered(k):
        v = np.zeros((2, NB))
        v[rng.integers(0, 2, k), rng.choice(NB, k, replace=False)] = rng.uniform(1, 1e4, k)
        return v

    def below(b):
        v = base.copy()
        v[:, :b] = 0.0
        return v

    neg0 = base.copy()
    neg0[:, ::2] = -0.0
    fe = base / 1e3
    fe[:, 40:60] = 1e-6
    fe[1, 100:110] = 3e-6
    big = base.copy()
    big[:, 30:35] = 1e9
    allbig = np.where(base > 0, 1e9, 0.0)
    return {
        "one_bin_first_epoch": [one(0, first), one(1, first), one(0, first, 1e-6), one(1, first, 1e9)],
        "one_bin_last_epoch": [one(0, last), one(1, last), one(0, NB - 1), one(1, NB - 1)],
        "one_bin_age0": [one(0, 0), one(1, 0), one(0, 1), one(1, 2)],
        "scattered": [scattered(2), scattered(3), scattered(4), scattered(5)],
        "zero_below_age": [below(40), below(90), below(150), below(NB - 1)],
        "all_zero_and_inactive": [np.zeros((2, NB)), np.full((2, NB), -0.0), neg0, np.where(base > 0, -0.0, 0.0)],
        "front_end_sized": [fe, base / 1e3, np.where(base > 0, 1e-6, 0.0), fe[::-1].copy()],
        "huge": [big, allbig, base * 1e9 / base.max(), one(0, 60, 1e9) + one(1, 61, 1e9)],
    }


@gpu
@pytest.mark.parametrize("case", ["one_bin_first_epoch", "one_bin_last_epoch", "one_bin_age0", "scattered", "zero_below_age",
                                  "all_zero_and_inactive", "front_end_sized", "huge"])
def test_sparse_and_extreme_counts(handle, monkeypatch, case):
    ep, _ = _grid()
    rows = _count_cases()[case]
    check_case(handle, monkeypatch, ep, _flat(ep), rows, 60)
    if case == "all_zero_and_inactive":     # ll = 0, so ll / prev is NaN and the stop rule never fires
        rates, iters, ll = em(handle, monkeypatch, "cta", ep, _flat(ep), np.array(rows[:2]), 1003)
        assert (iters == 1003).all() and (ll == 0).all() and (rates == 0).all()


# =========================================================================================================================
# 4. Warm-start rates
# =========================================================================================================================
def _warm_cases():
    out = {}
    for tag, age in (("age0", 0.0), ("ancient", 250.0)):
        ep, null = _grid("3,7,0.2", age)
        for p in sorted({2, 3, null + 1}):
            r = _flat(ep)
            r[:p] = 0.0
            out[f"zero_prefix_{p}_{tag}"] = (ep, r, age)
    ep, _ = _grid()
    E = len(ep)
    rng = np.random.default_rng(7)
    deep01, deep1, mid1 = _flat(ep), _flat(ep), _flat(ep)
    deep01[E // 2:] = 0.1
    deep1[E // 2:] = 1.0
    mid1[5:9] = 1.0
    out.update({"floor_5e-9": (ep, np.full(E, 5e-9), 0.0), "deep_0.1": (ep, deep01, 0.0), "deep_1": (ep, deep1, 0.0),
                "mid_1": (ep, mid1, 0.0), "tiny_1e-300": (ep, np.full(E, 1e-300), 0.0),
                "log_uniform": (ep, np.exp(rng.uniform(np.log(1e-12), 0.0, E)), 0.0)})
    cep, cr = api.epochs_from_coal_file(os.path.join(GOLDEN, "cli_ancient.coal"), 250.0)
    out["cli_ancient_coal"] = (cep, cr, 250.0)
    return out


WARM = ["zero_prefix_1_age0", "zero_prefix_2_age0", "zero_prefix_3_age0", "zero_prefix_2_ancient", "zero_prefix_3_ancient", "zero_prefix_6_ancient",
        "floor_5e-9", "deep_0.1", "deep_1", "mid_1", "tiny_1e-300", "log_uniform", "cli_ancient_coal"]


def test_warm_start_cases_reach_the_branches(built):
    """(oracle only) the warm starts do what they are here for: zero-rate prefixes reach epochs that hold age bins (tasks with
    a non-finite normaliser), the deep rates underflow the numerators mid-grid (the M-step's copy-below rule), the tiny
    rates leave the log-likelihood at 0."""
    cases = _warm_cases()
    assert sorted(cases) == sorted(WARM)
    ab = po.age_bins()
    for name in WARM:
        ep, r, age = cases[name]
        if name.startswith("zero_prefix") and name != "zero_prefix_1_age0":      # (epoch 0 of an age-0 grid is [0, 0))
            p = int(name.split("_")[2])
            c = _normal(age)[0]
            held = [b for b in range(NB) if _epoch_of(ep, ab[b]) < p and (c[:, b] > 0).any()]
            assert held, name                                           # counts in the zero-rate epochs
            ll_bad = [po.estep(True, ep, r, ab[b])[0] for b in held]
            assert any(ll == 0.0 for ll in ll_bad), name           # coal_EM's `nc` is not finite: the task adds nothing
    for name in ("deep_0.1", "deep_1"):
        ep, r, _ = cases[name]
        tn = _numerators(ep, r, _normal(0.0)[0])
        first = int(np.argmax(tn != 0))
        assert tn[first] != 0 and (tn[first:] == 0).any(), name      # num == 0 above a non-zero one: the copy-below rule
    _, _, ll = oracle(*cases["tiny_1e-300"][:2], _normal(0.0)[0], 3)
    assert ll == 0.0


def _numerators(ep, rates, counts):
    """sum over the tasks of count * num[e] (the M-step's numerators), from the oracle's E-step probes"""
    tn = np.zeros(len(ep))
    for b, t in enumerate(po.age_bins()):
        for typ in (0, 1):
            if counts[typ, b] > 0:
                tn += counts[typ, b] * po.estep(typ == 0, ep, rates, t)[1]
    return tn


@gpu
@pytest.mark.parametrize("case", WARM)
def test_warm_start_rates(handle, monkeypatch, case):
    ep, r, age = _warm_cases()[case]
    check_case(handle, monkeypatch, ep, r, _normal(age)[:2], 60, age=age)


# =========================================================================================================================
# 5. Grids
# =========================================================================================================================
def _mid_zero_width():
    ep, _ = _grid()
    return np.insert(ep, 10, ep[10])               # two equal points mid-grid, age bins on both sides


GRIDS = {"E2": np.array([0.0, 1000.0]), "E3": np.array([0.0, 50.0, 5000.0]), "E3_age0": np.array([0.0, 0.0, 5000.0]),
         "mid_zero_width": None, "ypg1": ("3,7,0.2", 1.0), "ypg100": ("3,7,0.2", 100.0)}


def _grid_case(name):
    g = GRIDS[name]
    if name == "mid_zero_width":
        return _mid_zero_width()
    if isinstance(g, tuple):
        return _grid(g[0], 0.0, g[1])[0]
    return g


def test_grid_cases_are_what_they_claim(built):
    """(oracle only) the mid-grid zero-width epoch has age bins on both sides; ypg 1 puts no age bin in the last epoch,
    ypg 100 many."""
    ab = po.age_bins()
    ep = _mid_zero_width()
    assert ep[10] == ep[11] and any(_epoch_of(ep, t) == 9 for t in ab) and any(_epoch_of(ep, t) == 11 for t in ab)
    last = lambda ep: sum(_epoch_of(ep, t) == len(ep) - 1 for t in ab)
    assert last(_grid_case("ypg1")) == 0 and last(_grid_case("ypg100")) > 15


@gpu
@pytest.mark.parametrize("name", list(GRIDS))
def test_small_and_degenerate_grids(handle, monkeypatch, name):
    """E = 2 and 3 (on a 16-CTA cluster most CTAs of k_em_split own no column), a zero-width epoch mid-grid, years per
    generation 1 and 100."""
    ep = _grid_case(name)
    rows = [_normal(0.0)[0], _count_cases()["scattered"][3]]
    check_case(handle, monkeypatch, ep, _flat(ep), rows, 60)
    r = _flat(ep)
    r[: len(ep) // 2] = 0.0                          # zero rates in the epochs that hold most bins
    check_case(handle, monkeypatch, ep, r, rows[:1], 40, routes=("cta", "split16", "task1"))


def _limit(pred, lo=4, hi=1024):
    E = lo
    while E + 1 <= hi and pred(E + 1):
        E += 1
    return E


@gpu
def test_launcher_limits(handle, monkeypatch):
    """The largest grid k_em_cta fits and one epoch more (the launch moves to k_em), the largest grid k_em_split fits on
    16- and on 8-CTA clusters and one epoch more."""
    sms = sm_count()
    e_cta = _limit(lambda E: cta_fits(_geom_grid(E)))
    e16 = _limit(lambda E: split_fits(E, 16))
    e8 = _limit(lambda E: split_fits(E, 8))
    R = sms // 8 + 1                                 # one CTA per replicate
    for E, want in ((e_cta, ("cta", 1)), (e_cta + 1, ("task", 1))):
        ep = _geom_grid(E)
        assert default_kernel(R, ep, sms) == want
        counts = _normal(0.0, R, seed=22)
        assert_rows(em(handle, monkeypatch, None, ep, _flat(ep), counts, 30, want=want), ep, _flat(ep), counts, 30, rows=(0, R - 1))
    for E, route, want in ((e16, None, ("split", 16)), (e16 + 1, None, ("task", 8)), (e8, "split8", ("split", 8))):
        ep = _geom_grid(E)
        counts = _normal(0.0, 1, seed=23)
        if route is None:
            assert default_kernel(1, ep, sms) == want
        assert_rows(em(handle, monkeypatch, route, ep, _flat(ep), counts, 20, want=want), ep, _flat(ep), counts, 20)
    ep = _geom_grid(e8 + 1)
    counts = _normal(0.0, 1, seed=23)
    with monkeypatch.context() as m:
        m.setenv("COLATE_EM_CLUSTER", "8")
        res = handle.stage3_em(1, ep, _flat(ep), counts, 20)
    assert handle.last_em() == ("task", 8)
    assert_rows(res, ep, _flat(ep), counts, 20)


@gpu
@pytest.mark.parametrize("E", [207, 208, 243])
def test_k_em_one_cta_per_replicate_on_wide_grids(handle, monkeypatch, E):
    """k_em with one CTA per replicate sums 2E + 1 columns with 416 threads: from E = 208 on a thread owns several
    columns (the log-likelihood column first, then the exposures)."""
    ep = _grid("2,8,0.025")[0] if E == 243 else _geom_grid(E)
    assert len(ep) == E
    counts = _normal(0.0, 10, seed=24)
    res = em(handle, monkeypatch, "task1", ep, _flat(ep), counts, 4)
    assert_rows(res, ep, _flat(ep), counts, 4, rows=(0, 4, 9))
    if E == 208:                                     # the stop rule needs the log-likelihood column
        res = em(handle, monkeypatch, "task1", ep, _flat(ep), counts[:2], 3000)
        assert_rows(res, ep, _flat(ep), counts[:2], 3000)
        assert 1001 <= res[1].min() < 3000
    if E == 243:                                     # reached by the default launcher once replicates outnumber SMs / 8
        R = sm_count() // 8 + 1
        counts = _normal(0.0, R, seed=24)
        res = em(handle, monkeypatch, None, ep, _flat(ep), counts, 3, want=("task", 1))
        assert_rows(res, ep, _flat(ep), counts, 3, rows=(0, R - 1))


@gpu
@pytest.mark.parametrize("E", [513, 1024])
def test_largest_grids_against_the_raised_oracle(handle, monkeypatch, E):
    """E above the oracle's former 512: the E-step probe (k_estep: 8 (6E + 1) bytes of shared memory, over 48 KB at
    E = 1024) and k_em on one CTA and on clusters of 8, a few iterations."""
    ep = _geom_grid(E)
    rates = np.exp(np.random.default_rng(E).uniform(np.log(1e-6), np.log(1e-2), E))
    ab = po.age_bins()
    for sh in (True, False):
        ll, num, den = handle.estep(sh, ep, rates, ab)
        for b in range(0, NB, 4):
            lo, no, do = po.estep(sh, ep, rates, ab[b])
            assert bits_equal(num[b], no) and bits_equal(den[b], do) and bits_equal(ll[b], lo), (sh, b)
    counts = _normal(0.0, 1, seed=25)
    for route in ("task1", None):
        res = em(handle, monkeypatch, route, ep, _flat(ep), counts, 2, want=("task", 8))
        assert_rows(res, ep, _flat(ep), counts, 2)


def test_oracle_above_512_epochs(built):
    """(oracle only) the oracle takes grids up to the ABI's 1024 epochs: one EM iteration equals the M-step of the per-task
    E-step probes summed in the reference's order, and the probes equal the compiled reference where it is present."""
    E = 600
    ep = _geom_grid(E)
    init = np.exp(np.random.default_rng(9).uniform(np.log(1e-6), np.log(1e-2), E))
    c = _count_cases()["scattered"][3] + _count_cases()["one_bin_last_epoch"][1]
    ab = po.age_bins()
    tn, td, ll = np.zeros(E), np.zeros(E), 0.0
    for b in range(NB):
        for sh in (True, False):
            cnt = c[0 if sh else 1, b]
            if cnt > 0:
                lo, no, do = po.estep(sh, ep, init, ab[b])
                ll += cnt * lo
                for e in range(E):
                    tn[e] += cnt * no[e]
                    td[e] += cnt * do[e]
    want = init.copy()
    for e in range(E):
        if tn[e] == 0:
            want[e] = want[e - 1] if e > 0 else 0.0
        elif td[e] != 0:
            want[e] = max(tn[e] / td[e], 5e-9)
    r, it, llo = po.em_run(ep, init, c, max_iter=1)
    assert it == 1 and bits_equal(r, want) and bits_equal(llo, ll)
    assert po.em_run(_geom_grid(1024), _flat(_geom_grid(1024)), c, max_iter=1)[1] == 1
    if not po.ref_available():
        pytest.skip("the compiled reference is not present")
    for t in ab[::23]:
        for sh in (True, False):
            a, b = po.estep(sh, ep, init, t), po.ref_estep(sh, ep, init, t)
            assert all(bits_equal(x, y) for x, y in zip(a, b))


# =========================================================================================================================
# 6. Iteration limits
# =========================================================================================================================
# seed of the bootstrap weights and initial rate of runs found with the oracle: seed 5 from the flat rate stops at the first
# iteration allowed to stop (1001); from 1e-9 everywhere it stops at 1164
STOP_FIRST = (5, FLAT, 1001)
STOP_LATER = (5, 1e-9, 1164)


def test_oracle_stop_iterations(built):
    """(oracle only) the runs of the iteration-limit test stop where it expects them to."""
    ep, _ = _grid()
    for seed, r0, stop in (STOP_FIRST, STOP_LATER):
        c = _normal(0.0, 1, seed)[0]
        assert oracle(ep, np.full(len(ep), r0), c, 100000)[1] == stop
        capped = oracle(ep, np.full(len(ep), r0), c, stop)
        assert capped[1] == stop and not bits_equal(capped[0], oracle(ep, np.full(len(ep), r0), c, 100000)[0])


@gpu
@pytest.mark.parametrize("max_iter", [0, 1, 2])
def test_tiny_iteration_limits(handle, monkeypatch, max_iter):
    ep, _ = _grid()
    rows = [_normal(0.0)[1], _count_cases()["one_bin_first_epoch"][0]]
    check_case(handle, monkeypatch, ep, _flat(ep), rows, max_iter)


@gpu
@pytest.mark.parametrize("route", ["cta", "task1", "split16", "split8"])
def test_stop_rule(handle, monkeypatch, route):
    """A run that stops at iteration 1001, one that stops later, and the latter capped one iteration before it would stop."""
    ep, _ = _grid()
    for seed, r0, stop in (STOP_FIRST, STOP_LATER):
        c = _normal(0.0, 1, seed)
        init = np.full(len(ep), r0)
        res = em(handle, monkeypatch, route, ep, init, c, 100000)
        assert res[1][0] == stop
        assert_rows(res, ep, init, c, 100000)
        capped = em(handle, monkeypatch, route, ep, init, c, stop)     # one M-step fewer, same iteration count
        assert capped[1][0] == stop and not bits_equal(capped[0], res[0])
        assert_rows(capped, ep, init, c, stop)


# =========================================================================================================================
# 7. Stage ii (k_bootstrap) against po.stage2
# =========================================================================================================================
def _blocks(nb, seed, emp=True):
    rng = np.random.default_rng(seed)
    mk = lambda: np.where(rng.random((nb, NB)) < 0.4, 0.0, rng.random((nb, NB)) * 100)
    b = {"shared": mk(), "notshared": mk(), "shared_emp": mk(), "notshared_emp": mk()}
    if not emp:
        b["shared_emp"][:] = 0.0
        b["notshared_emp"][:] = 0.0
    return b


def _stage2(handle, w, blk, age, front_end):
    stack = np.stack([blk["shared"], blk["notshared"], blk["shared_emp"], blk["notshared_emp"]], axis=1)
    handle.set_option("front_end", front_end)
    try:
        return handle.stage2_bootstrap(w, stack, age)
    finally:
        handle.set_option("front_end", 0)


def _stage2_cases():
    ab = po.age_bins()
    ages = [0.0, 2.0 ** -1074]
    for k in (1, 2, 3, 50, 120, 183, 184):
        ages += [np.nextafter(ab[k], 0), ab[k], np.nextafter(ab[k], np.inf)] if k < 184 else [np.nextafter(ab[k], 0)]
    blk20, w20 = _blocks(20, 1), api.draw_block_weights(api.mt_seed(3), 3, 20)
    some_emp = _blocks(20, 2)
    some_emp["shared_emp"][::2] = 0.0
    some_emp["notshared_emp"][::2] = 0.0
    w_zero = w20.copy()
    w_zero[1] = 0
    blk500 = _blocks(500, 3)
    one500 = np.zeros((2, 500), np.int32)
    one500[0, 17] = 500
    one500[1, 499] = 500
    cases = [(f"age_{a!r}", w20, blk20, a) for a in ages]
    cases += [("no_emp", w20, _blocks(20, 1, emp=False), 300.0), ("no_emp_age0", w20, _blocks(20, 1, emp=False), 0.0),
              ("some_blocks_no_emp", w20, some_emp, 40.0), ("zero_weights", w_zero, blk20, 10.0),
              ("one_block", api.draw_block_weights(api.mt_seed(4), 3, 1), _blocks(1, 4), 5.0),
              ("500_blocks", api.draw_block_weights(api.mt_seed(5), 3, 500), blk500, 100.0),
              ("one_block_500_times", one500, blk500, 1.0)]
    return cases


@gpu
@pytest.mark.parametrize("front_end", [0, 1])
def test_stage2_edges(handle, front_end):
    """Ages on and one ulp either side of age_bin[k] (the `<=` that picks the first bin of the redistribution), the largest
    age the ABI accepts, blocks without emp counts (normf = 0), a replicate whose weights are all zero, one block, 500 blocks,
    one block drawn 500 times; tmp/tmp and the 1e3-normalised front-ends."""
    for name, w, blk, age in _stage2_cases():
        got = _stage2(handle, w, blk, age, front_end)
        want = po.stage2(w, blk, age, norm_1e3=bool(front_end))
        assert bits_equal(got, want), name
    ab = po.age_bins()
    w, blk = api.draw_block_weights(api.mt_seed(3), 1, 20), _blocks(20, 1)
    for age in (ab[184], np.nextafter(ab[184], np.inf), -1e-300, np.nan):
        with pytest.raises(ColateError):
            _stage2(handle, w, blk, age, front_end)
