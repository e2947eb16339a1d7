"""GPU: every layout of the generator stream word for word against std::mt19937.

Stage i draws every age from one MT19937 stream that kernels_mt.cu produces on the device: k_jump reaches the chunk
windows, one of six generator kernels writes the words (k_gen<TILED, PRE, W32>, k_gen_tma) in k_sample's tile order
(internal.h: stream_phys), and the state after the last word comes from the tail the generator leaves or from
k_tail_gather.  A misplaced word does not fault, it moves samples between bins; so each layout is compared here word for
word, including the words no kernel may write, the state after the stream, and streams past 2^31 words.

Reference: oracle_mt_words (std::mt19937 restated in C, pinned to libstdc++ by test_random_streams_match_libstdcxx); far
into a stream, the host jump-ahead (colate_test_jump_window_host, pinned to the oracle by
test_characteristic_polynomial_and_jumps) followed by colate_mt_generate.
"""
import time

import numpy as np
import pytest

from colate_b200 import api, synth
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

TILE = api.SAMPLE_TILE_WORDS
CANARY = 0xA5A5A5A5
PATHS = {"tma": (2, 0), "w32": (1, 0), "w64": (1, 1)}     # (gen_path, gen_w64)
SEEN = set()        # generator kernels the tests of this file reached
PAST_2_31 = set()   # ... on streams longer than 2^31 words


@pytest.fixture
def gen(handle):
    """The session handle with the generator options reset after the test."""
    yield handle
    handle.set_stream_cache(False)
    handle.set_option("gen_path", 0)
    handle.set_option("gen_w64", 0)


def _state_at(seed, word0):
    """State window in front of word `word0` of the seed's stream: one host jump of 200 * 2^q words per set bit q of
    word0 // 200, then the remaining words one by one."""
    w = api.mt_seed(seed)
    r, rest = divmod(word0, 200)
    q = 0
    while r:
        if r & 1:
            jw = np.zeros(624, np.uint32)
            assert api.lib().colate_test_jump_window_host(w, q, jw) == 0
            w = jw
        r >>= 1
        q += 1
    if rest:
        api.lib().colate_mt_generate(w, rest, np.zeros(rest, np.uint32))
    return w


def ref_words(seed, word0, n):
    out = np.zeros(max(n, 1), np.uint32)
    if word0 <= 1 << 22:
        po.lib().oracle_mt_words(seed, word0, n, out)
    else:
        api.lib().colate_mt_generate(_state_at(seed, word0), n, out)
    return out[:n]


def _phys(o, off):
    """internal.h: stream_phys for arrays (20-word chunks)."""
    o = np.asarray(o, np.int64)
    q = o - off
    row = q // 200
    w = q - row * 200
    c = w // 20
    p = off + (((row >> 5) * 10 + c) * 32 + (row & 31)) * 20 + (w - c * 20)
    return np.where(o < off, o, p)


def _after_ok(after, seed, word):
    nxt = np.zeros(50, np.uint32)
    api.lib().colate_mt_generate(after.copy(), 50, nxt)
    return np.array_equal(nxt, ref_words(seed, word, 50))


def _check_layout(buf, ref, off, n_rows, tma, lo=0):
    """buf = physical words [lo, lo + len(buf)) of a stream whose tiling starts at `off` and holds n_rows rows; ref = the
    oracle's words from physical / logical word lo on (lo: a tile boundary past off, or 0).  Words in front of off are
    linear, row words sit at stream_phys, everything else is the canary -- except that k_gen_tma's last group of 4 rows may
    carry up to 3 rows of ring contents past the last row (inside the last tile)."""
    exp = np.full(buf.shape, CANARY, np.uint32)
    free = np.zeros(buf.shape, bool)
    total = off + 200 * n_rows
    if lo == 0:
        exp[:off] = ref[:off]
    o = np.arange(max(lo, off), min(total, lo + len(buf)))
    exp[_phys(o, off) - lo] = ref[o - lo]
    if tma:
        rows = np.arange(n_rows, -(-n_rows // 4) * 4)
        p = _phys((off + rows[:, None] * 200 + np.arange(200)).ravel(), off) - lo
        free[p[(p >= 0) & (p < len(buf))]] = True
    bad = np.nonzero((buf != exp) & ~free)[0]
    assert bad.size == 0, (bad.size, bad[:8] + lo, buf[bad[:4]], exp[bad[:4]])


def test_stream_phys_formula(built):
    """The array form above against the library's own stream_phys."""
    rng = np.random.default_rng(0)
    for off in (0, 200, 200 * 37):
        o = np.concatenate([np.arange(0, 20000), rng.integers(0, 1 << 34, 2000)])
        got = np.array([api.lib().colate_test_stream_phys(int(x), off) for x in o])
        assert np.array_equal(got, _phys(o, off))


@pytest.mark.parametrize("k", [0, 1, 2, 3, 5, 8, 12])
def test_linear_stream(gen, k):
    """k_gen<false> (the layout-free kernel): starts at 0, on a chunk boundary, mid-chunk and behind a long jump chain into
    window 0 (a chunk index with many set bits); lengths around a round and a chunk; chunk counts M that are powers of two
    and not, with an odd and an even number of index bits (the radix-2 top level, then radix-4 levels)."""
    S = 200 << k
    seed = 11 + k
    st = api.mt_seed(seed)
    many_bits = (1 << 13) - 1 - (1 << 4) - (1 << 9)
    for word0 in (0, 5 * S, 3 * S + 377, many_bits * S + 200):
        for n in (0, 1, 623, 624, 625, S - 1, S, S + 1, 4 * S, 8 * S - 3, 5 * S + 7, 11 * S - S // 2):
            got, after = gen.mt_stream(st, word0, n, k)
            ref = ref_words(seed, word0, n + 50)
            assert np.array_equal(got, ref[:n]), (k, word0, n)
            nxt = np.zeros(50, np.uint32)
            api.lib().colate_mt_generate(after, 50, nxt)
            assert np.array_equal(nxt, ref[n:]), (k, word0, n)
            if word0 % S or n:
                assert gen.last_gen() == "linear"
                SEEN.add("linear")


def _tiled_case(h, path, k, pre, n_rows, seed):
    S = 200 << k
    r = 5 * 2 ** k + max(1, 3 * 2 ** k // 4) if pre else 3 * 2 ** k     # PRE: a first row that is not a chunk boundary
    word0 = 200 * r
    c0 = word0 // S
    off = word0 - c0 * S
    assert (off > 0) == pre
    buf, after = h.mt_stream_tiled(api.mt_seed(seed), word0, 200 * n_rows, k)
    kern = h.last_gen()
    want = ("pre_" if pre else "tiled_") + ("w64" if path == "w64" else "w32")
    if path == "tma" and k >= 2 and not pre:
        want = "tma"
    assert kern == want, (path, k, pre, kern)
    SEEN.add(kern)
    total = off + 200 * n_rows
    _check_layout(buf, ref_words(seed, c0 * S, total), off, n_rows, kern == "tma")
    assert _after_ok(after, seed, word0 + 200 * n_rows), (path, k, pre, n_rows)


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("pre", [False, True])
@pytest.mark.parametrize("k", [0, 1, 2, 3, 4, 7])
def test_tiled_stream(gen, path, pre, k):
    """The tile-ordered kernels: k_gen_tma (k >= 2, stream from a chunk boundary), k_gen<true, PRE, W32> with 32- and 64-bit
    addressing, from a chunk boundary and from a row inside a chunk (PRE); chunks of 1 and 2 rows (a 624-word round spans
    several chunks), 4 rows (the smallest the TMA path takes) and more; used rows around a group of 4, a tile of 32, a chunk
    and several tiles, down to one row (T < 624 words for the state after)."""
    if pre and k == 0:
        pytest.skip("with 1-row chunks every row starts a chunk")
    gp, w64 = PATHS[path]
    gen.set_option("gen_path", gp)
    gen.set_option("gen_w64", w64)
    m = 2 ** k
    for n in sorted({1, 3, 4, 5, 31, 32, 33, 3 * m - 1, 3 * m + 1, 32 * 5 + 1}):
        _tiled_case(gen, path, k, pre, n, seed=1000 + 7 * k + n)


def test_stream_cache_requests(gen):
    """colate_set_stream_cache as pairs.cohort uses it: a long request, then a shorter one (served from the cached stream,
    the state after through k_tail_gather), an equal one, a longer one (regenerated), one with another seed and one with
    another chunk size.  Every request gives the oracle's words at stream_phys and the oracle's state after."""
    gen.set_stream_cache(True)
    n1 = 5000
    reqs = [(5, n1, 3, False), (5, 1234, 3, True), (5, n1, 3, True), (5, 777, 2, True), (5, 3, 3, True),
            (5, 2 * n1, 3, False), (6, 1234, 3, False), (6, 1234, 4, True), (5, 900, 3, False)]
    for seed, n, k, cached in reqs:
        launches, kern = gen.launch_count(), gen.last_gen()
        buf, after = gen.mt_stream_tiled(api.mt_seed(seed), 0, 200 * n, k, n_phys=200 * n + TILE)
        if cached:
            assert gen.launch_count() - launches == 1 and gen.last_gen() == kern, (seed, n, k)   # k_tail_gather only
        else:
            assert gen.launch_count() - launches > 1, (seed, n, k)
        ref = ref_words(seed, 0, 200 * n)
        assert np.array_equal(buf[_phys(np.arange(200 * n), 0)], ref), (seed, n, k)
        assert _after_ok(after, seed, 200 * n), (seed, n, k)


def _same_stage1(a, b):
    """(stats, tallies, state) of two runs: bit for bit."""
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def _oracle(sites, gt, gr, seed):
    """po.stage1 with the 64 words after the stage in o["next"] (drawing them advances o["rng"])."""
    o = po.stage1(sites, gt, gr, seed=seed)
    o["next"] = np.array([po.lib().oracle_mt_next(o["rng"]) for _ in range(64)], np.uint32)
    return o


def _next_words(state, n=64):
    a = np.zeros(n, np.uint32)
    api.lib().colate_mt_generate(state.copy(), n, a)
    return a


def _stage1_whole(h, mt_state):
    s1 = h.stage1(mt_state)
    return s1.block_stats, s1.block_tallies, s1.mt_state


def _stage1_shards(h, sites, gt, gr, mt_state, cut):
    """Stage i as two chromosome shards (chromosomes [0, cut) and [cut, n_chr)) on one handle, the second sampled at its
    used-row offset of the stream (colate_stage1_sample with used_rank_base > 0): concatenated blocks, the last shard's state
    after, and the generator kernel of each shard."""
    n_chr = len(sites.chr_names)
    used_base = block_base = 0
    stats, tallies, kerns, state = [], [], [], None
    for lo, hi in ((0, cut), (cut, n_chr)):
        s0, s1 = int(sites.site_off[lo]), int(sites.site_off[hi])
        h.set_sites(sites.site_off[lo:hi + 1] - sites.site_off[lo], sites.pos[s0:s1], sites.age_begin[s0:s1],
                    sites.age_end[s0:s1], sites.meta()[s0:s1])
        for slot, g in ((0, gt), (1, gr)):
            first, end = api.chr_ranges(n_chr, g.chrom)
            al = g.anc.astype(np.uint16) | (g.der.astype(np.uint16) << 8)
            api.check(api.lib().colate_set_genome(h._h, slot, g.n, api.ptr(np.ascontiguousarray(first[lo:hi])),
                                                  api.ptr(np.ascontiguousarray(end[lo:hi])), api.ptr(g.bp), api.ptr(g.aaf),
                                                  api.ptr(g.daf), api.ptr(al), 0))
        h.set_mask(0, None)
        h.set_mask(1, None)
        used_chr, blocks_chr = h.stage1_flags()
        nb = int(np.sum(blocks_chr))
        st, tl, state = h.stage1_sample(mt_state, used_base, block_base, nb)
        stats.append(st[:nb])
        tallies.append(tl[:nb])
        kerns.append((used_base, h.last_gen()))
        used_base += int(np.sum(used_chr))
        block_base += nb
    return np.concatenate(stats), np.concatenate(tallies), state, kerns


def _check_oracle(o, res):
    stats, tallies, state = res
    assert stats.shape[0] == o["num_blocks"]
    assert np.array_equal(tallies[:, 0], o["n_shared"]) and np.array_equal(tallies[:, 1], o["n_notshared"])
    assert np.array_equal(tallies[:, 2], o["n_emp"])
    for v, k in enumerate(("shared", "notshared", "shared_emp", "notshared_emp")):
        assert np.array_equal(stats[:, v], o[k]), k
    assert np.array_equal(_next_words(state), o["next"])


def test_stage1_on_small_chunks(gen, monkeypatch):
    """Stage i with chunks of 1, 2 and 4 rows (COLATE_CHUNK_LOG2 = 0, 1, 2: k_gen<true> with rounds spanning chunks, and
    k_gen_tma at its smallest chunk), with 64-bit addressing forced, and as two shards whose second one starts inside a chunk
    (PRE): histograms, tallies and the state after bit for bit against the oracle."""
    seed = 1
    sites = synth.make_sites(seed, [4000, 3000, 5000], [2.5e8, 1.2e8, 0.9e8], weird=0.1)
    gt = synth.make_genome(seed + 100, sites, 0.7, weird=0.1)
    gr = synth.make_genome(seed + 200, sites, 0.6, weird=0.1)
    o = _oracle(sites, gt, gr, seed)
    pre_seen = set()
    for k, w64, want in ((0, 0, "tiled_w32"), (1, 0, "tiled_w32"), (2, 0, "tma"), (3, 0, "tma"), (1, 1, "tiled_w64")):
        monkeypatch.setenv("COLATE_CHUNK_LOG2", str(k))
        gen.set_option("gen_w64", w64)
        gen.set_option("gen_path", 1 if w64 else 2)
        gen.load(sites, gt, gr)
        res = _stage1_whole(gen, api.mt_seed(seed))
        assert gen.last_gen() == want, (k, w64)
        SEEN.add(want)
        _check_oracle(o, res)
        stats, tallies, state, kerns = _stage1_shards(gen, sites, gt, gr, api.mt_seed(seed), 1)
        base, kern = kerns[1]
        if base % 2 ** k:
            assert kern == ("pre_w64" if w64 else "pre_w32"), (k, w64, kern)
        else:
            assert kern == want, (k, w64, kern)
        if kern.startswith("pre"):
            pre_seen.add(kern)
        SEEN.add(kern)
        _check_oracle(o, (stats, tallies, state))
    assert pre_seen == {"pre_w32", "pre_w64"}


# ---- streams past 2^31 words -------------------------------------------------------------------------------------------
BIG_ROWS = 11_000_003        # 2.2e9 words > 2^31; the last tile is partial and its last group of 4 rows too
BIG_K = 16                   # stage i's chunk size at this many rows (pick_chunk_log2)


@pytest.fixture
def big_handle(built):
    """A handle of its own (about 10 GB of stream and 2 GB of count tiles), freed after the test."""
    h = api.Handle(0)
    yield h
    h.close()


def _big_sites(seed, rows_per_chr, chrom_len):
    """Every row passes the site filter and both genomes have a record with the row's alleles, a derived read in the
    reference and a read in the target at every row: (almost) every row is used."""
    sites = synth.make_sites(seed, rows_per_chr, chrom_len)
    sites.flipped[:] = 0
    sites.n_branch[:] = 1
    gt = synth.make_genome(seed + 100, sites, 1.0)
    gr = synth.make_genome(seed + 200, sites, 1.0)
    gr.aaf[:] = np.maximum(gr.aaf - (gr.daf == 0), 0)
    gr.daf[:] = np.maximum(gr.daf, 1)
    return sites, gt, gr


def test_streams_past_2_31_words(big_handle):
    """Streams longer than 2^31 words (k_gen_tma, and k_gen with 64-bit addressing, which run_mt_stream picks by itself at
    this size): the tiles around physical word 2^31, the first and the last tiles, the canary behind the last tile and a spread
    of tiles in between word for word, and the state after; then stage i on 11 M used rows on both paths and as two shards
    below 2^31 words each (W32, PRE), bit for bit against each other and against the oracle."""
    h = big_handle
    seed = 2024
    n_tiles = -(-BIG_ROWS // 32)
    t31 = (1 << 31) // TILE
    tiles = sorted({0, 1, t31 - 1, t31, t31 + 1, n_tiles - 2, n_tiles - 1} | {int(t) for t in np.linspace(2, n_tiles - 3, 9)})
    times = {}
    for path in ("tma", "w64"):
        h.set_option("gen_path", PATHS[path][0])
        t0 = time.time()
        for t in tiles:
            buf, after = h.mt_stream_tiled(api.mt_seed(seed), 0, 200 * BIG_ROWS, BIG_K, p0=t * TILE, n_phys=TILE)
            kern = h.last_gen()
            assert kern == ("tma" if path == "tma" else "tiled_w64")
            rows = min(32, BIG_ROWS - 32 * t)
            _check_layout(buf, ref_words(seed, t * TILE, 200 * rows), 0, 32 * t + rows, kern == "tma", lo=t * TILE)
        # behind the last tile: untouched up to one tile past the stream's end
        buf, _ = h.mt_stream_tiled(api.mt_seed(seed), 0, 200 * BIG_ROWS, BIG_K, p0=n_tiles * TILE,
                                   n_phys=200 * BIG_ROWS + TILE - n_tiles * TILE)
        assert (buf == CANARY).all()
        assert _after_ok(after, seed, 200 * BIG_ROWS)
        SEEN.add(kern)
        PAST_2_31.add(kern)
        times[path] = time.time() - t0
    # stage i at that size
    sites, gt, gr = _big_sites(seed, [5_600_000, BIG_ROWS - 5_600_000], [2.49e8, 2.43e8])
    h.set_option("gen_path", 2)
    h.load(sites, gt, gr)
    t0 = time.time()
    s1 = h.stage1(api.mt_seed(seed))
    times["stage1_tma"] = time.time() - t0
    tma = (s1.block_stats, s1.block_tallies, s1.mt_state)
    assert h.last_gen() == "tma"
    assert 200 * s1.n_used > 1 << 31 and int(s1.block_tallies[:, 1].sum()) == 100 * s1.n_used
    h.set_option("gen_path", 1)
    w64 = _stage1_whole(h, api.mt_seed(seed))
    assert h.last_gen() == "tiled_w64"
    _same_stage1(tma, w64)
    h.set_option("gen_path", 0)
    stats, tallies, state, kerns = _stage1_shards(h, sites, gt, gr, api.mt_seed(seed), 1)
    assert kerns[1][0] % (1 << 15) and kerns[1][1] == "pre_w32"
    _same_stage1(tma, (stats, tallies, state))
    t0 = time.time()
    o = _oracle(sites, gt, gr, seed)
    times["oracle_stage1"] = time.time() - t0
    assert o["n_used_total"] == s1.n_used
    _check_oracle(o, tma)
    print("past 2^31 words, wall s:", {k: round(v, 2) for k, v in times.items()})


def test_every_generator_kernel_ran():
    """The tests above reached all six generator kernels, and both the TMA and the 64-bit k_gen path past 2^31 words."""
    if not SEEN:
        pytest.skip("run with the rest of the file")
    assert SEEN == set(api.Handle.GEN_KERNELS), sorted(SEEN)
    assert PAST_2_31 == {"tma", "tiled_w64"}
