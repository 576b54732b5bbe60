"""Mask sets across palette-group (1,024 masks), mask-chunk and 32,768-mask boundaries, against the oracle on every cell.

Masks and targets are built from small pools of distinct images: mask i = mask pool[(A i) mod P], target t = target pool[(C t) mod Q]
with P and Q prime, so the expected score of every cell is E[(A i) mod P, (C t) mod Q], E being the oracle's pool-by-pool matrix.  The rows
of E are pairwise distinct and so are its columns, and no shift of a mask index by 1, 1,024, 32,768 or a chunk size (nor of a target
index by 1 or a stream chunk) lands on the same pool image: a search that reads or writes the wrong mask or target changes a value.

What each case reaches is asserted from the search's statistics (`match_kernel`, `match_kernel_launches`, `chunked`), computed from the
chunk formulas of cds_search_dense / cds_search_topk (csrc/cds_api.cu), so that a change to them cannot quietly leave a case testing
something else."""
import os

import numpy as np
import pytest

from colormipsearch_b200 import capi
from oracle import oracle as O

pytestmark = pytest.mark.gpu

GROUP = 1024                       # CDS_PALETTE_GROUP
SLICE = 32768                      # masks per grid-y slice of the host loops
DENSE_BUDGET = 64 << 20            # score words per device and mask chunk, cds_search_dense
TOPK_BUDGET = 512 << 20            # the same for cds_search_topk
KERNEL = {"cand": 1, "band": 2, "gather": 3}
NUM_RANKS, SECTOR_STRIDE, NUM_SECTORS = 19820, 32768, 6

W, H = 40, 20                      # pool images
P, Q = 251, 257                    # mask / target pool sizes (primes)
A, C = 3, 5                        # index multipliers
PARAMS = (20, 20, 0.02, 2, True)   # mask threshold, data threshold, zTolerance, xyShift, mirror


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(n_dev=1)
    yield c
    c.close()


def mask_chunk(M, T, budget):
    """the mask chunk of a search over T targets on one device (cds_search_dense / cds_search_topk)"""
    mc = max(1, min(M, budget // max(T, 1)))
    if mc < M and mc > GROUP:
        mc -= mc % GROUP
    return mc


def chunk_kernels(M, mc, kernel="cand"):
    """(launches, kernel of the last chunk): a chunk that starts inside a palette group runs on the gather kernel"""
    starts = range(0, M, mc)
    last = kernel if starts[-1] % GROUP == 0 else "gather"
    return len(starts), KERNEL[last]


def oracle_mask(rgb):
    mthr, dthr, ztol, shift, mirror = PARAMS
    return O.PixelMatchMask(rgb, mthr, mirror, dthr, ztol, shift, np.zeros((0, 4), np.int32))


def is_prime(n):
    return n > 1 and all(n % d for d in range(2, int(n ** 0.5) + 1))


def rand_img(rng, w, h, density, lut, colours=None):
    img = np.zeros((h, w, 3), np.uint8)
    sel = rng.random((h, w)) < density
    if colours is None:
        col = (lut[rng.integers(0, 256, (h, w))].astype(np.int64) * rng.integers(20, 256, (h, w, 1)) // 255).astype(np.uint8)
    else:
        col = colours[rng.integers(0, len(colours), (h, w))]
    img[sel] = col[sel]
    return img


def embed(rng, target, mask, frac):
    lit = mask.max(-1) > 20
    take = lit & (rng.random(lit.shape) < frac)
    target[take] = mask[take]


def classes(ctx, rgb):
    """colour class of every pixel, sector * ranks + rank; -1 without a sector"""
    codes = ctx.debug_encode_colors(rgb.reshape(-1, 3), 0).reshape(rgb.shape[:-1])
    sr = (codes >> 8) & 0x3FFFF
    valid = ((codes & 0xC0000000) == 0) & (sr < NUM_SECTORS * SECTOR_STRIDE)
    return np.where(valid, (sr // SECTOR_STRIDE) * NUM_RANKS + sr % SECTOR_STRIDE, -1).astype(np.int64)


def group_classes(ctx, imgs):
    """(sector classes, classes incl. 'no sector') of the lit mask pixels of a group's distinct images: its palette lies in between"""
    cls = np.unique(classes(ctx, imgs)[imgs.max(-1) > PARAMS[0]])
    return int(np.count_nonzero(cls >= 0)), len(cls)


@pytest.fixture(scope="module")
def pools(ctx):
    """(mask pool [P], target pool [Q], E scores [P][Q], E mirrored [P][Q], mask sizes [P])"""
    assert is_prime(P) and is_prime(Q)
    rng = np.random.default_rng(1024)
    lut = O.lut().astype(np.uint8)
    masks = np.stack([rand_img(rng, W, H, 0.2, None, lut) for _ in range(P)])
    # every group holds every pool mask, so every group's palette is the pool's: a staged palette, not a WIDE list
    assert group_classes(ctx, masks)[1] < 2048
    targets = np.stack([rand_img(rng, W, H, 0.35, lut) for _ in range(Q)])
    for q in range(Q):                                # real matches: parts of two pool masks in every target
        embed(rng, targets[q], masks[q % P], rng.uniform(0.3, 1.0))
        embed(rng, targets[q], masks[(7 * q + 3) % Q % P][:, ::-1], rng.uniform(0.3, 1.0))    # mirrored
    oms = [oracle_mask(m) for m in masks]
    es, em, _ = O.search_dense(oms, targets)
    sizes = np.array([m.size for m in oms], np.int32)
    # a mix-up of masks or of targets changes a value
    assert np.unique(es, axis=0).shape[0] == P and np.unique(es, axis=1).shape[1] == Q
    assert es.max() > 50 and em.any()
    # no index shift the searches work with maps a mask or a target onto the same pool image
    for d in (1, GROUP, SLICE, 256):
        assert (A * d) % P != 0 and (C * d) % Q != 0
    return masks, targets, es, em, sizes


def mask_index(M):
    return (A * np.arange(M, dtype=np.int64)) % P


def target_index(T):
    return (C * np.arange(T, dtype=np.int64)) % Q


def build_maskset(ctx, pools, M, block=4096):
    masks, _, _, _, sizes = pools
    ms = capi.MaskSet(ctx, W, H, *PARAMS, [])
    pm = mask_index(M)
    for i0 in range(0, M, block):
        got = ms.add_rgb(masks[pm[i0:i0 + block]])
        assert np.array_equal(got, sizes[pm[i0:i0 + block]]), i0
    assert len(ms) == M
    return ms


def build_library(ctx, pools, T, block=Q * 64):
    targets = pools[1]
    lib = capi.Library(ctx, W, H, T)
    pt = target_index(T)
    for t0 in range(0, T, block):
        assert lib.add_rgb(targets[pt[t0:t0 + block]]) == t0
    assert len(lib) == T
    return lib


def host_targets(pools, T):
    return pools[1][target_index(T)]


def check_dense(pools, M, T, got):
    _, _, es, em, _ = pools
    pm, pt = mask_index(M), target_index(T)
    scores, mirrored = got
    exp_s = es[pm[:, None], pt[None, :]]
    bad = np.argwhere(scores != exp_s)
    assert bad.size == 0, ("scores", M, T, len(bad), bad[:5].tolist())
    exp_m = em[pm[:, None], pt[None, :]]
    bad = np.argwhere(mirrored != exp_m)
    assert bad.size == 0, ("mirrored", M, T, len(bad), bad[:5].tolist())


def match_table(pools, pct):
    """[P][Q] bool: O.is_match of every pool pair"""
    _, _, es, _, sizes = pools
    ok = np.zeros(es.shape, bool)
    for p in range(P):
        for q in np.nonzero(es[p] > 0)[0]:
            ok[p, q] = O.is_match(int(es[p, q]), es[p, q] / sizes[p], pct)
    return ok


def expected_topk(pools, T, k, pct):
    """per mask pool image: (targets, scores, mirrored) of the reference's list -- every isMatch target, descending score, ties by
    ascending index, the first k"""
    _, _, es, em, _ = pools
    ok = match_table(pools, pct)
    pt = target_index(T)
    out = []
    for p in range(P):
        s = np.where(ok[p], es[p], -1)[pt]
        n = int(np.count_nonzero(s >= 0))
        if n > k:
            kth = np.partition(s, len(s) - k)[len(s) - k]
            cand = np.nonzero(s >= kth)[0]
        else:
            cand = np.nonzero(s >= 0)[0]
        cand = cand[np.lexsort((cand, -s[cand]))][:k]
        out.append((cand, s[cand], em[p][pt[cand]]))
    return out


def check_topk(pools, M, T, k, pct, got, exp=None):
    score, target, mirrored, count = got
    exp = exp if exp is not None else expected_topk(pools, T, k, pct)
    pm = mask_index(M)
    n = np.array([len(e[0]) for e in exp])[pm]
    assert np.array_equal(count, n), (M, T, k, pct, np.nonzero(count != n)[0][:5].tolist())
    et = np.full((P, k), -1, np.int64)
    esc = np.zeros((P, k), np.int32)
    emi = np.zeros((P, k), np.uint8)
    for p, (t, s, m) in enumerate(exp):
        et[p, :len(t)], esc[p, :len(t)], emi[p, :len(t)] = t, s, m
    valid = np.arange(k)[None, :] < count[:, None]
    for name, g, e in (("target", target, et), ("score", score, esc), ("mirrored", mirrored, emi)):
        bad = np.argwhere((g != e[pm]) & valid)
        assert bad.size == 0, (name, M, T, k, pct, len(bad), bad[:5].tolist())


def expected_matches(pools, M, T, pct):
    """every (mask, target, score, mirrored) passing isMatch, by mask, descending score, ascending target"""
    _, _, es, em, _ = pools
    ok = match_table(pools, pct)
    pm, pt = mask_index(M), target_index(T)
    mi, ti = np.nonzero(ok[pm[:, None], pt[None, :]])
    s = es[pm[mi], pt[ti]]
    order = np.lexsort((ti, -s, mi))
    return mi[order], ti[order], s[order], em[pm[mi], pt[ti]][order]


def check_matches(exp, got):
    assert len(got[0]) == len(exp[0]), (len(got[0]), len(exp[0]))
    for name, g, e in zip(("mask", "target", "score", "mirrored"), got, exp):
        assert np.array_equal(g, e), (name, int(np.count_nonzero(g != e)))


def both_filters(fn, noband):
    if noband:
        os.environ["CDSGPU_CAND_NOBAND"] = "1"
    try:
        return fn()
    finally:
        os.environ.pop("CDSGPU_CAND_NOBAND", None)


# ---------------------------------------------------------------------------------------------------------- 1. group edges, every kernel

@pytest.mark.parametrize("M", [1023, 1024, 1025, 2049])
def test_group_edges_every_kernel(ctx, pools, M):
    T = 300
    ms = build_maskset(ctx, pools, M, block=1000)
    lib = build_library(ctx, pools, T)
    targets = host_targets(pools, T)
    topk_exp = {(k, pct): expected_topk(pools, T, k, pct) for k in (5, 300) for pct in (0.0, 1.0)}
    match_exp = {pct: expected_matches(pools, M, T, pct) for pct in (0.0, 1.0)}
    try:
        for kern in ("cand", "band", "gather"):
            ctx.set_match_kernel(kern)
            for resident in (1, 0):
                ctx.set_option("resident_occupancy", resident)
                for noband in ((0, 1) if kern == "cand" else (0,)):
                    what = (M, kern, resident, noband)
                    got = both_filters(lambda: ms.search_dense(lib), noband)
                    st = ctx.last_stats()
                    assert (st["match_kernel"], st["match_kernel_launches"]) == (KERNEL[kern], 1), (what, st)
                    check_dense(pools, M, T, got)
                    for (k, pct), exp in topk_exp.items():
                        got = both_filters(lambda: ms.search_topk(lib, k, pct), noband)
                        st = ctx.last_stats()
                        assert st["match_kernel"] == KERNEL[kern] and st["chunked"] == 1 - resident, (what, k, pct, st)
                        check_topk(pools, M, T, k, pct, got, exp)
                    for pct, exp in match_exp.items():
                        got = both_filters(lambda: ms.search_matches(lib, pct), noband)
                        assert ctx.last_stats()["match_kernel"] == KERNEL[kern], what
                        check_matches(exp, got)
        ctx.set_match_kernel("auto")
        ctx.set_option("stream_chunk", 128)           # streamed targets: chunk boundaries inside the target pool's period
        check_matches(match_exp[1.0], ms.search_stream_matches(targets, 1.0))
        assert ctx.last_stats()["match_kernel"] == 1
    finally:
        ctx.set_match_kernel("auto")
        ctx.set_option("resident_occupancy", 1)
        ctx.set_option("stream_chunk", 256)
    ms.close()
    lib.close()


# -------------------------------------------------------------------------------------------------- 2. different palettes in one launch

PW, PH = 1210, 64          # at this width the palette size sets the band height, as at 1210 x 566 (asserted below)


def distinct_class_colours(ctx, rng, n):
    """n colours of n different colour classes, all with a sector and above the thresholds"""
    pool = rng.integers(0, 256, (400000, 3), dtype=np.uint8)
    pool = pool[pool.max(1) > 40]
    cls = classes(ctx, pool)
    _, first = np.unique(cls, return_index=True)
    first = first[cls[first] >= 0]
    assert len(first) >= n
    return pool[rng.permutation(first)[:n]]


def palette_rows(pal_entries, wide=False):
    return capi.cand_config(PW, PH, PARAMS[3], pal_entries, wide)[1]


@pytest.fixture(scope="module")
def palette_images(ctx):
    """distinct images of four kinds of groups at PW x PH: 'large' (above the 12-row palette limit, below a WIDE list), 'wide' (2,048
    classes or more), 'one' (one colour class), 'plain' (an ordinary palette); and targets holding parts of all of them"""
    rng = np.random.default_rng(1935)
    lut = O.lut().astype(np.uint8)
    limit = next(p for p in range(2, 2049) if palette_rows(p) < palette_rows(2))     # smallest staged palette with lower bands
    kinds = {}
    for name, n_colours in (("large", limit + 60), ("wide", 2200)):
        colours = distinct_class_colours(ctx, rng, n_colours)
        kinds[name] = np.stack([rand_img(rng, PW, PH, 0.1, None, colours[j::4]) for j in range(4)])
    one = np.array([[200, 90, 30]], np.uint8)
    kinds["one"] = np.stack([rand_img(rng, PW, PH, 0.1, None, one) for _ in range(2)])
    kinds["plain"] = np.stack([rand_img(rng, PW, PH, 0.1, None, lut[::2]) for _ in range(3)])
    n = {name: group_classes(ctx, imgs) for name, imgs in kinds.items()}
    assert limit - 1 <= n["large"][0] and n["large"][1] < 2048, (limit, n)
    assert n["wide"][0] >= 2048 and n["one"][1] == 1 and n["plain"][1] <= 256, n
    # the large group's palette lowers the launch's band height; the others' would not
    assert palette_rows(n["large"][0] + 1) < palette_rows(max(n["one"][1], n["plain"][1]) + 1) == palette_rows(2)
    names = list(kinds)
    first = {}
    imgs = []
    for name in names:
        first[name] = len(imgs)
        imgs += list(kinds[name])
    imgs = np.stack(imgs)
    # more targets than CTAs per group: every CTA moves from group to group and restages the palette
    targets = np.stack([rand_img(rng, PW, PH, 0.2, lut) for _ in range(300)])
    for t in range(len(targets)):
        for j in (t, t + 8, t + 3):
            embed(rng, targets[t], imgs[j % len(imgs)], 0.6)
    oms = [oracle_mask(m) for m in imgs]
    es, em, _ = O.search_dense(oms, targets)
    assert len(np.unique(es, axis=0)) == len(imgs) and es.max() > 100
    count = {name: len(kinds[name]) for name in names}
    return imgs, first, count, targets, es, em, np.array([m.size for m in oms], np.int32)


@pytest.mark.parametrize("layout", [
    (("large", 1024), ("one", 1024), ("plain", 1024), ("plain", 300)),       # a large palette followed by small ones, a short last group
    (("plain", 1024), ("one", 1024), ("large", 777)),                        # a large palette last (and short)
    (("wide", 1024), ("plain", 1024), ("one", 200)),                         # one group makes the whole set WIDE
    (("one", 1024), ("plain", 1024), ("wide", 500)),
], ids=["large_first", "large_last", "wide_first", "wide_last"])
def test_different_palettes_in_one_launch(ctx, palette_images, layout):
    imgs, first, count, targets, es, em, img_sizes = palette_images
    ids = np.concatenate([first[name] + np.arange(n) % count[name] for name, n in layout])
    M = len(ids)
    lib = capi.Library(ctx, PW, PH, len(targets))
    lib.add_rgb(targets)
    ms = capi.MaskSet(ctx, PW, PH, *PARAMS, [])
    sizes = np.concatenate([ms.add_rgb(imgs[ids[i0:i0 + 256]]) for i0 in range(0, M, 256)])
    assert np.array_equal(sizes, img_sizes[ids])
    for noband in (0, 1):
        scores, mirrored = both_filters(lambda: ms.search_dense(lib), noband)
        st = ctx.last_stats()
        assert (st["match_kernel"], st["match_kernel_launches"]) == (1, 1), st
        bad = np.argwhere((scores != es[ids]) | (mirrored != em[ids]))
        assert bad.size == 0, (noband, len(bad), bad[:5].tolist())
        got = both_filters(lambda: ms.search_topk(lib, 5, 1.0), noband)
        for i in sorted({0, M - 1} | {g * GROUP + d for g in range(1, (M - 1) // GROUP + 1) for d in (-2, -1, 0, 1)} | set(range(0, M, 97))):
            exp = [t for t in np.lexsort((np.arange(len(targets)), -es[ids[i]]))
                   if O.is_match(int(es[ids[i], t]), es[ids[i], t] / sizes[i], 1.0)][:5]
            c = int(got[3][i])
            assert got[1][i, :c].tolist() == exp and got[0][i, :c].tolist() == es[ids[i], exp].tolist(), (noband, i)
    ms.close()
    lib.close()


# -------------------------------------------------------------------------------------------------------------------- 3. dense mask chunks

@pytest.mark.parametrize("M,T", [(2100, 40000), (1100, 68000)], ids=["aligned", "mid_group"])
def test_dense_mask_chunks(ctx, pools, M, T):
    mc = mask_chunk(M, T, DENSE_BUDGET)
    if M == 2100:
        assert DENSE_BUDGET // T > GROUP and mc == GROUP and M % mc == 52        # rounded to a group; a 52-mask partial group last
    else:
        assert mc < GROUP and mc < M                                            # a chunk ends inside group 0: the rest runs on gather
    ms = build_maskset(ctx, pools, M, block=700)
    lib = build_library(ctx, pools, T)
    got = ms.search_dense(lib)
    st = ctx.last_stats()
    assert (st["match_kernel_launches"], st["match_kernel"]) == chunk_kernels(M, mc), st
    check_dense(pools, M, T, got)
    ms.close()
    lib.close()


# -------------------------------------------------------------------------------------------------------------------- 4. top-K mask chunks

@pytest.mark.parametrize("M,T", [(2100, 300000), (1100, 600000)], ids=["aligned", "mid_group"])
def test_topk_mask_chunks(ctx, pools, M, T):
    K, pct = 300, 1.0
    mc = mask_chunk(M, T, TOPK_BUDGET)
    if M == 2100:
        assert TOPK_BUDGET // T > GROUP and mc == GROUP and M % mc == 52
    else:
        assert mc < GROUP and mc < M
    ms = build_maskset(ctx, pools, M, block=700)
    lib = build_library(ctx, pools, T)
    got = ms.search_topk(lib, K, pct)
    st = ctx.last_stats()
    assert (st["match_kernel_launches"], st["match_kernel"], st["chunked"]) == chunk_kernels(M, mc) + (0,), st
    check_topk(pools, M, T, K, pct, got)
    ms.close()
    lib.close()


# ----------------------------------------------------------------------------------------------------------- 5. more than 32,768 masks

@pytest.mark.parametrize("M,block", [(SLICE + 1, SLICE + 1), (33000, 4093)], ids=["one_call", "blocks"])
def test_more_than_32768_masks(ctx, pools, M, block):
    T, K, pct = 300, 20, 5.0                                  # (fewer random pairs pass: ~3 M listed matches)
    ms = build_maskset(ctx, pools, M, block=block)            # checks the sizes add_rgb returns against the oracle's
    assert np.array_equal(ms.sizes(), pools[4][mask_index(M)])
    lib = build_library(ctx, pools, T)
    try:
        for kern in ("cand", "gather"):
            ctx.set_match_kernel(kern)
            got = ms.search_dense(lib)
            st = ctx.last_stats()
            launches = 1 if kern == "cand" else (M + SLICE - 1) // SLICE
            assert (st["match_kernel"], st["match_kernel_launches"]) == (KERNEL[kern], launches), st
            check_dense(pools, M, T, got)
    finally:
        ctx.set_match_kernel("auto")
    got = ms.search_topk(lib, K, pct)
    assert ctx.last_stats()["match_kernel"] == 1
    check_topk(pools, M, T, K, pct, got)
    exp = expected_matches(pools, M, T, pct)
    check_matches(exp, ms.search_matches(lib, pct))
    assert ctx.last_stats()["match_kernel"] == 1
    targets = host_targets(pools, T)
    check_matches(exp, ms.search_stream_matches(targets, pct))
    n = len(exp[0])
    with pytest.raises(capi.CdsError) as e:
        ms.search_stream_matches(targets, pct, capacity=n - 1)
    assert e.value.status == capi.CDS_ERR_CAPACITY and str(n) in e.value.message
    ms.close()
    lib.close()
