"""Rank-band bytes of the candidate kernel's word filter (csrc/cds_kernels.cuh, csrc/cds_cand.cu).

* The library's tile bytes equal a numpy recomputation from the code words: a byte that is missing a band would drop words that can
  match (the search tests would see it), a byte with a band too many only makes the filter weaker, which no equality test of the
  search results can see.
* Mask sets whose palette is too large for 12-row bands (cds_debug_cand_config) and a palette of a single colour class (staged as 16
  entries, the idle one last at index 15) give the oracle's results, with and without the filter."""
import os

import numpy as np
import pytest

from colormipsearch_b200 import capi
from oracle import oracle as O

pytestmark = pytest.mark.gpu

W, H = 1210, 566
SEED = 0xC0FFEE
NUM_RANKS, SECTOR_STRIDE, NUM_SECTORS, BANDS = 19820, 32768, 6, 8


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(n_dev=1)
    yield c
    c.close()


def classes(ctx, rgb, threshold):
    """(sector, rank) of every pixel as the device encodes it; sector -1 for pixels at or below the threshold or without a sector."""
    codes = ctx.debug_encode_colors(rgb.reshape(-1, 3), threshold).reshape(rgb.shape[:-1])
    sr = (codes >> 8) & 0x3FFFF
    valid = ((codes & 0xC0000000) == 0) & (sr < NUM_SECTORS * SECTOR_STRIDE)
    return np.where(valid, sr // SECTOR_STRIDE, -1).astype(np.int64), (sr % SECTOR_STRIDE).astype(np.int64)


def expected_bands(ctx, targets, threshold, S):
    """uint8 [n][tile rows][6 * tp]: bit b of byte [t][ty][sector * tp + tx] = a pixel of that sector above the threshold, inside the
    image and in [8 tx - S, 8 tx + 7 + S] x [4 ty - S, 4 ty + 3 + S], has rank band b."""
    n, h, w = targets.shape[:3]
    tp = ((w + 7) // 8 + 3) // 4 * 4
    ht = (h + 3) // 4
    sec, rank = classes(ctx, targets, threshold)
    bits = np.where(sec >= 0, np.left_shift(np.uint64(1), (np.maximum(sec, 0) * BANDS + rank * BANDS // NUM_RANKS).astype(np.uint64)),
                    np.uint64(0)).astype(np.uint64)
    pad = np.zeros((n, ht * 4 + 2 * S, tp * 8 + 2 * S), np.uint64)     # zeros outside the image
    pad[:, S:S + h, S:S + w] = bits
    for axis in (1, 2):                                               # OR over the (2 S + 1)-wide box, axis by axis
        pad = _box_or(pad, S, axis)
    core = pad[:, S:S + ht * 4, S:S + tp * 8]
    tiles = np.bitwise_or.reduce(np.bitwise_or.reduce(core.reshape(n, ht, 4, tp, 8), axis=4), axis=2)    # [n][ht][tp]
    out = np.zeros((n, ht, NUM_SECTORS * tp), np.uint8)
    for s in range(NUM_SECTORS):
        out[:, :, s * tp:(s + 1) * tp] = ((tiles >> np.uint64(BANDS * s)) & np.uint64(0xFF)).astype(np.uint8)
    return out


def _box_or(a, S, axis):
    out = a.copy()
    L = a.shape[axis]
    for d in range(1, S + 1):
        lo = [slice(None)] * a.ndim
        hi = [slice(None)] * a.ndim
        lo[axis], hi[axis] = slice(0, L - d), slice(d, L)
        out[tuple(hi)] |= a[tuple(lo)]
        out[tuple(lo)] |= a[tuple(hi)]
    return out


def test_library_band_bytes_match_numpy(ctx):
    h = 565                                                            # the last tile row holds a single image row
    targets = capi.synth_rgb_host(1, SEED, 0, 4, W, h)
    lib = capi.Library(ctx, W, h, len(targets))
    lib.add_rgb(targets)
    for dt in (20, 60, 20):                                            # a new data threshold re-bakes the planes and rebuilds the bytes
        for S in (0, 2, 4):
            got = lib.debug_bands(dt, S)
            want = expected_bands(ctx, targets, dt, S)
            assert got.shape == want.shape
            assert np.array_equal(got, want), (dt, S, int(np.count_nonzero(got != want)))
            # the bytes are neither empty nor saturated: the filter has something to drop
            nz = want[want != 0]
            assert nz.size > 0 and np.count_nonzero(nz != 0xFF) > 0
    lib.close()


def both(fn):
    os.environ.pop("CDSGPU_CAND_NOBAND", None)
    on = fn()
    os.environ["CDSGPU_CAND_NOBAND"] = "1"
    try:
        off = fn()
    finally:
        os.environ.pop("CDSGPU_CAND_NOBAND", None)
    return on, off


def same(a, b):
    if isinstance(a, (tuple, list)):
        return len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    return np.array_equal(np.asarray(a), np.asarray(b))


def class_index(ctx, rgb):
    """colour class of every pixel, sector * ranks + rank; -1 without a sector"""
    sec, rank = classes(ctx, rgb, 0)
    return np.where(sec >= 0, sec * NUM_RANKS + rank, -1)


def palette_classes(ctx, masks, threshold, with_none=True):
    """number of distinct colour classes of the masks' pixels above the threshold, with or without the 'no sector' class"""
    cls = np.unique(class_index(ctx, masks)[masks.max(-1) > threshold])
    return len(cls) if with_none else int(np.count_nonzero(cls >= 0))


def check_search(ctx, masks, targets, params):
    lib = capi.Library(ctx, W, H, len(targets))
    lib.add_rgb(targets)
    ms = capi.MaskSet(ctx, W, H, *params, [])
    ms.add_rgb(masks)
    (d_on, t_on), (d_off, t_off) = both(lambda: (ms.search_dense(lib), ms.search_topk(lib, 5, 0.0)))
    assert ctx.last_stats()["match_kernel"] == 1                       # the candidate kernel ran
    assert same(d_on, d_off) and same(t_on, t_off)
    mt, dt, tol, shift, mirror = params
    scores, mirrored = d_on
    assert scores.any()
    for i in range(3):
        om = O.PixelMatchMask(masks[i], mt, mirror, dt, tol, shift, np.zeros((0, 4), np.int32))
        es, em, _ = O.search_dense([om], targets)
        assert np.array_equal(scores[i], es[0]) and np.array_equal(mirrored[i], em[0]), i
    ms.close()
    lib.close()


def test_palette_above_twelve_row_limit(ctx):
    masks = capi.synth_rgb_host(0, SEED, 0, 20, W, H)
    targets = capi.synth_rgb_host(1, SEED, 0, 6, W, H)
    # colours of classes the masks do not have, painted over lit mask pixels until the group has ~1,990 classes
    rng = np.random.default_rng(22)
    pool = rng.integers(0, 256, (400000, 3), dtype=np.uint8)
    pool = pool[pool.max(1) > 40]
    cls = class_index(ctx, pool)
    have = set(np.unique(class_index(ctx, masks)[masks.max(-1) > 20]).tolist())
    _, first = np.unique(cls, return_index=True)
    new = [i for i in first if cls[i] >= 0 and int(cls[i]) not in have][:1990 - len(have)]
    colours = pool[new]
    k = 0
    for m in masks:
        ys, xs = np.nonzero(m.max(-1) > 20)
        pick = rng.choice(len(ys), size=min(len(ys), (len(colours) + len(masks) - 1) // len(masks)), replace=False)
        for j in pick:
            m[ys[j], xs[j]] = colours[k % len(colours)]
            k += 1
    # the group's palette has between n_lo (sector classes) and n_hi (the 'no sector' class too) entries, whichever way it is counted
    n_lo, n_hi = palette_classes(ctx, masks, 20, with_none=False), palette_classes(ctx, masks, 20)
    limit = 1936                                                      # palette + idle entry with 12-row bands at xyShift 2 (DESIGN.md §4.1)
    assert limit <= n_lo and n_hi < 2048, (n_lo, n_hi)                # above the limit, below a WIDE list
    assert capi.cand_config(W, H, 2, n_lo + 1)[:3] == (31, 8, 2)      # so the launch runs 8-row bands
    check_search(ctx, masks, targets, (20, 20, 0.01, 2, True))


@pytest.mark.parametrize("shift", [0, 2])
def test_palette_of_one_class(ctx, shift):
    masks = capi.synth_rgb_host(0, SEED, 0, 20, W, H)
    targets = capi.synth_rgb_host(1, SEED, 0, 6, W, H)
    # one colour over every lit mask pixel, and over the lit pixels of mask t in target t, so that there is something to match
    colour = np.array([200, 90, 30], np.uint8)
    lit = masks.max(-1) > 20
    masks[lit] = colour
    for t in range(len(targets)):
        targets[t][lit[t]] = colour
    assert palette_classes(ctx, masks, 20) == 1
    check_search(ctx, masks, targets, (20, 20, 0.01, shift, True))
