"""The candidate kernel's rank-band word filter (csrc/cds_cand.cu scan_one) drops only words that cannot match: every result with the
filter equals the result without it (CDSGPU_CAND_NOBAND=1, read at every launch) and the oracle on sampled cells.  Only the library's
resident occupancy carries the nibbles; streamed chunks and the chunked fallback run without the filter and must agree as well."""
import os

import numpy as np
import pytest

from colormipsearch_b200 import capi
from oracle import oracle as O

pytestmark = pytest.mark.gpu

W, H = 1210, 566
SEED = 0xC0FFEE


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(n_dev=1)
    yield c
    c.close()


@pytest.fixture(scope="module")
def data():
    masks = capi.synth_rgb_host(0, SEED, 0, 40, W, H)
    targets = capi.synth_rgb_host(1, SEED, 0, 24, W, H)
    return masks, targets


def both(fn):
    """fn() with the filter, then without it."""
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


def oracle_cells(masks, targets, params, scores, mirrored, n=3):
    rects = O.label_rects(W, H)
    mt, dt, tol, shift, mirror = params
    for i in range(min(n, len(masks))):
        om = O.PixelMatchMask(masks[i], mt, mirror, dt, tol, shift, rects)
        es, em, _ = O.search_dense([om], targets[:6])
        assert np.array_equal(scores[i, :6], es[0]) and np.array_equal(mirrored[i, :6], em[0]), (i, params)


@pytest.mark.parametrize("shift", [0, 2, 4])
@pytest.mark.parametrize("mirror", [True, False])
def test_dense_and_topk_equal_without_filter(ctx, data, shift, mirror):
    masks, targets = data
    params = (20, 20, 0.01, shift, mirror)
    lib = capi.Library(ctx, W, H, len(targets))
    lib.add_rgb(targets)
    ms = capi.MaskSet(ctx, W, H, *params, O.label_rects(W, H))
    ms.add_rgb(masks)
    (d_on, t_on), (d_off, t_off) = both(lambda: (ms.search_dense(lib), ms.search_topk(lib, 5, 0.0)))
    assert same(d_on, d_off) and same(t_on, t_off)
    oracle_cells(masks, targets, params, *d_on)
    ms.close()
    lib.close()


def test_wide_lists_and_reverse_search(ctx):
    fx = np.load(os.path.join(os.path.dirname(__file__), "golden", "cdsearch_fixtures.npz"))
    lm = np.stack([fx[k] for k in ("lm_BJD", "lm_GMR", "lm_VT016795", "lm_VT033614")])
    em = np.stack([fx[k] for k in ("em_12191", "em_12191_FL", "em_LPLC2")])
    params = (20, 20, 0.01, 2, True)
    for wide in (0, 1):
        ctx.set_option("wide_lists", wide)
        for masks, targets in ((em, lm), (lm, em)):
            lib = capi.Library(ctx, W, H, len(targets))
            lib.add_rgb(targets)
            ms = capi.MaskSet(ctx, W, H, *params, O.label_rects(W, H))
            ms.add_rgb(masks)
            on, off = both(lambda: ms.search_dense(lib))
            assert same(on, off), wide
            oracle_cells(masks, targets, params, *on)
            ms.close()
            lib.close()
    ctx.set_option("wide_lists", 0)


def test_rebake_and_chunked_occupancy(ctx, data):
    masks, targets = data
    lib = capi.Library(ctx, W, H, len(targets))
    lib.add_rgb(targets)
    for resident in (1, 0):
        ctx.set_option("resident_occupancy", resident)
        for dt in (20, 60, 20):            # a new data threshold re-bakes the planes and rebuilds the occupancy and its nibbles
            params = (20, dt, 0.01, 2, True)
            ms = capi.MaskSet(ctx, W, H, *params, O.label_rects(W, H))
            ms.add_rgb(masks)
            on, off = both(lambda: ms.search_dense(lib))
            assert same(on, off), (resident, dt)
            oracle_cells(masks, targets, params, *on, n=2)
            ms.close()
    ctx.set_option("resident_occupancy", 1)
    lib.close()


def test_streamed_pixel_and_tiff_searches(ctx, data):
    masks, targets = data
    params = (20, 20, 0.01, 2, True)
    ms = capi.MaskSet(ctx, W, H, *params, O.label_rects(W, H))
    ms.add_rgb(masks)
    lib = capi.Library(ctx, W, H, len(targets))
    lib.add_rgb(targets)
    ref = ms.search_topk(lib, 5, 0.0)
    files = [capi.tiff_encode_rgb(t, 8, 32773) for t in targets]
    on, off = both(lambda: (ms.search_stream(targets, 5, 0.0), ms.search_stream_tiff(files, 5, 0.0)))
    assert same(on, off)
    for got in on:
        assert same(got, ref)
    ms.close()
    lib.close()
