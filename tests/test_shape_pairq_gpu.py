"""GPU tests of the shape score's single-pair queue (cds_shape_pairq_*): every pair it scores equals what the batched call
cds_shape_score_pairs returns for the same pair, whatever the threads, batch sizes, cache size and keys."""
import threading

import numpy as np
import pytest

from colormipsearch_b200 import capi
from oracle import oracle as O
from tests import golden_vectors as GV

pytestmark = pytest.mark.gpu

W, H = 1210, 566
SMALL = (333, 151)          # odd width: unaligned slice-plane rows, a partly filled last bitmap word


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(n_dev=1)
    yield c
    c.close()


def _rects(w, h):
    return O.label_rects(W, H) if (w, h) == (W, H) else np.array([[0, 0, 40, 12], [w - 17, h - 9, w, h]], np.int32)


def _roi(w, h):
    roi = np.zeros((h, w, 3), np.uint8)
    roi[h // 5: h - 3, w // 7: w - w // 9] = 255          # asymmetric: the ROI is not mirrored with the query
    return roi


def _data(ctx, size, n_masks, n_targets, seed):
    """synthetic EM masks and LM targets (with gradients and zgap images made on the device) at full size; sparse random images at others"""
    w, h = size
    if size == (W, H):
        masks = capi.synth_rgb_host(0, seed, 0, n_masks, W, H)
        targets = capi.synth_rgb_host(1, seed, 0, n_targets, W, H)
        grads = capi.synth_gradient_host(seed, 0, n_targets, W, H)
    else:
        rng = np.random.default_rng(seed)

        def sparse(n):
            img = np.zeros((h, w, 3), np.uint8)
            img.reshape(-1, 3)[rng.integers(0, h * w, n)] = rng.integers(1, 256, (n, 3))
            img[0, :5] = 200; img[-1, -5:] = 90
            return img

        masks = np.stack([sparse(300 + 100 * i) for i in range(n_masks)])
        targets = np.stack([sparse(2000 + 300 * i) for i in range(n_targets)])
        grads = rng.integers(0, 700, (n_targets, h, w)).astype(np.uint16)
    zgaps = ctx.make_zgap(targets, 20, 10, _rects(w, h))
    return masks, targets, grads, zgaps


def _pairs(n_masks, n_targets, seed, n=None):
    if n is None:
        pm = np.repeat(np.arange(n_masks), n_targets)
        pt = np.tile(np.arange(n_targets), n_masks)
    else:
        rng = np.random.default_rng(seed)
        pm, pt = rng.integers(0, n_masks, n), rng.integers(0, n_targets, n)
    return pm.astype(np.int32), pt.astype(np.int64)


def _same(a, b):
    return all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(a, b))


@pytest.mark.parametrize("size", [(W, H), SMALL], ids=["full", "odd"])
def test_queue_equals_batched_call(ctx, size):
    """zgap given and derived, mirror on and off, label rectangles and an ROI, 1 / 8 / 40 native threads, max_batch 1 / 7 / 64,
    keys and key 0."""
    w, h = size
    n_masks, n_targets = 4, 10
    masks, targets, grads, zgaps = _data(ctx, size, n_masks, n_targets, 11)
    pm, pt = _pairs(n_masks, n_targets, 0)
    keys = np.arange(1, n_targets + 1, dtype=np.uint64) * 7919
    for mirror in (True, False):
        sms = capi.ShapeMaskSet(ctx, w, h, 20, mirror, _rects(w, h), roi=_roi(w, h))
        sms.add_rgb(masks)
        for zg in (zgaps, None):
            ref = sms.score_pairs(targets, grads, zg, pm, pt)
            assert (ref[0] > 0).any()
            for threads in (1, 8, 40):
                for max_batch in (1, 7, 64):
                    q = capi.ShapePairQueue(ctx, sms, max_batch=max_batch)
                    k = None if (threads, max_batch) == (8, 7) else keys
                    got = q.drive(targets, grads, zg, k, pm, pt, threads)
                    assert _same(got[:3], ref), (size, mirror, zg is not None, threads, max_batch)
                    q.close()
        sms.close()


def test_batches_of_more_than_one_launch(ctx):
    """Batches of up to 512 requests: several launches of 128 pairs share the accumulators in stream order."""
    w, h = SMALL
    masks, targets, grads, zgaps = _data(ctx, SMALL, 3, 4, 12)
    pm, pt = _pairs(3, 4, 3, n=1500)
    sms = capi.ShapeMaskSet(ctx, w, h, 20, True, _rects(w, h))
    sms.add_rgb(masks)
    ref = sms.score_pairs(targets, grads, zgaps, pm, pt)
    q = capi.ShapePairQueue(ctx, sms, max_batch=512, max_wait_us=2000)
    keys = np.arange(1, 5, dtype=np.uint64) * 720720          # multiples of every queue count up to 16: all requests meet in one queue
    got = q.drive(targets, grads, zgaps, keys, pm, pt, 300)
    assert _same(got[:3], ref)
    st = q.stats()
    assert st["requests"] == 1500 and st["uploads"] == 4
    q.close()
    sms.close()


def test_cache_smaller_than_the_targets(ctx):
    """max_batch 1 and cache_targets 1: two slots per queue for 24 targets, so slots are taken over while other callers wait."""
    w, h = SMALL
    masks, targets, grads, zgaps = _data(ctx, SMALL, 3, 24, 13)
    pm, pt = _pairs(3, 24, 4, n=400)
    sms = capi.ShapeMaskSet(ctx, w, h, 20, True, _rects(w, h), roi=_roi(w, h))
    sms.add_rgb(masks)
    keys = np.arange(1, 25, dtype=np.uint64)
    for zg in (zgaps, None):
        ref = sms.score_pairs(targets, grads, zg, pm, pt)
        q = capi.ShapePairQueue(ctx, sms, max_batch=1, cache_targets=1)
        for threads in (1, 8):
            got = q.drive(targets, grads, zg, keys, pm, pt, threads)
            assert _same(got[:3], ref), (zg is not None, threads)
        assert q.stats()["uploads"] > 24           # targets were evicted and uploaded again
        q.close()
    sms.close()


def test_golden_vectors_through_the_queue(ctx, fixtures):
    rects = O.label_rects(W, H)
    sms = capi.ShapeMaskSet(ctx, W, H, 20, True, rects)
    mask_keys = ["em_12191", "em_12191_FL"]
    sms.add_rgb(np.stack([fixtures[k] for k in mask_keys]))
    q = capi.ShapePairQueue(ctx, sms, max_batch=8)
    for i, c in enumerate(GV.SHAPE):
        zg = None if c[3] is None else fixtures[c[3]]
        # the key names the (target, gradient, zgap) combination: the mismatched-gradient case must not reuse a cached slot
        key = 1 + GV.SHAPE.index(next(d for d in GV.SHAPE if d[1:4] == c[1:4]))
        gap, he, mir = q.score(mask_keys.index(c[0]), fixtures[c[1]], fixtures[c[2]], zg, key=key)
        assert (gap, he, mir) == (c[4], c[5], c[7]), c
        assert capi.shape_score_2d(gap, he) == c[6]
    q.close()
    sms.close()


def test_masks_added_after_the_queue(ctx):
    w, h = SMALL
    masks, targets, grads, zgaps = _data(ctx, SMALL, 6, 8, 14)
    sms = capi.ShapeMaskSet(ctx, w, h, 20, True, _rects(w, h))
    sms.add_rgb(masks[:2])
    q = capi.ShapePairQueue(ctx, sms, max_batch=16)
    keys = np.arange(100, 108, dtype=np.uint64)
    pm, pt = _pairs(2, 8, 5, n=64)
    assert _same(q.drive(targets, grads, None, keys, pm, pt, 8)[:3], sms.score_pairs(targets, grads, None, pm, pt))
    sms.add_rgb(masks[2:])
    pm, pt = _pairs(6, 8, 6, n=300)
    got = q.drive(targets, grads, None, keys, pm, pt, 8)
    assert _same(got[:3], sms.score_pairs(targets, grads, None, pm, pt))
    q.close()
    sms.close()


def test_batched_calls_while_the_queue_runs(ctx):
    """Batched calls on the same mask set -- which reallocate its device descriptors once it outgrows them -- and masks added to it
    while the queue scores from 40 threads."""
    w, h = SMALL
    masks, targets, grads, zgaps = _data(ctx, SMALL, 2, 8, 15)
    extra = np.concatenate([_data(ctx, SMALL, 5, 1, 100 + i)[0] for i in range(16)])     # 80 more masks: past the 64 descriptors
    sms = capi.ShapeMaskSet(ctx, w, h, 20, True, _rects(w, h))
    sms.add_rgb(masks)
    keys = np.arange(1, 9, dtype=np.uint64)
    pm, pt = _pairs(2, 8, 7, n=4000)
    q = capi.ShapePairQueue(ctx, sms, max_batch=64)
    out = {}
    th = threading.Thread(target=lambda: out.update(r=q.drive(targets, grads, zgaps, keys, pm, pt, 40)))
    th.start()
    batched = []
    bm, bt = _pairs(2, 8, 8)
    batched.append((bm, bt, sms.score_pairs(targets, grads, zgaps, bm, bt)))
    sms.add_rgb(extra)
    bm, bt = _pairs(82, 8, 9, n=500)
    batched.append((bm, bt, sms.score_pairs(targets, grads, zgaps, bm, bt)))
    th.join()
    assert _same(out["r"][:3], sms.score_pairs(targets, grads, zgaps, pm, pt))
    ref = capi.ShapeMaskSet(ctx, w, h, 20, True, _rects(w, h))
    ref.add_rgb(np.concatenate([masks, extra]))
    for bm, bt, got in batched:
        assert _same(got, ref.score_pairs(targets, grads, zgaps, bm, bt))
    ref.close()
    q.close()
    sms.close()


def test_errors_and_edges(ctx):
    w, h = SMALL
    masks, targets, grads, zgaps = _data(ctx, SMALL, 2, 6, 16)
    masks = np.concatenate([masks, np.zeros((1, h, w, 3), np.uint8)])        # mask 2 is empty
    sms = capi.ShapeMaskSet(ctx, w, h, 20, True, _rects(w, h))
    sms.add_rgb(masks)
    capi.ShapePairQueue(ctx, sms).close()                                    # a queue that never scored
    q = capi.ShapePairQueue(ctx, sms, max_batch=64)
    # a missing gradient: (-1, -1, not mirrored) without a request
    assert q.score(0, targets[0], None, key=1) == (-1, -1, False)
    assert q.stats()["requests"] == 0
    with pytest.raises(capi.CdsIllegalArgument) as e:
        q.score(0, np.zeros((h + 1, w, 3), np.uint8), np.zeros((h + 1, w), np.uint16), key=2)
    assert e.value.status == capi.CDS_ERR_SIZE_MISMATCH
    for bad in (3, -1):
        with pytest.raises(capi.CdsIllegalArgument) as e:
            q.score(bad, targets[0], grads[0], key=1)
        assert e.value.status == capi.CDS_ERR_BAD_ARG
    with pytest.raises(capi.CdsIllegalArgument) as e:
        q.score(0, None, grads[0], key=1)
    assert e.value.status == capi.CDS_ERR_BAD_ARG
    # the empty mask scores what the batched call gives it
    pm, pt = _pairs(3, 6, 0)
    ref = sms.score_pairs(targets, grads, None, pm, pt)
    keys = np.arange(1, 7, dtype=np.uint64)
    got = q.drive(targets, grads, None, keys, pm, pt, 40)
    assert _same(got[:3], ref)
    # the cache holds every target: one upload per key, none on a second pass
    assert q.stats()["uploads"] == 6
    pm, pt = _pairs(3, 6, 1, n=2000)
    got = q.drive(targets, grads, None, keys, pm, pt, 40)
    assert _same(got[:3], sms.score_pairs(targets, grads, None, pm, pt))
    st = q.stats()
    assert st["uploads"] == 6
    assert st["requests"] == 2018 and st["batches"] < st["requests"]
    q.close()
    sms.close()


def test_two_devices():
    probe = capi.Context(n_dev=0)
    n_visible = probe.num_devices
    probe.close()
    if n_visible < 2:
        pytest.skip("one device visible")
    c = capi.Context(n_dev=2)
    masks, targets, grads, zgaps = _data(c, (W, H), 3, 8, 17)
    sms = capi.ShapeMaskSet(c, W, H, 20, True, O.label_rects(W, H))
    sms.add_rgb(masks)
    pm, pt = _pairs(3, 8, 2, n=200)
    keys = np.arange(1, 9, dtype=np.uint64)
    for zg in (zgaps, None):
        q = capi.ShapePairQueue(c, sms)
        assert _same(q.drive(targets, grads, zg, keys, pm, pt, 40)[:3], sms.score_pairs(targets, grads, zg, pm, pt))
        q.close()
    sms.close()
    c.close()
