"""The best-matches selection on the device (cds_search_best_matches, the streamed variants and the selection hook) against the
two-step path it replaces: every pair that passes isMatch (cds_search_matches), then cds_select_best_matches mask by mask."""
import ctypes as C

import numpy as np
import pytest

from colormipsearch_b200 import capi
from oracle import oracle as O
from tests.test_select_cpu import reference_test_data

pytestmark = pytest.mark.gpu

W, H = 1210, 566
LIMITS = [(0, 0, 0), (1, 1, 1), (2, 3, 2), (3, 2, 0), (2, 0, 1), (300, 1, 1), (300, 0, 0), (300, 3, 2), (0, 1, 0), (1, 0, 0)]


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(n_dev=1)
    yield c
    c.close()


def make_groups(line, sample, line_hash, sample_hash):
    g = capi.TargetGroups.__new__(capi.TargetGroups)
    g.line, g.sample, g.line_hash, g.sample_hash = [np.ascontiguousarray(a, np.int32) for a in (line, sample, line_hash, sample_hash)]
    return g


def host_select(g, target, score, limits):
    n = len(target)
    lid = np.ascontiguousarray(g.line[target]); sid = np.ascontiguousarray(g.sample[target]); sc = np.ascontiguousarray(score, np.int32)
    sel = np.zeros(max(n, 1), np.int64)
    cnt = C.c_int64(0)
    capi._check(capi.lib().cds_select_best_matches(lid.ctypes.data_as(capi._i32p), sid.ctypes.data_as(capi._i32p), sc.ctypes.data_as(capi._i32p), n,
                                                   g.line_hash.ctypes.data_as(capi._i32p), len(g.line_hash), g.sample_hash.ctypes.data_as(capi._i32p),
                                                   len(g.sample_hash), *[int(x) for x in limits], sel.ctypes.data_as(capi._i64p), C.byref(cnt)))
    return sel[: cnt.value]


def two_step(mask, target, score, g, limits):
    """indices into the (mask, score desc, target asc) list of what the per-mask host selection keeps, masks ascending"""
    out = []
    if len(mask):
        bounds = np.searchsorted(mask, np.arange(int(mask.max()) + 2))
        for a, b in zip(bounds[:-1], bounds[1:]):
            if a < b:
                out.append(a + host_select(g, target[a:b], score[a:b], limits))
    return np.concatenate(out) if out else np.zeros(0, np.int64)


def expected(matches, g, limits):
    idx = two_step(matches[0], matches[1], matches[2], g, limits)
    return tuple(a[idx] for a in matches)


def assert_same(got, exp):
    assert len(got[0]) == len(exp[0])
    for x, y in zip(got, exp):
        assert np.array_equal(x, y)


# ---- 1. the selection hook against cds_select_best_matches ----

def random_list(rng, n_masks, n_targets, n_lines, n_samples, n_scores):
    mask, target, score = [], [], []
    for m in range(n_masks):
        k = 0 if rng.random() < 0.15 else (1 if rng.random() < 0.1 else int(rng.integers(1, n_targets + 1)))
        t = np.sort(rng.choice(n_targets, k, replace=False))
        s = rng.integers(1, n_scores + 1, k)
        order = np.lexsort((t, -s))
        mask.append(np.full(k, m)); target.append(t[order]); score.append(s[order])
    return (np.concatenate(mask).astype(np.int32), np.concatenate(target).astype(np.int64), np.concatenate(score).astype(np.int32))


def test_hook_random_lists(ctx):
    rng = np.random.default_rng(2024)
    for trial in range(240):
        n_targets = int(rng.integers(1, 400))
        n_lines = int(rng.choice([1, 5, 12, 13, 24, 25, 48, 49, 96, 97, 150]))
        n_samples = int(rng.choice([1, 7, 12, 13, 24, 25, 48, 49, 96, 97, 300]))
        line = rng.integers(0, n_lines, n_targets)
        sample = rng.integers(0, n_samples, n_targets)
        if trial % 3 == 0:        # colliding buckets: few distinct hashes
            lh = rng.integers(-4, 4, n_lines) * 65536 * int(rng.choice([1, 16]))
            sh = rng.integers(0, 3, n_samples) * 16
        else:                     # the names' own String hashes, one of them "UNKNOWN" (blank names)
            lh = np.array([capi.java_string_hash("UNKNOWN" if i == 0 else "R%dG%02d" % (10 + i % 90, i)) for i in range(n_lines)])
            sh = np.array([capi.java_string_hash("%d" % (2000000 + 7919 * i)) for i in range(n_samples)])
        g = make_groups(line, sample, lh, sh)
        mask, target, score = random_list(rng, int(rng.integers(1, 6)), n_targets, n_lines, n_samples, int(rng.choice([2, 3, 11, 500])))
        limits = LIMITS[trial % len(LIMITS)], (int(rng.integers(0, 30)), int(rng.integers(0, 5)), int(rng.integers(0, 4)))
        for lim in limits:
            got = capi.debug_select_best_matches_device(ctx, mask, target, score, None, g, *lim)
            assert np.array_equal(got, two_step(mask, target, score, g, lim)), (trial, lim)


def test_hook_reference_data(ctx):
    data = reference_test_data()
    order = sorted(range(len(data)), key=lambda i: (-data[i][2], i))
    enc = [data[i] + (i,) for i in order]                      # encounter order: score desc, target asc
    g = capi.TargetGroups([m[0] for m in data], [m[1] for m in data])
    target = np.array([m[3] for m in enc], np.int64)
    score = np.array([m[2] for m in enc], np.int32)
    for lim in LIMITS:
        got = capi.debug_select_best_matches_device(ctx, np.zeros(len(enc), np.int32), target, score, None, g, *lim)
        assert [enc[i] for i in got.tolist()] == O.select_best_matches(list(enc), *lim), lim


# ---- 2-4, 6. searches ----

def random_groups(rng, n_targets, blank_every=17):
    """lines of 1-40 targets, inside them samples of 1-6 targets, over a shuffled target order"""
    perm = rng.permutation(n_targets)
    lines, samples = [None] * n_targets, [None] * n_targets
    i = li = si = 0
    while i < n_targets:
        ln = "" if li % blank_every == 5 else "R%dG%02d_AE_01" % (10 + li % 80, li)
        end = min(n_targets, i + int(rng.integers(1, 41)))
        while i < end:
            send = min(end, i + int(rng.integers(1, 7)))
            for t in perm[i:send]:
                lines[t], samples[t] = ln, "%d" % (1000000 + 7919 * si)
            i, si = send, si + 1
        li += 1
    return capi.TargetGroups(lines, samples)


@pytest.fixture(scope="module")
def resident(ctx):
    rng = np.random.default_rng(7)
    n_targets = 3000
    lib = capi.Library(ctx, W, H, n_targets)
    lib.generate_synthetic(0xB357, 0, n_targets)
    masks = capi.synth_rgb_host(0, 0xB357, 0, 24, W, H)
    groups = random_groups(rng, n_targets)
    yield lib, masks, groups
    lib.close()


def make_maskset(ctx, masks, xy_shift=2, mirror=True):
    ms = capi.MaskSet(ctx, W, H, 20, 20, 0.01, xy_shift, mirror, O.label_rects(W, H))
    ms.add_rgb(masks)
    return ms


@pytest.mark.parametrize("params", [(2, True), (0, False)])
@pytest.mark.parametrize("pct", [0.0, 1.0])
def test_resident_search_equals_two_steps(ctx, resident, params, pct):
    lib, masks, groups = resident
    ms = make_maskset(ctx, masks, *params)
    try:
        matches = ms.search_matches(lib, pct)
        assert len(matches[0]) > 100
        for occ in (1, 0):
            ctx.set_option("resident_occupancy", occ)
            for lim in ((300, 0, 0), (300, 1, 1), (300, 3, 2), (5, 2, 1), (0, 0, 0), (20, 0, 3)):
                assert_same(ms.search_best_matches(lib, groups, pct, *lim), expected(matches, groups, lim))
    finally:
        ctx.set_option("resident_occupancy", 1)
        ms.close()


def test_d2h_bytes_follow_the_selection(ctx, resident):
    lib, masks, groups = resident
    ms = make_maskset(ctx, masks)
    try:
        matches = ms.search_matches(lib, 0.0)
        assert ctx.last_stats()["d2h_bytes"] == 12 * len(matches[0])
        sel = ms.search_best_matches(lib, groups, 0.0, 300, 1, 1)
        assert 0 < len(sel[0]) < len(matches[0]) // 4
        assert ctx.last_stats()["d2h_bytes"] <= 17 * len(sel[0]) + 4096
    finally:
        ms.close()


@pytest.fixture(scope="module")
def streamed(ctx):
    rng = np.random.default_rng(11)
    n_targets = 400
    targets = capi.synth_rgb_host(1, 0x57EA, 0, n_targets, W, H)
    files = [capi.tiff_encode_rgb(t, 8, 32773) for t in targets]
    lib = capi.Library(ctx, W, H, n_targets)
    lib.add_rgb(targets)
    masks = capi.synth_rgb_host(0, 0x57EA, 0, 24, W, H)
    yield targets, files, lib, masks, random_groups(rng, n_targets)
    lib.close()


def test_streamed_files_and_pixels_equal_resident(ctx, streamed):
    targets, files, lib, masks, groups = streamed
    ms = make_maskset(ctx, masks)
    try:
        ctx.set_option("stream_chunk_tiff", 48)
        ctx.set_option("stream_chunk", 48)
        matches = ms.search_matches(lib, 1.0)
        for lim in ((300, 1, 1), (300, 3, 2), (4, 2, 0)):
            res = ms.search_best_matches(lib, groups, 1.0, *lim)
            assert_same(res, expected(matches, groups, lim))
            assert_same(ms.search_stream_best_matches_tiff(files, groups, 1.0, *lim), res)
            assert_same(ms.search_stream_best_matches_rgb(targets, groups, 1.0, *lim), res)
    finally:
        ctx.set_option("stream_chunk_tiff", 4096)
        ctx.set_option("stream_chunk", 256)
        ms.close()


def test_compaction_and_capacity(ctx, streamed):
    targets, files, lib, masks, groups = streamed
    ms = make_maskset(ctx, masks)
    chunk = 16
    try:
        ctx.set_option("stream_chunk_tiff", chunk)
        ctx.set_option("stream_chunk", chunk)
        matches = ms.search_matches(lib, 0.0)
        n_pass = len(matches[0])
        keys = {(int(m), int(groups.line[t]), int(groups.sample[t])) for m, t in zip(matches[0], matches[1])}
        for tm in (2, 1):
            budget = tm * len(keys) + len(masks) * chunk + 16            # pairs: room for a compacted list and one chunk
            assert budget < n_pass or tm > 1
            ctx.set_option("best_list_bytes", 12 * budget)
            for lim in ((300, 3, tm), (2, 1, tm), (0, 0, tm)):
                exp = expected(matches, groups, lim)
                assert_same(ms.search_best_matches(lib, groups, 0.0, *lim), exp)
                assert_same(ms.search_stream_best_matches_tiff(files, groups, 0.0, *lim), exp)
        # the same budget without a per-sample limit: the list cannot shrink, CDS_ERR_CAPACITY names the bytes of all passing pairs
        with pytest.raises(capi.CdsError) as e:
            ms.search_best_matches(lib, groups, 0.0, 300, 3, 0)
        assert e.value.status == capi.CDS_ERR_CAPACITY and str(12 * n_pass) in e.value.message
        ctx.set_option("best_list_bytes", 1 << 30)
        # output capacity below the selection: nothing written, the count reported
        exp = expected(matches, groups, (300, 1, 1))
        n_sel = len(exp[0])
        cap = n_sel - 1
        out = [np.full(cap, -7, np.int32), np.full(cap, -7, np.int64), np.full(cap, -7, np.int32), np.zeros(cap, np.uint8)]
        cnt = C.c_int64(0)
        g = groups.struct()
        st = capi.lib().cds_search_best_matches(ctx.h, ms.h, lib.h, C.byref(g), 0.0, 300, 1, 1, cap, out[0].ctypes.data_as(capi._i32p),
                                                out[1].ctypes.data_as(capi._i64p), out[2].ctypes.data_as(capi._i32p), out[3].ctypes.data_as(capi._u8p),
                                                C.byref(cnt))
        assert st == capi.CDS_ERR_CAPACITY and cnt.value == n_sel
        assert (out[0] == -7).all() and (out[1] == -7).all()
        assert_same(ms.search_best_matches(lib, groups, 0.0, 300, 1, 1, capacity=n_sel), exp)
    finally:
        ctx.set_option("best_list_bytes", 1 << 30)
        ctx.set_option("stream_chunk_tiff", 4096)
        ctx.set_option("stream_chunk", 256)
        ms.close()


def test_bad_group_ids_and_size_mismatch(ctx, streamed):
    targets, files, lib, masks, groups = streamed
    ms = make_maskset(ctx, masks[:2])
    try:
        bad = make_groups(groups.line, groups.sample, groups.line_hash, groups.sample_hash)
        bad.line = bad.line.copy(); bad.line[len(bad.line) - 1] = len(bad.line_hash)
        with pytest.raises(capi.CdsIllegalArgument, match="line id"):
            ms.search_best_matches(lib, bad, 0.0, 300, 1, 1)
        small = capi.Library(ctx, 64, 64, 4)
        with pytest.raises(capi.CdsIllegalArgument, match="Invalid image size"):
            ms.search_best_matches(small, make_groups([], [], [0], [0]), 0.0, 300, 1, 1)
        small.close()
    finally:
        ms.close()


# ---- 5. the reference's fixture images against the oracle ----

def test_golden_fixtures_against_oracle(ctx, fixtures):
    rects = O.label_rects(W, H, 270)
    lm_keys = ["lm_VT033614", "lm_BJD", "lm_VT016795", "lm_GMR"]
    em_keys = ["em_12191", "em_12191_FL", "em_LPLC2"]
    targets = np.stack([fixtures[k] for k in lm_keys])
    lines = [k.split("_")[1][:2] for k in lm_keys]            # VT, BJ, VT, GM
    samples = [k.split("_")[1] for k in lm_keys]
    lib = capi.Library(ctx, W, H, 8)
    lib.add_rgb(targets)
    ms = capi.MaskSet(ctx, W, H, 20, 20, 0.01, 2, True, rects)
    sizes = ms.add_rgb(np.stack([fixtures[k] for k in em_keys]))
    oms = [O.PixelMatchMask(fixtures[k], 20, True, 20, 0.01, 2, rects) for k in em_keys]
    es, _, _ = O.search_dense(oms, targets)
    groups = capi.TargetGroups(lines, samples)
    try:
        for pct in (0.0, 1.0):
            for lim in ((300, 1, 1), (1, 1, 1), (0, 0, 0), (2, 1, 0)):
                got = ms.search_best_matches(lib, groups, pct, *lim)
                exp_mask, exp_target, exp_score = [], [], []
                for m in range(len(em_keys)):
                    passing = [t for t in range(len(lm_keys)) if O.is_match(int(es[m, t]), es[m, t] / sizes[m], pct)]
                    passing.sort(key=lambda t: (-es[m, t], t))
                    sel = O.select_best_matches([(lines[t], samples[t], int(es[m, t]), t) for t in passing], *lim)
                    exp_mask += [m] * len(sel); exp_target += [s[3] for s in sel]; exp_score += [s[2] for s in sel]
                assert got[0].tolist() == exp_mask and got[1].tolist() == exp_target and got[2].tolist() == exp_score, (pct, lim)
    finally:
        ms.close()
        lib.close()


# ---- 7. two devices ----

def two_device_context():
    probe = capi.Context(n_dev=0)
    n_visible = probe.num_devices
    probe.close()
    # with one GPU, a context that names it twice still runs the two-device path (library shards, two lists moved to the first device)
    return capi.Context(n_dev=2) if n_visible >= 2 else capi.Context(device_ids=[0, 0])


def test_two_devices_equal_one(ctx, streamed):
    targets, files, lib, masks, groups = streamed
    ctx2 = two_device_context()
    try:
        assert ctx2.num_devices == 2
        ms1 = make_maskset(ctx, masks)
        ms2 = make_maskset(ctx2, masks)
        lib2 = capi.Library(ctx2, W, H, len(targets))
        lib2.add_rgb(targets)
        for c in (ctx, ctx2):
            c.set_option("stream_chunk_tiff", 48)
        for lim in ((300, 1, 1), (300, 3, 2), (300, 0, 0)):
            one = ms1.search_best_matches(lib, groups, 1.0, *lim)
            assert_same(ms2.search_best_matches(lib2, groups, 1.0, *lim), one)
            assert_same(ms2.search_stream_best_matches_tiff(files, groups, 1.0, *lim), one)
        ms1.close(); ms2.close(); lib2.close()
    finally:
        ctx.set_option("stream_chunk_tiff", 4096)
        ctx2.close()


def test_two_devices_compaction_of_a_resident_library(ctx, streamed):
    """A resident library sharded over two devices keeps shard-local target indices in its lists until the search ends; a list that
    fills during the search is compacted by the targets' real lines and samples, and the result is the one-device two-step result."""
    targets, files, lib, masks, groups = streamed
    ctx2 = two_device_context()
    chunk = 4
    compacted = False
    try:
        ms = make_maskset(ctx, masks)
        matches = ms.search_matches(lib, 0.0)
        ms.close()
        ms2 = make_maskset(ctx2, masks)
        lib2 = capi.Library(ctx2, W, H, len(targets))
        lib2.add_rgb(targets)
        ctx2.set_option("stream_chunk", chunk)
        shard = (matches[1] // 64) % 2                              # block-cyclic sharding, 64 targets a block
        passing = [int((shard == d).sum()) for d in (0, 1)]
        keys = [{(int(m), int(groups.line[t]), int(groups.sample[t])) for m, t, sh in zip(*matches[:2], shard) if sh == d} for d in (0, 1)]
        for tm in (1, 2):
            budget = tm * max(len(k) for k in keys) + len(masks) * chunk + 16     # pairs: a compacted list and one chunk
            if budget >= max(passing):
                continue
            ctx2.set_option("best_list_bytes", 12 * budget)
            for lim in ((300, 3, tm), (2, 1, tm), (0, 0, tm)):
                assert_same(ms2.search_best_matches(lib2, groups, 0.0, *lim), expected(matches, groups, lim))
            compacted = True
        assert compacted
        ms2.close(); lib2.close()
    finally:
        ctx2.close()
