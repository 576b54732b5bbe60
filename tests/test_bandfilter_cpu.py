"""The host count of the rank-band word filter (tools/cand_band_count.py): the word filter removes no more than the per-pixel
bound, eight bands remove at least what four remove, and the fixed band table splits every sector's ranks evenly."""
import importlib.util
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tool():
    spec = importlib.util.spec_from_file_location("cand_band_count", os.path.join(ROOT, "tools", "cand_band_count.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_band_table_is_even_and_fixed():
    T = _tool()
    bands = T.band_of(np.arange(T.NUM_RANKS), 4)
    counts = np.bincount(bands)
    assert len(counts) == 4 and counts.max() - counts.min() <= 1
    assert np.array_equal(T.FOLD4[1 << T.band_of(np.arange(T.NUM_RANKS), 8)], 1 << bands)


def test_word_filter_counts_are_bounded_by_per_pixel_filter():
    T = _tool()
    res = T.run("synthetic", T.S.synth_rgb(0, T.SEED, 0, 2, T.W, T.H), T.S.synth_rgb(1, T.SEED, 0, 3, T.W, T.H))
    for nb in (4, 8):
        assert 0.0 <= res["word%d_removed" % nb] <= res["pixel%d_removed" % nb] + 1e-12
    assert res["word8_removed"] >= res["word4_removed"]
