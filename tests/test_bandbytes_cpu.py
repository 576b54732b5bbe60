"""The candidate kernel's launch configuration (cds_debug_cand_config, no device needed).  The staged palette is sized to the launch's
largest palette, which pays for one rank-band byte per sector tile word: at the bench's 1210 x 566 with xyShift 2 the kernel keeps two
stages of 12-row bands with 31 consumer warps up to the palette size that DESIGN.md §4.1 states."""
from colormipsearch_b200 import capi

W, H = 1210, 566
BUDGET = 227 * 1024
PALETTE_LIMIT = 1936       # the largest palette + idle entry with 12-row bands at xyShift 2 (DESIGN.md §4.1)


def test_headline_palette_keeps_twelve_row_bands():
    # the bench's synthetic mask group: 256 colour classes + the idle entry
    warps, rows, stages, smem = capi.cand_config(W, H, 2, 257)
    assert (warps, rows, stages) == (31, 12, 2)
    assert 0 < smem <= BUDGET


def test_wide_lists_keep_twelve_row_bands():
    # WIDE lists read no palette, whatever size is asked for
    assert capi.cand_config(W, H, 2, 2048, wide=True) == capi.cand_config(W, H, 2, 1, wide=True)
    warps, rows, stages, smem = capi.cand_config(W, H, 2, 2048, wide=True)
    assert (warps, rows, stages) == (31, 12, 2)
    assert 0 < smem <= BUDGET


def test_xyshift_0_and_4_band_heights():
    # with the largest palette the band heights are those of the 4-band layout, which always staged 2,048 entries: 12 rows at
    # xyShift 0, 8 at xyShift 4, 31 warps and 2 stages at both
    assert capi.cand_config(W, H, 0, 2048)[:3] == (31, 12, 2)
    assert capi.cand_config(W, H, 4, 2048)[:3] == (31, 8, 2)
    # xyShift 4 stays at 8 rows with the headline palette; at xyShift 0 the room the small palette leaves fits 16-row bands
    assert capi.cand_config(W, H, 4, 257)[:3] == (31, 8, 2)
    assert capi.cand_config(W, H, 0, 257)[:3] == (31, 16, 2)


def test_largest_palette_with_twelve_row_bands():
    assert capi.cand_config(W, H, 2, PALETTE_LIMIT)[:3] == (31, 12, 2)
    assert capi.cand_config(W, H, 2, PALETTE_LIMIT)[3] <= BUDGET
    # one more entry rounds the staged palette up by 16 and no longer fits: the search falls back to 8-row bands
    assert capi.cand_config(W, H, 2, PALETTE_LIMIT + 1)[:3] == (31, 8, 2)
    assert capi.cand_config(W, H, 2, 2048)[:3] == (31, 8, 2)


def test_staged_palette_is_rounded_to_16_entries():
    smem = [capi.cand_config(W, H, 2, p)[3] for p in (1, 16, 17, 32, 257, 272)]
    assert smem[0] == smem[1] and smem[2] == smem[3] and smem[4] == smem[5]
    assert smem[2] - smem[1] == 16 * 8


def test_bad_arguments_are_refused():
    import pytest
    for args in ((W, H, 1, 257), (W, H, 2, 0), (W, H, 2, 2049), (0, H, 2, 257), (4096, H, 2, 257)):
        with pytest.raises(capi.CdsIllegalArgument):
            capi.cand_config(*args)
