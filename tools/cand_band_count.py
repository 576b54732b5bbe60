"""Counts, on the host, the candidate bits of the candidate kernel (mask pixels whose dilated target neighbourhood has a pixel of
the right colour sector, csrc/cds_cand.cu) and how many of them a finer test would remove when every sector's 19 820 ranks are
cut into NB fixed rank bands (band = rank * NB // 19820):

  today       word & occupancy word of the same (tile, sector): the kernel's candidates
  word NB     the same, minus the words whose band byte (OR over the word's set bits of the bands the pixel's interval in the
              list's sector touches) shares no band with the target tile's band byte (OR over the pixels that set the tile's
              occupancy bits of 1 << band(rank))
  pixel NB    per-pixel (sector x rank band) occupancy: a candidate stays only when a band its interval touches is occupied at
              its own position -- an upper bound on what any word-level filter can remove

Production parameters (mask / data threshold 20, zTolerance 0.01, xyShift 2, mirror).  Needs no GPU: the images come from the
host generator (oracle/synth.py) and the reference fixtures, the intervals from the library's host tables.

    python tools/cand_band_count.py [--masks 64] [--targets 256] [--data synthetic,real_fixture,dense_synthetic]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from colormipsearch_b200 import capi  # noqa: E402
from oracle import oracle as O  # noqa: E402
from oracle import synth as S  # noqa: E402

SEED = 0xC0FFEE
W, H = 1210, 566
MASK_T, DATA_T, TOL, XYSHIFT = 20, 20, 0.01, 2
NUM_RANKS, STRIDE, EMPTY = 19820, 32768, 0xFFFFFFFF
NBS = (4, 8)


def ratio_rank_table():
    """rank[second * 256 + max] of the distinct doubles second / max, 0 <= second < max <= 255 (csrc/cds_tables.cpp)."""
    a, b = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    valid = a < b
    r = np.where(valid, a / np.maximum(b, 1), 0.0)
    uniq = np.unique(r[valid])
    assert len(uniq) == NUM_RANKS
    return np.where(valid, np.searchsorted(uniq, r), 0).astype(np.int32).reshape(-1)


RANK = ratio_rank_table()


def classify(rgb):
    """-> sector (-1 = none), rank, max channel; the strict-inequality ladder of cds_tables.h classify_color."""
    r, g, b = (rgb[..., i].astype(np.int32) for i in range(3))
    sector = np.full(r.shape, -1, np.int32)
    second = np.zeros(r.shape, np.int32)
    mx = np.maximum(np.maximum(r, g), b)
    for s, cond, sec in ((0, (b > r) & (b > g) & (r > g), r), (1, (b > r) & (b > g) & ~(r > g), g),
                         (2, (g > b) & (g > r) & (b > r), b), (3, (g > b) & (g > r) & ~(b > r), r),
                         (4, (r > b) & (r > g) & (g > b), g), (5, (r > b) & (r > g) & ~(g > b), b)):
        sector[cond] = s
        second[cond] = sec[cond]
    rank = np.where(sector >= 0, RANK[second * 256 + mx], 0)
    return sector, rank, mx


def band_of(rank, nb):
    return (rank * nb) // NUM_RANKS


def shift_offsets():
    return [(dx, dy) for dx in (-2, 0, 2) for dy in (-2, 0, 2)] if XYSHIFT == 2 else [(0, 0)]


def target_planes(rgb):
    """-> per-pixel band masks [sectors, H, W] uint8 (bit b: some shifted position is in the image, above the threshold, of
    this sector and of rank band b, NB = 8; non-zero exactly where the sector's occupancy bit is set) and the tiles' band bytes
    [sectors, tile rows, tile cols]."""
    sector, rank, mx = classify(rgb)
    valid = (sector >= 0) & (mx > DATA_T)
    src = np.zeros((6, H, W), np.uint8)
    bit = (1 << band_of(rank, 8)).astype(np.uint8)
    for s in range(6):
        src[s] = np.where(valid & (sector == s), bit, 0)
    pad = 2
    sp = np.zeros((6, H + 2 * pad, W + 2 * pad), np.uint8)
    sp[:, pad:pad + H, pad:pad + W] = src
    occ = np.zeros((6, H, W), np.uint8)
    for dx, dy in shift_offsets():
        occ |= sp[:, pad + dy:pad + dy + H, pad + dx:pad + dx + W]
    HT, WT = (H + 3) // 4, (W + 7) // 8
    t = np.zeros((6, HT * 4, WT * 8), np.uint8)
    t[:, :H, :W] = occ
    tile = np.bitwise_or.reduce(t.reshape(6, HT, 4, WT, 8).transpose(0, 1, 3, 2, 4).reshape(6, HT, WT, 32), axis=3)
    return occ, tile


_IV = {}


def intervals(cls_sector, cls_rank):
    key = (int(cls_sector), int(cls_rank))
    if key not in _IV:
        _IV[key] = capi.class_intervals(TOL, *key)
    return _IV[key]


def band_span(lo_rank, hi_rank):
    """uint8 of the NB = 8 bands that ranks [lo_rank, hi_rank] touch."""
    b0, b1 = band_of(lo_rank, 8), band_of(min(hi_rank, NUM_RANKS - 1), 8)
    return ((1 << (b1 + 1)) - (1 << b0)) & 0xFF


def mask_lists(rgb):
    """The mask's list pixels in target coordinates: (sector, y, x, band byte of the pixel's interval in that sector,
    word id), sorted by word; word = (orientation, sector, tile row, tile column)."""
    om = O.PixelMatchMask(rgb, MASK_T, True, DATA_T, TOL, XYSHIFT, O.label_rects(W, H))
    pos = om.positions()
    y, x = pos // W, pos % W
    sector, rank, _ = classify(rgb[y, x])
    rows = []
    for i in np.nonzero(sector >= 0)[0]:
        lo1, len1, lo2, len2 = intervals(sector[i], rank[i])
        for lo, ln in ((lo1, len1), (lo2, len2)):
            if lo == EMPTY:
                continue
            s, r0 = lo // STRIDE, lo % STRIDE
            bb = band_span(r0, r0 + ln)
            for o, xo in ((0, x[i]), (1, W - 1 - x[i])):
                rows.append((o, s, y[i], xo, bb))
    a = np.array(rows, np.int64).reshape(-1, 5)
    o, s, yy, xx, bb = a.T
    word = ((o * 6 + s) * 1024 + yy // 4) * 1024 + xx // 8
    order = np.argsort(word, kind="stable")
    o, s, yy, xx, bb, word = (v[order] for v in (o, s, yy, xx, bb, word))
    _, wid = np.unique(word, return_inverse=True)
    return dict(s=s, y=yy, x=xx, bb=bb.astype(np.uint8), wid=wid)


FOLD4 = np.array([(v | v >> 1) & 1 | (v >> 1 | v >> 2) & 2 | (v >> 2 | v >> 3) & 4 | (v >> 3 | v >> 4) & 8 for v in range(256)],
                 np.uint8)   # NB 8 -> 4: band4 = band8 // 2


def prepare(ml):
    starts = np.r_[0, np.nonzero(np.diff(ml["wid"]))[0] + 1] if len(ml["wid"]) else np.zeros(0, np.int64)
    ml["starts"] = starts
    ml["wty"] = ml["y"][starts] // 4
    ml["wtx"] = ml["x"][starts] // 8
    ml["wsec"] = ml["s"][starts]
    ml["wbb"] = {8: np.bitwise_or.reduceat(ml["bb"], starts) if len(starts) else np.zeros(0, np.uint8)}
    ml["wbb"][4] = FOLD4[ml["wbb"][8]]
    ml["bb4"] = FOLD4[ml["bb"]]
    return ml


def count_pair(ml, occ, tile):
    """-> dict of candidate bits (and words with candidates) for one (mask, target)."""
    pb = occ[ml["s"], ml["y"], ml["x"]]
    cand = pb != 0
    out = {"today": int(cand.sum()), "words_today": int(np.bitwise_or.reduceat(cand, ml["starts"]).sum()) if len(cand) else 0}
    tb8 = tile[ml["wsec"], ml["wty"], ml["wtx"]]
    for nb in NBS:
        tb = tb8 if nb == 8 else FOLD4[tb8]
        keep = (tb & ml["wbb"][nb]) != 0
        kc = cand & keep[ml["wid"]]
        out["word%d" % nb] = int(kc.sum())
        out["words_word%d" % nb] = int(np.bitwise_or.reduceat(kc, ml["starts"]).sum()) if len(kc) else 0
        pbn = pb if nb == 8 else FOLD4[pb]
        out["pixel%d" % nb] = int(((pbn & (ml["bb"] if nb == 8 else ml["bb4"])) != 0).sum())
    return out


def run(name, masks, targets):
    mls = [prepare(mask_lists(m)) for m in masks]
    tot = {}
    for t in targets:
        occ, tile = target_planes(t)
        for ml in mls:
            for k, v in count_pair(ml, occ, tile).items():
                tot[k] = tot.get(k, 0) + v
    res = {"data": name, "masks": len(masks), "targets": len(targets), "candidate_bits_per_pair": tot["today"] / (len(masks) * len(targets))}
    for nb in NBS:
        res["word%d_removed" % nb] = 1.0 - tot["word%d" % nb] / max(tot["today"], 1)
        res["word%d_words_removed" % nb] = 1.0 - tot["words_word%d" % nb] / max(tot["words_today"], 1)
        res["pixel%d_removed" % nb] = 1.0 - tot["pixel%d" % nb] / max(tot["today"], 1)
    return res


def fixture_sets(n_masks, n_targets):
    """real_fixture and dense_synthetic as bench.py's data_dependence builds them (same seeds and jitter)."""
    rects = O.label_rects(W, H)
    rng = np.random.default_rng(7)
    fx = np.load(os.path.join(ROOT, "tests", "golden", "cdsearch_fixtures.npz"))

    def clear(img):
        img = img.copy()
        for x0, y0, x1, y1 in rects:
            img[y0:y1, x0:x1] = 0
        return img

    def jitter(img, scale):
        out = np.roll(img, (int(rng.integers(-40, 41)), int(rng.integers(-60, 61))), axis=(0, 1))
        if scale < 1.0:
            out = ((out.astype(np.uint16) * int(scale * 256)) >> 8).astype(np.uint8)
        return out

    em = [clear(fx[k]) for k in ("em_12191", "em_12191_FL", "em_LPLC2")]
    lm = [clear(fx[k]) for k in ("lm_BJD", "lm_GMR", "lm_VT016795", "lm_VT033614")]
    masks = np.stack([jitter(em[i % 3], 1.0) for i in range(n_masks)])
    targets = np.stack([jitter(lm[i % 4], float(rng.uniform(0.5, 1.0))) for i in range(n_targets)])
    real = (masks, targets)
    base = S.synth_rgb(1, SEED, 100000, 6 * 128, W, H)
    pool = []
    for i in range(128):
        out = base[6 * i].copy()
        for k in range(1, 6):
            nxt = base[6 * i + k]
            empty = ~out.any(axis=2)
            out[empty] = nxt[empty]
        pool.append(out)
    dense_t = np.stack([jitter(pool[i % 128], 1.0) for i in range(n_targets)])
    return real, dense_t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--masks", type=int, default=64)
    ap.add_argument("--targets", type=int, default=256)
    ap.add_argument("--data", default="synthetic,real_fixture,dense_synthetic")
    a = ap.parse_args()
    want = a.data.split(",")
    synth_masks = S.synth_rgb(0, SEED, 0, a.masks, W, H)
    if "synthetic" in want:
        print(json.dumps(run("synthetic", synth_masks, S.synth_rgb(1, SEED, 0, a.targets, W, H))), flush=True)
    if "real_fixture" in want or "dense_synthetic" in want:
        (rm, rt), dt = fixture_sets(a.masks, a.targets)
        if "real_fixture" in want:
            print(json.dumps(run("real_fixture", rm, rt)), flush=True)
        if "dense_synthetic" in want:
            print(json.dumps(run("dense_synthetic", synth_masks, dt)), flush=True)


if __name__ == "__main__":
    main()
