"""One cds_ctx over all visible devices: dense / top-K / streaming searches (pixels and TIFF files, library from TIFF files, all
matches, best matches selected on the device) must equal the single-device results."""
import sys, numpy as np
sys.path.insert(0, ".")
from colormipsearch_b200 import capi
from oracle import oracle as O
W, H = 1210, 566
masks = capi.synth_rgb_host(0, 0xC0FFEE, 0, 24, W, H)
targets = capi.synth_rgb_host(1, 0xC0FFEE, 0, 200, W, H)
rects = O.label_rects(W, H)
files = [capi.tiff_encode_rgb(t, 8 if i % 3 else 566, 32773 if i % 5 else 1) for i, t in enumerate(targets)]
NS = 72                                   # targets of the shape part: three windows of 32, so both devices get work
grads = np.stack([capi.synth_gradient_host(0xC0FFEE, i, 1, W, H)[0] if i < 6 else np.roll(capi.synth_gradient_host(0xC0FFEE, i % 6, 1, W, H)[0], i, axis=1) for i in range(NS)])
rng = np.random.default_rng(3)
pm = rng.integers(0, 6, 600); pt = rng.integers(0, NS, 600)
has = (np.arange(NS) % 11 != 5).astype(np.uint8)
pfiles = [capi.png_encode_gray16(g, -1 if i % 2 else 0) for i, g in enumerate(grads)]
tfiles = [capi.tiff_encode_rgb(t, 8, 32773) for t in targets[:NS]]
lines = ["R%dG%02d" % (10 + i // 7, i // 7) for i in range(200)]           # lines of 7 targets, samples of 2
groups = capi.TargetGroups(lines, ["%d" % (i // 2) for i in range(200)])
res = {}
for nd in (1, 0):
    ctx = capi.Context(n_dev=nd)
    print("devices", ctx.num_devices)
    ctx.set_option("stream_chunk", 16)
    ctx.set_option("stream_chunk_tiff", 24)
    lib = capi.Library(ctx, W, H, 256); lib.add_rgb(targets)
    ms = capi.MaskSet(ctx, W, H, 20, 20, 0.01, 2, True, rects); ms.add_rgb(masks)
    lib2 = capi.Library(ctx, W, H, 256); lib2.add_tiff(files)
    res[nd] = (ms.search_dense(lib), ms.search_topk(lib, 50, 0.0), ms.search_stream(targets, 50, 0.0), ms.search_stream_tiff(files, 50, 0.0),
               ms.search_topk(lib2, 50, 0.0), ms.search_stream_matches_tiff(files, 1.0), ms.search_matches(lib, 1.0))
    # shape score across the context's devices (windows of targets dealt out over the devices, masks replicated), pixels / TIFF / TIFF + PNG
    sms = capi.ShapeMaskSet(ctx, W, H, 20, True, rects)
    qm, he = sms.add_rgb(masks[:6])
    shape_res = (qm, he, sms.score_pairs(targets[:NS], grads, None, pm, pt, has), sms.score_pairs_tiff(tfiles, grads, None, pm, pt, has),
                 sms.score_pairs_files(tfiles, pfiles, None, pm, pt, has))
    sms.close()
    # the single-pair queue: one dispatcher per device, targets spread by key
    q = capi.PairQueue(ctx, ms, max_batch=32, max_wait_us=100, cache_targets=128)
    qpm = np.repeat(np.arange(24), 40).astype(np.int32); qpt = np.tile(np.arange(40), 24).astype(np.int64)
    qs, qmir, _ = q.drive(targets[:40], (np.arange(40) + 1).astype(np.uint64), qpm, qpt, 16)
    q.close()
    res[nd] = res[nd] + (shape_res, (qs, qmir, qpm, qpt))
    res[nd] = res[nd] + ([(ms.search_best_matches(lib, groups, 1.0, *lim), ms.search_stream_best_matches_tiff(files, groups, 1.0, *lim))
                          for lim in ((300, 1, 1), (5, 3, 2), (0, 0, 0))],)
    ms.close(); lib.close(); lib2.close(); ctx.close()
a, b = res[1], res[0]
print("dense equal:", np.array_equal(a[0][0], b[0][0]), np.array_equal(a[0][1], b[0][1]))
for name, i in (("topk", 1), ("stream", 2), ("stream_tiff", 3), ("topk over a TIFF-built library", 4)):
    ok = np.array_equal(a[i][3], b[i][3]) and all(np.array_equal(a[i][j][m, :a[i][3][m]], b[i][j][m, :a[i][3][m]]) for j in range(3) for m in range(24))
    print(name, "equal:", ok)
ok = all(np.array_equal(a[1][j][m, :a[1][3][m]], a[2][j][m, :a[1][3][m]]) for j in range(3) for m in range(24))
print("stream == topk:", ok)
for i in (3, 4):
    ok = all(np.array_equal(a[1][j][m, :a[1][3][m]], b[i][j][m, :a[1][3][m]]) for j in range(3) for m in range(24))
    print("multi-device result %d == single-device topk:" % i, ok)
print("all-matches over TIFF files == all-matches over the resident library (single, multi):",
      all(np.array_equal(x, y) for x, y in zip(a[5], a[6])), all(np.array_equal(x, y) for x, y in zip(b[5], b[6])),
      "; single == multi:", all(np.array_equal(x, y) for x, y in zip(a[5], b[5])))
sa, sb = a[7], b[7]
print("shape mask sizes equal:", np.array_equal(sa[0], sb[0]) and np.array_equal(sa[1], sb[1]))
for name, i in (("shape pairs (pixels)", 2), ("shape pairs (TIFF)", 3), ("shape pairs (TIFF + PNG)", 4)):
    print(name, "single == multi:", all(np.array_equal(x, y) for x, y in zip(sa[i], sb[i])), "; == pixel call:", all(np.array_equal(x, y) for x, y in zip(sb[i], sa[2])))
for nd, r in ((1, a), (0, b)):
    qs, qmir, qpm, qpt = r[8]
    print("pair queue (devices %s) == dense:" % ("1" if nd else "all"), np.array_equal(qs, r[0][0][qpm, qpt]) and np.array_equal(qmir, r[0][1][qpm, qpt].astype(bool)))
best_ok = all(all(np.array_equal(x, y) for x, y in zip(r1, r2)) for p1, p2 in zip(a[9], b[9]) for r1, r2 in zip(p1, p2))
files_ok = all(all(np.array_equal(x, y) for x, y in zip(p[0], p[1])) for r in (a, b) for p in r[9])
print("best matches (resident, TIFF files) single == multi:", best_ok, "; files == resident:", files_ok)
