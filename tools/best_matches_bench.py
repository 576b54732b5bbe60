"""Best-matches selection fused into the search (cds_search_best_matches, cds_search_stream_best_matches_tiff) against the two-step
path it replaces: every passing pair to the host (cds_search_matches / cds_search_stream_matches_tiff), then
cds_select_best_matches for every mask.  configs[1] share: 1 000 masks x 12 500 resident synthetic targets, production parameters
(xyShift 2, mirror, pct 1); the TIFF leg streams PackBits files of the first --tiff-targets of those targets.  Lines of 1-40 targets,
samples of 1-6 targets inside them (seeded).  Per leg and limit set it prints one JSON line: passing and selected pairs, wall time and
d2h_bytes of both paths (outputs compared), and the device time of the selection stage (kernels of csrc/cds_bestsel.cu and the cub
sorts / scans it launches, from torch.profiler over one more call).

    python tools/best_matches_bench.py [--masks 1000] [--targets 12500] [--tiff-targets 2000] [--reps 3]
"""
import argparse, ctypes as C, json, subprocess, sys, time
import numpy as np
sys.path.insert(0, ".")
from colormipsearch_b200 import capi
from oracle import oracle as O

W, H, SEED = 1210, 566, 0xC0FFEE
ap = argparse.ArgumentParser()
ap.add_argument("--masks", type=int, default=1000)
ap.add_argument("--targets", type=int, default=12500)
ap.add_argument("--tiff-targets", type=int, default=2000)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--pct", type=float, default=1.0)
a = ap.parse_args()
LIMITS = [(300, 0, 0), (300, 1, 1), (300, 3, 2)]


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        return "unknown"


def groups_for(n_targets, seed=5):
    rng = np.random.default_rng(seed)
    perm = rng.permutation(n_targets)
    line = np.zeros(n_targets, np.int32); sample = np.zeros(n_targets, np.int32)
    i = li = si = 0
    while i < n_targets:
        end = min(n_targets, i + int(rng.integers(1, 41)))
        while i < end:
            send = min(end, i + int(rng.integers(1, 7)))
            line[perm[i:send]] = li; sample[perm[i:send]] = si
            i, si = send, si + 1
        li += 1
    g = capi.TargetGroups.__new__(capi.TargetGroups)
    g.line, g.sample = line, sample
    g.line_hash = np.array([capi.java_string_hash("R%dG%02d_AE_01" % (10 + j % 80, j)) for j in range(li)], np.int32)
    g.sample_hash = np.array([capi.java_string_hash("%d" % (1000000 + 7919 * j)) for j in range(si)], np.int32)
    return g


def host_selection(matches, g, lim):
    """cds_select_best_matches over every mask's slice of the all-pairs output"""
    mask, target, score, mir = matches
    keep = []
    bounds = np.searchsorted(mask, np.arange(a.masks + 1))
    sel = np.zeros(max(len(mask), 1), np.int64)
    cnt = C.c_int64(0)
    lid = np.ascontiguousarray(g.line[target]); sid = np.ascontiguousarray(g.sample[target])
    for m in range(a.masks):
        lo, hi = int(bounds[m]), int(bounds[m + 1])
        if lo == hi:
            continue
        capi._check(capi.lib().cds_select_best_matches(lid[lo:].ctypes.data_as(capi._i32p), sid[lo:].ctypes.data_as(capi._i32p),
                                                       score[lo:].ctypes.data_as(capi._i32p), hi - lo, g.line_hash.ctypes.data_as(capi._i32p),
                                                       len(g.line_hash), g.sample_hash.ctypes.data_as(capi._i32p), len(g.sample_hash),
                                                       *lim, sel.ctypes.data_as(capi._i64p), C.byref(cnt)))
        keep.append(lo + sel[:cnt.value])
    idx = np.concatenate(keep) if keep else np.zeros(0, np.int64)
    return tuple(x[idx] for x in matches)


def timed(fn):
    best, out = None, None
    for _ in range(a.reps):
        t0 = time.perf_counter()
        out = fn()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best, out, ctx.last_stats()


def selection_device_ms(fn):
    import torch
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    total = 0.0
    for ev in prof.key_averages():
        if "bestsel" in ev.key or "cub::" in ev.key:
            total += getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0))
    return total / 1000.0


ctx = capi.Context(device_ids=[0])
rects = O.label_rects(W, H)
gpu = gpu_name()
lib = capi.Library(ctx, W, H, a.targets)
lib.generate_synthetic(SEED, 0, a.targets)
masks = np.concatenate([ctx.synth_rgb(0, SEED, i, min(64, a.masks - i), W, H, on_device=True) for i in range(0, a.masks, 64)])
ms = capi.MaskSet(ctx, W, H, 20, 20, 0.01, 2, True, rects)
ms.add_rgb(masks)
n_files = min(a.tiff_targets, a.targets)
files = []
for i in range(0, n_files, 64):
    files += [capi.tiff_encode_rgb(t, 8, 32773) for t in ctx.synth_rgb(1, SEED, i, min(64, n_files - i), W, H, on_device=True)]
legs = {
    "resident": (groups_for(a.targets), lambda cap: ms.search_matches(lib, a.pct, capacity=cap),
                 lambda g, lim, cap: ms.search_best_matches(lib, g, a.pct, *lim, capacity=cap), a.targets),
    "tiff": (groups_for(n_files), lambda cap: ms.search_stream_matches_tiff(files, a.pct, capacity=cap),
             lambda g, lim, cap: ms.search_stream_best_matches_tiff(files, g, a.pct, *lim, capacity=cap), n_files),
}
for leg, (g, all_pairs, fused, n_targets) in legs.items():
    n_pass = len(all_pairs(None)[0])            # (sizes the outputs, so that the timed calls are not retried)
    t_all, matches, st_all = timed(lambda: all_pairs(max(n_pass, 1)))
    for lim in LIMITS:
        t0 = time.perf_counter()
        exp = host_selection(matches, g, lim)
        t_host_sel = time.perf_counter() - t0
        cap = max(len(exp[0]), 1)
        t_new, got, st_new = timed(lambda: fused(g, lim, cap))
        same = len(got[0]) == len(exp[0]) and all(np.array_equal(x, y) for x, y in zip(got, exp))
        sel_ms = selection_device_ms(lambda: fused(g, lim, cap))
        print(json.dumps({"leg": leg, "masks": a.masks, "targets": n_targets, "pct": a.pct, "limits": lim, "gpu": gpu,
                          "passing_pairs": int(len(matches[0])), "selected_pairs": int(len(got[0])), "equal_to_two_step": bool(same),
                          "two_step_s": round(t_all + t_host_sel, 4), "two_step_search_s": round(t_all, 4), "two_step_host_select_s": round(t_host_sel, 4),
                          "two_step_d2h_bytes": int(st_all["d2h_bytes"]), "fused_s": round(t_new, 4), "fused_d2h_bytes": int(st_new["d2h_bytes"]),
                          "selection_device_ms": round(sel_ms, 3)}), flush=True)
ms.close(); lib.close(); ctx.close()
