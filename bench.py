#!/usr/bin/env python
"""Benchmark of the colour-depth pixel-match hot path (BASELINE.json metric: mask x target CDS comparisons / s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[1], "1,000 EM masks x 100,000 LM targets pixel-match search, 1210x566, on
8xB200", i.e. 12,500 targets per GPU.  100,000 encoded targets do not fit one GPU, so the benchmark is weak-scaled: every
rank holds its own 12,500-target shard (masks replicated, no data-path collective), N = 8 is the full configuration and
N = 1 is one GPU's share of it.  Parameters are the production ones (cdsparams.sh): mask/data threshold 20, zTolerance
0.01, xyShift 2, mirror, top-300 per mask, pctPositivePixels 1.  One step = all masks against the rank's resident
library, per-mask top-K on the device, results on the host.  Inputs are synthetic (cds_synth.h).

One JSON line on stdout (rank 0).  `value` uses device time (CUDA events on the library's launch stream, summed over the
step's kernels, max over ranks); `e2e` is wall clock through the C ABI with host buffers (uploads + encoding + mask
preparation + search + read-back inside the timed region).

--dump-outputs DIR writes what the last timed step returned (rank 0, after the host merge): score, target, mirrored [M, K] and
count [M] of the per-mask top-K (the --impl reference arm: its dense score and mirrored [M, T]).  The inputs are seeded, so two
builds run with the same arguments can be compared file for file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H = 1210, 566
ALGO_BYTES_PER_COMPARISON = 3 * W * H          # SURVEY.md 8(d): the target's RGB bytes as the reference stores them
SEED = 0xC0FFEE
PARAMS = dict(mask_threshold=20, data_threshold=20, z_tolerance=0.01, xy_shift=2, mirror=True)
TOPK = 300
PCT_POSITIVE = 1.0


def label_rects():
    return np.array([[W - 270, 0, W, 90], [0, 0, 330, 100]], np.int32)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons while the timed region runs (NVML in-process; nvidia-smi would do the same query
    but spawning it every 200 ms stalls CUDA calls of this process)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            hnd = nv.nvmlDeviceGetHandleByIndex(self.gpu_index)
            bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                    "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                    "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            mx = nv.nvmlDeviceGetMaxClockInfo(hnd, nv.NVML_CLOCK_SM)
            while not self.stop_flag.is_set():
                sm = nv.nvmlDeviceGetClockInfo(hnd, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(hnd)
                self.samples.append((float(sm), float(mx), [k for k, b in bits.items() if r & b]))
                self.stop_flag.wait(0.1)
        except Exception:
            q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            while not self.stop_flag.is_set():
                try:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                         capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                    self.samples.append((float(out[0]), float(out[1]),
                                         [n for n, v in zip(names, out[2:6]) if v.strip().lower().startswith("active")]))
                except Exception:
                    pass
                self.stop_flag.wait(1.0)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        reasons = sorted({r for s in self.samples for r in s[2]})
        return {"sm_mhz": float(np.median([s[0] for s in self.samples])), "sm_max_mhz": float(max(s[1] for s in self.samples)),
                "reasons": reasons, "samples": len(self.samples)}


def host_threads():
    """All the host threads this process may use (torchrun exports OMP_NUM_THREADS=1, which is not what a CPU baseline wants)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def bind_to_gpu(gpu_index):
    """Moves this rank onto the CPUs next to its GPU (sysfs local_cpulist of the GPU's PCI function) BEFORE it allocates and
    first-touches its pinned buffers, so that host->device uploads of N ranks do not all pull from one NUMA node.  Returns what
    was found, for the JSON line.  Best effort."""
    info = {"bound": False}
    try:
        import pynvml as nv
        nv.nvmlInit()
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(gpu_index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.lower().split(":", 1)
        dev = "/sys/bus/pci/devices/%s:%s" % (dom[-4:], rest)
        info["pci"] = dev.rsplit("/", 1)[1]
        info["numa_node"] = int(open(dev + "/numa_node").read().strip())
        cpus = set()
        for part in open(dev + "/local_cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = (cpus & allowed) or allowed
        info["local_cpus"] = len(cpus)
        info["host_cpus_allowed"] = len(allowed)
        if use != allowed:
            os.sched_setaffinity(0, use)
            info["bound"] = True
        info["cpus_used"] = len(use)
    except Exception as e:
        info["error"] = repr(e)
    return info


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return rank, local_rank, world


def cpu_baseline(masks_host, targets_fn, budget_s=12.0):
    """The oracle (CPU port of the Java algorithm), OpenMP over all host cores, on a bounded sample of the workload:
    32 masks x 1024 targets, repeated until ~budget_s of CPU work has been timed."""
    from oracle import oracle as O
    rects = label_rects()
    cores = host_threads()
    p = PARAMS
    n_m, n_t = min(32, len(masks_host)), 1024
    oms = [O.PixelMatchMask(m, p["mask_threshold"], p["mirror"], p["data_threshold"], p["z_tolerance"], p["xy_shift"], rects)
           for m in masks_host[:n_m]]
    tg = targets_fn(n_t)
    O.search_dense(oms[:2], tg[:64], cores)      # warm the threads
    passes, dt = 0, 0.0
    t0 = time.perf_counter()
    while dt < budget_s and passes < 64:
        O.search_dense(oms, tg, cores)
        passes += 1
        dt = time.perf_counter() - t0
    return {"value": n_m * n_t * passes / dt, "unit": "comparisons/s", "cores": cores, "kind": "port",
            "sample": "%d masks x %d targets of the same synthetic workload x %d passes, %.1f s, OpenMP over targets" % (n_m, n_t, passes, dt)}


def shape_bench(ctx, n_masks=64, n_targets=600, per_mask=300, cpu_pairs=48):
    """BASELINE configs[2] in miniature: shape / area-gap scoring of `per_mask` targets for each of `n_masks` masks
    (thr 20, mirror, zgap derived on the device, synthetic gradient images).  Reports pairs/s of the pair kernel (device
    events), end-to-end pairs/s through cds_shape_score_pairs with host buffers, mask preparation time, and the oracle."""
    from colormipsearch_b200 import capi
    rects = label_rects()
    masks = np.concatenate([ctx.synth_rgb(0, SEED, i, min(64, n_masks - i), W, H, on_device=True) for i in range(0, n_masks, 64)])
    # target and gradient images live in pinned host memory, like the pixel-match e2e leg
    t_arr, t_ptr = ctx.host_alloc(n_targets * 3 * W * H)
    g_arr, g_ptr = ctx.host_alloc(n_targets * 2 * W * H)
    targets = t_arr.reshape(n_targets, H, W, 3)
    grads = g_arr.view(np.uint16).reshape(n_targets, H, W)
    for i in range(0, n_targets, 64):
        n = min(64, n_targets - i)
        targets[i:i + n] = ctx.synth_rgb(1, SEED, i, n, W, H, on_device=True)
        grads[i:i + n] = ctx.synth_gradient(SEED, i, n, W, H, on_device=True)
    # mask preparation: the first call of a size also pays for the device pools' first allocations; the steady figure is a repeat
    prep_first_s = prep_s = None
    for _ in range(2):
        t0 = time.perf_counter()
        sms = capi.ShapeMaskSet(ctx, W, H, 20, True, rects)
        sms.add_rgb(masks)
        prep_s = time.perf_counter() - t0
        if prep_first_s is None:
            prep_first_s = prep_s
            sms.close()
    pm = np.repeat(np.arange(n_masks, dtype=np.int32), per_mask)
    pt = ((pm.astype(np.int64) * 7) + np.tile(np.arange(per_mask, dtype=np.int64) * 2, n_masks)) % n_targets
    sms.score_pairs(targets, grads, None, pm, pt)                                # warm-up: first-use allocations of the pooled buffers
    e2e_s = None
    for _ in range(2):                                                           # the better of two calls (each one complete: H2D .. D2H)
        t0 = time.perf_counter()
        gap, he, mir = sms.score_pairs(targets, grads, None, pm, pt)
        dt = time.perf_counter() - t0
        e2e_s = dt if e2e_s is None else min(e2e_s, dt)
    st = ctx.last_stats()
    # the same call with the targets as PackBits TIFF files (decoded on the device); gradients stay pixels (PNG in the reference)
    from concurrent.futures import ThreadPoolExecutor as _TPE
    with _TPE(max_workers=host_threads()) as ex:
        files = list(ex.map(lambda i: capi.tiff_encode_rgb(targets[i], 8, 32773), range(n_targets)))
    foff = np.zeros(n_targets + 1, np.int64)
    np.cumsum([len(f) for f in files], out=foff[1:])
    f_arr, f_ptr = ctx.host_alloc(int(foff[-1]) + 64)
    for i, f in enumerate(files):
        f_arr[foff[i]:foff[i + 1]] = np.frombuffer(f, np.uint8)
    del files
    sms.score_pairs_tiff((f_arr, foff), grads, None, pm, pt, blob_ptr=f_ptr)
    tiff_s = None
    for _ in range(2):
        t0 = time.perf_counter()
        gap2, he2, mir2 = sms.score_pairs_tiff((f_arr, foff), grads, None, pm, pt, blob_ptr=f_ptr)
        dt = time.perf_counter() - t0
        tiff_s = dt if tiff_s is None else min(tiff_s, dt)
    tiff_same = bool(np.array_equal(gap2, gap) and np.array_equal(he2, he) and np.array_equal(mir2, mir))
    ctx.host_free(f_ptr)
    n_pairs = len(pm)
    bytes_per_pair = 3 * W * H + 2 * W * H + 3 * W * H          # SURVEY 8(d): target RGB + gradient + zgap RGB
    peak, peak_src = measured_peak()
    kernel_pairs_s = n_pairs / (st["match_kernel_ms"] * 1e-3)
    out = {"metric": "shape-score pairs/sec", "pairs": n_pairs, "masks": n_masks, "targets": n_targets,
           "value": kernel_pairs_s, "unit": "pairs/s", "kernel_ms": st["match_kernel_ms"],
           "e2e": {"value": n_pairs / e2e_s, "unit": "pairs/s", "ms": e2e_s * 1e3,
                   "h2d_bytes": int(n_targets * (3 * W * H + 2 * W * H)), "what": "cds_shape_score_pairs: H2D of targets + gradients, "
                   "zgap = maxFilter(10) on device, slice planes, pair kernel, D2H"},
           "e2e_tiff": {"value": n_pairs / tiff_s, "unit": "pairs/s", "ms": tiff_s * 1e3,
                        "h2d_bytes": int(foff[-1]) + int(n_targets * 2 * W * H), "equals_pixel_call": tiff_same,
                        "what": "cds_shape_score_pairs_tiff: targets as PackBits TIFF files decoded on the device, gradients as pixels"},
           "mask_prep_ms_per_mask": prep_s / n_masks * 1e3, "mask_prep_first_use_ms_per_mask": prep_first_s / n_masks * 1e3,
           "roofline": shape_roofline(kernel_pairs_s, bytes_per_pair, peak, peak_src)}
    # oracle on a few pairs, one pair per host thread
    if cpu_pairs <= 0:
        sms.close()
        del targets, grads
        ctx.host_free(t_ptr)
        ctx.host_free(g_ptr)
        return out
    try:
        from concurrent.futures import ThreadPoolExecutor
        from oracle import oracle as O
        cores = host_threads()
        n_cm = 2
        oms = [O.ShapeMask(masks[i], 20, True, rects) for i in range(n_cm)]
        zg = [O.make_zgap(targets[int(pt[i])], 20, rects) for i in range(cpu_pairs)]

        def one(i):
            return oms[i % n_cm].score(targets[int(pt[i])], grads[int(pt[i])], zg[i])

        t0 = time.perf_counter()
        with ThreadPoolExecutor(cores) as ex:
            res = list(ex.map(one, range(cpu_pairs)))
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": cpu_pairs / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
                               "sample": "%d pairs (zgap images prepared outside the timed region), one pair per host thread" % cpu_pairs}
        # parity spot check of the bench itself
        for i in range(min(cpu_pairs, 8)):
            m = i % n_cm
            j = int(np.nonzero((pm == m) & (pt == pt[i]))[0][0]) if ((pm == m) & (pt == pt[i])).any() else None
            if j is not None:
                assert (int(gap[j]), int(he[j]), bool(mir[j])) == res[i], "shape bench parity"
    except Exception as e:  # the baseline is reporting only
        out["cpu_baseline"] = {"error": str(e)}
    sms.close()
    del targets, grads
    ctx.host_free(t_ptr)
    ctx.host_free(g_ptr)
    return out


def shape_roofline(kernel_pairs_s, bytes_per_pair, peak, peak_src):
    """The shape step's device time is the per-TARGET kernel (zgap dilation + slice planes), not the pair kernel: both are reported
    with their physical DRAM traffic from the ncu capture named in profiles/ncu_shape.json."""
    nc = {}
    try:
        nc = json.load(open(os.path.join(ROOT, "profiles", "ncu_shape.json")))
    except Exception:
        pass
    dk, pk = nc.get("shape_target_derive_kernel", {}), nc.get("shape_pair_kernel", {})
    out = {"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_src, "counters_source": nc.get("source"),
           "kernel": "shape_pair_kernel", "algorithmic_bytes_per_pair": bytes_per_pair,
           "achieved_algorithmic": kernel_pairs_s * bytes_per_pair / 1e9, "frac_algorithmic": kernel_pairs_s * bytes_per_pair / 1e9 / peak,
           "note": "frac is physical: ncu DRAM bytes per pair x pairs/s of the pair kernel / HBM copy peak (the kernel gathers the query's "
                   "non-black pixels, ~1-3 % of each plane; frac_algorithmic counts target RGB + gradient + zgap RGB per pair, SURVEY 8d)"}
    if pk.get("dram_bytes_per_pair"):
        out["traffic_per_pair"] = pk["dram_bytes_per_pair"]
        out["achieved"] = kernel_pairs_s * pk["dram_bytes_per_pair"] / 1e9
        out["frac"] = out["achieved"] / peak
    else:
        out["achieved"] = out["frac"] = None
    if dk:
        # the per-target kernel at the rate the capture ran it (32 targets per launch)
        tps = dk["targets_per_launch"] / (dk["ncu_us_per_launch"] * 1e-6)
        out["target_kernel"] = {"kernel": "shape_target_derive_kernel", "targets_per_s_in_capture": tps,
                                "dram_gbs": tps * dk["dram_bytes_per_target"] / 1e9, "frac": tps * dk["dram_bytes_per_target"] / 1e9 / peak,
                                "issue_active": dk["issue_active"], "warp_inst_per_target": dk["warp_inst_per_target"],
                                "note": "issue-bound (VIMNMX3 / shuffle / PRMT), not HBM-bound"}
    return out


def shape_config2_mix(ctx, topk, n_masks, t_first, t_limit=4096, inflate_windows=(0,)):
    """BASELINE configs[2] with its REAL pair mix: the pairs are the top-300 isMatch targets of every mask from the pixel-match
    step this bench has just run (about 8 pairs per target, not 32), restricted to the first `t_limit` targets of the shard so
    that targets + gradients fit comfortably in pinned host memory.  End to end through cds_shape_score_pairs(_tiff) with host buffers."""
    from concurrent.futures import ThreadPoolExecutor
    from colormipsearch_b200 import capi
    rects = label_rects()
    score, target, mirrored, count = topk
    pm = np.repeat(np.arange(n_masks, dtype=np.int32), count[:n_masks])
    pt = np.concatenate([target[m, :count[m]] for m in range(n_masks)]).astype(np.int64)
    keep = pt < t_limit
    pm, pt = pm[keep], pt[keep]
    n_pairs, n_t = len(pm), t_limit
    if n_pairs == 0:
        return {"error": "no pairs"}
    masks = np.concatenate([ctx.synth_rgb(0, SEED, i, min(64, n_masks - i), W, H, on_device=True) for i in range(0, n_masks, 64)])
    t_arr, t_ptr = ctx.host_alloc(n_t * 3 * W * H)
    g_arr, g_ptr = ctx.host_alloc(n_t * 2 * W * H)
    targets = t_arr.reshape(n_t, H, W, 3)
    grads = g_arr.view(np.uint16).reshape(n_t, H, W)
    for i in range(0, n_t, 64):
        n = min(64, n_t - i)
        targets[i:i + n] = ctx.synth_rgb(1, SEED, t_first + i, n, W, H, on_device=True)
        grads[i:i + n] = ctx.synth_gradient(SEED, t_first + i, n, W, H, on_device=True)
    m_arr, m_ptr = ctx.host_alloc(n_masks * 3 * W * H)
    np.copyto(m_arr, masks.reshape(-1))
    sms = capi.ShapeMaskSet(ctx, W, H, 20, True, rects)
    sms.add_rgb(masks[:64])                                                       # warm-up: pooled buffers
    sms.close()
    prep_first_s = prep_s = None
    for _ in range(2):                                                            # the first call of this size grows the device pools
        t0 = time.perf_counter()
        sms = capi.ShapeMaskSet(ctx, W, H, 20, True, rects)
        sms.add_rgb_ptr(m_ptr, n_masks)
        prep_s = time.perf_counter() - t0
        if prep_first_s is None:
            prep_first_s = prep_s
            sms.close()
    sms.score_pairs(targets[:64], grads[:64], None, pm[:8] * 0, pt[:8] % 64)      # warm-up
    best = None
    for _ in range(2):
        t0 = time.perf_counter()
        gap, he, mir = sms.score_pairs(targets, grads, None, pm, pt)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    st = ctx.last_stats()
    with ThreadPoolExecutor(max_workers=host_threads()) as ex:
        files = list(ex.map(lambda i: capi.tiff_encode_rgb(targets[i], 8, 32773), range(n_t)))
    foff = np.zeros(n_t + 1, np.int64)
    np.cumsum([len(f) for f in files], out=foff[1:])
    f_arr, f_ptr = ctx.host_alloc(int(foff[-1]) + 64)
    for i, f in enumerate(files):
        f_arr[foff[i]:foff[i + 1]] = np.frombuffer(f, np.uint8)
    del files
    sms.score_pairs_tiff((f_arr, foff), grads, None, pm[:64], pt[:64], blob_ptr=f_ptr)
    best_t = None
    for _ in range(2):
        t0 = time.perf_counter()
        gap2, he2, mir2 = sms.score_pairs_tiff((f_arr, foff), grads, None, pm, pt, blob_ptr=f_ptr)
        dt = time.perf_counter() - t0
        best_t = dt if best_t is None else min(best_t, dt)
    st_t = ctx.last_stats()
    same = bool(np.array_equal(gap2, gap) and np.array_equal(he2, he) and np.array_equal(mir2, mir))
    # the same pairs with BOTH inputs as files, the way gradientScores meets them on disk: targets as PackBits TIFF, gradients as 16-bit
    # PNG.  Writing PNG files is host work outside the timed region (70 ms each), so only P distinct gradient files are written and target
    # i gets file i % P; the scores are checked against the pixel call on the targets below P and between the two inflate paths on all.
    # Gradient streams are inflated on the device (one warp per stream) or, for comparison, by host threads (zlib).
    n_f, P = min(n_t, 4096), min(n_t, 512)
    kf = pt < n_f
    files_leg = None
    if kf.sum() >= 64:
        with ThreadPoolExecutor(max_workers=host_threads()) as ex:
            pngs = list(ex.map(lambda i: capi.png_encode_gray16(grads[i], 2), range(P)))
        poff = np.zeros(n_f + 1, np.int64)
        np.cumsum([len(pngs[i % P]) for i in range(n_f)], out=poff[1:])
        p_arr, p_ptr = ctx.host_alloc(int(poff[-1]) + 64)
        for i in range(n_f):
            p_arr[poff[i]:poff[i + 1]] = np.frombuffer(pngs[i % P], np.uint8)
        del pngs
        tsub = (f_arr[:int(foff[n_f])], foff[:n_f + 1])
        psub = (p_arr[:int(poff[-1])], poff)
        in_p = pt[kf] < P
        files_leg = {"pairs": int(kf.sum()), "targets": int(n_f), "distinct_gradient_files": int(P), "png_bytes_mean": float(poff[-1]) / n_f,
                     "tiff_bytes_mean": float(foff[n_f]) / n_f}
        res = {}
        legs = [(1, w, "device_inflate" if w == 0 else "device_inflate_window_%d" % w) for w in inflate_windows] + [(0, 0, "host_inflate")]
        for mode, window, key in legs:
            ctx.set_option("device_inflate", mode)
            ctx.set_option("shape_inflate_window", window)
            sms.score_pairs_files(tsub, psub, None, pm[kf][:64], pt[kf][:64])
            best_f = None
            for _ in range(2):
                t0 = time.perf_counter()
                res[key] = sms.score_pairs_files(tsub, psub, None, pm[kf], pt[kf])
                dt = time.perf_counter() - t0
                best_f = dt if best_f is None else min(best_f, dt)
            st_f = ctx.last_stats()
            gap3, he3, mir3 = res[key]
            files_leg[key] = {"value": int(kf.sum()) / best_f, "unit": "pairs/s", "ms": best_f * 1e3, "h2d_bytes": int(st_f["h2d_bytes"]),
                              "targets_per_s": int(len(np.unique(pt[kf]))) / best_f, "host_inflate_fallbacks": int(st_f["host_inflate_fallbacks"]),
                              "equals_pixel_call_below_P": bool(np.array_equal(gap3[in_p], gap[kf][in_p]) and np.array_equal(he3[in_p], he[kf][in_p])
                                                                and np.array_equal(mir3[in_p], mir[kf][in_p]))}
        files_leg["inflate_paths_agree"] = bool(all(np.array_equal(x, y) for x, y in zip(res["device_inflate"], res["host_inflate"])))
        ctx.set_option("device_inflate", 1)
        ctx.set_option("shape_inflate_window", 0)
        ctx.host_free(p_ptr)
    n_active = int(len(np.unique(pt)))
    out = {"pairs": int(n_pairs), "distinct_targets": n_active, "masks": n_masks,
           "e2e": {"value": n_pairs / best, "unit": "pairs/s", "ms": best * 1e3, "h2d_bytes": int(st["h2d_bytes"]),
                   "h2d_gbs": st["h2d_bytes"] / best / 1e9},
           "e2e_tiff": {"value": n_pairs / best_t, "unit": "pairs/s", "ms": best_t * 1e3, "h2d_bytes": int(st_t["h2d_bytes"]),
                        "h2d_gbs": st_t["h2d_bytes"] / best_t / 1e9, "equals_pixel_call": same},
           "e2e_files": files_leg,
           "pair_kernel_ms": st["match_kernel_ms"], "pair_kernel_pairs_per_s": n_pairs / (st["match_kernel_ms"] * 1e-3),
           "mask_prep_ms_per_mask": prep_s / n_masks * 1e3, "mask_prep_first_use_ms_per_mask": prep_first_s / n_masks * 1e3,
           "mask_prep_h2d_bytes_per_mask": 3 * W * H,
           "what": "pairs = top-300 isMatch targets per mask from this run's pixel-match search, targets < %d; only targets with pairs are "
                   "uploaded (RGB or TIFF file + gray16 gradient, or TIFF + PNG files in e2e_files), zgap dilation + slice planes + pair kernel per window of "
                   "32 / 128 targets (up to 2048 when the gradient PNG streams are inflated on the device)" % t_limit}
    sms.close()
    del targets, grads
    for q in (t_ptr, g_ptr, m_ptr, f_ptr):
        ctx.host_free(q)
    return out


def data_dependence(ctx, masks_synth, n_masks=1000, n_targets=1024, reps=3):
    """The candidate kernel's speed depends on the data (its ticket tests skip mask tiles where the target has nothing in that
    colour sector), so the headline workload is not the whole story.  Two more settings at reduced size, each with its own
    comparisons/s (device time of cds_search_topk over a resident library) and an oracle check of sampled cells:
      real_fixture     masks = the reference's three EM fixtures, targets = its four LM fixtures, label regions cleared, replicated
                       with translation (and brightness scaling for the targets) jitter
      dense_synthetic  the synthetic masks against targets that overlay six synthetic targets each (~20-30 % of the pixels lit)
      reverse_search   the LM fixtures (brightness-scaled: tens of thousands of colour classes per mask group) as masks against the
                       EM fixtures as targets -- the word lists then carry rank intervals instead of palette references"""
    from colormipsearch_b200 import capi
    from oracle import oracle as O
    rects = label_rects()
    p = PARAMS
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

    def leg(masks, targets, what):
        lib = capi.Library(ctx, W, H, len(targets))
        for i in range(0, len(targets), 256):
            lib.add_rgb(targets[i:i + 256])
        ms = capi.MaskSet(ctx, W, H, p["mask_threshold"], p["data_threshold"], p["z_tolerance"], p["xy_shift"], p["mirror"], rects)
        sizes = np.concatenate([ms.add_rgb(masks[i:i + 64]) for i in range(0, len(masks), 64)])
        ms.search_topk(lib, TOPK, PCT_POSITIVE)
        dev_ms, kern = 0.0, 0
        for _ in range(reps):
            res = ms.search_topk(lib, TOPK, PCT_POSITIVE)
            st = ctx.last_stats()
            dev_ms += st["total_device_ms"]
            kern = st["match_kernel"]
        # oracle: 4 masks x 8 targets, every cell
        pm = np.sort(rng.choice(len(masks), 4, replace=False))
        pt = np.sort(rng.choice(len(targets), 8, replace=False))
        sub = capi.MaskSet(ctx, W, H, p["mask_threshold"], p["data_threshold"], p["z_tolerance"], p["xy_shift"], p["mirror"], rects)
        sub.add_rgb(masks[pm])
        dense, dmir = sub.search_dense(lib)
        sub.close()
        oms = [O.PixelMatchMask(masks[i], p["mask_threshold"], p["mirror"], p["data_threshold"], p["z_tolerance"], p["xy_shift"], rects) for i in pm]
        es, em, _ = O.search_dense(oms, targets[pt])
        ok = bool(np.array_equal(dense[:, pt], es) and np.array_equal(dmir[:, pt], em))
        lit = float(np.mean([(t.max(axis=2) > p["data_threshold"]).mean() for t in targets[:: max(1, len(targets) // 32)]]))
        out = {"value": len(masks) * len(targets) * reps / (dev_ms * 1e-3), "unit": "comparisons/s", "masks": len(masks), "targets": len(targets),
               "ms_per_search": dev_ms / reps, "match_kernel": {1: "candidate", 2: "band", 3: "gather"}.get(kern, "?"),
               "target_pixels_above_threshold": lit, "mask_pixels_mean": float(np.mean(sizes)),
               "matches_returned": int(res[3].sum()), "equals_oracle_on_sampled_cells": ok, "what": what}
        ms.close()
        lib.close()
        return out

    legs = {}
    em = [clear(fx[k]) for k in ("em_12191", "em_12191_FL", "em_LPLC2")]
    lm = [clear(fx[k]) for k in ("lm_BJD", "lm_GMR", "lm_VT016795", "lm_VT033614")]
    masks = np.stack([jitter(em[i % 3], 1.0) for i in range(n_masks)])
    targets = np.stack([jitter(lm[i % 4], float(rng.uniform(0.5, 1.0))) for i in range(n_targets)])
    legs["real_fixture"] = leg(masks, targets, "the reference's EM / LM fixture images (labels cleared), replicated with jitter")
    n_rev = max(16, min(128, n_masks // 8))
    legs["reverse_search"] = leg(targets[:n_rev], masks,
                                 "the LM fixture images (brightness-scaled, jittered) as %d masks x the EM fixture images as targets" % n_rev)
    del masks, targets
    base = np.concatenate([ctx.synth_rgb(1, SEED, 100000 + i, min(64, 6 * 128 - i), W, H, on_device=True) for i in range(0, 6 * 128, 64)])
    pool = []
    for i in range(128):
        out = base[6 * i].copy()
        for k in range(1, 6):
            nxt = base[6 * i + k]
            empty = ~out.any(axis=2)
            out[empty] = nxt[empty]
        pool.append(out)
    del base
    targets = np.stack([jitter(pool[i % 128], 1.0) for i in range(n_targets)])
    legs["dense_synthetic"] = leg(masks_synth[:n_masks], targets, "synthetic masks x overlays of six synthetic targets each, replicated with jitter")
    return legs


def pair_provider_bench(ctx, masks_host, n_masks=64, n_targets=256, threads=40):
    """The reference's own calling convention: ColorDepthSearchAlgorithm.calculateMatchingScore, one (mask, target) pair per call,
    from a pool of ~40 threads (LocalColorMIPSearchProcessor.java:93-105; 2 x cores - 1 = 39 workers in submitCDSJob.sh), the same
    target images recurring across masks.  Here: cds_pairq_score driven by `threads` native threads (cds_debug_pairq_drive), mask by
    mask over all targets like the reference's loop.  `cold` includes uploading + encoding every target once; `warm` finds them all
    in the device cache (the reference keeps its targets in a 100 000-image cache)."""
    from colormipsearch_b200 import capi
    rects = label_rects()
    p = PARAMS
    ms = capi.MaskSet(ctx, W, H, p["mask_threshold"], p["data_threshold"], p["z_tolerance"], p["xy_shift"], p["mirror"], rects)
    ms.add_rgb(masks_host[:n_masks])
    targets = np.concatenate([ctx.synth_rgb(1, SEED, i, min(64, n_targets - i), W, H, on_device=True) for i in range(0, n_targets, 64)])
    lib = capi.Library(ctx, W, H, n_targets)
    lib.add_rgb(targets)
    dense, dmir = ms.search_dense(lib)
    lib.close()
    pm = np.repeat(np.arange(n_masks, dtype=np.int32), n_targets)
    pt = np.tile(np.arange(n_targets, dtype=np.int64), n_masks)
    keys = np.arange(n_targets, dtype=np.uint64) + 1
    q = capi.PairQueue(ctx, ms, max_batch=128, max_wait_us=60, cache_targets=max(512, 2 * n_targets))
    sc, mir, cold_s = q.drive(targets, keys, pm, pt, threads)
    st_cold = q.stats()
    sc2, mir2, warm_s = q.drive(targets, keys, pm, pt, threads)
    st = q.stats()
    ok = bool(np.array_equal(sc, dense[pm, pt]) and np.array_equal(sc2, dense[pm, pt]) and np.array_equal(mir2, dmir[pm, pt].astype(bool)))
    # the same with twice the callers (the reference sizes its pool by the host: 2 x cores - 1 threads)
    sc3, mir3, warm2_s = q.drive(targets, keys, pm, pt, 2 * threads)
    ok = ok and bool(np.array_equal(sc3, dense[pm, pt]))
    q.close()
    ms.close()
    n = len(pm)
    return {"metric": "single-pair calls/sec through cds_pairq_score", "threads": threads, "masks": n_masks, "targets": n_targets, "pairs": n,
            "warm_twice_the_threads": {"value": n / warm2_s, "unit": "pairs/s", "threads": 2 * threads},
            "cold": {"value": n / cold_s, "unit": "pairs/s", "uploads": st_cold["uploads"], "batches": st_cold["batches"]},
            "warm": {"value": n / warm_s, "unit": "pairs/s", "uploads": st["uploads"] - st_cold["uploads"], "batches": st["batches"] - st_cold["batches"],
                     "mean_batch": n / max(1, st["batches"] - st_cold["batches"])},
            "equals_dense_search": ok,
            "what": "blocking single-pair calls from %d native threads, micro-batched into one kernel launch per batch; targets keyed like the "
                    "reference's image cache" % threads}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  The reference is Java and there is no JVM on
    this image, so this is the oracle port (oracle/cds_oracle.c, pinned on the reference's golden vectors) on all host
    cores; each step is a bounded sample of the workload.  Nothing here maps the GPU library: the synthetic inputs come from
    the host-only build of the generator (oracle/synth_host.cpp)."""
    rank, local_rank, world = dist_env()
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as O
    from oracle import synth as S
    rects = label_rects()
    cores = host_threads()
    p = PARAMS
    n_m, n_t = args.ref_masks, max(args.ref_targets, cores)

    def gen(kind, n):
        chunks = [(i, min(8, n - i)) for i in range(0, n, 8)]
        with ThreadPoolExecutor(cores) as ex:
            return np.concatenate(list(ex.map(lambda c: S.synth_rgb(kind, SEED, c[0], c[1], W, H), chunks)))

    masks = gen(0, n_m)
    targets = gen(1, n_t)
    oms = [O.PixelMatchMask(m, p["mask_threshold"], p["mirror"], p["data_threshold"], p["z_tolerance"], p["xy_shift"], rects)
           for m in masks]
    for _ in range(args.warmup):
        O.search_dense(oms[:4], targets[: max(cores, 8)], cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        scores, mirrored, _ = O.search_dense(oms, targets, cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"score": scores, "mirrored": mirrored})
    value = n_m * n_t * args.steps / dt
    sample = "%d masks x %d targets per step (bounded sample of the workload), OpenMP over targets" % (n_m, n_t)
    cfg = workload_config(args, world)
    cfg["workload"] += "; THIS ARM: CPU port timed on a bounded sample of it, %d masks x %d targets per step" % (n_m, n_t)
    cfg["sample"] = {"masks": n_m, "targets": n_t}
    line = {
        "impl": "reference", "metric": "mask x target CDS comparisons/sec", "value": value, "unit": "comparisons/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": "comparisons/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "comparisons/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_library_mapped": "libcdsgpu" in open("/proc/self/maps").read(),
        "note": "Java reference cannot run here (no JVM); this is the C port of its algorithm pinned on its golden vectors",
    }
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays):
    """Writes the last timed step's per-mask result arrays (`name` -> array, one row per mask) as out_dir/<name>.npy in float64,
    so that two builds can be compared output for output.  When they would exceed DUMP_LIMIT_BYTES, a fixed sample of mask rows
    (seeded, sorted) is written instead; mask_index.npy always names the rows written."""
    n = len(next(iter(arrays.values())))
    row_bytes = sum(8 * int(np.prod(a.shape[1:])) for a in arrays.values()) + 8
    budget = DUMP_LIMIT_BYTES - 1024 * (len(arrays) + 1)          # room for the .npy headers
    rows = np.arange(n)
    if n * row_bytes > budget:
        rows = np.sort(np.random.default_rng(SEED).choice(n, budget // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "mask_index.npy"), rows.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a)[rows].astype(np.float64))


def workload_config(args, world):
    return {
        "workload": "BASELINE configs[1]: %d masks x %d targets per GPU (x%d GPUs = %d targets), 1210x566, maskThr 20, dataThr 20, "
                    "zTol 0.01, xyShift 2, mirror (18 variants), top-%d per mask, pctPositivePixels %g"
                    % (args.masks, args.targets_per_gpu, world, args.targets_per_gpu * world, TOPK, PCT_POSITIVE),
        "masks": args.masks, "targets_per_gpu": args.targets_per_gpu, "image": [W, H],
        "parallelism": "targets sharded over %d GPU(s), masks replicated, host merge, no collective" % world,
        "l2": "library shard (%.1f GB) is far larger than L2; every step re-streams it" % (args.targets_per_gpu * 2.79e-3),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--masks", type=int, default=1000)
    ap.add_argument("--targets-per-gpu", type=int, default=12500)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--e2e-targets", type=int, default=0, help="targets per e2e step (0 = same as --targets-per-gpu)")
    ap.add_argument("--ref-masks", type=int, default=32)
    ap.add_argument("--ref-targets", type=int, default=1024)
    ap.add_argument("--kernel", default="auto", choices=["auto", "cand", "band"], help="batched match kernel (auto = candidate kernel)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-e2e-tiff", action="store_true", help="skip the TIFF-file variant of the end-to-end step")
    ap.add_argument("--e2e-tiff", action="store_true", help="(default now) the TIFF-file variant of the end-to-end step runs at every N")
    ap.add_argument("--no-shape", action="store_true")
    ap.add_argument("--no-pair-provider", action="store_true", help="skip the single-pair (micro-batching queue) leg")
    ap.add_argument("--no-bind", action="store_true", help="do not move the rank onto the CPUs next to its GPU")
    ap.add_argument("--no-data-dependence", action="store_true", help="skip the real-fixture / dense-target legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)

    if args.impl == "reference":
        run_reference(args)
        return

    rank, local_rank, world = dist_env()
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    binding = bind_to_gpu(local_rank) if not args.no_bind else {"bound": False, "disabled": True}
    from colormipsearch_b200 import capi
    ctx = capi.Context(device_ids=[local_rank])
    ctx.set_match_kernel(args.kernel)
    rects = label_rects()
    M, T = args.masks, args.targets_per_gpu
    t_first = rank * T                       # this rank's shard of the synthetic target numbering

    # ---- resident inputs: synthetic library generated on the device, masks generated on the device and prepared
    t0 = time.perf_counter()
    lib = capi.Library(ctx, W, H, T)
    lib.generate_synthetic(SEED, t_first, T)
    masks_host = np.concatenate([ctx.synth_rgb(0, SEED, i, min(64, M - i), W, H, on_device=True) for i in range(0, M, 64)])
    ms = capi.MaskSet(ctx, W, H, PARAMS["mask_threshold"], PARAMS["data_threshold"], PARAMS["z_tolerance"], PARAMS["xy_shift"],
                      PARAMS["mirror"], rects)
    mask_sizes = ms.add_rgb(masks_host)
    setup_s = time.perf_counter() - t0

    def step():
        out = ms.search_topk(lib, TOPK, PCT_POSITIVE)
        return out, ctx.last_stats()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    dev_ms, match_ms, launches, match_launches, kernel_used = 0.0, 0.0, 0, 0, 0
    t0 = time.perf_counter()
    last = None
    for _ in range(args.steps):
        last, st = step()
        dev_ms += st["total_device_ms"]
        match_ms += st["match_kernel_ms"]
        launches += st["kernel_launches"]
        match_launches += st["match_kernel_launches"]
        kernel_used = st["match_kernel"]
    barrier()
    wall_s = time.perf_counter() - t0
    sampler.stop_flag.set()
    sampler.join()

    # the job's result: per-rank top-K lists merged on the host (rank 0); no data-path collective
    from colormipsearch_b200 import sharding
    merged = None
    if world > 1:
        merged = sharding.gather_and_merge_topk(last, TOPK, t_first)
    elif last is not None:
        merged = last
    if args.dump_outputs and merged is not None:
        score, target, mirrored, count = merged
        dump_outputs(args.dump_outputs, {"score": score, "target": target, "mirrored": mirrored, "count": count})

    # max over ranks of the device time
    times = torch.tensor([dev_ms, match_ms, wall_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, match_ms, wall_ms = [float(x) for x in times.tolist()]
    comparisons_per_step = M * T * world
    value = comparisons_per_step * args.steps / (dev_ms * 1e-3)

    # ---- end to end through the C ABI with host buffers (pinned), every step: upload + encode targets, upload +
    # prepare masks, search, top-K back on the host
    e2e = None
    if not args.no_e2e:
        Te = args.e2e_targets or T
        img_bytes = 3 * W * H
        avail = 0
        try:
            for ln in open("/proc/meminfo"):
                if ln.startswith("MemAvailable"):
                    avail = int(ln.split()[1]) * 1024
        except Exception:
            pass
        pool_t = Te
        budget = int(avail * 0.5 / max(world, 1)) if avail else 8 << 30
        if pool_t * img_bytes > budget:
            pool_t = max(64, budget // img_bytes // 64 * 64)
        pool_arr, pool_ptr = ctx.host_alloc(pool_t * img_bytes)
        mask_arr, mask_ptr = ctx.host_alloc(M * img_bytes)
        np.copyto(mask_arr, masks_host.reshape(-1))
        for i in range(0, pool_t, 64):
            n = min(64, pool_t - i)
            pool_arr[i * img_bytes:(i + n) * img_bytes] = ctx.synth_rgb(1, SEED, t_first + i, n, W, H, on_device=True).reshape(-1)
        lib.close()
        ms.close()
        barrier()
        e2e_steps = max(1, args.e2e_steps)
        import ctypes
        from colormipsearch_b200 import sharding as _sh
        phases = {"masks_h2d_prepare": 0.0, "stream_search": 0.0, "destroy": 0.0}

        def e2e_step():
            ta = time.perf_counter()
            ms_e = capi.MaskSet(ctx, W, H, PARAMS["mask_threshold"], PARAMS["data_threshold"], PARAMS["z_tolerance"],
                                PARAMS["xy_shift"], PARAMS["mirror"], rects)
            ms_e.add_rgb_ptr(mask_ptr, M)
            tb = time.perf_counter(); phases["masks_h2d_prepare"] += tb - ta
            parts, done = [], 0
            while done < Te:                      # one call when the pinned pool holds the whole step (the normal case)
                n = min(pool_t, Te - done)
                sc, tg, mi, cn = ms_e.search_stream(pool_ptr, TOPK, PCT_POSITIVE, n=n)
                parts.append((sc, np.where(tg >= 0, tg + done, -1), mi, cn))
                done += n
            res = parts[0] if len(parts) == 1 else _sh.merge_topk(parts, TOPK)
            tc = time.perf_counter(); phases["stream_search"] += tc - tb
            ms_e.close()
            phases["destroy"] += time.perf_counter() - tc
            return res

        e2e_step()                                 # untimed: first-use allocations of the streaming buffers
        for kph in phases:
            phases[kph] = 0.0
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            res = e2e_step()
        barrier()
        e2e_s = time.perf_counter() - t0
        te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_s = float(te.item())
        d2h = M * TOPK * 8 + M * 4
        e2e_equal = None
        if last is not None and Te == T:
            e2e_equal = bool(np.array_equal(res[3], last[3]) and all(
                np.array_equal(res[i][m, :res[3][m]], last[i][m, :last[3][m]]) for i in range(3) for m in range(0, M, max(1, M // 64))))
        e2e = {"value": M * Te * world * e2e_steps / e2e_s, "unit": "comparisons/s",
               "h2d_bytes_per_step": (Te + M) * img_bytes * world, "d2h_bytes_per_step": d2h * world,
               "steps": e2e_steps, "ms_per_step": e2e_s / e2e_steps * 1e3, "targets_per_gpu": Te,
               "pinned_pool_targets": pool_t, "phase_ms_per_step": {k: v / e2e_steps * 1e3 for k, v in phases.items()},
               "equals_resident_search": e2e_equal,
               "what": "every step, from pinned HOST buffers through the C ABI: cds_maskset_create + cds_maskset_add_rgb (H2D + mask "
                       "preparation) + cds_search_stream_rgb (chunked H2D of the targets overlapping encode + match + top-K, "
                       "result D2H, host merge) + destroy"}
        # ---- the same step with the targets as PackBits TIFF FILES in pinned host memory (how colour-depth MIP libraries are
        # stored; SURVEY 8f row f4): the files cross PCIe as they are and are decoded on the device
        if not args.no_e2e_tiff:
            from concurrent.futures import ThreadPoolExecutor
            t_enc = time.perf_counter()
            # the files are written from the pinned pool where it holds the whole step, otherwise chunk by chunk from the generator: the
            # TIFF leg needs 1.7 GB of host memory per rank, whatever the pixel leg could get
            files = []
            with ThreadPoolExecutor(max_workers=host_threads()) as ex:
                if pool_t >= Te:
                    pool_img = pool_arr[:Te * img_bytes].reshape(Te, H, W, 3)
                    files = list(ex.map(lambda i: capi.tiff_encode_rgb(pool_img[i], 8, 32773), range(Te)))
                else:
                    for i in range(0, Te, 64):
                        blk = ctx.synth_rgb(1, SEED, t_first + i, min(64, Te - i), W, H, on_device=True)
                        files += list(ex.map(lambda im: capi.tiff_encode_rgb(im, 8, 32773), blk))
            offsets = np.zeros(Te + 1, np.int64)
            np.cumsum([len(f) for f in files], out=offsets[1:])
            blob_arr, blob_ptr = ctx.host_alloc(int(offsets[-1]) + 64)
            for i, f in enumerate(files):
                blob_arr[offsets[i]:offsets[i + 1]] = np.frombuffer(f, np.uint8)
            del files
            with ThreadPoolExecutor(max_workers=host_threads()) as ex:
                mfiles = list(ex.map(lambda i: capi.tiff_encode_rgb(masks_host[i], 8, 32773), range(M)))
            moffsets = np.zeros(M + 1, np.int64)
            np.cumsum([len(f) for f in mfiles], out=moffsets[1:])
            mblob_arr, mblob_ptr = ctx.host_alloc(int(moffsets[-1]) + 64)
            for i, f in enumerate(mfiles):
                mblob_arr[moffsets[i]:moffsets[i + 1]] = np.frombuffer(f, np.uint8)
            del mfiles
            enc_s = time.perf_counter() - t_enc
            tphases = {"masks_h2d_prepare": 0.0, "stream_search": 0.0, "destroy": 0.0}

            def e2e_tiff_step():
                ta = time.perf_counter()
                ms_e = capi.MaskSet(ctx, W, H, PARAMS["mask_threshold"], PARAMS["data_threshold"], PARAMS["z_tolerance"],
                                    PARAMS["xy_shift"], PARAMS["mirror"], rects)
                ms_e.add_tiff((mblob_arr, moffsets), blob_ptr=mblob_ptr)
                tb = time.perf_counter(); tphases["masks_h2d_prepare"] += tb - ta
                r = ms_e.search_stream_tiff((blob_arr, offsets), TOPK, PCT_POSITIVE, blob_ptr=blob_ptr)
                tc = time.perf_counter(); tphases["stream_search"] += tc - tb
                ms_e.close()
                tphases["destroy"] += time.perf_counter() - tc
                return r

            e2e_tiff_step()
            for kph in tphases:
                tphases[kph] = 0.0
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                rt = e2e_tiff_step()
            barrier()
            tiff_s = time.perf_counter() - t0
            tt = torch.tensor([tiff_s], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            tiff_s = float(tt.item())
            same = bool(np.array_equal(rt[3], res[3]) and all(np.array_equal(rt[i][m, :rt[3][m]], res[i][m, :res[3][m]])
                                                              for i in range(3) for m in range(0, M, max(1, M // 64))))
            e2e["tiff"] = {"value": M * Te * world * e2e_steps / tiff_s, "unit": "comparisons/s",
                           "h2d_bytes_per_step": (int(offsets[-1]) + int(moffsets[-1])) * world, "d2h_bytes_per_step": d2h * world,
                           "ms_per_step": tiff_s / e2e_steps * 1e3, "file_bytes_mean": float(offsets[-1]) / Te,
                           "compression_ratio": Te * img_bytes / float(offsets[-1]),
                           "phase_ms_per_step": {k: v / e2e_steps * 1e3 for k, v in tphases.items()},
                           "equals_rgb_search": same, "encode_setup_s": enc_s,
                           "what": "the same step with masks and targets as PackBits RGB TIFF files (71 strips of 8 rows, written by "
                                   "cds_tiff_encode_rgb outside the timed region) in pinned host memory: cds_maskset_add_tiff + "
                                   "cds_search_stream_tiff parse the tags on the host, upload the files as stored and decode them on "
                                   "the device"}
            ctx.host_free(blob_ptr)
            ctx.host_free(mblob_ptr)
        ctx.host_free(pool_ptr)
        ctx.host_free(mask_ptr)

    # shape score at every N: each rank scores its own pairs on its own GPU (no exchange: pairs go to the device that holds the target);
    # the job's rate is the sum over the ranks, timed as the slowest rank
    shape_line = None
    if not args.no_shape:
        shape_line = shape_bench(ctx, cpu_pairs=48 if (rank == 0 and world == 1) else 0)
        if world > 1:
            ts = torch.tensor([shape_line["e2e"]["ms"], shape_line["e2e_tiff"]["ms"], shape_line["kernel_ms"]], dtype=torch.float64, device="cuda")
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
            e_ms, t_ms, k_ms = [float(x) for x in ts.tolist()]
            n_pairs = shape_line["pairs"] * world
            shape_line["pairs"] = n_pairs
            shape_line["value"] = n_pairs / (k_ms * 1e-3)
            shape_line["kernel_ms"] = k_ms
            shape_line["e2e"].update({"value": n_pairs / (e_ms * 1e-3), "ms": e_ms, "h2d_bytes": shape_line["e2e"]["h2d_bytes"] * world})
            shape_line["e2e_tiff"].update({"value": n_pairs / (t_ms * 1e-3), "ms": t_ms, "h2d_bytes": shape_line["e2e_tiff"]["h2d_bytes"] * world})
            shape_line["roofline"] = None
            shape_line["n_gpus"] = world
    # The headline end-to-end number is the step fed with the library AS THE REFERENCE STORES IT: PackBits RGB TIFF files held in
    # (pinned) host memory, uploaded as they are and decoded on the device.  The same step fed with decoded pixels is kept next to
    # it as e2e.rgb_pixels: it moves 16 x the bytes over PCIe and is bound by the link, not by anything this library does.
    e2e_line = e2e
    if e2e and "tiff" in e2e:
        rgb = dict(e2e)
        e2e_line = rgb.pop("tiff")
        e2e_line["steps"] = rgb.get("steps")
        e2e_line["targets_per_gpu"] = rgb.get("targets_per_gpu")
        e2e_line["input"] = "masks and targets as PackBits RGB TIFF files in pinned host memory (the reference's storage format)"
        e2e_line["rgb_pixels"] = rgb
    if rank == 0:
        peak, peak_src = measured_peak()
        per_launch_cmp = M * T / max(match_launches / args.steps, 1)
        avg_launch_s = match_ms * 1e-3 / max(match_launches, 1)
        cmp_per_s_kernel = per_launch_cmp / avg_launch_s
        achieved_algo = cmp_per_s_kernel * ALGO_BYTES_PER_COMPARISON / 1e9
        # counters of the dominant kernel from one `ncu --set full` capture of this command at reduced size (profiles/ncu_traffic.json
        # names the capture): DRAM bytes and executed warp instructions per comparison scale with the launch
        nc = {}
        tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tp):
            try:
                nc = json.load(open(tp))
            except Exception:
                nc = {}
        traffic = nc["dram_bytes_per_comparison"] * per_launch_cmp if "dram_bytes_per_comparison" in nc else None
        n_groups = -(-M // 1024)
        # what ONE pass of the kernel's own layout over the resident shard costs: code plane + occupancy bitmaps of every target, per mask group
        plane_bytes = (H + 4) * 1224 * 4 + 142 * (7 * 152 + 32) * 4
        pass_floor = float(plane_bytes) * T * n_groups
        clocks = sampler.summary()
        sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
        issue_peak = 148 * 4 * sm_hz                    # warp instructions / s: 148 SMs x 4 schedulers x clock
        wipc = nc.get("warp_inst_per_comparison")
        line = {
            "metric": "mask x target CDS comparisons/sec", "value": value, "unit": "comparisons/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
            "wall_ms_per_step": wall_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic", "config": workload_config(args, world),
            "clocks": clocks, "gpu_launches": int(launches),
            "roofline": {"bound": "hbm",
                         # frac = PHYSICAL DRAM traffic of the dominant kernel (ncu dram__bytes_read + write, per launch) / its launch time / HBM copy peak
                         "achieved": (traffic / avg_launch_s / 1e9) if traffic else None, "peak": peak, "unit": "GB/s",
                         "frac": (traffic / avg_launch_s / 1e9 / peak) if traffic else None,
                         "traffic": traffic, "peak_source": peak_src,
                         "kernel": {1: "pixelmatch_cand_kernel<1,1024,31>", 2: "pixelmatch_band_kernel<1,true,128,24>", 3: "pixelmatch_gather_kernel"}.get(kernel_used, "?"),
                         "comparisons_per_launch": per_launch_cmp, "avg_launch_ms": avg_launch_s * 1e3,
                         # SURVEY 8(d)'s accounting: 3*W*H bytes per comparison, as if every mask re-read every target
                         "algorithmic_bytes_per_comparison": ALGO_BYTES_PER_COMPARISON,
                         "achieved_algorithmic": achieved_algo, "frac_algorithmic": achieved_algo / peak,
                         # the kernel's own layout read exactly once per mask group: the HBM floor of this formulation
                         "pass_floor_bytes": pass_floor, "pass_floor_frac": pass_floor / avg_launch_s / 1e9 / peak,
                         # the ceiling that binds: issue slots
                         "warp_inst_per_comparison": wipc,
                         "issue_frac": (wipc * cmp_per_s_kernel / issue_peak) if wipc else None,
                         "issue_peak_warp_inst_per_s": issue_peak,
                         "spin_share_of_instructions": nc.get("spin_share_of_instructions"),
                         "counters_source": nc.get("source"),
                         "note": "frac is physical (ncu DRAM bytes per comparison x this launch's comparisons / launch time / measured "
                                 "HBM copy peak).  frac_algorithmic follows SURVEY 8(d) (3*W*H bytes per comparison) and exceeds 1 because "
                                 "up to 1024 masks share one pass over a target.  The kernel is bound by instruction issue: issue_frac = "
                                 "warp instructions per comparison x comparisons/s / (148 SMs x 4 schedulers x SM clock)"},
            "e2e": e2e_line, "host_binding": binding,
            "mask_pixels_mean": float(np.mean(mask_sizes)), "setup_s": setup_s,
            "matches_returned": int(merged[3].sum()) if merged is not None else None,
        }
        if shape_line is not None:
            line["shape"] = shape_line
        if not args.no_shape and world == 1:
            try:
                line["shape"]["config2_mix"] = shape_config2_mix(ctx, last, M, t_first, min(T, 4096))
            except Exception as e:      # reporting only
                line["shape"]["config2_mix"] = {"error": repr(e)}
        if not args.no_pair_provider and world == 1:
            try:
                line["pair_provider"] = pair_provider_bench(ctx, masks_host)
            except Exception as e:      # reporting only
                line["pair_provider"] = {"error": repr(e)}
        if not args.no_data_dependence and world == 1:
            try:
                line["data_dependence"] = data_dependence(ctx, masks_host)
            except Exception as e:      # reporting only
                line["data_dependence"] = {"error": repr(e)}
        if not args.no_cpu_baseline and world == 1:
            def targets_fn(n):
                return np.concatenate([ctx.synth_rgb(1, SEED, i, min(64, n - i), W, H, on_device=True) for i in range(0, n, 64)])
            line["cpu_baseline"] = cpu_baseline(masks_host, targets_fn)
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
