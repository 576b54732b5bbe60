"""The shape score's single-pair call three ways, on a gradientScores-like mix:  python tools/shape_pairq_bench.py [--legs abc] [--threads 1,8,40,80]

64 synthetic EM masks, each scoring 300 targets drawn from a pool of 512 synthetic LM targets at 1210 x 566, with gradients from
cds_synth_gradient and zgap images from cds_make_zgap passed as pixels (the way the Java provider passes them).
  (a) today's single-pair path: one cds_shape_score_pairs call per pair from 40 Python threads (ctypes releases the interpreter lock;
      the context's lock serialises the calls anyway), over the first A_PAIRS pairs
  (b) the queue: cds_debug_shape_pairq_drive with native threads, the cache holding the whole pool, then with a cache of 128 slots
      per device (max_batch 16: targets are evicted and uploaded again)
  (c) the ceiling: all pairs in one batched cds_shape_score_pairs call
Every leg is run once to warm up, then timed with host clocks around the blocking calls.  (b) and (a) must equal (c) bit for bit."""
import argparse
import json
import subprocess
import sys
import threading
import time

import numpy as np

sys.path.insert(0, ".")
from colormipsearch_b200 import capi
from oracle import oracle as O

W, H = 1210, 566
SEED = 0x5EED
N_MASKS, N_POOL, PER_MASK = 64, 512, 300
A_PAIRS = 1000


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = "unknown (%s)" % e
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--legs", default="abc")
    ap.add_argument("--threads", default="1,8,40,80")
    args = ap.parse_args()
    threads = [int(t) for t in args.threads.split(",")]
    print(json.dumps({"gpu": gpu_info()}), flush=True)

    ctx = capi.Context(device_ids=[0])
    rects = O.label_rects(W, H)
    masks = ctx.synth_rgb(0, SEED, 0, N_MASKS, W, H, on_device=True)
    targets = np.concatenate([ctx.synth_rgb(1, SEED, i, 128, W, H, on_device=True) for i in range(0, N_POOL, 128)])
    grads = np.concatenate([ctx.synth_gradient(SEED, i, 128, W, H, on_device=True) for i in range(0, N_POOL, 128)])
    zgaps = np.concatenate([ctx.make_zgap(targets[i:i + 128], 20, 10, rects) for i in range(0, N_POOL, 128)])
    rng = np.random.default_rng(SEED)
    pm = np.repeat(np.arange(N_MASKS, dtype=np.int32), PER_MASK)
    pt = np.concatenate([rng.choice(N_POOL, PER_MASK, replace=False) for _ in range(N_MASKS)]).astype(np.int64)
    keys = np.arange(1, N_POOL + 1, dtype=np.uint64) * 2654435761
    n = len(pm)
    sms = capi.ShapeMaskSet(ctx, W, H, 20, True, rects)
    sms.add_rgb(masks)

    # (c) the ceiling, and the reference of the other legs
    ref = sms.score_pairs(targets, grads, zgaps, pm, pt)
    t0 = time.perf_counter()
    ref = sms.score_pairs(targets, grads, zgaps, pm, pt)
    secs = time.perf_counter() - t0
    if "c" in args.legs:
        print(json.dumps({"leg": "c_batched_call", "pairs": n, "seconds": round(secs, 4), "pairs_per_s": round(n / secs)}), flush=True)

    if "a" in args.legs:
        na = A_PAIRS
        out = [None] * na

        def one(i):
            t = int(pt[i])
            out[i] = sms.score_pairs(targets[t:t + 1], grads[t:t + 1], zgaps[t:t + 1], pm[i:i + 1], [0])

        for timed in (False, True):
            nxt = iter(range(na))
            lock = threading.Lock()

            def worker():
                while True:
                    with lock:
                        i = next(nxt, None)
                    if i is None:
                        return
                    one(i)

            t0 = time.perf_counter()
            pool = [threading.Thread(target=worker) for _ in range(40)]
            for th in pool:
                th.start()
            for th in pool:
                th.join()
            secs = time.perf_counter() - t0
        got = [np.concatenate([o[k] for o in out]) for k in range(3)]
        assert all(np.array_equal(g, r[:na]) for g, r in zip(got, ref)), "leg (a) differs from the batched call"
        print(json.dumps({"leg": "a_single_pair_calls", "threads": 40, "pairs": na, "seconds": round(secs, 4), "pairs_per_s": round(na / secs)}), flush=True)

    if "b" in args.legs:
        for name, max_batch, cache in (("b_queue_pool_resident", 64, N_POOL), ("b_queue_cache_128", 16, 128)):
            for nt in threads:
                q = capi.ShapePairQueue(ctx, sms, max_batch=max_batch, cache_targets=cache)
                q.drive(targets, grads, zgaps, keys, pm, pt, nt)                  # warm-up: fills the cache
                s0 = q.stats()
                gap, he, mir, secs = q.drive(targets, grads, zgaps, keys, pm, pt, nt)
                s1 = q.stats()
                q.close()
                assert np.array_equal(gap, ref[0]) and np.array_equal(he, ref[1]) and np.array_equal(mir, ref[2]), \
                    "leg (b) differs from the batched call (%s, %d threads)" % (name, nt)
                print(json.dumps({"leg": name, "threads": nt, "max_batch": max_batch, "cache_targets": cache, "pairs": n,
                                  "seconds": round(secs, 4), "pairs_per_s": round(n / secs),
                                  "requests": s1["requests"] - s0["requests"], "batches": s1["batches"] - s0["batches"],
                                  "uploads": s1["uploads"] - s0["uploads"]}), flush=True)
    sms.close()
    ctx.close()
    print(json.dumps({"gpu": gpu_info(), "equal_to_batched_call": True}), flush=True)


if __name__ == "__main__":
    main()
