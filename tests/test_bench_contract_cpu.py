"""The reference arm of bench.py (`--impl reference`: the oracle port on the host cores) prints one JSON line with the keys the
driver reads.  Runs on CPU only; the GPU arm shares the same line layout (checked on the GPU box by the driver itself)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--ref-masks", "2", "--ref-targets", "8"], capture_output=True, text=True, timeout=600, check=True).stdout
    lines = [ln for ln in out.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "mask x target CDS comparisons/sec" and d["unit"] == "comparisons/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "comparisons/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the arm says what it actually timed: at least one target per host core, so that every core has work
    n_t = max(8, len(os.sched_getaffinity(0)))
    assert d["config"]["sample"] == {"masks": 2, "targets": n_t}
    assert "workload" in d["config"] and "2 masks x %d targets" % n_t in d["config"]["workload"]
    assert d["gpu_library_mapped"] is False        # the CPU arm takes its inputs from the host-only generator: libcdsgpu.so is not mapped


def test_dump_outputs_are_the_last_steps_results(tmp_path):
    """--dump-outputs writes the timed path's results as float64 .npy files, the same ones from run to run (seeded inputs)."""
    import numpy as np
    from oracle import oracle as O
    from oracle import synth as S
    dumps = []
    for run in range(2):
        d = tmp_path / ("run%d" % run)
        subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
                        "--ref-masks", "2", "--ref-targets", "8", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, check=True)
        dumps.append({p.stem: np.load(p) for p in d.glob("*.npy")})
    assert sorted(dumps[0]) == ["mask_index", "mirrored", "score"]
    assert all(a.dtype == np.float64 for a in dumps[0].values())
    assert all(np.array_equal(dumps[0][k], dumps[1][k]) for k in dumps[0])
    # what the arm computed: both masks against its targets (at least one per host core), in order
    n_t = dumps[0]["score"].shape[1]
    masks, targets = S.synth_rgb(0, 0xC0FFEE, 0, 2, 1210, 566), S.synth_rgb(1, 0xC0FFEE, 0, n_t, 1210, 566)
    rects = O.label_rects(1210, 566)
    es, em, _ = O.search_dense([O.PixelMatchMask(m, 20, True, 20, 0.01, 2, rects) for m in masks], targets)
    assert dumps[0]["mask_index"].tolist() == [0, 1]
    assert np.array_equal(dumps[0]["score"], es) and np.array_equal(dumps[0]["mirrored"], em)


def test_steps_must_be_positive():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True, text=True,
                       timeout=600)
    assert p.returncode != 0 and "--steps" in p.stderr


def test_reference_arm_under_torchrun_prints_once():
    """Launched like the driver launches N > 1 (torchrun, one process per GPU): rank 0 alone runs and prints the reference line,
    the other ranks exit 0 without work."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29547", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0",
           "--ref-masks", "2", "--ref-targets", "8"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0
