"""bench.py's driver-facing contract, as far as a CPU box can exercise it: the reference arm
(`--impl reference`: the reference's CPU path on the host cores, no GPU involved) prints ONE
JSON line with the agreed keys, and ranks other than 0 of a torchrun launch exit quietly."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None):
    env = dict(os.environ, **(env_extra or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                           "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                          cwd=ROOT, env=env, timeout=600)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    baseline = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["impl"] == "reference" and d["metric"] == baseline["metric"]
    for k in ("value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_runs_on_rank_zero_only():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


_DUMP_CASE = """
import sys, torch
sys.path.insert(0, {root!r})
import bench
B, M = 40, 5
g = torch.Generator().manual_seed(1)
y_true = [torch.randn((B, s, s, 7), generator=g) for s in (2, 4)]
det = {{"boxes_xyxy": torch.randint(-1, 700, (B, M, 4), dtype=torch.int32, generator=g),
       "scores": torch.rand((B, M), dtype=torch.float64, generator=g),
       "classes": torch.randint(-1, 80, (B, M), dtype=torch.int32, generator=g),
       "counts": torch.randint(0, M + 1, (B,), dtype=torch.int32, generator=g)}}
bench.DUMP_BYTES = bench.DUMP_Y_IMAGES * (sum(y[0].numel() for y in y_true) * 4 + 8) + 10 * (8 + (M * 4 + M + M + 1) * 8)
if __name__ == "__main__":
    bench.dump_outputs(sys.argv[1], det, y_true)
"""


def test_dump_outputs_writes_a_fixed_sample_within_the_budget(tmp_path):
    """--dump-outputs on host tensors laid out like the step's outputs, in two separate processes:
    float32 / float64 files only, no more than DUMP_BYTES, the same seeded sample in every run,
    the values of the tensors given."""
    import numpy as np
    code = _DUMP_CASE.format(root=ROOT)
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, "-c", code, str(tmp_path / d)], capture_output=True, text=True,
                           timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
    sys.path.insert(0, ROOT)
    import bench
    budget = bench.DUMP_BYTES
    scope = {}
    try:
        exec(code, scope)                  # the same tensors and budget, in this process
        det, y_true, limit = scope["det"], scope["y_true"], bench.DUMP_BYTES
    finally:
        bench.DUMP_BYTES = budget
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == sorted(["y_true_2.npy", "y_true_4.npy", "y_true_images.npy", "boxes_xyxy.npy",
                            "scores.npy", "classes.npy", "counts.npy", "detections_images.npy"])
    a = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        assert np.array_equal(a[f[:-4]], np.load(tmp_path / "b" / f)), f
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= limit
    yi, di = a["y_true_images"].astype(int), a["detections_images"].astype(int)
    assert len(yi) == bench.DUMP_Y_IMAGES and len(set(yi)) == len(yi)
    assert len(di) == 10 and len(set(di)) == 10
    for y in y_true:
        assert np.array_equal(a[f"y_true_{y.shape[1]}"], y.numpy()[yi])
    for k, v in det.items():
        assert np.array_equal(a[k], v.numpy()[di].astype(np.float64)), k


@pytest.mark.gpu
def test_dump_outputs_hold_what_the_timed_step_computed(tmp_path):
    """bench.py --dump-outputs on the device at a small batch: the files hold the fused step's
    detections and y_true for bench's own seeded inputs (one direct engine.grid_step on them)."""
    import numpy as np
    import torch
    B = 64
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                        "--batch", str(B), "--strong-batch", str(B), "--no-e2e", "--no-extras",
                        "--no-cpu-baseline", "--no-overlap-run", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    assert len([ln for ln in r.stdout.splitlines() if ln.strip()]) == 1
    sys.path.insert(0, ROOT)
    import bench
    from multigriddet_b200 import engine, synth
    device = torch.device("cuda", 0)
    anchors, _, d_boxes, preds = bench.make_device_inputs(B, device, seed=1)
    y = [torch.empty((B, g, g, bench.D), dtype=torch.float32, device=device) for g in (19, 38, 76)]
    d_hw = torch.from_numpy(synth.image_shapes(0, B, mixed=True)).to(device)
    det = engine.grid_step(d_boxes, y, preds, d_hw, (bench.S, bench.S), anchors, bench.C,
                           want=("boxes_xyxy", "scores", "classes"), **bench.POST)
    a = {p.name[:-4]: np.load(p) for p in tmp_path.iterdir()}
    yi, di = a["y_true_images"].astype(int), a["detections_images"].astype(int)
    assert len(yi) == bench.DUMP_Y_IMAGES and np.array_equal(di, np.arange(B))
    for t in y:
        assert np.array_equal(a[f"y_true_{t.shape[1]}"], t.cpu().numpy()[yi])
    for k in ("boxes_xyxy", "scores", "classes", "counts"):
        assert np.array_equal(a[k], det[k].cpu().numpy().astype(np.float64)), k
    assert a["counts"].sum() > 0
