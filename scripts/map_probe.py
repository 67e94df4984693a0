"""Streaming mAP (evaluation.MapAccumulator) against the drop-in calculate_map at COCO-val shape.

5 000 images, max_boxes=100, 80 classes, the 10 COCO thresholds, per-scale APs on.  Times
each 256-image update and compute() with CUDA events, and the drop-in path (the reference's
dicts, then calculate_map) with a host clock, in the same run; checks the two results agree
(rel 1e-12) and prints the card's name and power limit beside the numbers.  NumPy is pinned
like the test suite pins it (oracle/ref_loader.py): the drop-in's AP depends on NumPy's argsort
tie order, and the reference's numbers were produced without its SIMD sort dispatch.

    python scripts/map_probe.py [--images 5000] [--out map_probe.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import ref_loader  # noqa: E402

ref_loader.pin_numpy_env()                                 # before NumPy is first imported

import numpy as np
import torch

from multigriddet_b200.evaluation import MapAccumulator, calculate_map
from oracle import metrics_oracle as MO
from oracle.gen_golden import synth_eval_set


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def differences(a, b, path="result"):
    """Paths where the two result dicts differ (floats at rel 1e-12)."""
    if isinstance(b, dict):
        if set(a) != set(b):
            return [f"{path}: keys {sorted(set(a) ^ set(b))}"]
        return [d for k in b for d in differences(a[k], b[k], f"{path}[{k!r}]")]
    if isinstance(b, float):
        return [] if abs(a - b) <= 1e-12 * abs(b) + 1e-15 else [f"{path}: {a!r} != {b!r}"]
    return [] if a == b else [f"{path}: {a!r} != {b!r}"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    B, M, N, C = args.images, 100, 20, 80
    t0 = time.perf_counter()
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(5, B, M, N, C)
    dn[:] = M                                              # max_boxes detections on every image
    ds = np.round(ds, 3)
    host = (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
    print(f"inputs: {B} images x {M} detections, {C} classes ({time.perf_counter() - t0:.1f} s to synthesise)")
    dev = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in host]

    def run(acc, ev=None):
        for b0 in range(0, B, args.batch):
            if ev is not None:
                ev[0].append(torch.cuda.Event(enable_timing=True)); ev[0][-1].record()
            acc.update(*[t[b0:b0 + args.batch] for t in dev])
            if ev is not None:
                ev[1].append(torch.cuda.Event(enable_timing=True)); ev[1][-1].record()
        if ev is not None:
            ev[2].record()
        res = acc.compute()
        if ev is not None:
            ev[3].record()
        return res

    acc = MapAccumulator(C)
    run(acc)                                               # warm-up: modules, workspace, pool
    reps = []
    for _ in range(5):
        acc.reset()
        torch.cuda.synchronize()
        ev = ([], [], torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        got = run(acc, ev)
        torch.cuda.synchronize()
        upd = [a.elapsed_time(b) for a, b in zip(ev[0], ev[1])]
        reps.append({"update_ms_per_batch_median": float(np.median(upd)), "update_ms_total": float(sum(upd)),
                     "compute_ms": ev[2].elapsed_time(ev[3]), "end_to_end_ms": ev[0][0].elapsed_time(ev[3])})

    t0 = time.perf_counter()
    preds, gts = MO.to_dicts(*host)
    t_dicts = time.perf_counter() - t0
    t0 = time.perf_counter()
    ref = calculate_map(preds, gts, C)
    t_map = time.perf_counter() - t0
    diff = differences(got, ref)
    same = not diff
    for d in diff[:10]:
        print("differs:", d)
    out = {"card": card(), "images": B, "max_boxes": M, "classes": C, "thresholds": 10, "per_scale": True,
           "batch": args.batch, "device_runs": reps,
           "dropin_build_dicts_s": t_dicts, "dropin_calculate_map_s": t_map,
           "numpy_pinned": ref_loader.numpy_is_pinned(),
           "num_predictions": got["num_predictions"], "mAP": float(got["mAP"]), "equal_to_dropin": bool(same)}
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)
    if not same:
        sys.exit("MapAccumulator and calculate_map disagree")


if __name__ == "__main__":
    main()
