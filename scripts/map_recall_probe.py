"""Cost of COCO-style average recall: MapAccumulator.update and compute() without and with
recall_max_dets=(1, 10, 100), alternating in the same run, at the COCO-val shape of map_probe.py.

5 000 images, max_boxes=100 detections on every image, 80 classes, the 10 COCO thresholds,
per-scale APs on, default matcher settings, inputs from oracle.gen_golden.synth_eval_set, batches of
--batch images.  One update pass = reset() then every batch through update(), timed with CUDA
events around the pass; the two accumulators alternate, --reps passes each after 3 warm-ups, and
the numbers are medians.  compute() is timed with a host clock around the call and a device
synchronise, alternating the same way.  Checks that every key of the plain dict is identical (==) in
the dict with recall.  Prints the card's name and power limit beside the numbers.

    python scripts/map_recall_probe.py [--images 5000] [--reps 15] [--out map_recall_probe.json]
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

from multigriddet_b200.evaluation import MapAccumulator
from oracle.gen_golden import synth_eval_set

LIMITS = (1, 10, 100)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def same(a, b):
    """== on every value of two result dicts."""
    if isinstance(b, dict):
        return set(a) == set(b) and all(same(a[k], b[k]) for k in b)
    return type(a) is type(b) and a == b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    B, M, N, C = args.images, 100, 20, 80
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(5, B, M, N, C)
    dn[:] = M                                              # max_boxes detections on every image
    ds = np.round(ds, 3)
    host = (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
    dev = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in host]
    accs = {"plain": MapAccumulator(C), "recall": MapAccumulator(C, recall_max_dets=LIMITS)}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def one_pass(acc):
        acc.reset()
        torch.cuda.synchronize()
        ev0.record()
        for b0 in range(0, B, args.batch):
            acc.update(*[t[b0:b0 + args.batch] for t in dev])
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1)

    def timed_compute(acc):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = acc.compute()
        torch.cuda.synchronize()
        return res, (time.perf_counter() - t0) * 1e3

    for _ in range(3):                                     # warm-up: modules, workspace, pool
        for acc in accs.values():
            one_pass(acc)
            timed_compute(acc)
    update_ms = {k: [] for k in accs}
    for _ in range(args.reps):                             # alternate in the same run
        for k, acc in accs.items():
            update_ms[k].append(one_pass(acc))
    compute_ms = {k: [] for k in accs}
    results = {}
    for _ in range(args.reps):
        for k, acc in accs.items():
            results[k], t = timed_compute(acc)
            compute_ms[k].append(t)

    plain, with_ar = results["plain"], results["recall"]
    equal = set(with_ar) - set(plain) == {f"AR{m}" for m in LIMITS} | {"ARS", "ARM", "ARL", "recall"} and \
        same({k: with_ar[k] for k in plain}, plain)
    med = {k: float(np.median(v)) for k, v in update_ms.items()}
    out = {"card": card(), "images": B, "max_boxes": M, "max_gt": N, "classes": C, "thresholds": 10,
           "per_scale": True, "recall_max_dets": list(LIMITS), "batch": args.batch, "reps": args.reps,
           "update_pass_ms_median": med, "update_pass_ms_all": update_ms,
           "recall_adds_ms": med["recall"] - med["plain"],
           "compute_ms_median": {k: float(np.median(v)) for k, v in compute_ms.items()},
           "compute_ms_all": compute_ms,
           "matcher": with_ar["recall"]["matcher"],
           "ar": {k: with_ar[k] for k in [f"AR{m}" for m in LIMITS] + ["ARS", "ARM", "ARL"]},
           "map": plain["mAP"], "ap_part_identical": bool(equal)}
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)
    if not equal:
        sys.exit("recall_max_dets changed the AP part of the result")


if __name__ == "__main__":
    main()
