"""Cost of the precision-recall curves: MapAccumulator.compute() against
compute(precision_recall=True) in the same run, at the COCO-val shape of map_probe.py.

5 000 images, max_boxes=100, 80 classes, the 10 COCO thresholds, per-scale APs on, default
matcher settings (both full-set views are matched, so the curves of both are computed and the
one calculate_map's rule selects is kept).  The records are accumulated once; the two computes
then alternate, each timed with a host clock around the call (it ends in a device synchronise),
median after warm-up.  Checks that the AP part of the curve result is identical (==) to compute()'s,
and reports the device memory of the kept curves and the peak added by the curve call.  Prints
the card's name and power limit beside the numbers.

    python scripts/map_pr_probe.py [--images 5000] [--reps 15] [--out map_pr_probe.json]
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

CONFS = [0.05, 0.1, 0.25, 0.5, 0.75]


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
    acc = MapAccumulator(C)
    for b0 in range(0, B, args.batch):
        acc.update(*[t[b0:b0 + args.batch] for t in dev])
    torch.cuda.synchronize()

    def timed(pr):
        t0 = time.perf_counter()
        res = acc.compute(precision_recall=True, confidences=CONFS) if pr else acc.compute()
        torch.cuda.synchronize()
        return res, (time.perf_counter() - t0) * 1e3

    for _ in range(3):                                     # warm-up: modules, workspace, pool
        timed(False)
        timed(True)
    plain_ms, pr_ms = [], []
    for _ in range(args.reps):                             # alternate the two in the same run
        plain, t = timed(False)
        plain_ms.append(t)
        res, t = timed(True)
        pr_ms.append(t)
        del res

    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    res = acc.compute(precision_recall=True, confidences=CONFS)
    torch.cuda.synchronize()
    peak_extra = torch.cuda.max_memory_allocated() - base
    pr = res.pop("precision_recall")
    kept = sum(pr[k].numel() * pr[k].element_size() for k in ("offsets", "scores", "precision", "recall"))
    equal = same(res, plain)
    out = {"card": card(), "images": B, "max_boxes": M, "classes": C, "thresholds": 10, "per_scale": True,
           "confidences": len(CONFS), "matcher": pr["matcher"], "curve_records": int(pr["scores"].numel()),
           "reps": args.reps,
           "compute_ms_median": float(np.median(plain_ms)),
           "compute_pr_ms_median": float(np.median(pr_ms)),
           "compute_ms_all": plain_ms, "compute_pr_ms_all": pr_ms,
           "curve_bytes_kept": int(kept), "peak_extra_bytes_during_compute_pr": int(peak_extra),
           "ap_part_identical": bool(equal)}
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)
    if not equal:
        sys.exit("compute(precision_recall=True) changed the AP part")


if __name__ == "__main__":
    main()
