"""Cost of the detection confusion matrix: ConfusionMatrixAccumulator.update at Q = 1 and Q = 32
confidences against MapAccumulator.update, at the COCO-val shape of map_probe.py, and a check of
the matrices against a host pass.

5 000 images, max_boxes=100 detections on every image, 80 classes, inputs from
oracle.gen_golden.synth_eval_set (20 % of the detection labels are wrong, so confusions occur).
One pass = reset() then every batch of --batch images through update(); the passes of the
accumulators alternate in the same run, each timed with CUDA events around the pass, median after
warm-up.  compute() is timed with a host clock (it ends in a synchronise).

Check: engine.match_detections(return_matched=True) on host arrays gives stage 1, NumPy does stage 2
and the counts; the Q = 1 matrix and four of the 32 are compared whole (==), all 32 by the
diagonal and the row and column sums.  Prints the card's name and power limit beside the numbers.

    python scripts/confusion_probe.py [--images 5000] [--reps 15] [--out confusion_probe.json]
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

from multigriddet_b200 import engine
from multigriddet_b200.evaluation import ConfusionMatrixAccumulator, MapAccumulator
from oracle.gen_golden import synth_eval_set

THR = 0.5
CONFS32 = [round(0.03 * k, 2) for k in range(32)]          # 0.00 .. 0.93, on the scores' 0.001 grid


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def iou_rows(p, g):
    """Corner IoU of every (detection, ground truth) pair in the matcher's operation order."""
    x1 = np.maximum(p[:, None, 0], g[None, :, 0]); y1 = np.maximum(p[:, None, 1], g[None, :, 1])
    x2 = np.minimum(p[:, None, 2], g[None, :, 2]); y2 = np.minimum(p[:, None, 3], g[None, :, 3])
    inter = np.maximum(0.0, x2 - x1) * np.maximum(0.0, y2 - y1)
    a1 = (p[:, 2] - p[:, 0]) * (p[:, 3] - p[:, 1])
    a2 = (g[:, 2] - g[:, 0]) * (g[:, 3] - g[:, 1])
    uni = (a1[:, None] + a2[None, :]) - inter
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(uni > 0, inter / np.where(uni > 0, uni, 1.0), 0.0)


def host_matrix(args, who, C, conf):
    """One (C+1, C+1) matrix from the host matcher's claims (stage 1) and a NumPy stage 2."""
    db, ds, dc, dn, gtb, gtc, gtn = args
    m = np.zeros((C + 1, C + 1), np.int64)
    for b in range(len(dn)):
        n, g = int(dn[b]), int(gtn[b])
        s, c, w = ds[b, :n], dc[b, :n], who[b, :n]
        keep = s >= conf
        order = np.argsort(s, kind="stable")[::-1]
        order = order[keep[order]]
        taken = np.zeros(g, bool)
        hit = keep & (w >= 0)
        taken[w[hit]] = True
        np.add.at(m, (c[hit], c[hit]), 1)
        iou = iou_rows(db[b, :n].astype(np.float64), gtb[b, :g])
        for d in order:
            if w[d] >= 0:
                continue
            v = np.where(taken, -1.0, iou[d]) if g else iou[d]
            j = int(np.argmax(v)) if g else -1
            if j >= 0 and v[j] > 0 and v[j] >= THR:
                taken[j] = True
                m[gtc[b, j], c[d]] += 1
            else:
                m[C, c[d]] += 1
        np.add.at(m, (gtc[b, :g][~taken], C), 1)
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    B, M, N, C = args.images, 100, 20, 80
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(5, B, M, N, C)
    dn[:] = M
    ds = np.round(ds, 3)
    host = (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
    dev = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in host]
    accs = {"map": MapAccumulator(C), "confusion_q1": ConfusionMatrixAccumulator(C, THR),
            "confusion_q32": ConfusionMatrixAccumulator(C, THR, CONFS32)}
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

    for _ in range(3):                                     # warm-up: modules, workspace, pool
        for acc in accs.values():
            one_pass(acc)
    times = {k: [] for k in accs}
    for _ in range(args.reps):                             # alternate in the same run
        for k, acc in accs.items():
            times[k].append(one_pass(acc))

    compute_ms = []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        m32 = accs["confusion_q32"].compute()
        compute_ms.append((time.perf_counter() - t0) * 1e3)
    m1 = accs["confusion_q1"].compute()

    # host check: stage 1 of the host matcher, stage 2 in NumPy
    tp, who = engine.match_detections(*host, [THR], iou_mode="corner", return_matched=True)
    tp, who = tp[0], who[0]
    checks = {"q1_whole": bool(np.array_equal(m1[0], host_matrix(host, who, C, -np.inf)))}
    whole = [0, 10, 17, 31]
    checks["q32_whole"] = {CONFS32[q]: bool(np.array_equal(m32[q], host_matrix(host, who, C, CONFS32[q])))
                           for q in whole}
    n_gt = np.bincount(gtc[np.arange(N)[None, :] < gtn[:, None]], minlength=C)
    sums = True
    for q, conf in enumerate(CONFS32):
        kept = ds >= conf
        sums &= np.array_equal(np.diag(m32[q])[:C], np.bincount(dc[kept & (tp == 1)], minlength=C))
        sums &= np.array_equal(m32[q, :C].sum(1), n_gt)
        sums &= np.array_equal(m32[q, :, :C].sum(0), np.bincount(dc[kept], minlength=C)) and m32[q, C, C] == 0
    checks["q32_diagonal_and_sums"] = bool(sums)
    ok = checks["q1_whole"] and all(checks["q32_whole"].values()) and sums

    off = int(m1[0, :C, :C].sum() - np.trace(m1[0, :C, :C]))
    out = {"card": card(), "images": B, "max_boxes": M, "max_gt": N, "classes": C, "iou_threshold": THR,
           "batch": args.batch, "reps": args.reps,
           "update_pass_ms_median": {k: float(np.median(v)) for k, v in times.items()},
           "update_pass_ms_all": times,
           "compute_q32_ms_median": float(np.median(compute_ms)), "compute_q32_ms_all": compute_ms,
           "q1_cells": {"true_positives": int(np.trace(m1[0, :C, :C])), "class_confusions": off,
                        "background_fp": int(m1[0, C].sum()), "missed": int(m1[0, :, C].sum())},
           "checks": checks}
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)
    if not ok:
        sys.exit("the device matrices differ from the host pass")


if __name__ == "__main__":
    main()
