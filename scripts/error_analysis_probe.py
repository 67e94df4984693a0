"""Cost of the detection error analysis: ErrorAnalysisAccumulator.update against MapAccumulator.update
at the COCO-val shape of map_probe.py, compute() time, the records' device memory, and a check of the
dict against the CPU restatement of tests/test_error_analysis.py on a subset.

5 000 images, max_boxes=100 detections on every image, 80 classes, inputs from
oracle.gen_golden.synth_eval_set (20 % of the detection labels are wrong, so every error type occurs).
One pass = reset() then every batch of --batch images through update(); the passes of the two
accumulators alternate in the same run, each timed with CUDA events around the pass, median after
warm-up.  compute() is timed with a host clock (it ends in a synchronise).  Prints the card's name and
power limit beside the numbers.

    python scripts/error_analysis_probe.py [--images 5000] [--reps 15] [--check 256] [--out error_analysis.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_loader  # noqa: E402

ref_loader.pin_numpy_env()                                 # before NumPy is first imported

import numpy as np
import torch

from multigriddet_b200.evaluation import ErrorAnalysisAccumulator, MapAccumulator
from oracle.gen_golden import synth_eval_set
sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_error_analysis import tide_batch, tide_result  # noqa: E402  the CPU restatement of the rule


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def same(got, want):
    close = lambda a, b: np.allclose(a, b, rtol=1e-12, atol=1e-14)
    return bool(close(got["AP"], want["AP"]) and all(close(got["dAP"][k], want["dAP"][k]) for k in want["dAP"])
                and got["counts"] == want["counts"] and close(got["per_class"]["AP"], want["per_class"]["AP"])
                and close(got["per_class"]["dAP"], want["per_class"]["dAP"])
                and np.array_equal(got["per_class"]["counts"], want["per_class"]["counts"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--check", type=int, default=256, help="images of the subset checked on the CPU")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    B, M, N, C = args.images, 100, 20, 80
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(5, B, M, N, C)
    dn[:] = M
    ds = np.round(ds, 3)
    host = (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
    dev = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in host]
    accs = {"map": MapAccumulator(C), "error_analysis": ErrorAnalysisAccumulator(C)}
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

    ea = accs["error_analysis"]
    compute_ms = []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        res = ea.compute()
        torch.cuda.synchronize()
        compute_ms.append((time.perf_counter() - t0) * 1e3)
    record_bytes = ea._slots * 40

    n = min(args.check, B)
    sub = ErrorAnalysisAccumulator(C)
    sub.update(*[t[:n] for t in dev])
    sub_host = tuple(a[:n] for a in host)
    cls, flag, gt, counts = tide_batch(*sub_host, C)
    check = same(sub.compute(), tide_result(cls, flag, sub_host[1], gt, counts, C))

    out = {"card": card(), "images": B, "max_boxes": M, "max_gt": N, "classes": C, "pos_threshold": 0.5,
           "background_threshold": 0.1, "batch": args.batch, "reps": args.reps,
           "update_pass_ms_median": {k: float(np.median(v)) for k, v in times.items()},
           "update_pass_ms_all": times,
           "compute_ms_median": float(np.median(compute_ms)), "compute_ms_all": compute_ms,
           "record_bytes": record_bytes,
           "AP": res["AP"], "dAP": res["dAP"], "counts": res["counts"],
           "check_images": n, "check_equal": check}
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)
    if not check:
        sys.exit("the device dict differs from the CPU restatement")


if __name__ == "__main__":
    main()
