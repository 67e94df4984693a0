"""Sharded streaming mAP (evaluation.ShardedMapAccumulator) at COCO-val shape, under torchrun.

The data of scripts/map_probe.py: 5 000 images, max_boxes=100, 80 classes, the 10 COCO
thresholds, per-scale APs on, fed as 256-image global batches, each split over the ranks by
shard_bounds.  Every rank synthesises the whole set from the same seed and updates with its
shard.  Reports, median of 5 runs after a warm-up:
- the per-rank update time (CUDA events, all updates of the run);
- compute() split into its phases (the update-sequence check, partition, exchange, merged
  compute, all-reduce and copy to the host), each closed by a device synchronise and timed with
  a host clock, the slowest rank per phase;
- the time from the first update to the result dict (host clock, ends in a synchronise);
- rank 0's single-GPU MapAccumulator over the whole set in the same run (CUDA events);
- the card's name and power limit.
Checks that every rank's dict equals the single-GPU dict exactly (== on every value).

    torchrun --nproc_per_node N scripts/map_sharded_probe.py [--images 5000] [--out FILE]
    python scripts/map_sharded_probe.py                      (world size 1)
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch

from multigriddet_b200.evaluation import MapAccumulator, ShardedMapAccumulator
from multigriddet_b200.sharding import shard_bounds
from oracle.gen_golden import synth_eval_set

PHASES = ("check", "partition", "exchange", "merged", "reduce")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def differences(a, b, path="result"):
    """Paths where two result dicts differ (exact comparison)."""
    if isinstance(b, dict):
        if set(a) != set(b):
            return [f"{path}: keys {sorted(set(a) ^ set(b))}"]
        return [d for k in b for d in differences(a[k], b[k], f"{path}[{k!r}]")]
    same_type = type(a) is type(b) or (isinstance(a, float) and isinstance(b, float))
    return [] if same_type and a == b else [f"{path}: {a!r} != {b!r}"]


class TimedSharded(ShardedMapAccumulator):
    """Host clock per compute() phase, each closed by a device synchronise."""

    def compute(self):
        self.phase_s = {}
        torch.cuda.synchronize()
        self._t = time.perf_counter()
        return super().compute()

    def _mark(self, phase):
        torch.cuda.synchronize()
        t = time.perf_counter()
        self.phase_s[phase] = t - self._t
        self._t = t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")
    rank = dist.get_rank() if dist else 0
    B, M, N, C = args.images, 100, 20, 80
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(5, B, M, N, C)
    dn[:] = M                                              # max_boxes detections on every image
    ds = np.round(ds, 3)
    host = (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
    dev = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in host]
    batches = [(b0, min(b0 + args.batch, B)) for b0 in range(0, B, args.batch)]

    def run_sharded(acc):
        ev = []
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for b0, b1 in batches:
            lo, hi = shard_bounds(b1 - b0, rank, world)
            ev.append((torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)))
            ev[-1][0].record()
            acc.update(*[t[b0 + lo:b0 + hi] for t in dev], n_total=b1 - b0)
            ev[-1][1].record()
        res = acc.compute()
        end_to_end = time.perf_counter() - t0
        return res, sum(a.elapsed_time(b) for a, b in ev), end_to_end

    acc = TimedSharded(C)
    run_sharded(acc)                                       # warm-up: modules, workspace, pool, NCCL
    reps = []
    for _ in range(args.reps):
        acc.reset()
        if dist:
            dist.barrier()
        got, upd_ms, e2e_s = run_sharded(acc)
        row = {"update_ms": upd_ms, "end_to_end_ms": e2e_s * 1e3,
               **{f"{p}_ms": acc.phase_s[p] * 1e3 for p in PHASES}}
        row["compute_ms"] = sum(row[f"{p}_ms"] for p in PHASES)
        if dist:                                           # the slowest rank of each number
            rows = [None] * world
            dist.all_gather_object(rows, row)
            row = {k: max(r[k] for r in rows) for k in row}
        reps.append(row)
    median = {k: float(np.median([r[k] for r in reps])) for k in reps[0]}
    results = [None] * world
    if dist:
        dist.all_gather_object(results, got)
    else:
        results = [got]

    out = None
    if rank == 0:
        single = MapAccumulator(C)

        def run_single():
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record()
            for b0, b1 in batches:
                single.update(*[t[b0:b1] for t in dev])
            e[1].record()
            res = single.compute()
            e[2].record()
            torch.cuda.synchronize()
            return res, e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2]), e[0].elapsed_time(e[2])

        run_single()
        single_reps = []
        for _ in range(args.reps):
            single.reset()
            torch.cuda.synchronize()
            ref, u, c, t = run_single()
            single_reps.append({"update_ms": u, "compute_ms": c, "end_to_end_ms": t})
        diffs = {r: differences(res, ref) for r, res in enumerate(results)}
        for r, d in diffs.items():
            for line in d[:5]:
                print(f"rank {r} differs:", line)
        out = {"card": card(), "world_size": world, "images": B, "max_boxes": M, "classes": C,
               "thresholds": 10, "per_scale": True, "batch": args.batch, "reps": args.reps,
               "sharded_median": median, "sharded_runs": reps,
               "single_gpu_median": {k: float(np.median([r[k] for r in single_reps])) for k in single_reps[0]},
               "num_predictions": ref["num_predictions"], "mAP": float(ref["mAP"]),
               "identical_to_single_gpu": all(not d for d in diffs.values())}
        print(json.dumps(out, indent=1))
        if args.out:
            os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
            with open(args.out, "w") as fh:
                json.dump(out, fh, indent=1)
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    if out is not None and not out["identical_to_single_gpu"]:
        sys.exit("ShardedMapAccumulator and MapAccumulator disagree")


if __name__ == "__main__":
    main()
