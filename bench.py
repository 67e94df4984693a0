#!/usr/bin/env python
"""Headline benchmark: encode + decode/NMS images/sec on COCO-shaped synthetic data.

    python bench.py --gpus N --steps K --warmup W              (this repo's CUDA path)
    python bench.py --impl reference --gpus N --steps K ...    (reference CPU path)
    python bench.py ... --dump-outputs DIR      (also save the last timed step's outputs)

One *step* = one pass of the hot path over one batch: `mgd_encode_targets` on B
images' ground-truth boxes (B x 3 grids of y_true written) followed by
`mgd_decode_nms` on B images of raw head outputs (decode, threshold, NMS, top-k),
both through the C ABI.  Workload (BASELINE.json configs[4], the configuration the
metric is quoted on): COCO 80 classes, 608x608, grids 19/38/76, up to 100
boxes/image, planted head outputs, confidence 0.001, DIoU-NMS 0.45, max 100
detections.  Images are independent, so N GPUs shard by image with no collective
(weak scaling: every rank processes its own batch).

`value` is measured with inputs and outputs resident in HBM (CUDA events on the
launching stream, max over ranks); the step is ONE library call
(`mgd_encode_decode_nms`), which overlaps the two halves internally.  `e2e` is the
same step through the same C ABI with pinned HOST buffers, so host<->device copies
are inside the timed region.  The batch is far larger than L2 (2 x 2.67 MB per
image), so no L2 flush is needed.

`--scaling strong` (BASELINE.json configs[4] as written): 4 096 images IN TOTAL are
split over the ranks and every rank ends the step holding all detections: the NMS
kernels store each image's rows into every rank's tensors as they produce them
(`sharding.DetectionExchange`: peer stores over NVLink, no collective call; the NCCL
all-gather and the host gather it replaces are timed beside it).  The default weak line
(4 096 images per rank, no collective) carries the strong numbers as `strong_scaling`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

def _baseline_metric():
    """The metric string of BASELINE.json, verbatim (the driver matches lines on it)."""
    try:
        with open(os.path.join(ROOT, "BASELINE.json"), encoding="utf-8") as fh:
            return str(json.load(fh)["metric"])
    except Exception:
        return "encode+decode/NMS images/sec, COCO 608\u00d7608, 1\u20138 B200; % HBM peak"


METRIC = _baseline_metric()
UNIT = "images/s"
S, C, A, NBOX = 608, 80, 3, 100
CELLS = 19 * 19 + 38 * 38 + 76 * 76                    # 7581
D = 5 + A + C                                           # 88
BYTES_ENCODE = CELLS * D * 4 + NBOX * 5 * 4             # y_true written + boxes read
BYTES_DECODE = CELLS * D * 4 + 100 * (32 + 16 + 8 + 4 + 4) + 4
POST = dict(max_boxes=100, confidence=0.001, nms_threshold=0.45, nms_method="diou")
WORKLOAD = ("COCO 80c 608x608 (grids 19/38/76, 88 ch): encode <=100 boxes/img + decode/DIoU-NMS "
            "(conf 0.001, thr 0.45, max 100), planted head outputs, mixed letterbox shapes")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="images per rank per step")
    ap.add_argument("--e2e-batch", type=int, default=512)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-overlap-run", action="store_true",
                    help="skip the extra separate-calls measurement")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the extra workloads (dense-random, small batches, drop-in latency)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="strong: --strong-batch images in total, split over the ranks, gather on the clock")
    ap.add_argument("--strong-batch", type=int, default=4096)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed step returned in its last call to DIR/<name>.npy "
                         "(rank 0's outputs only when several ranks run)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    return args


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def dram_traffic(kernel):
    """Per-image DRAM bytes of a kernel from the committed ncu --set full capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            return json.load(fh).get(kernel)
    except Exception:
        return None


class ClockSampler:
    """SM clock and throttle reasons sampled (NVML, every ~5 ms) while the timed region runs."""

    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("hw_thermal_slowdown", 0x40),
               ("sw_thermal_slowdown", 0x20), ("hw_power_brake_slowdown", 0x80))

    def __init__(self, index):
        self.index = index
        self.sm, self.mask, self.stop = [], 0, False
        self.max_mhz = None
        self.thread = None

    def _visible_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v for v in vis.split(",") if v.strip()]
            if self.index < len(ids) and ids[self.index].strip().isdigit():
                return int(ids[self.index])
        return self.index

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._visible_index())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None
        return self

    def _run(self):
        nv = self.nv
        while not self.stop:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                try:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                except Exception:
                    pass
            time.sleep(0.005)

    def __exit__(self, *exc):
        self.stop = True
        if self.thread is not None:
            self.thread.join(timeout=1)

    def summary(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": [n for n, bit in self.REASONS if self.mask & bit], "samples": len(sm)}


# ------------------------------------------------------------------------------
# CPU side: the oracle port of the reference, timed on host cores
# ------------------------------------------------------------------------------

def _cpu_inputs(n_images, seed=0):
    import numpy as np
    import torch
    from multigriddet_b200 import synth
    from oracle import c_oracle
    anchors = synth.coco_anchors(np.float32)
    boxes = synth.synth_boxes(seed, n_images, NBOX, S, C)
    yt = c_oracle.encode_targets(boxes, (S, S), anchors, C)       # input prep, not timed
    preds = [p.numpy() for p in
             synth.planted_head_outputs([torch.from_numpy(y) for y in yt], A, seed)]
    return anchors, boxes, preds


_SHARDS = []          # filled before the worker pool forks: inputs are inherited, not pickled


def _cpu_worker_indexed(i):
    return _cpu_worker(_SHARDS[i])


def _reference_staged():
    try:
        from oracle import ref_loader
        return ref_loader.staged()
    except Exception:
        return False


def _cpu_worker(args):
    """One shard of the workload on one host core: the REAL reference
    (oracle/_ref: preprocess_true_boxes, then MultiGridDecoder.postprocess image by image,
    like evaluator.py:254-273) when it is staged, else the NumPy port."""
    boxes, preds = args
    import numpy as np
    from multigriddet_b200 import synth
    anchors = synth.coco_anchors(np.float32)
    shapes = synth.image_shapes(0, boxes.shape[0], mixed=True)
    if _reference_staged():
        from oracle import ref_loader
        enc = ref_loader.load_staged_encoder()
        post = ref_loader.load_postprocess(staged_copy=True)
        dec = post.MultiGridDecoder(anchors, C, input_shape=(S, S))
        t0 = time.perf_counter()
        enc(boxes.copy(), (S, S), anchors, C, False)
        t1 = time.perf_counter()
        for b in range(boxes.shape[0]):
            dec.postprocess([p[b:b + 1] for p in preds], tuple(int(v) for v in shapes[b]), (S, S),
                            max_boxes=POST["max_boxes"], confidence=POST["confidence"],
                            nms_threshold=POST["nms_threshold"], nms_method=POST["nms_method"])
        t2 = time.perf_counter()
        return t1 - t0, t2 - t1
    from oracle import mgd_oracle as O
    t0 = time.perf_counter()
    O.encode_targets(boxes, (S, S), anchors, C)
    t1 = time.perf_counter()
    O.postprocess_batch(preds, shapes, (S, S), anchors, C, **POST)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def _cpu_kind():
    if _reference_staged():
        return "reference", ("the reference's own sources staged under oracle/_ref by oracle/build_ref.py "
                             "(preprocess_true_boxes + MultiGridDecoder.postprocess per image)")
    return "port", "oracle/mgd_oracle.py (NumPy port of the reference path; oracle/_ref is not staged)"


def cpu_baseline_single(n_images=320):
    """The reference's CPU path on ONE host core, bounded sample (~10-15 s)."""
    _, boxes, preds = _cpu_inputs(n_images)
    te, td = _cpu_worker((boxes, preds))
    kind, what = _cpu_kind()
    return {"value": n_images / (te + td), "unit": UNIT, "cores": 1, "kind": kind,
            "sample": f"{n_images} images (same COCO-608 workload): encode {n_images / te:.1f} img/s, "
                      f"decode+DIoU-NMS {n_images / td:.1f} img/s, {what}, 1 host core",
            "encode_images_per_s": n_images / te, "decode_nms_images_per_s": n_images / td}


def run_reference(args):
    """--impl reference: the reference's CPU path on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    per_worker = 8
    n_images = cores * per_worker
    _, boxes, preds = _cpu_inputs(n_images)
    _SHARDS[:] = [(boxes[i * per_worker:(i + 1) * per_worker],
                   [p[i * per_worker:(i + 1) * per_worker] for p in preds]) for i in range(cores)]
    kind, what = _cpu_kind()
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        for _ in range(args.warmup):
            pool.map(_cpu_worker_indexed, range(cores), chunksize=1)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_cpu_worker_indexed, range(cores), chunksize=1)
        dt = time.perf_counter() - t0
    value = n_images * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "images_per_step": n_images},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{n_images} images/step sharded over {cores} processes: {what}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    return json.dumps(line)


# ------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------

def bind_near_gpu(index):
    """One process per GPU: run this rank's host threads on the CPUs next to its GPU, so the
    page-locked buffers of the host-memory path are first-touched on that NUMA node and the
    PCIe traffic does not cross the socket interconnect.  Returns the CPU count or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if index < len(ids) and ids[index].isdigit():
                index = int(ids[index])
        handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        return len(os.sched_getaffinity(0))
    except Exception:
        return None


def make_device_inputs(batch, device, seed):
    import numpy as np
    import torch
    from multigriddet_b200 import engine, synth
    anchors = synth.coco_anchors(np.float32)
    unique = min(batch, 512)
    base = synth.synth_boxes(seed, unique, NBOX, S, C)
    reps = (batch + unique - 1) // unique
    boxes = np.tile(base, (reps, 1, 1))[:batch]
    d_boxes = torch.from_numpy(boxes).to(device)
    preds = [torch.empty((batch, g, g, D), dtype=torch.float32, device=device)
             for g in (19, 38, 76)]
    chunk = 256
    for b0 in range(0, batch, chunk):
        yt = engine.encode_targets(d_boxes[b0:b0 + chunk], (S, S), anchors, C)
        pl = synth.planted_head_outputs(yt, A, seed * 1000 + b0)
        for dst, src in zip(preds, pl):
            dst[b0:b0 + chunk].copy_(src)
        del yt, pl
    torch.cuda.synchronize()
    return anchors, boxes, d_boxes, preds


def _time_gpu(fn, steps, warmup, barrier):
    """Device time of `steps` calls of fn (CUDA events on the current stream), in ms."""
    import torch
    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    return e0.elapsed_time(e1)


DUMP_BYTES = 63 * 10 ** 6         # array bytes: under 64 MB on disk, .npy headers included
DUMP_Y_IMAGES = 16


def dump_outputs(out_dir, det, y_true):
    """--dump-outputs: the detection tensors and y_true of the timed step's last call, as
    float32 / float64 .npy files of at most DUMP_BYTES in all, so that two builds can be
    compared output for output.  y_true is DUMP_Y_IMAGES images drawn with a fixed seed (a
    batch is gigabytes); the detections are every image's, or a seeded sample of images when
    they do not fit.  `<part>_images.npy` holds the batch indices each part was taken from."""
    import numpy as np
    import torch
    rng = np.random.default_rng(0)

    def pick(n, k):
        return np.sort(rng.choice(n, k, replace=False)) if k < n else np.arange(n)

    n_y = int(y_true[0].shape[0])
    y_img = pick(n_y, min(n_y, DUMP_Y_IMAGES))
    sel = torch.from_numpy(y_img).to(y_true[0].device)
    arrays = {f"y_true_{int(y.shape[1])}": y.index_select(0, sel).cpu().numpy() for y in y_true}
    arrays["y_true_images"] = y_img.astype(np.float64)
    left = DUMP_BYTES - sum(a.nbytes for a in arrays.values())
    # integer outputs go out as float64, which holds every int32 exactly
    keys = ("boxes_xyxy", "scores", "classes", "counts")
    n_det = int(det["counts"].shape[0])
    per_image = 8 + sum(det[k][0].numel() * 8 for k in keys)
    d_img = pick(n_det, min(n_det, left // per_image))
    sel = torch.from_numpy(d_img).to(det["counts"].device)
    for k in keys:
        arrays[k] = det[k].index_select(0, sel).cpu().numpy().astype(np.float64)
    arrays["detections_images"] = d_img.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from multigriddet_b200 import engine, sharding, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: multigriddet_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    numa = bind_near_gpu(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    strong = args.scaling == "strong"
    Bs = args.strong_batch                                  # strong scaling: images in total
    lo_s, hi_s = sharding.shard_bounds(Bs, rank, world)
    B = (hi_s - lo_s) if strong else args.batch             # images of this rank per step
    n_alloc = max(B, hi_s - lo_s)
    anchors, boxes_np, d_boxes, preds = make_device_inputs(n_alloc, device, seed=1 + rank)
    y_out = [torch.empty((n_alloc, g, g, D), dtype=torch.float32, device=device) for g in (19, 38, 76)]
    d_hw = torch.from_numpy(synth.image_shapes(rank, n_alloc, mixed=True)).to(device)
    WANT = ("boxes_xyxy", "scores", "classes")
    out_keep = []

    def fused(n=None):
        """The step: ONE library call, mgd_encode_decode_nms (the library runs the y_true writer
        underneath the NMS on an internal stream and joins before the call's work completes)."""
        n = B if n is None else n
        det = engine.grid_step(d_boxes[:n], [y[:n] for y in y_out], [p[:n] for p in preds], d_hw[:n],
                               (S, S), anchors, C, sync=False, want=WANT, **POST)
        out_keep[:] = [det]           # keep this step's outputs alive until the next one
        return det

    def separate(n=None):
        """The same work as two calls on one stream (mgd_encode_targets, mgd_decode_nms)."""
        n = B if n is None else n
        engine.encode_targets(d_boxes[:n], (S, S), anchors, C, out=[y[:n] for y in y_out], sync=False)
        det = engine.decode_nms([p[:n] for p in preds], d_hw[:n], (S, S), anchors, C, sync=False,
                                want=WANT, **POST)
        out_keep[:] = [det]
        return det

    # the detection exchange is set up collectively, once; a host whose GPUs cannot map each
    # other's memory falls back to the NCCL gather (and says so in the line)
    exchange, exchange_error = [None], None
    try:
        exchange[0] = sharding.DetectionExchange(Bs, POST["max_boxes"], device=local)
    except Exception as e:
        exchange_error = repr(e)

    def strong_step(gather="exchange"):
        """configs[4] as written: this rank's slice of the 4 096-image batch plus the exchange
        step -- every rank ends with all detections.  "exchange": the NMS kernels store every
        image's rows into all ranks' tensors while they run (sharding.DetectionExchange: peer
        stores over NVLink, no collective call); "device": one NCCL all-gather of the packed
        lists after the step; "host": all_gather_object of host copies."""
        n = hi_s - lo_s
        if gather == "exchange" and exchange[0] is None:
            gather = "device"
        if gather == "exchange":
            ex = exchange[0]
            engine.grid_step(d_boxes[:n], [y[:n] for y in y_out], [p[:n] for p in preds], d_hw[:n],
                             (S, S), anchors, C, sync=False, want=WANT, out=ex.local(WANT), **POST)
            return ex.full()
        det = fused(n)
        det = {k: v for k, v in det.items() if not k.startswith("_")}
        if gather == "device":
            full = sharding.gather_detections_device(det, Bs)
        else:
            full = sharding.gather_detections(det)
        out_keep[:] = [det, full]
        return full

    step = strong_step if strong else fused
    for _ in range(args.warmup):
        step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        engine.profile_begin()
        barrier()
        ev0.record()
        for _ in range(args.steps):
            out = step()
        ev1.record()
        barrier()
        prof = engine.profile_end()
    engine.poll_status(local)
    n_step_images = (hi_s - lo_s) if strong else B
    if args.dump_outputs and rank == 0:
        # before the measurements below overwrite y_out
        dump_outputs(args.dump_outputs, out, [y[:n_step_images] for y in y_out])
    ms = ev0.elapsed_time(ev1)
    ms_max = max_over_ranks(ms)
    total_images = (Bs if strong else B * world) * args.steps
    value = total_images / (ms_max / 1e3)
    n_det = int(out["counts"].sum().item())

    # ---- the same work as two separate calls on one stream (what the fused call saves) -------
    overlap = None
    if not args.no_overlap_run:
        t_sep = max_over_ranks(_time_gpu(separate, args.steps, 1, barrier))
        overlap = {"value": B * world * args.steps / (t_sep / 1e3), "unit": UNIT,
                   "ms_per_step": t_sep / args.steps,
                   "note": "mgd_encode_targets then mgd_decode_nms as two calls on one stream "
                           "(no overlap); the headline step is the single fused call"}

    # ---- configs[4] as written: strong scaling with the gather on the clock --------------------
    strong_line = None
    if not strong:
        res = {}
        for how in ("exchange", "device", "host"):
            fn = (lambda h=how: strong_step(h))
            if how == "host":
                # host gather synchronises inside (all_gather_object): wall clock, max over ranks
                for _ in range(2):
                    fn()
                barrier()
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    fn()
                torch.cuda.synchronize()
                t = max_over_ranks((time.perf_counter() - t0) * 1e3)
            else:
                t = max_over_ranks(_time_gpu(fn, args.steps, 2, barrier))
            res[how] = {"value": Bs * args.steps / (t / 1e3), "ms_per_step": t / args.steps}
        t_nog = max_over_ranks(_time_gpu(lambda: fused(hi_s - lo_s), args.steps, 1, barrier))
        strong_line = {"scaling": "strong", "total_images_per_step": Bs, "images_per_rank": hi_s - lo_s,
                       "unit": UNIT, "value": res["exchange"]["value"],
                       "ms_per_step": res["exchange"]["ms_per_step"],
                       "gather": "sharding.DetectionExchange: the NMS kernels store each image's rows into "
                                 "every rank's tensors as they produce them (peer stores through CUDA-IPC "
                                 "mappings, NVLink for N > 1; two one-warp flag barriers per step, no "
                                 "collective call); every rank ends with all detections",
                       "exchange_timeouts": exchange[0].timeouts() if exchange[0] is not None else None,
                       "exchange_error": exchange_error,
                       "nccl_gather": dict(res["device"], note="gather_detections_device: one NCCL all-gather "
                                           "of the packed lists after the step (the baseline the exchange replaces)"),
                       "host_gather": dict(res["host"], note="gather_detections: all_gather_object of host copies"),
                       "compute_only_ms_per_step": t_nog / args.steps}

    # ---- rooflines (per-launch CUDA events on the launching stream) ----------------------------
    peak, peak_src = measured_peak()
    kernels = {}
    for kind, nbytes in (("encode_fill", BYTES_ENCODE), ("decode_compact", BYTES_DECODE)):
        tot_ms, launches = prof[kind]
        if launches:
            per_launch_images = n_step_images * args.steps / launches
            sec = tot_ms / launches / 1e3
            gbs = per_launch_images * nbytes / sec / 1e9
            traffic = dram_traffic(kind)
            kernels[kind] = {"ms_total": tot_ms, "launches": launches,
                             "avg_launch_ms": tot_ms / launches,
                             "images_per_launch": per_launch_images,
                             "achieved_gbs": gbs, "frac": gbs / peak,
                             "frac_algorithmic": gbs / peak,
                             "dram_bytes_per_image_ncu": traffic,
                             "dram_gbs": per_launch_images * traffic / sec / 1e9 if traffic else None,
                             "frac_dram": per_launch_images * traffic / sec / 1e9 / peak if traffic else None}
    for kind in ("encode_assign", "nms"):
        tot_ms, launches = prof[kind]
        kernels[kind] = {"ms_total": tot_ms, "launches": launches,
                         "avg_launch_ms": tot_ms / max(launches, 1)}
    dominant = max(("encode_fill", "decode_compact"), key=lambda k: prof[k][0])
    dk = kernels[dominant]
    roofline = {"bound": "hbm", "kernel": dominant, "achieved": dk["achieved_gbs"], "peak": peak,
                "unit": "GB/s", "frac": dk["frac"],
                "frac_algorithmic": dk["frac_algorithmic"], "frac_dram": dk["frac_dram"],
                "traffic": dk["dram_bytes_per_image_ncu"] * dk["images_per_launch"]
                           if dk["dram_bytes_per_image_ncu"] else None,
                "peak_source": peak_src, "frac_of_nominal_8tbs": dk["achieved_gbs"] / 8000.0,
                "algorithmic_bytes_per_image": BYTES_ENCODE if dominant == "encode_fill" else BYTES_DECODE,
                "note": "achieved / frac(_algorithmic): the bytes the reference's algorithm touches per "
                        "launch over the launch's CUDA-event time; frac_dram: the DRAM bytes ncu counted "
                        "for the kernel (profiles/traffic.json) over the same time.  The decoder reads "
                        "less than the algorithmic bytes (its filter never asks for the rest), so its "
                        "frac_algorithmic can exceed 1; see kernels.decode_compact",
                "step_frac_of_hbm_peak": (BYTES_ENCODE + BYTES_DECODE) * n_step_images * args.steps
                                         / (ms / 1e3) / 1e9 / peak}
    gpu_launches = sum(v[1] for v in prof.values())

    # ---- end to end through the C ABI with pinned host buffers ----------------------------------
    e2e = None
    if not args.no_e2e:
        Be = min(args.e2e_batch, B)
        h_boxes = torch.from_numpy(boxes_np[:Be].copy()).pin_memory()
        h_preds = [p[:Be].cpu().pin_memory() for p in preds]
        h_y = [torch.empty((Be, g, g, D), dtype=torch.float32).pin_memory() for g in (19, 38, 76)]
        hw_np = d_hw[:Be].cpu().numpy()
        np_preds = [p.numpy() for p in h_preds]
        np_y = [y.numpy() for y in h_y]

        # encode (device->host heavy) and decode (host->device heavy) are independent calls of
        # the same C ABI; issued from two host threads they use both PCIe directions at once
        from concurrent.futures import ThreadPoolExecutor
        pool = ThreadPoolExecutor(2)

        zc = [False, False]            # [decoder reads the page-locked predictions in place,
                                       #  writer stores y_true straight into host memory]

        def e2e_encode():
            torch.cuda.set_device(local)
            return engine.encode_targets(h_boxes.numpy(), (S, S), anchors, C, out=np_y, zerocopy=zc[1])

        def e2e_decode():
            torch.cuda.set_device(local)
            return engine.decode_nms(np_preds, hw_np, (S, S), anchors, C, want=WANT, zerocopy=zc[0], **POST)

        def e2e_concurrent():
            fe, fd = pool.submit(e2e_encode), pool.submit(e2e_decode)
            fe.result()
            return fd.result()

        def e2e_sequential():
            e2e_encode()
            return e2e_decode()

        # How to issue the two independent calls is the caller's choice and depends on the
        # host: alone on its link a GPU moves both directions at once (concurrent wins); with
        # several GPUs saturating the host's memory interface the directions only get in each
        # other's way.  Time both on warm-up steps, all ranks together, and use the faster one.
        # The same goes for HOW the predictions reach the decoder: staged through device memory
        # in bulk copies, or read in place by the kernel (MGD_FLAG_HOST_ZEROCOPY: only the
        # sectors the filter asks for cross the link -- fewer bytes through the host's memory
        # interface, which is what several GPUs on one host run out of; finer-grained traffic on
        # the link, which is what a single GPU runs out of).
        trial = {}
        zc_modes = {"": (False, False), "+zerocopy": (True, False), "+zerocopy_both": (True, True)}
        for suffix, mode in zc_modes.items():
            zc[:] = mode
            for name, fn in (("concurrent", e2e_concurrent), ("sequential", e2e_sequential)):
                fn()
                barrier()
                tt = time.perf_counter()
                fn()
                fn()
                torch.cuda.synchronize()
                trial[name + suffix] = max_over_ranks(time.perf_counter() - tt) / 2
        issue = min(trial, key=trial.get)
        zc[:] = zc_modes[issue[issue.index("+"):] if "+" in issue else ""]
        e2e_step = e2e_concurrent if issue.startswith("concurrent") else e2e_sequential
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            res = e2e_step()
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)

        # what the links themselves do with the same bytes: one bulk H2D and one bulk D2H of the
        # step's tensors from the same pinned buffers (no kernels, no chunking), ALL RANKS AT ONCE
        # (barriered), the directions together and one after the other -- the contended rate is
        # the honest denominator on a multi-GPU host
        d_in = [torch.empty_like(p, device=device) for p in h_preds]
        d_outb = [torch.empty_like(y, device=device) for y in h_y]
        s_up, s_dn = torch.cuda.Stream(device=device), torch.cuda.Stream(device=device)

        def link_step(both=True):
            with torch.cuda.stream(s_up):
                for d, h in zip(d_in, h_preds):
                    d.copy_(h, non_blocking=True)
            if not both:
                s_up.synchronize()
            with torch.cuda.stream(s_dn):
                for h, d in zip(h_y, d_outb):
                    h.copy_(d, non_blocking=True)

        link = {}
        for name, both in (("concurrent", True), ("sequential", False)):
            link_step(both)
            barrier()
            t1 = time.perf_counter()
            for _ in range(args.e2e_steps):
                link_step(both)
            torch.cuda.synchronize()
            link[name] = max_over_ranks(time.perf_counter() - t1) / args.e2e_steps
        dt_link = min(link.values())
        del d_in, d_outb
        h2d = Be * NBOX * 5 * 4 + sum(p.numel() * 4 for p in h_preds) + Be * 8
        d2h = sum(y.numel() * 4 for y in h_y) + Be * (100 * (16 + 8 + 4) + 4)
        e2e = {"value": Be * world * args.e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "batch": Be, "steps": args.e2e_steps,
               "detections_last_step": int(res["counts"].sum()),
               "pcie": {"bound": "pcie / host memory", "bare_copy_ms": {k: v * 1e3 for k, v in link.items()},
                        "achieved_gbs_per_rank": (h2d + d2h) / (dt / args.e2e_steps) / 1e9,
                        "peak_gbs_per_rank": (h2d + d2h) / dt_link / 1e9,
                        "frac": dt_link / (dt / args.e2e_steps),
                        "note": "peak = the same bytes as bare bulk copies (H2D and D2H, together or one "
                                "after the other, whichever is faster) issued by ALL ranks at once behind "
                                "a barrier, max over ranks: the contended rate of this host"},
               "issue": issue, "issue_trial_ms": {k: v * 1e3 for k, v in trial.items()},
               "note": "pinned host buffers, host<->device traffic inside; the two calls of a step are "
                       "issued concurrently from two host threads or back to back, and the decoder gets "
                       "its predictions staged in bulk copies or reads them in place over the link "
                       "(+zerocopy: MGD_FLAG_HOST_ZEROCOPY, then only the sectors its filter asks for "
                       "cross, h2d_bytes_per_step stays the size of the tensors handed over; "
                       "+zerocopy_both: the writer also stores y_true straight into host memory) -- whichever "
                       "the warm-up steps found fastest on this host (see issue / issue_trial_ms)"}
        pool.shutdown()
        del h_preds, h_y, np_preds, np_y

    # ---- extra workloads (never the headline; each guarded: an extra must not cost the line) ----
    extras = {}
    if rank == 0 and not args.no_extras:
        def guarded(name, fn):
            try:
                extras[name] = fn()
            except Exception as exc:
                extras[name] = {"error": repr(exc)}

        def solo(fn, n=10):
            """ms per call, this rank alone (no barrier: the other ranks are idle or in their own extras)."""
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n

        def x_dense():
            # SURVEY 8d (ii): every channel N(0,1) -- every cell a candidate, the decoder's worst case
            Bd = 256
            dp = synth.dense_random_head_outputs(Bd, S, A, C, seed=5, device=device)
            hw = d_hw[:Bd]
            engine.profile_begin()
            t = solo(lambda: engine.decode_nms(dp, hw, (S, S), anchors, C, sync=False, want=WANT, **POST))
            pr = engine.profile_end()
            dec_ms = pr["decode_compact"][0] / max(pr["decode_compact"][1], 1)
            return {"workload": "dense random head (all channels N(0,1)): 7 581 candidates per image",
                    "batch": Bd, "ms_per_call": t, "images_per_s": Bd / (t / 1e3),
                    "decode_ms": dec_ms, "nms_ms": pr["nms"][0] / max(pr["decode_compact"][1], 1),
                    "decode_frac_of_hbm_peak": Bd * BYTES_DECODE / (dec_ms / 1e3) / 1e9 / peak,
                    "note": "every row takes the exact path and every byte is read: algorithmic == DRAM bytes"}

        def x_small():
            # BASELINE configs 2 and 3 as written (device tensors, one call each)
            r = {}
            t = solo(lambda: engine.encode_targets(d_boxes[:64], (S, S), anchors, C,
                                                   out=[y[:64] for y in y_out], sync=False), 20)
            r["encode_b64"] = {"ms_per_call": t, "images_per_s": 64 / (t / 1e3),
                               "frac_of_hbm_peak": 64 * BYTES_ENCODE / (t / 1e3) / 1e9 / peak}
            for name, pc in (("decode_nms_b256", False), ("decode_nms_b256_per_class", True)):
                kw = dict(POST, per_class=pc)
                t = solo(lambda: engine.decode_nms([p[:256] for p in preds], d_hw[:256], (S, S), anchors, C,
                                                   sync=False, want=WANT, **kw), 20)
                r[name] = {"ms_per_call": t, "images_per_s": 256 / (t / 1e3),
                           "frac_of_hbm_peak": 256 * BYTES_DECODE / (t / 1e3) / 1e9 / peak}
            r["note"] = ("BASELINE.json configs[1] (B = 64 encode) and configs[2] (B = 256 decode + NMS, "
                         "class-agnostic and per-class), whole call, algorithmic bytes over the call's time")
            return r

        def x_dropin():
            # the reference's own calling convention (evaluator.py:254-289): one image per
            # MultiGridDecoder.postprocess call, ordinary pageable NumPy arrays in and out
            from concurrent.futures import ThreadPoolExecutor
            from multigriddet_b200.postprocess import MultiGridDecoder
            n = 64
            imgs = [[p[b:b + 1].cpu().numpy() for p in preds] for b in range(n)]
            shp = d_hw[:n].cpu().numpy()
            dec = MultiGridDecoder(anchors, C, input_shape=(S, S))

            def one(b):
                torch.cuda.set_device(local)
                return dec.postprocess(imgs[b], tuple(int(v) for v in shp[b]), (S, S), max_boxes=100,
                                       confidence=POST["confidence"], nms_threshold=POST["nms_threshold"],
                                       nms_method="diou")
            one(0)
            t0 = time.perf_counter()
            for b in range(n):
                one(b)
            t_serial = (time.perf_counter() - t0) / n
            with ThreadPoolExecutor(8) as ex:
                list(ex.map(one, range(8)))
                t0 = time.perf_counter()
                list(ex.map(one, range(n)))
                t_thr = (time.perf_counter() - t0) / n
            batch_in = [np.concatenate([im[l] for im in imgs]) for l in range(3)]     # pageable, like the rest

            def batched():
                return dec.postprocess_batch(batch_in, shp, (S, S), 100, POST["confidence"],
                                             POST["nms_threshold"], "diou")
            batched()                                      # warm-up (staging buffers), like `one(0)` above
            t0 = time.perf_counter()
            for _ in range(3):
                batched()
            t_batch = (time.perf_counter() - t0) / 3 / n
            return {"images": n, "ms_per_image_serial": t_serial * 1e3, "images_per_s_serial": 1 / t_serial,
                    "ms_per_image_8_threads": t_thr * 1e3, "images_per_s_8_threads": 1 / t_thr,
                    "ms_per_image_one_batched_call": t_batch * 1e3,
                    "note": "e2e_dropin: pageable NumPy in / out through MultiGridDecoder.postprocess, one "
                            "image per call (the evaluator's usage, serial and from 8 threads), and the "
                            "same images as one postprocess_batch call"}

        def x_map():
            Bm = min(B, 1024)
            det = fused(Bm)
            gt = torch.from_numpy(boxes_np[:Bm]).to(device)
            gt_boxes = gt[..., :4].double().contiguous()
            gt_cls = gt[..., 4].int().contiguous()
            gt_n = ((gt[..., 2] - gt[..., 0]) * (gt[..., 3] - gt[..., 1]) > 0).sum(1).int()
            thr = [0.5 + 0.05 * i for i in range(10)]
            margs = (det["boxes_xyxy"].double(), det["scores"], det["classes"], det["counts"],
                     gt_boxes, gt_cls, gt_n, thr)
            tp = engine.match_detections(*margs)
            t = solo(lambda: engine.match_detections(*margs, sync=False), 5)
            return {"images_per_s": Bm / (t / 1e3), "images": Bm, "iou_thresholds": 10,
                    "tp_at_0.5": int(tp[0].sum().item()), "detections": int(det["counts"].sum().item()),
                    "note": "mgd_match_detections on device tensors (latency-bound, no roofline claimed)"}

        guarded("dense_random", x_dense)
        guarded("small_batch", x_small)
        guarded("e2e_dropin", x_dropin)
        guarded("map_matching", x_map)
    barrier()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_single()

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "images_per_rank_per_step": n_step_images,
                       "images_per_step_total": Bs if strong else B * world,
                       "sharding": (f"image-sharded x{world}; " +
                                    (("detections written into every rank's tensors by the NMS kernels (peer stores, no collective call)"
                                      if exchange[0] is not None else "detection lists all-gathered every step (NCCL)")
                                     if strong else "no collective")),
                       "step": "one mgd_encode_decode_nms call per rank (encode + decode + NMS; the library "
                               "overlaps the y_true writer with the NMS internally)",
                       "cpus_bound_to_rank": numa,
                       "l2": "inputs larger than L2 (2 x 2.67 MB/image x batch), no flush needed"},
            "roofline": roofline, "kernels": kernels, "separate_calls": overlap,
            "strong_scaling": strong_line,
            "cpu_baseline": cpu, "e2e": e2e,
            "clocks": clocks.summary(), "gpu_launches": gpu_launches,
            "detections_last_step": n_det, "extras": extras or None,
        }
    if world > 1:
        dist.destroy_process_group()
    return json.dumps(line) if rank == 0 else None


def main():
    args = parse()
    # stdout carries exactly one JSON line: anything a library prints there meanwhile (NCCL's
    # version banner, for one) is sent to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        line = run_reference(args) if args.impl == "reference" else run_b200(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    if line:
        print(line, flush=True)


if __name__ == "__main__":
    main()
