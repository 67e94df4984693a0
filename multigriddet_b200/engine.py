"""Array-level entry points over the C ABI.

Accepts NumPy arrays (host memory: the library stages through the GPU), torch
CUDA tensors (device memory, zero-copy, enqueued on the current torch stream)
and any other object exporting ``__dlpack__`` (e.g. TensorFlow tensors via
``tf.experimental.dlpack``), which goes through the ``*_dlpack`` entry points.
Outputs are allocated here, in the same memory space as the inputs, and handed
to the library: the library never owns tensor memory.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib

_NMS_METHODS = {"diou": _lib.NMS_DIOU, "standard": _lib.NMS_IOU, "iou": _lib.NMS_IOU,
                "cluster": _lib.NMS_IOU, "soft": _lib.NMS_SOFT, "wbf": _lib.NMS_WBF}


def _is_torch(x) -> bool:
    return type(x).__module__.split(".")[0] == "torch"


def _torch_stream(device_index: int) -> int:
    import torch
    return int(torch.cuda.current_stream(device_index).cuda_stream)


def _current_device() -> int:
    # host-memory calls run on the caller's current CUDA device when torch is in the
    # process (one rank per GPU under torchrun), else on device 0
    import sys
    torch = sys.modules.get("torch")
    if torch is not None and torch.cuda.is_available():
        return int(torch.cuda.current_device())
    return 0


def device_count() -> int:
    return int(_lib.load().mgd_device_count())


def post_config(max_boxes=100, confidence=0.1, nms_threshold=0.5, nms_method="diou",
                per_class=False, use_softmax=True, rescore_confidence=True,
                soft_sigma=0.5, soft_score_threshold=0.001) -> _lib.PostConfig:
    if nms_method not in _NMS_METHODS:
        raise NotImplementedError(
            f"nms_method={nms_method!r}: the CUDA path implements 'diou', 'standard', "
            "'cluster' (greedy hard NMS), 'soft' (Gaussian SoftNMS) and 'wbf' (use_wbf=True)")
    pc = _lib.PostConfig()
    pc.use_softmax = int(bool(use_softmax))
    pc.rescore_confidence = int(bool(rescore_confidence))
    pc.confidence = float(confidence)
    pc.nms_threshold = float(nms_threshold)
    pc.nms_method = _NMS_METHODS[nms_method]
    pc.per_class = int(bool(per_class))
    pc.max_boxes = int(max_boxes)
    pc.soft_sigma = float(soft_sigma)
    pc.soft_score_threshold = float(soft_score_threshold)
    return pc


# ------------------------------------------------------------------------------
# encode
# ------------------------------------------------------------------------------

def encode_targets(true_boxes, input_shape, anchors, num_classes, grid_shapes=None,
                   out=None, sync=True, return_stats=False, semantics="numpy", zerocopy=False):
    """Multi-grid y_true encoder.  ``semantics="numpy"``: the reference's
    ``preprocess_true_boxes``; ``"tf_compat"``: its TensorFlow encoder
    ``tf_preprocess_true_boxes`` (MGD_FLAG_TF_COMPAT, include/mgd.h).

    true_boxes: (B, N, 5) NumPy array (any dtype) or torch CUDA float32 tensor.
    Returns a list of L arrays/tensors (B, Gh, Gw, 5+A+C) float32 in the same
    memory space.  ``sync=False`` (device tensors only) returns right after the
    kernels are enqueued on the current stream; class-range errors then surface
    at the next ``poll_status``.  ``zerocopy=True`` (host arrays in page-locked memory): the
    writer stores y_true straight into host memory (MGD_FLAG_HOST_ZEROCOPY).
    """
    lib = _lib.load()
    if semantics not in ("numpy", "tf_compat"):
        raise ValueError(f"semantics must be 'numpy' or 'tf_compat', got {semantics!r}")
    mode = _lib.FLAG_TF_COMPAT if semantics == "tf_compat" else 0
    cfg = _lib.make_head_config(anchors, num_classes, input_shape, grid_shapes)
    L = cfg.num_layers
    stats = (ctypes.c_longlong * 4)()
    if _is_torch(true_boxes):
        import torch
        if not true_boxes.is_cuda:
            raise ValueError("torch tensors must live on a CUDA device (pass NumPy for host data)")
        boxes = true_boxes.to(torch.float32).contiguous()
        if boxes.dim() != 3 or boxes.shape[2] != 5:
            raise ValueError(f"true_boxes must be (B, N, 5), got {tuple(boxes.shape)}")
        B, N = int(boxes.shape[0]), int(boxes.shape[1])
        dev = boxes.device.index or 0
        if out is None:
            out = [torch.empty((B, cfg.grid_h[l], cfg.grid_w[l], 5 + cfg.num_anchors[l] + cfg.num_classes),
                               dtype=torch.float32, device=boxes.device) for l in range(L)]
        ptrs = _lib.ptr_array([o.data_ptr() for o in out])
        rc = lib.mgd_encode_targets(ctypes.byref(cfg), ctypes.c_void_p(boxes.data_ptr()), B, N,
                                    ptrs, _lib.MEM_DEVICE, dev,
                                    ctypes.c_void_p(_torch_stream(dev)),
                                    (_lib.FLAG_SYNC if sync else 0) | mode, stats)
    else:
        boxes = np.ascontiguousarray(np.asarray(true_boxes), dtype=np.float32)
        if boxes.ndim != 3 or boxes.shape[2] != 5:
            raise ValueError(f"true_boxes must be (B, N, 5), got {boxes.shape}")
        B, N = boxes.shape[0], boxes.shape[1]
        if out is None:
            # page-locked, recycled: pageable outputs crawl through the driver's bounce buffer
            out = [_lib.pinned.empty((B, cfg.grid_h[l], cfg.grid_w[l],
                                      5 + cfg.num_anchors[l] + cfg.num_classes), np.float32)
                   for l in range(L)]
        ptrs = _lib.ptr_array([o.ctypes.data for o in out])
        rc = lib.mgd_encode_targets(ctypes.byref(cfg), ctypes.c_void_p(boxes.ctypes.data), B, N,
                                    ptrs, _lib.MEM_HOST, _current_device(), None,
                                    _lib.FLAG_SYNC | mode | (_lib.FLAG_HOST_ZEROCOPY if zerocopy else 0), stats)
    _lib.raise_for_status(rc)
    if return_stats:
        return out, {"n_valid_boxes": int(stats[0]), "n_skipped_writes": int(stats[1]),
                     "n_positive_cells": int(stats[2])}
    return out


def poll_status(device=None, stream=None):
    """Synchronise and raise any deferred device-side error of async calls."""
    lib = _lib.load()
    dev = _current_device() if device is None else int(device)
    st = _torch_stream(dev) if stream is None else int(stream)
    _lib.raise_for_status(lib.mgd_poll_status(dev, ctypes.c_void_p(st)))


# ------------------------------------------------------------------------------
# decode + NMS
# ------------------------------------------------------------------------------

def _check_out(given, spec, B, device):
    """Validate caller-provided output tensors (decode_nms / grid_step ``out=``)."""
    import torch
    if "counts" not in given:
        raise ValueError("out= needs a 'counts' tensor")
    res = {}
    for k, t in given.items():
        shape, dt = ((B,), "int32") if k == "counts" else spec.get(k, (None, None))
        if shape is None:
            raise ValueError(f"out= has an unknown tensor {k!r}")
        dt = getattr(torch, dt) if isinstance(dt, str) else dt
        if not (_is_torch(t) and t.is_cuda and t.device == device and t.is_contiguous()
                and t.dtype == dt and tuple(t.shape) == tuple(shape)):
            raise ValueError(f"out[{k!r}] must be a contiguous {dt} CUDA tensor of shape {tuple(shape)}")
        res[k] = t
    return res


def decode_nms(preds, image_shapes, model_image_size, anchors, num_classes, max_boxes=100,
               confidence=0.1, nms_threshold=0.5, nms_method="diou", per_class=False,
               use_softmax=True, rescore_confidence=True, sync=True, return_stats=False,
               want=("boxes_xywh", "boxes_xyxy", "scores", "classes", "index"), out=None,
               zerocopy=False):
    """Batched decode -> threshold -> NMS -> top-k (B independent reference calls).

    preds: list of L (B, Gh, Gw, 5+A+C) float32 NumPy arrays or torch CUDA tensors.
    image_shapes: None (model input size), one (h, w), or (B, 2).
    out: (torch path) dict of preallocated contiguous CUDA tensors to write into -- 'counts'
    (B,) int32 plus any of ``want`` with the shapes / dtypes below; tensors taken from a
    ``sharding.DetectionExchange`` are mirrored to every rank by the kernels.
    zerocopy=True (NumPy predictions in page-locked memory): the decoder reads them in place
    over the link, only the sectors its filter asks for (MGD_FLAG_HOST_ZEROCOPY).
    Returns a dict of padded arrays/tensors + 'counts' (B,).
    """
    lib = _lib.load()
    L = len(preds)
    if L != len(anchors):
        raise ValueError(f"Expected {len(anchors)} predictions, got {L}")   # multigrid_decode.py:62-63
    grid_shapes = [(int(p.shape[1]), int(p.shape[2])) for p in preds]
    cfg = _lib.make_head_config(anchors, num_classes, model_image_size, grid_shapes)
    pc = post_config(max_boxes, confidence, nms_threshold, nms_method, per_class, use_softmax,
                     rescore_confidence)
    B = int(preds[0].shape[0])
    for l, p in enumerate(preds):
        exp = (B, cfg.grid_h[l], cfg.grid_w[l], 5 + cfg.num_anchors[l] + cfg.num_classes)
        if tuple(int(v) for v in p.shape) != exp:
            raise ValueError(f"preds[{l}] has shape {tuple(p.shape)}, expected {exp}")
    M = int(max_boxes)
    stats = (ctypes.c_longlong * 4)()
    hw = None
    d_hw = None
    if image_shapes is not None and _is_torch(image_shapes):
        import torch
        d_hw = image_shapes.to(torch.int32).contiguous()
        if tuple(d_hw.shape) != (B, 2) or not d_hw.is_cuda:
            raise ValueError("a tensor image_shapes must be a CUDA (B, 2) tensor")
    elif image_shapes is not None:
        hw = np.asarray(image_shapes, dtype=np.int32).reshape(-1, 2)
        if hw.shape[0] == 1 and B != 1:
            hw = np.tile(hw, (B, 1))
        if hw.shape[0] != B:
            raise ValueError(f"image_shapes must be (h, w) or (B, 2); got {hw.shape} for B={B}")
        hw = np.ascontiguousarray(hw)
    spec = {"boxes_xywh": ((B, M, 4), "float64"), "boxes_xyxy": ((B, M, 4), "int32"),
            "scores": ((B, M), "float64"), "classes": ((B, M), "int32"),
            "index": ((B, M), "int32")}
    given, out = out, {}
    if given is not None and not _is_torch(preds[0]):
        raise ValueError("out= is only supported with torch CUDA tensors")
    if _is_torch(preds[0]):
        import torch
        dev = preds[0].device.index or 0
        tp = [p.to(torch.float32).contiguous() for p in preds]
        if given is not None:
            out = _check_out(given, spec, B, tp[0].device)
        else:
            for k in want:
                out[k] = torch.empty(spec[k][0], dtype=getattr(torch, spec[k][1]), device=tp[0].device)
            out["counts"] = torch.empty((B,), dtype=torch.int32, device=tp[0].device)
        if d_hw is None and hw is not None:
            d_hw = torch.from_numpy(hw).to(tp[0].device, non_blocking=False)
        addr = lambda k: ctypes.c_void_p(out[k].data_ptr()) if k in out else None
        rc = lib.mgd_decode_nms(
            ctypes.byref(cfg), ctypes.byref(pc), _lib.ptr_array([p.data_ptr() for p in tp]), B,
            ctypes.c_void_p(d_hw.data_ptr()) if d_hw is not None else None,
            addr("boxes_xywh"), addr("boxes_xyxy"), addr("scores"), addr("classes"),
            addr("index"), addr("counts"), _lib.MEM_DEVICE, dev,
            ctypes.c_void_p(_torch_stream(dev)), _lib.FLAG_SYNC if sync else 0, stats)
        out["_keepalive"] = (tp, d_hw)
    else:
        npreds = [np.ascontiguousarray(np.asarray(p), dtype=np.float32) for p in preds]
        for k in want:
            out[k] = _lib.pinned.empty(spec[k][0], spec[k][1])
        out["counts"] = np.empty((B,), dtype=np.int32)
        addr = lambda k: ctypes.c_void_p(out[k].ctypes.data) if k in out else None
        rc = lib.mgd_decode_nms(
            ctypes.byref(cfg), ctypes.byref(pc), _lib.ptr_array([p.ctypes.data for p in npreds]), B,
            ctypes.c_void_p(hw.ctypes.data) if hw is not None else None,
            addr("boxes_xywh"), addr("boxes_xyxy"), addr("scores"), addr("classes"),
            addr("index"), addr("counts"), _lib.MEM_HOST, _current_device(), None,
            _lib.FLAG_SYNC | (_lib.FLAG_HOST_ZEROCOPY if zerocopy else 0), stats)
    _lib.raise_for_status(rc)
    if not sync:
        return out
    out.pop("_keepalive", None)
    if return_stats:
        out["stats"] = {"n_candidates": int(stats[0]), "n_detections": int(stats[1])}
    return out


def grid_step(true_boxes, y_true, preds, image_shapes, input_shape, anchors, num_classes,
              max_boxes=100, confidence=0.1, nms_threshold=0.5, nms_method="diou", per_class=False,
              use_softmax=True, rescore_confidence=True, sync=True,
              want=("boxes_xywh", "boxes_xyxy", "scores", "classes", "index"), out=None):
    """Both halves of the grid path in one library call on torch CUDA tensors
    (``mgd_encode_decode_nms``): ``y_true`` (list of preallocated (Be, G, G, D) tensors) is
    overwritten with the targets of ``true_boxes`` while ``preds`` are decoded and suppressed;
    the library overlaps the two internally.  Returns the detection dict of ``decode_nms``."""
    import torch
    lib = _lib.load()
    if len(preds) != len(anchors) or len(y_true) != len(anchors):
        raise ValueError(f"Expected {len(anchors)} tensors per list")
    grid_shapes = [(int(p.shape[1]), int(p.shape[2])) for p in preds]
    cfg = _lib.make_head_config(anchors, num_classes, input_shape, grid_shapes)
    pc = post_config(max_boxes, confidence, nms_threshold, nms_method, per_class, use_softmax,
                     rescore_confidence)
    B = int(preds[0].shape[0])
    Be, N = int(true_boxes.shape[0]), int(true_boxes.shape[1])
    dev = preds[0].device.index or 0
    for l, (p, y) in enumerate(zip(preds, y_true)):
        d = 5 + cfg.num_anchors[l] + cfg.num_classes
        if tuple(p.shape) != (B, cfg.grid_h[l], cfg.grid_w[l], d) or \
                tuple(y.shape) != (Be, cfg.grid_h[l], cfg.grid_w[l], d):
            raise ValueError(f"layer {l}: unexpected tensor shape")
        if not (p.is_cuda and y.is_cuda and p.is_contiguous() and y.is_contiguous()
                and p.dtype == torch.float32 and y.dtype == torch.float32):
            raise ValueError("grid_step takes contiguous float32 CUDA tensors")
    tb = true_boxes.to(torch.float32).contiguous()
    d_hw = None
    if image_shapes is not None:
        d_hw = image_shapes if _is_torch(image_shapes) else torch.from_numpy(
            np.ascontiguousarray(np.broadcast_to(np.asarray(image_shapes, np.int32).reshape(-1, 2), (B, 2)))).to(preds[0].device)
        d_hw = d_hw.to(torch.int32).contiguous()
    M = int(max_boxes)
    spec = {"boxes_xywh": ((B, M, 4), torch.float64), "boxes_xyxy": ((B, M, 4), torch.int32),
            "scores": ((B, M), torch.float64), "classes": ((B, M), torch.int32),
            "index": ((B, M), torch.int32)}
    if out is not None:
        out = _check_out(out, spec, B, preds[0].device)
    else:
        out = {k: torch.empty(spec[k][0], dtype=spec[k][1], device=preds[0].device) for k in want}
        out["counts"] = torch.empty((B,), dtype=torch.int32, device=preds[0].device)
    addr = lambda k: ctypes.c_void_p(out[k].data_ptr()) if k in out else None
    rc = lib.mgd_encode_decode_nms(
        ctypes.byref(cfg), ctypes.byref(pc), ctypes.c_void_p(tb.data_ptr()), Be, N,
        _lib.ptr_array([y.data_ptr() for y in y_true]),
        _lib.ptr_array([p.data_ptr() for p in preds]), B,
        ctypes.c_void_p(d_hw.data_ptr()) if d_hw is not None else None,
        addr("boxes_xywh"), addr("boxes_xyxy"), addr("scores"), addr("classes"), addr("index"),
        addr("counts"), dev, ctypes.c_void_p(_torch_stream(dev)), _lib.FLAG_SYNC if sync else 0)
    _lib.raise_for_status(rc)
    if not sync:
        out["_keepalive"] = (tb, d_hw)
    return out


def decode_dense(preds, anchors, num_classes, model_image_size, image_shapes=None,
                 use_softmax=True, rescore_confidence=True):
    """Dense decode (reference ``decode_predictions`` [+ ``correct_boxes``]):
    (B, cells, 5+C) float64."""
    lib = _lib.load()
    if len(preds) != len(anchors):
        raise ValueError(f"Expected {len(anchors)} predictions, got {len(preds)}")
    grid_shapes = [(int(p.shape[1]), int(p.shape[2])) for p in preds]
    cfg = _lib.make_head_config(anchors, num_classes, model_image_size, grid_shapes)
    pc = post_config(use_softmax=use_softmax, rescore_confidence=rescore_confidence)
    B = int(preds[0].shape[0])
    cells = sum(g[0] * g[1] for g in grid_shapes)
    hw = None
    if image_shapes is not None:
        hw = np.asarray(image_shapes, dtype=np.int32).reshape(-1, 2)
        if hw.shape[0] == 1 and B != 1:
            hw = np.tile(hw, (B, 1))
        hw = np.ascontiguousarray(hw)
    if _is_torch(preds[0]):
        import torch
        dev = preds[0].device.index or 0
        tp = [p.to(torch.float32).contiguous() for p in preds]
        out = torch.empty((B, cells, 5 + int(num_classes)), dtype=torch.float64, device=tp[0].device)
        d_hw = torch.from_numpy(hw).to(tp[0].device) if hw is not None else None
        rc = lib.mgd_decode_dense(ctypes.byref(cfg), ctypes.byref(pc),
                                  _lib.ptr_array([p.data_ptr() for p in tp]), B,
                                  ctypes.c_void_p(d_hw.data_ptr()) if d_hw is not None else None,
                                  ctypes.c_void_p(out.data_ptr()), _lib.MEM_DEVICE, dev,
                                  ctypes.c_void_p(_torch_stream(dev)), _lib.FLAG_SYNC)
    else:
        npreds = [np.ascontiguousarray(np.asarray(p), dtype=np.float32) for p in preds]
        out = np.empty((B, cells, 5 + int(num_classes)), dtype=np.float64)
        rc = lib.mgd_decode_dense(ctypes.byref(cfg), ctypes.byref(pc),
                                  _lib.ptr_array([p.ctypes.data for p in npreds]), B,
                                  ctypes.c_void_p(hw.ctypes.data) if hw is not None else None,
                                  ctypes.c_void_p(out.ctypes.data), _lib.MEM_HOST,
                                  _current_device(), None, _lib.FLAG_SYNC)
    _lib.raise_for_status(rc)
    return out


_WBF_CONF = {"avg": 0, "max": 1, "box_and_model_avg": 2, "absent_model_aware_avg": 2}


def wbf(boxes, scores, classes, box_weights=None, iou_thr=0.55, skip_box_thr=0.0, conf_type="avg"):
    """Weighted boxes fusion of (n,4) xywh float64 boxes (reference wbf.py semantics):
    (fused boxes, fused scores, classes) in (class asc, leader score desc) order."""
    lib = _lib.load()
    b = np.ascontiguousarray(np.asarray(boxes, dtype=np.float64).reshape(-1, 4))
    s = np.ascontiguousarray(np.asarray(scores, dtype=np.float64).reshape(-1))
    c = np.ascontiguousarray(np.asarray(classes).astype(np.int32).reshape(-1))
    n = b.shape[0]
    if s.shape[0] != n or c.shape[0] != n:
        raise ValueError("boxes, scores and classes disagree on n")
    w = None
    if box_weights is not None:
        w = np.ascontiguousarray(np.asarray(box_weights, dtype=np.float64).reshape(-1))
    ob = np.empty((max(n, 1), 4), dtype=np.float64)
    osc = np.empty((max(n, 1),), dtype=np.float64)
    oc = np.empty((max(n, 1),), dtype=np.int32)
    n_out = ctypes.c_int(0)
    rc = lib.mgd_wbf(ctypes.c_void_p(b.ctypes.data), ctypes.c_void_p(s.ctypes.data),
                     ctypes.c_void_p(c.ctypes.data),
                     ctypes.c_void_p(w.ctypes.data) if w is not None else None, n, float(iou_thr),
                     float(skip_box_thr), _WBF_CONF.get(conf_type, 0), ctypes.c_void_p(ob.ctypes.data),
                     ctypes.c_void_p(osc.ctypes.data), ctypes.c_void_p(oc.ctypes.data),
                     ctypes.cast(ctypes.byref(n_out), ctypes.c_void_p), _lib.MEM_HOST,
                     _current_device(), None, _lib.FLAG_SYNC)
    _lib.raise_for_status(rc)
    k = n_out.value
    return ob[:k].copy(), osc[:k].copy(), oc[:k].copy()


def soft_nms(boxes, scores, sigma=0.5, score_threshold=0.001):
    """Gaussian SoftNMS on (n,4) xywh float64 boxes: (kept positions in input order,
    their decayed scores)."""
    lib = _lib.load()
    b = np.ascontiguousarray(np.asarray(boxes, dtype=np.float64).reshape(-1, 4))
    s = np.ascontiguousarray(np.asarray(scores, dtype=np.float64).reshape(-1))
    n = b.shape[0]
    if s.shape[0] != n:
        raise ValueError("boxes and scores disagree on n")
    keep = np.empty((max(n, 1),), dtype=np.int32)
    soft = np.empty((max(n, 1),), dtype=np.float64)
    n_keep = ctypes.c_int(0)
    rc = lib.mgd_soft_nms(ctypes.c_void_p(b.ctypes.data), ctypes.c_void_p(s.ctypes.data), n,
                          float(sigma), float(score_threshold), ctypes.c_void_p(keep.ctypes.data),
                          ctypes.c_void_p(soft.ctypes.data),
                          ctypes.cast(ctypes.byref(n_keep), ctypes.c_void_p), _lib.MEM_HOST,
                          _current_device(), None, _lib.FLAG_SYNC)
    _lib.raise_for_status(rc)
    k = n_keep.value
    return keep[:k].astype(np.int64), soft[:k].copy()


def nms(boxes, scores, classes=None, nms_threshold=0.5, nms_method="diou", per_class=False,
        max_keep=0):
    """Greedy NMS on (n,4) xywh float64 boxes; returns kept positions (descending score)."""
    lib = _lib.load()
    if nms_method not in _NMS_METHODS or nms_method in ("soft", "wbf"):
        raise NotImplementedError(f"nms_method={nms_method!r} is not a greedy hard NMS")
    b = np.ascontiguousarray(np.asarray(boxes, dtype=np.float64).reshape(-1, 4))
    s = np.ascontiguousarray(np.asarray(scores, dtype=np.float64).reshape(-1))
    n = b.shape[0]
    if s.shape[0] != n:
        raise ValueError("boxes and scores disagree on n")
    c = None
    if classes is not None:
        c = np.ascontiguousarray(np.asarray(classes).astype(np.int32).reshape(-1))
    keep = np.empty((max(n, 1),), dtype=np.int32)
    n_keep = ctypes.c_int(0)
    rc = lib.mgd_nms(ctypes.c_void_p(b.ctypes.data), ctypes.c_void_p(s.ctypes.data),
                     ctypes.c_void_p(c.ctypes.data) if c is not None else None, n,
                     float(nms_threshold), _NMS_METHODS[nms_method], int(bool(per_class)),
                     int(max_keep), ctypes.c_void_p(keep.ctypes.data),
                     ctypes.cast(ctypes.byref(n_keep), ctypes.c_void_p), _lib.MEM_HOST,
                     _current_device(), None, _lib.FLAG_SYNC)
    _lib.raise_for_status(rc)
    return keep[:n_keep.value].astype(np.int64)


PROFILE_KINDS = ("encode_assign", "encode_fill", "decode_compact", "nms", "other")


def profile_begin():
    """Start per-kernel CUDA-event timing of this thread's library calls."""
    _lib.raise_for_status(_lib.load().mgd_profile_begin())


def profile_end():
    """Stop timing; returns {kernel kind: (total ms, launches)}."""
    ms = (ctypes.c_double * len(PROFILE_KINDS))()
    n = (ctypes.c_longlong * len(PROFILE_KINDS))()
    _lib.raise_for_status(_lib.load().mgd_profile_end(ms, n))
    return {k: (float(ms[i]), int(n[i])) for i, k in enumerate(PROFILE_KINDS)}


# ------------------------------------------------------------------------------
# mAP matching (reference multigriddet/evaluation/metrics.py)
# ------------------------------------------------------------------------------

_IOU_MODES = {"corner": _lib.IOU_CORNER, "centre": _lib.IOU_CENTRE, "center": _lib.IOU_CENTRE}


def match_detections(det_boxes, det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts,
                     iou_thresholds, iou_mode="corner", return_matched=False, sync=True):
    """TP flags of padded per-image detections against padded per-image ground truth
    (``mgd_match_detections``).  NumPy arrays (host) or torch CUDA tensors (device).

    det_boxes (B, M, 4), det_scores (B, M), det_classes (B, M), det_counts (B,),
    gt_boxes (B, N, 4), gt_classes (B, N), gt_counts (B,).  Returns ``tp`` (T, B, M) uint8
    (and ``matched_gt`` (T, B, M) int32 when asked) in the same memory space.
    """
    lib = _lib.load()
    mode = _IOU_MODES[iou_mode]
    thr = np.ascontiguousarray(np.asarray(iou_thresholds, dtype=np.float64).reshape(-1))
    T = int(thr.shape[0])
    thr_p = thr.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    if _is_torch(det_boxes):
        import torch
        dev = det_boxes.device
        f64 = lambda x: x.to(device=dev, dtype=torch.float64).contiguous()
        i32 = lambda x: x.to(device=dev, dtype=torch.int32).contiguous()
        db, ds, dc, dn = f64(det_boxes), f64(det_scores), i32(det_classes), i32(det_counts)
        gb, gc, gn = f64(gt_boxes), i32(gt_classes), i32(gt_counts)
        B, M, N = int(ds.shape[0]), int(ds.shape[1]), int(gc.shape[1])
        tp = torch.empty((T, B, M), dtype=torch.uint8, device=dev)
        who = torch.empty((T, B, M), dtype=torch.int32, device=dev) if return_matched else None
        p = lambda x: ctypes.c_void_p(x.data_ptr()) if x is not None and x.numel() else None
        idx = dev.index or 0
        rc = lib.mgd_match_detections(p(db), p(ds), p(dc), p(dn), B, M, p(gb), p(gc), p(gn), N, thr_p, T,
                                      mode, p(tp), p(who), _lib.MEM_DEVICE, idx,
                                      ctypes.c_void_p(_torch_stream(idx)), _lib.FLAG_SYNC if sync else 0)
    else:
        f64 = lambda x: np.ascontiguousarray(np.asarray(x), dtype=np.float64)
        i32 = lambda x: np.ascontiguousarray(np.asarray(x), dtype=np.int32)
        db, ds, dc, dn = f64(det_boxes), f64(det_scores), i32(det_classes), i32(det_counts)
        gb, gc, gn = f64(gt_boxes), i32(gt_classes), i32(gt_counts)
        B, M, N = ds.shape[0], ds.shape[1], gc.shape[1]
        tp = np.zeros((T, B, M), dtype=np.uint8)
        who = np.full((T, B, M), -1, dtype=np.int32) if return_matched else None
        p = lambda x: ctypes.c_void_p(x.ctypes.data) if x is not None and x.size else None
        rc = lib.mgd_match_detections(p(db), p(ds), p(dc), p(dn), B, M, p(gb), p(gc), p(gn), N, thr_p, T,
                                      mode, p(tp), p(who), _lib.MEM_HOST, _current_device(), None,
                                      _lib.FLAG_SYNC)
    _lib.raise_for_status(rc)
    return (tp, who) if return_matched else tp


_MAP_METHODS = {"coco": _lib.MAP_COCO, "voc": _lib.MAP_VOC}


def map_config(num_classes, iou_thresholds, method="coco", views=(_lib.MAP_VIEW_CORNER,)) -> _lib.MapConfig:
    """``mgd_map_config`` for ``map_update`` / ``map_compute``; raises ValueError on what the
    library would refuse, before any device work."""
    if method not in _MAP_METHODS:
        raise ValueError(f"Unknown method: {method}")
    thr = [float(t) for t in iou_thresholds]
    if not 1 <= len(thr) <= _lib.MAP_MAX_THRESHOLDS:
        raise ValueError(f"between 1 and {_lib.MAP_MAX_THRESHOLDS} IoU thresholds supported, got {len(thr)}")
    if int(num_classes) < 1:
        raise ValueError(f"num_classes must be >= 1, got {num_classes}")
    if not views or any(not 0 <= v < _lib.MAP_VIEWS for v in views):
        raise ValueError(f"views must be a non-empty subset of range({_lib.MAP_VIEWS})")
    cfg = _lib.MapConfig()
    cfg.num_classes = int(num_classes)
    cfg.num_thresholds = len(thr)
    cfg.method = _MAP_METHODS[method]
    cfg.views = sum(1 << v for v in set(views))
    for t, v in enumerate(thr):
        cfg.iou_thresholds[t] = v
    for k, x in enumerate(np.arange(0, 1.1, 0.1)):     # compute_average_precision's VOC recalls
        cfg.voc_recalls[k] = float(x)
    return cfg


def map_record_bytes() -> int:
    """Bytes of the record buffer per padded detection slot (``mgd_map_record_bytes``)."""
    return int(_lib.load().mgd_map_record_bytes())


def map_update(cfg, records, slot_offset, gt_hist, det_boxes, det_scores, det_classes, det_counts,
               gt_boxes, gt_classes, gt_counts, sync=False):
    """Match one batch and write its records at ``slot_offset`` of ``records`` (a CUDA byte
    tensor), adding its ground-truth counts to ``gt_hist`` ((MAP_VIEWS, C) int64 CUDA tensor)
    (``mgd_map_update``).  Torch CUDA tensors in ``match_detections``' layout; boxes may be
    int32 (``decode_nms``' ``boxes_xyxy``).  Enqueued on the current stream; class-range errors
    surface at the next ``poll_status`` unless ``sync``."""
    import torch
    lib = _lib.load()
    dev = records.device
    for name, t in (("det_boxes", det_boxes), ("det_scores", det_scores), ("det_classes", det_classes),
                    ("det_counts", det_counts), ("gt_boxes", gt_boxes), ("gt_classes", gt_classes),
                    ("gt_counts", gt_counts)):
        if not (_is_torch(t) and t.device == dev):
            raise ValueError(f"{name} must be a torch tensor on {dev}")
    f64 = lambda x: x.to(torch.float64).contiguous()
    i32 = lambda x: x.to(torch.int32).contiguous()
    db, ds, dc, dn = f64(det_boxes), f64(det_scores), i32(det_classes), i32(det_counts)
    gb, gc, gn = f64(gt_boxes), i32(gt_classes), i32(gt_counts)
    if ds.dim() != 2 or tuple(db.shape) != (*ds.shape, 4) or dc.shape != ds.shape or tuple(dn.shape) != (ds.shape[0],):
        raise ValueError("detections must be det_boxes (B, M, 4), det_scores / det_classes (B, M), det_counts (B,)")
    B, M = int(ds.shape[0]), int(ds.shape[1])
    if gc.dim() != 2 or gc.shape[0] != B or tuple(gb.shape) != (*gc.shape, 4) or tuple(gn.shape) != (B,):
        raise ValueError("ground truth must be gt_boxes (B, N, 4), gt_classes (B, N), gt_counts (B,)")
    N = int(gc.shape[1])
    if records.dtype != torch.uint8 or records.numel() < (slot_offset + B * M) * map_record_bytes():
        raise ValueError("records is not a uint8 tensor large enough for this update")
    p = lambda x: ctypes.c_void_p(x.data_ptr()) if x.numel() else None
    idx = dev.index or 0
    rc = lib.mgd_map_update(ctypes.byref(cfg), p(db), p(ds), p(dc), p(dn), B, M, p(gb), p(gc), p(gn), N,
                            int(slot_offset), p(records), p(gt_hist), idx,
                            ctypes.c_void_p(_torch_stream(idx)), _lib.FLAG_SYNC if sync else 0)
    _lib.raise_for_status(rc)


def recall_limits(max_dets):
    """Check average-recall detection limits (pycocotools' ``maxDets``) the way
    ``mgd_map_recall_update`` would, before any device work: 1 to 8 int32 values >= 1, strictly
    increasing.  Returns them as a tuple of ints."""
    try:
        lim = list(max_dets)
    except TypeError:
        raise ValueError(f"recall_max_dets must be a sequence of integers, got {max_dets!r}") from None
    if not 1 <= len(lim) <= _lib.MAP_MAX_RECALL_LIMITS:
        raise ValueError(f"between 1 and {_lib.MAP_MAX_RECALL_LIMITS} recall limits supported, got {len(lim)}")
    for k in lim:
        if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, np.integer)) or not 1 <= k < 2 ** 31:
            raise ValueError(f"recall limits must be int32 values >= 1, got {k!r}")
    if any(b <= a for a, b in zip(lim, lim[1:])):
        raise ValueError(f"recall limits must be strictly increasing, got {lim}")
    return tuple(int(k) for k in lim)


def map_recall_update(cfg, records, slot_offset, batch, max_dets, limits, tp):
    """Count the true positives of the ``batch * max_dets`` records ``map_update`` wrote at
    ``slot_offset`` by their first limit bucket: adds to ``tp`` ((MAP_VIEWS, C, T, K) int64 CUDA
    tensor) (``mgd_map_recall_update``).  Enqueued on the current stream, behind that
    ``map_update``."""
    import torch
    lib = _lib.load()
    lim = recall_limits(limits)
    V, C, T, K = _lib.MAP_VIEWS, cfg.num_classes, cfg.num_thresholds, len(lim)
    if not (_is_torch(tp) and tp.is_cuda and tp.dtype == torch.int64 and tp.is_contiguous()
            and tuple(tp.shape) == (V, C, T, K)):
        raise ValueError(f"tp must be a contiguous int64 CUDA tensor of shape {(V, C, T, K)}")
    dev = tp.device
    if not (_is_torch(records) and records.device == dev and records.dtype == torch.uint8
            and records.numel() >= (slot_offset + batch * max_dets) * map_record_bytes()):
        raise ValueError(f"records is not a uint8 tensor on {dev} large enough for this update")
    arr = (ctypes.c_int * K)(*lim)
    idx = dev.index or 0
    rc = lib.mgd_map_recall_update(ctypes.byref(cfg), ctypes.c_void_p(records.data_ptr()) if records.numel() else None,
                                   int(slot_offset), int(batch), int(max_dets), arr, K, ctypes.c_void_p(tp.data_ptr()),
                                   idx, ctypes.c_void_p(_torch_stream(idx)), 0)
    _lib.raise_for_status(rc)


def map_compute(cfg, records, num_slots, gt_hist):
    """Sort the first ``num_slots`` records and compute every view's per-(class, threshold)
    AP (``mgd_map_compute``).  Returns NumPy ``det_hist`` (MAP_VIEWS, C) int64 and ``ap``
    (MAP_VIEWS, C, T) for 'coco' or ``voc`` (MAP_VIEWS, C, T, 11) for 'voc'; synchronises."""
    import torch
    lib = _lib.load()
    dev = gt_hist.device
    V, C, T = _lib.MAP_VIEWS, cfg.num_classes, cfg.num_thresholds
    det_hist = torch.empty((V, C), dtype=torch.int64, device=dev)
    coco = cfg.method == _lib.MAP_COCO
    out = torch.empty((V, C, T) if coco else (V, C, T, _lib.MAP_VOC_POINTS), dtype=torch.float64, device=dev)
    idx = dev.index or 0
    rc = lib.mgd_map_compute(ctypes.byref(cfg),
                             ctypes.c_void_p(records.data_ptr()) if records is not None and num_slots else None,
                             int(num_slots), ctypes.c_void_p(gt_hist.data_ptr()),
                             ctypes.c_void_p(out.data_ptr()) if coco else None,
                             None if coco else ctypes.c_void_p(out.data_ptr()),
                             ctypes.c_void_p(det_hist.data_ptr()), idx, ctypes.c_void_p(_torch_stream(idx)), 0)
    _lib.raise_for_status(rc)
    return {"det_hist": det_hist.cpu().numpy(), "ap" if coco else "voc": out.cpu().numpy()}


def _check_owner(owner, cfg, dev):
    import torch
    if not (_is_torch(owner) and owner.device == dev and owner.dtype == torch.int32 and owner.is_contiguous()
            and tuple(owner.shape) == (cfg.num_classes,)):
        raise ValueError(f"owner must be a contiguous int32 tensor of shape ({cfg.num_classes},) on {dev}")


def map_partition(cfg, records, num_slots, segments, global_slots, owner, world):
    """Group this rank's first ``num_slots`` records by the rank that owns their class, for the
    sharded accumulator (``mgd_map_partition``).  ``segments``: (S, 2) int64 ``(L_u, G_u +
    lo_r * M_u)`` per update with local images (a CUDA tensor or a sequence of pairs);
    ``global_slots``: slots of all ranks over all updates; ``owner``: (C,) int32 CUDA tensor of
    ranks in [0, world).  Padding slots are dropped and each record gets its global slot.
    Returns the grouped records (a uint8 CUDA tensor with room for ``num_slots`` records) and
    the records per destination rank, (world,) int64 on the device.  Enqueued on the current
    stream; nothing synchronises."""
    import torch
    lib = _lib.load()
    dev = records.device if _is_torch(records) else None
    if not (_is_torch(records) and records.is_cuda and records.dtype == torch.uint8 and records.is_contiguous()):
        raise ValueError("records must be a contiguous uint8 CUDA tensor")
    num_slots, world = int(num_slots), int(world)
    rb = map_record_bytes()
    if num_slots < 0 or records.numel() < num_slots * rb:
        raise ValueError(f"records holds {records.numel() // rb} records, num_slots is {num_slots}")
    if world < 1:
        raise ValueError(f"world must be >= 1, got {world}")
    _check_owner(owner, cfg, dev)
    if not _is_torch(segments):
        segments = torch.tensor(np.asarray(segments, dtype=np.int64).reshape(-1, 2), device=dev)
    if not (segments.device == dev and segments.dtype == torch.int64 and segments.is_contiguous()
            and segments.dim() == 2 and segments.shape[1] == 2):
        raise ValueError(f"segments must be a contiguous (S, 2) int64 tensor on {dev}")
    if num_slots > 0 and segments.shape[0] == 0:
        raise ValueError("segments is empty but there are records")
    if int(global_slots) < num_slots:
        raise ValueError(f"global_slots ({global_slots}) < num_slots ({num_slots})")
    out = torch.empty((max(num_slots, 1) * rb,), dtype=torch.uint8, device=dev)
    counts = torch.empty((world,), dtype=torch.int64, device=dev)
    idx = dev.index or 0
    p = lambda x: ctypes.c_void_p(x.data_ptr()) if x.numel() else None
    rc = lib.mgd_map_partition(ctypes.byref(cfg), p(records) if num_slots else None, num_slots, p(segments),
                               int(segments.shape[0]), int(global_slots), p(owner), world, p(out), p(counts),
                               idx, ctypes.c_void_p(_torch_stream(idx)), 0)
    _lib.raise_for_status(rc)
    return out, counts


def map_compute_merged(cfg, records, num_records, gt_hist, owner, rank):
    """``map_compute`` over the records a rank received from ``map_partition`` of every rank
    (``mgd_map_compute_merged``): ``gt_hist`` is the sum over the ranks, and only the classes
    with ``owner[c] == rank`` get their APs and detection counts, the others exact zeros.
    Returns CUDA tensors ``det_hist`` (MAP_VIEWS, C) int64 and ``ap`` (MAP_VIEWS, C, T) for
    'coco' or ``voc`` (MAP_VIEWS, C, T, 11) for 'voc'.  Enqueued on the current stream."""
    import torch
    lib = _lib.load()
    V, C, T = _lib.MAP_VIEWS, cfg.num_classes, cfg.num_thresholds
    if not (_is_torch(gt_hist) and gt_hist.is_cuda and gt_hist.dtype == torch.int64 and gt_hist.is_contiguous()
            and tuple(gt_hist.shape) == (V, C)):
        raise ValueError(f"gt_hist must be a contiguous ({V}, {C}) int64 CUDA tensor")
    dev = gt_hist.device
    num_records = int(num_records)
    if num_records < 0 or (num_records and not (
            _is_torch(records) and records.device == dev and records.dtype == torch.uint8
            and records.is_contiguous() and records.numel() >= num_records * map_record_bytes())):
        raise ValueError(f"records must be a contiguous uint8 tensor on {dev} holding {num_records} records")
    _check_owner(owner, cfg, dev)
    if int(rank) < 0:
        raise ValueError(f"rank must be >= 0, got {rank}")
    det_hist = torch.empty((V, C), dtype=torch.int64, device=dev)
    coco = cfg.method == _lib.MAP_COCO
    out = torch.empty((V, C, T) if coco else (V, C, T, _lib.MAP_VOC_POINTS), dtype=torch.float64, device=dev)
    idx = dev.index or 0
    rc = lib.mgd_map_compute_merged(ctypes.byref(cfg), ctypes.c_void_p(records.data_ptr()) if num_records else None,
                                    num_records, ctypes.c_void_p(gt_hist.data_ptr()),
                                    ctypes.c_void_p(owner.data_ptr()), int(rank),
                                    ctypes.c_void_p(out.data_ptr()) if coco else None,
                                    None if coco else ctypes.c_void_p(out.data_ptr()),
                                    ctypes.c_void_p(det_hist.data_ptr()), idx, ctypes.c_void_p(_torch_stream(idx)), 0)
    _lib.raise_for_status(rc)
    return {"det_hist": det_hist, "ap" if coco else "voc": out}


_MAP_PR_TABLES = ("best_f1", "best_index", "at_confidence")


def _map_pr_request(cfg, views, confidences, num_records, dev):
    """Check a curve request and allocate its outputs: ``(mgd_map_pr, host confidences, CUDA
    tensors)``; raises ValueError before any device work."""
    import torch
    views = sorted(set(int(v) for v in views))
    if not views or any(v not in (_lib.MAP_VIEW_CORNER, _lib.MAP_VIEW_CENTRE) for v in views):
        raise ValueError("curve views must be a non-empty subset of (MAP_VIEW_CORNER, MAP_VIEW_CENTRE)")
    if any(not (cfg.views >> v) & 1 for v in views):
        raise ValueError(f"curve views {views} are not all matched by the configuration")
    conf = np.ascontiguousarray(np.asarray([] if confidences is None else confidences, dtype=np.float64).reshape(-1))
    if len(conf) > _lib.MAP_MAX_CONFIDENCES:
        raise ValueError(f"at most {_lib.MAP_MAX_CONFIDENCES} confidences supported, got {len(conf)}")
    if not np.all(np.isfinite(conf)):
        raise ValueError("confidences must be finite")
    V, C, T, Q = len(views), cfg.num_classes, cfg.num_thresholds, len(conf)
    cap = max(int(num_records), 1)
    f64 = dict(dtype=torch.float64, device=dev)
    out = {"views": views,
           "offsets": torch.empty((C + 1,), dtype=torch.int64, device=dev),
           "scores": torch.empty((cap,), **f64),
           "precision": torch.empty((V, T, cap), **f64),
           "recall": torch.empty((V, T, cap), **f64),
           "best_f1": torch.empty((V, C, T, 4), **f64),
           "best_index": torch.empty((V, C, T), dtype=torch.int64, device=dev),
           "at_confidence": torch.empty((V, C, T, Q, 3), **f64)}
    pr = _lib.MapPr()
    pr.views = sum(1 << v for v in views)
    pr.num_confidences = Q
    pr.confidences = conf.ctypes.data if Q else None
    pr.capacity = cap
    for k in ("offsets", "scores", "precision", "recall", "best_f1", "best_index"):
        setattr(pr, k, out[k].data_ptr())
    pr.at_confidence = out["at_confidence"].data_ptr() if Q else None
    return pr, conf, out


def map_compute_pr(cfg, records, num_slots, gt_hist, views, confidences=None):
    """``map_compute`` plus the precision-recall curves and operating points of the full-set
    ``views`` (MAP_VIEW_CORNER and / or MAP_VIEW_CENTRE, matched by ``cfg``) in one call
    (``mgd_map_compute_pr``); ``confidences``: up to 32 finite scores to evaluate p / r / F1 at.
    Returns ``map_compute``'s dict (NumPy) with ``"pr"``: ``views`` (the list, in order), CUDA
    tensors ``offsets`` (C+1,), ``scores`` (cap,), ``precision`` / ``recall`` (V, T, cap) -- the
    first ``offsets[C]`` entries of a row are used -- and NumPy ``best_f1`` (V, C, T, 4),
    ``best_index`` (V, C, T), ``at_confidence`` (V, C, T, Q, 3).  Synchronises."""
    import torch
    lib = _lib.load()
    dev = gt_hist.device
    V, C, T = _lib.MAP_VIEWS, cfg.num_classes, cfg.num_thresholds
    num_slots = int(num_slots)
    if num_slots < 0:
        raise ValueError(f"num_slots must be >= 0, got {num_slots}")
    pr, conf, tensors = _map_pr_request(cfg, views, confidences, num_slots, dev)
    det_hist = torch.empty((V, C), dtype=torch.int64, device=dev)
    coco = cfg.method == _lib.MAP_COCO
    out = torch.empty((V, C, T) if coco else (V, C, T, _lib.MAP_VOC_POINTS), dtype=torch.float64, device=dev)
    idx = dev.index or 0
    rc = lib.mgd_map_compute_pr(ctypes.byref(cfg),
                                ctypes.c_void_p(records.data_ptr()) if records is not None and num_slots else None,
                                num_slots, ctypes.c_void_p(gt_hist.data_ptr()),
                                ctypes.c_void_p(out.data_ptr()) if coco else None,
                                None if coco else ctypes.c_void_p(out.data_ptr()),
                                ctypes.c_void_p(det_hist.data_ptr()), ctypes.byref(pr), idx,
                                ctypes.c_void_p(_torch_stream(idx)), 0)
    _lib.raise_for_status(rc)
    for k in _MAP_PR_TABLES:
        tensors[k] = tensors[k].cpu().numpy()
    return {"det_hist": det_hist.cpu().numpy(), "ap" if coco else "voc": out.cpu().numpy(), "pr": tensors}


def map_compute_merged_pr(cfg, records, num_records, gt_hist, owner, rank, views, confidences=None):
    """``map_compute_merged`` plus ``map_compute_pr``'s curves and operating points for the
    classes with ``owner[c] == rank`` (``mgd_map_compute_merged_pr``): the other classes have
    empty curve segments and exact zeros in ``best_f1`` / ``best_index`` / ``at_confidence``, so
    summing the tables over the ranks assembles them.  Every output is a CUDA tensor; enqueued on
    the current stream."""
    import torch
    lib = _lib.load()
    V, C, T = _lib.MAP_VIEWS, cfg.num_classes, cfg.num_thresholds
    if not (_is_torch(gt_hist) and gt_hist.is_cuda and gt_hist.dtype == torch.int64 and gt_hist.is_contiguous()
            and tuple(gt_hist.shape) == (V, C)):
        raise ValueError(f"gt_hist must be a contiguous ({V}, {C}) int64 CUDA tensor")
    dev = gt_hist.device
    num_records = int(num_records)
    if num_records < 0 or (num_records and not (
            _is_torch(records) and records.device == dev and records.dtype == torch.uint8
            and records.is_contiguous() and records.numel() >= num_records * map_record_bytes())):
        raise ValueError(f"records must be a contiguous uint8 tensor on {dev} holding {num_records} records")
    _check_owner(owner, cfg, dev)
    if int(rank) < 0:
        raise ValueError(f"rank must be >= 0, got {rank}")
    pr, conf, tensors = _map_pr_request(cfg, views, confidences, num_records, dev)
    det_hist = torch.empty((V, C), dtype=torch.int64, device=dev)
    coco = cfg.method == _lib.MAP_COCO
    out = torch.empty((V, C, T) if coco else (V, C, T, _lib.MAP_VOC_POINTS), dtype=torch.float64, device=dev)
    idx = dev.index or 0
    rc = lib.mgd_map_compute_merged_pr(ctypes.byref(cfg),
                                       ctypes.c_void_p(records.data_ptr()) if num_records else None,
                                       num_records, ctypes.c_void_p(gt_hist.data_ptr()),
                                       ctypes.c_void_p(owner.data_ptr()), int(rank),
                                       ctypes.c_void_p(out.data_ptr()) if coco else None,
                                       None if coco else ctypes.c_void_p(out.data_ptr()),
                                       ctypes.c_void_p(det_hist.data_ptr()), ctypes.byref(pr), idx,
                                       ctypes.c_void_p(_torch_stream(idx)), 0)
    _lib.raise_for_status(rc)
    return {"det_hist": det_hist, "ap" if coco else "voc": out, "pr": tensors}


def confusion_config(num_classes, iou_threshold=0.5, confidences=None, iou_mode="corner"):
    """Check the settings of a confusion matrix the way ``mgd_confusion_update`` would, before any
    device work.  Returns ``(num_classes, iou_threshold, confidences (Q,) float64, iou_mode code)``;
    ``confidences=None`` is one matrix over every detection (the most negative float64, which
    every finite score passes)."""
    if isinstance(num_classes, bool) or int(num_classes) != num_classes or int(num_classes) < 1:
        raise ValueError(f"num_classes must be an integer >= 1, got {num_classes}")
    thr = float(iou_threshold)
    if not 0.0 < thr <= 1.0:
        raise ValueError(f"iou_threshold must be in (0, 1], got {iou_threshold}")
    if iou_mode not in _IOU_MODES:
        raise ValueError(f"iou_mode must be 'corner' or 'centre', got {iou_mode!r}")
    conf = np.asarray([np.finfo(np.float64).min] if confidences is None else confidences, dtype=np.float64)
    conf = np.ascontiguousarray(conf.reshape(-1))
    if not 1 <= len(conf) <= _lib.MAP_MAX_CONFIDENCES:
        raise ValueError(f"between 1 and {_lib.MAP_MAX_CONFIDENCES} confidences supported, got {len(conf)}")
    if not np.all(np.isfinite(conf)):
        raise ValueError("confidences must be finite")
    return int(num_classes), thr, conf, _IOU_MODES[iou_mode]


def confusion_update(matrix, confidences, iou_threshold, iou_mode, det_boxes, det_scores, det_classes, det_counts,
                     gt_boxes, gt_classes, gt_counts, sync=False):
    """Add one batch's detection confusion matrices to ``matrix`` ((Q, C+1, C+1) int64 CUDA tensor;
    rows: true class, columns: detected class, index C: background) at each of the Q
    ``confidences``, one IoU threshold and ``iou_mode`` 'corner' / 'centre'
    (``mgd_confusion_update``).  Torch CUDA tensors in ``match_detections``' layout; boxes may be
    int32 (``decode_nms``' ``boxes_xyxy``).  Enqueued on the current stream; class-range errors
    surface at the next ``poll_status`` unless ``sync``."""
    import torch
    lib = _lib.load()
    if not (_is_torch(matrix) and matrix.dim() == 3 and matrix.shape[1] == matrix.shape[2] and matrix.shape[1] >= 2):
        raise ValueError("matrix must be a (Q, C+1, C+1) tensor")
    C, thr, conf, mode = confusion_config(int(matrix.shape[1]) - 1, iou_threshold, confidences, iou_mode)
    if matrix.shape[0] != len(conf):
        raise ValueError(f"matrix holds {matrix.shape[0]} confidences, {len(conf)} given")
    tensors = (("det_boxes", det_boxes), ("det_scores", det_scores), ("det_classes", det_classes),
               ("det_counts", det_counts), ("gt_boxes", gt_boxes), ("gt_classes", gt_classes), ("gt_counts", gt_counts))
    for name, t in tensors:
        if not _is_torch(t):
            raise ValueError(f"{name} must be a torch tensor")
    db, ds, dc, dn, gb, gc, gn = (t for _, t in tensors)
    if ds.dim() != 2 or tuple(db.shape) != (*ds.shape, 4) or dc.shape != ds.shape or tuple(dn.shape) != (ds.shape[0],):
        raise ValueError("detections must be det_boxes (B, M, 4), det_scores / det_classes (B, M), det_counts (B,)")
    B, M = int(ds.shape[0]), int(ds.shape[1])
    if gc.dim() != 2 or gc.shape[0] != B or tuple(gb.shape) != (*gc.shape, 4) or tuple(gn.shape) != (B,):
        raise ValueError("ground truth must be gt_boxes (B, N, 4), gt_classes (B, N), gt_counts (B,)")
    N = int(gc.shape[1])
    if not (matrix.is_cuda and matrix.dtype == torch.int64 and matrix.is_contiguous()):
        raise ValueError("matrix must be a contiguous int64 CUDA tensor")
    dev = matrix.device
    for name, t in tensors:
        if t.device != dev:
            raise ValueError(f"{name} must be a torch tensor on {dev}")
    f64 = lambda x: x.to(torch.float64).contiguous()
    i32 = lambda x: x.to(torch.int32).contiguous()
    db, ds, dc, dn, gb, gc, gn = f64(db), f64(ds), i32(dc), i32(dn), f64(gb), i32(gc), i32(gn)
    p = lambda x: ctypes.c_void_p(x.data_ptr()) if x.numel() else None
    idx = dev.index or 0
    rc = lib.mgd_confusion_update(p(db), p(ds), p(dc), p(dn), B, M, p(gb), p(gc), p(gn), N, C, thr, mode,
                                  conf.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), len(conf),
                                  ctypes.c_void_p(matrix.data_ptr()), idx, ctypes.c_void_p(_torch_stream(idx)),
                                  _lib.FLAG_SYNC if sync else 0)
    _lib.raise_for_status(rc)


def tide_config(num_classes, pos_threshold=0.5, background_threshold=0.1, iou_mode="corner"):
    """Check the settings of an error analysis the way ``mgd_tide_update`` would, before any device
    work.  Returns ``(num_classes, pos_threshold, background_threshold, iou_mode code)``."""
    if isinstance(num_classes, bool) or int(num_classes) != num_classes or int(num_classes) < 1:
        raise ValueError(f"num_classes must be an integer >= 1, got {num_classes}")
    if int(num_classes) * _lib.TIDE_SETS > 2 ** 31 - 1:
        raise ValueError(f"num_classes must be below 2^31 / {_lib.TIDE_SETS}, got {num_classes}")
    t_f, t_b = float(pos_threshold), float(background_threshold)
    if not 0.0 < t_f <= 1.0:
        raise ValueError(f"pos_threshold must be in (0, 1], got {pos_threshold}")
    if not 0.0 < t_b <= t_f:
        raise ValueError(f"background_threshold must be in (0, pos_threshold], got {background_threshold}")
    if iou_mode not in _IOU_MODES:
        raise ValueError(f"iou_mode must be 'corner' or 'centre', got {iou_mode!r}")
    return int(num_classes), t_f, t_b, _IOU_MODES[iou_mode]


def tide_update(records, slot_offset, gt_hist, counts, pos_threshold, background_threshold, iou_mode,
                det_boxes, det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts, sync=False):
    """Type one batch's errors and write the records of every error-fixed set (``mgd_tide_update``):
    ``TIDE_SETS * B * M`` records at ``slot_offset`` of ``records`` (a CUDA byte tensor), image by
    image, one block of M per set; the sets' ground-truth counts are added to the MAP_VIEW_CORNER row
    of ``gt_hist`` ((MAP_VIEWS, TIDE_SETS * C) int64) and the error counts to ``counts`` ((C,
    TIDE_ERRORS) int64).  Torch CUDA tensors in ``match_detections``' layout; boxes may be int32
    (``decode_nms``' ``boxes_xyxy``).  Enqueued on the current stream; class-range errors surface at
    the next ``poll_status`` unless ``sync``."""
    import torch
    lib = _lib.load()
    if not (_is_torch(counts) and counts.dim() == 2 and counts.shape[1] == _lib.TIDE_ERRORS):
        raise ValueError(f"counts must be a (C, {_lib.TIDE_ERRORS}) tensor")
    C, t_f, t_b, mode = tide_config(int(counts.shape[0]), pos_threshold, background_threshold, iou_mode)
    tensors = (("det_boxes", det_boxes), ("det_scores", det_scores), ("det_classes", det_classes),
               ("det_counts", det_counts), ("gt_boxes", gt_boxes), ("gt_classes", gt_classes), ("gt_counts", gt_counts))
    for name, t in tensors:
        if not _is_torch(t):
            raise ValueError(f"{name} must be a torch tensor")
    db, ds, dc, dn, gb, gc, gn = (t for _, t in tensors)
    if ds.dim() != 2 or tuple(db.shape) != (*ds.shape, 4) or dc.shape != ds.shape or tuple(dn.shape) != (ds.shape[0],):
        raise ValueError("detections must be det_boxes (B, M, 4), det_scores / det_classes (B, M), det_counts (B,)")
    B, M = int(ds.shape[0]), int(ds.shape[1])
    if gc.dim() != 2 or gc.shape[0] != B or tuple(gb.shape) != (*gc.shape, 4) or tuple(gn.shape) != (B,):
        raise ValueError("ground truth must be gt_boxes (B, N, 4), gt_classes (B, N), gt_counts (B,)")
    N = int(gc.shape[1])
    if not (counts.is_cuda and counts.dtype == torch.int64 and counts.is_contiguous()):
        raise ValueError("counts must be a contiguous int64 CUDA tensor")
    dev = counts.device
    if not (_is_torch(gt_hist) and gt_hist.device == dev and gt_hist.dtype == torch.int64 and gt_hist.is_contiguous()
            and tuple(gt_hist.shape) == (_lib.MAP_VIEWS, _lib.TIDE_SETS * C)):
        raise ValueError(f"gt_hist must be a contiguous ({_lib.MAP_VIEWS}, {_lib.TIDE_SETS * C}) int64 tensor on {dev}")
    slot_offset = int(slot_offset)
    if not (_is_torch(records) and records.device == dev and records.dtype == torch.uint8 and slot_offset >= 0
            and records.numel() >= (slot_offset + _lib.TIDE_SETS * B * M) * map_record_bytes()):
        raise ValueError(f"records is not a uint8 tensor on {dev} large enough for this update")
    for name, t in tensors:
        if t.device != dev:
            raise ValueError(f"{name} must be a torch tensor on {dev}")
    f64 = lambda x: x.to(torch.float64).contiguous()
    i32 = lambda x: x.to(torch.int32).contiguous()
    db, ds, dc, dn, gb, gc, gn = f64(db), f64(ds), i32(dc), i32(dn), f64(gb), i32(gc), i32(gn)
    p = lambda x: ctypes.c_void_p(x.data_ptr()) if x.numel() else None
    idx = dev.index or 0
    rc = lib.mgd_tide_update(p(db), p(ds), p(dc), p(dn), B, M, p(gb), p(gc), p(gn), N, C, t_f, t_b, mode,
                             slot_offset, p(records), p(gt_hist), p(counts), idx, ctypes.c_void_p(_torch_stream(idx)),
                             _lib.FLAG_SYNC if sync else 0)
    _lib.raise_for_status(rc)


def iou_matrix(boxes1, boxes2):
    """(n, m) float64 IoU matrix of xyxy boxes (``mgd_iou_matrix``), NumPy in / out."""
    lib = _lib.load()
    b1 = np.ascontiguousarray(np.asarray(boxes1, dtype=np.float64).reshape(-1, 4))
    b2 = np.ascontiguousarray(np.asarray(boxes2, dtype=np.float64).reshape(-1, 4))
    out = np.zeros((b1.shape[0], b2.shape[0]), dtype=np.float64)
    if out.size:
        rc = lib.mgd_iou_matrix(ctypes.c_void_p(b1.ctypes.data), b1.shape[0],
                                ctypes.c_void_p(b2.ctypes.data), b2.shape[0],
                                ctypes.c_void_p(out.ctypes.data), _lib.MEM_HOST, _current_device(),
                                None, _lib.FLAG_SYNC)
        _lib.raise_for_status(rc)
    return out


# ------------------------------------------------------------------------------
# box-side pre-step of the encoder (reference multigriddet/data/augmentation.py)
# ------------------------------------------------------------------------------

def reshape_boxes_batch(boxes, params, counts=None, want_f32=True, sync=True):
    """``reshape_boxes`` over a batch (``mgd_reshape_boxes``).

    boxes (B, N, 5) int32 or float64, NumPy or torch CUDA; params (B, 10) int32
    ``[src_w, src_h, target_w, target_h, padding_w, padding_h, dx, dy, hflip, vflip]``;
    counts (B,) valid rows or None.  Returns ``(out, out_f32 or None, out_counts)`` in the same
    memory space; ``out_f32`` is what ``encode_targets`` takes.
    """
    lib = _lib.load()
    if _is_torch(boxes):
        import torch
        dev = boxes.device
        i32 = boxes.dtype == torch.int32
        b = boxes.contiguous() if i32 else boxes.to(torch.float64).contiguous()
        B, N = int(b.shape[0]), int(b.shape[1])
        par = torch.as_tensor(params).to(device=dev, dtype=torch.int32).contiguous()
        cnt = None if counts is None else torch.as_tensor(counts).to(device=dev, dtype=torch.int32).contiguous()
        out = torch.empty_like(b)
        o32 = torch.empty((B, N, 5), dtype=torch.float32, device=dev) if want_f32 else None
        ocn = torch.empty((B,), dtype=torch.int32, device=dev)
        p = lambda x: ctypes.c_void_p(x.data_ptr()) if x is not None and x.numel() else None
        idx = dev.index or 0
        rc = lib.mgd_reshape_boxes(p(b), _lib.BOXES_I32 if i32 else _lib.BOXES_F64, p(cnt), p(par), B, N,
                                   p(out), p(o32), p(ocn), _lib.MEM_DEVICE, idx,
                                   ctypes.c_void_p(_torch_stream(idx)), _lib.FLAG_SYNC if sync else 0)
    else:
        b = np.asarray(boxes)
        i32 = b.dtype == np.int32
        b = np.ascontiguousarray(b, dtype=np.int32 if i32 else np.float64)
        B, N = b.shape[0], b.shape[1]
        par = np.ascontiguousarray(np.asarray(params), dtype=np.int32).reshape(B, 10)
        cnt = None if counts is None else np.ascontiguousarray(np.asarray(counts), dtype=np.int32)
        out = np.zeros_like(b)
        o32 = np.zeros((B, N, 5), dtype=np.float32) if want_f32 else None
        ocn = np.zeros((B,), dtype=np.int32)
        p = lambda x: ctypes.c_void_p(x.ctypes.data) if x is not None and x.size else None
        rc = lib.mgd_reshape_boxes(p(b), _lib.BOXES_I32 if i32 else _lib.BOXES_F64, p(cnt), p(par), B, N,
                                   p(out), p(o32), p(ocn), _lib.MEM_HOST, _current_device(), None,
                                   _lib.FLAG_SYNC)
    _lib.raise_for_status(rc)
    return out, o32, ocn


def letterbox_boxes_batch(boxes, src_shapes, input_shape, max_boxes_per_image, counts=None,
                          expansion=1, multiscale_shapes=None, hflip=None, sync=True):
    """The tf.data box pre-step of the reference's default training path
    (``mgd_letterbox_boxes``; generators.py:1859-1916 letterbox / multi-scale transform,
    :227-256 flip, :1963-1976 padded_batch, :1983-2034 ``_expand_box_capacity``).

    boxes (B, N, 5) float32 NumPy or torch CUDA, original-image pixels; src_shapes (B, 2)
    (h, w); multiscale_shapes (B, 2) or None; hflip (B,) bool or None.  Returns the
    (B, max_boxes_per_image * expansion, 5) float32 tensor ``encode_targets`` consumes."""
    lib = _lib.load()
    B, N = int(boxes.shape[0]), int(boxes.shape[1])
    par = np.zeros((B, 6), dtype=np.int32)
    par[:, 0:2] = np.asarray(src_shapes, dtype=np.int64).reshape(B, 2)
    if multiscale_shapes is not None:
        par[:, 2:4] = np.asarray(multiscale_shapes, dtype=np.int64).reshape(B, 2)
    if hflip is not None:
        par[:, 4] = np.asarray(hflip).astype(np.int32).reshape(B)
    cap = int(max_boxes_per_image) * int(expansion)
    ih, iw = int(input_shape[0]), int(input_shape[1])
    if _is_torch(boxes):
        import torch
        dev = boxes.device
        b = boxes.to(torch.float32).contiguous()
        d_par = torch.from_numpy(par).to(dev)
        cnt = None if counts is None else torch.as_tensor(counts).to(device=dev, dtype=torch.int32).contiguous()
        out = torch.empty((B, cap, 5), dtype=torch.float32, device=dev)
        p = lambda x: ctypes.c_void_p(x.data_ptr()) if x is not None and x.numel() else None
        idx = dev.index or 0
        rc = lib.mgd_letterbox_boxes(p(b), p(cnt), p(d_par), B, N, ih, iw, int(max_boxes_per_image),
                                     int(expansion), p(out), _lib.MEM_DEVICE, idx,
                                     ctypes.c_void_p(_torch_stream(idx)), _lib.FLAG_SYNC if sync else 0)
    else:
        b = np.ascontiguousarray(np.asarray(boxes), dtype=np.float32)
        cnt = None if counts is None else np.ascontiguousarray(np.asarray(counts), dtype=np.int32)
        out = np.zeros((B, cap, 5), dtype=np.float32)
        p = lambda x: ctypes.c_void_p(x.ctypes.data) if x is not None and x.size else None
        rc = lib.mgd_letterbox_boxes(p(b), p(cnt), p(par), B, N, ih, iw, int(max_boxes_per_image),
                                     int(expansion), p(out), _lib.MEM_HOST, _current_device(), None,
                                     _lib.FLAG_SYNC)
    _lib.raise_for_status(rc)
    return out


def mosaic_merge_boxes_batch(boxes, sample_index, crop_xy, image_size, want_f32=True, sync=True):
    """``merge_mosaic_bboxes`` for a batch of mosaics (``mgd_mosaic_merge_boxes``).

    boxes (n_src, N, 5) float64 (zero rows = padding); sample_index (B, 4) source image of
    each quadrant (top-left, bottom-left, bottom-right, top-right); crop_xy (B, 2);
    image_size (height, width).  Returns ``(out (B, N, 5) f64, out_f32 or None, counts)``.
    """
    lib = _lib.load()
    H, W = int(image_size[0]), int(image_size[1])
    if _is_torch(boxes):
        import torch
        dev = boxes.device
        b = boxes.to(torch.float64).contiguous()
        n_src, N = int(b.shape[0]), int(b.shape[1])
        par = torch.cat([torch.as_tensor(sample_index).reshape(-1, 4).to(dev),
                         torch.as_tensor(crop_xy).reshape(-1, 2).to(dev)], 1).to(torch.int32).contiguous()
        B = int(par.shape[0])
        out = torch.empty((B, N, 5), dtype=torch.float64, device=dev)
        o32 = torch.empty((B, N, 5), dtype=torch.float32, device=dev) if want_f32 else None
        ocn = torch.empty((B,), dtype=torch.int32, device=dev)
        p = lambda x: ctypes.c_void_p(x.data_ptr()) if x is not None and x.numel() else None
        idx = dev.index or 0
        rc = lib.mgd_mosaic_merge_boxes(p(b), n_src, N, p(par), B, H, W, p(out), p(o32), p(ocn),
                                        _lib.MEM_DEVICE, idx, ctypes.c_void_p(_torch_stream(idx)),
                                        _lib.FLAG_SYNC if sync else 0)
    else:
        b = np.ascontiguousarray(np.asarray(boxes), dtype=np.float64)
        n_src, N = b.shape[0], b.shape[1]
        par = np.ascontiguousarray(np.concatenate([np.asarray(sample_index).reshape(-1, 4),
                                                   np.asarray(crop_xy).reshape(-1, 2)], 1), dtype=np.int32)
        B = par.shape[0]
        out = np.zeros((B, N, 5), dtype=np.float64)
        o32 = np.zeros((B, N, 5), dtype=np.float32) if want_f32 else None
        ocn = np.zeros((B,), dtype=np.int32)
        p = lambda x: ctypes.c_void_p(x.ctypes.data) if x is not None and x.size else None
        rc = lib.mgd_mosaic_merge_boxes(p(b), n_src, N, p(par), B, H, W, p(out), p(o32), p(ocn),
                                        _lib.MEM_HOST, _current_device(), None, _lib.FLAG_SYNC)
    _lib.raise_for_status(rc)
    return out, o32, ocn


# ------------------------------------------------------------------------------
# loss-side ignore mask (reference multigriddet/losses/multigrid_loss.py:494-703)
# ------------------------------------------------------------------------------

def ignore_masks(y_preds, y_trues, anchors, input_shape, num_classes, ignore_thresh=0.5, eps=1e-7,
                 sync=True):
    """Per layer ``(ignore_mask, assigned_anchor_iou, max_iou_map)``, each (B, G, G, 1) float32
    (``mgd_ignore_mask``).  Lists of NumPy arrays (host) or torch CUDA tensors (device)."""
    lib = _lib.load()
    L = len(y_preds)
    grids = [(int(p.shape[1]), int(p.shape[2])) for p in y_preds]
    cfg = _lib.make_head_config([np.asarray(a, dtype=np.float32) for a in anchors], num_classes,
                                input_shape, grids)
    B = int(y_preds[0].shape[0])
    outs = []
    if _is_torch(y_preds[0]):
        import torch
        dev = y_preds[0].device
        yp = [t.to(torch.float32).contiguous() for t in y_preds]
        yt = [t.to(device=dev, dtype=torch.float32).contiguous() for t in y_trues]
        for gh, gw in grids:
            outs.append(tuple(torch.empty((B, gh, gw, 1), dtype=torch.float32, device=dev) for _ in range(3)))
        ptr = lambda ts: _lib.ptr_array([t.data_ptr() for t in ts])
        idx = dev.index or 0
        rc = lib.mgd_ignore_mask(ctypes.byref(cfg), ptr(yp), ptr(yt), B, float(ignore_thresh), float(eps),
                                 ptr([o[0] for o in outs]), ptr([o[1] for o in outs]), ptr([o[2] for o in outs]),
                                 _lib.MEM_DEVICE, idx, ctypes.c_void_p(_torch_stream(idx)),
                                 _lib.FLAG_SYNC if sync else 0)
    else:
        yp = [np.ascontiguousarray(np.asarray(t), dtype=np.float32) for t in y_preds]
        yt = [np.ascontiguousarray(np.asarray(t), dtype=np.float32) for t in y_trues]
        for gh, gw in grids:
            outs.append(tuple(np.zeros((B, gh, gw, 1), dtype=np.float32) for _ in range(3)))
        ptr = lambda ts: _lib.ptr_array([t.ctypes.data for t in ts])
        rc = lib.mgd_ignore_mask(ctypes.byref(cfg), ptr(yp), ptr(yt), B, float(ignore_thresh), float(eps),
                                 ptr([o[0] for o in outs]), ptr([o[1] for o in outs]), ptr([o[2] for o in outs]),
                                 _lib.MEM_HOST, _current_device(), None, _lib.FLAG_SYNC)
    _lib.raise_for_status(rc)
    return outs


def encode_ignore_masks(true_boxes, y_preds, anchors, input_shape, num_classes, ignore_thresh=0.5,
                        eps=1e-7, want_y_true=True, sync=True, semantics="numpy"):
    """Target encoding and loss-side ignore mask in one call on torch CUDA tensors
    (``mgd_encode_ignore_mask``): the mask kernels read the encoder's owner table instead of a
    dense ``y_true``.  Returns ``(y_true list or None, [(ignore, assigned_iou, max_iou)] per layer)``;
    identical to ``encode_targets`` followed by ``ignore_masks``."""
    import torch
    lib = _lib.load()
    grids = [(int(p.shape[1]), int(p.shape[2])) for p in y_preds]
    cfg = _lib.make_head_config([np.asarray(a, dtype=np.float32) for a in anchors], num_classes,
                                input_shape, grids)
    dev = y_preds[0].device
    B, N = int(true_boxes.shape[0]), int(true_boxes.shape[1])
    tb = true_boxes.to(device=dev, dtype=torch.float32).contiguous()
    yp = [t.to(torch.float32).contiguous() for t in y_preds]
    yt = [torch.empty_like(t) for t in yp] if want_y_true else None
    outs = [tuple(torch.empty((B, gh, gw, 1), dtype=torch.float32, device=dev) for _ in range(3))
            for gh, gw in grids]
    ptr = lambda ts: _lib.ptr_array([t.data_ptr() for t in ts])
    idx = dev.index or 0
    flags = (_lib.FLAG_SYNC if sync else 0) | (_lib.FLAG_TF_COMPAT if semantics == "tf_compat" else 0)
    rc = lib.mgd_encode_ignore_mask(ctypes.byref(cfg), ctypes.c_void_p(tb.data_ptr()), B, N, ptr(yp),
                                    ptr(yt) if yt is not None else None, float(ignore_thresh), float(eps),
                                    ptr([o[0] for o in outs]), ptr([o[1] for o in outs]),
                                    ptr([o[2] for o in outs]), idx, ctypes.c_void_p(_torch_stream(idx)), flags)
    _lib.raise_for_status(rc)
    return yt, outs
