"""Drop-in for ``multigriddet/evaluation/metrics.py`` of the reference: same function
names, arguments, return containers and conventions; the IoU and the greedy
detection-to-ground-truth matching (the O(P x G) part, a Python double loop in the
reference) run in ``libmgd.so`` (``mgd_match_detections``, ``mgd_iou_matrix``).  The
precision / recall / AP arithmetic on the resulting flag vectors is a few NumPy
reductions per class, exactly as in the reference.

Tie rule (the reference's ``np.argsort(scores)[::-1]``, metrics.py:93, is unstable):
equal scores are ordered like a reversed stable argsort, i.e. later prediction first.
"""
from __future__ import annotations

from typing import Any, Dict, List, Tuple

import numpy as np

from .. import _lib, engine

COCO_THRESHOLDS = [0.5, 0.55, 0.6, 0.65, 0.7, 0.75, 0.8, 0.85, 0.9, 0.95]


def calculate_iou_matrix(boxes1: np.ndarray, boxes2: np.ndarray) -> np.ndarray:
    """(N, M) IoU of xyxy boxes -- metrics.py:28-70."""
    boxes1, boxes2 = np.asarray(boxes1), np.asarray(boxes2)
    if len(boxes1) == 0 or len(boxes2) == 0:
        return np.zeros((len(boxes1), len(boxes2)))
    if boxes1.shape[1] != 4 or boxes2.shape[1] != 4:
        raise ValueError("Boxes must have 4 coordinates")
    return engine.iou_matrix(boxes1, boxes2)


class _Packed:
    """Lists of dicts -> the padded per-image tensors the library takes."""

    def __init__(self, predictions: List[Dict], ground_truths: List[Dict]):
        ids = {}
        for rec in list(predictions) + list(ground_truths):
            ids.setdefault(rec["image_id"], len(ids))
        B = max(len(ids), 1)
        p_img = np.array([ids[p["image_id"]] for p in predictions], dtype=np.int64)
        g_img = np.array([ids[g["image_id"]] for g in ground_truths], dtype=np.int64)
        self.det_counts = np.bincount(p_img, minlength=B).astype(np.int32)
        self.gt_counts = np.bincount(g_img, minlength=B).astype(np.int32)
        M = max(int(self.det_counts.max(initial=0)), 1)
        N = max(int(self.gt_counts.max(initial=0)), 1)

        def slots(img, counts):
            order = np.argsort(img, kind="stable")
            start = np.concatenate([[0], np.cumsum(counts)[:-1]])
            slot = np.empty(len(img), dtype=np.int64)
            slot[order] = np.arange(len(img)) - np.repeat(start, counts)
            return slot
        self.p_img, self.p_slot = p_img, slots(p_img, self.det_counts)
        g_slot = slots(g_img, self.gt_counts)
        self.det_boxes = np.zeros((B, M, 4)); self.det_scores = np.zeros((B, M))
        self.det_classes = np.full((B, M), -1, dtype=np.int32)
        self.gt_boxes = np.zeros((B, N, 4)); self.gt_classes = np.full((B, N), -2, dtype=np.int32)
        if len(predictions):
            self.det_boxes[p_img, self.p_slot] = np.array([p["bbox"] for p in predictions], dtype=np.float64)
            self.det_scores[p_img, self.p_slot] = np.array([p["score"] for p in predictions], dtype=np.float64)
            self.det_classes[p_img, self.p_slot] = np.array([p["class"] for p in predictions])
        if len(ground_truths):
            self.gt_boxes[g_img, g_slot] = np.array([g["bbox"] for g in ground_truths], dtype=np.float64)
            self.gt_classes[g_img, g_slot] = np.array([g["class"] for g in ground_truths])
        self.pred_scores = np.array([p["score"] for p in predictions], dtype=np.float64)
        self.pred_classes = np.array([p["class"] for p in predictions], dtype=np.int64)
        self.gt_class_flat = np.array([g["class"] for g in ground_truths], dtype=np.int64)

    def flags(self, thresholds, mode) -> np.ndarray:
        """(T, P) uint8 TP flags in the order of the ``predictions`` list."""
        tp = engine.match_detections(self.det_boxes, self.det_scores, self.det_classes, self.det_counts,
                                     self.gt_boxes, self.gt_classes, self.gt_counts, thresholds,
                                     iou_mode=mode)
        return tp[:, self.p_img, self.p_slot] if len(self.p_img) else np.zeros((len(thresholds), 0), np.uint8)


def _sorted_flags(tp: np.ndarray, scores: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    order = np.argsort(scores, kind="stable")[::-1]
    flags = tp[order].astype(bool)
    return flags, ~flags, scores[order]


def match_predictions_to_gt(predictions: List[Dict], ground_truths: List[Dict],
                            iou_threshold: float = 0.5) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(tp_flags, fp_flags, scores) in descending-score order -- metrics.py:73-144 (the
    un-cached matcher: ``BoxUtils.box_iou`` reads the boxes as centre format).  Like the
    reference it matches on 'class' and 'image_id' of whatever lists it is given."""
    if len(predictions) == 0:
        return np.array([]), np.array([]), np.array([])
    pk = _Packed(predictions, ground_truths)
    return _sorted_flags(pk.flags([iou_threshold], "centre")[0], pk.pred_scores)


def match_predictions_to_gt_cached(predictions: List[Dict], ground_truths: List[Dict],
                                   iou_threshold: float, iou_cache=None):
    """metrics.py:147-218.  ``iou_cache`` is accepted for signature compatibility and not
    read: the corner-format IoUs it holds are recomputed on the device."""
    if len(predictions) == 0:
        return np.array([]), np.array([]), np.array([])
    pk = _Packed(predictions, ground_truths)
    return _sorted_flags(pk.flags([iou_threshold], "corner")[0], pk.pred_scores)


def compute_iou_cache_for_class(predictions: List[Dict], ground_truths: List[Dict], class_id: int):
    """metrics.py:456-514: ``{(pred_idx, gt_idx): iou}`` for same-image pairs of one class
    (indices into the class-filtered lists)."""
    cp = [p for p in predictions if p["class"] == class_id]
    cg = [g for g in ground_truths if g["class"] == class_id]
    if not cp or not cg:
        return {}
    cache = {}
    by_img_p, by_img_g = {}, {}
    for i, p in enumerate(cp):
        by_img_p.setdefault(p["image_id"], []).append(i)
    for j, g in enumerate(cg):
        by_img_g.setdefault(g["image_id"], []).append(j)
    for img, pi in by_img_p.items():
        gi = by_img_g.get(img)
        if not gi:
            continue
        mat = calculate_iou_matrix(np.array([cp[i]["bbox"] for i in pi]), np.array([cg[j]["bbox"] for j in gi]))
        for a, i in enumerate(pi):
            for b, j in enumerate(gi):
                cache[(i, j)] = float(mat[a, b])
    return cache


def compute_precision_recall(tp_flags: np.ndarray, fp_flags: np.ndarray, num_gt: int):
    """metrics.py:221-246."""
    if len(tp_flags) == 0:
        return np.array([0.0]), np.array([0.0])
    cum_tp, cum_fp = np.cumsum(tp_flags), np.cumsum(fp_flags)
    return cum_tp / (cum_tp + cum_fp + 1e-8), cum_tp / (num_gt + 1e-8)


def compute_average_precision(precisions: np.ndarray, recalls: np.ndarray, method: str = "coco") -> float:
    """metrics.py:249-300 ('coco': all-point interpolation + trapezoid; 'voc': 11 points)."""
    if len(precisions) == 0 or len(recalls) == 0:
        return 0.0
    if method == "voc":
        vals = []
        for r in np.arange(0, 1.1, 0.1):
            sel = precisions[recalls >= r]
            vals.append(np.max(sel) if len(sel) > 0 else 0.0)
        return np.mean(vals)
    if method == "coco":
        idx = np.argsort(recalls)
        r, p = recalls[idx], precisions[idx]
        interp = np.maximum.accumulate(p[::-1])[::-1]
        if len(r) > 1:
            return float(np.sum((r[1:] - r[:-1]) * (interp[1:] + interp[:-1]) / 2.0))
        return interp[0] * r[0]
    raise ValueError(f"Unknown method: {method}")


def _special_ap(n_pred: int, n_gt: int):
    """The AP of a class without predictions or without ground truth (metrics.py:303-385);
    None when the class has both."""
    if n_pred == 0:
        return 0.0 if n_gt > 0 else 1.0
    if n_gt == 0:
        return 0.0
    return None


def _class_ap(tp_row, pk: _Packed, class_id: int, method: str) -> float:
    sel = pk.pred_classes == class_id
    n_gt = int(np.sum(pk.gt_class_flat == class_id))
    special = _special_ap(int(np.count_nonzero(sel)), n_gt)
    if special is not None:
        return special
    tp, fp, _ = _sorted_flags(tp_row[sel], pk.pred_scores[sel])
    return compute_average_precision(*compute_precision_recall(tp, fp, n_gt), method)


def calculate_ap_for_class(predictions, ground_truths, class_id: int, iou_threshold: float = 0.5,
                           method: str = "coco") -> float:
    """metrics.py:303-341 (un-cached matcher)."""
    pk = _Packed(predictions, ground_truths)
    return _class_ap(pk.flags([iou_threshold], "centre")[0], pk, class_id, method)


def calculate_ap_for_class_cached(predictions, ground_truths, class_id: int, iou_threshold: float,
                                  iou_cache=None, method: str = "coco") -> float:
    """metrics.py:344-385 (cached matcher; ``iou_cache`` not read)."""
    pk = _Packed(predictions, ground_truths)
    return _class_ap(pk.flags([iou_threshold], "corner")[0], pk, class_id, method)


def _box_area(bbox) -> float:
    x1, y1, x2, y2 = bbox
    return (x2 - x1) * (y2 - y1)


def _filter_by_area(predictions, ground_truths, min_area=None, max_area=None):
    keep = lambda r: ((min_area is None or _box_area(r["bbox"]) >= min_area) and
                      (max_area is None or _box_area(r["bbox"]) < max_area))
    return [p for p in predictions if keep(p)], [g for g in ground_truths if keep(g)]


_SCALES = (("APS", None, 1024.0), ("APM", 1024.0, 9216.0), ("APL", 9216.0, None))


class _DictSource:
    """What ``_map_results`` reads, from the reference's lists of dicts."""

    def __init__(self, predictions: List[Dict], ground_truths: List[Dict]):
        self.predictions, self.ground_truths = predictions, ground_truths
        self.num_predictions, self.num_ground_truths = len(predictions), len(ground_truths)

    def classes(self):
        return set(p["class"] for p in self.predictions) | set(g["class"] for g in self.ground_truths)

    def scale(self, lo, hi) -> "_DictSource":
        return _DictSource(*_filter_by_area(self.predictions, self.ground_truths, lo, hi))

    def ap_table(self, iou_thresholds, matcher: str, method: str):
        pk = _Packed(self.predictions, self.ground_truths)
        tp = pk.flags(iou_thresholds, matcher) if iou_thresholds else None
        return lambda class_id, t: _class_ap(tp[t], pk, class_id, method)


def _map_results(src, num_classes, iou_thresholds, class_names, method, use_parallel, optimize_classes,
                 cache_ious, compute_per_scale) -> Dict[str, Any]:
    """calculate_map's result dict (metrics.py:541-815) from an AP source: the class set, the
    matcher choice, the means over classes and thresholds and the per-scale rules.
    ``src.ap_table(thresholds, matcher, method)(class_id, t)`` is the AP of one class at
    threshold t; ``src.scale(lo, hi)`` is the source of the area-filtered sub-call."""
    results = {"mAP": 0.0, "mAP50": 0.0, "mAP75": 0.0, "per_class": {}, "per_iou": {},
               "num_predictions": src.num_predictions, "num_ground_truths": src.num_ground_truths}
    if optimize_classes:
        active = sorted(src.classes())
    else:
        active = list(range(num_classes))
    if use_parallel and len(active) > 1 and cache_ious and src.num_predictions > 10000:
        cache_ious = False
    ap_of = src.ap_table(iou_thresholds, "corner" if cache_ious else "centre", method)
    iou_aps = {thr: [] for thr in iou_thresholds}
    class_aps = {}
    for class_id in active:
        name = class_names[class_id] if class_id < len(class_names) else f"class_{class_id}"
        res = {}
        for t, thr in enumerate(iou_thresholds):
            ap = ap_of(class_id, t)
            res[f"AP{thr:.2f}"] = ap
            iou_aps[thr].append(ap)
        res["AP"] = np.mean(list(res.values()))
        class_aps[name] = res
    results["per_class"] = class_aps
    for thr in iou_thresholds:
        if len(iou_aps[thr]) > 0:
            results["per_iou"][f"mAP{thr:.2f}"] = np.mean(iou_aps[thr])
    if 0.5 in iou_thresholds:
        results["mAP50"] = results["per_iou"].get("mAP0.50", 0.0)
    if 0.75 in iou_thresholds:
        results["mAP75"] = results["per_iou"].get("mAP0.75", 0.0)
    if len(iou_thresholds) > 0:
        results["mAP"] = np.mean([results["per_iou"].get(f"mAP{thr:.2f}", 0.0) for thr in iou_thresholds])
    for key, lo, hi in _SCALES:
        results[key], results[key + "50"] = 0.0, 0.0
        if compute_per_scale:
            sub_src = src.scale(lo, hi)
            if sub_src.num_ground_truths > 0:
                sub = _map_results(sub_src, num_classes, iou_thresholds, class_names, method,
                                   use_parallel=False, optimize_classes=optimize_classes,
                                   cache_ious=False, compute_per_scale=False)
                results[key], results[key + "50"] = sub["mAP"], sub.get("mAP50", 0.0)
    return results


def calculate_map(predictions: List[Dict], ground_truths: List[Dict], num_classes: int,
                  iou_thresholds: List[float] = None, class_names: List[str] = None,
                  method: str = "coco", use_parallel: bool = True, optimize_classes: bool = True,
                  cache_ious: bool = True, compute_per_scale: bool = True) -> Dict[str, Any]:
    """mAP over classes and IoU thresholds -- metrics.py:541-815, same result keys.

    One ``mgd_match_detections`` launch covers every class and threshold.  Which matcher
    (and with it which IoU formula) the reference would have used is reproduced: the cached
    corner-IoU matcher by default; the un-cached centre-format one when ``cache_ious`` is
    false, when the parallel branch sees more than 10000 predictions (:604-606), and for
    the per-scale APs (:745-800).  ``use_parallel`` only takes part in that decision.
    """
    if iou_thresholds is None:
        iou_thresholds = list(COCO_THRESHOLDS)
    if class_names is None:
        class_names = [f"class_{i}" for i in range(num_classes)]
    return _map_results(_DictSource(predictions, ground_truths), num_classes, iou_thresholds, class_names,
                        method, use_parallel, optimize_classes, cache_ious, compute_per_scale)


class _DeviceSource:
    """What ``_map_results`` reads, from ``mgd_map_compute``'s per-view outputs.  ``view`` is
    the view the detections and ground truth are counted in: one of the two full-set views,
    or an area band's view (``band``), which is also the one its APs come from."""

    _BANDS = {(None, 1024.0): _lib.MAP_VIEW_S, (1024.0, 9216.0): _lib.MAP_VIEW_M, (9216.0, None): _lib.MAP_VIEW_L}

    def __init__(self, out, gt_hist, view: int, band: bool = False):
        self.out, self.gt_hist, self.view, self.band = out, gt_hist, view, band
        self._det, self._gt = out["det_hist"][view], gt_hist[view]
        self.num_predictions, self.num_ground_truths = int(self._det.sum()), int(self._gt.sum())

    def classes(self):
        return set(np.flatnonzero((self._det > 0) | (self._gt > 0)).tolist())

    def scale(self, lo, hi) -> "_DeviceSource":
        return _DeviceSource(self.out, self.gt_hist, self._BANDS[(lo, hi)], band=True)

    def ap_table(self, iou_thresholds, matcher: str, method: str):
        v = self.view if self.band else (_lib.MAP_VIEW_CORNER if matcher == "corner" else _lib.MAP_VIEW_CENTRE)
        if not self.band:
            self.matcher_view = v                         # the view of the main APs, for the curves
        det, gt = self.out["det_hist"][v], self.gt_hist[v]

        def ap_of(class_id, t):
            special = _special_ap(int(det[class_id]), int(gt[class_id]))
            if special is not None:
                return special
            if method == "voc":
                return np.mean(self.out["voc"][v, class_id, t])
            ap = self.out["ap"][v, class_id, t]
            # compute_average_precision: float(np.sum(...)), or interp[0] * r[0] for one record
            return ap if det[class_id] == 1 else float(ap)
        return ap_of


def _full_views(cfg):
    """The full-set views a configuration matches (one or both of corner and centre)."""
    return [v for v in (_lib.MAP_VIEW_CORNER, _lib.MAP_VIEW_CENTRE) if (cfg.views >> v) & 1]


def _check_pr_args(precision_recall, confidences):
    if confidences is not None and not precision_recall:
        raise ValueError("confidences are evaluated with precision_recall=True only")


def _precision_recall(pr, view, num_records, gt_hist, confidences) -> Dict[str, Any]:
    """compute()'s "precision_recall" entry: the curves and tables of ``view`` out of the
    compute's (``engine.map_compute_pr``) outputs, the curves trimmed to ``num_records`` and no
    longer sharing memory with the other view's."""
    import torch
    vi = pr["views"].index(view)
    own = lambda t: t.clone(memory_format=torch.contiguous_format)
    res = {"matcher": "corner" if view == _lib.MAP_VIEW_CORNER else "centre",
           "offsets": pr["offsets"], "scores": own(pr["scores"][:num_records]),
           "precision": own(pr["precision"][vi, :, :num_records]), "recall": own(pr["recall"][vi, :, :num_records]),
           "num_gt": np.array(gt_hist[view]), "best_f1": pr["best_f1"][vi], "best_index": pr["best_index"][vi]}
    if confidences is not None:
        res["at_confidence"] = pr["at_confidence"][vi]
    return res


def _average_recall(tp, gt_hist, view, max_dets, per_scale) -> Dict[str, Any]:
    """compute()'s average-recall keys from the ``(MAP_VIEWS, C, T, K)`` true positives counted by
    ``mgd_map_recall_update`` in the first limit bucket above their rank.  ``recall[v, c, t, k]`` is
    the prefix sum over the buckets over ``gt_hist[v, c]``, -1.0 where that is 0; an AR is its mean
    over the classes with ground truth and every threshold, 0.0 when no class has any."""
    gt = np.asarray(gt_hist, dtype=np.int64)[:, :, None, None]
    cum = np.cumsum(np.asarray(tp, dtype=np.int64), axis=-1)
    with np.errstate(divide="ignore", invalid="ignore"):
        recall = np.where(gt > 0, cum / gt, -1.0)

    def mean(v, k):
        has = gt_hist[v] > 0
        return float(np.mean(recall[v][has][:, :, k])) if has.any() else 0.0
    res = {f"AR{m}": mean(view, k) for k, m in enumerate(max_dets)}
    for key, v in (("ARS", _lib.MAP_VIEW_S), ("ARM", _lib.MAP_VIEW_M), ("ARL", _lib.MAP_VIEW_L)):
        res[key] = mean(v, len(max_dets) - 1) if per_scale else 0.0
    res["recall"] = {"max_dets": tuple(max_dets), "matcher": "corner" if view == _lib.MAP_VIEW_CORNER else "centre",
                     "num_gt": np.array(gt_hist[view]), "recall": recall[view]}
    return res


class MapAccumulator:
    """``calculate_map`` fed batch by batch with device tensors, without the lists of dicts.

    ``update`` takes the padded per-image tensors ``match_detections`` takes (torch CUDA
    tensors; ``det_boxes`` may be the int32 ``boxes_xyxy`` of ``engine.decode_nms``) and only
    enqueues work on the current stream: it matches the batch with every matcher the
    configuration can need and appends one record per padded detection slot
    (``mgd_map_update``).  ``compute`` sorts the records and computes the APs on the device
    (``mgd_map_compute``) and returns ``calculate_map``'s result dict for all updates so far,
    the detections listed image by image in slot order.  The arguments are
    ``calculate_map``'s.  Scores must be finite and class ids in [0, num_classes);
    ``compute`` raises AssertionError for a class id outside that range.

    The AP follows ``np.argsort`` of the recalls as NumPy's generic introsort orders equal
    ones, which is how the reference's numbers were produced (NumPy without its SIMD sort
    dispatch, the pin of ``oracle/ref_loader.py``).  Where NumPy dispatches its argsort to
    AVX-512 or AVX2 it orders those ties differently, and ``calculate_map`` itself then gives
    different numbers from one CPU to another.

    ``recall_max_dets`` (e.g. pycocotools' ``(1, 10, 100)``; up to 8 increasing limits) adds
    COCO-style average recall to every ``compute()`` dict: ``AR{k}`` per limit, ``ARS`` / ``ARM`` /
    ``ARL`` at the largest limit (0.0 without ``compute_per_scale``, as ``APS`` is), and ``"recall"``
    (see ``compute``).  It is pycocotools' AR with this matcher: per (image, class) the first k
    detections by descending score (equal scores: later slot first, where pycocotools takes the
    earlier first) are kept, and there are no crowd or ignore regions, so the numbers are not
    pycocotools' own.  It costs one more kernel per ``update``; ``None`` adds nothing.
    """

    def __init__(self, num_classes: int, iou_thresholds: List[float] = None, class_names: List[str] = None,
                 method: str = "coco", use_parallel: bool = True, optimize_classes: bool = True,
                 cache_ious: bool = True, compute_per_scale: bool = True, device=None, recall_max_dets=None):
        self._recall_limits = None if recall_max_dets is None else engine.recall_limits(recall_max_dets)
        if iou_thresholds is None:
            iou_thresholds = list(COCO_THRESHOLDS)
        if class_names is None:
            class_names = [f"class_{i}" for i in range(num_classes)]
        # the matcher of the full set is chosen at compute() (it depends on the prediction
        # count): with cache_ious and use_parallel both are matched
        views = [_lib.MAP_VIEW_CORNER] if cache_ious else [_lib.MAP_VIEW_CENTRE]
        if cache_ious and use_parallel:
            views.append(_lib.MAP_VIEW_CENTRE)
        if compute_per_scale:
            views += [_lib.MAP_VIEW_S, _lib.MAP_VIEW_M, _lib.MAP_VIEW_L]
        self._cfg = engine.map_config(num_classes, iou_thresholds, method, views)
        self._args = (int(num_classes), list(iou_thresholds), list(class_names), method, use_parallel,
                      optimize_classes, cache_ious, compute_per_scale)
        import torch
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self._record_bytes = engine.map_record_bytes()
        self.reset()

    def reset(self) -> None:
        """Forget every update."""
        import torch
        self._records = torch.empty((0,), dtype=torch.uint8, device=self.device)
        self._slots = 0
        self._gt_hist = torch.zeros((_lib.MAP_VIEWS, self._cfg.num_classes), dtype=torch.int64, device=self.device)
        if self._recall_limits is not None:
            self._recall_tp = torch.zeros((_lib.MAP_VIEWS, self._cfg.num_classes, self._cfg.num_thresholds,
                                           len(self._recall_limits)), dtype=torch.int64, device=self.device)

    def update(self, det_boxes, det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts) -> None:
        """Add one batch: det_boxes (B, M, 4) xyxy, det_scores (B, M), det_classes (B, M),
        det_counts (B,), gt_boxes (B, N, 4) xyxy, gt_classes (B, N), gt_counts (B,)."""
        slots = int(det_scores.shape[0]) * int(det_scores.shape[1])
        self._reserve(slots)
        engine.map_update(self._cfg, self._records, self._slots, self._gt_hist, det_boxes, det_scores,
                          det_classes, det_counts, gt_boxes, gt_classes, gt_counts)
        if self._recall_limits is not None:
            engine.map_recall_update(self._cfg, self._records, self._slots, int(det_scores.shape[0]),
                                     int(det_scores.shape[1]), self._recall_limits, self._recall_tp)
        self._slots += slots

    def _reserve(self, slots: int) -> None:
        """Room for ``slots`` more records behind the used ones (grown by doubling, on the stream)."""
        import torch
        need = (self._slots + slots) * self._record_bytes
        if need > self._records.numel():
            grown = torch.empty((max(need, 2 * self._records.numel()),), dtype=torch.uint8, device=self.device)
            used = self._slots * self._record_bytes
            grown[:used].copy_(self._records[:used])
            self._records = grown

    def compute(self, precision_recall: bool = False, confidences=None) -> Dict[str, Any]:
        """``calculate_map``'s result dict over every update since construction or ``reset``.

        With ``precision_recall`` the same dict gains ``"precision_recall"``, computed in the same
        library call (``mgd_map_compute_pr``) for the matcher ``calculate_map`` uses for its main
        APs (``"matcher"``: 'corner' or 'centre'), per class ``c`` and threshold ``t``:

        - ``offsets`` (C+1,), ``scores`` (n,), ``precision`` / ``recall`` (T, n): CUDA tensors.
          The curve of class c is ``[offsets[c], offsets[c+1])``: its detections by descending
          score (equal scores: later detection first), with ``compute_precision_recall``'s
          values of the sorted TP / FP flags of ``match_predictions_to_gt(_cached)``, bit for bit.
          A class without detections has an empty segment, not the reference's ``([0.0], [0.0])``.
        - ``num_gt`` (C,): ground truth per class.
        - ``best_f1`` (C, T, 4): (confidence, precision, recall, F1) at the first maximum of
          ``F1 = 2 p r / (p + r)`` among the detections that end a run of equal scores -- the
          points a ``score >= confidence`` filter can produce; zeros when that maximum is 0.
          ``best_index`` (C, T): its position in the class's curve, -1 where ``best_f1`` is zeros.
        - ``at_confidence`` (C, T, Q, 3), with ``confidences`` (up to 32 finite values): the
          (precision, recall, F1) of the detections with ``score >= confidences[q]``, zeros where
          none is left.  Equal to filtering the detections by that score and evaluating again.

        With ``recall_max_dets`` the dict also holds ``AR{k}``, ``ARS`` / ``ARM`` / ``ARL`` and
        ``"recall"``: ``max_dets``, ``matcher`` (the main APs' view, as above), ``num_gt`` (C,) and
        ``recall`` (C, T, K) float64, the true positives among the first ``max_dets[k]`` detections of
        every (image, class) over ``num_gt``, -1.0 for a class without ground truth.  ``AR{k}`` is
        the mean of ``recall[..., k]`` over the classes with ground truth and every threshold (0.0
        if there are none); at a limit >= the detections per image it is the final recall of the
        curves above.  The band ARs do the same in the area band's view at the largest limit.
        """
        _check_pr_args(precision_recall, confidences)
        if precision_recall:
            return self._compute_pr(confidences)
        out = engine.map_compute(self._cfg, self._records, self._slots, self._gt_hist)
        engine.poll_status(self.device.index or 0)
        full = _lib.MAP_VIEW_CORNER if self._args[6] else _lib.MAP_VIEW_CENTRE    # a view always matched
        gt = self._gt_hist.cpu().numpy()
        src = _DeviceSource(out, gt, full)
        return self._with_recall(_map_results(src, *self._args), src, gt, self._recall_tp_host())

    def _recall_tp_host(self):
        return None if self._recall_limits is None else self._recall_tp.cpu().numpy()

    def _with_recall(self, res, src, gt, recall_tp) -> Dict[str, Any]:
        """``res`` with the average-recall keys, in the view ``_map_results`` took its APs from."""
        if recall_tp is not None:
            res.update(_average_recall(recall_tp, gt, src.matcher_view, self._recall_limits, self._args[7]))
        return res

    def _compute_pr(self, confidences) -> Dict[str, Any]:
        # the matcher of the main APs is only known from the counts: curves of both full-set views
        out = engine.map_compute_pr(self._cfg, self._records, self._slots, self._gt_hist, _full_views(self._cfg),
                                    confidences)
        engine.poll_status(self.device.index or 0)
        full = _lib.MAP_VIEW_CORNER if self._args[6] else _lib.MAP_VIEW_CENTRE
        gt = self._gt_hist.cpu().numpy()
        src = _DeviceSource(out, gt, full)
        res = _map_results(src, *self._args)
        n = int(out["det_hist"][src.matcher_view].sum())
        res["precision_recall"] = _precision_recall(out["pr"], src.matcher_view, n, gt, confidences)
        return self._with_recall(res, src, gt, self._recall_tp_host())


def global_slot_segments(updates, rank: int, world_size: int):
    """The sharded accumulator's global slots.  ``updates``: ``(n_total, max_dets)`` of every
    update in order, the global batch of each split over the ranks by ``shard_bounds``.  Local
    slot j of update u on ``rank`` is global slot ``G_u + lo * M_u + (j - L_u)``: ``G_u`` the
    slots of all ranks over the earlier updates, ``lo`` the rank's first image, ``L_u`` its
    local slot offset.  Returns the segments ``[(L_u, G_u + lo * M_u)]`` of the updates where
    this rank has slots, and the global slot count."""
    from ..sharding import shard_bounds
    segments, local, glob = [], 0, 0
    for n_total, m in updates:
        lo, hi = shard_bounds(n_total, rank, world_size)
        if (hi - lo) * m:
            segments.append((local, glob + lo * m))
        local += (hi - lo) * m
        glob += n_total * m
    return segments, glob


def check_same_updates(updates, error=None, group=None) -> None:
    """Collective over ``group`` (nothing to do without ``torch.distributed`` or at world size
    1): raises ValueError on every rank if the ranks' ``(n_total, max_dets)`` update sequences
    differ, and AssertionError on every rank if any rank passes an ``error`` (the class-range
    report of its updates).  One ``all_gather_object``; no device is needed."""
    from ..sharding import _dist
    d = _dist()
    if d is not None and d.get_world_size(group) > 1:
        infos = [None] * d.get_world_size(group)
        d.all_gather_object(infos, ([tuple(int(x) for x in u) for u in updates], error), group=group)
        seqs = [seq for seq, _ in infos]
        bad = [r for r, seq in enumerate(seqs) if seq != seqs[0]]
        if bad:
            raise ValueError(f"ranks {[0] + bad} made different update sequences (n_total, max_dets): "
                             f"{len(seqs[0])} updates on rank 0, {[len(seqs[r]) for r in bad]} on the others")
        errors = [(r, e) for r, (_, e) in enumerate(infos) if e]
    else:
        errors = [(0, error)] if error else []
    if errors:
        r, e = errors[0]
        raise AssertionError(f"rank {r}: {e}")


class ShardedMapAccumulator(MapAccumulator):
    """``MapAccumulator`` over a batch sharded across the ranks of ``group`` (contiguous shards,
    ``sharding.shard_bounds``), e.g. fed by ``ShardedGridPath.decode_nms(gather=False)``.

    ``update`` takes this rank's shard of a global batch and, like ``MapAccumulator.update``,
    only enqueues the matching on the current stream; it makes no collective call.  Every rank
    makes the same sequence of updates.  ``compute`` is collective: each rank groups its
    records by the rank that owns their class (class ``c`` belongs to rank ``c % world``;
    ``mgd_map_partition``), the records are exchanged with ``all_to_all_single`` (device
    tensors with NCCL, host memory with any other backend), each rank sorts what it received and
    computes the APs of its own classes (``mgd_map_compute_merged``), and one all-reduce
    assembles the tables.  Every rank returns the same dict, equal to ``MapAccumulator``'s over
    the whole data: equal scores of a class are ordered later detection first in global image
    order, because every record carries its global slot (``global_slot_segments``).  The
    update sequences and the class-range status of all ranks are compared first, so a class id
    out of range raises AssertionError on every rank.  Without ``torch.distributed`` or at world
    size 1 the same partition and merged compute run without collectives.  With
    ``recall_max_dets`` each rank counts the true positives of its own images by rank, and the
    counts join the one all-reduce."""

    def __init__(self, num_classes: int, iou_thresholds: List[float] = None, class_names: List[str] = None,
                 method: str = "coco", use_parallel: bool = True, optimize_classes: bool = True,
                 cache_ious: bool = True, compute_per_scale: bool = True, device=None, group=None,
                 recall_max_dets=None):
        import torch
        from ..sharding import _dist
        d = _dist()
        self.group = group
        self.rank, self.world_size = (d.get_rank(group), d.get_world_size(group)) if d else (0, 1)
        super().__init__(num_classes, iou_thresholds, class_names, method, use_parallel, optimize_classes,
                         cache_ious, compute_per_scale, device, recall_max_dets)
        self._owner = (torch.arange(int(num_classes), device=self.device) % self.world_size).to(torch.int32)

    def reset(self) -> None:
        """Forget every update (on this rank; every rank resets together)."""
        super().reset()
        self._updates = []

    def update(self, det_boxes, det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts,
               n_total: int = None) -> None:
        """Add this rank's shard of a global batch of ``n_total`` images (default: the local batch
        times the world size).  The shard must be the one ``shard_bounds(n_total)`` gives this
        rank, possibly empty (a (0, M) / (0, N) batch), with the same M on every rank."""
        n_total = self._shard_total(int(det_scores.shape[0]), n_total)
        super().update(det_boxes, det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts)
        self._updates.append((n_total, int(det_scores.shape[1])))

    def _shard_total(self, n_local: int, n_total) -> int:
        """``n_total`` (default: ``n_local`` times the world size), checked against this rank's shard."""
        from ..sharding import shard_bounds
        n_total = n_local * self.world_size if n_total is None else int(n_total)
        lo, hi = shard_bounds(n_total, self.rank, self.world_size)
        if hi - lo != n_local:
            raise ValueError(f"rank {self.rank} holds {n_local} images, shard_bounds({n_total}) says {hi - lo}")
        return n_total

    def _mark(self, phase: str) -> None:
        """Called as each phase of ``compute`` has been enqueued ('check', 'partition', 'exchange',
        'merged', 'reduce'); a hook for timing."""

    def compute(self, precision_recall: bool = False, confidences=None) -> Dict[str, Any]:
        """``calculate_map``'s result dict over every rank's updates (collective).

        ``precision_recall`` / ``confidences`` as for ``MapAccumulator.compute``, in the same
        collective calls: every rank holds the whole ``best_f1`` / ``best_index`` /
        ``at_confidence`` tables (they join the one all-reduce), while the curves stay on the
        rank that owns the class.  ``owned`` (C,) marks this rank's classes; the other classes
        have empty curve segments here.  The average-recall keys are the same on every rank."""
        _check_pr_args(precision_recall, confidences)
        host, gt, pr = self._merged_tables(precision_recall, confidences)
        full = _lib.MAP_VIEW_CORNER if self._args[6] else _lib.MAP_VIEW_CENTRE
        src = _DeviceSource(host, gt, full)
        res = self._with_recall(_map_results(src, *self._args), src, gt, host.pop("recall_tp", None))
        if pr is not None:
            for k in engine._MAP_PR_TABLES:
                pr[k] = pr[k].cpu().numpy()
            owned = (self._owner == self.rank).cpu().numpy()
            n = int(host["det_hist"][src.matcher_view][owned].sum())     # this rank's records
            res["precision_recall"] = _precision_recall(pr, src.matcher_view, n, gt, confidences)
            res["precision_recall"]["owned"] = owned
        return res

    def _rank_counts(self):
        """Counts of this rank's own images that the all-reduce sums, by name (int64 CUDA tensors)."""
        return {} if self._recall_limits is None else {"recall_tp": self._recall_tp}

    def _merged_tables(self, precision_recall: bool = False, confidences=None):
        """The collective part of ``compute``: the update check, the record exchange, the merged
        compute and the all-reduce.  Returns the summed tables as NumPy arrays (``det_hist``, ``ap``
        or ``voc``, and every ``_rank_counts`` entry), the summed ground-truth counts (NumPy) and
        the curve outputs (or None)."""
        error = None
        try:
            engine.poll_status(self.device.index or 0)
        except AssertionError as e:
            error = str(e)
        check_same_updates(self._updates, error, self.group)
        self._mark("check")
        segments, global_slots = global_slot_segments(self._updates, self.rank, self.world_size)
        send, counts = engine.map_partition(self._cfg, self._records, self._slots, segments, global_slots,
                                            self._owner, self.world_size)
        self._mark("partition")
        if self.world_size == 1:
            recs, n_recv, gt_hist = send, int(counts[0]), self._gt_hist
        else:
            recs, n_recv, gt_hist = self._exchange(send, counts)
        self._mark("exchange")
        if precision_recall:
            out = engine.map_compute_merged_pr(self._cfg, recs, n_recv, gt_hist, self._owner, self.rank,
                                               _full_views(self._cfg), confidences)
        else:
            out = engine.map_compute_merged(self._cfg, recs, n_recv, gt_hist, self._owner, self.rank)
        out.update(self._rank_counts())
        self._mark("merged")
        if self.world_size > 1:
            out = self._all_reduce(out)
        pr = out.pop("pr", None)
        host = {k: v.cpu().numpy() for k, v in out.items()}
        self._mark("reduce")
        return host, gt_hist.cpu().numpy(), pr

    def _wire(self):
        """Where the collectives' tensors live: the device with NCCL, host memory otherwise."""
        import torch
        from ..sharding import _dist
        return self.device if _dist().get_backend(self.group) == "nccl" else torch.device("cpu")

    def _exchange(self, send, counts):
        """Each rank's records to the ranks that own their classes; the summed ground truth."""
        import torch
        from ..sharding import _dist
        d, g, rb, wire = _dist(), self.group, self._record_bytes, self._wire()
        counts = counts.to(wire)
        recv_counts = torch.empty_like(counts)
        gt_hist = self._gt_hist.to(wire, copy=True)            # the local one stays: more updates may follow
        d.all_to_all_single(recv_counts, counts, group=g)
        d.all_reduce(gt_hist, group=g)
        send_splits = [c * rb for c in counts.tolist()]
        recv_splits = [c * rb for c in recv_counts.tolist()]
        recs = torch.empty((sum(recv_splits),), dtype=torch.uint8, device=wire)
        d.all_to_all_single(recs, send[:sum(send_splits)].to(wire), recv_splits, send_splits, group=g)
        return recs.to(self.device), sum(recv_splits) // rb, gt_hist.to(self.device)

    def _all_reduce(self, out):
        """Sum the ranks' tables: each (view, class) is non-zero on its owner only, so the sums are
        exact.  One float64 all-reduce; the detection counts, best indices and the counts of each
        rank's own images (``_rank_counts``) travel as float64 (exact below 2^53).  The curves are
        not sent."""
        import torch
        from ..sharding import _dist
        key = "ap" if "ap" in out else "voc"
        pr = out.get("pr")
        counts = [k for k in out if k not in (key, "det_hist", "pr")]
        tables = [out[key], out["det_hist"]] + [out[k] for k in counts] + \
            ([pr[k] for k in engine._MAP_PR_TABLES] if pr else [])
        flat = torch.cat([t.reshape(-1).to(torch.float64) for t in tables]).to(self._wire())
        _dist().all_reduce(flat, group=self.group)
        summed, lo = [], 0
        for t in tables:
            summed.append(flat[lo:lo + t.numel()].to(t.dtype).reshape(t.shape))
            lo += t.numel()
        res = {key: summed.pop(0), "det_hist": summed.pop(0)}
        for k in counts:
            res[k] = summed.pop(0)
        if pr:
            res["pr"] = dict(pr, **dict(zip(engine._MAP_PR_TABLES, summed)))
        return res


class ConfusionMatrixAccumulator:
    """Detection confusion matrix at chosen confidences, fed batch by batch with device tensors.

    For each confidence ``confidences[q]`` the detections with ``score >= confidences[q]`` are
    matched first with the reference's matcher of their own class (``match_predictions_to_gt_cached``
    with ``iou_mode='corner'``, ``match_predictions_to_gt`` with 'centre'), then the ones left
    unmatched claim, in the same order, the still-unclaimed ground truth of any class with the
    highest IoU when it is ``>= iou_threshold`` (``mgd_confusion_update``).  ``compute`` returns a
    host int64 array ``(Q, C+1, C+1)``: rows are the true class, columns the detected class, as in
    ``sklearn.metrics.confusion_matrix``, and index C is background -- row C holds the false
    positives on nothing, column C the missed objects.  The diagonal is the matcher's TP count at
    that confidence; row g < C sums to the ground truth of class g, column d < C to the class-d
    detections kept.

    ``confidences=None`` is a single matrix (Q = 1) over every detection passed in; a typical
    choice is the confidence ``MapAccumulator.compute(precision_recall=True)`` gives in
    ``best_f1``, or up to 32 of them.  ``iou_mode='centre'`` is there only so that the diagonal
    agrees with ``calculate_map`` where the reference switches to its un-cached matcher, which reads
    the xyxy boxes as centre format (more than 10 000 predictions with ``use_parallel``, i.e. every
    COCO-val-sized run); 'corner' is the correct IoU.

    ``update`` takes ``MapAccumulator.update``'s tensors (``det_boxes`` may be the int32
    ``boxes_xyxy`` of ``engine.decode_nms``) and only enqueues work on the current stream.  Scores
    must be finite; ``compute`` raises AssertionError for a class id outside [0, num_classes).
    """

    def __init__(self, num_classes: int, iou_threshold: float = 0.5, confidences=None, iou_mode: str = "corner",
                 device=None):
        self.num_classes, self.iou_threshold, self.confidences, _ = engine.confusion_config(
            num_classes, iou_threshold, confidences, iou_mode)
        self.iou_mode = iou_mode
        import torch
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.reset()

    def reset(self) -> None:
        """Forget every update."""
        import torch
        C1 = self.num_classes + 1
        self._matrix = torch.zeros((len(self.confidences), C1, C1), dtype=torch.int64, device=self.device)

    def update(self, det_boxes, det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts) -> None:
        """Add one batch: det_boxes (B, M, 4) xyxy, det_scores (B, M), det_classes (B, M),
        det_counts (B,), gt_boxes (B, N, 4) xyxy, gt_classes (B, N), gt_counts (B,)."""
        engine.confusion_update(self._matrix, self.confidences, self.iou_threshold, self.iou_mode, det_boxes,
                                det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts)

    def compute(self) -> np.ndarray:
        """The (Q, C+1, C+1) int64 matrices over every update since construction or ``reset``."""
        engine.poll_status(self.device.index or 0)
        return self._matrix.cpu().numpy()


class ShardedConfusionMatrixAccumulator(ConfusionMatrixAccumulator):
    """``ConfusionMatrixAccumulator`` over a batch sharded across the ranks of ``group``.

    ``update`` takes this rank's shard (any split of the images, possibly empty) and makes no
    collective call.  ``compute`` is collective: one int64 all-reduce sums the ranks' matrices (on
    the device with NCCL, through host memory with any other backend), with one more element for
    the rank's class-range error, so a rank that saw one still joins the reduce and every rank then
    raises AssertionError.  Every rank returns the same matrix, equal to the single-process one.
    Without ``torch.distributed`` or at world size 1 it makes no collective call."""

    def __init__(self, num_classes: int, iou_threshold: float = 0.5, confidences=None, iou_mode: str = "corner",
                 device=None, group=None):
        from ..sharding import _dist
        d = _dist()
        self.group = group
        self.world_size = d.get_world_size(group) if d else 1
        super().__init__(num_classes, iou_threshold, confidences, iou_mode, device)

    def compute(self) -> np.ndarray:
        """The (Q, C+1, C+1) int64 matrices over every rank's updates (collective)."""
        import torch
        from ..sharding import _dist
        error = None
        try:
            engine.poll_status(self.device.index or 0)
        except AssertionError as e:
            error = str(e)
        if self.world_size == 1:
            if error:
                raise AssertionError(error)
            return self._matrix.cpu().numpy()
        d = _dist()
        wire = self.device if d.get_backend(self.group) == "nccl" else torch.device("cpu")
        flat = torch.cat([self._matrix.reshape(-1),
                          torch.tensor([1 if error else 0], dtype=torch.int64, device=self.device)]).to(wire)
        d.all_reduce(flat, group=self.group)
        flat = flat.cpu()
        if int(flat[-1]):
            raise AssertionError(error or f"class id outside [0, num_classes) on {int(flat[-1])} other rank(s)")
        return flat[:-1].reshape(self._matrix.shape).numpy()


TIDE_FIXES = ("Cls", "Loc", "Both", "Dupe", "Bkg", "Miss", "FP", "FN")     # record sets 1 .. 8
TIDE_ERRORS = ("Cls", "Loc", "Both", "Dupe", "Bkg", "Miss")


def _error_analysis(out, gt_hist, num_classes: int, method: str) -> Dict[str, Any]:
    """``ErrorAnalysisAccumulator.compute``'s dict from one map compute over the ``TIDE_SETS * C``
    classes of the record sets (``det_hist``, ``ap`` / ``voc``) plus the ``counts`` (C, 6)."""
    C, F = num_classes, _lib.TIDE_SETS
    ap_of = _DeviceSource(out, gt_hist, _lib.MAP_VIEW_CORNER).ap_table([None], "corner", method)
    ap = np.array([[ap_of(f * C + c, 0) for c in range(C)] for f in range(F)], dtype=np.float64)
    det, gt = out["det_hist"][_lib.MAP_VIEW_CORNER], gt_hist[_lib.MAP_VIEW_CORNER]
    active = np.flatnonzero((det[:C] > 0) | (gt[:C] > 0))       # calculate_map's optimize_classes set
    mean = lambda row: float(np.mean(row[active])) if len(active) else 0.0
    base = mean(ap[0])
    counts = np.asarray(out["counts"], dtype=np.int64)
    return {"AP": base,
            "dAP": {k: mean(ap[f + 1]) - base for f, k in enumerate(TIDE_FIXES)},
            "counts": {k: int(counts[:, e].sum()) for e, k in enumerate(TIDE_ERRORS)},
            "per_class": {"AP": ap[0], "dAP": (ap[1:] - ap[0]).T.copy(), "counts": counts}}


class ErrorAnalysisAccumulator(MapAccumulator):
    """TIDE-style detection error analysis (Bolya et al., ECCV 2020): what each kind of error costs
    in AP, fed batch by batch with device tensors (``mgd_tide_update``).

    The base is the reference's matcher at ``pos_threshold`` t_f (``iou_mode`` 'corner':
    ``match_predictions_to_gt_cached``, 'centre': ``match_predictions_to_gt``, as in
    ``ConfusionMatrixAccumulator``); every detection is used.  Each false positive d gets one type
    from its best IoU ``s`` with the ground truth of its own class (claimed or not) and ``o`` with
    that of the other classes, the first that applies: Bkg ``max(s, o) < background_threshold``;
    Cls ``o >= t_f``; Dupe ``s >= t_f``; Loc ``s >= background_threshold``; Both otherwise.  A Miss is
    a ground truth the base left unclaimed that no Cls or Loc error targets (the ground truth
    attaining ``o`` or ``s``; equal IoU: the lowest index).

    Each fix is applied alone to the base, and the AP of the fixed detections is ``calculate_map``'s
    AP arithmetic at one threshold: Cls gives d its target's class and Loc keeps d's class, and in
    the visiting order (score descending, equal scores later slot first) d then claims the target
    as a TP if no one holds it yet, or is dropped; Both / Dupe / Bkg drop those detections; Miss
    removes the missed ground truth; FP drops every false positive; FN leaves each class only its
    claimed ground truth.  ``dAP[e]`` is the mean AP over classes with fix e minus the base mean,
    both over the classes with detections or ground truth (``calculate_map``'s ``optimize_classes``
    set); the base ``AP`` is ``MapAccumulator``'s mAP at ``iou_thresholds=[pos_threshold]`` with the
    same matcher.  This is TIDE's definition with this project's matcher and AP arithmetic, with
    no crowd or ignore regions and these tie rules, so the numbers are not ``tidecv``'s own (which
    also uses 101-point AP).

    ``update`` takes ``MapAccumulator.update``'s tensors (``det_boxes`` may be the int32
    ``boxes_xyxy`` of ``engine.decode_nms``) and only enqueues work on the current stream; it keeps
    ``TIDE_SETS`` (9) records of 40 bytes per padded detection slot.  Scores must be finite;
    ``compute`` raises AssertionError for a class id outside [0, num_classes).  ``class_names``
    label the rows of ``per_class`` for the caller; the dict does not use them.
    """

    def __init__(self, num_classes: int, pos_threshold: float = 0.5, background_threshold: float = 0.1,
                 iou_mode: str = "corner", method: str = "coco", class_names: List[str] = None, device=None):
        C, self.pos_threshold, self.background_threshold, _ = engine.tide_config(
            num_classes, pos_threshold, background_threshold, iou_mode)
        self.num_classes, self.iou_mode = C, iou_mode
        self.class_names = [f"class_{i}" for i in range(C)] if class_names is None else list(class_names)
        self._init_map(method, device)

    def _init_map(self, method, device):
        # the record sets are blocks of C classes of one map evaluation: one threshold, corner view
        MapAccumulator.__init__(self, _lib.TIDE_SETS * self.num_classes, [self.pos_threshold], None, method,
                                use_parallel=False, compute_per_scale=False, device=device)

    def reset(self) -> None:
        """Forget every update."""
        import torch
        super().reset()
        self._counts = torch.zeros((self.num_classes, _lib.TIDE_ERRORS), dtype=torch.int64, device=self.device)

    def update(self, det_boxes, det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts) -> None:
        """Add one batch: det_boxes (B, M, 4) xyxy, det_scores (B, M), det_classes (B, M),
        det_counts (B,), gt_boxes (B, N, 4) xyxy, gt_classes (B, N), gt_counts (B,)."""
        slots = _lib.TIDE_SETS * int(det_scores.shape[0]) * int(det_scores.shape[1])
        self._reserve(slots)
        engine.tide_update(self._records, self._slots, self._gt_hist, self._counts, self.pos_threshold,
                           self.background_threshold, self.iou_mode, det_boxes, det_scores, det_classes,
                           det_counts, gt_boxes, gt_classes, gt_counts)
        self._slots += slots

    def compute(self) -> Dict[str, Any]:
        """Over every update since construction or ``reset``:

        - ``AP``: the base mAP at ``pos_threshold``;
        - ``dAP``: ``{"Cls", "Loc", "Both", "Dupe", "Bkg", "Miss", "FP", "FN"}``, the rise of that
          mAP when only that error is fixed;
        - ``counts``: ``{"Cls", "Loc", "Both", "Dupe", "Bkg", "Miss"}``, the number of errors;
        - ``per_class``: ``AP`` (C,) float64, ``dAP`` (C, 8) float64 in the order above, ``counts``
          (C, 6) int64 (a false positive counts under its detection's class, a Miss under its
          ground truth's).  A class's AP follows ``calculate_map``: 0.0 with ground truth but no
          detections or detections but no ground truth, 1.0 with neither.
        """
        out, gt = self._tables()
        return _error_analysis(out, gt, self.num_classes, self._args[3])

    def _tables(self):
        out = engine.map_compute(self._cfg, self._records, self._slots, self._gt_hist)
        engine.poll_status(self.device.index or 0)
        out["counts"] = self._counts.cpu().numpy()
        return out, self._gt_hist.cpu().numpy()


class ShardedErrorAnalysisAccumulator(ErrorAnalysisAccumulator, ShardedMapAccumulator):
    """``ErrorAnalysisAccumulator`` over a batch sharded across the ranks of ``group``, with
    ``ShardedMapAccumulator``'s machinery: ``update`` takes this rank's shard (as
    ``ShardedMapAccumulator.update``, with ``n_total``) and makes no collective call; ``compute`` is
    collective.  The record sets are exchanged and their APs computed class by class on the rank
    that owns the class, and the error counts of each rank's images join the one all-reduce.  The
    update sequences and class-range status of all ranks are compared first, so a class id out of
    range raises AssertionError on every rank.  Every rank returns the same dict, equal to the
    single-process one.  Without ``torch.distributed`` or at world size 1 it makes no collective
    call."""

    def __init__(self, num_classes: int, pos_threshold: float = 0.5, background_threshold: float = 0.1,
                 iou_mode: str = "corner", method: str = "coco", class_names: List[str] = None, device=None,
                 group=None):
        self.group = group
        super().__init__(num_classes, pos_threshold, background_threshold, iou_mode, method, class_names, device)

    def _init_map(self, method, device):
        ShardedMapAccumulator.__init__(self, _lib.TIDE_SETS * self.num_classes, [self.pos_threshold], None, method,
                                       use_parallel=False, compute_per_scale=False, device=device, group=self.group)

    def update(self, det_boxes, det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts,
               n_total: int = None) -> None:
        """Add this rank's shard of a global batch of ``n_total`` images (default: the local batch
        times the world size), as ``ShardedMapAccumulator.update``."""
        n_total = self._shard_total(int(det_scores.shape[0]), n_total)
        super().update(det_boxes, det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts)
        self._updates.append((n_total, _lib.TIDE_SETS * int(det_scores.shape[1])))

    def _rank_counts(self):
        return {"counts": self._counts}

    def _tables(self):
        out, gt, _ = self._merged_tables()
        return out, gt
