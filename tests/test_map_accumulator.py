"""Streaming mAP on the device (evaluation.MapAccumulator, mgd_map_update / mgd_map_compute).

CPU: argument validation before any device work, the entry points without a device, and the
property the device AP walk relies on (only the record NumPy's argsort of the recalls leaves at
the end of each run of equal recall enters the AP).  GPU: the accumulator against the real reference's calculate_map numbers
(tests/golden/metrics_cases.npz) and against the drop-in calculate_map on the same detections.
"""
import ctypes
import os

import numpy as np
import pytest

from multigriddet_b200 import _lib, engine
from oracle import metrics_oracle as MO
from oracle.gen_golden import synth_eval_set

GOLD = os.path.join(os.path.dirname(__file__), "golden", "metrics_cases.npz")
MAP_KEYS = ("mAP", "mAP50", "mAP75", "APS", "APM", "APL", "APS50", "APM50", "APL50")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    return _lib.load()


def _case(z, name):
    return tuple(z[f"{name}_{k}"] for k in ("db", "ds", "dc", "dn", "gtb", "gtc", "gtn")) + (int(z[f"{name}_C"]),)


# ------------------------------------------------------------------------------ CPU

def test_configuration_is_validated_before_any_device_call():
    from multigriddet_b200.evaluation import MapAccumulator
    for kw in (dict(num_classes=0), dict(num_classes=3, iou_thresholds=[]),
               dict(num_classes=3, iou_thresholds=[0.5] * 33), dict(num_classes=3, method="coco101")):
        with pytest.raises(ValueError):
            MapAccumulator(**kw)
    with pytest.raises(ValueError):
        engine.map_config(3, [0.5], views=())


def test_entry_points_validate_then_need_a_device(lib):
    assert lib.mgd_map_record_bytes() == 40
    cfg = engine.map_config(3, [0.5, 0.75], "coco", views=(_lib.MAP_VIEW_CORNER, _lib.MAP_VIEW_S))
    one = ctypes.c_void_p(8)                                # never dereferenced: validation or no device
    upd = lambda c, B=1: lib.mgd_map_update(ctypes.byref(c), one, one, one, one, B, 4, one, one, one, 2,
                                            0, one, one, 0, None, 0)
    cmp = lambda c, n=4: lib.mgd_map_compute(ctypes.byref(c), one, n, one, one, one, one, 0, None, 0)
    for field, bad in (("num_thresholds", 0), ("num_thresholds", 33), ("num_classes", 0), ("method", 7),
                       ("views", 0), ("views", 1 << _lib.MAP_VIEWS)):
        c = engine.map_config(3, [0.5, 0.75])
        setattr(c, field, bad)
        assert upd(c) == _lib.ERR_INVALID_ARGUMENT, field
        assert cmp(c) == _lib.ERR_INVALID_ARGUMENT, field
    assert upd(cfg, B=-1) == _lib.ERR_INVALID_ARGUMENT
    assert cmp(cfg, n=-1) == _lib.ERR_INVALID_ARGUMENT
    assert lib.mgd_map_compute(ctypes.byref(cfg), one, 4, one, None, one, one, 0, None, 0) == \
        _lib.ERR_INVALID_ARGUMENT                           # coco without ap_out
    if lib.mgd_device_count() == 0:
        assert upd(cfg) == _lib.ERR_NO_DEVICE
        assert cmp(cfg) == _lib.ERR_NO_DEVICE
        with pytest.raises(_lib.MgdError, match="no CPU fallback"):
            _lib.raise_for_status(cmp(cfg))


def _ap_at_run_ends(tp, n_gt, perm):
    """The AP as map_ap_kernel computes it: the records in sorted order; where the recall steps
    up, the interpolated precision of the run's last point is that of the record ``perm`` (the
    argsort of the recalls) leaves there."""
    cum_tp = np.cumsum(tp)
    p, r = MO.precision_recall(tp, n_gt)
    if len(r) == 1:
        return float(p[0] * r[0])
    later = np.maximum.accumulate(p[::-1])[::-1]           # max over the records at and after i
    ap = 0.0
    for i in np.flatnonzero(r[1:] != r[:-1]):
        q = cum_tp[i] / ((perm[i] + 1) + 1e-8)
        ap += (r[i + 1] - r[i]) * (later[i + 1] + max(q, later[i + 1])) / 2.0
    return ap


def test_ap_depends_only_on_the_argsort_of_each_recall_run_end():
    """compute_average_precision sorts the (already non-decreasing) recalls with NumPy's
    unstable argsort, which permutes runs of equal recall; the device takes the records in
    order and only asks which record the sort leaves at the end of each run."""
    z = np.load(GOLD)
    cases = [_case(z, n)[:7] for n in ("a", "b", "ties")] + [synth_eval_set(31, 30, 40, 12, 3, ties=True)]
    permuted = 0
    for db, ds, dc, dn, gtb, gtc, gtn in cases:
        for cached in (True, False):
            tp, _ = MO.match_batch(db, ds, dc, dn, gtb, gtc, gtn, [0.5, 0.75], cached)
            B = len(dn)
            ftp = np.concatenate([tp[:, b, :dn[b]] for b in range(B)], 1)
            fs = np.concatenate([ds[b, :dn[b]] for b in range(B)])
            fc = np.concatenate([dc[b, :dn[b]] for b in range(B)])
            ngt = np.bincount(np.concatenate([gtc[b, :gtn[b]] for b in range(B)]), minlength=int(fc.max()) + 1)
            for c in np.unique(fc):
                sel = fc == c
                order = np.argsort(fs[sel], kind="stable")[::-1]
                for t in range(2):
                    if ngt[c] == 0:
                        continue
                    flags = ftp[t][sel][order].astype(bool)
                    p, r = MO.precision_recall(flags, int(ngt[c]))
                    assert np.all(np.diff(r) >= 0)
                    perm = np.argsort(r)
                    permuted += not np.array_equal(perm, np.arange(len(r)))
                    ref = MO.average_precision(p, r)
                    assert _ap_at_run_ends(flags, int(ngt[c]), perm) == pytest.approx(ref, rel=1e-12, abs=1e-15)
    assert permuted > 0                                     # the sort did reorder equal recalls


# ------------------------------------------------------------------------------ GPU

def _dev(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _accumulate(C, pieces, args, **kw):
    from multigriddet_b200.evaluation import MapAccumulator
    acc = MapAccumulator(C, **kw)
    B = len(args[3])
    lo = 0
    for n in pieces:
        acc.update(*_dev(*[a[lo:lo + n] for a in args]))
        lo += n
    assert lo == B
    return acc.compute()


def _assert_same(got, ref, rel, path="result"):
    assert type(got) is type(ref) or (isinstance(got, float) and isinstance(ref, float)), (path, type(got), type(ref))
    if isinstance(ref, dict):
        assert set(got) == set(ref), (path, sorted(set(got) ^ set(ref)))
        for k in ref:
            _assert_same(got[k], ref[k], rel, f"{path}[{k!r}]")
    elif isinstance(ref, float) and rel:
        assert got == pytest.approx(ref, rel=rel, abs=1e-15), path
    else:
        assert got == ref, path


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["a", "b", "ties"])
def test_gpu_accumulator_against_reference_golden(name):
    z = np.load(GOLD)
    db, ds, dc, dn, gtb, gtc, gtn, C = _case(z, name)
    args = (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
    thr = [float(t) for t in z["thresholds"]]
    for cached, tag in ((True, "cached"), (False, "plain")):
        res = _accumulate(C, [len(dn)], args, use_parallel=False, cache_ious=cached)
        for key in MAP_KEYS:
            assert float(res[key]) == pytest.approx(float(z[f"{name}_{tag}_map_{key}"]), rel=1e-12, abs=1e-15), key
        for c in range(C):
            per = res["per_class"].get(f"class_{c}")
            if per is None:
                continue
            for t, th in enumerate(thr):
                ref = float(z[f"{name}_{tag}_c{c}_t{t}_ap"])
                assert float(per[f"AP{th:.2f}"]) == pytest.approx(ref, rel=1e-12, abs=1e-15), (tag, c, t)
        voc = _accumulate(C, [len(dn)], args, iou_thresholds=[0.5], method="voc", use_parallel=False,
                          cache_ious=cached, compute_per_scale=False)
        assert float(voc["mAP50"]) == pytest.approx(float(z[f"{name}_{tag}_map_voc50"]), rel=1e-12)


@pytest.mark.gpu
def test_gpu_streaming_is_invariant_to_how_the_images_are_split():
    args = synth_eval_set(41, 40, 30, 20, 6, ties=True)
    args = (args[0].astype(np.int32),) + args[1:]
    for kw in (dict(), dict(cache_ious=False), dict(method="voc", use_parallel=False)):
        whole = _accumulate(6, [40], args, **kw)
        split = _accumulate(6, [1, 7, 32], args, **kw)          # the record buffer grows twice
        _assert_same(split, whole, rel=0)


def _at_size_inputs():
    B, M, N, C = 2000, 100, 20, 80
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(43, B, M, N, C)
    ds = np.round(ds, 2)                                    # ties across images are common
    ds[1::97, 3] = -0.0
    ds[2::89, 5] = 0.0
    return (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn), C


@pytest.mark.gpu
def test_gpu_accumulator_equals_dropin_at_size():
    from multigriddet_b200.evaluation import calculate_map
    args, C = _at_size_inputs()
    preds, gts = MO.to_dicts(*args)
    assert len(preds) > 10000 and any(p["score"] == 0.0 and np.signbit(p["score"]) for p in preds)
    for kw in (dict(), dict(use_parallel=False), dict(optimize_classes=False),
               dict(method="voc", use_parallel=False)):
        ref = calculate_map(preds, gts, C, **kw)
        got = _accumulate(C, [256] * 7 + [208], args, **kw)
        _assert_same(got, ref, rel=1e-12, path=str(kw))


@pytest.mark.gpu
def test_gpu_accumulator_straight_from_decode_nms():
    import torch
    from multigriddet_b200 import synth
    from multigriddet_b200.evaluation import MapAccumulator, calculate_map
    S, C, B, N = 416, 20, 24, 40
    anchors = synth.coco_anchors(np.float32)
    boxes = synth.synth_boxes(44, B, N, S, C)
    y = engine.encode_targets(torch.from_numpy(boxes).cuda(), (S, S), anchors, C)
    preds = synth.planted_head_outputs(y, 3, seed=44)
    det = engine.decode_nms(preds, None, (S, S), anchors, C, max_boxes=100, confidence=0.05,
                            nms_threshold=0.45, nms_method="diou")
    gt_counts = ((boxes[..., 2] - boxes[..., 0]) * (boxes[..., 3] - boxes[..., 1]) > 0).sum(1).astype(np.int32)
    gt_boxes, gt_classes = boxes[..., :4].astype(np.float64), boxes[..., 4].astype(np.int32)
    acc = MapAccumulator(C)
    acc.update(det["boxes_xyxy"], det["scores"], det["classes"], det["counts"], *_dev(gt_boxes, gt_classes, gt_counts))
    got = acc.compute()
    host = [det[k].cpu().numpy() for k in ("boxes_xyxy", "scores", "classes", "counts")]
    p, g = MO.to_dicts(*host, gt_boxes, gt_classes, gt_counts)
    assert len(p) > 0 and got["num_predictions"] == len(p)
    _assert_same(got, calculate_map(p, g, C), rel=1e-12)


@pytest.mark.gpu
def test_gpu_accumulator_edge_cases():
    from multigriddet_b200.evaluation import MapAccumulator, calculate_map
    C = 4
    # every box large: no ground truth in the S and M bands; class 3 has predictions only
    gtb = np.array([[[0, 0, 200, 200], [50, 50, 300, 260], [0, 0, 0, 0]]], np.float64)
    gtc = np.array([[0, 1, 0]], np.int32)
    db = np.array([[[0, 0, 201, 199], [10, 10, 20, 20], [50, 50, 300, 250], [0, 0, 150, 150]]], np.int32)
    ds = np.array([[0.9, 0.8, 0.8, 0.3]])
    dc = np.array([[0, 0, 1, 3]], np.int32)
    args = (db, ds, dc, np.array([4], np.int32), gtb, gtc, np.array([2], np.int32))
    empty = (np.zeros((2, 5, 4), np.int32), np.zeros((2, 5)), np.zeros((2, 5), np.int32), np.zeros(2, np.int32),
             np.zeros((2, 3, 4)), np.zeros((2, 3), np.int32), np.zeros(2, np.int32))
    acc = MapAccumulator(C)
    acc.update(*_dev(*empty))                                # all counts 0
    assert acc.compute()["num_predictions"] == 0
    acc.update(*_dev(*args))
    got = acc.compute()
    ref = calculate_map(*MO.to_dicts(*args), C)
    _assert_same(got, ref, rel=1e-12)
    assert got["APS"] == 0.0 and got["APM"] == 0.0 and got["APL"] > 0.0
    assert got["per_class"]["class_3"]["AP"] == 0.0
    acc.reset()
    assert acc.compute()["num_predictions"] == 0
    bad = (db, ds, np.array([[0, 0, 1, 4]], np.int32)) + args[3:]
    acc.update(*_dev(*bad))
    with pytest.raises(AssertionError, match="class id"):
        acc.compute()
