"""Precision-recall curves and confidence operating points of the streaming mAP accumulators
(MapAccumulator / ShardedMapAccumulator.compute(precision_recall=True), mgd_map_compute_pr /
mgd_map_compute_merged_pr).

CPU: argument validation of both entry points before any device work, the mgd_map_pr layout,
and the two operating-point rules (restated here) (at a confidence: equal to filtering the detections
and evaluating again; best F1: run ends only).  GPU: the curves equal the drop-in host functions
bit for bit (match_predictions_to_gt(_cached) + compute_precision_recall), their APs equal
calculate_map's, the operating points equal the rules restated here, and the sharded tables and owned curves
equal the single-process ones (every comparison exact ==).
"""
import ctypes
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from multigriddet_b200 import _lib, engine
from oracle import metrics_oracle as MO
from oracle.gen_golden import synth_eval_set

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(os.path.dirname(__file__), "golden", "metrics_cases.npz")
CONFS = [-1.0, 0.0, 0.05, 0.3, 0.5, 0.75, 0.9, 0.99, 1.0, 2.0]      # 0.3 / 0.5 / 0.75 sit inside runs of ties


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    return _lib.load()


def _case(z, name):
    return tuple(z[f"{name}_{k}"] for k in ("db", "ds", "dc", "dn", "gtb", "gtc", "gtn")) + (int(z[f"{name}_C"]),)


# ------------------------------------------------------------------------------ operating-point rules
# A restatement of the two rules the device applies to one class's curve (scores descending, equal
# scores later detection first, with compute_precision_recall's values); the tests compare against it.

def f1_score(p, r):
    """F1 of one precision / recall pair: ``2.0 * p * r / (p + r)`` in that operation order, 0
    where ``p + r == 0``."""
    return 0.0 if p + r == 0 else 2.0 * p * r / (p + r)


def best_f1(scores, precisions, recalls):
    """The best-F1 operating point: only a record that ends a run of equal scores (the last record,
    or one whose successor's score differs) is a point a ``score >= confidence`` filter can
    produce.  Returns ``((confidence, precision, recall, f1), k)`` at the first maximum of F1 among
    those records, or ``((0, 0, 0, 0), -1)`` when that maximum is 0 or the curve is empty."""
    n = len(scores)
    best, best_k = 0.0, -1
    for k in range(n):
        if k + 1 < n and scores[k + 1] == scores[k]:
            continue
        f1 = f1_score(precisions[k], recalls[k])
        if f1 > best:
            best, best_k = f1, k
    if best_k < 0:
        return (0.0, 0.0, 0.0, 0.0), -1
    return (float(scores[best_k]), float(precisions[best_k]), float(recalls[best_k]), best), best_k


def at_confidence(scores, precisions, recalls, confidence):
    """(precision, recall, f1) of the curve cut at ``score >= confidence``: at record ``K - 1``,
    ``K`` the records with that score, or zeros when ``K == 0``.  The greedy match visits
    detections by descending score, so dropping the lower scores changes no earlier flag: this
    equals filtering the detections and evaluating again."""
    K = int(np.count_nonzero(np.asarray(scores) >= confidence))
    if K == 0:
        return 0.0, 0.0, 0.0
    p, r = float(precisions[K - 1]), float(recalls[K - 1])
    return p, r, f1_score(p, r)


# ------------------------------------------------------------------------------ CPU

def _pr_struct(views=1 << _lib.MAP_VIEW_CORNER, conf=(0.5,), capacity=4, **null):
    one = 8                                                 # never dereferenced: validation or no device
    arr = (ctypes.c_double * max(len(conf), 1))(*conf)
    pr = _lib.MapPr()
    pr.views, pr.num_confidences, pr.confidences, pr.capacity = views, len(conf), ctypes.addressof(arr), capacity
    for k in ("offsets", "scores", "precision", "recall", "best_f1", "best_index", "at_confidence"):
        setattr(pr, k, None if null.get(k) else one)
    pr._keep = arr
    return pr


def test_entry_points_validate_then_need_a_device(lib):
    cfg = engine.map_config(3, [0.5, 0.75], "coco", views=(_lib.MAP_VIEW_CORNER, _lib.MAP_VIEW_S))
    one = ctypes.c_void_p(8)

    def single(c=cfg, n=4, pr="ok", ap=one):
        p = _pr_struct() if pr == "ok" else pr
        return lib.mgd_map_compute_pr(ctypes.byref(c), one, n, one, ap, one, one,
                                      ctypes.byref(p) if p is not None else None, 0, None, 0)

    def merged(c=cfg, n=4, rank=0, owner=one, pr="ok", ap=one):
        p = _pr_struct() if pr == "ok" else pr
        return lib.mgd_map_compute_merged_pr(ctypes.byref(c), one, n, one, owner, rank, ap, one, one,
                                             ctypes.byref(p) if p is not None else None, 0, None, 0)

    for field, bad in (("num_thresholds", 0), ("num_classes", 0), ("method", 7), ("views", 0)):
        c = engine.map_config(3, [0.5, 0.75])
        setattr(c, field, bad)
        assert single(c) == _lib.ERR_INVALID_ARGUMENT, field
        assert merged(c) == _lib.ERR_INVALID_ARGUMENT, field
    bad_pr = [None,
              _pr_struct(views=0),
              _pr_struct(views=1 << _lib.MAP_VIEW_S),                      # a band view has no curve
              _pr_struct(views=1 << _lib.MAP_VIEW_CENTRE),                 # not matched by cfg
              _pr_struct(views=(1 << _lib.MAP_VIEW_CORNER) | (1 << _lib.MAP_VIEW_CENTRE)),
              _pr_struct(conf=[0.5] * 33),
              _pr_struct(conf=[0.5, float("nan")]),
              _pr_struct(conf=[float("inf")]),
              _pr_struct(conf=[-float("inf")]),
              _pr_struct(capacity=3),                                      # below the 4 records
              _pr_struct(offsets=True), _pr_struct(scores=True), _pr_struct(precision=True),
              _pr_struct(recall=True), _pr_struct(best_f1=True), _pr_struct(best_index=True),
              _pr_struct(at_confidence=True)]
    neg = _pr_struct()
    neg.num_confidences = -1
    nulls = _pr_struct()
    nulls.confidences = None
    bad_pr += [neg, nulls]
    for i, p in enumerate(bad_pr):
        assert single(pr=p) == _lib.ERR_INVALID_ARGUMENT, i
        assert merged(pr=p) == _lib.ERR_INVALID_ARGUMENT, i
    for kw in (dict(n=-1), dict(ap=None)):
        assert single(**kw) == _lib.ERR_INVALID_ARGUMENT, kw
    for kw in (dict(n=-1), dict(rank=-1), dict(owner=None), dict(ap=None)):
        assert merged(**kw) == _lib.ERR_INVALID_ARGUMENT, kw
    ok = [_pr_struct(conf=()), _pr_struct(conf=(), at_confidence=True),    # no confidences: no table
          _pr_struct(capacity=9), _pr_struct(conf=[0.5] * 32)]
    empty = _pr_struct(capacity=0, scores=True, precision=True, recall=True)
    if lib.mgd_device_count() == 0:
        for p in ok:
            assert single(pr=p) == _lib.ERR_NO_DEVICE
            assert merged(pr=p) == _lib.ERR_NO_DEVICE
        assert single(n=0, pr=empty) == _lib.ERR_NO_DEVICE                 # no records: no curve memory
        assert merged(n=0, pr=empty) == _lib.ERR_NO_DEVICE
        with pytest.raises(_lib.MgdError, match="no CPU fallback"):
            _lib.raise_for_status(single())


def test_pr_struct_layout_matches_c(tmp_path):
    src = tmp_path / "layout.c"
    fields = [f for f, _ in _lib.MapPr._fields_]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mgd.h"\n'
                   'int main(void){printf("%zu' + ' %zu' * len(fields) + '\\n", sizeof(mgd_map_pr)' +
                   "".join(f", offsetof(mgd_map_pr, {f})" for f in fields) + ");return 0;}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    assert got == [ctypes.sizeof(_lib.MapPr)] + [getattr(_lib.MapPr, f).offset for f in fields]


def test_python_wrappers_validate_before_any_device_work():
    import torch
    cfg = engine.map_config(3, [0.5], views=(_lib.MAP_VIEW_CORNER, _lib.MAP_VIEW_M))
    gt = torch.zeros((_lib.MAP_VIEWS, 3), dtype=torch.int64)
    owner = torch.zeros(3, dtype=torch.int32)
    for views, conf in (([], None), ([_lib.MAP_VIEW_M], None), ([_lib.MAP_VIEW_CENTRE], None),
                        ([_lib.MAP_VIEW_CORNER], [0.1] * 33), ([_lib.MAP_VIEW_CORNER], [0.1, float("nan")])):
        with pytest.raises(ValueError):
            engine.map_compute_pr(cfg, None, 0, gt, views, conf)
    with pytest.raises(ValueError, match="gt_hist"):
        engine.map_compute_merged_pr(cfg, None, 0, gt, owner, 0, [_lib.MAP_VIEW_CORNER])


def _filter_padded(args, q):
    """The padded tensors with only the detections of score >= q, in slot order."""
    db, ds, dc, dn = args[:4]
    B, M = ds.shape
    fb, fs, fc = np.zeros_like(db), np.zeros_like(ds), np.full_like(dc, -1)
    fn = np.zeros_like(dn)
    for b in range(B):
        keep = [i for i in range(int(dn[b])) if ds[b, i] >= q]
        fn[b] = len(keep)
        fb[b, :len(keep)], fs[b, :len(keep)], fc[b, :len(keep)] = db[b, keep], ds[b, keep], dc[b, keep]
    return (fb, fs, fc, fn) + tuple(args[4:])


def _oracle_curves(args, thresholds, cached):
    """{(class, t): (scores, precision, recall)} of the oracle's matcher and precision_recall,
    the detections listed image by image in slot order like the reference's dicts."""
    db, ds, dc, dn, gtb, gtc, gtn = args
    tp, _ = MO.match_batch(db, ds, dc, dn, gtb, gtc, gtn, thresholds, cached)
    B = len(dn)
    ftp = np.concatenate([tp[:, b, :dn[b]] for b in range(B)], 1)
    fs = np.concatenate([ds[b, :dn[b]] for b in range(B)])
    fc = np.concatenate([dc[b, :dn[b]] for b in range(B)])
    gcl = np.concatenate([gtc[b, :gtn[b]] for b in range(B)])
    out = {}
    for c in np.unique(fc):
        sel = fc == c
        order = np.argsort(fs[sel], kind="stable")[::-1]
        for t in range(len(thresholds)):
            p, r = MO.precision_recall(ftp[t][sel][order], int(np.sum(gcl == c)))
            out[(int(c), t)] = (fs[sel][order], p, r)
    return out


def test_oracle_at_confidence_equals_filtering_and_evaluating_again():
    args = synth_eval_set(53, 24, 30, 10, 4, ties=True)          # scores on a 0.01 grid: many ties
    thr = [0.5, 0.75]
    for cached in (True, False):
        full = _oracle_curves(args, thr, cached)
        inside = 0
        for (c, t), (s, p, r) in full.items():
            vals, counts = np.unique(s, return_counts=True)
            qs = [-1.0, 2.0, float(s.min()), float(s.max())] + [float(v) for v in vals[counts > 1][:6]]
            for q in qs:
                inside += bool(np.sum(s == q) > 1 and np.any(s > q))
                filt = _oracle_curves(_filter_padded(args, q), thr, cached).get((c, t))
                want = (0.0, 0.0, 0.0) if filt is None else (filt[1][-1], filt[2][-1], f1_score(filt[1][-1], filt[2][-1]))
                assert at_confidence(s, p, r, q) == want, (cached, c, t, q)
        assert inside > 10                                      # cuts inside runs of equal scores were tried


def test_oracle_best_f1_takes_run_ends_only():
    # scores 0.9, 0.8, 0.8, 0.7; TP, TP, FP, FP; 2 ground truths: the mid-run record k = 1 has
    # F1 = 1, but no threshold stops there; the run's end k = 2 (F1 0.8) is the best point
    s = np.array([0.9, 0.8, 0.8, 0.7])
    p, r = MO.precision_recall(np.array([1, 1, 0, 0]), 2)
    f1 = [f1_score(a, b) for a, b in zip(p, r)]
    assert int(np.argmax(f1)) == 1
    point, k = best_f1(s, p, r)
    assert k == 2 and point == (0.8, p[2], r[2], f1[2])
    assert at_confidence(s, p, r, 0.8) == (p[2], r[2], f1[2])
    # the first maximum in descending-score order
    tie_s = np.array([0.9, 0.8])
    tp, tr = np.array([1.0, 1.0]), np.array([0.5, 0.5])         # equal F1 twice: the first one
    assert best_f1(tie_s, tp, tr)[1] == 0
    # nothing to choose: no detections, or F1 0 everywhere
    assert best_f1(np.array([]), np.array([]), np.array([])) == ((0.0, 0.0, 0.0, 0.0), -1)
    z = MO.precision_recall(np.array([0, 0]), 3)
    assert best_f1(np.array([0.5, 0.4]), *z) == ((0.0, 0.0, 0.0, 0.0), -1)
    # the best run end is the best threshold: no confidence gives a higher F1
    for (c, t), (s, p, r) in _oracle_curves(synth_eval_set(54, 16, 30, 10, 4, ties=True), [0.5], True).items():
        point, k = best_f1(s, p, r)
        sweep = [at_confidence(s, p, r, q)[2] for q in np.unique(s)]
        assert point[3] == max(sweep + [0.0]), (c, t)
        if k >= 0:
            assert (k == len(s) - 1 or s[k + 1] != s[k]) and at_confidence(s, p, r, point[0])[2] == point[3]


# ------------------------------------------------------------------------------ GPU

def _dev(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _accumulator(C, pieces, args, **kw):
    from multigriddet_b200.evaluation import MapAccumulator
    acc = MapAccumulator(C, **kw)
    lo = 0
    for n in pieces:
        acc.update(*_dev(*[a[lo:lo + n] for a in args]))
        lo += n
    assert lo == len(args[3])
    return acc


def _without_pr(res):
    return {k: v for k, v in res.items() if k != "precision_recall"}


def _assert_equal(got, ref, path="result"):
    """== on every value (and the same types), no tolerance."""
    assert type(got) is type(ref) or (isinstance(got, float) and isinstance(ref, float)), (path, type(got), type(ref))
    if isinstance(ref, dict):
        assert set(got) == set(ref), (path, sorted(set(got) ^ set(ref)))
        for k in ref:
            _assert_equal(got[k], ref[k], f"{path}[{k!r}]")
    elif isinstance(ref, np.ndarray):
        assert got.dtype == ref.dtype and np.array_equal(got, ref), path
    elif hasattr(ref, "cpu"):
        assert got.dtype == ref.dtype and got.shape == ref.shape and bool((got.cpu() == ref.cpu()).all()), path
    else:
        assert got == ref, (path, got, ref)


def _segments(pr):
    """{class: (scores, precision (T, k), recall (T, k))} on the host."""
    off = pr["offsets"].cpu().numpy()
    s, p, r = (pr[k].cpu().numpy() for k in ("scores", "precision", "recall"))
    assert off[0] == 0 and np.all(np.diff(off) >= 0) and off[-1] == len(s) == p.shape[1] == r.shape[1]
    return {c: (s[off[c]:off[c + 1]], p[:, off[c]:off[c + 1]], r[:, off[c]:off[c + 1]]) for c in range(len(off) - 1)}


def _check_against_dropin(res, args, C, thr, matcher, confidences=None, brute_q=(), **kw):
    """Every class's curve at every threshold equals the drop-in host functions; the curves' APs
    equal the drop-in calculate_map's per-class APs (``kw``: its keyword arguments); the operating
    points equal the rules restated above."""
    from multigriddet_b200.evaluation import metrics as G
    pr = res["precision_recall"]
    assert pr["matcher"] == matcher
    match = G.match_predictions_to_gt_cached if matcher == "corner" else G.match_predictions_to_gt
    preds, gts = MO.to_dicts(*args)
    ref = G.calculate_map(preds, gts, C, iou_thresholds=thr, **kw)
    seg = _segments(pr)
    T = len(thr)
    assert pr["best_f1"].shape == (C, T, 4) and pr["best_index"].shape == (C, T)
    checked_ap = 0
    for c in range(C):
        pc = [p for p in preds if p["class"] == c]
        gc = [g for g in gts if g["class"] == c]
        assert pr["num_gt"][c] == len(gc)
        s, P, R = seg[c]
        assert len(s) == len(pc), c
        for t, th in enumerate(thr):
            if pc:
                tp, fp, sc = match(pc, gc, th)
                p, r = G.compute_precision_recall(tp, fp, len(gc))
                assert np.array_equal(s, sc) and np.array_equal(P[t], p) and np.array_equal(R[t], r), (c, t)
                if gc:
                    want = ref["per_class"][f"class_{c}"][f"AP{th:.2f}"]
                    assert G.compute_average_precision(P[t], R[t]) == want, (c, t)
                    checked_ap += 1
            point, k = best_f1(s, P[t], R[t])
            assert tuple(pr["best_f1"][c, t]) == point and pr["best_index"][c, t] == k, (c, t)
            if confidences is not None:
                for q, conf in enumerate(confidences):
                    assert tuple(pr["at_confidence"][c, t, q]) == at_confidence(s, P[t], R[t], conf), (c, t, q)
            for q in brute_q:                                # filter the dicts and run the drop-in again
                keep = [x for x in pc if x["score"] >= confidences[q]]
                if keep:
                    tp, fp, _ = match(keep, gc, th)
                    p, r = G.compute_precision_recall(tp, fp, len(gc))
                    want = (p[-1], r[-1], f1_score(p[-1], r[-1]))
                else:
                    want = (0.0, 0.0, 0.0)
                assert tuple(pr["at_confidence"][c, t, q]) == want, (c, t, q)
    return checked_ap


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["a", "b", "ties"])
def test_gpu_curves_equal_dropin_on_golden_cases(name):
    z = np.load(GOLD)
    db, ds, dc, dn, gtb, gtc, gtn, C = _case(z, name)
    args = (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
    thr = [float(t) for t in z["thresholds"]]
    confs = sorted(set(CONFS + [float(v) for v in np.unique(ds[ds > 0])[:8]]))[:32]
    checked = 0
    for cached in (True, False):
        acc = _accumulator(C, [len(dn)], args, use_parallel=False, cache_ious=cached)
        plain = acc.compute()
        res = acc.compute(precision_recall=True, confidences=confs)
        _assert_equal(_without_pr(res), plain)
        checked += _check_against_dropin(res, args, C, thr, "corner" if cached else "centre", confs,
                                         brute_q=range(len(confs)) if name == "ties" else (),
                                         use_parallel=False, cache_ious=cached)
    assert checked > 0


def _at_size_inputs():
    B, M, N, C = 2000, 100, 20, 80
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(43, B, M, N, C)
    ds = np.round(ds, 2)                                    # ties across images are common
    ds[1::97, 3] = -0.0
    ds[2::89, 5] = 0.0
    return (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn), C


@pytest.mark.gpu
@pytest.mark.parametrize("kw,matcher", [(dict(use_parallel=False), "corner"), (dict(cache_ious=False), "centre"),
                                        (dict(), "centre")])          # defaults: > 10 000 predictions
def test_gpu_curves_equal_dropin_at_size(kw, matcher):
    args, C = _at_size_inputs()
    acc = _accumulator(C, [256] * 7 + [208], args, **kw)
    plain = acc.compute()
    res = acc.compute(precision_recall=True, confidences=CONFS)
    assert res["num_predictions"] > 10000
    _assert_equal(_without_pr(res), plain, str(kw))
    assert _check_against_dropin(res, args, C, [0.5, 0.55, 0.6, 0.65, 0.7, 0.75, 0.8, 0.85, 0.9, 0.95],
                                 matcher, CONFS, **kw) > 700


@pytest.mark.gpu
def test_gpu_curves_are_invariant_to_how_the_images_are_split():
    args = synth_eval_set(41, 40, 30, 20, 6, ties=True)
    args = (args[0].astype(np.int32),) + args[1:]
    for kw in (dict(), dict(cache_ious=False), dict(method="voc", use_parallel=False)):
        whole = _accumulator(6, [40], args, **kw).compute(precision_recall=True, confidences=CONFS)
        split = _accumulator(6, [1, 7, 32], args, **kw).compute(precision_recall=True, confidences=CONFS)
        _assert_equal(split, whole, str(kw))


@pytest.mark.gpu
def test_gpu_best_f1_takes_the_run_end():
    # one image: 0.9 TP, then two detections of score 0.8 (the later one, slot 2, first: TP), 0.7 FP
    db = np.array([[[0, 0, 100, 100], [500, 500, 520, 520], [200, 200, 300, 300], [600, 600, 620, 620]]], np.int32)
    ds = np.array([[0.9, 0.8, 0.8, 0.7]])
    dc = np.zeros((1, 4), np.int32)
    gtb = np.array([[[0, 0, 100, 100], [200, 200, 300, 300]]], np.float64)
    args = (db, ds, dc, np.array([4], np.int32), gtb, np.zeros((1, 2), np.int32), np.array([2], np.int32))
    res = _accumulator(2, [1], args).compute(precision_recall=True, confidences=[0.85, 0.8, 0.75])
    pr = res["precision_recall"]
    s, P, R = _segments(pr)[0]
    assert s.tolist() == [0.9, 0.8, 0.8, 0.7]
    p, r = MO.precision_recall(np.array([1, 1, 0, 0]), 2)
    assert np.array_equal(P[0], p) and np.array_equal(R[0], r)
    assert pr["best_index"][0, 0] == 2 and tuple(pr["best_f1"][0, 0]) == (0.8, p[2], r[2], f1_score(p[2], r[2]))
    assert tuple(pr["at_confidence"][0, 0, 1]) == tuple(pr["best_f1"][0, 0, 1:])
    assert len(_segments(pr)[1][0]) == 0 and pr["best_index"][1, 0] == -1      # class 1: nothing


@pytest.mark.gpu
def test_gpu_curve_edge_cases():
    import torch
    from multigriddet_b200.evaluation import MapAccumulator
    C = 4
    # class 1: ground truth only; class 2: predictions only; class 3: nothing
    gtb = np.array([[[0, 0, 200, 200], [50, 50, 300, 260], [0, 0, 0, 0]]], np.float64)
    gtc = np.array([[0, 1, 0]], np.int32)
    db = np.array([[[0, 0, 201, 199], [10, 10, 20, 20], [50, 50, 300, 250], [0, 0, 150, 150]]], np.int32)
    ds = np.array([[0.9, 0.8, 0.8, 0.3]])
    dc = np.array([[0, 0, 2, 2]], np.int32)
    args = (db, ds, dc, np.array([4], np.int32), gtb, gtc, np.array([2], np.int32))
    empty = (np.zeros((2, 5, 4), np.int32), np.zeros((2, 5)), np.zeros((2, 5), np.int32), np.zeros(2, np.int32),
             np.zeros((2, 3, 4)), np.zeros((2, 3), np.int32), np.zeros(2, np.int32))
    thr = [0.5, 0.75]
    acc = MapAccumulator(C, iou_thresholds=thr)
    for _ in range(2):                                       # nothing at all, then all-padding updates
        res = acc.compute(precision_recall=True, confidences=[0.5])
        pr = res["precision_recall"]
        assert pr["offsets"].cpu().tolist() == [0] * (C + 1)
        assert tuple(pr["scores"].shape) == (0,) and tuple(pr["precision"].shape) == (2, 0)
        assert np.all(pr["best_f1"] == 0) and np.all(pr["best_index"] == -1) and np.all(pr["at_confidence"] == 0)
        acc.update(*_dev(*empty))
    acc.update(*_dev(*args))
    res = acc.compute(precision_recall=True, confidences=[-5.0, 2.0])
    _assert_equal(_without_pr(res), acc.compute())
    _check_against_dropin(res, args, C, thr, "corner", [-5.0, 2.0], brute_q=(0, 1))
    pr = res["precision_recall"]
    seg = _segments(pr)
    assert [len(seg[c][0]) for c in range(C)] == [2, 0, 2, 0]
    assert pr["num_gt"].tolist() == [1, 1, 0, 0]
    assert np.all(pr["best_index"][1:] == -1) and np.all(pr["best_f1"][1:] == 0)   # F1 0 without TP
    assert np.all(pr["at_confidence"][:, :, 1] == 0)                             # above every score
    for c in (0, 2):                                                              # below every score
        assert np.array_equal(pr["at_confidence"][c, :, 0, 0], seg[c][1][:, -1])
    assert set(pr) == {"matcher", "offsets", "scores", "precision", "recall", "num_gt", "best_f1", "best_index",
                       "at_confidence"}
    assert "at_confidence" not in acc.compute(precision_recall=True)["precision_recall"]
    with pytest.raises(ValueError, match="precision_recall"):
        acc.compute(confidences=[0.5])
    with pytest.raises(ValueError):
        acc.compute(precision_recall=True, confidences=[0.5, float("inf")])
    assert isinstance(pr["precision"], torch.Tensor) and pr["precision"].is_cuda and pr["precision"].is_contiguous()


@pytest.mark.gpu
def test_gpu_curves_straight_from_decode_nms():
    import torch
    from multigriddet_b200 import synth
    from multigriddet_b200.evaluation import MapAccumulator
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
    res = acc.compute(precision_recall=True, confidences=CONFS)
    host = [det[k].cpu().numpy() for k in ("boxes_xyxy", "scores", "classes", "counts")]
    assert res["num_predictions"] > 0
    _check_against_dropin(res, (*host, gt_boxes, gt_classes, gt_counts), C,
                          [0.5, 0.55, 0.6, 0.65, 0.7, 0.75, 0.8, 0.85, 0.9, 0.95], "corner", CONFS)


# ------------------------------------------------------------------------------ GPU, sharded

def _free_port():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def _spawn(target, world, *args, timeout=900):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=target, args=(r, world, port, q) + args) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=timeout) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    return dict(res)


def _split(args, sizes):
    out, lo = [], 0
    for n in sizes:
        out.append(tuple(a[lo:lo + n] for a in args))
        lo += n
    assert lo == len(args[3])
    return out


def _reference(C, batches, **kw):
    from multigriddet_b200.evaluation import MapAccumulator
    acc = MapAccumulator(C, **kw)
    for b in batches:
        acc.update(*_dev(*b))
    return acc.compute(precision_recall=True, confidences=CONFS)


def _sharded(C, batches, rank=0, world=1, **kw):
    from multigriddet_b200.evaluation import ShardedMapAccumulator
    from multigriddet_b200.sharding import shard_bounds
    acc = ShardedMapAccumulator(C, **kw)
    for b in batches:
        lo, hi = shard_bounds(len(b[3]), rank, world)
        acc.update(*_dev(*[a[lo:hi] for a in b]), n_total=len(b[3]))
    return acc.compute(precision_recall=True, confidences=CONFS)


def _assert_sharded_equal(got, ref, rank, world, path="result"):
    """The tables and the AP dict equal the single-process ones; the curves of the classes this
    rank owns equal the single-process curves, the others are empty here."""
    gpr, rpr = dict(got["precision_recall"]), ref["precision_recall"]
    owned = gpr.pop("owned")
    C = len(rpr["num_gt"])
    assert owned.tolist() == [c % world == rank for c in range(C)], path
    _assert_equal(_without_pr(got), _without_pr(ref), path)
    for k in ("matcher", "num_gt", "best_f1", "best_index", "at_confidence"):
        _assert_equal(gpr[k], rpr[k], f"{path}[{k}]")
    gs, rs = _segments(gpr), _segments(rpr)
    for c in range(C):
        for a, b in zip(gs[c], rs[c]):
            assert np.array_equal(a, b) if owned[c] else a.size == 0, (path, c)


_KWS = (dict(), dict(use_parallel=False), dict(method="voc", use_parallel=False), dict(cache_ious=False))


@pytest.mark.gpu
def test_gpu_sharded_world_of_one_equals_accumulator():
    z = np.load(GOLD)
    db, ds, dc, dn, gtb, gtc, gtn, C = _case(z, "ties")
    cases = [((db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn), C, [len(dn) // 3, len(dn) - len(dn) // 3])]
    args, C2 = _at_size_inputs()
    cases.append((args, C2, [256] * 7 + [208]))
    for args, C, sizes in cases:
        batches = _split(args, sizes)
        for kw in _KWS:
            got, ref = _sharded(C, batches, **kw), _reference(C, batches, **kw)
            assert got["precision_recall"]["owned"].all()
            _assert_sharded_equal(got, ref, 0, 1, str(kw))


def _crafted_ties():
    """Class 0: one detection of score 0.5 per image in two updates of one image per rank; only
    global image 2 (update 1, rank 0) has ground truth, so the curve depends on ordering equal
    scores later detection first in global image order."""
    C, M, N = 2, 2, 1
    batches = []
    for u in range(2):
        db = np.zeros((2, M, 4), np.int32)
        db[:, 0] = [10, 10, 50, 50]
        db[:, 1] = [100, 100, 300, 300]
        ds = np.array([[0.5, 0.25], [0.5, 0.25]])
        dc = np.array([[0, 1], [0, 1]], np.int32)
        gtb, gtc, gtn = np.zeros((2, N, 4)), np.zeros((2, N), np.int32), np.zeros(2, np.int32)
        if u == 1:
            gtb[0, 0] = [10, 10, 50, 50]
            gtn[0] = 1
        batches.append((db, ds, dc, np.array([2, 2], np.int32), gtb, gtc, gtn))
    return C, batches


def _rank_main(rank, world, port, q):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(0)
    out = {}

    def case(name, C, batches, **kw):
        try:
            _assert_sharded_equal(_sharded(C, batches, rank, world, **kw), _reference(C, batches, **kw), rank, world,
                                  f"{name} {kw}")
            out[name] = "equal"
        except AssertionError as e:
            out[name] = f"differs: {str(e)[:300]}"

    try:
        args = synth_eval_set(47, 31, 40, 12, 7, ties=True)
        args = (args[0].astype(np.int32),) + tuple(args[1:])
        for i, kw in enumerate(_KWS):
            case(f"uneven{i}", 7, _split(args, [31]), **kw)                  # 16 + 15 images
        case("empty_shard", 7, _split(args, [1, 19, 11]))                      # rank 1 holds nothing in update 0
        C, crafted = _crafted_ties()
        case("crafted_ties", C, crafted)
        sizes = [256] * 7 + [208]
        big, C2 = _at_size_inputs()
        case("at_size", C2, _split(big, sizes))
        q.put((rank, out))
    except Exception:                                         # pragma: no cover
        import traceback
        q.put((rank, {"error": traceback.format_exc()[-2000:]}))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_gpu_two_ranks_hold_the_tables_and_their_own_curves():
    res = _spawn(_rank_main, 2)
    for rank in (0, 1):
        got = res[rank]
        assert "error" not in got, (rank, got.get("error"))
        assert all(v == "equal" for v in got.values()), (rank, {k: v for k, v in got.items() if v != "equal"})
        assert len(got) == len(_KWS) + 3, (rank, sorted(got))
