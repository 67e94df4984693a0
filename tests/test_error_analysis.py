"""TIDE-style detection error analysis (evaluation.ErrorAnalysisAccumulator /
ShardedErrorAnalysisAccumulator, mgd_tide_update).

CPU: argument validation of the entry point and the Python wrappers before any device work; known
answers of the rule (restated here on top of oracle.metrics_oracle's matcher and AP arithmetic) on
hand-built images; its invariants on random batches with heavy score ties.  GPU: the device's error
counts, fixed ground-truth counts and fixed records equal the restatement's (exact ==), the fixed APs
equal it to rel 1e-12, the base APs equal MapAccumulator's, whatever the split over updates or ranks.
"""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest

from multigriddet_b200 import _lib, engine
from oracle import metrics_oracle as MO
from oracle.gen_golden import synth_eval_set

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(os.path.dirname(__file__), "golden", "metrics_cases.npz")
F = 9                                                       # base + 8 fixes
BASE, FCLS, FLOC, FBOTH, FDUPE, FBKG, FMISS, FFP, FFN = range(F)
CLS, LOC, BOTH, DUPE, BKG, MISS = range(6)
TP = -1
FIXES = ("Cls", "Loc", "Both", "Dupe", "Bkg", "Miss", "FP", "FN")
ERRORS = ("Cls", "Loc", "Both", "Dupe", "Bkg", "Miss")
REC = np.dtype([("score", "<f8"), ("cls", "<i4"), ("band", "<i4"), ("bits", "<u4", (5,)), ("pad", "<u4")])


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    return _lib.load()


def _case(z, name):
    return tuple(z[f"{name}_{k}"] for k in ("db", "ds", "dc", "dn", "gtb", "gtc", "gtn")) + (int(z[f"{name}_C"]),)


# ------------------------------------------------------------------------------ the rule, restated
# A restatement of the rule on top of the oracle's matcher; every other test compares against it.
def tide_image(det_boxes, det_scores, det_classes, gt_boxes, gt_classes, num_classes, t_f=0.5, t_b=0.1,
               cached=True):
    """One image.  Returns ``kind`` (n,) (TP = -1, else the error type), ``target`` (n,) (-1: none),
    ``claimed`` (g,) and ``miss`` (g,) bools, and the fixed sets' ``cls`` / ``tp`` (F, n) (class -1:
    dropped).

    1. base: ``oracle.metrics_oracle.match_image`` at t_f;
    2. each unmatched d: s / o = its largest IoU (``match_image``'s IoU) with the ground truth of its
       own / of the other classes, claimed or not, target the first index attaining it; the first of
       Bkg max(s, o) < t_b, Cls o >= t_f (target: o's), Dupe s >= t_f, Loc s >= t_b (target: s's), Both;
    3. Miss: unclaimed by the base and no Cls / Loc error's target;
    4. fixes, each alone: Cls (Loc) errors in visiting order (score descending, equal scores later slot
       first) claim their target with the target's (their own) class when neither the base nor an
       earlier error of the same fix holds it, else are dropped; Both / Dupe / Bkg and FP drop.
    """
    det_classes, gt_classes = np.asarray(det_classes), np.asarray(gt_classes)
    n, g = len(det_scores), len(gt_classes)
    iou = MO.iou_corner if cached else MO.iou_centre
    tp, who = MO.match_image(det_boxes, det_scores, det_classes, gt_boxes, gt_classes, [t_f], cached)
    claimed = np.zeros(g, bool)
    claimed[who[0][who[0] >= 0]] = True
    kind, target = np.full(n, TP), np.full(n, -1)
    for d in range(n):
        if tp[0, d]:
            continue
        s, sj, o, oj = 0.0, -1, 0.0, -1
        for j in range(g):
            v = iou([float(x) for x in det_boxes[d]], [float(x) for x in gt_boxes[j]])
            if gt_classes[j] == det_classes[d]:
                if v > s:
                    s, sj = v, j
            elif v > o:
                o, oj = v, j
        if max(s, o) < t_b:
            kind[d] = BKG
        elif o >= t_f:
            kind[d], target[d] = CLS, oj
        elif s >= t_f:
            kind[d] = DUPE
        elif s >= t_b:
            kind[d], target[d] = LOC, sj
        else:
            kind[d] = BOTH
    named = np.zeros(g, bool)
    named[target[target >= 0]] = True
    miss = ~claimed & ~named
    cls = np.tile(det_classes.astype(np.int64), (F, 1))
    flag = np.tile(tp[0].astype(np.int64), (F, 1))
    held = {FCLS: claimed.copy(), FLOC: claimed.copy()}
    for d in np.argsort(np.asarray(det_scores), kind="stable")[::-1]:
        k = kind[d]
        if k in (CLS, LOC):
            f = FCLS if k == CLS else FLOC
            t = target[d]
            if held[f][t]:
                cls[f, d] = -1
            else:
                held[f][t] = True
                cls[f, d], flag[f, d] = (gt_classes[t] if k == CLS else det_classes[d]), 1
        elif k in (BOTH, DUPE, BKG):
            cls[{BOTH: FBOTH, DUPE: FDUPE, BKG: FBKG}[k], d] = -1
        if k != TP:
            cls[FFP, d] = -1
    return kind, target, claimed, miss, cls, flag


def tide_batch(det_boxes, det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts, num_classes,
               t_f=0.5, t_b=0.1, cached=True):
    """``tide_image`` over padded batches: the records' ``cls`` / ``tp`` (B, F, M) (padding: class -1),
    the sets' ground-truth counts (F, C) and the error counts (C, 6)."""
    B, M = det_scores.shape
    C = num_classes
    cls = np.full((B, F, M), -1, np.int64)
    flag = np.zeros((B, F, M), np.int64)
    gt = np.zeros((F, C), np.int64)
    counts = np.zeros((C, 6), np.int64)
    for b in range(B):
        n, g = int(det_counts[b]), int(gt_counts[b])
        kind, _, claimed, miss, c, t = tide_image(det_boxes[b, :n], det_scores[b, :n], det_classes[b, :n],
                                                  gt_boxes[b, :g], gt_classes[b, :g], C, t_f, t_b, cached)
        cls[b, :, :n], flag[b, :, :n] = c, t
        for d in range(n):
            if kind[d] != TP:
                counts[det_classes[b, d], kind[d]] += 1
        gc = gt_classes[b, :g]
        total = np.bincount(gc, minlength=C)
        gt += total
        gt[FMISS] -= np.bincount(gc[miss], minlength=C)
        gt[FFN] -= np.bincount(gc[~claimed], minlength=C)
        counts[:, MISS] += np.bincount(gc[miss], minlength=C)
    flag[cls < 0] = 0
    return cls, flag, gt, counts


def tide_aps(cls, flag, det_scores, gt, num_classes, method="coco"):
    """(F, C) AP of every fixed set with ``calculate_map``'s per-class arithmetic; the records of a
    class in image-then-slot order, sorted like ``np.argsort(kind='stable')[::-1]``."""
    C = num_classes
    ap = np.zeros((F, C))
    for f in range(F):
        fc, ft = cls[:, f, :].reshape(-1), flag[:, f, :].reshape(-1)
        fs = np.asarray(det_scores, np.float64).reshape(-1)
        for c in range(C):
            sel = fc == c
            n_pred, n_gt = int(sel.sum()), int(gt[f, c])
            if n_pred == 0:
                ap[f, c] = 0.0 if n_gt > 0 else 1.0
            elif n_gt == 0:
                ap[f, c] = 0.0
            else:
                order = np.argsort(fs[sel], kind="stable")[::-1]
                ap[f, c] = MO.average_precision(*MO.precision_recall(ft[sel][order], n_gt), method)
    return ap


def tide_result(cls, flag, det_scores, gt, counts, num_classes, method="coco"):
    """The ``compute()`` dict of the restatement."""
    C = num_classes
    ap = tide_aps(cls, flag, det_scores, gt, C, method)
    active = np.flatnonzero(((cls[:, BASE, :, None] == np.arange(C)).any((0, 1))) | (gt[BASE] > 0))
    mean = lambda row: float(np.mean(row[active])) if len(active) else 0.0
    base = mean(ap[BASE])
    return {"AP": base, "dAP": {k: mean(ap[f + 1]) - base for f, k in enumerate(FIXES)},
            "counts": {k: int(counts[:, e].sum()) for e, k in enumerate(ERRORS)},
            "per_class": {"AP": ap[BASE], "dAP": (ap[1:] - ap[BASE]).T, "counts": counts}}


# ------------------------------------------------------------------------------ CPU: validation

def test_entry_point_validates_then_needs_a_device(lib):
    one = ctypes.c_void_p(8)                                # never dereferenced: validation or no device

    def call(batch=2, M=4, N=3, C=5, t_f=0.5, t_b=0.1, mode=_lib.IOU_CORNER, off=0, recs=one, hist=one, counts=one,
             dets=one, dn=one, gts=one, gn=one):
        return lib.mgd_tide_update(dets, dets, dets, dn, batch, M, gts, gts, gn, N, C, t_f, t_b, mode, off, recs,
                                   hist, counts, 0, None, 0)

    bad = [dict(batch=-1), dict(M=-1), dict(N=-1), dict(off=-1), dict(C=0), dict(C=-3),
           dict(t_f=0.0), dict(t_f=-0.5), dict(t_f=1.0000001), dict(t_f=float("nan")), dict(t_f=float("inf")),
           dict(t_b=0.0), dict(t_b=-0.1), dict(t_b=0.6), dict(t_f=0.3, t_b=0.5), dict(t_b=float("nan")),
           dict(mode=2), dict(mode=-1),
           dict(recs=None), dict(hist=None), dict(counts=None), dict(dn=None), dict(gn=None), dict(dets=None),
           dict(gts=None)]
    for kw in bad:
        assert call(**kw) == _lib.ERR_INVALID_ARGUMENT, kw
    for kw in (dict(M=65536), dict(M=30000, N=8 * 1024), dict(N=131072), dict(C=2 ** 28),
               dict(batch=2 ** 20, M=1000), dict(off=2 ** 31 - 10)):
        assert call(**kw) == _lib.ERR_UNSUPPORTED, kw
    ok = [dict(), dict(t_f=1.0, t_b=1.0), dict(t_f=0.5, t_b=0.5), dict(t_b=1e-9), dict(mode=_lib.IOU_CENTRE),
          dict(batch=0, dn=None, gn=None, dets=None, gts=None, recs=None, hist=None, counts=None),
          dict(M=0, dets=None, recs=None), dict(N=0, gts=None)]
    if lib.mgd_device_count() == 0:
        for kw in ok:
            assert call(**kw) == _lib.ERR_NO_DEVICE, kw
        with pytest.raises(_lib.MgdError, match="no CPU fallback"):
            _lib.raise_for_status(call())


def test_python_wrappers_validate_before_any_device_work():
    import torch
    from multigriddet_b200.evaluation import ErrorAnalysisAccumulator, ShardedErrorAnalysisAccumulator
    for kw in (dict(num_classes=0), dict(num_classes=2.5), dict(num_classes=True), dict(pos_threshold=0.0),
               dict(pos_threshold=1.5), dict(pos_threshold=float("nan")), dict(background_threshold=0.0),
               dict(background_threshold=0.6), dict(pos_threshold=0.3, background_threshold=0.4),
               dict(background_threshold=float("nan")), dict(iou_mode="xyxy"), dict(method="coco101")):
        args = dict(num_classes=3, **kw) if "num_classes" not in kw else kw
        for cls in (ErrorAnalysisAccumulator, ShardedErrorAnalysisAccumulator):
            with pytest.raises(ValueError):
                cls(**args, device="cpu")
        if "method" not in kw:
            with pytest.raises(ValueError):
                engine.tide_config(**args)
    C, B, M, N = 3, 2, 4, 3
    good = dict(det_boxes=torch.zeros(B, M, 4, dtype=torch.int32), det_scores=torch.zeros(B, M),
                det_classes=torch.zeros(B, M, dtype=torch.int32), det_counts=torch.zeros(B, dtype=torch.int32),
                gt_boxes=torch.zeros(B, N, 4), gt_classes=torch.zeros(B, N, dtype=torch.int32),
                gt_counts=torch.zeros(B, dtype=torch.int32))
    recs = torch.zeros(F * B * M * 40, dtype=torch.uint8)
    hist = torch.zeros((_lib.MAP_VIEWS, F * C), dtype=torch.int64)
    counts = torch.zeros((C, 6), dtype=torch.int64)

    def upd(records=recs, offset=0, gt_hist=hist, cnt=counts, t_f=0.5, t_b=0.1, mode="corner", **over):
        t = dict(good, **over)
        engine.tide_update(records, offset, gt_hist, cnt, t_f, t_b, mode, *t.values())

    for over, match in ((dict(det_boxes=torch.zeros(B, M, 5)), "detections"),
                        (dict(det_scores=torch.zeros(B, M + 1)), "detections"),
                        (dict(det_counts=torch.zeros(B + 1, dtype=torch.int32)), "detections"),
                        (dict(gt_boxes=torch.zeros(B, N)), "ground truth"),
                        (dict(gt_counts=torch.zeros(B - 1, dtype=torch.int32)), "ground truth"),
                        (dict(gt_classes=np.zeros((B, N), np.int32)), "torch tensor"),
                        (dict(cnt=torch.zeros((C, 5), dtype=torch.int64)), "counts"),
                        (dict(cnt=np.zeros((C, 6), np.int64)), "counts"),
                        (dict(t_f=0.0), "pos_threshold"), (dict(t_b=0.7), "background_threshold"),
                        (dict(mode="x"), "iou_mode"),
                        (dict(), "CUDA")):                      # everything right but on the host
        with pytest.raises(ValueError, match=match):
            upd(**over)
    if torch.cuda.is_available():
        dev = lambda t: t.cuda()
        for over, match in ((dict(gt_hist=dev(torch.zeros((_lib.MAP_VIEWS, C), dtype=torch.int64))), "gt_hist"),
                            (dict(records=dev(recs[:-1])), "records"), (dict(offset=-1), "records")):
            with pytest.raises(ValueError, match=match):
                upd(**dict(dict(records=dev(recs), gt_hist=dev(hist), cnt=dev(counts)), **over),
                    **{k: dev(v) for k, v in good.items()})


# ------------------------------------------------------------------------------ CPU: the rule, known answers

def _img(dets, gts):
    """One image from [(box, score, class)] and [(box, class)]."""
    db = np.array([d[0] for d in dets], np.float64).reshape(-1, 4)
    ds = np.array([d[1] for d in dets], np.float64)
    dc = np.array([d[2] for d in dets], np.int32)
    gb = np.array([g[0] for g in gts], np.float64).reshape(-1, 4)
    gc = np.array([g[1] for g in gts], np.int32)
    return db, ds, dc, gb, gc


def _batch(*images):
    """A padded batch from ``_img`` tuples."""
    B = len(images)
    M = max(max(len(im[1]) for im in images), 1)
    N = max(max(len(im[4]) for im in images), 1)
    db, ds, dc = np.zeros((B, M, 4)), np.zeros((B, M)), np.full((B, M), -1, np.int32)
    gb, gc = np.zeros((B, N, 4)), np.full((B, N), -1, np.int32)
    dn, gn = np.zeros(B, np.int32), np.zeros(B, np.int32)
    for b, (a, s, c, g, k) in enumerate(images):
        dn[b], gn[b] = len(s), len(k)
        db[b, :len(s)], ds[b, :len(s)], dc[b, :len(s)] = a, s, c
        gb[b, :len(k)], gc[b, :len(k)] = g, k
    return db, ds, dc, dn, gb, gc, gn


CAT, DOG = 0, 1                                             # C = 2
BOX = [0, 0, 100, 100]


def test_oracle_each_of_the_six_types():
    img = _img([(BOX, 0.9, CAT),                           # TP on the cat
                (BOX, 0.8, CAT),                           # Dupe: IoU 1 with the claimed cat
                ([0, 0, 100, 70], 0.7, DOG),               # Cls: IoU 0.7 with the cat, no dog overlaps
                ([300, 300, 400, 340], 0.6, DOG),          # Loc: IoU 0.4 with the dog
                ([300, 0, 400, 30], 0.5, CAT),             # Both: IoU 0.3 with the (other-class) mouse
                ([900, 900, 950, 950], 0.4, DOG)],         # Bkg: nothing
               [(BOX, CAT), ([300, 300, 400, 400], DOG), ([300, 0, 400, 100], 2),
                ([600, 600, 700, 700], DOG)])              # missed dog
    kind, target, claimed, miss, cls, flag = tide_image(*img, 3)
    assert kind.tolist() == [TP, DUPE, CLS, LOC, BOTH, BKG]
    assert target.tolist() == [-1, -1, 0, 1, -1, -1]
    assert claimed.tolist() == [True, False, False, False] and miss.tolist() == [False, False, True, True]
    # the Cls fix turns det 2 into a TP cat... on a claimed cat: dropped; the Loc fix claims the dog
    assert cls[FCLS].tolist() == [CAT, CAT, -1, DOG, CAT, DOG] and flag[FCLS, 2] == 0
    assert cls[FLOC].tolist() == [CAT, CAT, DOG, DOG, CAT, DOG] and flag[FLOC].tolist() == [1, 0, 0, 1, 0, 0]
    for f, d in ((FBOTH, 4), (FDUPE, 1), (FBKG, 5)):
        want = [CAT, CAT, DOG, DOG, CAT, DOG]
        want[d] = -1
        assert cls[f].tolist() == want
    assert cls[FFP].tolist() == [CAT, -1, -1, -1, -1, -1]
    for f in (BASE, FMISS, FFN):
        assert cls[f].tolist() == [CAT, CAT, DOG, DOG, CAT, DOG] and flag[f].tolist() == [1, 0, 0, 0, 0, 0]
    _, _, gt, counts = tide_batch(*_batch(img), 3)
    assert gt[BASE].tolist() == [1, 2, 1] and gt[FMISS].tolist() == [1, 1, 0] and gt[FFN].tolist() == [1, 0, 0]
    assert counts.tolist() == [[0, 0, 1, 1, 0, 0], [1, 1, 0, 0, 1, 1], [0, 0, 0, 0, 0, 1]]


def test_oracle_cls_and_loc_errors_racing_for_one_ground_truth():
    # a cat box and a dog box on one unclaimed dog: the cat is a Cls error, the dog a Loc error,
    # with the same target; each fix is applied alone, so each claims it in its own fix
    img = _img([([0, 0, 100, 60], 0.9, CAT), ([0, 0, 100, 40], 0.8, DOG)], [(BOX, DOG)])
    kind, target, claimed, miss, cls, flag = tide_image(*img, 2)
    assert kind.tolist() == [CLS, LOC] and target.tolist() == [0, 0] and not miss.any()
    assert cls[FCLS].tolist() == [DOG, DOG] and flag[FCLS].tolist() == [1, 0]
    assert cls[FLOC].tolist() == [CAT, DOG] and flag[FLOC].tolist() == [0, 1]
    # two Cls errors on one dog: the higher score claims it, the other is dropped
    img = _img([([0, 0, 100, 60], 0.5, CAT), ([0, 0, 100, 90], 0.5, CAT)], [(BOX, DOG)])
    kind, target, _, _, cls, flag = tide_image(*img, 2)
    assert kind.tolist() == [CLS, CLS] and cls[FCLS].tolist() == [-1, DOG]     # equal scores: later slot first
    args = _batch(img)
    cls, flag, gt, counts = tide_batch(*args, 2)
    res = tide_result(cls, flag, args[1], gt, counts, 2)
    # base: cats without ground truth and a dog without detections, AP 0 each; fixed: the cat class
    # is left with neither (1.0) and the dog found (1.0)
    assert res["AP"] == 0.0 and res["dAP"]["Cls"] == pytest.approx(1.0, abs=1e-6)


def test_oracle_cls_fix_whose_target_is_claimed_and_claimed_loc_target():
    # the dog box lies on a cat that the cat box claimed: Cls error, dropped by its fix
    img = _img([(BOX, 0.9, CAT), ([0, 0, 100, 80], 0.8, DOG), ([0, 0, 100, 30], 0.7, CAT)], [(BOX, CAT)])
    kind, target, claimed, miss, cls, flag = tide_image(*img, 2)
    assert kind.tolist() == [TP, CLS, LOC] and target.tolist() == [-1, 0, 0]
    assert cls[FCLS].tolist() == [CAT, -1, CAT] and flag[FCLS].tolist() == [1, 0, 0]
    # the Loc error's target is claimed by the base: it stays Loc, and its fix drops it
    assert cls[FLOC].tolist() == [CAT, DOG, -1] and not miss.any()


def test_oracle_equal_iou_to_two_targets_takes_the_lowest_index():
    img = _img([(BOX, 0.9, CAT)], [(BOX, DOG), (BOX, DOG), ([0, 0, 100, 30], CAT)])
    kind, target, _, miss, cls, flag = tide_image(*img, 2)
    assert kind.tolist() == [CLS] and target.tolist() == [0] and miss.tolist() == [False, True, True]
    img = _img([([0, 0, 100, 40], 0.9, CAT)], [(BOX, CAT), (BOX, CAT)])
    kind, target, _, miss, _, _ = tide_image(*img, 2)
    assert kind.tolist() == [LOC] and target.tolist() == [0] and miss.tolist() == [False, True]


def test_oracle_fn_fix_empties_a_class_and_a_class_without_ground_truth():
    # every dog missed; a mouse detection (class 2) without any mouse in the data
    img = _img([(BOX, 0.9, CAT), ([500, 500, 600, 600], 0.8, 2)], [(BOX, CAT), ([300, 300, 400, 400], DOG)])
    args = _batch(img)
    cls, flag, gt, counts = tide_batch(*args, 3)
    assert gt[FFN].tolist() == [1, 0, 0] and gt[FMISS].tolist() == [1, 0, 0] and counts[DOG, MISS] == 1
    res = tide_result(cls, flag, args[1], gt, counts, 3)
    ap = tide_aps(cls, flag, args[1], gt, 3)
    assert ap[BASE].tolist() == [pytest.approx(1.0, abs=1e-6), 0.0, 0.0]      # no dog detection, no mouse gt
    assert ap[FFN, DOG] == 1.0 and ap[FMISS, DOG] == 1.0                      # no detections, no ground truth
    assert ap[FFP, 2] == 1.0 and ap[FBKG, 2] == 1.0                           # its only detection dropped
    assert res["dAP"]["FN"] == pytest.approx(1.0 / 3) and res["dAP"]["FP"] == pytest.approx(1.0 / 3)
    assert res["counts"] == {"Cls": 0, "Loc": 0, "Both": 0, "Dupe": 0, "Bkg": 1, "Miss": 1}


def test_oracle_iou_mode_switch():
    # corner IoU 64 / 136 < 0.5; read as [x, y, w, h] the same numbers overlap 361 / 523 >= 0.5
    img = _img([([12, 12, 22, 22], 0.9, CAT)], [([10, 10, 20, 20], DOG)])
    assert tide_image(*img, 2, cached=True)[0].tolist() == [BOTH]
    assert tide_image(*img, 2, cached=False)[0].tolist() == [CLS]


def _perturbed(seed, B, M, N, C, ties=True, p=0.3):
    """synth_eval_set with a share p of the detection labels redrawn, so that every type occurs."""
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(seed, B, M, N, C, ties=ties)
    rng = np.random.default_rng(seed + 1000)
    flip = rng.random(dc.shape) < p
    dc = np.where(flip, rng.integers(0, C, dc.shape), dc).astype(np.int32)
    return db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn


def _check_invariants(args, C, t_f, t_b, cached):
    db, ds, dc, dn, gtb, gtc, gtn = args
    cls, flag, gt, counts = tide_batch(*args, C, t_f, t_b, cached)
    tp = MO.match_batch(*args, [t_f], cached)[0][0]
    real = np.arange(ds.shape[1])[None, :] < dn[:, None]
    assert int(tp[real].sum()) + int(counts[:, :MISS].sum()) == int(real.sum())
    named = 0
    for b in range(len(dn)):
        n, g = int(dn[b]), int(gtn[b])
        kind, target, claimed, miss, c, t = tide_image(db[b, :n], ds[b, :n], dc[b, :n], gtb[b, :g], gtc[b, :g],
                                                       C, t_f, t_b, cached)
        assert np.array_equal(kind == TP, tp[b, :n] == 1)
        unclaimed_named = np.zeros(g, bool)
        unclaimed_named[target[target >= 0]] = True
        unclaimed_named &= ~claimed
        assert int(claimed.sum() + miss.sum() + unclaimed_named.sum()) == g
        named += int(unclaimed_named.sum())
        # each fix changes only the records it is about
        touched = {FCLS: kind == CLS, FLOC: kind == LOC, FBOTH: kind == BOTH, FDUPE: kind == DUPE,
                   FBKG: kind == BKG, FMISS: np.zeros(n, bool), FFP: kind != TP, FFN: np.zeros(n, bool)}
        for f, m in touched.items():
            same = (c[f] == c[BASE]) & (t[f] == t[BASE])
            assert same[~m].all(), f
    n_gt = np.bincount(np.concatenate([gtc[b, :gtn[b]] for b in range(len(gtn))]), minlength=C)
    for f in (BASE, FCLS, FLOC, FBOTH, FDUPE, FBKG, FFP):
        assert np.array_equal(gt[f], n_gt)
    assert np.array_equal(n_gt - gt[FMISS], counts[:, MISS])
    assert int(gt[FFN].sum()) + int(counts[:, MISS].sum()) + named == int(n_gt.sum())
    assert int(gt[FFN].sum()) == int(tp[real].sum())
    return counts


def test_oracle_invariants_on_random_batches():
    C = 6
    args = _perturbed(91, 24, 30, 12, C)
    seen = np.zeros(6, np.int64)
    for cached in (True, False):
        for t_f, t_b in ((0.5, 0.1), (0.3, 0.3), (0.9, 0.05)):
            seen += _check_invariants(args, C, t_f, t_b, cached).sum(0)
    assert (seen > 0).all()                                 # every type occurs


# ------------------------------------------------------------------------------ GPU

def _dev(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _acc(C, pieces, args, **kw):
    from multigriddet_b200.evaluation import ErrorAnalysisAccumulator
    acc = ErrorAnalysisAccumulator(C, **kw)
    lo = 0
    for n in pieces:
        acc.update(*_dev(*[a[lo:lo + n] for a in args]))
        lo += n
    assert lo == len(args[3])
    return acc


def _device_state(acc):
    """The accumulator's records (B, F, M) class / tp, fixed ground-truth counts (F, C), counts."""
    recs = np.frombuffer(acc._records[:acc._slots * 40].cpu().numpy().tobytes(), dtype=REC)
    C = acc.num_classes
    gt = acc._gt_hist.cpu().numpy()
    assert not np.delete(gt, _lib.MAP_VIEW_CORNER, 0).any()
    return recs, gt[_lib.MAP_VIEW_CORNER].reshape(F, C), acc._counts.cpu().numpy()


def _check_against_restatement(acc, args, C, t_f=0.5, t_b=0.1, cached=True, method="coco"):
    cls, flag, gt, counts = tide_batch(*args, C, t_f, t_b, cached)
    recs, dgt, dcounts = _device_state(acc)
    B, M = args[1].shape
    recs = recs.reshape(B, F, M)
    want_cls = np.where(cls >= 0, cls + np.arange(F)[None, :, None] * C, -1)
    assert np.array_equal(recs["cls"], want_cls), np.argwhere(recs["cls"] != want_cls)[:8]
    assert np.array_equal(recs["bits"][..., _lib.MAP_VIEW_CORNER], flag)
    assert not np.delete(recs["bits"], _lib.MAP_VIEW_CORNER, -1).any()
    assert np.array_equal(recs["score"], np.broadcast_to(args[1][:, None, :], (B, F, M)))
    assert dgt.dtype == np.int64 and np.array_equal(dgt, gt)
    assert dcounts.dtype == np.int64 and np.array_equal(dcounts, counts)
    got = acc.compute()
    want = tide_result(cls, flag, args[1], gt, counts, C, method)
    _assert_result(got, want)
    return got


def _assert_result(got, want):
    assert got["AP"] == pytest.approx(want["AP"], rel=1e-12, abs=1e-15)
    assert set(got["dAP"]) == set(FIXES) and set(got["counts"]) == set(ERRORS)
    for k in FIXES:
        assert got["dAP"][k] == pytest.approx(want["dAP"][k], rel=1e-12, abs=1e-14), k
    assert got["counts"] == want["counts"]
    pc = got["per_class"]
    assert pc["AP"].dtype == np.float64 and pc["dAP"].dtype == np.float64 and pc["counts"].dtype == np.int64
    np.testing.assert_allclose(pc["AP"], want["per_class"]["AP"], rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(pc["dAP"], want["per_class"]["dAP"], rtol=1e-12, atol=1e-14)
    assert np.array_equal(pc["counts"], want["per_class"]["counts"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["a", "b", "ties"])
def test_gpu_equals_restatement_on_golden_cases(name):
    z = np.load(GOLD)
    db, ds, dc, dn, gtb, gtc, gtn, C = _case(z, name)
    args = (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
    for mode in ("corner", "centre"):
        for t_f, t_b, method in ((0.5, 0.1, "coco"), (0.75, 0.3, "coco"), (0.5, 0.1, "voc")):
            acc = _acc(C, [len(dn)], args, pos_threshold=t_f, background_threshold=t_b, iou_mode=mode, method=method)
            _check_against_restatement(acc, args, C, t_f, t_b, mode == "corner", method)


@pytest.mark.gpu
def test_gpu_equals_restatement_on_random_data():
    C = 80
    args = _perturbed(93, 256, 100, 20, C)
    for mode in ("corner", "centre"):
        got = _check_against_restatement(_acc(C, [100, 156], args, iou_mode=mode), args, C, cached=mode == "corner")
        assert all(v > 0 for v in got["counts"].values()), got["counts"]


@pytest.mark.gpu
def test_gpu_at_size():
    C = 80
    args = _perturbed(95, 2000, 100, 20, C)
    _check_against_restatement(_acc(C, [256] * 7 + [208], args), args, C)


@pytest.mark.gpu
def test_gpu_base_equals_map_accumulator():
    from multigriddet_b200.evaluation import MapAccumulator
    C = 80
    args = _perturbed(97, 500, 100, 20, C)
    for mode, kw in (("corner", dict(use_parallel=False)), ("centre", dict(cache_ious=False))):
        for t_f in (0.5, 0.7):
            mp = MapAccumulator(C, iou_thresholds=[t_f], compute_per_scale=False, **kw)
            for lo in (0, 250):
                mp.update(*_dev(*[a[lo:lo + 250] for a in args]))
            ref = mp.compute()
            got = _acc(C, [250, 250], args, pos_threshold=t_f, iou_mode=mode).compute()
            assert got["AP"] == ref["mAP"], (mode, t_f)
            for c in range(C):
                per = ref["per_class"].get(f"class_{c}")
                if per is not None:
                    assert got["per_class"]["AP"][c] == per[f"AP{t_f:.2f}"], (mode, t_f, c)


@pytest.mark.gpu
def test_gpu_independent_of_the_split_over_updates():
    C = 7
    args = _perturbed(99, 40, 30, 12, C)
    for mode in ("corner", "centre"):
        whole = _acc(C, [40], args, iou_mode=mode).compute()
        _assert_result(_acc(C, [1, 0, 7, 32], args, iou_mode=mode).compute(), whole)
        acc = _acc(C, [40], args, iou_mode=mode)
        acc.reset()
        empty = acc.compute()
        assert empty["AP"] == 0.0 and not any(empty["dAP"].values()) and not any(empty["counts"].values())
        acc.update(*_dev(*args))
        _assert_result(acc.compute(), whole)


@pytest.mark.gpu
def test_gpu_straight_from_decode_nms():
    import torch
    from multigriddet_b200 import synth
    from multigriddet_b200.evaluation import ErrorAnalysisAccumulator
    S, C, B, N = 416, 20, 24, 40
    anchors = synth.coco_anchors(np.float32)
    boxes = synth.synth_boxes(46, B, N, S, C)
    y = engine.encode_targets(torch.from_numpy(boxes).cuda(), (S, S), anchors, C)
    preds = synth.planted_head_outputs(y, 3, seed=46)
    det = engine.decode_nms(preds, None, (S, S), anchors, C, max_boxes=100, confidence=0.05,
                            nms_threshold=0.45, nms_method="diou")
    assert det["boxes_xyxy"].dtype == torch.int32
    gt_counts = ((boxes[..., 2] - boxes[..., 0]) * (boxes[..., 3] - boxes[..., 1]) > 0).sum(1).astype(np.int32)
    gt_boxes, gt_classes = boxes[..., :4].astype(np.float64), boxes[..., 4].astype(np.int32)
    acc = ErrorAnalysisAccumulator(C)
    acc.update(det["boxes_xyxy"], det["scores"], det["classes"], det["counts"], *_dev(gt_boxes, gt_classes, gt_counts))
    host = [det[k].cpu().numpy() for k in ("boxes_xyxy", "scores", "classes", "counts")]
    assert (host[2] == -1).any() and host[3].sum() > 0              # -1 padding classes are there
    got = _check_against_restatement(acc, (*host, gt_boxes, gt_classes, gt_counts), C)
    assert sum(got["counts"].values()) > 0


@pytest.mark.gpu
def test_gpu_class_out_of_range_raises():
    C = 5
    args = list(_perturbed(101, 12, 20, 8, C))
    for which, value in (("det", C), ("det", -1), ("gt", C + 3), ("gt", -2)):
        bad = [a.copy() for a in args]
        b = int(np.flatnonzero((args[3] > 0) & (args[6] > 0))[0])
        if which == "det":
            bad[2][b, 0] = value
        else:
            bad[5][b, 0] = value
        acc = _acc(C, [12], bad)
        with pytest.raises(AssertionError, match="error analysis update: class id outside"):
            acc.compute()


# ------------------------------------------------------------------------------ GPU, sharded

def _same(got, want):
    """Exact equality of two compute() dicts."""
    return (got["AP"] == want["AP"] and got["dAP"] == want["dAP"] and got["counts"] == want["counts"]
            and all(np.array_equal(got["per_class"][k], want["per_class"][k]) for k in ("AP", "dAP", "counts")))


@pytest.mark.gpu
def test_gpu_sharded_world_of_one_equals_single():
    from multigriddet_b200.evaluation import ShardedErrorAnalysisAccumulator
    C = 80
    args = _perturbed(103, 300, 100, 20, C)
    for mode in ("corner", "centre"):
        ref = _acc(C, [300], args, iou_mode=mode).compute()
        sh = ShardedErrorAnalysisAccumulator(C, iou_mode=mode)
        for lo in (0, 100):
            sh.update(*_dev(*[a[lo:lo + [100, 200][lo > 0]] for a in args]))
        assert _same(sh.compute(), ref), mode


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


def _rank_main(rank, world, port, q):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from multigriddet_b200.evaluation import ErrorAnalysisAccumulator, ShardedErrorAnalysisAccumulator
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(0)
    out = {}
    C = 9
    args = _perturbed(105, 32, 40, 12, C)
    try:
        from multigriddet_b200.sharding import shard_bounds
        for mode in ("corner", "centre"):
            for name, batches in (("uneven", [(0, 31)]),                       # 16 + 15 images
                                  ("empty", [(0, 1), (1, 31), (31, 32)])):     # rank 1 holds nothing twice
                single = ErrorAnalysisAccumulator(C, iou_mode=mode)
                acc = ShardedErrorAnalysisAccumulator(C, iou_mode=mode)
                for a, b in batches:
                    single.update(*_dev(*[x[a:b] for x in args]))
                    lo, hi = shard_bounds(b - a, rank, world)
                    acc.update(*_dev(*[x[a + lo:a + hi] for x in args]), n_total=b - a)
                got, want = acc.compute(), single.compute()
                out[f"{name}_{mode}"] = "equal" if _same(got, want) else "differs"
        acc = ShardedErrorAnalysisAccumulator(C)
        bad = [a.copy() for a in args]
        if rank == 1:
            bad[2][:, 0] = C + 1                           # only rank 1 sees an out-of-range class
        acc.update(*_dev(*[x[rank * 15:rank * 15 + 15] for x in bad]))
        try:
            acc.compute()
            out["class_error"] = "no error"
        except AssertionError as e:
            out["class_error"] = "raised" if "class id outside" in str(e) else f"message: {e}"
        q.put((rank, out))
    except Exception:                                         # pragma: no cover
        import traceback
        q.put((rank, {"error": traceback.format_exc()[-2000:]}))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_gpu_two_ranks_equal_the_single_process():
    res = _spawn(_rank_main, 2)
    for rank in (0, 1):
        got = res[rank]
        assert "error" not in got, (rank, got.get("error"))
        assert got == {"uneven_corner": "equal", "uneven_centre": "equal", "empty_corner": "equal",
                       "empty_centre": "equal", "class_error": "raised"}, (rank, got)
