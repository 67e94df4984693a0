"""Detection confusion matrix at chosen confidences (evaluation.ConfusionMatrixAccumulator /
ShardedConfusionMatrixAccumulator, mgd_confusion_update).

CPU: argument validation of the entry point and the Python wrappers before any device work;
known answers of the rule (restated here on top of oracle.metrics_oracle.match_image) on hand-built
images; its invariants on random batches.  GPU: the device matrices equal the restatement's, the
reference matcher's TP counts, plain counts and MapAccumulator's operating points, whatever the
split over updates or ranks (every comparison exact == on int64).
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
CONFS = [-1.0, 0.0, 0.05, 0.3, 0.5, 0.75, 0.9, 0.99, 1.0, 2.0]      # 0.3 / 0.5 / 0.75 sit inside runs of ties
ALL = [float(np.finfo(np.float64).min)]                              # confidences=None


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    return _lib.load()


def _case(z, name):
    return tuple(z[f"{name}_{k}"] for k in ("db", "ds", "dc", "dn", "gtb", "gtc", "gtn")) + (int(z[f"{name}_C"]),)


# ------------------------------------------------------------------------------ the rule, restated
# A restatement of the rule on top of the oracle's matcher; every other test compares against it.
def confusion_image(det_boxes, det_scores, det_classes, gt_boxes, gt_classes, num_classes, iou_threshold,
                    confidences, cached=True, pairs=None):
    """Detection confusion matrices of one image, (Q, C+1, C+1) int64: rows true class, columns
    detected class, index C background.  For each confidence q, over the detections with
    ``score >= confidences[q]``:

    1. stage 1 is ``oracle.metrics_oracle.match_image`` (the reference's matcher) on those detections; each pair adds
       1 to ``[c, c]``;
    2. stage 2: the detections stage 1 left unmatched, in the same visiting order, each claim the
       still-unclaimed ground truth of any class with the highest IoU (``match_image``'s IoU;
       equal IoU: lowest index) when that IoU >= threshold; each pair adds 1 to
       ``[gt class, det class]``;
    3. every kept detection still unmatched adds 1 to ``[C, det class]``, every unclaimed ground
       truth 1 to ``[gt class, C]``.

    Stage 1 runs on the filtered detections, as the rule states it.  ``pairs``: a list that gets
    the stage-2 pairs ``(q, detection slot, ground-truth index)``.
    """
    C, n, g = int(num_classes), len(det_scores), len(gt_classes)
    Q = len(confidences)
    out = np.zeros((Q, C + 1, C + 1), np.int64)
    iou = MO.iou_corner if cached else MO.iou_centre
    cache = {}

    def iou_of(d, j):
        if (d, j) not in cache:
            cache[(d, j)] = iou([float(x) for x in det_boxes[d]], [float(x) for x in gt_boxes[j]])
        return cache[(d, j)]

    scores = np.asarray(det_scores, np.float64)
    for q, conf in enumerate(confidences):
        keep = np.flatnonzero(scores >= conf)
        tp, who = MO.match_image(np.asarray(det_boxes)[keep], scores[keep], np.asarray(det_classes)[keep],
                              gt_boxes, gt_classes, [iou_threshold], cached)
        taken = np.zeros(g, bool)
        matched = {}
        for i, d in enumerate(keep):
            if tp[0, i]:
                matched[int(d)] = int(who[0, i])
                taken[who[0, i]] = True
                out[q, det_classes[d], det_classes[d]] += 1
        order = keep[np.argsort(scores[keep], kind="stable")[::-1]]
        for d in order:
            d = int(d)
            if d in matched:
                continue
            best, best_j = 0.0, -1
            for j in range(g):
                if taken[j]:
                    continue
                v = iou_of(d, j)
                if v > best:
                    best, best_j = v, j
            if best_j >= 0 and best >= iou_threshold:
                taken[best_j] = True
                out[q, gt_classes[best_j], det_classes[d]] += 1
                if pairs is not None:
                    pairs.append((q, d, best_j))
            else:
                out[q, C, det_classes[d]] += 1
        for j in range(g):
            if not taken[j]:
                out[q, gt_classes[j], C] += 1
    return out


def confusion_batch(det_boxes, det_scores, det_classes, det_counts, gt_boxes, gt_classes, gt_counts,
                    num_classes, iou_threshold, confidences, cached=True, pairs=None):
    """``confusion_image`` summed over padded batches: det (B, M, ...), gt (B, N, ...).
    ``pairs`` gets ``(q, image, detection slot, ground-truth index)`` of every stage-2 pair."""
    out = np.zeros((len(confidences), num_classes + 1, num_classes + 1), np.int64)
    for b in range(len(det_counts)):
        n, g = int(det_counts[b]), int(gt_counts[b])
        got = [] if pairs is not None else None
        out += confusion_image(det_boxes[b, :n], det_scores[b, :n], det_classes[b, :n], gt_boxes[b, :g],
                               gt_classes[b, :g], num_classes, iou_threshold, confidences, cached, got)
        if pairs is not None:
            pairs += [(q, b, d, j) for q, d, j in got]
    return out


# ------------------------------------------------------------------------------ CPU: validation

def test_entry_point_validates_then_needs_a_device(lib):
    one = ctypes.c_void_p(8)                                # never dereferenced: validation or no device

    def call(batch=2, M=4, N=3, C=5, thr=0.5, mode=_lib.IOU_CORNER, conf=(0.5,), Q=None, matrix=one,
             dets=one, dn=one, gts=one, gn=one, conf_null=False):
        arr = (ctypes.c_double * max(len(conf), 1))(*conf)
        cp = None if conf_null else ctypes.cast(arr, ctypes.POINTER(ctypes.c_double))
        return lib.mgd_confusion_update(dets, dets, dets, dn, batch, M, gts, gts, gn, N, C, thr, mode, cp,
                                        len(conf) if Q is None else Q, matrix, 0, None, 0)

    bad = [dict(batch=-1), dict(M=-1), dict(N=-1), dict(C=0), dict(C=-3),
           dict(thr=0.0), dict(thr=-0.5), dict(thr=1.0000001), dict(thr=float("nan")), dict(thr=float("inf")),
           dict(mode=2), dict(mode=-1),
           dict(conf=()), dict(conf=[0.5] * 33), dict(conf=(0.5,), Q=0), dict(conf=(0.5,), Q=-1),
           dict(conf_null=True), dict(conf=(0.5, float("nan"))), dict(conf=(float("inf"),)),
           dict(conf=(-float("inf"),)),
           dict(matrix=None), dict(dn=None), dict(gn=None), dict(dets=None), dict(gts=None)]
    for kw in bad:
        assert call(**kw) == _lib.ERR_INVALID_ARGUMENT, kw
    for kw in (dict(M=65536), dict(M=30000, N=8 * 1024)):
        assert call(**kw) == _lib.ERR_UNSUPPORTED, kw
    ok = [dict(), dict(thr=1.0), dict(thr=1e-9), dict(mode=_lib.IOU_CENTRE), dict(conf=[0.5] * 32),
          dict(conf=(-np.finfo(np.float64).max,)), dict(batch=0, dn=None, gn=None, dets=None, gts=None),
          dict(M=0, dets=None), dict(N=0, gts=None)]
    if lib.mgd_device_count() == 0:
        for kw in ok:
            assert call(**kw) == _lib.ERR_NO_DEVICE, kw
        with pytest.raises(_lib.MgdError, match="no CPU fallback"):
            _lib.raise_for_status(call())


def test_python_wrappers_validate_before_any_device_work():
    import torch
    from multigriddet_b200.evaluation import ConfusionMatrixAccumulator, ShardedConfusionMatrixAccumulator
    for kw in (dict(num_classes=0), dict(num_classes=2.5), dict(iou_threshold=0.0), dict(iou_threshold=1.5),
               dict(iou_threshold=float("nan")), dict(iou_mode="xyxy"), dict(confidences=[]),
               dict(confidences=[0.1] * 33), dict(confidences=[0.5, float("nan")]), dict(confidences=[float("inf")])):
        args = dict(num_classes=3, **kw) if "num_classes" not in kw else kw
        for cls in (ConfusionMatrixAccumulator, ShardedConfusionMatrixAccumulator):
            with pytest.raises(ValueError):
                cls(**args, device="cpu")
        with pytest.raises(ValueError):
            engine.confusion_config(**args)
    C, B, M, N = 3, 2, 4, 3
    good = dict(det_boxes=torch.zeros(B, M, 4, dtype=torch.int32), det_scores=torch.zeros(B, M),
                det_classes=torch.zeros(B, M, dtype=torch.int32), det_counts=torch.zeros(B, dtype=torch.int32),
                gt_boxes=torch.zeros(B, N, 4), gt_classes=torch.zeros(B, N, dtype=torch.int32),
                gt_counts=torch.zeros(B, dtype=torch.int32))
    mat = torch.zeros((2, C + 1, C + 1), dtype=torch.int64)

    def upd(matrix=mat, conf=(0.1, 0.5), thr=0.5, mode="corner", **over):
        t = dict(good, **over)
        engine.confusion_update(matrix, conf, thr, mode, *t.values())

    for over, match in ((dict(det_boxes=torch.zeros(B, M, 5)), "detections"),
                        (dict(det_scores=torch.zeros(B, M + 1)), "detections"),
                        (dict(det_counts=torch.zeros(B + 1, dtype=torch.int32)), "detections"),
                        (dict(gt_boxes=torch.zeros(B, N)), "ground truth"),
                        (dict(gt_counts=torch.zeros(B - 1, dtype=torch.int32)), "ground truth"),
                        (dict(gt_classes=np.zeros((B, N), np.int32)), "torch tensor"),
                        (dict(matrix=torch.zeros((2, C + 1, C), dtype=torch.int64)), "matrix"),
                        (dict(matrix=torch.zeros((1, C + 1, C + 1), dtype=torch.int64)), "confidences"),
                        (dict(thr=0.0), "iou_threshold"), (dict(conf=(0.1, float("nan"))), "finite"),
                        (dict(mode="x"), "iou_mode"),
                        (dict(), "CUDA")):                      # everything right but on the host
        with pytest.raises(ValueError, match=match):
            upd(**over)


# ------------------------------------------------------------------------------ CPU: the rule, known answers

def _img(dets, gts):
    """One image from [(box, score, class)] and [(box, class)]."""
    db = np.array([d[0] for d in dets], np.float64).reshape(-1, 4)
    ds = np.array([d[1] for d in dets], np.float64)
    dc = np.array([d[2] for d in dets], np.int32)
    gb = np.array([g[0] for g in gts], np.float64).reshape(-1, 4)
    gc = np.array([g[1] for g in gts], np.int32)
    return db, ds, dc, gb, gc


def _cells(m):
    """{(row, col): count} of the non-zero cells of one (C+1, C+1) matrix."""
    return {(int(r), int(c)): int(m[r, c]) for r, c in zip(*np.nonzero(m))}


DOG, CAT, BG = 1, 0, 2                                     # C = 2


def test_oracle_dog_labelled_cat_is_one_confusion():
    img = _img([([10, 10, 110, 110], 0.9, CAT)], [([12, 10, 110, 112], DOG)])
    m = confusion_image(*img, 2, 0.5, ALL)
    assert _cells(m[0]) == {(DOG, CAT): 1}                  # not one FP [bg, cat] plus one FN [dog, bg]
    m = confusion_image(*img, 2, 0.5, [0.95])
    assert _cells(m[0]) == {(DOG, BG): 1}                   # filtered out: the dog is missed


def test_oracle_stage_one_claim_frees_the_ground_truth_at_a_higher_confidence():
    # det 0: cat on the cat, 0.4;  det 1: dog on the same cat, 0.9
    img = _img([([0, 0, 100, 100], 0.4, CAT), ([0, 0, 100, 100], 0.9, DOG)], [([0, 0, 100, 100], CAT)])
    m = confusion_image(*img, 2, 0.5, [0.3, 0.5, 0.95])
    assert _cells(m[0]) == {(CAT, CAT): 1, (BG, DOG): 1}    # the cat claimed it in stage 1
    assert _cells(m[1]) == {(CAT, DOG): 1}                  # cat detection dropped: free for stage 2
    assert _cells(m[2]) == {(CAT, BG): 1}                   # nothing kept: a miss


def test_oracle_run_of_equal_scores_straddling_a_confidence():
    # two cats of score 0.5, visited later slot first, and a dog of 0.8 on nothing
    img = _img([([0, 0, 100, 100], 0.5, CAT),               # IoU 1 with the cat, 0.73 with the dog
                ([0, 0, 100, 55], 0.5, CAT),                # IoU 0.55 with the cat, 0.32 with the dog
                ([600, 600, 700, 700], 0.8, DOG)],
               [([0, 0, 100, 100], CAT), ([0, 20, 100, 110], DOG)])
    conf = [0.5, float(np.nextafter(0.5, 1.0)), 0.8]
    m = confusion_image(*img, 2, 0.5, conf)
    # slot 1 claims the cat in stage 1, so slot 0 takes the dog in stage 2; the other order would
    # give [cat, cat], [bg, cat] and [dog, bg]
    assert _cells(m[0]) == {(CAT, CAT): 1, (DOG, CAT): 1, (BG, DOG): 1}
    assert _cells(m[1]) == _cells(m[2]) == {(CAT, BG): 1, (DOG, BG): 1, (BG, DOG): 1}   # the run goes whole


def test_oracle_two_detections_compete_for_one_ground_truth_in_stage_two():
    # both cats on the dog: the higher score claims it though its IoU is lower
    img = _img([([0, 0, 100, 60], 0.9, CAT), ([0, 0, 100, 95], 0.8, CAT)], [([0, 0, 100, 100], DOG)])
    pairs = []
    m = confusion_image(*img, 2, 0.5, ALL, pairs=pairs)
    assert _cells(m[0]) == {(DOG, CAT): 1, (BG, CAT): 1} and pairs == [(0, 0, 0)]
    # equal IoU with two unclaimed ground truths: the lower index
    img = _img([([0, 0, 100, 100], 0.9, CAT)], [([0, 0, 100, 100], DOG), ([0, 0, 100, 100], DOG)])
    pairs = []
    m = confusion_image(*img, 2, 0.5, ALL, pairs=pairs)
    assert _cells(m[0]) == {(DOG, CAT): 1, (DOG, BG): 1} and pairs == [(0, 0, 0)]


def test_oracle_both_iou_modes():
    # corner IoU 64 / 136 < 0.5; read as [x, y, w, h] the same numbers overlap 361 / 523 >= 0.5
    img = _img([([12, 12, 22, 22], 0.9, CAT)], [([10, 10, 20, 20], DOG)])
    assert MO.iou_corner([12, 12, 22, 22], [10, 10, 20, 20]) < 0.5 <= MO.iou_centre([12, 12, 22, 22], [10, 10, 20, 20])
    assert _cells(confusion_image(*img, 2, 0.5, ALL, cached=True)[0]) == {(DOG, BG): 1, (BG, CAT): 1}
    assert _cells(confusion_image(*img, 2, 0.5, ALL, cached=False)[0]) == {(DOG, CAT): 1}
    # stage 1 follows the same switch
    img = _img([([12, 12, 22, 22], 0.9, DOG)], [([10, 10, 20, 20], DOG)])
    assert _cells(confusion_image(*img, 2, 0.5, ALL, cached=True)[0]) == {(DOG, BG): 1, (BG, DOG): 1}
    assert _cells(confusion_image(*img, 2, 0.5, ALL, cached=False)[0]) == {(DOG, DOG): 1}


def _perturbed(seed, B, M, N, C, ties=True, p=0.3):
    """synth_eval_set with a share p of the detection labels redrawn, so that confusions occur."""
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(seed, B, M, N, C, ties=ties)
    rng = np.random.default_rng(seed + 1000)
    flip = rng.random(dc.shape) < p
    dc = np.where(flip, rng.integers(0, C, dc.shape), dc).astype(np.int32)
    return db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn


def _check_invariants(m, args, C, thr, confidences, cached, tp=None):
    """Diagonal = the reference matcher's TP count at each confidence; row g < C sums to the
    ground truth of g; column d < C to the kept class-d detections; [C, C] = 0."""
    db, ds, dc, dn, gtb, gtc, gtn = args
    if tp is None:
        tp = MO.match_batch(db, ds, dc, dn, gtb, gtc, gtn, [thr], cached)[0][0]
    real = np.arange(ds.shape[1])[None, :] < dn[:, None]
    greal = np.arange(gtc.shape[1])[None, :] < gtn[:, None]
    n_gt = np.bincount(gtc[greal], minlength=C)
    for q, conf in enumerate(confidences):
        kept = real & (ds >= conf)
        assert np.array_equal(np.diag(m[q])[:C], np.bincount(dc[kept & (tp == 1)], minlength=C)), q
        assert np.array_equal(m[q, :C].sum(1), n_gt), q
        assert np.array_equal(m[q, :, :C].sum(0), np.bincount(dc[kept], minlength=C)), q
        assert m[q, C, C] == 0 and m.dtype == np.int64


def test_oracle_invariants_on_random_batches():
    C = 6
    confs = CONFS[:3] + [0.35, 0.5, 0.51, 0.9]
    args = _perturbed(61, 24, 30, 12, C)
    for cached in (True, False):
        for thr in (0.3, 0.5, 0.9):
            pairs = []
            m = confusion_batch(*args, C, thr, confs, cached, pairs=pairs)
            _check_invariants(m, args, C, thr, confs, cached)
            assert len(pairs) > 0
            for q, b, d, j in pairs:                       # stage 2 is always cross-class
                assert args[2][b, d] != args[5][b, j]
            off = sum(int(m[q, :C, :C].sum() - np.trace(m[q][:C, :C])) for q in range(len(confs)))
            assert off == len(pairs)


# ------------------------------------------------------------------------------ GPU

def _dev(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _acc(C, pieces, args, **kw):
    from multigriddet_b200.evaluation import ConfusionMatrixAccumulator
    acc = ConfusionMatrixAccumulator(C, **kw)
    lo = 0
    for n in pieces:
        acc.update(*_dev(*[a[lo:lo + n] for a in args]))
        lo += n
    assert lo == len(args[3])
    return acc


def _eq(got, want, what=""):
    assert got.dtype == np.int64 and want.dtype == np.int64 and got.shape == want.shape, what
    assert np.array_equal(got, want), (what, np.argwhere(got != want)[:8])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["a", "b", "ties"])
def test_gpu_equals_oracle_on_golden_cases(name):
    z = np.load(GOLD)
    db, ds, dc, dn, gtb, gtc, gtn, C = _case(z, name)
    args = (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
    confs = sorted(set(CONFS + [float(v) for v in np.unique(ds[ds > 0])[:8]]))[:32]
    nonzero_off = 0
    for mode in ("corner", "centre"):
        for thr in (0.5, 0.75):
            got = _acc(C, [len(dn)], args, iou_threshold=thr, confidences=confs, iou_mode=mode).compute()
            want = confusion_batch(*args, C, thr, confs, cached=mode == "corner")
            _eq(got, want, (mode, thr))
            nonzero_off += int(got[:, :C, :C].sum() - np.trace(got[:, :C, :C], axis1=1, axis2=2).sum())
            _eq(_acc(C, [len(dn)], args, iou_threshold=thr, iou_mode=mode).compute(),
                confusion_batch(*args, C, thr, ALL, cached=mode == "corner"), (mode, thr, "all"))
    assert nonzero_off > 0 or name == "ties"                # ties: 2 classes, no cross-class overlap >= thr


@pytest.mark.gpu
def test_gpu_equals_oracle_on_random_data():
    C = 80
    args = _perturbed(71, 256, 100, 20, C)
    confs = [0.0, 0.3, 0.5, 0.75, 0.95]
    for mode in ("corner", "centre"):
        got = _acc(C, [100, 156], args, confidences=confs, iou_mode=mode).compute()
        want = confusion_batch(*args, C, 0.5, confs, cached=mode == "corner")
        _eq(got, want, mode)
        assert (got[:, :C, :C].sum() - np.trace(got[:, :C, :C], axis1=1, axis2=2).sum()) > 100


@pytest.mark.gpu
def test_gpu_at_size_against_matcher_and_counts():
    C = 80
    args = _perturbed(73, 2000, 100, 20, C)
    confs = CONFS + [0.25, 0.55]
    for mode, cached in (("corner", True), ("centre", False)):
        got = _acc(C, [256] * 7 + [208], args, confidences=confs, iou_mode=mode).compute()
        tp = engine.match_detections(*_dev(*args), [0.5], iou_mode=mode)[0].cpu().numpy()
        _check_invariants(got, args, C, 0.5, confs, cached, tp=tp)


@pytest.mark.gpu
def test_gpu_independent_of_the_split_over_updates():
    C = 7
    args = _perturbed(75, 40, 30, 12, C)
    for mode in ("corner", "centre"):
        whole = _acc(C, [40], args, confidences=CONFS, iou_mode=mode).compute()
        split = _acc(C, [1, 0, 7, 32], args, confidences=CONFS, iou_mode=mode).compute()
        _eq(split, whole, mode)
        acc = _acc(C, [40], args, confidences=CONFS, iou_mode=mode)
        acc.reset()
        assert not acc.compute().any()
        acc.update(*_dev(*args))
        _eq(acc.compute(), whole, mode)


@pytest.mark.gpu
def test_gpu_straight_from_decode_nms():
    import torch
    from multigriddet_b200 import synth
    from multigriddet_b200.evaluation import ConfusionMatrixAccumulator
    S, C, B, N = 416, 20, 24, 40
    anchors = synth.coco_anchors(np.float32)
    boxes = synth.synth_boxes(44, B, N, S, C)
    y = engine.encode_targets(torch.from_numpy(boxes).cuda(), (S, S), anchors, C)
    preds = synth.planted_head_outputs(y, 3, seed=44)
    det = engine.decode_nms(preds, None, (S, S), anchors, C, max_boxes=100, confidence=0.05,
                            nms_threshold=0.45, nms_method="diou")
    assert det["boxes_xyxy"].dtype == torch.int32
    gt_counts = ((boxes[..., 2] - boxes[..., 0]) * (boxes[..., 3] - boxes[..., 1]) > 0).sum(1).astype(np.int32)
    gt_boxes, gt_classes = boxes[..., :4].astype(np.float64), boxes[..., 4].astype(np.int32)
    acc = ConfusionMatrixAccumulator(C, confidences=CONFS)
    acc.update(det["boxes_xyxy"], det["scores"], det["classes"], det["counts"], *_dev(gt_boxes, gt_classes, gt_counts))
    got = acc.compute()
    host = [det[k].cpu().numpy() for k in ("boxes_xyxy", "scores", "classes", "counts")]
    assert (host[2] == -1).any() and host[3].sum() > 0              # -1 padding classes are there
    _eq(got, confusion_batch(*host, gt_boxes, gt_classes, gt_counts, C, 0.5, CONFS), "decode_nms")
    assert got[CONFS.index(0.0)].sum() > 0


@pytest.mark.gpu
def test_gpu_class_out_of_range_raises_and_padding_is_ignored():
    C = 5
    args = list(_perturbed(77, 12, 20, 8, C))
    want = confusion_batch(*args, C, 0.5, CONFS)
    # whatever the padding slots hold, nothing changes
    db, ds, dc, dn, gtb, gtc, gtn = (a.copy() for a in args)
    for b in range(len(dn)):
        dc[b, dn[b]:] = [-7, 99, C][b % 3]
        ds[b, dn[b]:] = [np.nan, np.inf, 5.0][b % 3]
        db[b, dn[b]:] = -123
        gtc[b, gtn[b]:] = [C, -1, 1000][b % 3]
        gtb[b, gtn[b]:] = np.nan
    padded = (db, ds, dc, dn, gtb, gtc, gtn)
    _eq(_acc(C, [5, 7], padded, confidences=CONFS).compute(), want, "padding")
    # a real slot out of range: AssertionError at compute, for a detection and for a ground truth
    for which, value in (("det", C), ("det", -1), ("gt", C + 3), ("gt", -2)):
        bad = [a.copy() for a in args]
        b = int(np.flatnonzero((args[3] > 0) & (args[6] > 0))[0])
        if which == "det":
            bad[2][b, 0] = value
        else:
            bad[5][b, 0] = value
        acc = _acc(C, [12], bad, confidences=CONFS)
        with pytest.raises(AssertionError, match="confusion update: class id outside"):
            acc.compute()
        m = acc.compute()                                   # reported once; the other cells are counted
        assert m.shape == (len(CONFS), C + 1, C + 1)


@pytest.mark.gpu
def test_gpu_diagonal_equals_map_accumulator_operating_points():
    from multigriddet_b200.evaluation import MapAccumulator
    C = 80
    args = _perturbed(79, 500, 100, 20, C)
    confs = CONFS + [0.45]
    for mode, kw in (("corner", dict(use_parallel=False)), ("centre", dict(cache_ious=False))):
        mp = MapAccumulator(C, iou_thresholds=[0.5], compute_per_scale=False, **kw)
        for lo in (0, 250):
            mp.update(*_dev(*[a[lo:lo + 250] for a in args]))
        pr = mp.compute(precision_recall=True, confidences=confs)["precision_recall"]
        assert pr["matcher"] == mode
        m = _acc(C, [250, 250], args, confidences=confs, iou_mode=mode).compute()
        rec = pr["at_confidence"][:, 0, :, 1]                               # (C, Q)
        want = np.rint(rec * (pr["num_gt"][:, None] + 1e-8)).astype(np.int64).T
        _eq(np.stack([np.diag(m[q])[:C] for q in range(len(confs))]), want, mode)


# ------------------------------------------------------------------------------ GPU, sharded

@pytest.mark.gpu
def test_gpu_sharded_world_of_one_equals_single():
    from multigriddet_b200.evaluation import ShardedConfusionMatrixAccumulator
    C = 80
    args = _perturbed(81, 300, 100, 20, C)
    for mode in ("corner", "centre"):
        ref = _acc(C, [300], args, confidences=CONFS, iou_mode=mode).compute()
        sh = ShardedConfusionMatrixAccumulator(C, confidences=CONFS, iou_mode=mode)
        for lo in (0, 100):
            sh.update(*_dev(*[a[lo:lo + [100, 200][lo > 0]] for a in args]))
        _eq(sh.compute(), ref, mode)


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
    from multigriddet_b200.evaluation import ShardedConfusionMatrixAccumulator
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(0)
    out = {}
    C = 9
    args = _perturbed(83, 31, 40, 12, C)
    try:
        for name, splits in (("uneven", [(0, 16), (16, 31)]),            # 16 + 15 images
                             ("empty", [(0, 0), (0, 31)])):              # rank 0 holds nothing
            for mode in ("corner", "centre"):
                lo, hi = splits[rank]
                acc = ShardedConfusionMatrixAccumulator(C, confidences=CONFS, iou_mode=mode)
                for a, b in ((lo, lo + (hi - lo) // 2), (lo + (hi - lo) // 2, hi)):
                    acc.update(*_dev(*[x[a:b] for x in args]))
                got = acc.compute()
                want = confusion_batch(*args, C, 0.5, CONFS, cached=mode == "corner")
                out[f"{name}_{mode}"] = "equal" if np.array_equal(got, want) and got.dtype == np.int64 else "differs"
        acc = ShardedConfusionMatrixAccumulator(C)
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
def test_gpu_two_ranks_sum_to_the_single_matrix():
    res = _spawn(_rank_main, 2)
    for rank in (0, 1):
        got = res[rank]
        assert "error" not in got, (rank, got.get("error"))
        assert got == {"uneven_corner": "equal", "uneven_centre": "equal", "empty_corner": "equal",
                       "empty_centre": "equal", "class_error": "raised"}, (rank, got)
