"""COCO-style average recall of the streaming mAP accumulators (MapAccumulator /
ShardedMapAccumulator with ``recall_max_dets``, mgd_map_recall_update).

The rule, restated here as filter-then-match: in each view keep the detections and ground truth of
the view's area band (none for the full-set views), then the first k detections of every (image,
class) in the matcher's visiting order (score descending, equal scores later slot first), match
what is left with the view's matcher and count the true positives.  CPU: argument validation of the
entry point and the wrappers; known answers of the restatement on hand-built images; on random
batches with heavy ties it equals the full walk's TP flags counted by rank, which is what the
kernel counts.  GPU: the device tables and every AR key equal the restatement (exact ==), whatever
the split over updates or ranks, and nothing the dict held before changes.
"""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest

from multigriddet_b200 import _lib, engine
from multigriddet_b200.sharding import shard_bounds
from oracle import metrics_oracle as MO
from oracle.gen_golden import synth_eval_set

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(os.path.dirname(__file__), "golden", "metrics_cases.npz")
COCO = [0.5, 0.55, 0.6, 0.65, 0.7, 0.75, 0.8, 0.85, 0.9, 0.95]
V = _lib.MAP_VIEWS
# view -> (cached matcher, area band or None), as mgd_map_update matches them
VIEW_RULES = {_lib.MAP_VIEW_CORNER: (True, None), _lib.MAP_VIEW_CENTRE: (False, None),
              _lib.MAP_VIEW_S: (False, 0), _lib.MAP_VIEW_M: (False, 1), _lib.MAP_VIEW_L: (False, 2)}
BAND_KEYS = (("ARS", _lib.MAP_VIEW_S), ("ARM", _lib.MAP_VIEW_M), ("ARL", _lib.MAP_VIEW_L))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    return _lib.load()


def _case(z, name):
    db, ds, dc, dn, gtb, gtc, gtn = (z[f"{name}_{k}"] for k in ("db", "ds", "dc", "dn", "gtb", "gtc", "gtn"))
    return (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn), int(z[f"{name}_C"])


# ------------------------------------------------------------------------------ the rule, restated

def area_band(boxes):
    """map_area_band of xyxy boxes: 0 = S, 1 = M, 2 = L, 3 = none (NaN area)."""
    b = np.asarray(boxes, np.float64)
    a = (b[..., 2] - b[..., 0]) * (b[..., 3] - b[..., 1])
    return np.select([a < 1024.0, (a >= 1024.0) & (a < 9216.0), a >= 9216.0], [0, 1, 2], 3)


def visit_rank(ds, dc, keep):
    """(B, M) rank of each slot among the ``keep`` slots of its image and class in the matcher's
    visiting order: score descending, equal scores later slot first."""
    M = ds.shape[1]
    si, sj = ds[:, :, None], ds[:, None, :]
    later = np.arange(M)[None, None, :] > np.arange(M)[None, :, None]
    ahead = keep[:, None, :] & (dc[:, :, None] == dc[:, None, :]) & ((sj > si) | ((sj == si) & later))
    return ahead.sum(2)


def compact(keep, *arrays):
    """The ``keep`` slots of every image moved to the front in slot order, and their counts."""
    order = np.argsort(~keep, axis=1, kind="stable")
    out = [np.take_along_axis(a, order if a.ndim == 2 else order[..., None], axis=1) for a in arrays]
    return out, keep.sum(1).astype(np.int32)


def oracle_match(db, ds, dc, dn, gtb, gtc, gtn, thresholds, cached):
    """(T, B, M) TP flags of the reference's matcher (oracle.metrics_oracle)."""
    return MO.match_batch(db, ds, dc, dn, gtb, gtc, gtn, thresholds, cached)[0]


def device_match(db, ds, dc, dn, gtb, gtc, gtn, thresholds, cached):
    """The same flags from mgd_match_detections (held to the oracle by the mAP tests)."""
    return engine.match_detections(np.asarray(db, np.float64), ds, dc, dn, gtb, gtc, gtn, thresholds,
                                   iou_mode="corner" if cached else "centre")


def _view_inputs(args, v):
    db, ds, dc, dn, gtb, gtc, gtn = args
    B, M = ds.shape
    N = gtc.shape[1]
    band = VIEW_RULES[v][1]
    dmask = np.arange(M)[None] < dn[:, None]
    gmask = np.arange(N)[None] < gtn[:, None]
    if band is not None:
        dmask, gmask = dmask & (area_band(db) == band), gmask & (area_band(gtb) == band)
    return dmask, compact(gmask, gtb, gtc)


def restated_tp(args, C, thresholds, limits, views, match=oracle_match):
    """Filter-then-match: ``tp (MAP_VIEWS, C, T, K)`` true positives among the first limits[k]
    detections of every (image, class), and ``gt (MAP_VIEWS, C)``, for each view in ``views``."""
    db, ds, dc = args[:3]
    M = ds.shape[1]
    tp = np.zeros((V, C, len(thresholds), len(limits)), np.int64)
    gt = np.zeros((V, C), np.int64)
    for v in views:
        dmask, ((gb, gc), gn) = _view_inputs(args, v)
        gt[v] = np.bincount(gc[np.arange(gc.shape[1])[None] < gn[:, None]], minlength=C)
        rank = visit_rank(ds, dc, dmask)
        for k, lim in enumerate(limits):
            (b, s, c), n = compact(dmask & (rank < lim), db, ds, dc)
            flags = match(b, s, c, n, gb, gc, gn, thresholds, VIEW_RULES[v][0])
            kept = np.arange(M)[None] < n[:, None]
            for t in range(len(thresholds)):
                tp[v, :, t, k] = np.bincount(c[kept & (flags[t] == 1)], minlength=C)
    return tp, gt


def ranked_tp(args, C, thresholds, limits, views, match=oracle_match):
    """The full walk's TP flags in each view, counted when the detection's rank is < limits[k]."""
    db, ds, dc = args[:3]
    M = ds.shape[1]
    tp = np.zeros((V, C, len(thresholds), len(limits)), np.int64)
    for v in views:
        dmask, ((gb, gc), gn) = _view_inputs(args, v)
        (b, s, c), n = compact(dmask, db, ds, dc)
        flags = match(b, s, c, n, gb, gc, gn, thresholds, VIEW_RULES[v][0])
        kept = np.arange(M)[None] < n[:, None]
        rank = visit_rank(s, c, kept)
        for k, lim in enumerate(limits):
            for t in range(len(thresholds)):
                tp[v, :, t, k] = np.bincount(c[kept & (flags[t] == 1) & (rank < lim)], minlength=C)
    return tp


def ar_keys(tp, gt, view, limits, per_scale=True):
    """The AR keys and the "recall" entry compute() should give for these counts."""
    rec = np.where(gt[:, :, None, None] > 0, tp / np.maximum(gt, 1)[:, :, None, None], -1.0)

    def mean(v, k):
        has = gt[v] > 0
        return float(np.mean(rec[v][has][:, :, k])) if has.any() else 0.0
    out = {f"AR{m}": mean(view, k) for k, m in enumerate(limits)}
    for key, v in BAND_KEYS:
        out[key] = mean(v, len(limits) - 1) if per_scale else 0.0
    out["recall"] = {"max_dets": tuple(limits), "matcher": "corner" if view == _lib.MAP_VIEW_CORNER else "centre",
                     "num_gt": gt[view], "recall": rec[view]}
    return out


def _same(got, want, path="result"):
    """== on every value, arrays and tensors included, with the same types."""
    import torch
    assert type(got) is type(want) or (isinstance(got, float) and isinstance(want, float)), (path, type(got), type(want))
    if isinstance(want, dict):
        assert set(got) == set(want), (path, sorted(set(got) ^ set(want)))
        for k in want:
            _same(got[k], want[k], f"{path}[{k!r}]")
    elif isinstance(want, np.ndarray):
        assert got.dtype == want.dtype and got.shape == want.shape and np.array_equal(got, want), path
    elif isinstance(want, torch.Tensor):
        assert got.dtype == want.dtype and torch.equal(got, want), path
    elif isinstance(want, (tuple, list)):
        assert len(got) == len(want), path
        for i, (a, b) in enumerate(zip(got, want)):
            _same(a, b, f"{path}[{i}]")
    else:
        assert got == want, (path, got, want)


# ------------------------------------------------------------------------------ CPU: validation

def test_entry_point_validates_then_needs_a_device(lib):
    one = ctypes.c_void_p(8)                                # never dereferenced: validation or no device

    def call(cfg_kw=None, records=one, slot_offset=0, batch=2, M=4, limits=(1, 10, 100), K=None, tp=one,
             limits_null=False):
        cfg = engine.map_config(3, [0.5, 0.75])
        for k, v in (cfg_kw or {}).items():
            setattr(cfg, k, v)
        arr = (ctypes.c_int * max(len(limits), 1))(*limits)
        return lib.mgd_map_recall_update(ctypes.byref(cfg), records, slot_offset, batch, M,
                                         None if limits_null else arr, len(limits) if K is None else K, tp,
                                         0, None, 0)

    bad = [dict(cfg_kw=dict(num_classes=0)), dict(cfg_kw=dict(num_thresholds=0)),
           dict(cfg_kw=dict(num_thresholds=33)), dict(cfg_kw=dict(method=2)), dict(cfg_kw=dict(views=0)),
           dict(cfg_kw=dict(views=1 << V)),
           dict(limits=()), dict(limits=tuple(range(1, 10))), dict(limits=(1,), K=0), dict(limits=(1,), K=-1),
           dict(limits_null=True), dict(limits=(0, 10)), dict(limits=(-1,)), dict(limits=(10, 10)),
           dict(limits=(1, 100, 10)),
           dict(batch=-1), dict(M=-1), dict(slot_offset=-1),
           dict(records=None), dict(tp=None)]
    for kw in bad:
        assert call(**kw) == _lib.ERR_INVALID_ARGUMENT, kw
    cfg = engine.map_config(3, [0.5])
    assert lib.mgd_map_recall_update(None, one, 0, 2, 4, (ctypes.c_int * 1)(1), 1, one, 0, None, 0) \
        == _lib.ERR_INVALID_ARGUMENT
    for kw in (dict(M=65536, batch=1), dict(slot_offset=(1 << 31) - 4, batch=1, M=4),
               dict(batch=1 << 20, M=4096)):
        assert call(**kw) == _lib.ERR_UNSUPPORTED, kw
    ok = [dict(), dict(limits=(1,)), dict(limits=tuple(range(1, 9))), dict(limits=(5, 1 << 30)),
          dict(slot_offset=(1 << 31) - 9, batch=2, M=4), dict(batch=0, records=None, tp=None),
          dict(M=0, records=None, tp=None)]
    if lib.mgd_device_count() == 0:
        for kw in ok:
            assert call(**kw) == _lib.ERR_NO_DEVICE, kw
        with pytest.raises(_lib.MgdError, match="no CPU fallback"):
            _lib.raise_for_status(call())
    del cfg


def test_python_wrappers_validate_before_any_device_work(lib):
    import torch
    from multigriddet_b200.evaluation import MapAccumulator, ShardedMapAccumulator
    for bad in ([], (0,), (1, 0), (10, 1), (1, 1), tuple(range(1, 10)), (1.5,), (True, 10), 100, "1", (1, None),
                (-5,), (1, 2 ** 31)):
        for cls in (MapAccumulator, ShardedMapAccumulator):
            with pytest.raises(ValueError):
                cls(3, recall_max_dets=bad, device="cpu")
        with pytest.raises(ValueError):
            engine.recall_limits(bad)
    assert engine.recall_limits((1, 10, 100)) == (1, 10, 100)
    assert engine.recall_limits(np.array([1, 5])) == (1, 5)
    cfg = engine.map_config(3, [0.5, 0.75])
    rec = torch.zeros(8 * engine.map_record_bytes(), dtype=torch.uint8)
    for tp in (torch.zeros((V, 3, 2, 3), dtype=torch.int64),      # everything right but on the host
               torch.zeros((V, 3, 2, 2), dtype=torch.int64), torch.zeros((V, 3, 2, 3), dtype=torch.int32)):
        with pytest.raises(ValueError, match="tp must be"):
            engine.map_recall_update(cfg, rec, 0, 2, 4, (1, 10, 100), tp)
    with pytest.raises(ValueError, match="strictly increasing"):
        engine.map_recall_update(cfg, rec, 0, 2, 4, (10, 1), torch.zeros((V, 3, 2, 2), dtype=torch.int64))


# ------------------------------------------------------------------------------ CPU: known answers

def _one(dets, gts):
    """One image, padded batch of 1, from [(box, score, class)] and [(box, class)]."""
    db = np.array([d[0] for d in dets], np.float64).reshape(1, -1, 4)
    ds = np.array([[d[1] for d in dets]], np.float64).reshape(1, -1)
    dc = np.array([[d[2] for d in dets]], np.int32).reshape(1, -1)
    gb = np.array([g[0] for g in gts], np.float64).reshape(1, -1, 4)
    gc = np.array([[g[1] for g in gts]], np.int32).reshape(1, -1)
    return db, ds, dc, np.array([len(dets)], np.int32), gb, gc, np.array([len(gts)], np.int32)


CORNER = _lib.MAP_VIEW_CORNER


def test_oracle_best_detection_ranked_second_lowers_ar1():
    # class 0: the 0.9 detection barely overlaps, the 0.8 one sits on the object
    img = _one([([0, 0, 100, 100], 0.9, 0), ([200, 200, 300, 300], 0.8, 0)], [([205, 200, 300, 305], 0)])
    tp, gt = restated_tp(img, 1, [0.5], (1, 10), [CORNER])
    assert tp[CORNER, 0, 0].tolist() == [0, 1] and gt[CORNER].tolist() == [1]
    ar = ar_keys(tp, gt, CORNER, (1, 10))
    assert ar["AR1"] == 0.0 and ar["AR10"] == 1.0


def test_oracle_run_of_equal_scores_straddling_a_limit():
    # two class-0 detections of score 0.5: the later slot is visited first, so it is the one kept
    # at k = 1 (pycocotools would keep the earlier one and find the object)
    img = _one([([0, 0, 100, 100], 0.5, 0), ([500, 500, 600, 600], 0.5, 0), ([0, 0, 50, 50], 0.2, 0)],
               [([0, 0, 100, 100], 0)])
    tp, gt = restated_tp(img, 1, [0.5, 0.9], (1, 2, 3), [CORNER])
    assert tp[CORNER, 0].tolist() == [[0, 1, 1], [0, 1, 1]]
    swapped = _one([([500, 500, 600, 600], 0.5, 0), ([0, 0, 100, 100], 0.5, 0), ([0, 0, 50, 50], 0.2, 0)],
                   [([0, 0, 100, 100], 0)])
    tp, gt = restated_tp(swapped, 1, [0.5, 0.9], (1, 2, 3), [CORNER])
    assert tp[CORNER, 0].tolist() == [[1, 1, 1], [1, 1, 1]]


def test_oracle_class_without_detections_counts_zero_and_without_ground_truth_is_left_out():
    # class 0 found, class 1 has an object and no detection, class 2 a detection and no object
    img = _one([([0, 0, 100, 100], 0.9, 0), ([300, 300, 400, 400], 0.7, 2)],
               [([0, 0, 100, 100], 0), ([300, 0, 400, 100], 1)])
    tp, gt = restated_tp(img, 3, [0.5, 0.75], (1, 100), [CORNER])
    ar = ar_keys(tp, gt, CORNER, (1, 100))
    rec = ar["recall"]["recall"]
    assert rec[1].tolist() == [[0.0, 0.0], [0.0, 0.0]] and rec[2].tolist() == [[-1.0, -1.0], [-1.0, -1.0]]
    assert ar["AR1"] == ar["AR100"] == 0.5                   # (1 + 0) / 2: class 2 does not enter
    assert ar["ARS"] == ar["ARM"] == ar["ARL"] == 0.0        # no band view restated here: no ground truth


def test_oracle_band_view_ranks_within_the_band():
    # class 0: a large detection of 0.9 on nothing, then a small one of 0.8 on the small object.
    # Over everything the small one ranks second; in the S band it ranks first.
    img = _one([([0, 0, 200, 200], 0.9, 0), ([300, 300, 320, 320], 0.8, 0)], [([300, 300, 320, 321], 0)])
    S = _lib.MAP_VIEW_S
    tp, gt = restated_tp(img, 1, [0.5], (1, 2), [_lib.MAP_VIEW_CENTRE, S, _lib.MAP_VIEW_L])
    assert tp[_lib.MAP_VIEW_CENTRE, 0, 0].tolist() == [0, 1]
    assert tp[S, 0, 0].tolist() == [1, 1] and gt[S].tolist() == [1] and gt[_lib.MAP_VIEW_L].tolist() == [0]
    assert np.array_equal(ranked_tp(img, 1, [0.5], (1, 2), [_lib.MAP_VIEW_CENTRE, S, _lib.MAP_VIEW_L]), tp)


def _tied(seed, B, M, N, C, decimals=1):
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(seed, B, M, N, C, ties=True)
    return db.astype(np.int32), np.round(ds, decimals), dc, dn, gtb, gtc, gtn


def test_oracle_filter_then_match_equals_full_walk_counted_by_rank():
    """The prefix argument: truncating each (image, class) to its first k detections and matching
    again gives the full walk's TP flags of those detections, in every view."""
    thr = [0.3, 0.5, 0.75]
    limits = (1, 2, 3, 5, 8, 40)
    for seed, C in ((91, 3), (92, 1)):
        args = _tied(seed, 10, 25, 10, C)
        views = list(VIEW_RULES)
        want, gt = restated_tp(args, C, thr, limits, views)
        assert np.array_equal(ranked_tp(args, C, thr, limits, views), want)
        assert (want[..., 0] < want[..., -1]).any()           # the limits do truncate
        assert all(gt[v].sum() > 0 for v in views)            # every band has ground truth
        assert np.all(np.diff(want, axis=-1) >= 0)


# ------------------------------------------------------------------------------ GPU

def _dev(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _acc(C, pieces, args, cls=None, **kw):
    from multigriddet_b200.evaluation import MapAccumulator
    acc = (cls or MapAccumulator)(C, **kw)
    lo = 0
    for n in pieces:
        acc.update(*_dev(*[a[lo:lo + n] for a in args]))
        lo += n
    assert lo == len(args[3])
    return acc


def _views(acc):
    return [v for v in range(V) if (acc._cfg.views >> v) & 1]


def _device_tp(acc):
    return np.cumsum(acc._recall_tp.cpu().numpy(), axis=-1)


def _matcher_view(args, kw):
    """The view calculate_map takes its main APs from for these settings (more than 10 000
    predictions with use_parallel and cache_ious: the centre one)."""
    if not kw.get("cache_ious", True):
        return _lib.MAP_VIEW_CENTRE
    many = kw.get("use_parallel", True) and int(args[3].sum()) > 10000
    return _lib.MAP_VIEW_CENTRE if many else _lib.MAP_VIEW_CORNER


def _check(acc, res, args, C, thresholds, limits, kw, match=oracle_match, want=None):
    """The device table (every matched view) and the dict's AR part against the restatement."""
    views = _views(acc)
    if want is None:
        want = restated_tp(args, C, thresholds, limits, views, match)
    tp, gt = want
    got = _device_tp(acc)
    for v in range(V):
        if v in views:
            assert np.array_equal(got[v], tp[v]), (v, np.argwhere(got[v] != tp[v])[:8])
        else:
            assert not got[v].any(), v
    view = _matcher_view(args, kw)
    exp = ar_keys(tp, gt, view, limits, per_scale=kw.get("compute_per_scale", True))
    _same({k: res[k] for k in exp}, exp)
    return tp


LIMITS = (1, 3, 10, 100)
_KWS = (dict(), dict(use_parallel=False), dict(cache_ious=False, compute_per_scale=False))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["a", "b", "ties"])
def test_gpu_equals_restatement_on_golden_cases(name):
    args, C = _case(np.load(GOLD), name)
    want = restated_tp(args, C, COCO, LIMITS, list(VIEW_RULES))
    for kw in _KWS:
        acc = _acc(C, [len(args[3])], args, recall_max_dets=LIMITS, **kw)
        res = acc.compute()
        tp = _check(acc, res, args, C, COCO, LIMITS, kw, want=want)
        assert res["AR1"] <= res["AR3"] <= res["AR10"] <= res["AR100"]
    assert (tp[..., 0] < tp[..., -1]).any()


@pytest.mark.gpu
def test_gpu_equals_restatement_on_random_ties_beyond_100_detections():
    C, thr, limits = 2, [0.5, 0.75, 0.9], (1, 10, 60, 101, 140)
    args = _tied(95, 12, 150, 20, C)
    args[3][:] = 150                                          # about 75 detections per (image, class)
    for kw in (dict(), dict(cache_ious=False)):
        acc = _acc(C, [5, 7], args, iou_thresholds=thr, recall_max_dets=limits, **kw)
        tp = _check(acc, acc.compute(), args, C, thr, limits, kw)
        assert all(tp[v].sum() > 0 for v in _views(acc))
        assert (tp[..., 2] < tp[..., 3]).any()                # 60 truncates


@pytest.mark.gpu
def test_gpu_at_size():
    C, B = 80, 2000
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(97, B, 100, 20, C)
    args = (db.astype(np.int32), np.round(ds, 2), dc, dn, gtb, gtc, gtn)
    limits = (1, 10, 100)
    for kw in (dict(), dict(use_parallel=False)):
        acc = _acc(C, [256] * 7 + [208], args, recall_max_dets=limits, **kw)
        res = acc.compute()
        assert res["recall"]["matcher"] == ("centre" if not kw else "corner")
        _check(acc, res, args, C, COCO, limits, kw, match=device_match)
        assert 0.0 < res["AR1"] < res["AR10"] <= res["AR100"] and res["ARS"] > 0 and res["ARL"] > 0


@pytest.mark.gpu
def test_gpu_independent_of_the_split_over_updates():
    C = 6
    args = _tied(99, 40, 30, 20, C)
    for kw in _KWS:
        whole = _acc(C, [40], args, recall_max_dets=LIMITS, **kw)
        split = _acc(C, [1, 0, 7, 32], args, recall_max_dets=LIMITS, **kw)
        assert np.array_equal(_device_tp(split), _device_tp(whole))
        _same(split.compute(), whole.compute())
        split.reset()
        assert not split._recall_tp.any()
        split.update(*_dev(*args))
        _same(split.compute(), whole.compute())


@pytest.mark.gpu
def test_gpu_ar_at_a_limit_covering_every_detection_is_the_curves_final_recall():
    C, M = 7, 30
    args = _tied(101, 60, M, 20, C, decimals=2)
    for kw in (dict(), dict(cache_ious=False)):
        res = _acc(C, [60], args, recall_max_dets=(1, 10, M), **kw).compute(precision_recall=True)
        pr, rc = res["precision_recall"], res["recall"]
        assert rc["matcher"] == pr["matcher"]
        assert np.array_equal(rc["num_gt"], pr["num_gt"])
        off = pr["offsets"].cpu().numpy()
        recall = pr["recall"].cpu().numpy()
        for c in range(C):
            if rc["num_gt"][c] == 0:
                assert (rc["recall"][c] == -1.0).all()
                continue
            tp_all = np.rint(rc["recall"][c, :, -1] * rc["num_gt"][c])
            if off[c + 1] == off[c]:
                assert (tp_all == 0).all(), c
                continue
            assert np.array_equal(recall[:, off[c + 1] - 1], tp_all / (rc["num_gt"][c] + 1e-8)), c


@pytest.mark.gpu
def test_gpu_keys_of_before_are_unchanged():
    C = 5
    args = _tied(103, 30, 40, 15, C, decimals=2)
    for kw in _KWS:
        plain = _acc(C, [12, 18], args, **kw)
        with_ar = _acc(C, [12, 18], args, recall_max_dets=(1, 10, 100), **kw)
        assert not hasattr(plain, "_recall_tp")
        for pr in (dict(), dict(precision_recall=True, confidences=[0.2, 0.5])):
            want = plain.compute(**pr)
            got = with_ar.compute(**pr)
            assert set(got) - set(want) == {"AR1", "AR10", "AR100", "ARS", "ARM", "ARL", "recall"}
            _same({k: got[k] for k in want}, want)


@pytest.mark.gpu
def test_gpu_class_out_of_range_still_raises():
    C = 4
    args = [np.array(a) for a in _tied(105, 10, 20, 8, C)]
    b = int(np.flatnonzero((args[3] > 0) & (args[6] > 0))[0])
    args[2][b, 0] = C
    acc = _acc(C, [10], args, recall_max_dets=(1, 10))
    with pytest.raises(AssertionError, match="class id outside"):
        acc.compute()


# ------------------------------------------------------------------------------ GPU, sharded

def _sharded(C, batches, rank=0, world=1, **kw):
    from multigriddet_b200.evaluation import ShardedMapAccumulator
    acc = ShardedMapAccumulator(C, **kw)
    for b in batches:
        lo, hi = shard_bounds(len(b[3]), rank, world)
        acc.update(*_dev(*[a[lo:hi] for a in b]), n_total=len(b[3]))
    return acc.compute()


def _single(C, batches, **kw):
    from multigriddet_b200.evaluation import MapAccumulator
    acc = MapAccumulator(C, **kw)
    for b in batches:
        acc.update(*_dev(*b))
    return acc.compute()


def _batches(args, sizes):
    out, lo = [], 0
    for n in sizes:
        out.append(tuple(a[lo:lo + n] for a in args))
        lo += n
    assert lo == len(args[3])
    return out


@pytest.mark.gpu
def test_gpu_sharded_world_of_one_equals_single():
    C = 80
    args = _tied(107, 300, 100, 20, C, decimals=2)
    for kw in (dict(), dict(use_parallel=False)):
        kw = dict(kw, recall_max_dets=(1, 10, 100))
        batches = _batches(args, [100, 200])
        _same(_sharded(C, batches, **kw), _single(C, batches, **kw), str(kw))


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
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(0)
    out = {}
    C = 7
    args = _tied(109, 31, 40, 12, C)
    try:
        for name, sizes in (("uneven", [31]),                      # 16 + 15 images
                            ("empty_update", [1, 19, 11]),          # rank 1 holds nothing in update 0
                            ("empty_rank", [1])):                   # rank 1 holds nothing at all
            for i, kw in enumerate((dict(), dict(cache_ious=False, compute_per_scale=False))):
                kw = dict(kw, recall_max_dets=(1, 5, 10, 40))
                batches = _batches(tuple(a[:sum(sizes)] for a in args), sizes)
                try:
                    _same(_sharded(C, batches, rank, world, **kw), _single(C, batches, **kw))
                    out[f"{name}{i}"] = "equal"
                except AssertionError as e:
                    out[f"{name}{i}"] = f"differs: {str(e)[:300]}"
        q.put((rank, out))
    except Exception:                                         # pragma: no cover
        import traceback
        q.put((rank, {"error": traceback.format_exc()[-2000:]}))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_gpu_two_ranks_equal_the_single_accumulator():
    res = _spawn(_rank_main, 2)
    for rank in (0, 1):
        got = res[rank]
        assert "error" not in got, (rank, got.get("error"))
        assert len(got) == 6 and all(v == "equal" for v in got.values()), (rank, got)
