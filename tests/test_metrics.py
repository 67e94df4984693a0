"""mAP matching (SURVEY.md 8(f)-4): reference multigriddet/evaluation/metrics.py.

CPU: the oracle restatement (oracle/metrics_oracle.py) against the golden vectors the
REAL reference produced (tests/golden/metrics_cases.npz, oracle/gen_golden.py) and against
the reference on fresh seeds (executed live where its tree exists, else its stored outputs,
tests/golden/live_metrics.npz).  GPU: the CUDA path
(mgd_match_detections / mgd_iou_matrix through the drop-in module) against both.
"""
import os

import numpy as np
import pytest

import golden_util as G
from oracle import metrics_oracle as MO
from oracle import ref_loader

GOLD = os.path.join(os.path.dirname(__file__), "golden", "metrics_cases.npz")


def _case(z, name):
    return tuple(z[f"{name}_{k}"] for k in ("db", "ds", "dc", "dn", "gtb", "gtc", "gtn")) + (int(z[f"{name}_C"]),)


def _flat(tp, ds, dc, dn, gtc, gtn):
    B = len(dn)
    cat = lambda a, n: np.concatenate([a[b, :n[b]] for b in range(B)]) if B else a[:0]
    return (np.concatenate([tp[:, b, :dn[b]] for b in range(B)], 1), cat(ds, dn), cat(dc, dn), cat(gtc, gtn))


def _check_against_golden(z, name, matcher):
    db, ds, dc, dn, gtb, gtc, gtn, C = _case(z, name)
    thr = z["thresholds"]
    for cached, tag in ((True, "cached"), (False, "plain")):
        tp = matcher(db, ds, dc, dn, gtb, gtc, gtn, thr, cached)
        ftp, fs, fc, fgc = _flat(np.asarray(tp), ds, dc, dn, gtc, gtn)
        for c in range(C):
            sel = fc == c
            order = np.argsort(fs[sel], kind="stable")[::-1]
            for t in range(len(thr)):
                key = f"{name}_{tag}_c{c}_t{t}_tp"
                if key in z.files:
                    assert np.array_equal(z[f"{name}_{tag}_c{c}_t{t}_scores"], fs[sel][order])
                    assert np.array_equal(z[key], ftp[t][sel][order].astype(bool)), (name, tag, c, t)
                ap = MO.class_ap(ftp[t], fs, fc, fgc, c)
                assert ap == pytest.approx(float(z[f"{name}_{tag}_c{c}_t{t}_ap"]), rel=1e-12, abs=1e-15)


@pytest.mark.parametrize("name", ["a", "b", "ties"])
def test_oracle_matches_reference_golden(name):
    z = np.load(GOLD)
    _check_against_golden(z, name, lambda *a: MO.match_batch(*a)[0])


def test_oracle_iou_matrix_golden():
    z = np.load(GOLD)
    for name in z["names"]:
        db, ds, dc, dn, gtb, gtc, gtn, C = _case(z, str(name))
        ref = z[f"{name}_ioumat"]
        n1, n2 = max(int(dn[0]), 1), max(int(gtn[0]), 1)
        got = np.array([[MO.iou_corner(db[0, i], gtb[0, j]) for j in range(n2)] for i in range(n1)])
        assert np.array_equal(got, ref)


def test_oracle_matches_live_reference_on_fresh_seeds():
    from oracle.gen_golden import synth_eval_set
    live = ref_loader.available()
    M = ref_loader.load_metrics() if live else None
    rec = G.Recorded("metrics")
    for seed in (11, 12):
        db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(seed, 6, 25, 10, 3)
        preds, gts = MO.to_dicts(db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
        for cached in (True, False):
            tp, _ = MO.match_batch(db, ds, dc, dn, gtb, gtc, gtn, [0.5, 0.8], cached)
            ftp, fs, fc, fgc = _flat(tp, ds, dc, dn, gtc, gtn)
            for c in range(3):
                cp = [p for p in preds if p["class"] == c]
                cg = [g for g in gts if g["class"] == c]
                for t, th in enumerate((0.5, 0.8)):
                    sel = fc == c
                    order = np.argsort(fs[sel], kind="stable")[::-1]
                    got = ftp[t][sel][order].astype(bool)
                    if live:
                        if cached:
                            cache = M.compute_iou_cache_for_class(preds, gts, c)
                            ref = M.match_predictions_to_gt_cached(cp, cg, th, cache)
                        else:
                            ref = M.match_predictions_to_gt(cp, cg, th)
                        assert np.array_equal(ref[0], got)
                    rec.check(f"s{seed}_{cached}_c{c}_t{t}", [got])


# ------------------------------------------------------------------------------ GPU

@pytest.mark.gpu
@pytest.mark.parametrize("name", ["a", "b", "ties"])
def test_gpu_matcher_against_reference_golden(name):
    from multigriddet_b200 import engine
    z = np.load(GOLD)

    def gpu(db, ds, dc, dn, gtb, gtc, gtn, thr, cached):
        return engine.match_detections(db, ds, dc, dn, gtb, gtc, gtn, thr,
                                       iou_mode="corner" if cached else "centre")
    _check_against_golden(z, name, gpu)


@pytest.mark.gpu
def test_gpu_matcher_matches_oracle_host_and_device():
    import torch
    from multigriddet_b200 import engine
    from oracle.gen_golden import synth_eval_set
    thr = [0.5, 0.55, 0.6, 0.65, 0.7, 0.75, 0.8, 0.85, 0.9, 0.95]
    for seed, B, M, N, C, ties in ((21, 16, 100, 40, 8, False), (22, 9, 33, 70, 2, True), (23, 3, 1, 1, 1, False)):
        args = synth_eval_set(seed, B, M, N, C, ties)
        for cached, mode in ((True, "corner"), (False, "centre")):
            ref_tp, ref_who = MO.match_batch(*args, thr, cached)
            tp, who = engine.match_detections(*args, thr, iou_mode=mode, return_matched=True)
            assert np.array_equal(tp, ref_tp) and np.array_equal(who, ref_who), (seed, mode)
            dev = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in args]
            tp_d = engine.match_detections(*dev, thr, iou_mode=mode)
            assert np.array_equal(tp_d.cpu().numpy(), ref_tp)
    # empty inputs
    e = engine.match_detections(np.zeros((2, 5, 4)), np.zeros((2, 5)), np.zeros((2, 5), np.int32),
                                np.zeros(2, np.int32), np.zeros((2, 3, 4)), np.zeros((2, 3), np.int32),
                                np.zeros(2, np.int32), [0.5])
    assert e.shape == (1, 2, 5) and not e.any()


@pytest.mark.gpu
def test_gpu_dropin_module_against_reference_golden():
    from multigriddet_b200.evaluation import metrics as G
    z = np.load(GOLD)
    for name in ("a", "ties"):
        db, ds, dc, dn, gtb, gtc, gtn, C = _case(z, name)
        preds, gts = MO.to_dicts(db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
        for cached, tag in ((True, "cached"), (False, "plain")):
            res = G.calculate_map(preds, gts, C, use_parallel=False, cache_ious=cached)
            for key in ("mAP", "mAP50", "mAP75", "APS", "APM", "APL", "APS50", "APM50", "APL50"):
                assert float(res[key]) == pytest.approx(float(z[f"{name}_{tag}_map_{key}"]), rel=1e-12, abs=1e-15), key
            voc = G.calculate_map(preds, gts, C, iou_thresholds=[0.5], method="voc", use_parallel=False,
                                  cache_ious=cached, compute_per_scale=False)
            assert float(voc["mAP50"]) == pytest.approx(float(z[f"{name}_{tag}_map_voc50"]), rel=1e-12)
            c = 1
            cp = [p for p in preds if p["class"] == c]
            cg = [g for g in gts if g["class"] == c]
            fn = G.match_predictions_to_gt_cached if cached else G.match_predictions_to_gt
            tp, fp, sc = fn(cp, cg, 0.5, None) if cached else fn(cp, cg, 0.5)
            assert np.array_equal(tp, z[f"{name}_{tag}_c{c}_t0_tp"]) and np.array_equal(fp, ~tp)
            assert np.array_equal(sc, z[f"{name}_{tag}_c{c}_t0_scores"])
        n1, n2 = max(int(dn[0]), 1), max(int(gtn[0]), 1)
        assert np.array_equal(G.calculate_iou_matrix(db[0, :n1], gtb[0, :n2]), z[f"{name}_ioumat"])
    assert G.match_predictions_to_gt([], [], 0.5)[0].shape == (0,)
    assert G.calculate_iou_matrix(np.zeros((0, 4)), np.zeros((3, 4))).shape == (0, 3)
