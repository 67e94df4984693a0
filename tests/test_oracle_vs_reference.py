"""The oracle against the reference on fresh seeds: executed live where the reference tree
exists, and everywhere against the reference's outputs on the same inputs as stored in
tests/golden/live_oracle_vs_reference.npz (golden_util.Recorded).
"""
import numpy as np
import pytest

import golden_util as G
from oracle import mgd_oracle as O
from oracle import ref_loader
from multigriddet_b200 import synth

LIVE = ref_loader.available()
REC = G.Recorded("oracle_vs_reference")


@pytest.mark.parametrize("S,C,N,B,layout,corners,padding,dt", [
    (608, 80, 100, 3, "uniform", "int", "tail", np.float32),
    (608, 80, 100, 2, "uniform", "frac", "interleaved", np.float64),
    (416, 20, 20, 8, "uniform", "int", "tail", np.float32),
    (320, 80, 300, 2, "mosaic", "frac", "tail", np.float32),
    (544, 80, 300, 2, "mosaic", "int", "interleaved", np.float64),
    (672, 80, 800, 1, "mosaic", "frac", "tail", np.float32),
])
def test_encoder_restatements_equal_reference(S, C, N, B, layout, corners, padding, dt, c_oracle):
    anchors = synth.coco_anchors(dt)
    boxes = synth.synth_boxes(31, B, N, S, C, corners=corners, layout=layout, padding=padding)
    ref = O.encode_targets(boxes, (S, S), anchors, C)
    if LIVE:
        live = ref_loader.load_encoder()(boxes.copy(), (S, S), anchors, C, False)
        assert all(np.array_equal(a, b) for a, b in zip(live, ref))
    REC.check(f"enc_{S}_{C}_{N}_{B}_{layout}_{corners}_{padding}_{np.dtype(dt).name}", [boxes, *ref])
    for impl in (O.encode_targets_parallel_scheme, c_oracle.encode_targets):
        got = impl(boxes, (S, S), anchors, C)
        assert all(np.array_equal(a, b) for a, b in zip(ref, got)), impl.__name__
    with pytest.raises(AssertionError):
        bad = boxes.copy()
        bad[0, 0, 4] = C
        O.encode_targets(bad, (S, S), anchors, C)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_decoder_restatements_equal_reference(dt, c_oracle):
    import torch
    S, C, B = 608, 80, 3
    anchors = synth.coco_anchors(dt)
    boxes = synth.synth_boxes(5, B, 100, S, C)
    yt = O.encode_targets(boxes, (S, S), anchors, C)
    preds = [p.numpy() for p in synth.planted_head_outputs([torch.from_numpy(y) for y in yt], 3, 9)]
    if LIVE:
        post = ref_loader.load_postprocess()
        dec = post.MultiGridDecoder(anchors, C, input_shape=(S, S))
    for k, (ishape, method, conf, thr) in enumerate((((608, 608), "diou", 0.001, 0.45),
                                                      ((480, 640), "diou", 0.1, 0.45),
                                                      ((427, 640), "cluster", 0.001, 0.5))):
        cc = c_oracle.decode_nms(preds, [ishape], (S, S), anchors, C, max_boxes=100, confidence=conf,
                                 nms_threshold=thr, nms_method=method)
        for b in range(B):
            one = [p[b:b + 1] for p in preds]
            m = O.postprocess_image(one, ishape, (S, S), anchors, C, max_boxes=100, confidence=conf,
                                    nms_threshold=thr, nms_method=method)
            rb, rc, rs = m["boxes_xyxy"], m["classes"], m["scores"]
            if LIVE:
                lb, lc, ls = dec.postprocess([o.copy() for o in one], ishape, (S, S), max_boxes=100,
                                             confidence=conf, nms_threshold=thr, nms_method=method)
                assert np.array_equal(lb, rb) and np.array_equal(lc, rc) and np.array_equal(ls, rs)
            REC.check(f"dec_{np.dtype(dt).name}_k{k}_b{b}", [rb, rc, rs])
            n = len(rs)
            assert int(cc["counts"][b]) == n
            assert np.array_equal(cc["scores"][b, :n], rs)
            assert np.array_equal(cc["boxes_xyxy"][b, :n], rb.reshape(-1, 4))
    # sigmoid mode and the dense decode tensor
    d_mine = O.decode_predictions(preds, anchors, (S, S), C, use_softmax=False, rescore_confidence=False)
    if LIVE:
        dec2 = post.MultiGridDecoder(anchors, C, input_shape=(S, S), use_softmax=False, rescore_confidence=False)
        assert np.array_equal(dec2.decode_predictions([p.copy() for p in preds]), d_mine)
    REC.check(f"dec_{np.dtype(dt).name}_dense_sigmoid", [d_mine])


@pytest.mark.skipif(not LIVE, reason="asserts the reference's own behaviour: needs the reference tree")
def test_reference_error_conventions():
    post = ref_loader.load_postprocess()
    anchors = synth.coco_anchors(np.float32)
    dec = post.MultiGridDecoder(anchors, 80)
    with pytest.raises(ValueError):
        dec.decode_predictions([np.zeros((1, 19, 19, 88), np.float32)])
    assert post.DIoUNMS().apply_nms(np.zeros((0, 4)), np.zeros(0), np.zeros(0), 0.5, 0.1) == ([], [], [])
    with pytest.raises(NotImplementedError):      # 'standard' is not wired in the reference
        dec.handle_predictions(np.ones((1, 3, 85)), (608, 608), nms_method="standard")


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_per_class_nms_equals_reference_per_partition(seed):
    """SURVEY 8a-9 / VERDICT r1 item 6a: O.greedy_nms(per_class=True) against the reference's
    DIoUNMS / StandardNMS (nms.py:83-187) run per argmax-class partition, merged by score,
    then the reference's top-k (multigrid_decode.py:336-345)."""
    from oracle.gen_golden import reference_per_class
    rng = np.random.default_rng(seed)
    n = int(rng.integers(50, 700))
    xy = rng.uniform(0, 300, size=(n, 2))
    wh = rng.uniform(4, 150, size=(n, 2))
    boxes = np.concatenate([xy, wh], 1)
    scores = rng.uniform(0.01, 1, size=n)
    classes = rng.integers(0, 5, size=n)
    REC.check(f"pcnms_s{seed}_inputs", [boxes, scores, classes])
    if LIVE:
        post = ref_loader.load_postprocess()
        dec = post.MultiGridDecoder(synth.coco_anchors(np.float32), 80)
    for name, diou in (("DIoUNMS", True), ("StandardNMS", False)):
        for thr in (0.3, 0.45, 0.6):
            keep = O.greedy_nms(boxes, scores, thr, diou, classes=classes, per_class=True)
            # stored: the rows the reference keeps, as positions in the inputs
            REC.check(f"pcnms_s{seed}_{name}_{thr}", [np.asarray(keep, np.int64)])
            for mx in (n, 30):
                if LIVE:
                    b, c, s = reference_per_class(post, dec, boxes, classes, scores, thr,
                                                  getattr(post, name), mx)
                    assert np.array_equal(scores[keep[:mx]], s)
                    assert np.array_equal(boxes[keep[:mx]], b)
                    assert np.array_equal(classes[keep[:mx]], c)


@pytest.mark.parametrize("S,C,N,B,layout,corners,padding,aset,seed", [
    (608, 80, 100, 3, "uniform", "int", "tail", "coco", 41),
    (608, 80, 100, 2, "mosaic", "frac", "interleaved", "coco", 42),
    (416, 20, 30, 4, "uniform", "frac", "tail", "coco", 43),
    (352, 1, 40, 2, "mosaic", "frac", "tail", "small_first", 44),
    (320, 80, 300, 2, "mosaic", "frac", "tail", "coco", 45),
    (672, 80, 400, 1, "mosaic", "int", "interleaved", "coco", 46),
])
def test_tf_encoder_restatement_equals_reference_code_over_tf_shim(S, C, N, B, layout, corners, padding,
                                                                   aset, seed):
    """SURVEY 8a-3: ``O.encode_targets_tf_compat`` against the reference's OWN TensorFlow encoder
    (generators.py:2696-3390), its source executed statement by statement with oracle/tf_shim.py
    answering the tf.* calls in NumPy (TensorFlow is not installed).  Bit for bit, logarithms
    included: both sides call the same float32 log here."""
    from oracle.gen_golden import SMALL_FIRST
    anchors = (synth.coco_anchors(np.float32) if aset == "coco"
               else [np.array(a, dtype=np.float32) for a in SMALL_FIRST])
    boxes = synth.synth_boxes(seed, B, N, S, C, corners=corners, layout=layout, padding=padding,
                              anchors=anchors)
    grids = [(S // 32,) * 2, (S // 16,) * 2, (S // 8,) * 2]
    got = O.encode_targets_tf_compat(boxes, (S, S), anchors, C, grids)
    if LIVE:
        ref = ref_loader.load_tf_encoder()(boxes.copy(), (S, S), anchors, C, grids)
        for g, r in zip(got, ref):
            assert np.array_equal(g, r)
    REC.check(f"tfenc_s{seed}", [boxes, *got])
    assert sum(int(g[..., 4].sum()) for g in got) > 0
    assert all(g.dtype == np.float32 for g in got)


def test_tf_encoder_restatement_on_the_adversarial_inputs():
    """Same, on the hand-made inputs of oracle/gen_golden.tf_adversarial_boxes: duplicate
    centres (scatter order), blocks leaving the grid, cell-boundary centres, zero-area rows,
    class ids outside [0, C)."""
    from oracle.gen_golden import tf_adversarial_boxes
    S, C = 608, 80
    anchors = synth.coco_anchors(np.float32)
    grids = [(19, 19), (38, 38), (76, 76)]
    boxes = tf_adversarial_boxes(S, C)
    got = O.encode_targets_tf_compat(boxes, (S, S), anchors, C, grids)
    if LIVE:
        ref = ref_loader.load_tf_encoder()(boxes.copy(), (S, S), anchors, C, grids)
        for g, r in zip(got, ref):
            assert np.array_equal(g, r)
    REC.check("tfenc_adversarial", [boxes, *got])
    ref = got
    # boxes 0, 1 (identical) and 2 share their centre and their layer: the LAST one (class 1) owns
    # every cell of the block, classes 3 and 7 appear nowhere; the ids outside [0, C) light no
    # class channel at all
    assert all(r[0][..., 5 + 3 + 3].sum() == 0 and r[0][..., 5 + 3 + 7].sum() == 0 for r in ref)
    assert sum(float(r[0][..., 5 + 3 + 1].sum()) for r in ref) >= 9
    assert any(np.any((r[0][..., 4] > 0) & (r[0][..., 8:].sum(-1) == 0)) for r in ref)


def test_tf_encoder_restatement_on_odd_geometries():
    """60 random heads (1-4 layers, 1-4 anchors per layer, grids down to 2 x 2) with boxes leaving
    the image, negative sizes and class ids outside [0, C): the reference's TF encoder over the
    TF-op stand-in against the restatement, bit for bit."""
    from fuzz_util import tf_encoder_odd_case
    rng = np.random.default_rng(77)
    for i in range(60):
        S, C, anchors, grids, boxes = tf_encoder_odd_case(rng)
        got = O.encode_targets_tf_compat(boxes, (S, S), anchors, C, grids)
        if LIVE:
            ref = ref_loader.load_tf_encoder()(boxes.copy(), (S, S), anchors, C, grids)
            assert all(np.array_equal(g, r) for g, r in zip(got, ref)), (S, C, [a.shape for a in anchors])
        REC.check(f"tfenc_odd{i}", [boxes, *anchors, *got])
