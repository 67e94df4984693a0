"""Box-side pre-step of the encoder (SURVEY.md 8(f)-3): reference
multigriddet/data/augmentation.py reshape_boxes (:112-164) and merge_mosaic_bboxes (:606-667).

CPU: the oracle restatement against golden vectors produced by the REAL reference
(tests/golden/boxes_cases.npz; reshape_boxes with its row shuffle disabled) and against the
reference on fresh seeds (live where its tree exists, else its stored outputs,
tests/golden/live_box_transforms.npz).  GPU: mgd_reshape_boxes /
mgd_mosaic_merge_boxes against both, and the device pipeline boxes -> reshape -> encode.
"""
import os

import numpy as np
import pytest

import golden_util as G
from oracle import mgd_oracle as O
from oracle import ref_loader
from oracle.gen_golden import synth_box_transform_cases

GOLD = os.path.join(os.path.dirname(__file__), "golden", "boxes_cases.npz")


def _golden_cases():
    z = np.load(GOLD)
    reshape, mosaic = synth_box_transform_cases(77, int(z["n_cases"]))
    return z, reshape, mosaic


def test_oracle_matches_reference_golden():
    z, reshape, mosaic = _golden_cases()
    for i, c in enumerate(reshape):
        for tag, dt in (("i32", np.int32), ("f64", np.float64)):
            got = O.reshape_boxes(c["boxes"].astype(dt), c["src"], c["target"], c["padding"], c["offset"],
                                  c["hflip"], c["vflip"])
            assert np.array_equal(np.asarray(got).reshape(-1, 5), z[f"r{i}_{tag}"]), (i, tag)
    for i, c in enumerate(mosaic):
        assert np.array_equal(O.merge_mosaic_bboxes(c["boxes"], *c["crop"], c["size"]), z[f"m{i}"]), i


REC = G.Recorded("box_transforms")


def test_oracle_matches_live_reference_on_fresh_seeds():
    live = ref_loader.available()
    R = ref_loader.load_box_transforms() if live else None
    reshape, mosaic = synth_box_transform_cases(5, 60)
    for i, c in enumerate(reshape):
        for dt in (np.int32, np.float64, np.float32):
            a = (c["boxes"].astype(dt), c["src"], c["target"], c["padding"], c["offset"], c["hflip"], c["vflip"])
            got = np.asarray(O.reshape_boxes(*a))
            if live:
                assert np.array_equal(np.asarray(R.reshape_boxes(*a)), got)
            REC.check(f"reshape{i}_{np.dtype(dt).name}", [a[0], got])
    for i, c in enumerate(mosaic):
        got = O.merge_mosaic_bboxes(c["boxes"], *c["crop"], c["size"])
        if live:
            assert np.array_equal(R.merge_mosaic_bboxes(c["boxes"], *c["crop"], c["size"]), got)
        REC.check(f"mosaic{i}", [c["boxes"], got])


def _reshape_batch_inputs(cases, dt, N):
    B = len(cases)
    boxes = np.zeros((B, N, 5), dt)
    counts = np.zeros(B, np.int32)
    params = np.zeros((B, 10), np.int32)
    for b, c in enumerate(cases):
        n = len(c["boxes"])
        boxes[b, :n] = c["boxes"].astype(dt)
        counts[b] = n
        params[b] = [*c["src"], *c["target"], *c["padding"], *c["offset"], int(c["hflip"]), int(c["vflip"])]
    return boxes, counts, params


@pytest.mark.gpu
def test_gpu_reshape_boxes_against_golden_and_oracle():
    import torch
    from multigriddet_b200 import engine
    from multigriddet_b200.data import reshape_boxes
    z, reshape, _ = _golden_cases()
    N = 24
    for tag, dt in (("i32", np.int32), ("f64", np.float64)):
        boxes, counts, params = _reshape_batch_inputs(reshape, dt, N)
        for dev in (False, True):
            args = (torch.from_numpy(boxes).cuda(), params, counts) if dev else (boxes, params, counts)
            out, o32, cnt = engine.reshape_boxes_batch(*args)
            if dev:
                out, o32, cnt = out.cpu().numpy(), o32.cpu().numpy(), cnt.cpu().numpy()
            for i in range(len(reshape)):
                ref = z[f"r{i}_{tag}"]
                assert cnt[i] == len(ref) and np.array_equal(out[i, :cnt[i]], ref), (tag, dev, i)
                assert not out[i, cnt[i]:].any()
                assert np.array_equal(o32[i], out[i].astype(np.float32))
        for i, c in enumerate(reshape[:8]):                        # the single-image drop-in
            got = reshape_boxes(c["boxes"].astype(dt), c["src"], c["target"], c["padding"], c["offset"],
                                c["hflip"], c["vflip"])
            assert got.dtype == dt and np.array_equal(np.asarray(got).reshape(-1, 5), z[f"r{i}_{tag}"])
    assert len(reshape_boxes(np.zeros((0, 5), np.int32), (10, 10), (5, 5), (5, 5), (0, 0))) == 0


@pytest.mark.gpu
def test_gpu_mosaic_merge_against_golden_and_oracle():
    import torch
    from multigriddet_b200 import engine
    from multigriddet_b200.data import merge_mosaic_bboxes
    z, _, mosaic = _golden_cases()
    for i, c in enumerate(mosaic):
        assert np.array_equal(merge_mosaic_bboxes(c["boxes"], *c["crop"], c["size"]), z[f"m{i}"]), i
    # batch form: 16 mosaics drawing their four samples from a batch of 16 images; cap at N
    rng = np.random.default_rng(3)
    N, S = 12, 416
    src = np.zeros((16, N, 5))
    for b in range(16):
        m = int(rng.integers(4, N + 1))
        xy = rng.uniform(0, S, (m, 2)); wh = rng.uniform(20, 200, (m, 2))
        src[b, :m] = np.concatenate([xy, np.minimum(xy + wh, S), rng.integers(0, 20, (m, 1))], 1)
    idx = np.stack([rng.permutation(16)[:4] for _ in range(16)])
    crop = rng.integers(int(S * .2), int(S * .8), (16, 2))
    ref = np.stack([O.merge_mosaic_bboxes(src[idx[b]], int(crop[b, 0]), int(crop[b, 1]), (S, S)) for b in range(16)])
    for dev in (False, True):
        out, o32, cnt = engine.mosaic_merge_boxes_batch(torch.from_numpy(src).cuda() if dev else src, idx, crop, (S, S))
        if dev:
            out, o32, cnt = out.cpu().numpy(), o32.cpu().numpy(), cnt.cpu().numpy()
        assert np.array_equal(out, ref)
        assert np.array_equal(cnt, (ref[..., 2] > 0).sum(1)) and cnt.max() == N      # the cap is hit
        assert np.array_equal(o32, ref.astype(np.float32))


@pytest.mark.gpu
def test_device_pipeline_reshape_then_encode():
    """int32 annotation boxes -> reshape on the device -> float32 (B, N, 5) -> encoder, no host hop."""
    import torch
    from multigriddet_b200 import engine, synth
    S, C, N = 416, 80, 24
    reshape, _ = synth_box_transform_cases(9, 32)
    for c in reshape:
        c["target"] = (S, S)
    boxes, counts, params = _reshape_batch_inputs(reshape, np.int32, N)
    anchors = synth.coco_anchors(np.float32)
    _, d32, _ = engine.reshape_boxes_batch(torch.from_numpy(boxes).cuda(), params, counts, sync=False)
    got = engine.encode_targets(d32, (S, S), anchors, C)
    host = np.zeros((len(reshape), N, 5), np.float32)
    for b, c in enumerate(reshape):
        r = np.asarray(O.reshape_boxes(c["boxes"].astype(np.int32), c["src"], c["target"], c["padding"],
                                       c["offset"], c["hflip"], c["vflip"])).reshape(-1, 5)
        host[b, :len(r)] = r
    ref = O.encode_targets(host, (S, S), anchors, C)
    for g, r in zip(got, ref):
        g = g.cpu().numpy()
        assert np.array_equal(g[..., 4:], r[..., 4:]) and np.array_equal(g[..., :2], r[..., :2])
        np.testing.assert_allclose(g[..., 2:4], r[..., 2:4], rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------
# tf.data box pre-step (generators.py:1859-1916, 1963-2034): the oracle is pinned against the
# reference's own TF source run over oracle/tf_shim.py (tests at the end of this file)
# ------------------------------------------------------------------------------

def _tfdata_case(seed, B=12, N=40):
    rng = np.random.default_rng(seed)
    src = np.stack([rng.integers(120, 1400, B), rng.integers(120, 1400, B)], 1)       # (h, w)
    counts = rng.integers(0, N + 1, B).astype(np.int32)
    boxes = np.zeros((B, N, 5), np.float32)
    for b in range(B):
        n = counts[b]
        xy = rng.uniform(0, [src[b, 1], src[b, 0]], (n, 2))
        wh = rng.uniform(2, [src[b, 1] / 2, src[b, 0] / 2], (n, 2))
        boxes[b, :n] = np.concatenate([xy, np.minimum(xy + wh, [src[b, 1], src[b, 0]]),
                                       rng.integers(0, 80, (n, 1))], 1)
    ms = np.stack([rng.choice([320, 416, 512, 608], B), ] * 2, 1)
    ms[::3] = 0                                                                      # some without
    flip = rng.integers(0, 2, B).astype(bool)
    return boxes, counts, src, ms, flip


def test_tf_letterbox_oracle_known_values():
    """Hand-derived: a 480x640 image into 608x608 -> scale 0.95, new size 608x456, pad_top 76."""
    sx, sy, pl, pt = O.tf_letterbox_params(480, 640, (608, 608))
    assert (float(sx), float(pl), float(pt)) == (np.float32(608) / np.float32(640), 0.0, 76.0) and sx == sy
    out = O.tf_letterbox_boxes(np.array([[[100, 50, 300, 250, 7]]], np.float32), None, [(480, 640)],
                               (608, 608), 100, expansion=4)
    assert out.shape == (1, 400, 5) and not out[0, 1:].any()
    np.testing.assert_allclose(out[0, 0], [95.0, 123.5, 285.0, 313.5, 7.0], rtol=1e-6)
    flipped = O.tf_letterbox_boxes(np.array([[[100, 50, 300, 250, 7]]], np.float32), None, [(480, 640)],
                                   (608, 608), 100, hflip=[True])
    np.testing.assert_allclose(flipped[0, 0], [608 - 285.0, 123.5, 608 - 95.0, 313.5, 7.0], rtol=1e-6)
    # multi-scale: sampled shape 320 -> image scaled by 320/608, then letterboxed back up
    sx, sy, pl, pt = O.tf_letterbox_params(480, 640, (608, 608), (320, 320))
    assert abs(float(sx) - 0.95) < 5e-3 and float(pl) in (0.0, 1.0)


@pytest.mark.gpu
def test_tf_letterbox_boxes_match_oracle_and_feed_the_encoder():
    import torch
    from multigriddet_b200 import engine, synth
    from multigriddet_b200.data import expand_box_capacity, letterbox_boxes
    for seed in (1, 2):
        boxes, counts, src, ms, flip = _tfdata_case(seed)
        for expansion, (mo, mi) in ((1, (False, False)), (2, (False, True)), (4, (True, False)), (8, (True, True))):
            ref = O.tf_letterbox_boxes(boxes, counts, src, (608, 608), 30, expansion, ms, flip)
            got = letterbox_boxes(boxes, src, (608, 608), 30, counts, mo, mi, ms, flip)
            assert got.dtype == np.float32 and np.array_equal(got, ref)
            dev = letterbox_boxes(torch.from_numpy(boxes).cuda(), src, (608, 608), 30, counts, mo, mi, ms, flip)
            assert np.array_equal(dev.cpu().numpy(), ref)
        # capacity expansion alone == what the fused kernel pads
        plain = letterbox_boxes(boxes, src, (608, 608), 30, counts, multiscale_shapes=ms, hflip=flip)
        assert np.array_equal(expand_box_capacity(plain, True, True),
                              letterbox_boxes(boxes, src, (608, 608), 30, counts, True, True, ms, flip))
    # device pipeline: raw annotation boxes -> letterbox kernel -> encoder, nothing on the host
    boxes, counts, src, ms, flip = _tfdata_case(5, B=6)
    d = letterbox_boxes(torch.from_numpy(boxes).cuda(), src, (608, 608), 40, counts, True, False)
    anchors = synth.coco_anchors(np.float32)
    y_dev = engine.encode_targets(d, (608, 608), anchors, 80)
    y_ref = O.encode_targets(O.tf_letterbox_boxes(boxes, counts, src, (608, 608), 40, 4), (608, 608), anchors, 80)
    for a, r in zip(y_dev, y_ref):
        assert np.array_equal(a.cpu().numpy()[..., 4:], r[..., 4:])


def _tfboxes_golden():
    import golden_util as G
    z = np.load(G.GOLDEN + "/tfboxes_cases.npz")
    cap = int(z["cap"])
    for i in range(int(z["n_cases"])):
        n, sh, sw, S, m0, m1, flip, exp = (int(v) for v in z[f"c{i}_meta"])
        yield z[f"c{i}_boxes"], n, (sh, sw), S, ((m0, m1) if m0 else None), bool(flip), exp, cap, z[f"c{i}_out"]


def test_tf_letterbox_oracle_matches_reference_code_golden():
    """tests/golden/tfboxes_cases.npz: outputs of the reference's own tf.data box functions
    (tf_letterbox_resize, _preprocess_image_and_boxes, tf_random_horizontal_flip,
    _expand_box_capacity; generators.py:167-256, 1859-2034) executed over oracle/tf_shim.py."""
    k = 0
    for boxes, n, src, S, ms, flip, exp, cap, ref in _tfboxes_golden():
        got = O.tf_letterbox_boxes(boxes[None], np.array([n]), [src], (S, S), cap, exp,
                                   multiscale_shapes=None if ms is None else [ms], hflip=[flip])[0]
        assert got.shape == ref.shape and np.array_equal(got, ref)
        k += 1
    assert k >= 40


def test_tf_letterbox_oracle_matches_live_reference_code_over_tf_shim():
    """Fresh seeds: live where the reference tree exists, else its stored outputs."""
    from oracle.gen_golden import tfboxes_inputs
    f = ref_loader.load_tf_box_prestep() if ref_loader.available() else None
    for i, (boxes, n, src, S, ms, flip, exp) in enumerate(tfboxes_inputs(701, 40)):
        got = O.tf_letterbox_boxes(boxes[None], np.array([n]), [src], (S, S), 12, exp,
                                   multiscale_shapes=[ms] if ms[0] else None, hflip=[flip])[0]
        if f is not None:
            ref = f(boxes[:n], src, (S, S), 12, exp, ms if ms[0] else None, flip)
            assert got.shape == ref.shape and np.array_equal(got, ref)
        REC.check(f"tfboxes{i}", [boxes, got])


@pytest.mark.gpu
def test_gpu_letterbox_boxes_match_reference_code_golden():
    """mgd_letterbox_boxes (host arrays and device tensors) against the fixtures made from the
    reference's own code: bit for bit (IEEE float32 multiplies / adds and int truncations)."""
    import torch
    from multigriddet_b200 import engine
    for boxes, n, src, S, ms, flip, exp, cap, ref in _tfboxes_golden():
        kw = dict(counts=np.array([n], np.int32), expansion=exp,
                  multiscale_shapes=None if ms is None else [ms], hflip=[flip])
        got = engine.letterbox_boxes_batch(boxes[None], [src], (S, S), cap, **kw)[0]
        assert np.array_equal(got, ref)
        dev = engine.letterbox_boxes_batch(torch.from_numpy(boxes[None]).cuda(), [src], (S, S), cap, **kw)[0]
        assert np.array_equal(dev.cpu().numpy(), ref)
