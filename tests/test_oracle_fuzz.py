"""The checker of the GPU sweep, checked: on the random geometries of tests/test_gpu_fuzz.py
the C oracle (what the CUDA path is compared with) must equal the NumPy oracle, and where
the reference exists the NumPy oracle must equal the reference itself (everywhere: its outputs
on these inputs as stored in tests/golden/live_oracle_fuzz.npz)."""
import warnings

import numpy as np
import pytest

import golden_util as G
from fuzz_util import random_boxes, random_head, tie_free
from multigriddet_b200 import synth
from oracle import mgd_oracle as O
from oracle import ref_loader


def _case(seed):
    rng = np.random.default_rng(1000 + seed)
    S, C, anchors, grids = random_head(rng)
    B, N = int(rng.integers(1, 4)), int(rng.integers(1, 25))
    boxes = tie_free(random_boxes(rng, B, N, S, C), anchors)
    return rng, S, C, anchors, grids, boxes


@pytest.mark.parametrize("seed", range(16))
def test_c_oracle_equals_numpy_oracle_on_random_geometries(c_oracle, seed):
    import torch
    rng, S, C, anchors, grids, boxes = _case(seed)
    y_np = O.encode_targets(boxes, (S, S), anchors, C, grids)
    y_c = c_oracle.encode_targets(boxes, (S, S), anchors, C, grids)
    for a, b in zip(y_np, y_c):
        assert np.array_equal(a[..., 4:], b[..., 4:]) and np.array_equal(a[..., :2], b[..., :2])
        np.testing.assert_allclose(a[..., 2:4], b[..., 2:4], rtol=1e-6, atol=1e-7)
    if len({len(a) for a in anchors}) == 1:
        preds = [p.numpy().copy() for p in synth.planted_head_outputs([torch.from_numpy(y) for y in y_c],
                                                                      len(anchors[0]), seed)]
    else:
        preds = [rng.normal(0, 2, y.shape).astype(np.float32) for y in y_c]
    shapes = np.stack([rng.integers(S // 2, 3 * S, len(boxes)), rng.integers(S // 2, 3 * S, len(boxes))], 1)
    kw = dict(max_boxes=int(rng.choice([5, 100])), confidence=float(rng.choice([0.001, 0.05, 0.3])),
              nms_threshold=float(rng.choice([0.3, 0.45, 0.7])), nms_method=str(rng.choice(["diou", "standard"])),
              per_class=bool(rng.integers(0, 2)))
    r_np = O.postprocess_batch(preds, shapes, (S, S), anchors, C, **kw)
    r_c = c_oracle.decode_nms(preds, shapes, (S, S), anchors, C, **kw)
    for b in range(len(boxes)):
        k = int(r_c["counts"][b])
        one = r_np[b]                                   # per-image dict of the NumPy oracle
        assert len(one["index"]) == k, (seed, b)
        assert np.array_equal(one["index"], r_c["index"][b, :k]), (seed, b)
        np.testing.assert_allclose(one["scores"], r_c["scores"][b, :k], rtol=1e-6)
        np.testing.assert_allclose(one["boxes_xywh"], r_c["boxes_xywh"][b, :k], rtol=1e-9, atol=1e-9)


REC = G.Recorded("oracle_fuzz")


@pytest.mark.parametrize("seed", range(16))
def test_numpy_oracle_equals_reference_on_random_geometries(seed):
    rng, S, C, anchors, grids, boxes = _case(seed)
    if len({len(a) for a in anchors}) != 1:
        pytest.skip("the reference itself needs the same number of anchors on every layer "
                    "(np.array(anchor_mask), generators.py:2531)")
    y_np = O.encode_targets(boxes, (S, S), anchors, C, grids)
    if ref_loader.available():
        enc = ref_loader.load_encoder()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            y_ref = enc(boxes.copy(), (S, S), anchors, C, False, grid_shapes=[np.array(g) for g in grids])
        for a, b in zip(y_ref, y_np):
            assert np.array_equal(np.asarray(a), b)
    REC.check(f"seed{seed}", [boxes, *anchors, *y_np])
