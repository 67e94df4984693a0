"""Loss-side ignore mask (SURVEY.md 8(f)-2): reference
multigriddet/losses/multigrid_loss.py:445-703.

TensorFlow is not installed here, so the reference's graph code cannot run as it is.  The pin
is its own source -- ``MultiGridLoss._compute_ignore_mask`` / ``_compute_iou_batch`` --
executed statement by statement with ``oracle/tf_shim.py`` answering the tf.* / K.* calls in
NumPy: live against the oracle restatement (oracle/loss_oracle.py) where the reference tree
exists, and as ``tests/golden/ignoremask_cases.npz`` everywhere else.  The CPU tests also check
hand-derived properties of the oracle; the GPU tests check the CUDA path against the oracle and
against the fixtures: IoU maps to 1e-5, masks exactly except on cells whose best IoU lies
within 1e-5 of the threshold (TF's float32 tanh / sigmoid / exp are Eigen's, the fixtures' are
libm's: neither side may claim more).
"""
import numpy as np
import pytest

from multigriddet_b200 import synth
from oracle import loss_oracle as LO
from oracle import mgd_oracle as O


def _inputs(seed, B, N, S, C, noise=0.05):
    import torch
    anchors = synth.coco_anchors(np.float32)
    boxes = synth.synth_boxes(seed, B, N, S, C)
    y = O.encode_targets(boxes, (S, S), anchors, C)
    preds = [p.numpy() for p in synth.planted_head_outputs([torch.from_numpy(a) for a in y], 3, seed)]
    rng = np.random.default_rng(seed)
    for p in preds:                                        # spread the IoUs away from 1
        p[..., 0:4] += rng.normal(0, noise, p[..., 0:4].shape).astype(np.float32)
    return anchors, y, preds


def test_oracle_properties():
    S, C = 160, 20
    anchors, y, preds = _inputs(0, 3, 8, S, C)
    for l, (ig, asg, mx) in enumerate(LO.ignore_masks(preds, y, anchors, (S, S))):
        pos = y[l][..., 4:5] > 0.5
        assert ig.shape == asg.shape == mx.shape == pos.shape and ig.dtype == np.float32
        assert not (ig[pos] != 0).any()                    # positives are never ignored
        assert set(np.unique(ig)) <= {0.0, 1.0}
        assert np.all(asg[~pos] == 0) and np.all(asg <= mx + 1e-7)
        assert np.all((mx >= 0) & (mx <= 1.0 + 1e-6))
        assert np.array_equal(ig[~pos] == 1, mx[~pos] > 0.5)
    # an image without boxes: every map is zero (multigrid_loss.py:634-642)
    empty = [np.zeros_like(t[:1]) for t in y]
    for ig, asg, mx in LO.ignore_masks([p[:1] for p in preds], empty, anchors, (S, S)):
        assert not ig.any() and not asg.any() and not mx.any()
    # a prediction that reproduces its own target exactly has IoU 1 with it:
    # raw xy = 0 activates to tanh(0) + sigmoid(0) = 0.5, raw wh = the stored log ratio
    t = np.zeros((1, 5, 5, 5 + 3 + C), np.float32)
    t[0, 2, 3, :5] = [0.5, 0.5, 0.1, -0.2, 1.0]
    t[0, 2, 3, 5 + 1] = 1.0
    p = np.zeros_like(t)
    p[0, 2, 3, 2:4] = [0.1, -0.2]
    ig, asg, mx = LO.ignore_mask_layer(p, t, anchors[0], (S, S))
    assert asg[0, 2, 3, 0] == pytest.approx(1.0, abs=1e-6) and ig[0, 2, 3, 0] == 0
    # the 'ij' meshgrid quirk: the ROW index feeds the x channel
    t2 = np.zeros_like(t); t2[0, 1, 4, :5] = [0.5, 0.5, 0.0, 0.0, 1.0]; t2[0, 1, 4, 5] = 1.0
    p2 = np.zeros_like(t)
    _, _, mx2 = LO.ignore_mask_layer(p2, t2, np.array([[8, 8], [4, 4], [2, 2]], np.float32), (S, S))
    best = np.unravel_index(np.argmax(mx2[0, ..., 0]), (5, 5))
    assert best == (1, 4)                                  # same tensor position: the offset is consistent


@pytest.mark.gpu
@pytest.mark.parametrize("seed,B,N,S,C", [(1, 6, 12, 160, 20), (2, 4, 60, 416, 20), (3, 3, 100, 608, 80)])
def test_gpu_ignore_mask_matches_oracle(seed, B, N, S, C):
    import torch
    from multigriddet_b200 import engine
    from multigriddet_b200.losses import compute_ignore_mask
    anchors, y, preds = _inputs(seed, B, N, S, C)
    ref = LO.ignore_masks(preds, y, anchors, (S, S), ignore_thresh=0.5)
    for dev in (False, True):
        yp = [torch.from_numpy(p).cuda() for p in preds] if dev else preds
        yt = [torch.from_numpy(t).cuda() for t in y] if dev else y
        got = engine.ignore_masks(yp, yt, anchors, (S, S), C, ignore_thresh=0.5)
        n_flagged = 0
        for (ig, asg, mx), (rig, rasg, rmx) in zip(got, ref):
            if dev:
                ig, asg, mx = ig.cpu().numpy(), asg.cpu().numpy(), mx.cpu().numpy()
            np.testing.assert_allclose(mx, rmx, rtol=1e-5, atol=1e-6)
            np.testing.assert_allclose(asg, rasg, rtol=1e-5, atol=1e-6)
            sure = np.abs(rmx - 0.5) > 1e-5
            assert np.array_equal(ig[sure], rig[sure])
            n_flagged += int(rig.sum())
        assert n_flagged > 0
    one = compute_ignore_mask(preds[1], y[1], anchors[1], (S, S))
    np.testing.assert_allclose(one[2], ref[1][2], rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
def test_ignore_mask_fed_by_the_encoder_table_equals_the_dense_path():
    """SURVEY 8f-2 as specified: mgd_encode_ignore_mask (owner table + box records feed the mask
    kernels) must give bit-identical masks and y_true to mgd_encode_targets + mgd_ignore_mask,
    also across the encoder's internal chunk boundary and with y_true switched off."""
    import os
    import torch
    from multigriddet_b200 import engine, synth
    S, C, B, N = 608, 80, 20, 60
    anchors = synth.coco_anchors(np.float32)
    boxes = torch.from_numpy(synth.synth_boxes(8, B, N, S, C, layout="mosaic")).cuda()
    y_ref = engine.encode_targets(boxes, (S, S), anchors, C)
    gen = torch.Generator(device="cuda"); gen.manual_seed(3)
    y_pred = [torch.randn(y.shape, generator=gen, device="cuda") for y in y_ref]
    m_ref = engine.ignore_masks(y_pred, y_ref, anchors, (S, S), C, 0.5)
    os.environ["MGD_ENCODE_CHUNK_IMAGES"] = "7"            # 20 images = chunks of 7, 7, 6
    try:
        y_got, m_got = engine.encode_ignore_masks(boxes, y_pred, anchors, (S, S), C, 0.5)
        none_y, m_got2 = engine.encode_ignore_masks(boxes, y_pred, anchors, (S, S), C, 0.5, want_y_true=False)
    finally:
        del os.environ["MGD_ENCODE_CHUNK_IMAGES"]
    assert none_y is None
    assert all(torch.equal(a, b) for a, b in zip(y_got, y_ref))
    # (the order of an image's ground-truth list depends on atomics, and the best pair is
    #  picked by cross-multiplication: equal pairs may round differently run to run -- the
    #  dense path has the same property, so compare like test_cuda_ignore_mask_matches_oracle)
    for got in (m_got, m_got2):
        for (gi, ga, gm), (ri, ra, rm) in zip(got, m_ref):
            assert float((gm - rm).abs().max()) < 1e-6 and float((ga - ra).abs().max()) < 1e-6
            clear = (rm - 0.5).abs() > 1e-5
            assert torch.equal(gi[clear], ri[clear])
    assert sum(float(m[0].sum()) for m in m_ref) > 0       # the mask is not trivially empty


def _golden_cases():
    import golden_util as G
    z = np.load(G.GOLDEN + "/ignoremask_cases.npz")
    for i in range(int(z["n_cases"])):
        seed, B, N, S, C = (int(v) for v in z[f"c{i}_meta"])
        anchors = [np.array(a, dtype=np.float32) for a in z[f"c{i}_anchors"]]
        y = G.dense_y_true(z, prefix=f"c{i}_y_")
        preds = [z[f"c{i}_pred{l}"].astype(np.float32) for l in range(3)]
        ref = []
        for l in range(3):
            shape = y[l].shape[:3] + (1,)
            ig = np.unpackbits(z[f"c{i}_ignore{l}"])[:int(np.prod(shape))].reshape(shape).astype(np.float32)
            ref.append((ig, z[f"c{i}_assigned{l}"], z[f"c{i}_maxiou{l}"]))
        yield S, C, anchors, y, preds, ref


def test_oracle_matches_reference_code_golden():
    """oracle/loss_oracle.py against the outputs of the reference's own _compute_ignore_mask
    (run over oracle/tf_shim.py when the fixture was made)."""
    import golden_util as G
    n = 0
    for S, C, anchors, y, preds, ref in _golden_cases():
        got = LO.ignore_masks(preds, y, anchors, (S, S), ignore_thresh=0.5)
        for (ig, asg, mx), (rig, rasg, rmx) in zip(got, ref):
            if G.numpy_pinned():
                assert np.array_equal(mx, rmx) and np.array_equal(asg, rasg) and np.array_equal(ig, rig)
            else:
                np.testing.assert_allclose(mx, rmx, rtol=1e-5, atol=1e-6)
                np.testing.assert_allclose(asg, rasg, rtol=1e-5, atol=1e-6)
                sure = np.abs(rmx - 0.5) > 1e-5
                assert np.array_equal(ig[sure], rig[sure])
            n += int(rig.sum())
    assert n > 1000


def test_oracle_matches_live_reference_code_over_tf_shim():
    """Fresh seeds: the two reference methods' own source executed over the TF-op stand-in
    against the restatement, bit for bit (both sides use the same float32 exp / tanh here),
    where the reference tree exists; everywhere against those outputs as stored in
    tests/golden/live_ignore_mask.npz."""
    import golden_util as G
    from oracle import ref_loader
    f = ref_loader.load_tf_ignore_mask() if ref_loader.available() else None
    rec = G.Recorded("ignore_mask")
    for seed, B, N, S, C, thr in ((11, 3, 12, 160, 20, 0.5), (12, 2, 60, 416, 20, 0.7), (13, 1, 100, 608, 80, 0.3)):
        anchors, y, preds = _inputs(seed, B, N, S, C)
        for l in range(3):
            got = LO.ignore_mask_layer(preds[l], y[l], anchors[l], (S, S), ignore_thresh=thr)
            if f is not None:
                ref = f(preds[l], y[l], anchors[l], (S, S), thr)
                for g, r in zip(got, ref):
                    assert g.shape == r.shape and np.array_equal(g, r)
            rec.check(f"s{seed}_l{l}", got)
    # an image without objects takes the reference's tf.cond zero branch (:634-642)
    anchors, y, preds = _inputs(14, 2, 5, 160, 20)
    y0 = [np.zeros_like(t) for t in y]
    for l in range(3):
        got = LO.ignore_mask_layer(preds[l], y0[l], anchors[l], (160, 160))
        if f is not None:
            for g, r in zip(got, f(preds[l], y0[l], anchors[l], (160, 160), 0.5)):
                assert np.array_equal(g, r)
        rec.check(f"empty_l{l}", got)
        assert not any(g.any() for g in got)


@pytest.mark.gpu
def test_gpu_ignore_mask_matches_reference_code_golden():
    """The CUDA path against the fixtures made from the reference's own code."""
    import torch
    from multigriddet_b200 import engine
    for S, C, anchors, y, preds, ref in _golden_cases():
        for dev in (False, True):
            yp = [torch.from_numpy(p).cuda() for p in preds] if dev else preds
            yt = [torch.from_numpy(t).cuda() for t in y] if dev else y
            got = engine.ignore_masks(yp, yt, anchors, (S, S), C, ignore_thresh=0.5)
            for (ig, asg, mx), (rig, rasg, rmx) in zip(got, ref):
                if dev:
                    ig, asg, mx = ig.cpu().numpy(), asg.cpu().numpy(), mx.cpu().numpy()
                np.testing.assert_allclose(mx, rmx, rtol=1e-5, atol=1e-6)
                np.testing.assert_allclose(asg, rasg, rtol=1e-5, atol=1e-6)
                sure = np.abs(rmx - 0.5) > 1e-5
                assert np.array_equal(ig[sure], rig[sure])
