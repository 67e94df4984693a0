"""Generate ``tests/golden/*.npz`` by running the REAL reference from /root/reference.

    python -m oracle.gen_golden          (build container only; needs /root/reference)

Test infrastructure (see ``oracle/__init__.py``).  The fixtures pin the oracle
(``tests/test_oracle_golden.py``) and, on the GPU box where the reference does not
exist, the CUDA path (``tests/test_gpu_golden.py``).  NumPy runs with its AVX
dispatch disabled (``ref_loader.pin_numpy_env``) so ``argsort`` ties and the float32
transcendentals are the portable libm ones.

``tests/golden/live_*.npz`` are not written here: they hold digests of the reference's outputs
on the inputs of the live-reference tests and are rewritten by those tests
(``golden_util.Recorded``, ``MGD_RECORD_REFERENCE_OUTPUTS=1``).

Fixtures are kept small: y_true is stored sparsely (positive cells only), head
outputs are quantised to float16-representable values so they store in half the
space while every consumer sees the identical float32 tensor.
"""
from __future__ import annotations

import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader  # noqa: E402

ref_loader.pin_numpy_env()

import numpy as np  # noqa: E402
import torch  # noqa: E402

from multigriddet_b200 import synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

SMALL_FIRST = (((10, 13), (16, 30), (33, 23)), ((30, 61), (62, 45), (59, 119)),
               ((116, 90), (156, 198), (373, 326)))


def sparse(y_true):
    """positive-cell coordinates and rows of each layer"""
    out = {}
    for l, y in enumerate(y_true):
        nz = np.argwhere(np.any(y != 0, axis=-1))
        out[f"idx{l}"] = nz.astype(np.int32)
        out[f"val{l}"] = y[nz[:, 0], nz[:, 1], nz[:, 2]].astype(np.float32)
        out[f"shape{l}"] = np.array(y.shape, dtype=np.int32)
    return out


def encode_cases():
    enc = ref_loader.load_encoder()
    cases = [
        # name, S, C, N, B, layout, corners, padding, anchor dtype, anchor set
        ("voc416", 416, 20, 20, 8, "uniform", "int", "tail", np.float32, "coco"),
        ("coco608", 608, 80, 100, 3, "uniform", "int", "tail", np.float32, "coco"),
        ("coco608_f64", 608, 80, 100, 2, "uniform", "frac", "interleaved", np.float64, "coco"),
        ("mosaic320", 320, 80, 300, 2, "mosaic", "frac", "tail", np.float32, "coco"),
        ("mosaic512_f64", 512, 80, 300, 2, "mosaic", "int", "tail", np.float64, "coco"),
        ("oneclass352", 352, 1, 40, 2, "uniform", "frac", "tail", np.float32, "small_first"),
    ]
    for i, (name, S, C, N, B, layout, corners, padding, dt, aset) in enumerate(cases):
        anchors = (synth.coco_anchors(dt) if aset == "coco"
                   else [np.array(a, dtype=dt) for a in SMALL_FIRST])
        boxes = synth.synth_boxes(100 + i, B, N, S, C, corners=corners, layout=layout,
                                  padding=padding, anchors=anchors)
        y = enc(boxes.copy(), (S, S), anchors, C, False)
        np.savez_compressed(os.path.join(OUT, f"encode_{name}.npz"), boxes=boxes,
                            anchors=np.stack(anchors).astype(np.float64),
                            anchors_f64=np.array(dt == np.float64), S=S, C=C, **sparse(y))
        print("encode", name, [int(a[..., 4].sum()) for a in y])
    # known-answer single boxes (the inputs of the reference's own two hot-path tests)
    small_first = [np.array(a, dtype=np.float32) for a in SMALL_FIRST]
    ka = []
    for box, C in (([254, 264, 354, 344, 0], 1), ([100, 200, 180, 260, 2], 80),
                   ([271.999, 271.999, 351.999, 351.999, 0], 1)):
        b = np.array([[box]], dtype=np.float32)
        y = enc(b.copy(), (608, 608), small_first, C, False)
        ka.append((b, C, y))
    np.savez_compressed(os.path.join(OUT, "encode_known_answer.npz"),
                        anchors=np.stack(small_first).astype(np.float64),
                        **{f"box{i}": k[0] for i, k in enumerate(ka)},
                        **{f"C{i}": np.array(k[1]) for i, k in enumerate(ka)},
                        **{f"c{i}_{key}": v for i, k in enumerate(ka) for key, v in sparse(k[2]).items()})


def tf_adversarial_boxes(S, C):
    """Hand-made inputs for the points where the TF encoder differs from the NumPy one or where
    its scatter is order-dependent: two boxes with the same centre (the later one must win every
    shared cell), boxes whose 3x3 block leaves the grid on each side, centres exactly on a cell
    boundary, zero-area and inverted rows between valid ones, class ids outside [0, C)."""
    rows = [
        [100, 200, 180, 260, 3], [100, 200, 180, 260, 7],            # identical boxes, classes differ
        [96, 196, 184, 264, 1],                                      # same centre, other size (other anchor?)
        [0, 0, 40, 30, 2], [S - 30, S - 44, S, S, 4],                # corners of the image
        [0, S / 2 - 20, 24, S / 2 + 20, 5], [S / 2 - 9, 0, S / 2 + 9, 20, 6],
        [296, 296, 312, 312, 0],                                     # centre 304 = a stride-8/16/32 boundary
        [50, 50, 50, 90, 1], [300, 300, 280, 320, 1],                # zero area, inverted
        [200, 400, 330, 560, C], [210, 410, 320, 550, -1],           # class ids out of range
        [411.5, 97.25, 468.75, 171.5, C - 1],                        # fractional corners
        [0, 0, 0, 0, 0],
        [5, 5, S - 5, S - 5, 0],                                     # almost the whole image
    ]
    return np.array([rows], dtype=np.float32)


def tf_encode_cases():
    """The reference's TensorFlow encoder (generators.py:2696-3390) run over oracle/tf_shim.py."""
    enc = ref_loader.load_tf_encoder()
    cases = [
        # name, S, C, N, B, layout, corners, padding, anchor set
        ("coco608", 608, 80, 100, 2, "uniform", "int", "tail", "coco"),
        ("coco608_frac", 608, 80, 100, 2, "mosaic", "frac", "interleaved", "coco"),
        ("voc416", 416, 20, 30, 3, "uniform", "frac", "tail", "coco"),
        ("oneclass352", 352, 1, 40, 2, "mosaic", "frac", "tail", "small_first"),
    ]
    for i, (name, S, C, N, B, layout, corners, padding, aset) in enumerate(cases):
        anchors = (synth.coco_anchors(np.float32) if aset == "coco"
                   else [np.array(a, dtype=np.float32) for a in SMALL_FIRST])
        boxes = synth.synth_boxes(500 + i, B, N, S, C, corners=corners, layout=layout,
                                  padding=padding, anchors=anchors)
        grids = [(S // 32, S // 32), (S // 16, S // 16), (S // 8, S // 8)]
        y = enc(boxes.copy(), (S, S), anchors, C, grids)
        np.savez_compressed(os.path.join(OUT, f"tfencode_{name}.npz"), boxes=boxes,
                            anchors=np.stack(anchors).astype(np.float64),
                            anchors_f64=np.array(False), S=S, C=C, **sparse(y))
        print("tf encode", name, [int(a[..., 4].sum()) for a in y])
    S, C = 608, 80
    anchors = synth.coco_anchors(np.float32)
    boxes = tf_adversarial_boxes(S, C)
    y = enc(boxes.copy(), (S, S), anchors, C, [(19, 19), (38, 38), (76, 76)])
    np.savez_compressed(os.path.join(OUT, "tfencode_adversarial608.npz"), boxes=boxes,
                        anchors=np.stack(anchors).astype(np.float64), anchors_f64=np.array(False),
                        S=S, C=C, **sparse(y))
    print("tf encode adversarial", [int(a[..., 4].sum()) for a in y])


def ignoremask_inputs(seed, B, N, S, C, noise=0.05):
    """Targets from the reference's NumPy encoder, planted head outputs with noisy boxes
    (IoUs spread over (0, 1)); float16-rounded so the fixture stays small."""
    enc = ref_loader.load_encoder()
    anchors = synth.coco_anchors(np.float32)
    boxes = synth.synth_boxes(seed, B, N, S, C, anchors=anchors)
    y = enc(boxes.copy(), (S, S), anchors, C, False)
    preds = [p.numpy() for p in synth.planted_head_outputs([torch.from_numpy(a) for a in y], 3, seed)]
    rng = np.random.default_rng(seed)
    for p in preds:
        p[..., 0:4] += rng.normal(0, noise, p[..., 0:4].shape).astype(np.float32)
    preds = [p.astype(np.float16).astype(np.float32) for p in preds]
    return anchors, y, preds


def ignoremask_cases():
    """The reference's loss-side ignore mask (losses/multigrid_loss.py:445-703) run over
    oracle/tf_shim.py: ``MultiGridLoss._compute_ignore_mask`` per layer, called like :285-320."""
    f = ref_loader.load_tf_ignore_mask()
    store = {}
    cases = [(600, 3, 10, 160, 4), (601, 2, 40, 320, 20)]
    store["n_cases"] = np.array(len(cases))
    for i, (seed, B, N, S, C) in enumerate(cases):
        anchors, y, preds = ignoremask_inputs(seed, B, N, S, C)
        store[f"c{i}_meta"] = np.array([seed, B, N, S, C])
        store[f"c{i}_anchors"] = np.stack(anchors).astype(np.float64)
        for key, v in sparse(y).items():
            store[f"c{i}_y_{key}"] = v
        n_ignored = 0
        for l in range(3):
            store[f"c{i}_pred{l}"] = preds[l].astype(np.float16)
            ig, asg, mx = f(preds[l], y[l], anchors[l], (S, S), 0.5)
            store[f"c{i}_ignore{l}"] = np.packbits(ig.astype(np.uint8).reshape(-1))
            store[f"c{i}_assigned{l}"] = asg
            store[f"c{i}_maxiou{l}"] = mx
            n_ignored += int(ig.sum())
        print("ignore mask case", i, "ignored cells", n_ignored)
    np.savez_compressed(os.path.join(OUT, "ignoremask_cases.npz"), **store)


def tfboxes_inputs(seed, n_cases, cap=12):
    """Random raw annotation boxes, source image sizes, multi-scale shapes, flips, capacity
    factors for the tf.data box pre-step."""
    rng = np.random.default_rng(seed)
    cases = []
    for t in range(n_cases):
        src_h, src_w = int(rng.integers(120, 1600)), int(rng.integers(120, 1600))
        S = int(rng.choice([320, 416, 608]))
        n = int(rng.integers(0, cap + 1))
        x1 = rng.uniform(0, src_w - 2, n)
        y1 = rng.uniform(0, src_h - 2, n)
        x2 = np.minimum(x1 + rng.uniform(1, src_w, n), src_w)
        y2 = np.minimum(y1 + rng.uniform(1, src_h, n), src_h)
        boxes = np.zeros((cap, 5), np.float32)
        boxes[:n] = np.stack([x1, y1, x2, y2, rng.integers(0, 80, n)], 1)
        if t % 4 == 0:
            boxes[:n, :4] = np.round(boxes[:n, :4])              # integer annotations, the common case
        ms = (0, 0) if t % 3 else (int(rng.choice([320, 352, 416, 480, 608, 672])),) * 2
        cases.append((boxes, n, (src_h, src_w), S, ms, bool(rng.integers(0, 2)), int(rng.choice([1, 2, 4, 8]))))
    return cases


def tfboxes_cases():
    """The box side of the reference's tf.data pipeline (generators.py:167-256, 1859-2034) run
    over oracle/tf_shim.py."""
    f = ref_loader.load_tf_box_prestep()
    cases = tfboxes_inputs(700, 48)
    store = {"n_cases": np.array(len(cases)), "cap": np.array(12)}
    for i, (boxes, n, src, S, ms, flip, exp) in enumerate(cases):
        store[f"c{i}_boxes"] = boxes
        store[f"c{i}_meta"] = np.array([n, src[0], src[1], S, ms[0], ms[1], int(flip), exp])
        store[f"c{i}_out"] = f(boxes[:n], src, (S, S), 12, exp, ms if ms[0] else None, flip)
    np.savez_compressed(os.path.join(OUT, "tfboxes_cases.npz"), **store)
    print("tf.data box cases", len(cases))


def decode_cases():
    post = ref_loader.load_postprocess()
    enc = ref_loader.load_encoder()
    cases = [
        # name, S, C, B, N, anchor dtype
        ("voc416", 416, 20, 2, 20, np.float32),
        ("coco160", 160, 80, 3, 12, np.float32),
        ("coco160_f64", 160, 80, 2, 12, np.float64),
    ]
    knobs = [
        dict(image_shape=None, confidence=0.001, nms_threshold=0.45, nms_method="diou", max_boxes=100),
        dict(image_shape=(480, 640), confidence=0.1, nms_threshold=0.45, nms_method="diou", max_boxes=100),
        dict(image_shape=(1080, 1920), confidence=0.001, nms_threshold=0.5, nms_method="cluster", max_boxes=5),
        dict(image_shape=(375, 500), confidence=0.3, nms_threshold=0.3, nms_method="diou", max_boxes=100),
        dict(image_shape=(480, 640), confidence=0.001, nms_threshold=0.45, nms_method="soft", max_boxes=100),
        dict(image_shape=None, confidence=0.001, nms_threshold=0.45, nms_method="soft", max_boxes=4),
        dict(image_shape=(427, 640), confidence=0.001, nms_threshold=0.55, nms_method="wbf", max_boxes=100),
        dict(image_shape=None, confidence=0.05, nms_threshold=0.4, nms_method="wbf", max_boxes=3),
    ]
    for i, (name, S, C, B, N, dt) in enumerate(cases):
        anchors = synth.coco_anchors(dt)
        boxes = synth.synth_boxes(200 + i, B, N, S, C, anchors=anchors)
        y = enc(boxes.copy(), (S, S), anchors, C, False)
        preds = synth.planted_head_outputs([torch.from_numpy(a) for a in y], 3, seed=300 + i)
        preds16 = [p.numpy().astype(np.float16) for p in preds]
        preds = [p.astype(np.float32) for p in preds16]
        dec = post.MultiGridDecoder(anchors, C, input_shape=(S, S))
        store = {"anchors": np.stack(anchors).astype(np.float64),
                 "anchors_f64": np.array(dt == np.float64), "S": S, "C": C,
                 "n_knobs": len(knobs)}
        for l, p in enumerate(preds16):
            store[f"pred{l}"] = p
        dense = dec.decode_predictions([p.copy() for p in preds])
        store["dense_sample_rows"] = np.arange(0, dense.shape[1], 37)
        store["dense_sample"] = dense[:, ::37, :]
        for k, kn in enumerate(knobs):
            ishape = kn["image_shape"] or (S, S)
            store[f"k{k}_image_shape"] = np.array(ishape)
            store[f"k{k}_conf"] = np.array(kn["confidence"])
            store[f"k{k}_thr"] = np.array(kn["nms_threshold"])
            store[f"k{k}_method"] = np.array(kn["nms_method"])
            store[f"k{k}_max"] = np.array(kn["max_boxes"])
            ties = 0
            for b in range(B):
                one = [p[b:b + 1].copy() for p in preds]
                for xyxy in (True, False):
                    bx, cl, sc = dec.postprocess(one, ishape, (S, S), max_boxes=kn["max_boxes"],
                                                 confidence=kn["confidence"],
                                                 nms_threshold=kn["nms_threshold"],
                                                 nms_method="diou" if kn["nms_method"] == "wbf" else kn["nms_method"],
                                                 use_wbf=kn["nms_method"] == "wbf", return_xyxy=xyxy)
                    tag = "xyxy" if xyxy else "xywh"
                    store[f"k{k}_b{b}_{tag}"] = np.asarray(bx)
                store[f"k{k}_b{b}_classes"] = np.asarray(cl)
                store[f"k{k}_b{b}_scores"] = np.asarray(sc)
                ties += int(len(sc) - len(np.unique(sc)))
            print("decode", name, "knob", k, "dets", [len(store[f"k{k}_b{b}_scores"]) for b in range(B)],
                  "equal-score detections", ties)
        np.savez_compressed(os.path.join(OUT, f"decode_{name}.npz"), **store)


def nms_cases():
    post = ref_loader.load_postprocess()
    rng = np.random.default_rng(7)
    store = {}
    for i, n in enumerate((1, 7, 120, 900)):
        xy = rng.uniform(0, 400, size=(n, 2))
        wh = rng.uniform(4, 150, size=(n, 2))
        boxes = np.concatenate([xy, wh], 1)
        scores = rng.uniform(0.01, 1, size=n)          # distinct with probability 1
        classes = rng.integers(0, 6, size=n)
        store[f"n{i}_boxes"], store[f"n{i}_scores"], store[f"n{i}_classes"] = boxes, scores, classes
        for name, cls in (("diou", post.DIoUNMS), ("standard", post.StandardNMS), ("cluster", post.ClusterNMS)):
            for thr in (0.3, 0.5):
                kb, kc, ks = cls().apply_nms(boxes, classes, scores, thr, 0.0)
                store[f"n{i}_{name}_{thr}_scores"] = ks[0]
                store[f"n{i}_{name}_{thr}_boxes"] = kb[0]
        half = n // 2
        for ct in ("avg", "max", "box_and_model_avg"):
            fb, fc, fs = post.WeightedBoxesFusion(iou_thr=0.4, skip_box_thr=0.05, conf_type=ct).fuse_boxes(
                [boxes[:half], boxes[half:]], [classes[:half], classes[half:]],
                [scores[:half], scores[half:]], (600, 600), weights=[1.0, 0.6])
            store[f"n{i}_wbf_{ct}_boxes"] = fb[0] if fb else np.zeros((0, 4))
            store[f"n{i}_wbf_{ct}_scores"] = fs[0] if fs else np.zeros((0,))
            store[f"n{i}_wbf_{ct}_classes"] = fc[0] if fc else np.zeros((0,), np.int64)
        for sigma in (0.5, 0.1):
            kb, kc, ks = post.SoftNMS(sigma=sigma).apply_nms(boxes, classes, scores, 0.5, 0.0)
            store[f"n{i}_soft_{sigma}_scores"] = ks[0]
            store[f"n{i}_soft_{sigma}_boxes"] = kb[0]
    np.savez_compressed(os.path.join(OUT, "nms_cases.npz"), **store)
    print("nms cases written")


def reference_per_class(post, dec, boxes, classes, scores, thr, nms_cls, max_boxes):
    """Per-class NMS out of reference code only (SURVEY 8a-9): partition by class, the
    reference's greedy NMS per partition (nms.py:83-187), concatenate, ``_filter_boxes``
    top-k (multigrid_decode.py:322-345).  Returned in descending-score order."""
    kb, kc, ks = [], [], []
    for c in np.unique(classes):
        m = classes == c
        b, cl, sc = nms_cls().apply_nms(boxes[m], classes[m], scores[m], thr, 0.0)
        if b:
            kb.append(b[0]); kc.append(cl[0]); ks.append(sc[0])
    if not kb:
        return np.zeros((0, 4)), np.zeros((0,), np.int64), np.zeros((0,))
    b, c, sc = dec._filter_boxes(np.concatenate(kb), np.concatenate(kc), np.concatenate(ks), max_boxes)
    order = np.argsort(-sc, kind="stable")
    return b[order], c[order], sc[order]


def perclass_cases():
    """tests/golden/perclass_cases.npz: per-class NMS composed of reference code, on the
    explicit boxes of nms_cases.npz and on a COCO-608 head (the north star's own wording)."""
    post = ref_loader.load_postprocess()
    enc = ref_loader.load_encoder()
    z = np.load(os.path.join(OUT, "nms_cases.npz"))
    dec = post.MultiGridDecoder(synth.coco_anchors(np.float32), 80)
    store = {}
    i = 0
    while f"n{i}_boxes" in z:
        boxes, scores, classes = z[f"n{i}_boxes"], z[f"n{i}_scores"], z[f"n{i}_classes"]
        for name, cls in (("diou", post.DIoUNMS), ("standard", post.StandardNMS)):
            for thr in (0.3, 0.5):
                for mx in (1000, 20):
                    b, c, sc = reference_per_class(post, dec, boxes, classes, scores, thr, cls, mx)
                    store[f"n{i}_{name}_{thr}_{mx}_boxes"] = b
                    store[f"n{i}_{name}_{thr}_{mx}_classes"] = c
                    store[f"n{i}_{name}_{thr}_{mx}_scores"] = sc
        i += 1
    np.savez_compressed(os.path.join(OUT, "perclass_cases.npz"), **store)
    print("per-class NMS cases written:", i)


def coco608_inputs(B=2, N=100, seed=400):
    """Deterministic COCO-608 head outputs (regenerated bit-identically by the tests from the
    same seeds: nothing of the 2.67 MB / image tensor is stored)."""
    S, C = 608, 80
    anchors = synth.coco_anchors(np.float32)
    boxes = synth.synth_boxes(seed, B, N, S, C, anchors=anchors)
    return S, C, anchors, boxes


def coco608_case():
    """tests/golden/coco608_detections.npz: the reference's detections on a full-size COCO head
    (class-agnostic DIoU and per-class mode), plus sampled rows of its dense decode tensor.
    Inputs are regenerated from seeds; a SHA-256 of the head tensor guards that."""
    import hashlib
    post = ref_loader.load_postprocess()
    enc = ref_loader.load_encoder()
    S, C, anchors, boxes = coco608_inputs()
    y = enc(boxes.copy(), (S, S), anchors, C, False)
    preds = [p.numpy() for p in synth.planted_head_outputs([torch.from_numpy(a) for a in y], 3, seed=401)]
    h = hashlib.sha256()
    for p in preds:
        h.update(np.ascontiguousarray(p).tobytes())
    dec = post.MultiGridDecoder(anchors, C, input_shape=(S, S))
    store = {"sha256": np.array(h.hexdigest()), "S": S, "C": C, "B": len(boxes)}
    dense = dec.decode_predictions([p.copy() for p in preds])
    store["dense_sample_rows"] = np.arange(0, dense.shape[1], 97)
    store["dense_sample"] = dense[:, ::97, :]
    knobs = [dict(image_shape=(608, 608), confidence=0.001, nms_threshold=0.45, max_boxes=100),
             dict(image_shape=(480, 640), confidence=0.1, nms_threshold=0.45, max_boxes=100),
             dict(image_shape=(1080, 1920), confidence=0.001, nms_threshold=0.5, max_boxes=30)]
    store["n_knobs"] = len(knobs)
    for k, kn in enumerate(knobs):
        for key, v in kn.items():
            store[f"k{k}_{key}"] = np.array(v)
        for b in range(len(boxes)):
            one = [p[b:b + 1].copy() for p in preds]
            bx, cl, sc = dec.postprocess(one, kn["image_shape"], (S, S), max_boxes=kn["max_boxes"],
                                         confidence=kn["confidence"], nms_threshold=kn["nms_threshold"],
                                         nms_method="diou")
            store[f"k{k}_b{b}_xyxy"], store[f"k{k}_b{b}_classes"], store[f"k{k}_b{b}_scores"] = \
                np.asarray(bx), np.asarray(cl), np.asarray(sc)
            # per-class mode: reference decode + letterbox + threshold (:262-278), then the
            # per-partition composition, then _convert_to_xyxy (:397-422)
            corrected = dec.correct_boxes(dec.decode_predictions(one), kn["image_shape"], (S, S))
            cls_all = np.argmax(corrected[..., 5:], axis=-1)
            pos = np.where(corrected[..., 4] >= kn["confidence"])
            cb, cc, cs = corrected[..., 0:4][pos], cls_all[pos], corrected[..., 4][pos]
            pb, pc, ps = reference_per_class(post, dec, cb, cc, cs, kn["nms_threshold"], post.DIoUNMS,
                                             kn["max_boxes"])
            store[f"k{k}_b{b}_pc_xyxy"] = dec._convert_to_xyxy(pb, kn["image_shape"]) if len(pb) else np.zeros((0, 4), np.int32)
            store[f"k{k}_b{b}_pc_classes"] = pc
            store[f"k{k}_b{b}_pc_scores"] = ps
            store[f"k{k}_b{b}_candidates"] = np.array(len(cs))
        print("coco608 knob", k, "dets", [len(store[f"k{k}_b{b}_scores"]) for b in range(len(boxes))],
              "per-class", [len(store[f"k{k}_b{b}_pc_scores"]) for b in range(len(boxes))])
    np.savez_compressed(os.path.join(OUT, "coco608_detections.npz"), **store)


def synth_eval_set(seed, B, M, N, C, ties=False):
    """Padded detections / ground truth shaped like an evaluation run: detections are
    jittered copies of ground-truth boxes (int32 xyxy like _convert_to_xyxy emits) with
    mostly-correct classes, ground truth is float xyxy."""
    rng = np.random.default_rng(seed)
    gtb = np.zeros((B, N, 4)); gtc = np.zeros((B, N), np.int32); gtn = rng.integers(0, N + 1, B).astype(np.int32)
    db = np.zeros((B, M, 4)); ds = np.zeros((B, M)); dc = np.zeros((B, M), np.int32)
    dn = rng.integers(0, M + 1, B).astype(np.int32)
    for b in range(B):
        xy = rng.uniform(0, 400, (N, 2)); wh = np.exp(rng.normal(np.log(60), 0.9, (N, 2))).clip(6, 300)
        gtb[b] = np.concatenate([xy, xy + wh], 1)
        gtc[b] = rng.integers(0, C, N)
        for i in range(M):
            j = int(rng.integers(0, N))
            db[b, i] = np.round(gtb[b, j] + rng.normal(0, 0.12, 4) * np.tile(wh[j], 2))
            dc[b, i] = gtc[b, j] if rng.random() < 0.8 else rng.integers(0, C)
        ds[b] = np.round(rng.uniform(0.05, 1, M), 2) if ties else rng.uniform(0.001, 1, M)
    return db, ds, dc, dn, gtb, gtc, gtn


def metrics_cases():
    """tests/golden/metrics_cases.npz: the reference's matcher flags, APs and calculate_map
    results (multigriddet/evaluation/metrics.py) on synthetic evaluation sets."""
    import contextlib, io
    from oracle import metrics_oracle as MO
    M = ref_loader.load_metrics()
    store = {}
    thr = [0.5, 0.55, 0.6, 0.65, 0.7, 0.75, 0.8, 0.85, 0.9, 0.95]
    cases = [("a", 1, 12, 40, 15, 5, False), ("b", 2, 5, 100, 30, 3, False), ("ties", 3, 8, 12, 6, 2, True)]
    store["names"] = np.array([c[0] for c in cases])
    store["thresholds"] = np.array(thr)
    for name, seed, B, Mx, N, C, ties in cases:
        db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(seed, B, Mx, N, C, ties)
        preds, gts = MO.to_dicts(db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
        for k, v in (("db", db), ("ds", ds), ("dc", dc), ("dn", dn), ("gtb", gtb), ("gtc", gtc), ("gtn", gtn)):
            store[f"{name}_{k}"] = v
        store[f"{name}_C"] = np.array(C)
        for cached in (True, False):
            tag = "cached" if cached else "plain"
            for c in range(C):
                cp = [p for p in preds if p["class"] == c]
                cg = [g for g in gts if g["class"] == c]
                cache = M.compute_iou_cache_for_class(preds, gts, c) if cached else None
                for t, th in enumerate(thr):
                    if cp:
                        r = (M.match_predictions_to_gt_cached(cp, cg, th, cache) if cached
                             else M.match_predictions_to_gt(cp, cg, th))
                        store[f"{name}_{tag}_c{c}_t{t}_tp"] = np.asarray(r[0], bool)
                        store[f"{name}_{tag}_c{c}_t{t}_scores"] = np.asarray(r[2], np.float64)
                    ap = (M.calculate_ap_for_class_cached(preds, gts, c, th, cache) if cached
                          else M.calculate_ap_for_class(preds, gts, c, th))
                    store[f"{name}_{tag}_c{c}_t{t}_ap"] = np.array(float(ap))
            with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
                res = M.calculate_map(preds, gts, C, use_parallel=False, cache_ious=cached)
                res_voc = M.calculate_map(preds, gts, C, iou_thresholds=[0.5], method="voc",
                                          use_parallel=False, cache_ious=cached, compute_per_scale=False)
            for key in ("mAP", "mAP50", "mAP75", "APS", "APM", "APL", "APS50", "APM50", "APL50"):
                store[f"{name}_{tag}_map_{key}"] = np.array(float(res[key]))
            store[f"{name}_{tag}_map_voc50"] = np.array(float(res_voc["mAP50"]))
            print("metrics", name, tag, {k: round(float(res[k]), 4) for k in ("mAP", "mAP50", "APS", "APM", "APL")})
        n1, n2 = int(dn[0]), int(gtn[0])
        store[f"{name}_ioumat"] = M.calculate_iou_matrix(db[0, :max(n1, 1)], gtb[0, :max(n2, 1)])
    np.savez_compressed(os.path.join(OUT, "metrics_cases.npz"), **store)


def synth_box_transform_cases(seed, n_cases, N=24):
    """Random inputs for reshape_boxes / merge_mosaic_bboxes (shared by the golden generator
    and the tests)."""
    rng = np.random.default_rng(seed)
    reshape, mosaic = [], []
    for _ in range(n_cases):
        n = int(rng.integers(0, N + 1))
        sw, sh = int(rng.integers(200, 1400)), int(rng.integers(200, 1400))
        tw = th = int(rng.choice([320, 416, 608]))
        pw, ph = int(rng.integers(100, int(tw * 1.3))), int(rng.integers(100, int(th * 1.3)))
        dx, dy = int(rng.integers(-120, 200)), int(rng.integers(-120, 200))
        xy = rng.uniform(0, [sw, sh], (n, 2)); wh = rng.uniform(1, [sw / 2, sh / 2], (n, 2))
        b = np.concatenate([xy, np.minimum(xy + wh, [sw, sh]), rng.integers(0, 80, (n, 1))], 1)
        reshape.append(dict(boxes=b, src=(sw, sh), target=(tw, th), padding=(pw, ph), offset=(dx, dy),
                            hflip=bool(rng.integers(0, 2)), vflip=bool(rng.integers(0, 2))))
        bx = np.zeros((4, N, 5))
        for q in range(4):
            m = int(rng.integers(0, N + 1))
            xy = rng.uniform(0, tw, (m, 2)); wh = np.exp(rng.normal(np.log(50), 1.0, (m, 2))).clip(2, tw)
            bx[q, :m] = np.concatenate([xy, np.minimum(xy + wh, tw), rng.integers(0, 80, (m, 1))], 1)
        mosaic.append(dict(boxes=bx, crop=(int(rng.integers(int(tw * .2), int(tw * .8))),
                                           int(rng.integers(int(th * .2), int(th * .8)))), size=(th, tw)))
    return reshape, mosaic


def boxes_cases():
    """tests/golden/boxes_cases.npz: the reference's reshape_boxes (shuffle disabled) and
    merge_mosaic_bboxes on random inputs."""
    R = ref_loader.load_box_transforms()
    reshape, mosaic = synth_box_transform_cases(77, 40)
    store = {"n_cases": np.array(len(reshape))}
    for i, c in enumerate(reshape):
        for tag, dt in (("i32", np.int32), ("f64", np.float64)):
            out = R.reshape_boxes(c["boxes"].astype(dt), c["src"], c["target"], c["padding"], c["offset"],
                                  c["hflip"], c["vflip"])
            store[f"r{i}_{tag}"] = np.asarray(out).reshape(-1, 5)
    for i, c in enumerate(mosaic):
        store[f"m{i}"] = R.merge_mosaic_bboxes(c["boxes"], c["crop"][0], c["crop"][1], c["size"])
    np.savez_compressed(os.path.join(OUT, "boxes_cases.npz"), **store)
    print("boxes cases written:", sum(len(store[f"r{i}_i32"]) for i in range(len(reshape))), "reshaped rows,",
          sum(int((store[f"m{i}"][:, 2] > 0).sum()) for i in range(len(mosaic))), "mosaic rows")


if __name__ == "__main__":
    if not ref_loader.available():
        raise SystemExit("reference tree not found at " + ref_loader.REFERENCE_ROOT)
    os.makedirs(OUT, exist_ok=True)
    only = sys.argv[1:] or ["encode", "tfencode", "ignoremask", "tfboxes", "decode", "nms", "metrics", "boxes", "perclass", "coco608"]
    if "encode" in only:
        encode_cases()
    if "tfencode" in only:
        tf_encode_cases()
    if "ignoremask" in only:
        ignoremask_cases()
    if "tfboxes" in only:
        tfboxes_cases()
    if "decode" in only:
        decode_cases()
    if "nms" in only:
        nms_cases()
    if "metrics" in only:
        metrics_cases()
    if "boxes" in only:
        boxes_cases()
    if "perclass" in only:
        perclass_cases()
    if "coco608" in only:
        coco608_case()
    total = sum(os.path.getsize(os.path.join(OUT, f)) for f in os.listdir(OUT))
    print(f"golden fixtures: {total / 1e6:.2f} MB in {OUT}")
