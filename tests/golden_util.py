"""Readers for tests/golden/*.npz (written by oracle/gen_golden.py from the reference)."""
import glob
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def numpy_pinned():
    """True when NumPy's float32 exp/log/tanh are the libm ones the goldens were made with."""
    return os.environ.get("MGD_NUMPY_PIN_EFFECTIVE") == "1"


def files(prefix):
    return sorted(glob.glob(os.path.join(GOLDEN, prefix + "_*.npz")))


def anchors_of(z):
    dt = np.float64 if bool(z["anchors_f64"]) else np.float32
    return [np.array(a, dtype=dt) for a in z["anchors"]]


def dense_y_true(z, prefix=""):
    out = []
    l = 0
    while f"{prefix}shape{l}" in z:
        y = np.zeros(tuple(z[f"{prefix}shape{l}"]), dtype=np.float32)
        idx = z[f"{prefix}idx{l}"]
        y[idx[:, 0], idx[:, 1], idx[:, 2]] = z[f"{prefix}val{l}"]
        out.append(y)
        l += 1
    return out


def preds_of(z):
    out = []
    l = 0
    while f"pred{l}" in z:
        out.append(z[f"pred{l}"].astype(np.float32))
        l += 1
    return out


def knobs_of(z):
    for k in range(int(z["n_knobs"])):
        yield k, dict(image_shape=tuple(int(v) for v in z[f"k{k}_image_shape"]),
                      confidence=float(z[f"k{k}_conf"]), nms_threshold=float(z[f"k{k}_thr"]),
                      nms_method=str(z[f"k{k}_method"]), max_boxes=int(z[f"k{k}_max"]))


def assert_encode_matches(got, ref, exact_floats):
    for g, r in zip(got, ref):
        g = np.asarray(g)
        assert g.shape == r.shape and g.dtype == np.float32
        assert np.array_equal(g[..., 4:], r[..., 4:]), "mask / one-hot channels differ"
        assert np.array_equal(g[..., 0:2], r[..., 0:2]), "cell offsets differ"
        if exact_floats:
            assert np.array_equal(g[..., 2:4], r[..., 2:4])
        else:
            np.testing.assert_allclose(g[..., 2:4], r[..., 2:4], rtol=1e-5, atol=1e-6)


RECORD = os.environ.get("MGD_RECORD_REFERENCE_OUTPUTS") == "1"
_recording = {}


def _require_reference():
    from oracle import ref_loader
    if not ref_loader.available():
        raise RuntimeError("recording needs the reference tree: what is stored must be what the "
                           "test has just checked against the reference itself")


def _write_recordings():
    for path, rows in _recording.items():
        cols = list(zip(*sorted(rows.items(), key=lambda kv: kv[0])))
        names, fields = cols[0], list(zip(*cols[1]))
        np.savez_compressed(path, names=np.array(names), shapes=np.array(fields[0]),
                            dtypes=np.array(fields[1]), sha256=np.array(fields[2]))


def _fields(a):
    return ",".join(str(n) for n in a.shape), a.dtype.str, _digest(a)


def _digest(a):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


class Recorded:
    """The reference's outputs on the inputs of a live-reference test, kept in
    tests/golden/live_<name>.npz so that the comparison also runs where the reference tree is
    absent.  ``check(key, arrays)`` asserts that ``arrays`` (the case's inputs and the
    restatement's outputs for case ``key``) equal the stored ones bit for bit: what is stored of
    each array is its shape, dtype and the SHA-256 of its bytes, which keeps the fixtures small
    where the arrays themselves (y_true grids, dense decode tensors) are megabytes.

    To rewrite the files, run the tests with the reference tree present and
    MGD_RECORD_REFERENCE_OUTPUTS=1.  Every test compares the restatement with the live reference
    before it calls ``check``, so what gets written is the reference's output."""

    def __init__(self, name):
        self.path = os.path.join(GOLDEN, f"live_{name}.npz")
        self._rows = None

    def check(self, key, arrays):
        arrays = [np.asarray(a) for a in arrays]
        if RECORD:
            _require_reference()
            if not _recording:
                import atexit
                atexit.register(_write_recordings)
            rows = _recording.setdefault(self.path, {})
            for i, a in enumerate(arrays):
                rows[f"{key}/{i}"] = _fields(a)
            return
        if self._rows is None:
            z = np.load(self.path)
            self._rows = {str(n): (str(s), str(d), str(h))
                          for n, s, d, h in zip(z["names"], z["shapes"], z["dtypes"], z["sha256"])}
        assert f"{key}/{len(arrays)}" not in self._rows, (key, "more arrays stored than given")
        for i, a in enumerate(arrays):
            want = self._rows[f"{key}/{i}"]
            got = _fields(a)
            assert got[:2] == want[:2], (key, i, "shape / dtype", got[:2], want[:2])
            assert got[2] == want[2], (key, i, "values differ")


def coco608_inputs(c_oracle_encode):
    """Regenerate the inputs of coco608_detections.npz from their seeds (oracle/gen_golden.py:
    coco608_inputs / coco608_case) and check them against the stored SHA-256."""
    import hashlib
    import torch
    from multigriddet_b200 import synth
    S, C = 608, 80
    anchors = synth.coco_anchors(np.float32)
    boxes = synth.synth_boxes(400, 2, 100, S, C, anchors=anchors)
    y = c_oracle_encode(boxes, (S, S), anchors, C)
    preds = [p.numpy() for p in synth.planted_head_outputs([torch.from_numpy(a) for a in y], 3, seed=401)]
    h = hashlib.sha256()
    for p in preds:
        h.update(np.ascontiguousarray(p).tobytes())
    return S, C, anchors, preds, h.hexdigest()
