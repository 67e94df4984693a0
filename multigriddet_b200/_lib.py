"""ctypes binding of ``libmgd.so`` (the C ABI in ``include/mgd.h``).

This is the only place the Python drop-ins touch native code.  There is no CPU
or NumPy fallback: if the library is missing, or no B200 is visible, every
compute call raises.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmgd.so")

MGD_MAX_LAYERS = 5
MGD_MAX_ANCHORS_PER_LAYER = 8
MEM_HOST, MEM_DEVICE = 0, 1
FLAG_SYNC = 1
FLAG_TF_COMPAT = 2
FLAG_HOST_ZEROCOPY = 4
NMS_IOU, NMS_DIOU, NMS_SOFT, NMS_WBF = 0, 1, 2, 3
IOU_CORNER, IOU_CENTRE = 0, 1
BOXES_I32, BOXES_F64 = 0, 1

MAP_MAX_THRESHOLDS, MAP_VOC_POINTS = 32, 11
MAP_MAX_CONFIDENCES = 32
MAP_COCO, MAP_VOC = 0, 1
MAP_VIEW_CORNER, MAP_VIEW_CENTRE, MAP_VIEW_S, MAP_VIEW_M, MAP_VIEW_L, MAP_VIEWS = range(6)

OK, ERR_INVALID_ARGUMENT, ERR_CLASS_RANGE, ERR_CUDA, ERR_NO_DEVICE, ERR_UNSUPPORTED = range(6)


class HeadConfig(ctypes.Structure):
    """``mgd_head_config``"""
    _fields_ = [
        ("num_layers", ctypes.c_int),
        ("num_classes", ctypes.c_int),
        ("input_h", ctypes.c_int),
        ("input_w", ctypes.c_int),
        ("grid_h", ctypes.c_int * MGD_MAX_LAYERS),
        ("grid_w", ctypes.c_int * MGD_MAX_LAYERS),
        ("num_anchors", ctypes.c_int * MGD_MAX_LAYERS),
        ("anchors", ((ctypes.c_double * 2) * MGD_MAX_ANCHORS_PER_LAYER) * MGD_MAX_LAYERS),
        ("anchors_f64", ctypes.c_int),
    ]


class PostConfig(ctypes.Structure):
    """``mgd_post_config``"""
    _fields_ = [
        ("use_softmax", ctypes.c_int),
        ("rescore_confidence", ctypes.c_int),
        ("confidence", ctypes.c_double),
        ("nms_threshold", ctypes.c_double),
        ("nms_method", ctypes.c_int),
        ("per_class", ctypes.c_int),
        ("max_boxes", ctypes.c_int),
        ("soft_sigma", ctypes.c_double),
        ("soft_score_threshold", ctypes.c_double),
    ]


class MapConfig(ctypes.Structure):
    """``mgd_map_config``"""
    _fields_ = [
        ("num_classes", ctypes.c_int),
        ("num_thresholds", ctypes.c_int),
        ("method", ctypes.c_int),
        ("views", ctypes.c_int),
        ("iou_thresholds", ctypes.c_double * MAP_MAX_THRESHOLDS),
        ("voc_recalls", ctypes.c_double * MAP_VOC_POINTS),
    ]


class MapPr(ctypes.Structure):
    """``mgd_map_pr``"""
    _fields_ = [
        ("views", ctypes.c_int),
        ("num_confidences", ctypes.c_int),
        ("confidences", ctypes.c_void_p),
        ("capacity", ctypes.c_longlong),
        ("offsets", ctypes.c_void_p),
        ("scores", ctypes.c_void_p),
        ("precision", ctypes.c_void_p),
        ("recall", ctypes.c_void_p),
        ("best_f1", ctypes.c_void_p),
        ("best_index", ctypes.c_void_p),
        ("at_confidence", ctypes.c_void_p),
    ]


class MgdError(RuntimeError):
    pass


_lib = None

_FP = ctypes.POINTER(ctypes.c_float)
_DP = ctypes.POINTER(ctypes.c_double)
_IP = ctypes.POINTER(ctypes.c_int)
_LLP = ctypes.POINTER(ctypes.c_longlong)

EXPORTS = ("mgd_version", "mgd_last_error", "mgd_device_count", "mgd_encode_targets",
           "mgd_decode_nms", "mgd_decode_dense", "mgd_nms", "mgd_soft_nms", "mgd_wbf", "mgd_poll_status",
           "mgd_encode_targets_dlpack", "mgd_decode_nms_dlpack", "mgd_profile_begin",
           "mgd_profile_end", "mgd_match_detections", "mgd_iou_matrix", "mgd_host_alloc",
           "mgd_host_free", "mgd_release_workspace", "mgd_reshape_boxes", "mgd_mosaic_merge_boxes",
           "mgd_ignore_mask", "mgd_encode_decode_nms", "mgd_letterbox_boxes",
           "mgd_encode_ignore_mask", "mgd_exchange_create", "mgd_exchange_connect",
           "mgd_exchange_buffer", "mgd_exchange_timeouts", "mgd_exchange_destroy",
           "mgd_map_record_bytes", "mgd_map_update", "mgd_map_compute", "mgd_map_partition",
           "mgd_map_compute_merged", "mgd_map_compute_pr", "mgd_map_compute_merged_pr")

IPC_HANDLE_BYTES = 64


def load():
    """Load ``libmgd.so`` (building it is ``__graft_entry__.build()``'s job)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise MgdError(
            f"{LIB_PATH} not found: build it with `python -m multigriddet_b200.build` "
            "(needs nvcc).  multigriddet_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.mgd_version.restype = ctypes.c_int
    lib.mgd_last_error.restype = ctypes.c_char_p
    lib.mgd_device_count.restype = ctypes.c_int
    lib.mgd_encode_targets.restype = ctypes.c_int
    lib.mgd_encode_targets.argtypes = [
        ctypes.POINTER(HeadConfig), ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
        ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
        ctypes.c_int, _LLP]
    lib.mgd_decode_nms.restype = ctypes.c_int
    lib.mgd_decode_nms.argtypes = [
        ctypes.POINTER(HeadConfig), ctypes.POINTER(PostConfig),
        ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_void_p,
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, _LLP]
    lib.mgd_encode_decode_nms.restype = ctypes.c_int
    lib.mgd_encode_decode_nms.argtypes = [
        ctypes.POINTER(HeadConfig), ctypes.POINTER(PostConfig),
        ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p),
        ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_void_p,
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    lib.mgd_decode_dense.restype = ctypes.c_int
    lib.mgd_decode_dense.argtypes = [
        ctypes.POINTER(HeadConfig), ctypes.POINTER(PostConfig),
        ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    lib.mgd_nms.restype = ctypes.c_int
    lib.mgd_nms.argtypes = [
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_double,
        ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    lib.mgd_wbf.restype = ctypes.c_int
    lib.mgd_wbf.argtypes = [
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
        ctypes.c_double, ctypes.c_double, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    lib.mgd_soft_nms.restype = ctypes.c_int
    lib.mgd_soft_nms.argtypes = [
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_double,
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
        ctypes.c_void_p, ctypes.c_int]
    lib.mgd_poll_status.restype = ctypes.c_int
    lib.mgd_poll_status.argtypes = [ctypes.c_int, ctypes.c_void_p]
    lib.mgd_encode_targets_dlpack.restype = ctypes.c_int
    lib.mgd_encode_targets_dlpack.argtypes = [
        ctypes.POINTER(HeadConfig), ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p),
        ctypes.c_void_p, ctypes.c_int, _LLP]
    lib.mgd_decode_nms_dlpack.restype = ctypes.c_int
    lib.mgd_decode_nms_dlpack.argtypes = [
        ctypes.POINTER(HeadConfig), ctypes.POINTER(PostConfig),
        ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_int, _LLP]
    lib.mgd_match_detections.restype = ctypes.c_int
    lib.mgd_match_detections.argtypes = [
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, _DP, ctypes.c_int,
        ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
        ctypes.c_int]
    lib.mgd_iou_matrix.restype = ctypes.c_int
    lib.mgd_iou_matrix.argtypes = [
        ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
        ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    lib.mgd_reshape_boxes.restype = ctypes.c_int
    lib.mgd_reshape_boxes.argtypes = [
        ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
        ctypes.c_int]
    lib.mgd_mosaic_merge_boxes.restype = ctypes.c_int
    lib.mgd_mosaic_merge_boxes.argtypes = [
        ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
        ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
        ctypes.c_void_p, ctypes.c_int]
    lib.mgd_encode_ignore_mask.restype = ctypes.c_int
    lib.mgd_encode_ignore_mask.argtypes = [
        ctypes.POINTER(HeadConfig), ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
        ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p), ctypes.c_double, ctypes.c_double,
        ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p),
        ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    lib.mgd_letterbox_boxes.restype = ctypes.c_int
    lib.mgd_letterbox_boxes.argtypes = [
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
        ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
        ctypes.c_void_p, ctypes.c_int]
    lib.mgd_ignore_mask.restype = ctypes.c_int
    lib.mgd_ignore_mask.argtypes = [
        ctypes.POINTER(HeadConfig), ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p),
        ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.POINTER(ctypes.c_void_p),
        ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_int,
        ctypes.c_void_p, ctypes.c_int]
    lib.mgd_host_alloc.restype = ctypes.c_int
    lib.mgd_host_alloc.argtypes = [ctypes.c_size_t, ctypes.POINTER(ctypes.c_void_p)]
    lib.mgd_host_free.restype = ctypes.c_int
    lib.mgd_host_free.argtypes = [ctypes.c_void_p]
    lib.mgd_release_workspace.restype = ctypes.c_int
    lib.mgd_exchange_create.restype = ctypes.c_int
    lib.mgd_exchange_create.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_size_t,
                                        ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p]
    lib.mgd_exchange_connect.restype = ctypes.c_int
    lib.mgd_exchange_connect.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.mgd_exchange_buffer.restype = ctypes.c_int
    lib.mgd_exchange_buffer.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p),
                                        ctypes.POINTER(ctypes.c_size_t)]
    lib.mgd_exchange_timeouts.restype = ctypes.c_int
    lib.mgd_exchange_timeouts.argtypes = [ctypes.c_void_p, ctypes.c_void_p, _IP]
    lib.mgd_exchange_destroy.restype = ctypes.c_int
    lib.mgd_exchange_destroy.argtypes = [ctypes.c_void_p]
    lib.mgd_map_record_bytes.restype = ctypes.c_int
    lib.mgd_map_record_bytes.argtypes = []
    lib.mgd_map_update.restype = ctypes.c_int
    lib.mgd_map_update.argtypes = [
        ctypes.POINTER(MapConfig), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
        ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    lib.mgd_map_compute.restype = ctypes.c_int
    lib.mgd_map_compute.argtypes = [
        ctypes.POINTER(MapConfig), ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    lib.mgd_map_partition.restype = ctypes.c_int
    lib.mgd_map_partition.argtypes = [
        ctypes.POINTER(MapConfig), ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_int,
        ctypes.c_longlong, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
        ctypes.c_void_p, ctypes.c_int]
    lib.mgd_map_compute_merged.restype = ctypes.c_int
    lib.mgd_map_compute_merged.argtypes = [
        ctypes.POINTER(MapConfig), ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
        ctypes.c_int]
    lib.mgd_map_compute_pr.restype = ctypes.c_int
    lib.mgd_map_compute_pr.argtypes = [
        ctypes.POINTER(MapConfig), ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(MapPr), ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    lib.mgd_map_compute_merged_pr.restype = ctypes.c_int
    lib.mgd_map_compute_merged_pr.argtypes = [
        ctypes.POINTER(MapConfig), ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(MapPr), ctypes.c_int,
        ctypes.c_void_p, ctypes.c_int]
    lib.mgd_profile_begin.restype = ctypes.c_int
    lib.mgd_profile_end.restype = ctypes.c_int
    lib.mgd_profile_end.argtypes = [_DP, _LLP]
    _lib = lib
    return lib


def raise_for_status(rc: int) -> None:
    """Map ``mgd_status`` to the reference's exception types."""
    if rc == OK:
        return
    msg = load().mgd_last_error().decode("utf-8", "replace")
    if rc == ERR_CLASS_RANGE:
        raise AssertionError(msg)              # generators.py:3409
    if rc == ERR_INVALID_ARGUMENT:
        raise ValueError(msg)
    if rc == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise MgdError(msg)


_cfg_cache: dict = {}


def make_head_config(anchors, num_classes, input_shape, grid_shapes=None) -> HeadConfig:
    """``anchors``: list of (A_l, 2) arrays; their dtype picks the arithmetic path
    (float64 only if the caller's anchors are float64, like NumPy promotion).
    Memoised on the values (the evaluator builds the same geometry for every image)."""
    arrs = [np.asarray(a) for a in anchors]
    key = (tuple((a.dtype.str, a.shape, a.tobytes()) for a in arrs), int(num_classes),
           int(input_shape[0]), int(input_shape[1]),
           None if grid_shapes is None else tuple((int(g[0]), int(g[1])) for g in grid_shapes))
    hit = _cfg_cache.get(key)
    if hit is not None:
        return hit
    cfg = _make_head_config(arrs, num_classes, input_shape, grid_shapes)
    if len(_cfg_cache) < 256:
        _cfg_cache[key] = cfg
    return cfg


def _make_head_config(arrs, num_classes, input_shape, grid_shapes=None) -> HeadConfig:
    num_layers = len(arrs)
    if not 1 <= num_layers <= MGD_MAX_LAYERS:
        raise ValueError(f"between 1 and {MGD_MAX_LAYERS} layers supported, got {num_layers}")
    cfg = HeadConfig()
    cfg.num_layers = num_layers
    cfg.num_classes = int(num_classes)
    cfg.input_h, cfg.input_w = int(input_shape[0]), int(input_shape[1])
    if grid_shapes is None:                     # generators.py:3423
        strides = (32, 16, 8, 4, 2)
        grid_shapes = [(cfg.input_h // strides[l], cfg.input_w // strides[l])
                       for l in range(num_layers)]
    f64 = False
    for l, a in enumerate(arrs):
        if a.ndim != 2 or a.shape[1] != 2 or not 1 <= a.shape[0] <= MGD_MAX_ANCHORS_PER_LAYER:
            raise ValueError(f"anchors[{l}] must have shape (1..{MGD_MAX_ANCHORS_PER_LAYER}, 2)")
        f64 = f64 or a.dtype == np.float64
        cfg.grid_h[l], cfg.grid_w[l] = int(grid_shapes[l][0]), int(grid_shapes[l][1])
        cfg.num_anchors[l] = a.shape[0]
        for i in range(a.shape[0]):
            cfg.anchors[l][i][0] = float(a[i, 0])
            cfg.anchors[l][i][1] = float(a[i, 1])
    cfg.anchors_f64 = int(f64)
    return cfg


def ptr_array(ptrs):
    return (ctypes.c_void_p * len(ptrs))(*[ctypes.c_void_p(int(p)) for p in ptrs])


class PinnedPool:
    """Recycling allocator of page-locked NumPy arrays (``mgd_host_alloc``).

    ``empty(shape, dtype)`` returns an ordinary ndarray whose memory is page-locked; when
    the array (and every view of it) is garbage collected the block goes back to the
    pool and is handed to the next request of the same size, so a training / evaluation
    loop that drops its previous batch allocates nothing in steady state.  The pool never
    holds more than ``cap_bytes`` of page-locked memory in total (in use + idle; env
    ``MGD_PINNED_CAP_MB``, default 4096): a caller that keeps every result alive gets
    pageable ``np.empty`` arrays once the cap is reached, as does a host without a GPU.
    """

    def __init__(self, cap_bytes=None):
        import threading
        if cap_bytes is None:
            cap_bytes = int(os.environ.get("MGD_PINNED_CAP_MB", "4096")) << 20
        self._lock = threading.Lock()
        self._free = {}
        self._idle = 0
        self._total = 0
        self.cap_bytes = cap_bytes

    def _give_back(self, ptr, nbytes):
        with self._lock:
            self._free.setdefault(nbytes, []).append(ptr)
            self._idle += nbytes

    def _trim(self, need):
        """Free idle blocks (largest first) until ``need`` more bytes fit under the cap."""
        victims = []
        with self._lock:
            for size in sorted(self._free, reverse=True):
                lst = self._free[size]
                while lst and self._total + need > self.cap_bytes:
                    victims.append(lst.pop())
                    self._idle -= size
                    self._total -= size
        for ptr in victims:
            load().mgd_host_free(ctypes.c_void_p(ptr))

    def empty(self, shape, dtype):
        import weakref
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
        if nbytes < (1 << 16):                    # tiny arrays: not worth a page-locked block
            return np.empty(shape, dtype)
        ptr = None
        with self._lock:
            lst = self._free.get(nbytes)
            if lst:
                ptr = lst.pop()
                self._idle -= nbytes
        if ptr is None:
            if self._total + nbytes > self.cap_bytes:
                self._trim(nbytes)
            if self._total + nbytes > self.cap_bytes:
                return np.empty(shape, dtype)
            out = ctypes.c_void_p()
            if load().mgd_host_alloc(nbytes, ctypes.byref(out)) != OK or not out.value:
                return np.empty(shape, dtype)
            ptr = out.value
            with self._lock:
                self._total += nbytes
        buf = (ctypes.c_char * nbytes).from_address(ptr)
        weakref.finalize(buf, self._give_back, ptr, nbytes)
        return np.frombuffer(buf, dtype=dtype).reshape(shape)


pinned = PinnedPool()
