"""Sharded streaming mAP (evaluation.ShardedMapAccumulator, mgd_map_partition /
mgd_map_compute_merged).

CPU: argument validation of the two entry points before any device work, the global-slot
arithmetic against a brute-force listing of global image order, and the update-sequence check
over gloo at world size 2.  GPU: the sharded accumulator equals MapAccumulator over the same
global data EXACTLY (== on every value of the result dict), at world size 1 and with two
processes on one GPU over gloo.
"""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest

from multigriddet_b200 import _lib, engine
from multigriddet_b200.evaluation.metrics import global_slot_segments
from multigriddet_b200.sharding import shard_bounds

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(os.path.dirname(__file__), "golden", "metrics_cases.npz")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    return _lib.load()


def _free_port():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def _spawn(target, world, *args, timeout=600):
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


# ------------------------------------------------------------------------------ CPU

def test_entry_points_validate_then_need_a_device(lib):
    cfg = engine.map_config(3, [0.5, 0.75], "coco", views=(_lib.MAP_VIEW_CORNER, _lib.MAP_VIEW_S))
    one = ctypes.c_void_p(8)                                # never dereferenced: validation or no device

    def part(c=cfg, n=4, nseg=1, glob=8, world=2, owner=one, counts=one):
        return lib.mgd_map_partition(ctypes.byref(c), one, n, one, nseg, glob, owner, world, one, counts,
                                     0, None, 0)

    def merged(c=cfg, n=4, rank=0, owner=one, ap=one):
        return lib.mgd_map_compute_merged(ctypes.byref(c), one, n, one, owner, rank, ap, one, one, 0, None, 0)

    for field, bad in (("num_thresholds", 0), ("num_classes", 0), ("method", 7), ("views", 0)):
        c = engine.map_config(3, [0.5, 0.75])
        setattr(c, field, bad)
        assert part(c) == _lib.ERR_INVALID_ARGUMENT, field
        assert merged(c) == _lib.ERR_INVALID_ARGUMENT, field
    for kw in (dict(n=-1), dict(n=1 << 31), dict(nseg=0), dict(nseg=-1), dict(glob=3), dict(world=0),
               dict(owner=None), dict(counts=None)):
        assert part(**kw) == _lib.ERR_INVALID_ARGUMENT, kw
    assert part(glob=(1 << 32) + 1) == _lib.ERR_UNSUPPORTED          # global slots must fit 32 bits
    assert part(world=257) == _lib.ERR_UNSUPPORTED                    # one radix digit of ranks
    for kw in (dict(n=-1), dict(rank=-1), dict(owner=None), dict(ap=None)):
        assert merged(**kw) == _lib.ERR_INVALID_ARGUMENT, kw
    if lib.mgd_device_count() == 0:
        assert part() == _lib.ERR_NO_DEVICE
        assert part(n=0, nseg=0, glob=1 << 32) == _lib.ERR_NO_DEVICE
        assert merged() == _lib.ERR_NO_DEVICE
        with pytest.raises(_lib.MgdError, match="no CPU fallback"):
            _lib.raise_for_status(merged())


def test_python_wrappers_validate_before_any_device_work():
    import torch
    from multigriddet_b200.evaluation import ShardedMapAccumulator
    cfg = engine.map_config(3, [0.5])
    cpu = torch.zeros(400, dtype=torch.uint8)
    owner = torch.zeros(3, dtype=torch.int32)
    with pytest.raises(ValueError, match="CUDA"):
        engine.map_partition(cfg, cpu, 10, [(0, 0)], 10, owner, 1)
    with pytest.raises(ValueError, match="gt_hist"):
        engine.map_compute_merged(cfg, cpu, 10, torch.zeros((_lib.MAP_VIEWS, 3), dtype=torch.int64), owner, 0)
    with pytest.raises(ValueError):
        ShardedMapAccumulator(0)


def _brute_force_slots(updates, world):
    """{(rank, local slot): global slot}, by listing every update's global batch image by image."""
    out, local = {}, [0] * world
    g = 0
    for n_total, m in updates:
        owner = [r for r in range(world) for _ in range(*shard_bounds(n_total, r, world))]
        for img in range(n_total):
            r = owner[img]
            for _ in range(m):
                out[(r, local[r])] = g
                local[r] += 1
                g += 1
    return out, g


@pytest.mark.parametrize("world,updates", [
    (1, [(5, 3), (2, 4)]),
    (2, [(11, 4)]),                                          # uneven shards
    (3, [(1, 5), (2, 5), (7, 2)]),                           # ranks without images
    (4, [(9, 3), (0, 3), (4, 7), (3, 1), (13, 2)]),          # an empty batch, every kind of shard
    (8, [(5, 100), (8, 100), (17, 1)]),
    (2, [(3, 0), (4, 2)]),                                   # max_dets 0
])
def test_global_slots_follow_global_image_order(world, updates):
    ref, total = _brute_force_slots(updates, world)
    seen = set()
    for r in range(world):
        segments, glob = global_slot_segments(updates, r, world)
        assert glob == total
        starts = [s for s, _ in segments]
        assert starts == sorted(set(starts))                  # strictly ascending local starts
        n_local = sum(m * (shard_bounds(n, r, world)[1] - shard_bounds(n, r, world)[0]) for n, m in updates)
        for j in range(n_local):
            L, base = [s for s in segments if s[0] <= j][-1]   # the kernel's lookup: last start <= j
            slot = base + (j - L)
            assert slot == ref[(r, j)], (r, j)
            seen.add(slot)
    assert seen == set(range(total))


def _agree_main(rank, world, port, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from multigriddet_b200.evaluation.metrics import check_same_updates
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    out = []
    try:
        for same, error in ((True, None), (False, None), (True, "class id" if rank == 1 else None),
                            (False, "class id")):
            seq = [(11, 100), (7, 100)] if same or rank == 0 else [(11, 100), (7, 50)]
            try:
                check_same_updates(seq, error)
                out.append("ok")
            except (ValueError, AssertionError) as e:
                out.append(type(e).__name__)
        q.put((rank, out))
    except Exception as e:                                    # pragma: no cover
        q.put((rank, repr(e)))
    finally:
        dist.destroy_process_group()


def test_update_sequences_are_checked_on_every_rank():
    res = _spawn(_agree_main, 2, timeout=300)
    want = ["ok", "ValueError", "AssertionError", "ValueError"]
    assert res == {0: want, 1: want}


# ------------------------------------------------------------------------------ GPU

def _dev(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _assert_equal(got, ref, path="result"):
    """== on every value (and the same types), no tolerance."""
    assert type(got) is type(ref) or (isinstance(got, float) and isinstance(ref, float)), (path, type(got), type(ref))
    if isinstance(ref, dict):
        assert set(got) == set(ref), (path, sorted(set(got) ^ set(ref)))
        for k in ref:
            _assert_equal(got[k], ref[k], f"{path}[{k!r}]")
    else:
        assert got == ref, (path, got, ref)


def _reference(C, batches, **kw):
    """MapAccumulator over the global batches, in one process."""
    from multigriddet_b200.evaluation import MapAccumulator
    acc = MapAccumulator(C, **kw)
    for b in batches:
        acc.update(*_dev(*b))
    return acc.compute()


def _sharded(C, batches, rank=0, world=1, **kw):
    """ShardedMapAccumulator fed with this rank's shard of every global batch."""
    from multigriddet_b200.evaluation import ShardedMapAccumulator
    acc = ShardedMapAccumulator(C, **kw)
    for b in batches:
        lo, hi = shard_bounds(len(b[3]), rank, world)
        acc.update(*_dev(*[a[lo:hi] for a in b]), n_total=len(b[3]))
    return acc.compute()


def _split(args, sizes, max_dets=None):
    """The global batches of one data set: consecutive images, optionally with fewer slots."""
    out, lo = [], 0
    for k, n in enumerate(sizes):
        b = [a[lo:lo + n] for a in args]
        if max_dets and max_dets[k]:
            m = max_dets[k]
            b[0], b[1], b[2], b[3] = b[0][:, :m], b[1][:, :m], b[2][:, :m], np.minimum(b[3], m).astype(np.int32)
        out.append(tuple(b))
        lo += n
    assert lo == len(args[3])
    return out


_KWS = (dict(), dict(use_parallel=False), dict(optimize_classes=False), dict(method="voc", use_parallel=False),
        dict(cache_ious=False, compute_per_scale=False))


_REC = np.dtype([("score", "<f8"), ("cls", "<i4"), ("band", "<i4"), ("bits", "<u4", (_lib.MAP_VIEWS,)),
                 ("pad", "<u4")])


@pytest.mark.gpu
def test_gpu_partition_groups_by_owner_and_stamps_global_slots():
    import torch
    from multigriddet_b200.evaluation import MapAccumulator
    from oracle.gen_golden import synth_eval_set
    args = synth_eval_set(47, 31, 40, 12, 7, ties=True)
    args = (args[0].astype(np.int32),) + tuple(args[1:])
    acc = MapAccumulator(7)
    for b in _split(args, [10, 21]):                         # 400 + 840 slots
        acc.update(*_dev(*b))
    rb = engine.map_record_bytes()
    assert _REC.itemsize == rb
    owner_np = np.array([2, 0, 1, 2, 0, 1, 2], np.int32)
    owner = torch.from_numpy(owner_np).cuda()
    segments = [(0, 1000), (400, 7000)]
    out, counts = engine.map_partition(acc._cfg, acc._records, acc._slots, segments, 1 << 32, owner, 3)
    src = acc._records[:acc._slots * rb].cpu().numpy().view(_REC)
    keep = np.flatnonzero(src["cls"] >= 0)
    dest = owner_np[src["cls"][keep]]
    order = keep[np.argsort(dest, kind="stable")]            # by destination, local order within
    want = src[order].copy()
    want["pad"] = np.where(order < 400, 1000 + order, 7000 + order - 400)
    assert counts.cpu().tolist() == np.bincount(dest, minlength=3).tolist()
    assert out[:len(order) * rb].cpu().numpy().tobytes() == want.tobytes()
    engine.poll_status()
    bad = torch.tensor([0, 1, 2, 3, 0, 1, 2], dtype=torch.int32, device="cuda")
    engine.map_partition(acc._cfg, acc._records, acc._slots, segments, 1 << 32, bad, 3)
    with pytest.raises(ValueError, match="owner"):
        engine.poll_status()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["a", "b", "ties"])
def test_gpu_world_of_one_equals_accumulator_on_golden_cases(name):
    z = np.load(GOLD)
    db, ds, dc, dn, gtb, gtc, gtn = (z[f"{name}_{k}"] for k in ("db", "ds", "dc", "dn", "gtb", "gtc", "gtn"))
    C = int(z[f"{name}_C"])
    args = (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
    B = len(dn)
    for kw in _KWS:
        ref = _reference(C, [args], **kw)
        _assert_equal(_sharded(C, [args], **kw), ref, str(kw))
        _assert_equal(_sharded(C, _split(args, [B // 3, B - B // 3]), **kw), ref, str(kw))


@pytest.mark.gpu
def test_gpu_world_of_one_equals_accumulator_at_size():
    from oracle.gen_golden import synth_eval_set
    B, M, N, C = 2000, 100, 20, 80
    db, ds, dc, dn, gtb, gtc, gtn = synth_eval_set(43, B, M, N, C)
    ds = np.round(ds, 2)                                     # ties across images are common
    ds[1::97, 3] = -0.0
    ds[2::89, 5] = 0.0
    args = (db.astype(np.int32), ds, dc, dn, gtb, gtc, gtn)
    batches = _split(args, [256] * 7 + [208])
    for kw in _KWS:
        _assert_equal(_sharded(C, batches, **kw), _reference(C, batches, **kw), str(kw))


def _crafted_ties():
    """Class 0: one detection per image, all of score 0.5, in two updates of one image per rank.
    Only global image 2 (update 1, rank 0) has ground truth.  Later detection first in global
    order puts image 2 second; concatenating the ranks' records puts it third, and the AP differs."""
    C, M, N = 2, 2, 1
    batches = []
    for u in range(2):
        db = np.zeros((2, M, 4), np.int32)
        db[:, 0] = [10, 10, 50, 50]
        db[:, 1] = [100, 100, 300, 300]
        ds = np.array([[0.5, 0.25], [0.5, 0.25]])
        dc = np.array([[0, 1], [0, 1]], np.int32)
        dn = np.array([2, 2], np.int32)
        gtb = np.zeros((2, N, 4))
        gtc = np.zeros((2, N), np.int32)
        gtn = np.zeros(2, np.int32)
        if u == 1:
            gtb[0, 0] = [10, 10, 50, 50]
            gtn[0] = 1
        batches.append((db, ds, dc, dn, gtb, gtc, gtn))
    return C, batches


def _rank_main(rank, world, port, q):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from oracle.gen_golden import synth_eval_set
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(0)
    out = {}

    def case(name, C, batches, **kw):
        try:
            _assert_equal(_sharded(C, batches, rank, world, **kw), _reference(C, batches, **kw), f"{name} {kw}")
            out[name] = "equal"
        except AssertionError as e:
            out[name] = f"differs: {str(e)[:300]}"

    try:
        args = synth_eval_set(47, 31, 40, 12, 7, ties=True)
        args = (args[0].astype(np.int32),) + tuple(args[1:])
        for i, kw in enumerate(_KWS):
            case(f"uneven{i}", 7, _split(args, [31]), **kw)                  # 16 + 15 images
        case("empty_shard", 7, _split(args, [1, 19, 11]))                      # rank 1 holds nothing in update 0
        case("updates", 7, _split(args, [7, 1, 12, 3, 8], max_dets=[None, 17, 40, 5, 23]))
        case("updates_voc", 7, _split(args, [7, 1, 12, 3, 8], max_dets=[None, 17, 40, 5, 23]),
             method="voc", use_parallel=False)
        C, crafted = _crafted_ties()
        case("crafted_ties", C, crafted)
        # the crafted case does tell the orders apart: rank-major concatenation gives another AP
        rank_major = [tuple(np.concatenate([b[k][r:r + 1] for b in crafted]) for k in range(7)) for r in range(2)]
        out["crafted_rank_major_differs"] = bool(_reference(C, rank_major)["mAP"] != _reference(C, crafted)["mAP"])
        # a class id out of range on one rank raises on both, and both go on
        bad = [np.array(a) for a in args]
        bad[2][20, 0] = 7                                                      # image 20: rank 1's shard
        try:
            _sharded(7, _split(tuple(bad), [31]), rank, world)
            out["class_range"] = "no error"
        except AssertionError as e:
            out["class_range"] = "AssertionError" if "class id" in str(e) else repr(e)
        case("after_error", 7, _split(args, [31]))
        # fed by ShardedGridPath.decode_nms(gather=False)
        from multigriddet_b200 import sharding, synth
        from multigriddet_b200.evaluation import ShardedMapAccumulator
        S, Cd, B, N = 416, 20, 13, 40
        anchors = synth.coco_anchors(np.float32)
        boxes = synth.synth_boxes(44, B, N, S, Cd)
        y = engine.encode_targets(torch.from_numpy(boxes).cuda(), (S, S), anchors, Cd)
        preds = synth.planted_head_outputs(y, 3, seed=44)
        kw = dict(max_boxes=100, confidence=0.05, nms_threshold=0.45, nms_method="diou")
        gt_counts = ((boxes[..., 2] - boxes[..., 0]) * (boxes[..., 3] - boxes[..., 1]) > 0).sum(1).astype(np.int32)
        gt = (boxes[..., :4].astype(np.float64), boxes[..., 4].astype(np.int32), gt_counts)
        path = sharding.ShardedGridPath(anchors, Cd, (S, S))
        det = path.decode_nms(preds, None, gather=False, **kw)
        sl = path.local_slice(B)
        acc = ShardedMapAccumulator(Cd)
        acc.update(det["boxes_xyxy"], det["scores"], det["classes"], det["counts"], *_dev(*[g[sl] for g in gt]),
                   n_total=B)
        full = engine.decode_nms(preds, None, (S, S), anchors, Cd, **kw)
        ref = _reference(Cd, [tuple(full[k].cpu().numpy() for k in ("boxes_xyxy", "scores", "classes", "counts"))
                              + gt])
        try:
            got = acc.compute()
            assert got["num_predictions"] > 0
            _assert_equal(got, ref, "decode_nms")
            out["decode_nms"] = "equal"
        except AssertionError as e:
            out["decode_nms"] = f"differs: {str(e)[:300]}"
        q.put((rank, out))
    except Exception as e:                                    # pragma: no cover
        import traceback
        q.put((rank, {"error": traceback.format_exc()[-2000:]}))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_gpu_two_ranks_equal_one_accumulator_over_the_global_data():
    res = _spawn(_rank_main, 2, timeout=900)
    for rank in (0, 1):
        got = res[rank]
        assert "error" not in got, (rank, got.get("error"))
        assert got.pop("class_range") == "AssertionError", rank
        assert got.pop("crafted_rank_major_differs") is True, rank
        assert all(v == "equal" for v in got.values()), (rank, {k: v for k, v in got.items() if v != "equal"})
        assert len(got) == len(_KWS) + 6, (rank, sorted(got))
