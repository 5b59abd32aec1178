"""CPU tier of the device-resident map (SURVEY.md §8f N1): the delta protocol of include/malio_mapsync.hpp is EXACT.
The real reference ikd-Tree (oracle/_ref) and a flat numpy mirror receive the same 50-scan scripted stream of
Add_Points (with and without down-sampling) / Delete_Point_Boxes; the mirror only ever sees what the device would see
(appends, boxes, per-voxel re-synchronisation records collected through KD_TREE::Box_Search).  After every scan the
mirror's live set must equal KD_TREE::flatten() point for point — whatever the tree's topology and re-build timing.
Where oracle/_ref is not built, the mirror replays the tree's answers to the same stream (tests/golden/make_ref_golden.py)."""
import hashlib
import os

import numpy as np
import pytest

import pyoracle as po
import np_mapops as nm

VOXEL = 0.5
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ikd_ref_golden.npz")


def scripted_stream(seed=1, M=20000, scans=50):
    """Yields ('build', xyz, ny, ids) then per scan ('scan', add_ds, ny, ids, add_plain, ny2, ids2, boxes|None)."""
    rng = np.random.default_rng(seed)
    xyz = rng.uniform(-20, 20, (M, 3)).astype(np.float32)
    xyz[:, 2] = rng.uniform(0, 4, M)
    yield ("build", xyz, np.full(M, 0.001, np.float32), np.arange(M, dtype=np.int32))
    nid = M
    for it in range(scans):
        k = 400
        a = (xyz[rng.integers(0, M, k)] + rng.normal(0, 0.4, (k, 3))).astype(np.float32)
        a[: k // 8] = a[k // 8: k // 4] + np.float32(0.01)          # several new points in the same voxel, in order
        ny = np.where(rng.uniform(size=k) < 0.5, 0.001, rng.uniform(0.0005, 0.01, k)).astype(np.float32)
        ids = np.arange(nid, nid + k, dtype=np.int32); nid += k
        b = (xyz[rng.integers(0, M, 60)] + rng.normal(0, 0.2, (60, 3))).astype(np.float32)
        ids2 = np.arange(nid, nid + 60, dtype=np.int32); nid += 60
        boxes = None
        if it % 7 == 3:
            c = xyz[rng.integers(0, M)]
            boxes = np.array([[c[0] - 3, c[1] - 3, c[2] - 1.5, c[0] + 3, c[1] + 3, c[2] + 1.5]], np.float32)
        yield ("scan", a, ny, ids, b, np.full(60, 0.002, np.float32), ids2, boxes)


def live_set_digest(xyz, ny, ids) -> bytes:
    """SHA-256 of a live point set ordered by id: equal digests <=> equal sets, point for point."""
    o = np.argsort(ids, kind="stable")
    h = hashlib.sha256(np.asarray(ids, np.int64)[o].tobytes())
    h.update(np.ascontiguousarray(xyz, np.float32)[o].tobytes())
    h.update(np.ascontiguousarray(ny, np.float32)[o].tobytes())
    return h.digest()


def recorded_stream():
    """The reference tree's answers to scripted_stream() (defaults), from the golden file: yields per scan
    (event, Delete_Point_Boxes count, Add_Points count, sync record as add_points_synced returns it, validnum, live-set digest)."""
    g = np.load(GOLD)
    events = list(scripted_stream())
    by_id = {}
    for ev in events:
        pairs = [(ev[1], ev[2], ev[3])] if ev[0] == "build" else [(ev[1], ev[2], ev[3]), (ev[4], ev[5], ev[6])]
        for xyz, ny, ids in pairs:
            by_id.update(zip(ids.tolist(), zip(xyz.copy(), ny.copy())))   # copies: callers may overwrite the event's arrays
    ob = om = 0
    for s, ev in enumerate(events[1:]):
        nb = int(g["stream_nb"][s])
        counts = g["stream_counts"][ob:ob + nb].astype(np.uint32)
        m = int(counts.sum())
        lo = g["stream_vox"][ob:ob + nb].astype(np.float32) * np.float32(VOXEL)
        ids = g["stream_ids"][om:om + m]
        sync = dict(boxes=np.concatenate([lo, lo + np.float32(VOXEL)], 1), counts=counts,
                    xyz=np.array([by_id[i][0] for i in ids.tolist()], np.float32).reshape(-1, 3),
                    normal_y=np.array([by_id[i][1] for i in ids.tolist()], np.float32), ids=ids.copy(), outside_own_box=0)
        ob += nb; om += m
        yield ev, int(g["stream_ndel"][s]), int(g["stream_added"][s]), sync, int(g["stream_valid"][s]), g["stream_digest"][s].tobytes()


def same_set(tree, mirror):
    fx, fny, fid = tree.flatten_points()
    lx, lny, lid = mirror
    if len(fid) != len(lid):
        return False
    a, b = np.argsort(fid, kind="stable"), np.argsort(lid, kind="stable")
    return np.array_equal(fid[a], np.asarray(lid)[b]) and np.array_equal(fx[a], lx[b]) and np.array_equal(fny[a], lny[b])


def _replay_recorded_stream():
    mir = nm.MirrorMap()
    ev0 = next(scripted_stream())
    mir.build(ev0[1], ev0[2], ev0[3])
    synced_pts = 0
    for ev, ndel, cnt, sync, valid, digest in recorded_stream():
        _, a, ny, ids, b, ny2, ids2, boxes = ev
        if boxes is not None:
            assert ndel == mir.delete_boxes(boxes)
        assert cnt > 0
        assert len(np.unique(sync["boxes"], axis=0)) == len(sync["boxes"])
        mir.sync_voxels(sync)
        synced_pts += len(sync["ids"])
        mir.add_points(b, ny2, ids2)
        live = mir.live_points()
        assert len(live[2]) == valid and live_set_digest(*live) == digest
    assert synced_pts < 50 * 400 * 3


@pytest.mark.parametrize("threads", [1, 8])
def test_delta_protocol_keeps_a_flat_mirror_equal_to_the_real_tree(threads):
    """With oracle/_ref: the live tree, read back with `threads` threads.  Without: the recorded answers of that tree (collected
    with 1 and with 8 threads, identical)."""
    if not po.ref_available():
        _replay_recorded_stream()
        return
    tree = po.RefTree(box_length=0.5)
    mir = nm.MirrorMap()
    synced_pts = 0
    for ev in scripted_stream():
        if ev[0] == "build":
            tree.build(ev[1], ev[2], ev[3]); mir.build(ev[1], ev[2], ev[3])
            continue
        _, a, ny, ids, b, ny2, ids2, boxes = ev
        if boxes is not None:
            assert tree.delete_boxes(boxes) == mir.delete_boxes(boxes)
        cnt, sync = tree.add_points_synced(a, ny, ids, 0.5, threads=threads)
        assert sync["outside_own_box"] == 0 and cnt > 0
        assert len(np.unique(sync["boxes"], axis=0)) == len(sync["boxes"])       # distinct voxels
        mir.sync_voxels(sync)
        synced_pts += len(sync["ids"])
        tree.add_points(b, ny2, ids2, downsample=False); mir.add_points(b, ny2, ids2)
        tree.wait_rebuild()
        assert same_set(tree, mir.live_points())
    assert synced_pts < 50 * 400 * 3      # the deltas stay proportional to the changed points
    tree.close()


@pytest.mark.skipif(not po.ref_available(), reason="oracle/_ref (the real ikd_Tree.cpp) was not built")
def test_collect_voxel_sync_edge_cases_and_thread_independence():
    """malio::collect_voxel_sync: nothing added -> empty record; many new points in ONE voxel -> one box; more threads than voxels;
    the record (boxes in order of first appearance, points in box order) does not depend on the thread count; a voxel the tree
    holds nothing in comes back with count 0 (its box still travels: the device must empty it)."""
    rng = np.random.default_rng(5)
    M = 5000
    xyz = rng.uniform(-10, 10, (M, 3)).astype(np.float32)
    tree = po.RefTree(box_length=0.5)
    tree.build(xyz, np.full(M, 0.001, np.float32), np.arange(M, dtype=np.int32))
    s = tree.collect_sync(np.zeros((0, 3), np.float32), 0.5, threads=4)
    assert s["boxes"].shape[0] == 0 and s["xyz"].shape[0] == 0
    one = (np.array([[1.1, 2.1, 3.1]], np.float32) + rng.uniform(0, 0.3, (40, 3)).astype(np.float32))
    tree.add_points(one, np.full(40, 0.001, np.float32), np.arange(M, M + 40, dtype=np.int32), downsample=True)
    s = tree.collect_sync(one, 0.5, threads=8)       # 8 threads, 1 voxel
    assert s["boxes"].shape[0] == 1 and s["counts"][0] == s["xyz"].shape[0] >= 1
    assert np.allclose(s["boxes"][0], [1.0, 2.0, 3.0, 1.5, 2.5, 3.5])
    inside = (s["xyz"] >= s["boxes"][0, :3]).all() and (s["xyz"] < s["boxes"][0, 3:]).all()
    assert inside
    # a box far outside the map: no live point, count 0, the box is still reported
    far = np.array([[500.2, 500.2, 500.2]], np.float32)
    s = tree.collect_sync(far, 0.5, threads=2)
    assert s["boxes"].shape[0] == 1 and s["counts"][0] == 0 and s["xyz"].shape[0] == 0
    # thread independence on a batch with repeats
    a = (xyz[rng.integers(0, M, 600)] + rng.normal(0, 0.3, (600, 3))).astype(np.float32)
    a[100:200] = a[0:100]
    tree.add_points(a, np.full(600, 0.001, np.float32), np.arange(M + 40, M + 640, dtype=np.int32), downsample=True)
    ref = tree.collect_sync(a, 0.5, threads=1)
    assert ref["boxes"].shape[0] < 600                      # repeats collapse
    for th in (2, 3, 8, 64):
        s = tree.collect_sync(a, 0.5, threads=th)
        for k in ("boxes", "counts", "xyz", "normal_y", "ids"):
            assert np.array_equal(s[k], ref[k]), (th, k)
    assert int(ref["counts"].sum()) == ref["xyz"].shape[0]
    tree.close()
