"""GPU parity of the device-resident map (SURVEY.md §8f N1): the real reference ikd-Tree (oracle/_ref) and the device
receive the same 50-scan scripted stream (Delete_Point_Boxes, Add_Points with and without down-sampling); the device
only gets deltas (boxes, appended points, per-voxel re-synchronisation records read back through KD_TREE::Box_Search by
include/malio_mapsync.hpp).  Checked: after every scan the device's live set is KD_TREE::flatten() point for point; every
10 scans the k-NN lists of 20k queries equal those of a FULL re-upload of the tree's snapshot (exact tree mode) — float
distances bit-identical everywhere, index lists identical except where two neighbours are at exactly tied distances (the
reference breaks those by traversal order; counted, SURVEY.md §7); a whole measurement pass agrees; H2D stays
proportional to the changed points.
Where oracle/_ref is not built, the device replays the tree's recorded answers to the stream of tests/test_mapops_cpu.py
(tests/golden/), and the full re-uploads are static snapshots of the same live points."""
import numpy as np
import pytest

import helpers as H
import pyoracle as po
from malio_b200 import capi, plugin, synth
from test_mapops_cpu import live_set_digest, recorded_stream, same_set, scripted_stream

pytestmark = pytest.mark.gpu


def static_snapshot_of(xyz, ny, ids):
    s = plugin.build_static_snapshot(xyz, ny)
    return plugin.MapSnapshot(s.nodes, s.node_cov, np.asarray(ids)[s.node_ids], s.max_depth)


def _check_knn(dev, snap, rng, n_q=20000):
    full = plugin.MeasurementModel(1)
    full.upload_map(snap)
    m = dev.map_download()
    slot_to_id = np.full(int(m["slots"].max()) + 1, -1, np.int64)
    slot_to_id[m["slots"]] = m["ids"]
    q = (m["xyz"][rng.integers(0, m["xyz"].shape[0], n_q)] + rng.normal(0, 0.4, (n_q, 3))).astype(np.float32)
    q[:200] += np.float32(60.0)            # far outside the map: ring expansion up to the whole grid
    q[200:400] *= np.float32(3.0)          # sparse fringe
    c0 = dev.counters()
    di, dd, _ = dev.Nearest_Search(q)
    c1 = dev.counters()
    fi, fd, _ = full.Nearest_Search(q)
    full.close()
    assert np.array_equal(dd, fd), "distances must be bit-identical"
    d_ids = np.where(di != 0xFFFFFFFF, slot_to_id[np.where(di != 0xFFFFFFFF, di, 0)], -1)
    f_ids = np.where(fi != 0xFFFFFFFF, snap.node_ids[np.where(fi != 0xFFFFFFFF, fi, 0)].astype(np.int64), -1)
    bad = np.argwhere(d_ids != f_ids)
    for (r, j) in bad:     # every difference must sit on an exact tie (or the k-th boundary)
        tied = (j > 0 and abs(dd[r, j] - dd[r, j - 1]) < 1e-10) or (j < 4 and abs(dd[r, j] - dd[r, j + 1]) < 1e-10) or j == 4
        assert tied, (r, j, dd[r], d_ids[r], f_ids[r])
    assert len(np.unique(bad[:, 0])) <= int(c1.knn_tie_queries - c0.knn_tie_queries) + 0 if len(bad) else True
    return len(bad)


def _replay_recorded_stream_on_the_device():
    rng = np.random.default_rng(17)
    dev = plugin.MeasurementModel(1)
    ev0 = next(scripted_stream())
    dev.map_build(ev0[1], ev0[2], ev0[3])
    h2d0 = dev.counters().h2d_bytes
    scans = 0
    for ev, ndel, cnt, sync, valid, digest in recorded_stream():
        _, a, ny, ids, b, ny2, ids2, boxes = ev
        if boxes is not None:
            assert ndel == dev.map_delete_boxes(boxes)
        dev.map_sync_voxels(sync, want_count=(scans % 2 == 0))
        if scans % 2:
            for k in ("boxes", "xyz", "normal_y", "ids"):
                sync[k][...] = 0
        dev.map_add_points(b, ny2, ids2)
        b[...] = 0
        m = dev.map_download()
        assert live_set_digest(m["xyz"], m["normal_y"], m["ids"]) == digest, scans
        live, slots = dev.map_info()
        assert live == valid
        scans += 1
        if scans % 10 == 0:
            _check_knn(dev, static_snapshot_of(m["xyz"], m["normal_y"], m["ids"]), rng)
    per_scan = (dev.counters().h2d_bytes - h2d0) / 50.0
    assert per_scan < 5 * 20000 * 12 / 50.0 + 40000, per_scan
    dev.close()


def test_fifty_scan_delta_stream_tracks_the_real_tree():
    if not po.ref_available():
        _replay_recorded_stream_on_the_device()
        return
    rng = np.random.default_rng(17)
    tree = po.RefTree(box_length=0.5)
    dev = plugin.MeasurementModel(1)
    h2d0 = None
    scans = 0
    for ev in scripted_stream(seed=2, M=60000, scans=50):
        if ev[0] == "build":
            tree.build(ev[1], ev[2], ev[3]); dev.map_build(ev[1], ev[2], ev[3])
            h2d0 = dev.counters().h2d_bytes
            continue
        _, a, ny, ids, b, ny2, ids2, boxes = ev
        if boxes is not None:
            assert tree.delete_boxes(boxes) == dev.map_delete_boxes(boxes)
        cnt, sync = tree.add_points_synced(a, ny, ids, 0.5)
        # every other scan without the kill count: the call then returns without waiting for the device, and the host arrays may be
        # overwritten at once (they went through the library's bounce buffer)
        dev.map_sync_voxels(sync, want_count=(scans % 2 == 0))
        if scans % 2:
            for k in ("boxes", "xyz", "normal_y", "ids"):
                sync[k][...] = 0
        tree.add_points(b, ny2, ids2, downsample=False); dev.map_add_points(b, ny2, ids2)
        b[...] = 0
        tree.wait_rebuild()
        m = dev.map_download()
        assert same_set(tree, (m["xyz"], m["normal_y"], m["ids"])), scans
        live, slots = dev.map_info()
        assert live == tree.validnum()
        scans += 1
        if scans % 10 == 0:
            nodes, cov, ids, depth, _ = tree.snapshot()
            _check_knn(dev, plugin.MapSnapshot(nodes, cov, ids, depth), rng)
    per_scan = (dev.counters().h2d_bytes - h2d0) / 50.0
    # k-NN test queries are uploads too (5 x 20k x 12 B); what remains is the deltas: ~500 points + boxes per scan
    assert per_scan < 5 * 20000 * 12 / 50.0 + 40000, per_scan
    dev.close(); tree.close()


def test_measurement_pass_on_the_device_resident_map_equals_snapshot_mode_and_compaction_keeps_it():
    """Snapshot mode on the churned reference tree where oracle/_ref is built, else on the static snapshot of the map."""
    case = synth.make_case("mapmode", 20000, 200000, 3, 3)
    snap, tree = H.snapshot_for(case, churn=True)
    if tree is not None:
        fx, fny, fid = tree.flatten_points()
    else:
        fx, fny, fid = case.map_xyz, case.map_normal_y, np.arange(case.map_xyz.shape[0], dtype=np.int32)
    ref = H.make_model(case, snap)                       # snapshot (tree) mode
    dev = plugin.MeasurementModel(3, params=case.params)  # device-resident map built from the same live points
    dev.map_build(fx, fny, fid)
    dev.upload_scan(case.pts, case.table, case.table_off, case.temporal_comp)

    def compare():
        ok1, H1, h1, s1 = ref.h_share_model(case.x_prop, True)
        c0 = dev.counters()
        ok2, H2, h2, s2 = dev.h_share_model(case.x_prop, True)
        ties = dev.counters().knn_tie_queries - c0.knn_tie_queries
        a1, a2 = ref.aux(), dev.aux()
        assert ok1 and ok2
        assert np.array_equal(a1["nn_sqdist"], a2["nn_sqdist"]) and np.array_equal(a1["world"], a2["world"])
        if ties == 0:
            assert np.array_equal(a1["selected"], a2["selected"]) and s1.n_eff == s2.n_eff
            assert H.rel_err(H2, H1) < 1e-11 and H.rel_err(h2, h1) < 1e-11
        x1, P1 = case.x_prop.copy(), case.P_prop.copy()
        x2, P2 = case.x_prop.copy(), case.P_prop.copy()
        ref.rearm_scan(); dev.rearm_scan()
        r1 = ref.update_iterated_dyn_share_modified(x1, P1, 3)
        r2 = dev.update_iterated_dyn_share_modified(x2, P2, 3)
        assert r1.passes == r2.passes and np.abs(synth.state_to_vec(x1, 3) - synth.state_to_vec(x2, 3)).max() < 1e-9
    compare()
    # kill 60 % of the map -> the next commit compacts; the survivors must answer exactly like a fresh snapshot of them
    lo = fx.min(0); hi = fx.max(0)
    cut = lo[0] + 0.6 * (hi[0] - lo[0])
    box = np.array([[lo[0] - 1, lo[1] - 1, lo[2] - 1, cut, hi[1] + 1, hi[2] + 1]], np.float32)
    if tree is not None:
        assert tree.delete_boxes(box) == dev.map_delete_boxes(box)
        tree.wait_rebuild()
        n_live = tree.validnum()
        nodes, cov, ids, depth, _ = tree.snapshot()
        survivors = plugin.MapSnapshot(nodes, cov, ids, depth)
    else:
        keep = ~np.all((box[0, :3] <= fx) & (box[0, 3:] > fx), axis=1)    # half-open boxes, as Delete_Point_Boxes
        assert int((~keep).sum()) == dev.map_delete_boxes(box)
        n_live = int(keep.sum())
        survivors = static_snapshot_of(fx[keep], fny[keep], fid[keep])
    live, slots = dev.map_info()
    assert live == slots == n_live and dev.counters().map_compactions == 1
    ref.upload_map(survivors)
    compare()
    ref.close(); dev.close()
    if tree is not None:
        tree.close()
