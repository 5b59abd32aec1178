"""Generates tests/golden/ikd_ref_golden.npz from the REAL reference ikd-Tree (oracle/_ref, built by `make -C oracle ref`
where the reference sources are present).  Run there:

    python tests/golden/make_ref_golden.py

Contents, so that the tests that compare with the reference tree also run where it cannot be built:
  * compact_*: what include/malio_flatten.hpp's compact flattener emits for the churned tree of make_golden.py (the tree is
    rebuilt here and checked to equal the committed snapshot of ikd_knn_golden.npz first): SHA-256 of the points and of the
    covariances, the depth and the root box.
  * stream_*: the 50-scan scripted stream of tests/test_mapops_cpu.py (seed 1, 20k-point map) as the tree answers it: per scan
    the Delete_Point_Boxes count, the Add_Points return value, the per-voxel re-synchronisation record of
    malio::collect_voxel_sync (voxel index of each box, live count per box, point ids; coordinates and normal_y follow from
    the ids through the seeded stream), KD_TREE::validnum() and a SHA-256 of KD_TREE::flatten() sorted by id.
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (os.path.join(ROOT, "ma-lio_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import pyoracle as po  # noqa: E402
from malio_b200 import synth  # noqa: E402
from test_mapops_cpu import scripted_stream, live_set_digest, VOXEL  # noqa: E402


def golden_tree():
    """The churned tree of make_golden.py, step for step."""
    rng = np.random.default_rng(2024)
    xyz = synth.make_world(6000, seed=11)
    ny = rng.uniform(0.0005, 0.01, xyz.shape[0]).astype(np.float32)
    tree = po.RefTree(box_length=0.5)
    tree.build(xyz, ny)
    add = xyz[rng.integers(0, 6000, 600)] + rng.normal(0, 0.3, (600, 3)).astype(np.float32)
    tree.add_points(add, rng.uniform(0.0005, 0.01, 600).astype(np.float32), downsample=True)
    add2 = xyz[rng.integers(0, 6000, 200)] + rng.normal(0, 0.2, (200, 3)).astype(np.float32)
    tree.add_points(add2, None, downsample=False)
    c = xyz[100]
    tree.delete_boxes([[c[0] - 4, c[1] - 4, c[2] - 2, c[0] + 4, c[1] + 4, c[2] + 2]])
    tree.wait_rebuild()
    return tree


def record_stream(threads):
    tree = po.RefTree(box_length=0.5)
    r = {k: [] for k in ("ndel", "added", "nb", "vox", "counts", "ids", "valid", "digest")}
    for ev in scripted_stream():
        if ev[0] == "build":
            tree.build(ev[1], ev[2], ev[3])
            continue
        _, a, ny, ids, b, ny2, ids2, boxes = ev
        r["ndel"].append(tree.delete_boxes(boxes) if boxes is not None else -1)
        cnt, sync = tree.add_points_synced(a, ny, ids, VOXEL, threads=threads)
        assert sync["outside_own_box"] == 0
        vox = np.floor(sync["boxes"][:, :3] / np.float32(VOXEL)).astype(np.int16)
        lo = vox.astype(np.float32) * np.float32(VOXEL)
        assert np.array_equal(np.concatenate([lo, lo + np.float32(VOXEL)], 1), sync["boxes"])   # boxes follow from the voxel index
        r["added"].append(cnt); r["nb"].append(len(vox)); r["vox"].append(vox)
        r["counts"].append(sync["counts"].astype(np.uint16)); r["ids"].append(sync["ids"])
        tree.add_points(b, ny2, ids2, downsample=False)
        tree.wait_rebuild()
        r["valid"].append(tree.validnum())
        r["digest"].append(np.frombuffer(live_set_digest(*tree.flatten_points()), np.uint8))
    tree.close()
    return {k: (np.concatenate(v) if k in ("vox", "counts", "ids") else np.stack(v) if k == "digest" else np.array(v, np.int32))
            for k, v in r.items()}


def main():
    g = np.load(os.path.join(HERE, "ikd_knn_golden.npz"))
    tree = golden_tree()
    nodes, cov, _, depth, _ = tree.snapshot()
    assert nodes.view(np.uint8).tobytes() == g["nodes"].tobytes() and np.array_equal(cov, g["node_cov"]), "tree differs from ikd_knn_golden"
    pts, pcov, pdepth, box = tree.snapshot_compact()
    tree.close()
    s1, s8 = record_stream(1), record_stream(8)
    assert all(np.array_equal(s1[k], s8[k]) for k in s1), "the record depends on the thread count"
    out = os.path.join(HERE, "ikd_ref_golden.npz")
    np.savez_compressed(out, compact_sha=np.frombuffer(hashlib.sha256(pts.tobytes()).digest(), np.uint8),
                        compact_cov_sha=np.frombuffer(hashlib.sha256(pcov.tobytes()).digest(), np.uint8),
                        compact_depth=pdepth, compact_root_box=box, **{"stream_" + k: v for k, v in s1.items()})
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
