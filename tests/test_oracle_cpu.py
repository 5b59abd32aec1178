"""CPU tests (no GPU): the oracle against the reference's golden vectors / the real reference ikd-Tree, the oracle's
hand-rolled algebra against numpy/scipy, host-side logic, and the C-ABI surface of the product library."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import helpers as H
import np_oracle as npo
import pyoracle as po
from malio_b200 import capi, plugin, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "ikd_knn_golden.npz")
REF_GOLD = os.path.join(ROOT, "tests", "golden", "ikd_ref_golden.npz")


def load_golden():
    g = np.load(GOLD)
    nodes = g["nodes"].view(capi.MAP_NODE).reshape(-1)
    return g, nodes


# ------------------------------------------------------------------ K / N: pinned by the real reference
def test_restated_search_matches_reference_golden():
    """oracle's restated KD_TREE::Search + MANUAL_HEAP on the flattened snapshot == the real Nearest_Search
    (fixture produced by tests/golden/make_golden.py from the reference ikd_Tree.cpp)."""
    g, nodes = load_golden()
    ids, d2, found, visits = po.knn_snapshot(nodes, g["node_cov"], g["queries"], nthreads=2)
    assert np.array_equal(found, g["ref_found"])
    m = ids >= 0
    mapped = np.where(m, g["node_ids"][np.clip(ids, 0, None)], -1)
    assert np.array_equal(mapped, g["ref_ids"])
    assert np.array_equal(d2[m], g["ref_d2"][m])
    assert visits > 0


def test_flattener_semantics_golden():
    g, nodes = load_golden()
    live = (nodes["link"] & capi.LINK_POINT_DELETED) == 0
    assert int(live.sum()) == int(g["n_live"]) == int(g["tree_valid"])
    # DFS pre-order: live points come out exactly in KD_TREE::flatten order (ikd_Tree.cpp:1638-1648)
    assert np.array_equal(g["node_ids"][live], g["flat_ids"])
    # links: left child is i+1, right index in range, boxes contain their child point
    n = nodes.shape[0]
    hl = (nodes["link"] & capi.LINK_HAS_LEFT) != 0
    hr = (nodes["link"] & capi.LINK_HAS_RIGHT) != 0
    ri = (nodes["link"] & capi.LINK_INDEX_MASK).astype(np.int64)
    idx = np.arange(n)
    assert np.all(idx[hl] + 1 < n) and np.all(ri[hr] < n) and np.all(ri[hr] > idx[hr])
    lc = nodes["xyz"][idx[hl] + 1]
    lb = nodes["lbox"][hl]
    child_live = live[idx[hl] + 1]
    inside = (lc[:, 0] >= lb[:, 0]) & (lc[:, 0] <= lb[:, 1]) & (lc[:, 1] >= lb[:, 2]) & (lc[:, 1] <= lb[:, 3]) & \
             (lc[:, 2] >= lb[:, 4]) & (lc[:, 2] <= lb[:, 5])
    assert np.all(inside[child_live])


def test_restated_search_vs_real_tree_after_churn():
    """With oracle/_ref: a live churned tree.  Without: the churned tree stored in the golden file and its own answers."""
    if po.ref_available():
        case = synth.make_case("t", 3000, 40000, 1, 3, varied_map_cov=True)
        snap, tree = H.snapshot_for(case, churn=True)
        rng = np.random.default_rng(1)
        q = case.map_xyz[rng.integers(0, 40000, 4000)] + rng.normal(0, 0.3, (4000, 3)).astype(np.float32)
        r_ids, r_d2, r_pts, r_found = tree.knn(q, 5, nthreads=4)
        nodes, node_cov, node_ids = snap.nodes, snap.node_cov, snap.node_ids
    else:
        g, nodes = load_golden()
        q, r_ids, r_d2, r_pts, r_found = g["queries"], g["ref_ids"], g["ref_d2"], g["ref_pts"], g["ref_found"]
        node_cov, node_ids = g["node_cov"], g["node_ids"]
    ids, d2, found, _ = po.knn_snapshot(nodes, node_cov, q, nthreads=4)
    assert np.array_equal(found, r_found)
    m = ids >= 0          # the stored queries include some with fewer than 5 neighbours in range
    assert np.array_equal(np.where(m, node_ids[np.clip(ids, 0, None)], -1), r_ids)
    assert np.array_equal(d2[m], r_d2[m])
    assert np.array_equal(node_cov[ids][m], r_pts[:, :, 3][m])


def test_compact_flattener_and_tight_box_rule_on_the_real_tree():
    """malio::flatten_ikdtree_compact emits exactly the first 16 bytes of every full record, and the boxes the full
    flattener copies out of the churned reference tree (node_range_*) ARE the tight boxes of the live points below —
    the rule the device uses to rebuild them after a compact upload (ikd_Tree.cpp:1469-1635).  Without oracle/_ref: the
    churned tree stored in the golden file, and digests of what the compact flattener made of the same tree."""
    if po.ref_available():
        case = synth.make_case("t", 2000, 30000, 1, 3, varied_map_cov=True)
        snap, tree = H.snapshot_for(case, churn=True)
        pts, cov, depth, root_box = tree.snapshot_compact()
        nodes, node_cov, max_depth = snap.nodes, snap.node_cov, snap.max_depth
        assert pts.shape[0] == nodes.shape[0]
        assert np.array_equal(pts["xyz"], nodes["xyz"]) and np.array_equal(pts["link"], nodes["link"])
        assert np.array_equal(cov, node_cov)
    else:
        import hashlib
        g, nodes = load_golden()
        r = np.load(REF_GOLD)
        node_cov, max_depth = g["node_cov"], int(g["max_depth"])
        depth, root_box = int(r["compact_depth"]), r["compact_root_box"]
        assert hashlib.sha256(plugin.compact_points(nodes).tobytes()).digest() == r["compact_sha"].tobytes()
        assert hashlib.sha256(node_cov.tobytes()).digest() == r["compact_cov_sha"].tobytes()
    assert depth == max_depth
    n = nodes.shape[0]
    link = nodes["link"]
    lo = np.full((n, 3), np.inf, np.float32)
    hi = np.full((n, 3), -np.inf, np.float32)
    for i in range(n - 1, -1, -1):            # children have larger indices than their parent (DFS pre-order)
        if not (link[i] & capi.LINK_POINT_DELETED):
            lo[i] = np.minimum(lo[i], nodes["xyz"][i]); hi[i] = np.maximum(hi[i], nodes["xyz"][i])
        if link[i] & capi.LINK_HAS_LEFT:
            c = i + 1
            assert np.array_equal(nodes["lbox"][i], np.stack([lo[c], hi[c]], 1).reshape(6)), i
            lo[i] = np.minimum(lo[i], lo[c]); hi[i] = np.maximum(hi[i], hi[c])
        if link[i] & capi.LINK_HAS_RIGHT:
            c = int(link[i] & capi.LINK_INDEX_MASK)
            assert np.array_equal(nodes["rbox"][i], np.stack([lo[c], hi[c]], 1).reshape(6)), i
            lo[i] = np.minimum(lo[i], lo[c]); hi[i] = np.maximum(hi[i], hi[c])
    assert np.array_equal(root_box, np.stack([lo[0], hi[0]], 1).reshape(6))


@pytest.mark.skipif(not po.ref_available(), reason="oracle/_ref (real ikd_Tree.cpp) only exists in the build container")
def test_parallel_flatteners_equal_the_serial_ones_on_the_real_tree():
    """malio::flatten_ikdtree_parallel / _compact_parallel (OpenMP, slots from subtree sizes) must produce the serial
    flatteners' output byte for byte on the churned reference tree, for grains from 'everything in one item' to 'tops
    all the way down'."""
    case = synth.make_case("t", 2000, 60000, 1, 3, varied_map_cov=True)
    snap, tree = H.snapshot_for(case, churn=True)
    nodes, cov, ids, depth, live = tree.snapshot()
    pts, pcov, pdepth, box = tree.snapshot_compact()
    for grain in (1 << 30, 16384, 4096, 1024):
        n2, c2, i2, d2, l2 = tree.snapshot_parallel(grain)
        assert n2.tobytes() == nodes.tobytes() and np.array_equal(c2, cov) and np.array_equal(i2, ids)
        assert d2 == depth and l2 == live
        p2, pc2, pd2, b2 = tree.snapshot_compact_parallel(grain)
        assert p2.tobytes() == pts.tobytes() and np.array_equal(pc2, pcov) and pd2 == pdepth and np.array_equal(b2, box)


def test_search_is_exact_knn_bruteforce():
    rng = np.random.default_rng(3)
    xyz = (rng.random((5000, 3)) * [40, 40, 4]).astype(np.float32)
    snap = plugin.build_static_snapshot(xyz)
    q = (rng.random((300, 3)) * [40, 40, 4]).astype(np.float32)
    ids, d2, found, _ = po.knn_snapshot(snap.nodes, snap.node_cov, q)
    d = q[:, None, :] - xyz[None, :, :]
    bd = (d[:, :, 0] * d[:, :, 0] + d[:, :, 1] * d[:, :, 1]) + d[:, :, 2] * d[:, :, 2]
    bi = np.argsort(bd, axis=1, kind="stable")[:, :5]
    assert np.array_equal(np.sort(snap.node_ids[ids], 1), np.sort(bi, 1))
    assert np.array_equal(d2, np.take_along_axis(bd, bi, 1))


def test_static_snapshot_builder_invariants():
    xyz = synth.make_world(20000, seed=5)
    snap = plugin.build_static_snapshot(xyz, np.linspace(0.001, 0.01, 20000, dtype=np.float32))
    assert sorted(snap.node_ids.tolist()) == list(range(20000))
    assert np.array_equal(snap.nodes["xyz"], xyz[snap.node_ids])
    assert np.allclose(snap.node_cov, np.linspace(0.001, 0.01, 20000, dtype=np.float32)[snap.node_ids])
    assert snap.max_depth == 15   # ceil(log2(20001))
    # subtree sizes implied by the links are consistent: right child index = i + 1 + size(left)
    n = 20000
    link = snap.nodes["link"]
    hr = (link & capi.LINK_HAS_RIGHT) != 0
    ri = (link & capi.LINK_INDEX_MASK)[hr]
    assert np.all(ri > np.arange(n)[hr])
    # the oracle's restated builder (bench.py's CPU arm) gives the same snapshot byte for byte
    o = po.build_static_snapshot(xyz, np.linspace(0.001, 0.01, 20000, dtype=np.float32))
    assert o.nodes.tobytes() == snap.nodes.tobytes() and np.array_equal(o.node_cov, snap.node_cov)
    assert np.array_equal(o.node_ids, snap.node_ids) and o.max_depth == snap.max_depth


# ------------------------------------------------------------------ P / U / algebra vs numpy
def test_esti_plane_vs_scipy_qr():
    L = po.oracle_lib()
    rng = np.random.default_rng(0)
    for trial in range(300):
        nrm = rng.normal(size=3); nrm /= np.linalg.norm(nrm)
        base = rng.normal(size=3) * 8
        u = np.cross(nrm, rng.normal(size=3)); u /= np.linalg.norm(u)
        v = np.cross(nrm, u)
        pts = base + rng.uniform(-1, 1, (5, 1)) * u + rng.uniform(-1, 1, (5, 1)) * v + rng.normal(0, 0.02 if trial % 3 else 0.3, (5, 1)) * nrm
        near = np.zeros((5, 4), np.float32)
        near[:, :3] = pts
        near[:, 3] = rng.uniform(0, 0.02, 5) if trial % 5 else 0.0
        pab = np.zeros(4, np.float32)
        pc = C.c_double(0)
        ok = L.orc_esti_plane(po.ptr(near), C.c_float(0.4), C.c_double(0.5), po.ptr(pab), C.byref(pc))
        ok2, pab2, pc2 = npo.esti_plane(near, np.float32(0.4), 0.5)
        resid = np.abs(near[:, :3].astype(np.float64) @ pab[:3] + pab[3])
        if abs(resid.max() - 0.4) > 1e-3:
            assert bool(ok) == ok2
        # float32 LSQ of A n = -1 is conditioned like |p|^2: two valid float QRs agree to ~1e-3 here
        np.testing.assert_allclose(pab, pab2, rtol=3e-3, atol=3e-4)
        assert pc.value == pytest.approx(pc2, rel=1e-12, abs=1e-18)


def test_eval_point_uncertainty_vs_numpy():
    L = po.oracle_lib()
    rng = np.random.default_rng(1)
    table, _ = synth.make_tables(1, 6, rng)
    for j in range(6):
        p = rng.normal(0, 30, 3).astype(np.float32)
        cov = np.zeros(9)
        L.orc_eval_point_uncertainty(po.ptr(p), po.ptr(table[j:j + 1]), po.ptr(cov))
        ref = npo.eval_point_uncertainty(p, table[j]["T"], table[j]["cov"])
        np.testing.assert_allclose(cov.reshape(3, 3), ref, rtol=1e-12)


def test_inverse_and_singular_values_vs_numpy():
    L = po.oracle_lib()
    rng = np.random.default_rng(2)
    A = rng.normal(size=(35, 35))
    A = A @ A.T + np.eye(35)
    inv = np.zeros((35, 35))
    assert L.orc_inverse(po.ptr(A), 35, po.ptr(inv)) == 1
    np.testing.assert_allclose(inv, np.linalg.inv(A), rtol=1e-9, atol=1e-12)
    M = rng.normal(size=(500, 24)) * [3, 1, 0.2] + [0] * 24 if False else rng.normal(size=(500, 24))
    M[:, :3] *= [3.0, 1.0, 0.2]
    sv = np.zeros(3)
    L.orc_singular_values_Nx3(po.ptr(M), 500, 24, po.ptr(sv))
    np.testing.assert_allclose(sv, np.linalg.svd(M[:, :3], compute_uv=False), rtol=1e-10)


def test_manifold_ops_vs_numpy_and_roundtrip():
    L = po.oracle_lib()
    case = synth.make_case("m", 100, 5000, 3, 3)
    rng = np.random.default_rng(4)
    for _ in range(20):
        d = rng.normal(0, 0.05, 35)
        x = case.x_prop.copy()
        L.orc_state_boxplus(3, C.byref(x), po.ptr(d))
        back = np.zeros(35)
        L.orc_state_boxminus(3, C.byref(x), C.byref(case.x_prop), po.ptr(back))
        np.testing.assert_allclose(back, d, atol=1e-9)
        xn = npo.NpState(case.x_prop, 3)
        npo.boxplus(xn, d)
        np.testing.assert_allclose(synth.state_to_vec(x, 3), xn.vec(), atol=1e-12)
        v = rng.normal(0, 0.3, 3)
        A = np.zeros(9)
        L.orc_A_matrix(po.ptr(v), po.ptr(A))
        np.testing.assert_allclose(A.reshape(3, 3), npo.A_matrix(v), atol=1e-14)
        g = np.array(x.grav[:])
        Nx = np.zeros(6); Mx = np.zeros(6)
        dl = rng.normal(0, 0.01, 2)
        L.orc_S2_Nx_yy(po.ptr(g), po.ptr(Nx)); L.orc_S2_Mx(po.ptr(g), po.ptr(dl), po.ptr(Mx))
        np.testing.assert_allclose(Nx.reshape(2, 3), npo.S2_Nx_yy(g), atol=1e-13)
        np.testing.assert_allclose(Mx.reshape(3, 2), npo.S2_Mx(g, dl), atol=1e-12)


# ------------------------------------------------------------------ B / A on a small case
@pytest.fixture(scope="module")
def small():
    case = synth.make_case("small-3L", 3000, 40000, 3, 3, varied_map_cov=True)
    snap = plugin.build_static_snapshot(case.map_xyz, case.map_normal_y)
    return case, snap


def test_oracle_reduction_equals_dense(small):
    case, snap = small
    orc = H.make_oracle(case, snap)
    assert orc.h_share_model(case.x_prop, True, 2)
    hx, h, R = orc.dense()
    Rc = np.where(R < 1e-4, 1e-3, R)
    HTH, HTh = orc.reduce()
    np.testing.assert_allclose(HTH, (hx.T / Rc) @ hx, rtol=1e-10)
    np.testing.assert_allclose(HTh, (hx.T / Rc) @ h, rtol=1e-10)
    st = orc.stats()
    assert st.n_eff == hx.shape[0] > 2000
    assert 0.3 <= st.loc_weight <= 2.0
    # each row has at most 12 non-zeros: cols 0-5, 6+3l, 6+3(L+l) of its LiDAR
    sel = orc.aux()["selected"].astype(bool)
    lid = case.pts["lidar"][sel]
    for l in range(3):
        rows = hx[lid == l]
        mask = np.ones(24, bool)
        mask[0:6] = False; mask[6 + 3 * l:9 + 3 * l] = False; mask[15 + 3 * l:18 + 3 * l] = False
        assert np.all(rows[:, mask] == 0)
        assert np.all(np.abs(rows[:, ~mask]).sum(1) > 0)


def test_jacobian_rows_match_finite_differences(small):
    """h_x (laserMapping.cpp:665-693) against d(pd2)/d(delta x) by central differences on the manifold, with the
    neighbours / planes frozen (converge = false)."""
    case, snap = small
    L_ = po.oracle_lib()
    orc = H.make_oracle(case, snap)
    x0 = case.x_prop.copy()
    assert orc.h_share_model(x0, True, 2)

    def unweighted(state):
        assert orc.h_share_model(state, False, 2)
        hx, h, _ = orc.dense()
        sel = np.flatnonzero(orc.aux()["selected"])
        w = np.linalg.norm(hx[:, :3], axis=1)          # = plane weight * localization weight (|n| = 1)
        return sel, hx / w[:, None], -h / w

    sel0, J0, pd0 = unweighted(x0)
    eps = 1e-6
    for k in list(range(0, 24)):
        d = np.zeros(35); d[k] = eps
        xp, xm = x0.copy(), x0.copy()
        L_.orc_state_boxplus(3, C.byref(xp), po.ptr(d))
        L_.orc_state_boxplus(3, C.byref(xm), po.ptr(-d))
        sp, _, pdp = unweighted(xp)
        sm, _, pdm = unweighted(xm)
        common = np.intersect1d(np.intersect1d(sp, sm), sel0)
        fd = (pdp[np.searchsorted(sp, common)] - pdm[np.searchsorted(sm, common)]) / (2 * eps)
        an = J0[np.searchsorted(sel0, common), k]
        # pd2 is evaluated in float32 on float32 world points: ~1e-6 m noise / 2e-6 => O(1) absolute noise per
        # point; compare in aggregate (robust) form
        err = np.abs(fd - an)
        assert np.median(err) < 0.6, (k, np.median(err))
        scale = max(np.abs(an).max(), 1.0)
        assert np.corrcoef(fd, an)[0, 1] > 0.99 or np.abs(an).max() < 1.0, k


def test_ieskf_update_vs_numpy_restatement(small):
    """oracle A (C++) against the numpy restatement fed with the same dense rows."""
    case, snap = small
    orc = H.make_oracle(case, snap)
    xo, Po = case.x_prop.copy(), case.P_prop.copy()
    rc, dx_log, flags, rep = orc.update_iterated(xo, Po, case.max_iter, nthreads=2)
    assert rc == 0
    orc2 = H.make_oracle(case, snap)

    def measure(xn, converge):
        s = capi.PassState()
        s.rot[:] = list(xn.rot); s.pos[:] = list(xn.pos)
        for l in range(3):
            s.ext[l].q[:] = list(xn.eq[l]); s.ext[l].t[:] = list(xn.et[l])
        ok = orc2.h_share_model(s, converge, 2)
        if not ok:
            return False, None, None, None
        return (True,) + orc2.dense()

    xn, Pn, dxn_log = npo.ieskf_update(measure, npo.NpState(case.x_prop, 3), case.P_prop.copy(), case.max_iter)
    np.testing.assert_allclose(synth.state_to_vec(xo, 3), xn.vec(), atol=1e-9)
    np.testing.assert_allclose(Po, Pn, rtol=1e-6, atol=1e-14)
    for a, b in zip(dx_log, dxn_log):
        if b is not None:
            np.testing.assert_allclose(a, b, atol=1e-9)
    assert rep.passes == len(dxn_log)


def test_degenerate_cases(small):
    case, snap = small
    # no effective points: empty map far away -> valid = false on every pass, state untouched
    far = plugin.build_static_snapshot(case.map_xyz[:50] + np.float32(1e4))
    orc = H.make_oracle(case, far)
    assert not orc.h_share_model(case.x_prop, True, 1)
    x, P = case.x_prop.copy(), case.P_prop.copy()
    rc, _, flags, rep = orc.update_iterated(x, P, 3)
    assert rc == 1 and np.all(flags & 1 == 0)
    assert np.array_equal(synth.state_to_vec(x, 3), synth.state_to_vec(case.x_prop, 3))
    # fewer effective points than state DOF: the dense branch (esekfom.hpp:574-582)
    sub = synth.make_case("tiny", 25, 40000, 3, 3, map_xyz=case.map_xyz)
    orc = H.make_oracle(sub, snap)
    assert orc.h_share_model(sub.x_prop, True, 1)
    assert 1 <= orc.n_eff() < 35
    x, P = sub.x_prop.copy(), sub.P_prop.copy()
    rc, dx_log, flags, rep = orc.update_iterated(x, P, 3)
    assert rc == 0 and np.all(np.isfinite(synth.state_to_vec(x, 3))) and np.all(np.isfinite(P))
    # all-equal point covariances: FIC 0/0 defined as mid-range (SURVEY.md quirk 8)
    eq = synth.make_case("eqcov", 500, 40000, 1, 3, map_xyz=case.map_xyz)
    eq.table["cov"][:] = 0.0
    eq.pts["xyz"][:] = eq.pts["xyz"][0]          # same point, same table entry -> identical traces
    eq.pts["table_idx"][:] = 0
    orc = po.Oracle(eq.params)
    orc.set_map_snapshot(snap.nodes, snap.node_cov)
    orc.set_scan(eq.pts, eq.table, eq.table_off, eq.temporal_comp)
    if orc.h_share_model(eq.x_prop, True, 1):
        _, _, R = orc.dense()
        assert np.all(R == (eq.params.point_cov_max + eq.params.point_cov_min) / 2)


# ------------------------------------------------------------------ the product library's surface (no compute calls)
def test_cabi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "malio_b200.h")).read()
    declared = set(re.findall(r"\b(malio_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"malio_flatten"}
    lib = capi.load()
    missing = [n for n in sorted(declared) if not hasattr(lib, n)]
    assert not missing, missing
    assert set(capi.EXPORTS) <= declared
    assert lib.malio_version().startswith(b"malio_b200")
    # struct layouts shared with the C side
    assert C.sizeof(capi.PassState) == 8 * (4 + 3 + 3 * 7)
    assert C.sizeof(capi.Rigid) == 56 and capi.MAP_NODE.itemsize == 64 and capi.SCAN_PT.itemsize == 16
    p = capi.default_params(3)
    assert p.n_lidar == 3 and p.plane_th == pytest.approx(0.4) and p.knn_max_sqdist == 5.0 and p.cov_threshold == 0.5


def test_product_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(capi.MalioError) as e:
        plugin.MeasurementModel(1)
    assert e.value.status == capi.ERR_CUDA
    cfg = capi.Config(); cfg.params = capi.default_params(5); cfg.params.n_lidar = 5
    h = C.c_void_p()
    assert capi.load().malio_create(C.byref(h), C.byref(cfg)) == capi.ERR_INVALID_ARG


def test_product_does_not_link_or_import_the_oracle():
    """The product must never route through oracle/ (no CPU fallback): no source under ma-lio_b200/ mentions it,
    and the shared library has no dependency on the checker libraries."""
    pkg = os.path.join(ROOT, "ma-lio_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cpp", ".cu", ".h", ".hpp")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                assert "pyoracle" not in txt and "liboracle" not in txt and "libikd_ref" not in txt, f
    import subprocess
    out = subprocess.run(["ldd", capi.lib_path()], capture_output=True, text=True).stdout
    assert "oracle" not in out and "ikd_ref" not in out


def test_map_incremental_decision_vs_numpy_restatement(small):
    """SURVEY §8f N1: the per-point decision of map_incremental (laserMapping.cpp:398-446) — the C++ restatement against
    an independent numpy one on the same Nearest_Points / normal_y / state."""
    case, snap = small
    orc = H.make_oracle(case, snap)
    x, P = case.x_prop.copy(), case.P_prop.copy()
    orc.update_iterated(x, P, case.max_iter)
    fs = 0.5
    cls, w = orc.map_incremental(x, fs, True)
    a = orc.aux()
    xyz = snap.nodes["xyz"]
    ids = a["nn_idx"]
    cnt = a["nn_cnt"]
    keep = ~(a["normal_y"].astype(np.float64) > case.params.cov_threshold)
    assert np.all(cls[~keep] == capi.MAP_SKIP) and np.all(cls[keep] != capi.MAP_SKIP)
    mid = (np.floor(w.astype(np.float64) / fs) * fs + 0.5 * fs).astype(np.float32)
    d = w - mid
    dist = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    exp = np.full(len(cls), capi.MAP_ADD, np.uint8)
    for i in np.nonzero(keep)[0]:
        if cnt[i] == 0:
            continue
        n0 = xyz[ids[i, 0]]
        if np.all(np.abs(n0 - mid[i]).astype(np.float64) > 0.5 * fs):
            exp[i] = capi.MAP_ADD_NO_DOWNSAMPLE
            continue
        if cnt[i] >= 5:
            q = xyz[ids[i]] - mid[i]
            dj = (q[:, 0] * q[:, 0] + q[:, 1] * q[:, 1]) + q[:, 2] * q[:, 2]
            if np.any(dj < dist[i]):
                exp[i] = capi.MAP_DROP
    exp[~keep] = capi.MAP_SKIP
    assert np.array_equal(cls, exp)
    assert len(set(cls.tolist())) >= 2          # the case exercises more than one branch
    # before the filter is initialised every kept point is added (:411, :439-440)
    cls0, _ = orc.map_incremental(x, fs, False)
    assert np.all(cls0[keep] == capi.MAP_ADD)


# ------------------------------------------------------------------ SURVEY §8f N3: pose-uncertainty table (host code)
def _rand_pose(rng, ang, tr, cov_scale):
    v = rng.normal(size=3); v *= ang / np.linalg.norm(v)
    q = npo.so3_exp(v)
    t = rng.normal(size=3) * tr
    A = rng.normal(size=(6, 6)) * np.sqrt(cov_scale)
    return npo.Pose(q, t, A @ A.T)


def _to_c(p):
    a = np.zeros(1, dtype=capi.POSE)
    a["q"][0] = p.q; a["t"][0] = p.t; a["T"][0] = p.T; a["cov"][0] = p.cov
    return a


def test_pose_compounding_and_table_vs_numpy():
    """Barfoot's 4th-order SE(3) covariance compounding (associate_uct.hpp:29-142) and the pose_unc table loop
    (laserMapping.cpp:1028-1048) in the product's host code against the numpy restatement — including the calls whose
    output aliases the second input (the adjoint then sees the overwritten T_, associate_uct.hpp:99)."""
    import ctypes as C
    lib = capi.load()
    rng = np.random.default_rng(7)
    p1, p2 = _rand_pose(rng, 0.3, 0.5, 1e-4), _rand_pose(rng, 0.2, 0.3, 1e-5)
    for fn_c, fn_np, sets_pose_cov in ((lib.malio_compound_pose_with_cov, npo.compound_pose_with_cov, True),
                                       (lib.malio_compound_inv_pose_with_cov, npo.compound_inv_pose_with_cov, False)):
        # (a) separate output
        c1, c2, co = _to_c(p1), _to_c(p2), np.zeros(1, dtype=capi.POSE)
        cov_out = np.zeros((6, 6))
        fn_c(capi.ptr(c1), capi.ptr(np.ascontiguousarray(p1.cov)), capi.ptr(c2), capi.ptr(np.ascontiguousarray(p2.cov)),
             capi.ptr(co), capi.ptr(cov_out))
        out = npo.Pose([1, 0, 0, 0], [0, 0, 0], np.zeros((6, 6)))
        ref_cov = fn_np(p1, p1.cov, p2.copy(), p2.cov, out)
        np.testing.assert_allclose(cov_out, ref_cov, rtol=1e-11, atol=1e-18)
        np.testing.assert_allclose(co["T"][0], out.T, rtol=1e-13, atol=1e-15)
        np.testing.assert_allclose(co["q"][0], out.q, rtol=1e-13, atol=1e-15)
        assert np.allclose(cov_out, cov_out.T, rtol=1e-12, atol=1e-20) and np.all(np.linalg.eigvalsh(cov_out) > -1e-15)
        if sets_pose_cov:
            assert np.array_equal(co["cov"][0], cov_out)
        # (b) output aliasing the second input, cov_cp = pose_cp.cov (the reference's call pattern)
        c2b = _to_c(p2)
        cov_alias = c2b["cov"][0]           # view into the struct: cov_cp IS pose_cp.cov
        fn_c(capi.ptr(c1), capi.ptr(np.ascontiguousarray(p1.cov)), capi.ptr(c2b), capi.ptr(np.ascontiguousarray(p2.cov)),
             capi.ptr(c2b), c2b["cov"].ctypes.data_as(C.c_void_p))
        pa = p2.copy()
        ref_alias = fn_np(p1, p1.cov, pa, pa.cov.copy(), pa)
        np.testing.assert_allclose(cov_alias, ref_alias, rtol=1e-11, atol=1e-18)
        np.testing.assert_allclose(c2b["T"][0], pa.T, rtol=1e-13, atol=1e-15)
    # first-order sanity: tiny covariances -> cov_cp ~= Ad cov_1 Ad^T + cov_2
    s1, s2 = _rand_pose(rng, 0.3, 0.5, 1e-12), _rand_pose(rng, 0.2, 0.3, 1e-12)
    out = npo.Pose([1, 0, 0, 0], [0, 0, 0], np.zeros((6, 6)))
    cov = npo.compound_pose_with_cov(s1, s1.cov, s2, s2.cov, out)
    Ad = npo.adjoint(np.linalg.inv(s2.T))
    np.testing.assert_allclose(cov, Ad @ s1.cov @ Ad.T + s2.cov, rtol=1e-9, atol=1e-24)
    # ---- the table of one scan, 3 LiDARs
    ext = [_rand_pose(rng, 0.05 + 0.5 * l, 0.3, 1e-8) for l in range(3)]
    tcomp = [_rand_pose(rng, 0.01, 0.05, 1e-8) for _ in range(2)]
    lists = [[_rand_pose(rng, 0.02, 0.02 * (j + 1), 1e-7 * (j + 1)) for j in range(n)] for n in (9, 6, 7)]
    ref = npo.build_pose_unc(ext, tcomp, lists)
    table, off = plugin.build_pose_unc(np.concatenate([_to_c(p) for p in ext]), np.concatenate([_to_c(p) for p in tcomp]),
                                       [np.concatenate([_to_c(p) for p in l]) for l in lists])
    assert off.tolist() == [0, 8, 13, 19] and table.shape[0] == 19
    k = 0
    for l in range(3):
        for p in ref[l]:
            np.testing.assert_allclose(table["T"][k], p.T, rtol=1e-12, atol=1e-14)
            np.testing.assert_allclose(table["cov"][k], p.cov, rtol=1e-10, atol=1e-20)
            k += 1
    # LiDAR 0's entries are copied verbatim (:1034-1036); single-LiDAR tables need no temporal_comp
    assert np.array_equal(table["cov"][0], lists[0][0].cov) and np.array_equal(table["T"][7], lists[0][7].T)
    t1, o1 = plugin.build_pose_unc(_to_c(ext[0]), None, [np.concatenate([_to_c(p) for p in lists[0]])])
    assert o1.tolist() == [0, 8] and np.array_equal(t1["cov"], table["cov"][:8])


def test_python_default_params_equal_the_library_defaults():
    """capi.default_params is restated in Python (so that bench.py --impl reference never maps the CUDA library): it must
    stay equal to malio_default_params()."""
    import ctypes as C
    for L in (1, 2, 3):
        a, b = capi.default_params(L), capi.default_params_from_library(L)
        assert bytes(C.string_at(C.byref(a), C.sizeof(a))) == bytes(C.string_at(C.byref(b), C.sizeof(b)))


def test_reference_arm_does_not_map_the_cuda_library_and_reports_the_split():
    """bench.py --impl reference: the CPU arm must not load libmalio_b200.so, must honour --steps and must report the
    K / B / A split at 3 threads and at all host threads (tiny stand-in workload: the arm itself is what is tested)."""
    import json, subprocess, sys, textwrap
    code = textwrap.dedent(f"""
        import sys, json
        sys.path.insert(0, {ROOT!r}); sys.argv = ['bench.py']
        import bench
        from malio_b200 import synth
        case = synth.make_case('mini', 3000, 30000, 3, 3)
        with bench.c_stdout_to_stderr():
            tree = bench.live_tree(case)
            best, runs = bench.cpu_arms(case, tree, 2, 1)
            if tree is not None: tree.close()
        mapped = [l for l in open('/proc/self/maps') if 'libmalio_b200' in l]
        print(json.dumps(dict(best=best, n_runs=len(runs), mapped=len(mapped))))
    """)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    r = json.loads(out.stdout.strip().splitlines()[-1])
    assert r["mapped"] == 0
    assert r["best"]["steps"] == 2 and set(r["best"]["split_ms_per_pass"]) == {"K_nearest_search", "B_h_share_model_rest", "A_ieskf_rest"}
    assert r["n_runs"] >= 1


def test_every_entry_point_survives_null_arguments():
    """C-ABI robustness without a GPU: every exported function called with NULL for every pointer and 0 for every scalar must
    return (an error code where it has one) instead of dereferencing — run in a subprocess, a missing check is a SIGSEGV."""
    import subprocess
    import sys
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "ma-lio_b200"))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "null_handle_probe.py")], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, (r.returncode, r.stdout[-400:], r.stderr[-400:])
    lines = [l.split() for l in r.stdout.strip().splitlines()]
    assert lines[-1] == ["DONE"]
    rc = {l[0]: l[1] for l in lines[:-1] if len(l) == 2}
    assert len(rc) >= 38
    for name, code in rc.items():
        takes_handle = name not in ("malio_default_params", "malio_build_static_snapshot", "malio_bspline_get_pose", "malio_pose_initial",
                                    "malio_compound_pose_with_cov", "malio_compound_inv_pose_with_cov", "malio_destroy", "malio_last_error")
        if takes_handle:
            assert code not in ("0", "ptr"), (name, code)      # an error code, never success
