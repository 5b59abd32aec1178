"""ctypes access to the CPU checkers.  TEST INFRASTRUCTURE ONLY.

  oracle/liboracle_malio.so   restated algorithm (oracle_malio.cpp)
  oracle/_ref/libikd_ref.so   the real reference ikd_Tree.cpp compiled in place (ref_ikd_capi.cpp)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
"""
from __future__ import annotations

import ctypes as C
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(_HERE), "ma-lio_b200"))
from malio_b200 import capi  # noqa: E402  (struct definitions only)

vp = C.c_void_p
_orc = None
_ref = None


def ptr(a):
    return capi.ptr(a)


def oracle_lib() -> C.CDLL:
    global _orc
    if _orc is None:
        path = os.path.join(_HERE, "liboracle_malio.so")
        if not os.path.exists(path):
            raise RuntimeError(f"{path} missing: make -C oracle")
        L = C.CDLL(path)
        L.orc_create.restype = vp
        L.orc_create.argtypes = [C.POINTER(capi.Params)]
        L.orc_destroy.argtypes = [vp]
        L.orc_set_map_snapshot.argtypes = [vp, vp, vp, C.c_uint32]
        L.orc_set_knn_hook.argtypes = [vp, vp, vp]
        L.orc_set_scan.argtypes = [vp, vp, C.c_uint32, vp, vp, vp]
        L.orc_knn_snapshot_batch.argtypes = [vp, vp, C.c_uint32, vp, C.c_int64, C.c_int, vp, vp, vp, C.POINTER(C.c_int64), C.c_int, vp]
        L.orc_esti_plane.argtypes = [vp, C.c_float, C.c_double, vp, C.POINTER(C.c_double)]
        L.orc_eval_point_uncertainty.argtypes = [vp, vp, vp]
        L.orc_qr_solve_5x3.argtypes = [vp, vp, vp]
        L.orc_inverse.argtypes = [vp, C.c_int, vp]
        L.orc_singular_values_Nx3.argtypes = [vp, C.c_int64, C.c_int64, vp]
        L.orc_state_boxplus.argtypes = [C.c_int, C.POINTER(capi.State), vp]
        L.orc_state_boxminus.argtypes = [C.c_int, C.POINTER(capi.State), C.POINTER(capi.State), vp]
        L.orc_A_matrix.argtypes = [vp, vp]
        L.orc_S2_Nx_yy.argtypes = [vp, vp]
        L.orc_S2_Mx.argtypes = [vp, vp, vp]
        L.orc_h_share_model.argtypes = [vp, C.POINTER(capi.PassState), C.c_int, C.c_int]
        L.orc_reduce.argtypes = [vp, vp, vp]
        L.orc_n_eff.argtypes = [vp]
        L.orc_set_minmax_override.argtypes = [vp, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double]
        L.orc_get_local_minmax.argtypes = [vp, vp]
        L.orc_partials.argtypes = [vp, vp, vp, vp]
        L.orc_get_stats.argtypes = [vp, C.POINTER(capi.PassStats)]
        L.orc_get_dense.argtypes = [vp, vp, vp, vp]
        L.orc_get_aux.argtypes = [vp, vp, vp, vp, vp, vp, vp]
        L.orc_map_incremental.restype = None
        L.orc_map_incremental.argtypes = [vp, vp, C.c_double, C.c_int, vp, vp]
        L.orc_get_visits.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.orc_reset_times.argtypes = [vp]
        L.orc_get_times.argtypes = [vp, vp, C.POINTER(C.c_int)]
        L.orc_set_fast_reduce.argtypes = [vp, C.c_int]
        L.orc_bspline_get_pose.argtypes = [vp, vp, C.c_int, C.c_double, vp, vp]
        L.orc_log_se3.argtypes = [vp, vp]
        L.orc_exp_se3.argtypes = [vp, vp]
        L.orc_quat_from_R.argtypes = [vp, vp]
        L.orc_undistort.restype = None
        L.orc_undistort.argtypes = [vp, C.c_int64, C.c_double, vp, vp, vp, vp, vp, vp, C.c_int, vp, C.c_int, C.c_int, vp, vp, vp, vp,
                                    C.POINTER(C.c_int32), vp]
        L.orc_voxel_grid.restype = C.c_int64
        L.orc_voxel_grid.argtypes = [vp, C.c_int64, C.c_float, vp, C.c_int64, vp]
        L.orc_update_iterated.argtypes = [vp, C.POINTER(capi.State), vp, C.c_int, C.c_double, C.c_int, vp, vp, C.POINTER(capi.UpdateReport)]
        L.orc_build_static_snapshot.argtypes = [vp, C.c_uint32, vp, vp, C.POINTER(C.c_uint32)]
        _orc = L
    return _orc


def ref_available() -> bool:
    return os.path.exists(os.path.join(_HERE, "_ref", "libikd_ref.so"))


def ref_lib() -> C.CDLL:
    global _ref
    if _ref is None:
        path = os.path.join(_HERE, "_ref", "libikd_ref.so")
        if not os.path.exists(path):
            raise RuntimeError(f"{path} missing (built only where /root/reference exists): make -C oracle ref")
        L = C.CDLL(path)
        L.ikdref_create.restype = vp
        L.ikdref_create.argtypes = [C.c_float, C.c_float, C.c_float]
        L.ikdref_destroy.argtypes = [vp]
        L.ikdref_build.argtypes = [vp, vp, vp, vp, C.c_int64]
        L.ikdref_add_points.argtypes = [vp, vp, vp, vp, C.c_int64, C.c_int]
        L.ikdref_delete_boxes.argtypes = [vp, vp, C.c_int]
        L.ikdref_wait_rebuild.argtypes = [vp]
        L.ikdref_size.argtypes = [vp]
        L.ikdref_validnum.argtypes = [vp]
        L.ikdref_knn.argtypes = [vp, vp, C.c_int64, C.c_int, vp, vp, vp, vp, C.c_int]
        L.ikdref_flatten_points.restype = C.c_int64
        L.ikdref_flatten_points.argtypes = [vp, vp, vp, vp, C.c_int64]
        L.ikdref_snapshot.restype = C.c_int64
        L.ikdref_snapshot.argtypes = [vp, vp, vp, vp, C.c_int64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.ikdref_snapshot_compact.restype = C.c_int64
        L.ikdref_snapshot_compact.argtypes = [vp, vp, vp, C.c_int64, C.POINTER(C.c_uint32), vp]
        L.ikdref_snapshot_parallel.restype = C.c_int64
        L.ikdref_snapshot_parallel.argtypes = [vp, vp, vp, vp, C.c_int64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.c_uint32]
        L.ikdref_snapshot_compact_parallel.restype = C.c_int64
        L.ikdref_snapshot_compact_parallel.argtypes = [vp, vp, vp, C.c_int64, C.POINTER(C.c_uint32), vp, C.c_uint32]
        L.ikdref_add_points_synced.argtypes = [vp, vp, vp, vp, C.c_int64, C.c_float, vp, C.c_int]
        L.ikdref_collect_sync.restype = None
        L.ikdref_collect_sync.argtypes = [vp, vp, C.c_int64, C.c_float, vp, C.c_int]
        L.ikdref_fetch_sync.restype = None
        L.ikdref_fetch_sync.argtypes = [vp, vp, vp, vp, vp]
        _ref = L
    return _ref


class RefTree:
    """The reference's KD_TREE<PointXYZINormal> (ikd_Tree.cpp compiled in place)."""

    def __init__(self, delete_param=0.5, balance_param=0.6, box_length=0.5):
        self.L = ref_lib()
        self.t = vp(self.L.ikdref_create(delete_param, balance_param, box_length))
        self.n_ids = 0

    def close(self):
        if self.t:
            self.L.ikdref_destroy(self.t)
            self.t = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def build(self, xyz, normal_y=None, ids=None):
        xyz = np.ascontiguousarray(xyz, np.float32)
        ny = None if normal_y is None else np.ascontiguousarray(normal_y, np.float32)
        ids = np.arange(xyz.shape[0], dtype=np.int32) if ids is None else np.ascontiguousarray(ids, np.int32)
        self.L.ikdref_build(self.t, ptr(xyz), ptr(ny), ptr(ids), xyz.shape[0])
        self.n_ids = max(self.n_ids, int(ids.max()) + 1 if len(ids) else 0)

    def add_points(self, xyz, normal_y=None, ids=None, downsample=True) -> int:
        xyz = np.ascontiguousarray(xyz, np.float32)
        ny = None if normal_y is None else np.ascontiguousarray(normal_y, np.float32)
        if ids is None:
            ids = np.arange(self.n_ids, self.n_ids + xyz.shape[0], dtype=np.int32)
        ids = np.ascontiguousarray(ids, np.int32)
        self.n_ids = max(self.n_ids, int(ids.max()) + 1 if len(ids) else 0)
        return self.L.ikdref_add_points(self.t, ptr(xyz), ptr(ny), ptr(ids), xyz.shape[0], 1 if downsample else 0)

    def add_points_synced(self, xyz, normal_y=None, ids=None, downsample_size=0.5, threads=1):
        """Add_Points(.., true) + the product's collect_voxel_sync on this tree (include/malio_mapsync.hpp).  Returns
        (tmp_counter, dict(boxes[nb,6], counts[nb], xyz[m,3], normal_y[m], ids[m], outside_own_box))."""
        xyz = np.ascontiguousarray(xyz, np.float32)
        ny = None if normal_y is None else np.ascontiguousarray(normal_y, np.float32)
        if ids is None:
            ids = np.arange(self.n_ids, self.n_ids + xyz.shape[0], dtype=np.int32)
        ids = np.ascontiguousarray(ids, np.int32)
        self.n_ids = max(self.n_ids, int(ids.max()) + 1 if len(ids) else 0)
        sz = np.zeros(3, np.int64)
        c = self.L.ikdref_add_points_synced(self.t, ptr(xyz), ptr(ny), ptr(ids), xyz.shape[0], C.c_float(downsample_size), ptr(sz), int(threads))
        nb, m = int(sz[0]), int(sz[1])
        boxes = np.zeros((nb, 6), np.float32); counts = np.zeros(nb, np.uint32)
        pxyz = np.zeros((m, 3), np.float32); pny = np.zeros(m, np.float32); pids = np.zeros(m, np.int32)
        self.L.ikdref_fetch_sync(ptr(boxes) if nb else None, ptr(counts) if nb else None, ptr(pxyz) if m else None,
                                 ptr(pny) if m else None, ptr(pids) if m else None)
        return c, dict(boxes=boxes, counts=counts, xyz=pxyz, normal_y=pny, ids=pids, outside_own_box=int(sz[2]))

    def collect_sync(self, xyz, downsample_size=0.5, out=None, threads=1):
        """malio::collect_voxel_sync alone (the caller already ran add_points(xyz, .., downsample=True)).  `out`: optional dict of
        pre-allocated arrays (boxes, counts, xyz, normal_y, ids) large enough to receive the record (e.g. pinned memory)."""
        xyz = np.ascontiguousarray(xyz, np.float32)
        sz = np.zeros(3, np.int64)
        self.L.ikdref_collect_sync(self.t, ptr(xyz), xyz.shape[0], C.c_float(downsample_size), ptr(sz), int(threads))
        nb, m = int(sz[0]), int(sz[1])
        if out is None:
            out = dict(boxes=np.zeros((max(nb, 1), 6), np.float32), counts=np.zeros(max(nb, 1), np.uint32), xyz=np.zeros((max(m, 1), 3), np.float32),
                       normal_y=np.zeros(max(m, 1), np.float32), ids=np.zeros(max(m, 1), np.int32))
        self.L.ikdref_fetch_sync(ptr(out["boxes"]), ptr(out["counts"]), ptr(out["xyz"]), ptr(out["normal_y"]), ptr(out["ids"]))
        return dict(boxes=out["boxes"][:nb], counts=out["counts"][:nb], xyz=out["xyz"][:m], normal_y=out["normal_y"][:m], ids=out["ids"][:m],
                    outside_own_box=int(sz[2]))

    def delete_boxes(self, boxes) -> int:
        b = np.ascontiguousarray(boxes, np.float32).reshape(-1, 6)
        return self.L.ikdref_delete_boxes(self.t, ptr(b), b.shape[0])

    def wait_rebuild(self):
        self.L.ikdref_wait_rebuild(self.t)

    def size(self):
        return self.L.ikdref_size(self.t)

    def validnum(self):
        return self.L.ikdref_validnum(self.t)

    def knn(self, q, k=5, nthreads=1):
        q = np.ascontiguousarray(q, np.float32)
        n = q.shape[0]
        ids = np.zeros((n, k), np.int32)
        d2 = np.zeros((n, k), np.float32)
        pts = np.zeros((n, k, 4), np.float32)
        found = np.zeros(n, np.int32)
        self.L.ikdref_knn(self.t, ptr(q), n, k, ptr(ids), ptr(d2), ptr(pts), ptr(found), nthreads)
        return ids, d2, pts, found

    def snapshot(self):
        """Flatten through include/malio_flatten.hpp.  Returns (nodes, node_cov, node_ids, max_depth, n_live)."""
        cap = max(self.size(), 1)
        nodes = np.zeros(cap, dtype=capi.MAP_NODE)
        cov = np.zeros(cap, np.float32)
        ids = np.zeros(cap, np.int32)
        depth = C.c_uint32(0)
        live = C.c_uint32(0)
        n = self.L.ikdref_snapshot(self.t, ptr(nodes), ptr(cov), ptr(ids), cap, C.byref(depth), C.byref(live))
        assert n >= 0
        return nodes[:n].copy(), cov[:n].copy(), ids[:n].copy(), int(depth.value), int(live.value)

    def snapshot_parallel(self, grain: int = 16384):
        """malio::flatten_ikdtree_parallel: same return as snapshot()."""
        cap = max(self.size(), 1)
        nodes = np.zeros(cap, dtype=capi.MAP_NODE)
        cov = np.zeros(cap, np.float32)
        ids = np.zeros(cap, np.int32)
        depth = C.c_uint32(0)
        live = C.c_uint32(0)
        n = self.L.ikdref_snapshot_parallel(self.t, ptr(nodes), ptr(cov), ptr(ids), cap, C.byref(depth), C.byref(live), grain)
        assert n >= 0
        return nodes[:n].copy(), cov[:n].copy(), ids[:n].copy(), int(depth.value), int(live.value)

    def snapshot_compact_parallel(self, grain: int = 16384):
        """malio::flatten_ikdtree_compact_parallel: same return as snapshot_compact()."""
        cap = max(self.size(), 1)
        pts = np.zeros(cap, dtype=capi.MAP_POINT)
        cov = np.zeros(cap, np.float32)
        depth = C.c_uint32(0)
        box = np.zeros(6, np.float32)
        n = self.L.ikdref_snapshot_compact_parallel(self.t, ptr(pts), ptr(cov), cap, C.byref(depth), ptr(box), grain)
        assert n >= 0
        return pts[:n].copy(), cov[:n].copy(), int(depth.value), box

    def snapshot_compact(self):
        """Flatten through malio::flatten_ikdtree_compact.  Returns (points, node_cov, max_depth, root_box)."""
        cap = max(self.size(), 1)
        pts = np.zeros(cap, dtype=capi.MAP_POINT)
        cov = np.zeros(cap, np.float32)
        depth = C.c_uint32(0)
        box = np.zeros(6, np.float32)
        n = self.L.ikdref_snapshot_compact(self.t, ptr(pts), ptr(cov), cap, C.byref(depth), ptr(box))
        assert n >= 0
        return pts[:n].copy(), cov[:n].copy(), int(depth.value), box

    def flatten_points(self):
        cap = max(self.size(), 1)
        xyz = np.zeros((cap, 3), np.float32)
        ny = np.zeros(cap, np.float32)
        ids = np.zeros(cap, np.int32)
        n = self.L.ikdref_flatten_points(self.t, ptr(xyz), ptr(ny), ptr(ids), cap)
        return xyz[:n], ny[:n], ids[:n]

    def knn1_fnptr(self):
        return C.cast(self.L.ikdref_knn1, vp)


def knn_snapshot(nodes, cov, q, k=5, nthreads=1):
    """Restated KD_TREE::Search over a snapshot.  Returns (idx, d2, found, total_visits)."""
    L = oracle_lib()
    q = np.ascontiguousarray(q, np.float32)
    n = q.shape[0]
    ids = np.zeros((n, k), np.int32)
    d2 = np.zeros((n, k), np.float32)
    found = np.zeros(n, np.int32)
    visits = C.c_int64(0)
    nodes = np.ascontiguousarray(nodes)
    cov = np.ascontiguousarray(cov, np.float32)
    L.orc_knn_snapshot_batch(ptr(nodes), ptr(cov), nodes.shape[0], ptr(q), n, k, ptr(ids), ptr(d2), ptr(found),
                             C.byref(visits), nthreads, None)
    return ids, d2, found, int(visits.value)


def build_static_snapshot(xyz, normal_y=0.001):
    """The static balanced snapshot of plugin.build_static_snapshot without mapping the product library."""
    from malio_b200 import plugin
    xyz = np.ascontiguousarray(xyz, np.float32)
    n = xyz.shape[0]
    nodes = np.zeros(n, dtype=capi.MAP_NODE)
    order = np.zeros(n, dtype=np.uint32)
    depth = C.c_uint32(0)
    oracle_lib().orc_build_static_snapshot(ptr(xyz), n, ptr(nodes), ptr(order), C.byref(depth))
    if np.isscalar(normal_y):
        cov = np.full(n, normal_y, dtype=np.float32)
    else:
        cov = np.ascontiguousarray(np.asarray(normal_y, dtype=np.float32)[order])
    return plugin.MapSnapshot(nodes, cov, order.astype(np.int64), int(depth.value))


class Oracle:
    """Restated h_share_model + update_iterated_dyn_share_modified on the CPU."""

    def __init__(self, params: capi.Params):
        self.L = oracle_lib()
        self.params = params
        self.n_lidar = params.n_lidar
        self.n_cols = 6 * (self.n_lidar + 1)
        self.n_dof = 17 + 6 * self.n_lidar
        self.c = vp(self.L.orc_create(C.byref(params)))
        self._keep = {}
        self.N = 0

    def close(self):
        if self.c:
            self.L.orc_destroy(self.c)
            self.c = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_map_snapshot(self, nodes, cov):
        nodes = np.ascontiguousarray(nodes)
        cov = np.ascontiguousarray(cov, np.float32)
        self._keep["map"] = (nodes, cov)
        self.L.orc_set_map_snapshot(self.c, ptr(nodes), ptr(cov), nodes.shape[0])

    def set_knn_ref(self, tree: RefTree):
        """k-NN through the real reference Nearest_Search (ids are the tree's point ids, not snapshot slots)."""
        self._keep["tree"] = tree
        self.L.orc_set_knn_hook(self.c, tree.knn1_fnptr(), tree.t)

    def set_scan(self, pts, table, table_off, tcomp):
        pts = np.ascontiguousarray(pts)
        table = np.ascontiguousarray(table)
        table_off = np.ascontiguousarray(table_off, np.uint32)
        tc = None if tcomp is None else np.ascontiguousarray(tcomp)
        self.N = pts.shape[0]
        self.L.orc_set_scan(self.c, ptr(pts), self.N, ptr(table), ptr(table_off), ptr(tc))

    def h_share_model(self, s, converge: bool, nthreads=1) -> bool:
        ps = s.pass_state() if isinstance(s, capi.State) else s
        return self.L.orc_h_share_model(self.c, C.byref(ps), 1 if converge else 0, nthreads) != 0

    def n_eff(self):
        return self.L.orc_n_eff(self.c)

    def set_minmax_override(self, enable, umin=0.0, umax=0.0, tmin=0.0, tmax=0.0):
        self.L.orc_set_minmax_override(self.c, 1 if enable else 0, umin, umax, tmin, tmax)

    def local_minmax(self):
        out = np.zeros(4)
        self.L.orc_get_local_minmax(self.c, ptr(out))
        return out

    def partials(self):
        G = np.zeros((self.n_cols, self.n_cols)); g = np.zeros(self.n_cols); S = np.zeros(6)
        self.L.orc_partials(self.c, ptr(G), ptr(g), ptr(S))
        return G, g, S

    def stats(self):
        st = capi.PassStats()
        self.L.orc_get_stats(self.c, C.byref(st))
        return st

    def dense(self):
        n = self.n_eff()
        hx = np.zeros((n, self.n_cols))
        h = np.zeros(n)
        R = np.zeros(n)
        self.L.orc_get_dense(self.c, ptr(hx), ptr(h), ptr(R))
        return hx, h, R

    def reduce(self):
        HTH = np.zeros((self.n_cols, self.n_cols))
        HTh = np.zeros(self.n_cols)
        self.L.orc_reduce(self.c, ptr(HTH), ptr(HTh))
        return HTH, HTh

    def aux(self):
        n = self.N
        ny = np.zeros(n, np.float32)
        ids = np.zeros((n, 5), np.int32)
        d2 = np.zeros((n, 5), np.float32)
        sel = np.zeros(n, np.uint8)
        w = np.zeros((n, 3), np.float32)
        cnt = np.zeros(n, np.int32)
        self.L.orc_get_aux(self.c, ptr(ny), ptr(ids), ptr(d2), ptr(sel), ptr(w), ptr(cnt))
        return dict(normal_y=ny, nn_idx=ids, nn_sqdist=d2, selected=sel, world=w, nn_cnt=cnt)

    def map_incremental(self, s, filter_size_map: float = 0.5, ekf_inited: bool = True):
        """map_incremental's per-point decision (laserMapping.cpp:398-446).  Returns (cls uint8[N], world float32[N,3])."""
        ps = s.pass_state() if isinstance(s, capi.State) else s
        cls = np.zeros(self.N, np.uint8)
        w = np.zeros((self.N, 3), np.float32)
        self.L.orc_map_incremental(self.c, C.byref(ps), C.c_double(filter_size_map), 1 if ekf_inited else 0, ptr(cls), ptr(w))
        return cls, w

    def visits(self):
        v, s = C.c_int64(0), C.c_int64(0)
        self.L.orc_get_visits(self.c, C.byref(v), C.byref(s))
        return int(v.value), int(s.value)

    def set_fast_reduce(self, enable: bool):
        """Timing arms only: esekfom.hpp:622-635 through the blocked / vectorised / threaded evaluation (orc_reduce_fast)."""
        self.L.orc_set_fast_reduce(self.c, 1 if enable else 0)

    def reset_times(self):
        self.L.orc_reset_times(self.c)

    def times(self):
        """(seconds in K = Nearest_Search, B = rest of h_share_model, A = rest of the update, passes) since reset_times()."""
        out = np.zeros(3)
        n = C.c_int(0)
        self.L.orc_get_times(self.c, ptr(out), C.byref(n))
        return float(out[0]), float(out[1]), float(out[2]), int(n.value)

    def update_iterated(self, x: capi.State, P: np.ndarray, max_iter: int, R=0.001, nthreads=1):
        n = self.n_dof
        dx_log = np.full((max_iter + 1, n), np.nan)
        flags = np.zeros(max_iter + 1, np.int32)
        rep = capi.UpdateReport()
        rc = self.L.orc_update_iterated(self.c, C.byref(x), ptr(P), max_iter, R, nthreads, ptr(dx_log), ptr(flags), C.byref(rep))
        return rc, dx_log, flags, rep


# ------------------------------------------------------------------ N2 / N3 restatements (oracle_undistort.cpp)
def bspline_get_pose(ctrl_t, ctrl_T, timestamp):
    L = oracle_lib()
    ct = np.ascontiguousarray(ctrl_t, np.float64)
    cT = np.ascontiguousarray(ctrl_T, np.float64).reshape(-1, 16)
    q, p = np.zeros(4), np.zeros(3)
    ok = L.orc_bspline_get_pose(ptr(ct), ptr(cT), ct.shape[0], float(timestamp), ptr(q), ptr(p))
    return bool(ok), q, p


def undistort(pts, beg_time, extrinsic, lt_imu_frame, ctrl_t, ctrl_T, imu_cov_t, cov_pointer, want_pose=False):
    """The per-point loop of UndistortPcl for one LiDAR (IMU_Processing.hpp:468-508), sequential, as the reference runs it."""
    L = oracle_lib()
    pts = np.ascontiguousarray(pts)
    n = pts.shape[0]
    raw = np.ascontiguousarray(pts.view(np.float32).reshape(n, 4))
    ct = np.ascontiguousarray(ctrl_t, np.float64)
    cT = np.ascontiguousarray(ctrl_T, np.float64).reshape(-1, 16)
    cv = np.ascontiguousarray(imu_cov_t, np.float64)
    eq, et = np.ascontiguousarray(extrinsic[0], np.float64), np.ascontiguousarray(extrinsic[1], np.float64)
    lq, lt = np.ascontiguousarray(lt_imu_frame[0], np.float64), np.ascontiguousarray(lt_imu_frame[1], np.float64)
    xyz = np.zeros((n, 3), np.float32); idx = np.zeros(n, np.int32); ok = np.zeros(n, np.uint8)
    pop = np.full(max(cv.shape[0], 1), -1, np.int32); npop = C.c_int32(0)
    pose = np.zeros((n, 7)) if want_pose else None
    L.orc_undistort(ptr(raw), n, float(beg_time), ptr(eq), ptr(et), ptr(lq), ptr(lt), ptr(ct), ptr(cT), ct.shape[0], ptr(cv),
                    cv.shape[0], int(cov_pointer), ptr(xyz), ptr(idx), ptr(ok), ptr(pop), C.byref(npop), ptr(pose))
    return dict(xyz=xyz, idx=idx, ok=ok, pop_point=pop[: min(npop.value, cv.shape[0])], n_pops=npop.value, pose=pose)


def voxel_grid(pts8, leaf):
    """pcl::VoxelGrid restated (all 8 float fields of PointXYZINormal averaged).  Returns (out[m,8], voxel_of[n])."""
    L = oracle_lib()
    p = np.ascontiguousarray(pts8, np.float32)
    n = p.shape[0]
    out = np.zeros((max(n, 1), 8), np.float32)
    vo = np.zeros(max(n, 1), np.int32)
    m = L.orc_voxel_grid(ptr(p), n, C.c_float(leaf), ptr(out), n, ptr(vo))
    return out[:m].copy(), vo[:n].copy()
