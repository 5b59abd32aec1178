#!/usr/bin/env python
"""bench.py — scans/sec & ms/IESKF-iter of the MA-LIO measurement hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # CUDA path (this repo), config C2 (the metric's config)
  python bench.py --impl reference --gpus N ...            # the reference's own CPU path on the host cores
  python bench.py --config C4|C5 ...                       # the other BASELINE configs (not the driver's bench line)
  torchrun ... bench.py --gpus N ...                       # N > 1: one rank per GPU

A *step* is one scan: the full iterated update (esekfom.hpp:495-721; max_iteration 3 => up to 4 measurement passes,
k-NN on the first pass and after a converged step) of the 3-LiDAR 100k-point merged scan against the 1M-point map
(BASELINE configs[1], "C2"; with --gpus N > 1 the same scan point-sharded over N ranks: configs[2]).  Synthetic, seeded
inputs (malio_b200/synth.py).  The map is a LIVE reference ikd-Tree (the real ikd_Tree.cpp, oracle/_ref: Build + the
scripted churn of SURVEY.md §8d — 2 % Add_Points with down-sampling, a no-down-sampling batch, one Delete_Point_Boxes —
so lazy flags and rebuilt subtrees exist); where oracle/_ref is not built the product's static builder stands in and the
line says so.  The tree is INPUT here, exactly what a MA-LIO checkout holds on its host; nothing under oracle/ computes
any part of the measured result.

`value`   scans/sec with every input already resident in HBM when the timed region starts (the per-scan state is
          re-armed on the device; sort, k-NN, plane fit, gate, reduction, D2H of the 3.5 KB system and the host 35x35
          algebra are all inside).
`e2e`     the same metric from HOST data through the public C-ABI, what a MA-LIO checkout would see per scan with the map kept
          on the device by deltas (SURVEY.md §8f N1, include/malio_mapsync.hpp): the host tree's own Add_Points of the scan's
          ~2.5k new points happens OUTSIDE the bracket (the reference does it too, and neither arm times map maintenance);
          INSIDE: read-back of the touched voxels from the tree (KD_TREE::Box_Search, `map_sync_host_ms`), upload of those
          deltas, device-side kill/append + cell-index rebuild, scan upload, iterated update, download of the per-point side
          outputs.  `e2e.full_snapshot` is the other integration path: flatten the live tree every scan
          (include/malio_flatten.hpp, OpenMP over the host threads; `flatten_ms`) + compact snapshot upload (20 B per node);
          `e2e.snapshot_only` is that step with the flatten left out (the round-1 definition), for comparison.
L2 is flushed (256 MiB write) between timed steps; each step is bracketed by CUDA events and the per-step times are
summed (max over ranks).  Only the cpu_baseline / --impl reference legs time anything under oracle/.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# stdout carries exactly one JSON line: NCCL's version banner (printed to stdout when the box exports NCCL_DEBUG) goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "ma-lio_b200"))

METRIC = "scans/sec & ms/IESKF-iter, 100k-pt scan vs 1M-pt map, 1/2/4/8 GPU"
UNIT = "scans/s"
WORKLOADS = {
    "C2": "C2: 3-LiDAR (Ouster+2xLivox) 100k-pt merged scan vs 1M-pt map (live ikd-Tree, churned), max_iteration=3",
    "C4": "C4: dense urban 300k-pt merged scan vs 5M-pt map, max_iteration=5",
    "C5": "C5: k-NN microbench, 1M queries vs 10M-pt tree, k=5",
}
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu captures (profiles/), C2 only
NCU_DRAM_BYTES = {"knn": 8.26e6, "pass": 10.1e6, "knn_c5": 535.6e6}   # profiles/r02_keys_pass_raw.csv (knn_keys_kernel, pass_kernel), r02_knn_direct_c5_raw.csv
SYNC_THREADS = 16          # host threads of the per-scan voxel read-back (include/malio_mapsync.hpp)
REF_CPU_BUDGET_S = 150.0   # bound of the CPU arms' total run time (both thread counts together)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=["C2", "C4", "C5"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sort", action="store_true")
    ap.add_argument("--static-map", action="store_true", help="static balanced snapshot instead of the live ikd-Tree")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step to DIR/<name>.npy (float32/float64), "
                         "so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the CUDA path's outputs (--impl ours)")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """One .npy per output, float32 or float64; integer outputs go to float64 (exact for the values they hold)."""
    conv = {k: (a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)) for k, a in arrays.items()}
    total = sum(a.nbytes for a in conv.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte budget")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in conv.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(a))


# ------------------------------------------------------------------ clocks sampler (recipe's nvidia-smi line)
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.rows = []
        self.proc = None
        self.t = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
            return
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if (t0 is None or t >= t0 - 0.1) and (t1 is None or t <= t1 + 0.1)] or \
               [r for (_, r) in self.rows]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for k, nm in enumerate(names):
                    if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class c_stdout_to_stderr:
    """The reference ikd-Tree printf()s thread start/stop notices on stdout; keep fd 1 clean for the JSON line."""

    def __enter__(self):
        self.libc = C.CDLL(None)
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *a):
        self.libc.fflush(None)
        os.dup2(self.saved, 1)
        os.close(self.saved)


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def load_case(config: str):
    from malio_b200 import synth
    return synth.case_C4() if config == "C4" else synth.case_C2()


# ------------------------------------------------------------------ the map as the host holds it
CHURN_NOTE = "Build + 2% Add_Points(downsample) + 0.5% Add_Points(no downsample) + one 12x12x6 m Delete_Point_Boxes"


def live_tree(case, seed=7):
    """The reference's KD_TREE (oracle/_ref = the real ikd_Tree.cpp) holding the case's map after the scripted churn of
    SURVEY.md §8d.  Returns a pyoracle.RefTree or None when oracle/_ref was not built."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle as po
    if not po.ref_available():
        return None
    tree = po.RefTree(box_length=0.5)
    tree.build(case.map_xyz, case.map_normal_y)
    rng = np.random.default_rng(seed)
    M = case.map_xyz.shape[0]
    k = max(M // 50, 10)
    add = case.map_xyz[rng.integers(0, M, k)] + rng.normal(0, 0.3, (k, 3)).astype(np.float32)
    tree.add_points(add, np.full(k, 0.001, np.float32), downsample=True)
    add2 = case.map_xyz[rng.integers(0, M, k // 4)] + rng.normal(0, 0.2, (k // 4, 3)).astype(np.float32)
    tree.add_points(add2, np.full(k // 4, 0.001, np.float32), downsample=False)
    c = case.map_xyz[rng.integers(0, M)]
    tree.delete_boxes([[c[0] - 6, c[1] - 6, c[2] - 3, c[0] + 6, c[1] + 6, c[2] + 3]])
    tree.wait_rebuild()
    return tree


# ------------------------------------------------------------------ reference / CPU arm
def cpu_reference_run(case, tree, steps: int, warmup: int, threads: int):
    """The reference's CPU path: real ikd_Tree.cpp (oracle/_ref) for the k-NN when it was compiled here, else the
    restated search; restated h_share_model + update_iterated_dyn_share_modified (oracle/), with esekfom.hpp:622-635
    evaluated the optimised way (orc_reduce_fast).  Returns a dict."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle as po
    orc = po.Oracle(case.params)
    orc.set_fast_reduce(True)
    if tree is not None:
        orc.set_knn_ref(tree)
        kind = "reference-knn+port"
    else:
        snap = po.build_static_snapshot(case.map_xyz, case.map_normal_y)
        orc.set_map_snapshot(snap.nodes, snap.node_cov)
        kind = "port"
    times, passes = [], 0
    for i in range(warmup + steps):
        orc.set_scan(case.pts, case.table, case.table_off, case.temporal_comp)
        x, P = case.x_prop.copy(), case.P_prop.copy()
        if i == warmup:
            orc.reset_times()
        t0 = time.perf_counter()
        rc, _, _, rep = orc.update_iterated(x, P, case.max_iter, nthreads=threads)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
            passes += rep.passes
    tK, tB, tA, npass = orc.times()
    tot = float(np.sum(times))
    orc.close()
    npass = max(npass, 1)
    return {"scans_per_s": steps / tot, "ms_per_pass": 1e3 * tot / max(passes, 1), "kind": kind, "threads": threads,
            "passes_per_scan": passes / max(steps, 1), "steps": steps, "warmup": warmup,
            "split_ms_per_pass": {"K_nearest_search": 1e3 * tK / npass, "B_h_share_model_rest": 1e3 * tB / npass,
                                  "A_ieskf_rest": 1e3 * tA / npass}}


def cpu_arms(case, tree, steps, warmup):
    """Both thread counts the survey asks for: 3 (what the reference ships, CMakeLists.txt:23-25) and all host threads.
    Steps are honoured up to a wall-clock budget (a full C2 scan is 0.2-0.7 s of CPU)."""
    th_all = host_threads()
    runs = []
    # 3 = the reference's MP_PROC_NUM; the serial stretches of h_share_model / the update (S2-S6, the c x c algebra) get slower
    # next to a large idle OpenMP team, so the best count lies between 3 and all: measured, not assumed
    counts = sorted({t for t in (3, 8, 16, 32, th_all) if t <= th_all})
    budget = REF_CPU_BUDGET_S / len(counts)
    for th in counts:
        probe = cpu_reference_run(case, tree, 1, 1, th)       # also the first warm-up
        est = 1.0 / probe["scans_per_s"]
        k = int(max(1, min(steps, budget / est - warmup)))
        w = int(max(0, min(warmup - 1, budget / est - k)))
        runs.append(cpu_reference_run(case, tree, k, w, th))
        runs[-1]["warmup"] = w + 2
    best = max(runs, key=lambda r: r["scans_per_s"])
    return best, runs


def cpu_baseline_obj(best, runs, what):
    return {"value": best["scans_per_s"], "unit": UNIT, "cores": best["threads"], "kind": best["kind"],
            "ms_per_ieskf_iter": best["ms_per_pass"], "split_ms_per_pass": best["split_ms_per_pass"],
            "by_threads": {str(r["threads"]): {"value": r["scans_per_s"], "ms_per_ieskf_iter": r["ms_per_pass"],
                                               "split_ms_per_pass": r["split_ms_per_pass"], "steps": r["steps"]} for r in runs},
            "sample": what,
            "notes": "K = KD_TREE::Nearest_Search of the real ikd_Tree.cpp (g++ -O3); B/A = line-by-line port (no Eigen in the "
                     "image) with the O(N) algebra of esekfom.hpp:622-635 blocked, AVX-dispatched and threaded (more generous than "
                     "the reference's baseline-x86-64 Eigen build); value = the fastest of the thread counts in by_threads (3 = the reference's default ... all host threads)"}


def run_reference(args, rank):
    if rank != 0:
        return
    if args.config == "C5":
        return run_reference_c5(args)
    case = load_case(args.config)
    with c_stdout_to_stderr():
        tree = None if args.static_map else live_tree(case)
        best, runs = cpu_arms(case, tree, args.steps, args.warmup)
        if tree is not None:
            tree.close()
    sps = best["scans_per_s"]
    line = {
        "impl": "reference", "metric": METRIC, "value": sps, "unit": UNIT, "n_gpus": args.gpus, "steps": best["steps"],
        "warmup": best["warmup"], "ms_per_step": 1e3 / sps, "ms_per_ieskf_iter": best["ms_per_pass"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64/f32", "data": "synthetic (seeded, malio_b200/synth.py)",
        "config": {"workload": WORKLOADS[args.config], "passes_per_scan": best["passes_per_scan"], "host_threads": host_threads(),
                   "steps_requested": args.steps, "warmup_requested": args.warmup,
                   "map": ("live reference ikd-Tree: " + CHURN_NOTE) if tree is not None else "static snapshot (restated search)"},
        "cpu_baseline": cpu_baseline_obj(best, runs, f"{best['steps']} full {args.config} scans per thread count (steps bounded by a "
                                                         f"{REF_CPU_BUDGET_S:.0f} s CPU budget)"),
        "e2e": {"value": sps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "clocks": None, "roofline": None,      # CPU arm: no GPU clocks, no kernel roofline
    }
    print(json.dumps(line))


# ------------------------------------------------------------------ C5: k-NN microbench
def c5_cpu(xyz, q, sample=200_000):
    """Reference KD_TREE::Nearest_Search (real ikd_Tree.cpp) on a bounded sample of the queries, 3 threads and all."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle as po
    if not po.ref_available():
        return None
    tree = po.RefTree(box_length=0.5)
    tree.build(xyz)
    out = {}
    th_all = host_threads()
    for th in ([3, th_all] if th_all > 3 else [th_all]):
        tree.knn(q[:20000], nthreads=th)
        t0 = time.perf_counter()
        tree.knn(q[:sample], nthreads=th)
        out[str(th)] = sample / (time.perf_counter() - t0)
    tree.close()
    best = max(out, key=lambda k: out[k])
    return {"value": out[best], "unit": "queries/s", "cores": int(best), "kind": "reference", "by_threads": out,
            "sample": f"{sample} of the 1M queries against the full 10M-point reference ikd-Tree (Build), after a 20k warm-up"}


def run_reference_c5(args):
    from malio_b200 import synth
    xyz, q = synth.knn_microbench()
    with c_stdout_to_stderr():
        cpu = c5_cpu(xyz, q)
    line = {"impl": "reference", "metric": "k-NN queries/s, 1M queries vs 10M-pt tree, k=5", "value": cpu["value"] if cpu else None,
            "unit": "queries/s", "n_gpus": args.gpus, "steps": 1, "warmup": 1, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded)", "config": {"workload": WORKLOADS["C5"]},
            "cpu_baseline": cpu, "e2e": {"value": cpu["value"] if cpu else None, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def run_ours_c5(args, rank, world):
    import torch
    import torch.distributed as dist
    from malio_b200 import plugin, synth
    from malio_b200 import dist as mdist
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
    xyz, q_all = synth.knn_microbench()
    lo, hi = mdist.shard_bounds(q_all.shape[0], rank, world)      # queries shard by block, tree replicated: no collective
    q = np.ascontiguousarray(q_all[lo:hi])
    snap = plugin.build_static_snapshot(xyz)
    m = plugin.MeasurementModel(1, device=local_rank, sort_queries=not args.no_sort)
    m.upload_map(snap)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        m.Nearest_Search(q)
    steps = args.steps
    c0 = m.counters()
    dev_ms, e2e_ms = [], []
    tw0 = time.time()
    for _ in range(steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        idx, d2, ms = m.Nearest_Search(q)      # host queries -> host lists (H2D 12 B, D2H 40 B per query inside)
        e1.record(); torch.cuda.synchronize()
        dev_ms.append(ms); e2e_ms.append(e0.elapsed_time(e1))
    tw1 = time.time()
    if args.dump_outputs and rank == 0:
        # a fixed sample of rank 0's queries keeps the dump small (1M x 5 lists would be 60 MB)
        pick = np.sort(np.random.default_rng(0).choice(idx.shape[0], min(idx.shape[0], 100_000), replace=False))
        dump_outputs(args.dump_outputs, {"knn_query_index": pick + lo, "knn_idx": idx[pick], "knn_sqdist": d2[pick]})
    c1 = m.counters()
    clocks = sampler.stop(tw0, tw1) if rank == 0 else None
    t = torch.tensor([float(np.sum(dev_ms)), float(np.sum(e2e_ms))], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank != 0:
        m.close()
        if world > 1:
            dist.destroy_process_group()
        return
    Q = q_all.shape[0]
    dev_s, e2e_s = t[0].item() * 1e-3 / steps, t[1].item() * 1e-3 / steps
    peak, peak_src = 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]); peak_src = "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        pass
    cand = float(c1.knn_candidates - c0.knn_candidates) / float((c1.knn_queries - c0.knn_queries) or 1)
    bytes_per_launch = (hi - lo) * (12 + 9 * 8 + cand * 16 + 40)
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        with c_stdout_to_stderr():
            cpu = c5_cpu(xyz, q_all)
    line = {"metric": "k-NN queries/s, 1M queries vs 10M-pt tree, k=5", "value": Q / dev_s, "unit": "queries/s", "n_gpus": world,
            "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_s * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded, malio_b200/synth.py knn_microbench)",
            "config": {"workload": WORKLOADS["C5"], "l2": "flushed between timed steps (256 MiB write); the 160 MB cell-sorted point array exceeds L2",
                       "queries_per_rank": hi - lo, "parallelism": f"query-block x{world}, replicated tree, no collective"},
            "clocks": clocks,
            "e2e": {"value": Q / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": (hi - lo) * 12, "d2h_bytes_per_step": (hi - lo) * 40,
                    "ms_per_step": e2e_s * 1e3, "what": "malio_knn: host queries -> sort -> search -> caller-order lists on the host"},
            "gpu_launches": int(c1.kernel_launches - c0.kernel_launches),
            "roofline": {"bound": "hbm", "kernel": "knn_direct_kernel (+ knn_list_kernel)", "achieved": bytes_per_launch / dev_s / 1e9,
                         "peak": peak, "unit": "GB/s", "frac": bytes_per_launch / dev_s / 1e9 / peak, "traffic": NCU_DRAM_BYTES["knn_c5"] if world == 1 else None,
                         "algorithmic_bytes_per_launch": bytes_per_launch, "us_per_launch": dev_s * 1e6, "candidates_per_query": cand,
                         "fallback_queries_per_search": float(c1.knn_fallback_queries - c0.knn_fallback_queries) / steps,
                         "ring2_queries_per_search": float(c1.knn_ring2_queries - c0.knn_ring2_queries) / steps, "peak_source": peak_src,
                         "note": "bytes = Q*(12 + 72 + C*16 + 40); device time = CUDA events around the search kernels (malio_knn ms_device)"},
            "cpu_baseline": cpu}
    print(json.dumps(line))
    m.close()
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------ CUDA arm
def run_ours(args, rank, world):
    import torch
    import torch.distributed as dist
    from malio_b200 import capi, plugin, synth
    from malio_b200 import dist as mdist

    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
    case = load_case(args.config)
    N_total = case.pts.shape[0]
    # contiguous block of the merged scan per rank (SURVEY.md §8e); map, tables and state are replicated
    lo, hi = mdist.shard_bounds(N_total, rank, world)

    def pinned(a):
        t = torch.empty(max(a.nbytes, 1), dtype=torch.uint8).pin_memory()
        v = t.numpy()[: a.nbytes].view(a.dtype).reshape(a.shape)
        v[...] = a
        return t, v

    keep = []
    tree = None
    with c_stdout_to_stderr():
        if not args.static_map:
            tree = live_tree(case)
    if tree is not None:
        nodes, cov, ids, depth, live = tree.snapshot()
        snap = plugin.MapSnapshot(nodes, cov, ids, depth)
        map_desc = "live reference ikd-Tree: " + CHURN_NOTE
    else:
        snap = plugin.build_static_snapshot(case.map_xyz, case.map_normal_y)
        map_desc = "static balanced snapshot (oracle/_ref not built)"
    M_nodes = snap.n_nodes
    cap_nodes = M_nodes + M_nodes // 8 + 1024
    t_pts, h_pts = pinned(np.ascontiguousarray(case.pts[lo:hi])); keep.append(t_pts)
    t_mp, h_mpts = pinned(np.zeros(cap_nodes, dtype=capi.MAP_POINT)); keep.append(t_mp)
    t_cv, h_cov = pinned(np.zeros(cap_nodes, dtype=np.float32)); keep.append(t_cv)
    h_mpts[:M_nodes] = plugin.compact_points(snap.nodes)
    h_cov[:M_nodes] = snap.node_cov

    model = plugin.MeasurementModel(case.n_lidar, device=local_rank, sort_queries=not args.no_sort, params=case.params)
    if world > 1:
        mdist.init_comm(model, rank, world, device=torch.device("cuda", local_rank))
    model.upload_map(snap)
    model.upload_scan(h_pts, case.table, case.table_off, case.temporal_comp)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step_resident():
        model.rearm_scan()
        x, P = case.x_prop.copy(), case.P_prop.copy()
        return model.update_iterated_dyn_share_modified(x, P, case.max_iter), x, P

    # root box of the map = the ikd-Tree root's node_range_* (node 0's point + its two children's boxes)
    n0 = snap.nodes[0]
    blo = np.array(n0["xyz"], np.float32); bhi = blo.copy()
    for b, bit in ((n0["lbox"], capi.LINK_HAS_LEFT), (n0["rbox"], capi.LINK_HAS_RIGHT)):
        if n0["link"] & bit:
            blo = np.minimum(blo, b[0::2]); bhi = np.maximum(bhi, b[1::2])
    root_box = np.stack([blo, bhi], axis=1).reshape(6).astype(np.float32)
    t_ny, h_ny = pinned(np.zeros(h_pts.shape[0], np.float32)); keep.append(t_ny)
    t_sel, h_sel = pinned(np.zeros(h_pts.shape[0], np.uint8)); keep.append(t_sel)
    aux_out = {"normal_y": h_ny, "selected": h_sel}
    flat = {"s": 0.0, "n": 0}
    if tree is not None:
        import pyoracle as po
        reflib = po.ref_lib()
        f_depth = C.c_uint32(0)
        f_box = np.zeros(6, np.float32)

    stages = {}

    def lap(name, t0):
        stages[name] = stages.get(name, 0.0) + (time.perf_counter() - t0)
        return time.perf_counter()

    def step_e2e_snapshot_only():
        t0 = time.perf_counter()
        sp = plugin.MapSnapshot(None, h_cov[:M_nodes], None, snap.max_depth)
        model.upload_map_compact(sp, points=h_mpts[:M_nodes], root_box=root_box)
        t0 = lap("upload_map_compact", t0)
        model.upload_scan(h_pts, case.table, case.table_off, case.temporal_comp)
        t0 = lap("upload_scan", t0)
        x, P = case.x_prop.copy(), case.P_prop.copy()
        rep = model.update_iterated_dyn_share_modified(x, P, case.max_iter)
        t0 = lap("update", t0)
        model.aux(out=aux_out)
        lap("aux", t0)
        return rep, x

    def step_e2e():
        if tree is None:
            return step_e2e_snapshot_only()
        # what a MA-LIO checkout does per scan: flatten the live tree (product header malio_flatten.hpp instantiated on
        # the real KD_TREE_NODE; OpenMP over the host threads) straight into pinned memory, then upload
        t0 = time.perf_counter()
        n = reflib.ikdref_snapshot_compact_parallel(tree.t, capi.ptr(h_mpts), capi.ptr(h_cov), cap_nodes, C.byref(f_depth),
                                                    capi.ptr(f_box), 16384)
        flat["s"] += time.perf_counter() - t0; flat["n"] += 1
        sp = plugin.MapSnapshot(None, h_cov[:n], None, int(f_depth.value))
        model.upload_map_compact(sp, points=h_mpts[:n], root_box=f_box)
        model.upload_scan(h_pts, case.table, case.table_off, case.temporal_comp)
        x, P = case.x_prop.copy(), case.P_prop.copy()
        rep = model.update_iterated_dyn_share_modified(x, P, case.max_iter)
        model.aux(out=aux_out)
        return rep, x

    # ---- device-resident map kept in step by deltas: a second handle in device-map mode, same scan
    inc = {"model": None}
    if tree is not None:
        fx, fny, fid = tree.flatten_points()
        mi = plugin.MeasurementModel(case.n_lidar, device=local_rank, sort_queries=not args.no_sort, params=case.params)
        if world > 1:
            mdist.init_comm(mi, rank, world, device=torch.device("cuda", local_rank))
        mi.map_build(fx, fny, fid)
        mi.upload_scan(h_pts, case.table, case.table_off, case.temporal_comp)
        mi.set_timing(False)
        inc["model"] = mi
        inc["rng"] = np.random.default_rng(99)
        inc["next_id"] = int(fid.max()) + 1
        K_DS, K_PLAIN = 2000, 500
        # one pinned record: header {n_boxes, n_points} | boxes | counts | xyz | normal_y | ids.  N > 1: rank 0 alone reads the deltas
        # back from ITS host tree (one tree, one read-back, as an integration would) and the record is broadcast over NVLink
        CAP_M = K_DS * 16
        off_b = 16; off_c = off_b + K_DS * 24; off_x = off_c + K_DS * 4; off_n = off_x + CAP_M * 12; off_i = off_n + CAP_M * 4
        pack_bytes = off_i + CAP_M * 4
        t_pack = torch.zeros(pack_bytes, dtype=torch.uint8).pin_memory(); keep.append(t_pack)
        h_pack = t_pack.numpy()
        inc["hdr"] = h_pack[0:8].view(np.int32)
        inc["boxes"] = h_pack[off_b:off_c].view(np.float32).reshape(K_DS, 6)
        inc["counts"] = h_pack[off_c:off_x].view(np.uint32)
        inc["xyz"] = h_pack[off_x:off_n].view(np.float32).reshape(CAP_M, 3)
        inc["ny"] = h_pack[off_n:off_i].view(np.float32)
        inc["ids"] = h_pack[off_i:pack_bytes].view(np.int32)
        d_pack = torch.zeros(pack_bytes, dtype=torch.uint8, device="cuda") if world > 1 else None
        inc["sync_s"] = 0.0; inc["sync_pts"] = 0; inc["n"] = 0
        inc["ny_plain"] = np.full(K_PLAIN, 0.001, np.float32)

        def prepare_scan_adds():
            # the reference's own map maintenance for one scan (laserMapping.cpp:443-444), NOT timed in either arm
            rng_i = inc["rng"]
            Mx = case.map_xyz.shape[0]
            a = (case.map_xyz[rng_i.integers(0, Mx, K_DS)] + rng_i.normal(0, 0.3, (K_DS, 3))).astype(np.float32)
            b = (case.map_xyz[rng_i.integers(0, Mx, K_PLAIN)] + rng_i.normal(0, 0.2, (K_PLAIN, 3))).astype(np.float32)
            ia = np.arange(inc["next_id"], inc["next_id"] + K_DS, dtype=np.int32); inc["next_id"] += K_DS
            ib = np.arange(inc["next_id"], inc["next_id"] + K_PLAIN, dtype=np.int32); inc["next_id"] += K_PLAIN
            with c_stdout_to_stderr():
                tree.add_points(a, np.full(K_DS, 0.001, np.float32), ia, downsample=True)
                tree.add_points(b, np.full(K_PLAIN, 0.001, np.float32), ib, downsample=False)
            inc["pending"] = (a, b, ib)

        from concurrent.futures import ThreadPoolExecutor
        inc["pool"] = ThreadPoolExecutor(max_workers=1)

        def step_e2e_incremental():
            a, b, ib = inc["pending"]
            t0 = time.perf_counter()
            # the scan upload does not depend on the map deltas: a helper thread issues it (H2D + per-scan reset on the handle) while
            # this thread reads the touched voxels back from the host tree (no handle involved); joined before the next handle call
            up = inc["pool"].submit(mi.upload_scan, h_pts, case.table, case.table_off, case.temporal_comp)
            if world == 1 or rank == 0:
                sync = tree.collect_sync(a, 0.5, out=dict(boxes=inc["boxes"], counts=inc["counts"], xyz=inc["xyz"], normal_y=inc["ny"], ids=inc["ids"]),
                                         threads=SYNC_THREADS)
            if world > 1:
                if rank == 0:
                    inc["hdr"][0] = sync["boxes"].shape[0]; inc["hdr"][1] = sync["xyz"].shape[0]
                    d_pack.copy_(t_pack, non_blocking=True)
                dist.broadcast(d_pack, 0)
                if rank != 0:
                    t_pack.copy_(d_pack, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                nb_, m_ = int(inc["hdr"][0]), int(inc["hdr"][1])
                sync = dict(boxes=inc["boxes"][:nb_], counts=inc["counts"][:nb_], xyz=inc["xyz"][:m_], normal_y=inc["ny"][:m_], ids=inc["ids"][:m_])
            inc["sync_s"] += time.perf_counter() - t0; inc["sync_pts"] += sync["xyz"].shape[0]; inc["n"] += 1
            t0 = lap("i_collect_sync_host", t0)
            up.result()
            t0 = lap("i_upload_scan_join", t0)
            mi.map_sync_voxels(sync, want_count=False)
            t0 = lap("i_map_sync_voxels", t0)
            mi.map_add_points(b, inc["ny_plain"], ib)
            t0 = lap("i_map_add_points", t0)
            x, P = case.x_prop.copy(), case.P_prop.copy()
            rep = mi.update_iterated_dyn_share_modified(x, P, case.max_iter)
            t0 = lap("i_update_incl_map_commit", t0)
            mi.aux(out=aux_out)
            lap("i_aux", t0)
            return rep, x

    def timed(fn, steps, warmup, before=None, ctr=None):
        ctr = ctr or model
        for _ in range(warmup):
            if before:
                before()
            fn()
            flush.fill_(1)
        barrier()
        flat["s"], flat["n"] = 0.0, 0
        ms, reps = [], []
        c0 = ctr.counters()
        t_wall0 = time.time()
        for _ in range(steps):
            if before:
                before()
            flush.fill_(1)          # L2 flush, outside the timed bracket
            torch.cuda.synchronize()
            if world > 1:           # start the ranks together: inside a pass they wait for each other (exchange), so any
                dist.barrier()      # start skew would be billed to the earlier rank's timed bracket
                torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
            reps.append(out[0])
        t_wall1 = time.time()
        barrier()
        c1 = ctr.counters()
        total = torch.tensor([float(np.sum(ms))], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(total, op=dist.ReduceOp.MAX)
        return float(total.item()), reps, c0, c1, out, (t_wall0, t_wall1)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    model.set_timing(False)       # no per-pass event records inside the measured loops
    tot_ms, reps, c0, c1, out, (tw0, tw1) = timed(step_resident, args.steps, args.warmup)
    x_res = out[1]
    dumped = None
    if args.dump_outputs and rank == 0:
        # what a caller of the timed step receives: the updated state and covariance, the report's deterministic fields and the
        # per-point side outputs of the last pass (rank 0's block of the scan when sharded); written after all timing
        rep_last, x_last, P_last = out
        aux = model.aux()
        dumped = {"state": synth.state_to_vec(x_last, case.n_lidar), "P": P_last, "dx_last": np.array(rep_last.dx_last[: case.n_dof]),
                  "report": np.array([rep_last.passes, rep_last.searches, rep_last.converged_count, rep_last.last_status,
                                      rep_last.n_eff_last], np.float64),
                  "normal_y": aux["normal_y"], "nn_idx": aux["nn_idx"], "nn_sqdist": aux["nn_sqdist"], "selected": aux["selected"],
                  "world": aux["world"]}
    passes = sum(r.passes for r in reps)
    searches = sum(r.searches for r in reps)
    launches = int(c1.kernel_launches - c0.kernel_launches)
    host_ms = float(np.sum([r.ms_host_solve for r in reps]))
    value = args.steps / (tot_ms * 1e-3)

    e_steps = max(3, min(args.steps, 10))
    e_ms, e_reps, ec0, ec1, e_out, _ = timed(step_e2e, e_steps, min(args.warmup, 3))
    flatten_ms = 1e3 * flat["s"] / max(flat["n"], 1) if tree is not None else None
    h2d = int(ec1.h2d_bytes - ec0.h2d_bytes) // e_steps
    d2h = int(ec1.d2h_bytes - ec0.d2h_bytes) // e_steps
    i_obj = None
    if inc["model"] is not None:
        inc["sync_s"], inc["sync_pts"], inc["n"] = 0.0, 0, 0
        mi = inc["model"]
        for _ in range(max(1, min(args.warmup, 3))):   # warm-up, untimed
            prepare_scan_adds(); step_e2e_incremental(); flush.fill_(1)
        inc["sync_s"], inc["sync_pts"], inc["n"] = 0.0, 0, 0
        stages.clear()
        i_ms, i_reps, ic0, ic1, i_out, _ = timed(step_e2e_incremental, e_steps, 0, before=prepare_scan_adds, ctr=mi)
        i_stage_ms = {k[2:]: 1e3 * v / e_steps for k, v in stages.items() if k.startswith("i_")}
        i_live, i_slots = mi.map_info()
        i_obj = {"value": e_steps / (i_ms * 1e-3), "unit": UNIT, "ms_per_step": i_ms / e_steps, "steps": e_steps,
                 "h2d_bytes_per_step": int(ic1.h2d_bytes - ic0.h2d_bytes) // e_steps, "d2h_bytes_per_step": int(ic1.d2h_bytes - ic0.d2h_bytes) // e_steps,
                 "map_sync_host_ms": 1e3 * inc["sync_s"] / max(inc["n"], 1), "map_sync_host_threads": SYNC_THREADS,
                 "map_sync_mode": "local read-back" if world == 1 else "rank 0 reads back from its host tree, one NCCL broadcast of the record (time included)",
                 "synced_points_per_step": inc["sync_pts"] / max(inc["n"], 1),
                 "host_wall_ms_per_stage": i_stage_ms,
                 "new_points_per_step": 2500, "map_live_points": i_live, "map_slots": i_slots,
                 "knn_tie_queries": int(ic1.knn_tie_queries - ic0.knn_tie_queries), "passes_per_scan": sum(r.passes for r in i_reps) / e_steps,
                 "what": "map kept on the device by deltas: Box_Search read-back of the voxels the scan's 2000 down-sampled adds touch (host, in the "
                         "bracket; the scan upload runs beside it on a helper thread) + upload of those points and boxes + 500 plain appends + device "
                         "kill/append + cell-index rebuild + IESKF update + download of normal_y/selected; the tree's own Add_Points runs outside "
                         "the bracket (untimed in both arms)"}
        inc["pool"].shutdown()
        mi.close()
    step_e2e_snapshot_only(); stages.clear()
    s_ms, _, _, _, _, _ = timed(step_e2e_snapshot_only, e_steps, 0)
    stage_ms = {k: 1e3 * v / e_steps for k, v in stages.items()}

    # separate short loop with per-kernel CUDA events on (same steps, L2 flushed): kernel times for the rooflines
    model.set_timing(True)
    r_steps = max(3, min(args.steps, 10))
    _, r_reps, rc0, rc1, _, (_, tw_end) = timed(step_resident, r_steps, 1)
    clocks = sampler.stop(tw0, tw_end) if rank == 0 else None
    knn_launches = int(rc1.knn_launches - rc0.knn_launches)
    knn_ms = float(rc1.knn_ms - rc0.knn_ms)
    pass_launches = int(rc1.pass_launches - rc0.pass_launches)
    pass_fit = int(rc1.pass_fit_launches - rc0.pass_fit_launches)
    pass_ms = float(rc1.pass_ms - rc0.pass_ms)
    dev_ms = float(np.sum([r.ms_device_total for r in r_reps])) * args.steps / r_steps
    e_value = e_steps / (e_ms * 1e-3)

    # ---- N > 1: the sharded result must equal a single-GPU run of the whole scan (outside every timed region)
    parity_n = None
    if world > 1:
        vec = synth.state_to_vec(x_res, case.n_lidar)
        tv = torch.from_numpy(vec.copy()).cuda()
        tv0 = tv.clone()
        dist.broadcast(tv0, 0)
        same = torch.tensor([1.0 if torch.equal(tv, tv0) else 0.0], device="cuda")
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        if rank == 0:
            single = plugin.MeasurementModel(case.n_lidar, device=local_rank, sort_queries=not args.no_sort, params=case.params)
            single.upload_map(snap)
            single.upload_scan(np.ascontiguousarray(case.pts), case.table, case.table_off, case.temporal_comp)
            x1, P1 = case.x_prop.copy(), case.P_prop.copy()
            rep1 = single.update_iterated_dyn_share_modified(x1, P1, case.max_iter)
            d = float(np.abs(synth.state_to_vec(x1, case.n_lidar) - vec).max())
            ok = bool(same.item() == 1.0) and d < 1e-9 and rep1.passes == reps[-1].passes and rep1.n_eff_last == reps[-1].n_eff_last
            parity_n = {"status": "ok" if ok else "FAILED", "ranks_bit_identical": bool(same.item() == 1.0), "state_max_abs_diff_vs_1gpu": d,
                        "passes": [int(rep1.passes), int(reps[-1].passes)], "n_eff_last": [int(rep1.n_eff_last), int(reps[-1].n_eff_last)]}
            single.close()

    if rank != 0:
        model.close()
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]); peak_src = "MEASURED_PEAKS.json hbm_gbs (burst copy)"
    except Exception:
        pass
    q_per_launch = (hi - lo)
    cand = int(rc1.knn_candidates - rc0.knn_candidates)
    roofs = []
    if knn_launches:
        cbar = cand / float(knn_launches * q_per_launch)
        bytes_per_launch = q_per_launch * (16 + 9 * 8 + cbar * 16 + 40 + 16 + 1)
        t_launch = knn_ms * 1e-3 / knn_launches
        achieved = bytes_per_launch / t_launch / 1e9
        n_q = case.pts.shape[0] // max(world, 1)
        knn_name = ("knn_keys_kernel, 4 lanes per query" if n_q <= 256 * 148 else
                    "knn_keys_kernel, 2 lanes per query" if n_q <= 1280 * 148 else "knn_direct_kernel, thread per query")
        roofs.append({"bound": "hbm", "kernel": f"k-NN search: {knn_name} (+ knn_list_kernel)",
                      "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                      "traffic": NCU_DRAM_BYTES["knn"] if (world == 1 and args.config == "C2") else None,
                      "algorithmic_bytes_per_launch": bytes_per_launch, "us_per_launch": t_launch * 1e6,
                      "us_per_step": knn_ms * 1e3 / r_steps, "launches_timed": knn_launches, "candidates_per_query": cbar,
                      "fallback_queries_per_search": float(rc1.knn_fallback_queries - rc0.knn_fallback_queries) / knn_launches,
                      "ring2_queries_per_search": float(rc1.knn_ring2_queries - rc0.knn_ring2_queries) / knn_launches,
                      "peak_source": peak_src,
                      "note": "bytes = Q*(16 + 72 + C*16 + 57), C = candidates scanned per query (device counter); the cell-sorted point "
                              "array and the scan are L2-resident at C2, so DRAM traffic is far below the algorithmic bytes; ncu: issue active 44 %, "
                              "17 of 32 lanes, 0.59 waves (782 blocks): bound by divergence and latency at a grid that does not fill the machine"})
    if pass_launches:
        # per point and pass: in 16 (scan point) + 16 (plane) + 8 (plane cov) + 16 (traces) + 1 (selected);
        # out 16 (world) + 4 (residual) + 8 (trace) + 4 (normal_y) + 96 (Jacobian row kept for the degenerate branch) + 1 + 1;
        # a search pass adds the plane fit: 20 (neighbour ids) + 5 x 20 (neighbour points + weights) + 24 (plane, plane cov)
        fit_frac = pass_fit / float(pass_launches)
        bytes_pt = 57 + 130 + fit_frac * 144
        bytes_per_launch = q_per_launch * bytes_pt + 434 * 8 * 2
        t_launch = pass_ms * 1e-3 / pass_launches
        achieved = bytes_per_launch / t_launch / 1e9
        roofs.append({"bound": "hbm", "kernel": "pass_kernel (plane fit on search passes + gate + Jacobian rows + H^T R^-1 [H|h] + fold)",
                      "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": NCU_DRAM_BYTES["pass"],
                      "algorithmic_bytes_per_launch": bytes_per_launch, "us_per_launch": t_launch * 1e6,
                      "us_per_step": pass_ms * 1e3 / r_steps, "launches_timed": pass_launches, "search_pass_fraction": fit_frac,
                      "peak_source": peak_src,
                      "note": "bytes/point = 57 in + 130 out (+144 on search passes); everything is L2-resident at C2: the kernel is "
                              "bound by FP64 dependent-chain latency and two grid barriers, not by HBM (see profiles/)"})
    roofs.sort(key=lambda r: -r["us_per_step"])
    roof = roofs[0] if roofs else None
    roof2 = roofs[1] if len(roofs) > 1 else None

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        try:
            with c_stdout_to_stderr():
                best, runs = cpu_arms(case, tree, 3, 1)
            cpu = cpu_baseline_obj(best, runs, f"3 full {args.config} scans after warm-up per thread count, same live ikd-Tree as the GPU arm")
        except Exception as e:   # the checker is optional for the product line
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": repr(e)}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tot_ms / args.steps, "ms_per_ieskf_iter": tot_ms / max(passes, 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64 (Jacobian, reduction, filter) / f32 (k-NN, plane fit)",
        "data": "synthetic (seeded, malio_b200/synth.py)",
        "config": {"workload": WORKLOADS[args.config], "parallelism": f"point-block x{world}", "passes_per_scan": passes / args.steps,
                   "knn_passes_per_scan": searches / args.steps, "l2": "flushed between timed steps (256 MiB write)",
                   "sort_queries": not args.no_sort, "points_per_rank": hi - lo, "map_nodes": M_nodes, "map": map_desc},
        "device_ms_per_step": dev_ms / args.steps, "host_solve_ms_per_step": host_ms / args.steps,
        "clocks": clocks,
        "e2e": None,
        "e2e_full": {"value": e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e_ms / e_steps, "steps": e_steps, "flatten_ms": flatten_ms, "flatten_host_threads": host_threads(),
                "snapshot_only": {"value": e_steps / (s_ms * 1e-3), "ms_per_step": s_ms / e_steps, "host_wall_ms_per_stage": stage_ms,
                                  "what": "the same step without the host flatten (pre-flattened pinned arrays)"},
                "what": "flatten of the live ikd-Tree (host, OpenMP) + upload_map_compact (20 B/node, boxes + cell index rebuilt on the "
                        "device) + upload_scan (pinned host buffers) + IESKF update + download of normal_y/selected"},
        "gpu_launches": launches,
        "roofline": roof, "roofline_secondary": roof2, "cpu_baseline": cpu,
    }
    full = line.pop("e2e_full")
    if i_obj is not None:
        line["e2e"] = dict(i_obj, mode="device-resident map (deltas)", full_snapshot={k: v for k, v in full.items() if k != "snapshot_only"},
                           snapshot_only=full["snapshot_only"], host_threads=host_threads())
    else:
        line["e2e"] = dict(full, mode="full snapshot per scan")
    if parity_n is not None:
        line["parity_n"] = parity_n
    if world > 1:
        xp = int(c1.exchange_passes - c0.exchange_passes)
        line["exchange_wait_us_per_pass"] = {
            "min_exchange": 1e3 * float(c1.exchange_min_wait_ms - c0.exchange_min_wait_ms) / max(xp, 1),
            "sum_exchange": 1e3 * float(c1.exchange_sum_wait_ms - c0.exchange_sum_wait_ms) / max(xp, 1), "passes": xp,
            "what": "rank 0, %globaltimer inside pass_kernel: push of this GPU's keys / system to every peer + wait for all of theirs; the "
                    "MIN exchange is where a rank waits for the slowest rank to have launched its pass (host launch skew)"}
    print(json.dumps(line))
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    model.close()
    if tree is not None:
        with c_stdout_to_stderr():
            tree.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        print(json.dumps({"error": f"--gpus {args.gpus} needs torchrun --nproc-per-node {args.gpus}"}))
        sys.exit(2)
    if args.config == "C5":
        run_ours_c5(args, rank, world)
    else:
        run_ours(args, rank, world)


if __name__ == "__main__":
    main()
