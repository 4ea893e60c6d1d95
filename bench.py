#!/usr/bin/env python
"""bench.py -- the headline benchmark of the hot path (BASELINE.json metric: k-NN queries/sec).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c2|t128|c1] [--no-extras] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic queries: batched exact k-NN (k = 10) on the
configuration BASELINE.json quotes the metric on, config 2: BallTree 1M x 16 f32 uniform points, 1M queries per GPU.
N > 1 shards the queries over ranks with the tree replicated -- built once on rank 0 and sent to the other ranks with
ncclBroadcast inside the library (pn_tree_replicate) -- and no data-path collective; weak scaling: every rank answers
its own 1M queries.

  value : whole-job queries/s with queries and outputs resident in HBM (pn_tree_query_knn_dev), CUDA events on the
          launching stream, max over ranks.
  e2e   : the same metric through the host-buffer C-ABI call (pn_balltree_query_f32) with pinned host buffers -- H2D of
          the queries and D2H of (idx, dist) inside the timed region.
  roofline / cpu_baseline : see DESIGN.md "Measurement".
  extra : the other BASELINE configurations, each with its own timing, e2e, pairs/(N*Q) and roofline:
            t128  BallTree 10M x 128 f32 uniform, 1M queries, k=10 (north-star target T; tensor roofline)
            c3    VantagePointTree 1M x 64 f32 Gaussian mixture, 1M queries, 1-NN
            c4    BallTree::query_radius 10M x 3 f32, 1M queries, r = 0.01
          and for N > 1 the two multi-GPU arms on T: `strong_t128` (ONE 1M-query batch split over the ranks, tree
          replicated over NCCL) and `sharded_t128` (points sharded by subtree, every rank scans all queries, lists
          exchanged by NCCL all-gather / slice exchange and merged), with scan / exchange / merge time and NCCL bytes.

`--impl reference` times the reference's own CPU implementation of the path (the oracle's C restatement of the Rust
crate -- no Rust toolchain exists in this image) on the host cores.

`--dump-outputs DIR` writes what the last timed step returned (rank 0's batch) as DIR/*.npy, so that two builds can be
compared output for output on the same seeded inputs: a fixed, seeded sample of query rows (`query_rows`), their
neighbour indices (`indices`, float64: exact below 2^53) and distances (`distances`, the tree's dtype), 32 MiB at most.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "knn_queries_per_sec_k10"
UNIT = "queries/s"

WORKLOADS = {
    # name: (n_points, dim, n_queries per GPU, k, dtype, generator, label)
    "c2": (1_000_000, 16, 1_000_000, 10, np.float32, "uniform",
           "BallTree 1M x 16 f32 uniform, 1M batched queries per GPU, k=10 (BASELINE config 2)"),
    "t128": (10_000_000, 128, 1_000_000, 10, np.float32, "uniform",
             "BallTree 10M x 128 f32 uniform, 1M batched queries per GPU, k=10 (north-star target shape)"),
    "c1": (10_000, 3, 10_000, 10, np.float64, "self",
           "BallTree 10k x 3 f64 uniform, every point a query, k=10 (BASELINE config 1)"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return {"hbm": float(j["hbm_gbs"]), "tc_burst": float(j.get("bf16_tflops", 1590.0)),
                    "tc_sustained": float(j.get("bf16_tflops_sustained", 1400.0)), "which": "measured"}
        except Exception:
            pass
    return {"hbm": 6650.0, "tc_burst": 1590.0, "tc_sustained": 1400.0, "which": "fallback"}


def config_dict(wl, world, nq, k):
    """identical for the B200 arm and the reference arm (the driver compares them)"""
    return {"workload": WORKLOADS[wl][6], "queries_per_gpu": nq, "k": k, "sharding": f"queries x{world}, tree replicated",
            "l2": "flushed between timed steps (256 MiB write, untimed)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            if ts < t0 or ts > t1 + 0.2:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 32 << 20


def dump_outputs(out_dir, idx, dist):
    """Writes the rows of a seeded sample of the (nq, k) result tensors `idx`, `dist` (see --dump-outputs)."""
    import torch
    nq, k = idx.shape
    m = min(nq, DUMP_BYTES // (8 + k * (8 + dist.element_size())))
    rows = np.sort(np.random.default_rng(0).choice(nq, size=m, replace=False))
    sel = torch.from_numpy(rows).to(idx.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "query_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "indices.npy"), idx.index_select(0, sel).cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "distances.npy"), dist.index_select(0, sel).cpu().numpy())


def make_inputs(wl, rank):
    import petal_neighbors_b200  # noqa: F401
    from petal_neighbors_b200 import synth
    n, d, nq, k, dtype, gen, _ = WORKLOADS[wl]
    pts = synth.fast_uniform(n, d, 2, dtype)
    if gen == "self":
        Q = pts.copy()
    else:
        Q = synth.fast_uniform(nq, d, 3, dtype, row0=rank * nq)  # each rank owns a slice of one query stream
    return pts, Q


def algorithmic_bytes(n, d, nq, k, s, pairs):
    """SURVEY.md 8d / BASELINE.md 4: B_alg = B_min + pairs*d*s/128."""
    b_min = n * d * s + nq * d * s + nq * k * (8 + s)
    return b_min + pairs * d * s / 128.0


def rooflines(n, d, nq, k, s, pairs, ms, kp=None):
    """Both rooflines of one launch: the contract's HBM formula and the tensor roof (2 d pairs useful flops, and the issued
    flops of the padded augmented contraction 2 Kp pairs) against the MEASURED 16-bit dense peak -- the MMA is kind::f16."""
    pk = peaks()
    t = ms * 1e-3
    b_alg = algorithmic_bytes(n, d, nq, k, s, pairs)
    hbm = b_alg / t / 1e9
    useful = 2.0 * d * pairs / t / 1e12
    out = {"hbm": {"achieved_gbs": hbm, "peak_gbs": pk["hbm"], "frac": hbm / pk["hbm"], "algorithmic_bytes": b_alg},
           "tensor": {"useful_tflops": useful, "frac_of_burst": useful / pk["tc_burst"], "frac_of_sustained": useful / pk["tc_sustained"],
                      "peak_burst_tflops": pk["tc_burst"], "peak_sustained_tflops": pk["tc_sustained"],
                      "peak_is": "measured dense bf16/fp16 GEMM (MEASURED_PEAKS.json); the filter MMA is tcgen05 kind::f16"},
           "peak_source": "of " + pk["which"]}
    if kp:
        issued = 2.0 * kp * pairs / t / 1e12
        out["tensor"].update({"issued_tflops": issued, "issued_frac_of_burst": issued / pk["tc_burst"],
                              "issued_frac_of_sustained": issued / pk["tc_sustained"], "k_padded": kp})
    return out


def cpu_reference(pts, Q, k, budget_s=20.0):
    """The reference's CPU path (oracle port) on a bounded sample of the same workload."""
    from oracle import pyoracle
    pyoracle.build()
    threads = pyoracle.max_threads()
    t0 = time.perf_counter()
    tree = pyoracle.BallTree.euclidean(pts)
    build_s = time.perf_counter() - t0
    # calibrate the sample on a few queries, then time about budget_s of CPU work
    probe = min(64, Q.shape[0])
    t0 = time.perf_counter()
    tree.query_batch(Q[:probe], k, n_threads=threads)
    per_q = (time.perf_counter() - t0) / probe
    sample = int(max(probe, min(Q.shape[0], budget_s / max(per_q, 1e-9))))
    t0 = time.perf_counter()
    _, _, ndist = tree.query_batch(Q[:sample], k, n_threads=threads)
    dt = time.perf_counter() - t0
    single = min(sample, max(16, int(3.0 / max(per_q * threads, 1e-9))))
    t0 = time.perf_counter()
    tree.query_batch(Q[:single], k, n_threads=1)
    dt1 = time.perf_counter() - t0
    return {
        "value": sample / dt, "unit": UNIT, "cores": threads, "kind": "port",
        "sample": f"first {sample} of the {Q.shape[0]} queries, reference tree (1-2 point leaves) built on all "
                  f"{pts.shape[0]} points, OpenMP outer loop over queries",
        "single_thread_value": single / dt1, "single_thread_sample": single,
        "build_seconds": build_s, "distance_evals_per_query": ndist / sample,
    }, tree, sample


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload
    n, d, nq, k, dtype, gen, label = WORKLOADS[wl]
    from petal_neighbors_b200 import synth  # noqa: F401  (numpy generators: no GPU is touched by this arm)
    import petal_neighbors_b200  # noqa: F401
    pts = synth.uniform(n, d, 2, dtype)
    Q = pts.copy() if gen == "self" else synth.uniform(min(nq, 200_000), d, 3, dtype)
    base, tree, sample = cpu_reference(pts, Q, k, budget_s=8.0)
    threads = base["cores"]
    for _ in range(args.warmup):
        tree.query_batch(Q[:max(16, sample // 8)], k, n_threads=threads)
    t0 = time.perf_counter()
    for s in range(args.steps):
        lo = (s * sample) % max(1, Q.shape[0] - sample + 1)
        tree.query_batch(Q[lo:lo + sample], k, n_threads=threads)
    dt = time.perf_counter() - t0
    v = args.steps * sample / dt
    base["value"] = v
    base["sample"] += f"; {sample} queries per step on the host cores (bounded sample)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32" if dtype == np.float32 else "f64", "data": "synthetic",
        "config": config_dict(wl, max(1, args.gpus), nq, k),
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------------------------------------------------
def timed_dev(tree, torch, stream, q_dev, nq, d, k, idx_dev, dist_dev, steps, warmup, flush):
    for _ in range(warmup):
        tree.query_knn_dev(q_dev.data_ptr(), nq, d, k, idx_dev.data_ptr(), dist_dev.data_ptr(), stream=stream.cuda_stream, sync=False)
    torch.cuda.synchronize()
    evs = []
    for _ in range(steps):
        flush.zero_()  # L2 flush between timed iterations (untimed)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        tree.query_knn_dev(q_dev.data_ptr(), nq, d, k, idx_dev.data_ptr(), dist_dev.data_ptr(), stream=stream.cuda_stream, sync=False)
        e1.record(stream)
        evs.append((e0, e1))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


def extra_t128(pn, torch, synth, stream, flush, steps):
    """North-star target T on one GPU: points generated and the tree BUILT on the device, 1M queries, k = 10."""
    n, d, nq, k = WORKLOADS["t128"][:4]
    t0 = time.perf_counter()
    pts_dev = synth.uniform_torch(n, d, 2, torch.float32)
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    tree = pn.BallTree.euclidean(pts_dev)
    info = tree.info()
    q_dev = synth.uniform_torch(nq, d, 3, torch.float32)
    idx_dev = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    dist_dev = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    ms = timed_dev(tree, torch, stream, q_dev, nq, d, k, idx_dev, dist_dev, steps, 1, flush)
    tree.query_knn_dev(q_dev.data_ptr(), nq, d, k, idx_dev.data_ptr(), dist_dev.data_ptr(), stream=stream.cuda_stream, sync=True)
    ctr = tree.counters()
    # end to end through the host-buffer ABI, pinned buffers
    q_pin = q_dev.cpu().pin_memory()
    idx_pin = torch.empty((nq, k), dtype=torch.int64).pin_memory()
    dist_pin = torch.empty((nq, k), dtype=torch.float32).pin_memory()
    from petal_neighbors_b200 import _ffi
    fn = _ffi.lib().pn_balltree_query_f32
    e2e_s = None
    for it in range(2):   # the first host-buffer call of a handle allocates its staging buffers: warm-up at full size
        t0 = time.perf_counter()
        rc = fn(tree._h, q_pin.data_ptr(), nq, d, k, idx_pin.data_ptr(), dist_pin.data_ptr())
        e2e_s = time.perf_counter() - t0
        if rc != 0:
            raise RuntimeError(_ffi.last_error())
    same = bool(torch.equal(idx_pin, idx_dev.cpu()) and torch.equal(dist_pin, dist_dev.cpu()))
    m = float(np.mean(ms))
    kp = (d + 6 + 31) // 32 * 32
    rl = rooflines(n, d, nq, k, 4, ctr["pairs"], ctr["scan_ms"], kp)
    out = {"workload": WORKLOADS["t128"][6], "ms_per_step": m, "value": nq / (m * 1e-3), "unit": UNIT, "steps": len(ms),
           "kernel_ms": ctr["scan_ms"], "pairs_over_NQ": ctr["pairs"] / (float(n) * nq), "rerank_per_query": ctr["rerank_pairs"] / nq,
           "e2e": {"value": nq / e2e_s, "unit": UNIT, "h2d_bytes_per_step": nq * d * 4, "d2h_bytes_per_step": nq * k * 12,
                   "matches_device_path": same},
           "build_seconds": info["build_seconds"], "build": "on the device (pn_balltree_create_dev_f32), points generated in HBM",
           "generate_seconds": gen_s, "device_bytes": info["device_bytes"],
           "roofline": {"bound": "tensor", "achieved": rl["tensor"]["useful_tflops"], "peak": rl["tensor"]["peak_sustained_tflops"],
                        "unit": "TFLOP/s", "frac": rl["tensor"]["frac_of_sustained"],
                        "note": "useful flops 2*d*pairs over the measured SUSTAINED 16-bit dense peak (a 2.3 s kernel runs under the power cap)",
                        "detail": rl}}
    del tree, pts_dev
    torch.cuda.empty_cache()
    return out


def extra_c3(pn, torch, synth, stream, flush, steps):
    """BASELINE config 3: VantagePointTree 1M x 64 f32 Gaussian mixture, 1M queries, query_nearest."""
    n = nq = 1_000_000
    d = 64
    pts = synth.fast_gaussian_mixture(n, d, 5, n_centers=1024, sigma=0.05, center_seed=4)
    Q = synth.fast_gaussian_mixture(nq, d, 6, n_centers=1024, sigma=0.05, center_seed=4)
    vp = pn.VantagePointTree.euclidean(pts)
    info = vp.info()
    q_dev = torch.from_numpy(Q).cuda()
    idx_dev = torch.empty((nq, 1), dtype=torch.int64, device="cuda")
    dist_dev = torch.empty((nq, 1), dtype=torch.float32, device="cuda")
    ms = timed_dev(vp, torch, stream, q_dev, nq, d, 1, idx_dev, dist_dev, steps, 1, flush)
    vp.query_knn_dev(q_dev.data_ptr(), nq, d, 1, idx_dev.data_ptr(), dist_dev.data_ptr(), stream=stream.cuda_stream, sync=True)
    ctr = vp.counters()
    q_pin = torch.from_numpy(Q).pin_memory()
    idx_pin = torch.empty((nq,), dtype=torch.int64).pin_memory()
    dist_pin = torch.empty((nq,), dtype=torch.float32).pin_memory()
    from petal_neighbors_b200 import _ffi
    fn = _ffi.lib().pn_vptree_query_nearest_f32
    wall = []
    for it in range(steps + 1):
        t0 = time.perf_counter()
        rc = fn(vp._h, q_pin.data_ptr(), nq, d, idx_pin.data_ptr(), dist_pin.data_ptr())
        dt = time.perf_counter() - t0
        if rc != 0:
            raise RuntimeError(_ffi.last_error())
        if it:
            wall.append(dt)
    ctr_host = vp.counters()
    same = bool(torch.equal(idx_pin, idx_dev[:, 0].cpu()) and torch.equal(dist_pin, dist_dev[:, 0].cpu()))
    m = float(np.mean(ms))
    kp = (d + 6 + 31) // 32 * 32
    rl = rooflines(n, d, nq, 1, 4, float(ctr["pairs"]), ctr["scan_ms"], kp)
    return {"workload": "VantagePointTree 1M x 64 f32 Gaussian mixture (1024 x sigma 0.05), 1M queries, query_nearest (BASELINE config 3)",
            "ms_per_step": m, "value": nq / (m * 1e-3), "unit": UNIT, "steps": len(ms), "kernel_ms": ctr["scan_ms"],
            "pairs_over_NQ": ctr["pairs"] / (float(n) * nq), "rerank_per_query": ctr["rerank_pairs"] / nq,
            "e2e": {"value": nq / float(np.mean(wall)), "unit": UNIT, "h2d_bytes_per_step": int(ctr_host["h2d_bytes"]),
                    "d2h_bytes_per_step": int(ctr_host["d2h_bytes"]), "matches_device_path": same},
            "build_seconds": info["build_seconds"],
            "build": "VP arrays on the host; the ball partitions the tensor path scans (reference rule, then two-means) on the device",
            "tensor_partition": "two-means" if info["tensor_partition"] == 1 else "reference", "seeded_scan": bool(info["prune_seeded"]),
            "tile_bitmaps": bool(info["prune_tiles"]), "est_tile_frac": info["est_tile_frac"],
            "roofline": {"bound": "tensor", "achieved": rl["tensor"]["useful_tflops"], "peak": rl["tensor"]["peak_burst_tflops"], "unit": "TFLOP/s",
                         "frac": rl["tensor"]["frac_of_burst"],
                         "note": "flops of the (query, point) pairs the pruned scan really evaluates, over the whole scan time (sort, seeds, tile "
                                 "bitmaps, filter); dense_equivalent_tflops = 2 d N Q / the same time, what a scan without pruning would need to do",
                         "dense_equivalent_tflops": 2.0 * d * float(n) * nq / (ctr["scan_ms"] * 1e-3) / 1e12 if ctr["scan_ms"] else None,
                         "detail": rl}}


def extra_c4(pn, torch, synth, steps):
    """BASELINE config 4: BallTree::query_radius 10M x 3 f32, 1M queries, r = 0.01, CSR output."""
    n, nq, d, r = 10_000_000, 1_000_000, 3, np.float32(0.01)
    pts_dev = synth.uniform_torch(n, d, 7, torch.float32)
    bt = pn.BallTree.euclidean(pts_dev)
    info = bt.info()
    Q = synth.fast_uniform(nq, d, 8, np.float32)
    wall, dev = [], []
    hits = 0
    ctr = None
    for it in range(steps + 1):
        t0 = time.perf_counter()
        offs, ind = bt.query_radius_batch(Q, r)
        dt = time.perf_counter() - t0
        ctr = bt.counters()
        hits = int(offs[-1])
        if it:
            wall.append(dt); dev.append(ctr["device_ms"])
        del offs, ind
    m = float(np.mean(dev))
    b_alg = n * d * 4 + nq * d * 4 + 8 * (nq + 1) + 8 * hits + ctr["pairs"] * d * 4 / 128.0
    pk = peaks()
    ach = b_alg / (m * 1e-3) / 1e9
    # k-NN (k = 10) on the same tree: narrow rows take the warp-per-query scan
    kw, kd, kc = [], [], None
    for it in range(steps + 1):
        t0 = time.perf_counter()
        bt.query_batch(Q, 10)
        dt = time.perf_counter() - t0
        kc = bt.counters()
        if it:
            kw.append(dt); kd.append(kc["device_ms"])
    knn = {"workload": "BallTree::query on the same tree, 1M queries, k = 10 (warp-per-query scan)", "ms_per_step": float(np.mean(kd)),
           "value": nq / (float(np.mean(kd)) * 1e-3), "unit": UNIT, "scan_ms": kc["scan_ms"], "pairs_per_query": kc["pairs"] / nq,
           "e2e": {"value": nq / float(np.mean(kw)), "unit": UNIT, "h2d_bytes_per_step": int(kc["h2d_bytes"]), "d2h_bytes_per_step": int(kc["d2h_bytes"]),
                   "note": "wall clock around pn_balltree_query_f32, pageable numpy buffers"}}
    return {"knn_k10": knn, "workload": "BallTree::query_radius 10M x 3 f32 uniform, 1M queries, r = 0.01 (BASELINE config 4)",
            "ms_per_step": m, "value": nq / (m * 1e-3), "unit": UNIT, "steps": len(dev),
            "timing": "device_ms of the host-buffer call (pipelined chunks: H2D, traversal, D2H of the CSR result)",
            "hits_per_query": hits / nq, "pairs_per_query": ctr["pairs"] / nq, "pairs_over_NQ": ctr["pairs"] / (float(n) * nq),
            "e2e": {"value": nq / float(np.mean(wall)), "unit": UNIT, "h2d_bytes_per_step": int(ctr["h2d_bytes"]), "d2h_bytes_per_step": int(ctr["d2h_bytes"]),
                    "note": "wall clock around pn_balltree_query_radius_f32 with pageable numpy buffers, result widened to u64 on the host"},
            "build_seconds": info["build_seconds"], "build": "on the device",
            "roofline": {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"], "algorithmic_bytes": b_alg,
                         "note": "d = 3 prunes to ~1.2e3 pairs per query: bound by traversal latency and host-side result handling, not by HBM"}}


def extra_c1(pn, synth, steps):
    """BASELINE config 1 (the reference's own bench, benches/ball_tree.rs:53-59): BallTree 10k x 3 f64, every point a
    query, k = 10; host buffers in and out (query_batch) and the no-upload self query."""
    n, d, k = 10_000, 3, 10
    pts = synth.uniform(n, d, 1, np.float64)
    bt = pn.BallTree.euclidean(pts)
    wall, dev, ctr = [], [], None
    for it in range(10 * steps + 1):
        t0 = time.perf_counter()
        idx, dist = bt.query_batch(pts, k)
        dt = time.perf_counter() - t0
        ctr = bt.counters()
        if it:
            wall.append(dt); dev.append(ctr["device_ms"])
    t0 = time.perf_counter()
    for it in range(10):
        si, sd = bt.query_self(k)
    self_s = (time.perf_counter() - t0) / 10
    return {"workload": "BallTree 10k x 3 f64, every point a query, k = 10 (BASELINE config 1)", "ms_per_step": float(np.mean(dev)),
            "value": n / (float(np.mean(dev)) * 1e-3), "unit": UNIT, "steps": len(dev), "scan_ms": ctr["scan_ms"], "pairs_over_NQ": ctr["pairs"] / float(n * n),
            "e2e": {"value": n / float(np.mean(wall)), "unit": UNIT, "h2d_bytes_per_step": int(ctr["h2d_bytes"]), "d2h_bytes_per_step": int(ctr["d2h_bytes"]),
                    "note": "wall clock around pn_balltree_query_f64, pageable numpy buffers"},
            "self_query": {"value": n / self_s, "unit": UNIT, "same_rows": bool(np.array_equal(si, idx) and np.array_equal(sd, dist))},
            "path": "warp-per-query scan (f64, d = 3)"}


def extra_multi_gpu(pn, torch, dist, synth, comm, rank, world, local, steps):
    """The two multi-GPU arms on the north-star shape T (10M x 128 f32, ONE batch of 1M queries, k = 10)."""
    from petal_neighbors_b200 import parallel
    n, d, nq, k = WORKLOADS["t128"][:4]
    out = {}
    q_all = synth.uniform_torch(nq, d, 3, torch.float32)
    stream = torch.cuda.current_stream()
    # ---- strong scaling, query sharding: the tree is built once on rank 0 and replicated with ncclBroadcast ----
    t0 = time.perf_counter()
    tree0 = None
    if rank == 0:
        tree0 = pn.BallTree.euclidean(synth.uniform_torch(n, d, 2, torch.float32))
    build_s = time.perf_counter() - t0
    torch.cuda.synchronize(); dist.barrier()
    t0 = time.perf_counter()
    tree = parallel.replicate(tree0, comm, 0)
    torch.cuda.synchronize(); dist.barrier()
    repl_s = time.perf_counter() - t0
    lo, hi = parallel.query_slice(nq, rank, world)
    mq = hi - lo
    oi = torch.empty((mq, k), dtype=torch.int64, device="cuda")
    od = torch.empty((mq, k), dtype=torch.float32, device="cuda")
    qs = q_all[lo:hi]
    ms = []
    for it in range(steps + 1):
        torch.cuda.synchronize(); dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        tree.query_knn_dev(qs.data_ptr(), mq, d, k, oi.data_ptr(), od.data_ptr(), stream=stream.cuda_stream, sync=False)
        e1.record(stream)
        torch.cuda.synchronize()
        if it:
            ms.append(e0.elapsed_time(e1))
    t = torch.tensor([float(np.mean(ms))], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    chk = torch.tensor([int(oi.sum().item())], dtype=torch.int64, device="cuda")
    dist.all_reduce(chk)
    m = float(t[0])
    out["strong_t128"] = {"workload": "ONE batch of 1M queries against BallTree 10M x 128 f32, k=10, split over the ranks; tree replicated",
                          "scaling": "strong", "n_gpus": world, "ms_per_batch": m, "value": nq / (m * 1e-3), "unit": UNIT,
                          "timing": "CUDA events per rank, max over ranks", "build_seconds_rank0": build_s,
                          "replicate_seconds": repl_s, "replicate": "pn_tree_replicate: ncclBroadcast of the flattened tree and the operand image",
                          "replicated_bytes": tree.info()["device_bytes"], "index_checksum": int(chk[0])}
    del tree, tree0, oi, od
    torch.cuda.empty_cache()
    # ---- point sharding by subtree + NCCL exchange + merge (the C5 structure at T's size) ----
    pts_dev = synth.uniform_torch(n, d, 2, torch.float32)
    t0 = time.perf_counter()
    st = parallel.ShardedBallTree(pts_dev, comm)
    shard_build_s = time.perf_counter() - t0
    del pts_dev
    torch.cuda.empty_cache()
    arms = {}
    for name, mode in (("allgather", parallel.PN_EXCHANGE_ALLGATHER), ("slice", parallel.PN_EXCHANGE_SLICE)):
        tms, stats = [], None
        for it in range(steps + 1):
            torch.cuda.synchronize(); dist.barrier()
            gi, gd = st.query_batch_dev(q_all, k, exchange=mode)
            if it:
                tms.append(st.stats["total_ms"])
            stats = dict(st.stats)
        t = torch.tensor([float(np.mean(tms)), stats["scan_ms"], stats["exchange_ms"], stats["merge_ms"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        b = torch.tensor([stats["nccl_bytes_sent"], int(gi.sum().item())], dtype=torch.int64, device="cuda")
        dist.all_reduce(b)
        m = float(t[0])
        arms[name] = {"ms_per_batch": m, "value": nq / (m * 1e-3), "unit": UNIT, "scan_ms": float(t[1]), "exchange_ms": float(t[2]),
                      "merge_ms": float(t[3]), "nccl_bytes_all_ranks": int(b[0]), "nccl_calls_per_rank": stats["nccl_calls"],
                      "chunks": stats["n_chunks"], "index_checksum": int(b[1]),
                      "note": "exchange_ms overlaps the next chunk's scan (separate stream); times are max over ranks"}
        del gi, gd
    out["sharded_t128"] = {"workload": "BallTree 10M x 128 f32 sharded by the depth-log2(N) subtrees, every rank scans ALL 1M queries, k=10; "
                                       "per-shard lists exchanged over NCCL and merged (the structure of BASELINE config 5)",
                           "n_gpus": world, "points_per_rank": st.tree.info()["n_points"], "shard_build_seconds": shard_build_s, **arms}
    # ---- the same sharding from ONE process (pn_multi_*): merge kernels read the other devices' lists over NVLink, no
    # collective.  Runs as a child process of rank 0 with a time limit while every rank's GPU is idle (the ranks wait at a
    # CPU-side barrier, never inside an NCCL kernel), so that a failure there cannot take the bench line down.
    del st, q_all
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    cpu_group = dist.new_group(backend="gloo")
    dist.barrier(group=cpu_group)
    if rank == 0:
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "multi_arm.py"), str(world)], capture_output=True, text=True, timeout=420)
            line = [l for l in r.stdout.splitlines() if l.startswith("{")]
            out["multi_one_process"] = json.loads(line[-1]) if line else {"error": (r.stderr or r.stdout)[-400:]}
        except Exception as e:  # noqa
            out["multi_one_process"] = {"error": repr(e)}
    dist.barrier(group=cpu_group)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--algo", default="auto", choices=["auto", "simt", "tensor"])
    ap.add_argument("--bucket", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra configurations (t128, c3, c4, multi-GPU arms)")
    ap.add_argument("--extras", default="", help="comma-separated subset of t128,c3,c4,multi (default: all)")
    ap.add_argument("--queries", type=int, default=0, help="override queries per GPU (profiling runs only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's outputs as DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the B200 arm (the reference arm's query sample depends on its timing)")
    sys.dont_write_bytecode = True  # the tree may be read-only; leave it as it was found

    if args.impl == "reference":
        run_reference_arm(args)
        return

    if os.environ.get("NCCL_DEBUG", "VERSION").upper() in ("VERSION", "WARN"):
        os.environ["NCCL_DEBUG"] = "NONE"   # NCCL prints its version banner on stdout; stdout carries the one JSON line
    import torch
    import torch.distributed as dist
    import petal_neighbors_b200 as pn
    from petal_neighbors_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the B200 arm")
    torch.cuda.set_device(local)
    comm = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        from petal_neighbors_b200 import parallel
        comm = parallel.Comm.from_torch(device=local)

    wl = args.workload
    reduced = False
    if args.queries:
        w = list(WORKLOADS[wl]); w[2] = args.queries; w[6] += f" [REDUCED to {args.queries} queries: profiling run, not a bench line]"
        WORKLOADS[wl] = tuple(w)
        reduced = True
    n, d, nq, k, dtype, gen, label = WORKLOADS[wl]
    s = np.dtype(dtype).itemsize
    tdtype = torch.float32 if dtype == np.float32 else torch.float64
    pts, Q = make_inputs(wl, rank)
    nq = Q.shape[0]
    algo = {"auto": pn.PN_ALGO_AUTO, "simt": pn.PN_ALGO_SIMT, "tensor": pn.PN_ALGO_TENSOR}[args.algo]
    # the tree: built once (rank 0) and, for N > 1, replicated to the other ranks with ncclBroadcast inside the library
    t0 = time.perf_counter()
    tree = pn.BallTree.euclidean(pts, device=local, algo=algo, bucket_size=args.bucket) if rank == 0 or world == 1 else None
    if world > 1:
        from petal_neighbors_b200 import parallel
        tree = parallel.replicate(tree, comm, 0)
    tree_s = time.perf_counter() - t0
    info = tree.info()

    stream = torch.cuda.Stream()  # explicit (non-default) stream: handle 0 would mean "the tree's own stream"
    torch.cuda.set_stream(stream)
    q_dev = torch.from_numpy(Q).cuda()
    idx_dev = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    dist_dev = torch.empty((nq, k), dtype=tdtype, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    q_pin = torch.from_numpy(Q).pin_memory()
    idx_pin = torch.empty((nq, k), dtype=torch.int64).pin_memory()
    dist_pin = torch.empty((nq, k), dtype=tdtype).pin_memory()

    def step_dev():
        tree.query_knn_dev(q_dev.data_ptr(), nq, d, k, idx_dev.data_ptr(), dist_dev.data_ptr(),
                           stream=stream.cuda_stream, sync=False)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # ---------------- kernel-resident timing (value) ----------------
    for _ in range(args.warmup):
        step_dev()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    t_wall0 = time.time()
    evs = []
    for _ in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations (untimed)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        step_dev()
        e1.record(stream)
        evs.append((e0, e1))
    barrier()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1)
    ms_steps = [a.elapsed_time(b) for a, b in evs]
    total_ms = float(sum(ms_steps))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, idx_dev, dist_dev)
    # one synchronous call to read the engine's work counters for exactly one step
    tree.query_knn_dev(q_dev.data_ptr(), nq, d, k, idx_dev.data_ptr(), dist_dev.data_ptr(),
                       stream=stream.cuda_stream, sync=True)
    ctr = tree.counters()

    # ---------------- end-to-end through the host-buffer C ABI (e2e) ----------------
    from petal_neighbors_b200 import _ffi
    fn = getattr(_ffi.lib(), "pn_balltree_query_f32" if dtype == np.float32 else "pn_balltree_query_f64")

    def step_host():
        rc = fn(tree._h, q_pin.data_ptr(), nq, d, k, idx_pin.data_ptr(), dist_pin.data_ptr())
        if rc != 0:
            raise RuntimeError(_ffi.last_error())

    for _ in range(min(args.warmup, 2)):
        step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    ctr_host = tree.counters()
    # sanity: both paths return the same answer
    same = bool(torch.equal(idx_pin, idx_dev.cpu()) and torch.equal(dist_pin, dist_dev.cpu()))

    if world > 1:
        t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_s = float(t[0]), float(t[1])

    # ---------------- the other configurations ----------------
    extra = {}
    want = set(x for x in args.extras.split(",") if x) or {"t128", "c3", "c4", "c1", "multi"}
    if not args.no_extras and not reduced and wl == "c2":
        del q_dev, idx_dev, dist_dev, q_pin, idx_pin, dist_pin
        esteps = max(1, min(args.steps, 3))
        torch.cuda.empty_cache()
        if world == 1:
            for name, fnx in (("t128", lambda: extra_t128(pn, torch, synth, stream, flush, esteps)),
                              ("c3", lambda: extra_c3(pn, torch, synth, stream, flush, esteps)),
                              ("c4", lambda: extra_c4(pn, torch, synth, esteps)),
                              ("c1", lambda: extra_c1(pn, synth, esteps))):
                if name not in want:
                    continue
                try:
                    t0 = time.perf_counter()
                    extra[name] = fnx()
                    extra[name]["wall_seconds"] = time.perf_counter() - t0
                except Exception as e:  # noqa: an extra must never take the headline line down
                    extra[name] = {"error": repr(e)}
                torch.cuda.empty_cache()
        elif "multi" in want:
            try:
                del tree
                torch.cuda.empty_cache()
                extra.update(extra_multi_gpu(pn, torch, dist, synth, comm, rank, world, local, max(1, min(args.steps, 2))))
            except Exception as e:  # noqa
                extra["multi_gpu_error"] = repr(e)

    if rank == 0:
        pk = peaks()
        pairs = ctr["pairs"]
        scan_ms = ctr["scan_ms"] if ctr["scan_ms"] > 0 else total_ms / args.steps
        kp = (d + 6 + 31) // 32 * 32 if ctr["filter_pairs"] else None
        rl = rooflines(n, d, nq, k, s, pairs, scan_ms, kp)
        traffic, traffic_src = None, None
        prof = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(prof):
            try:
                ent = json.load(open(prof)).get(wl if ctr["filter_pairs"] else wl + "_simt")
                if int(ent["queries"]) == nq:       # a measurement at this launch size, never an extrapolation
                    traffic, traffic_src = float(ent["bytes_per_launch"]), ent.get("source")
            except Exception:
                traffic = None
        out = {
            "metric": METRIC, "value": world * nq * args.steps / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if dtype == np.float32 else "f64", "data": "synthetic",
            "config": config_dict(wl, world, nq, k),
            "engine": {"bucket_size_max": info["bucket_size_max"], "tree_levels": info["n_levels"], "algo": args.algo,
                       "tree_build_seconds": info["build_seconds"], "tree_seconds_incl_replication": tree_s,
                       "seeded_scan": bool(info["prune_seeded"]), "tile_bitmaps": bool(info["prune_tiles"]),
                       "est_seed_candidates": info["est_seed_candidates"], "est_tile_frac": info["est_tile_frac"],
                       "tree": "built on the device on rank 0" + (", replicated with ncclBroadcast (pn_tree_replicate)" if world > 1 else "")},
            "e2e": {"value": world * nq * args.steps / e2e_s, "unit": UNIT,
                    "h2d_bytes_per_step": int(ctr_host["h2d_bytes"]), "d2h_bytes_per_step": int(ctr_host["d2h_bytes"]),
                    "timing": "wall clock around the synchronous host-buffer ABI call, pinned buffers, max over ranks",
                    "matches_device_path": same},
            "gpu_launches": int(ctr["kernel_launches"]) * args.steps,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": rl["hbm"]["achieved_gbs"], "peak": pk["hbm"], "unit": "GB/s", "frac": rl["hbm"]["frac"],
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": rl["peak_source"],
                         "kernel": ("tc::knn_filter_kernel (tcgen05 FP16 filter + exact rerank)" if ctr["filter_pairs"] else "knn_tile_kernel (exact SIMT scan)") + " + merge, CUDA events inside the engine, per step",
                         "rerank_pairs": int(ctr["rerank_pairs"]),
                         "kernel_ms": scan_ms, "algorithmic_bytes": rl["hbm"]["algorithmic_bytes"], "pairs": int(pairs),
                         "pairs_over_NQ": pairs / (float(n) * nq),
                         "tensor": rl["tensor"]},
            "extra": extra,
        }
        if not args.no_cpu_baseline:
            cap = 2_000_000 if d > 32 else n  # the reference tree of 10M x 128 needs ~9 GB of centroids and minutes to build
            base, _, _ = cpu_reference(pts[:cap], Q, k)
            if cap < n:
                base["sample"] += f" [reference tree built on the first {cap} of {n} points]"
            out["cpu_baseline"] = base
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        if comm is not None:
            comm.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
