"""Radius search from and into device memory (pn_tree_query_radius_dev) against the host-buffer call
(BallTree.query_radius_batch on numpy queries) on one GPU.  Two shapes: C4 (10M x 3 f32 uniform, 1M queries, r = 0.01)
and a 16-d clustered set (4M points, 1M queries) whose radius is the median distance to the 50th neighbour over a sample
of queries.  Each call is warmed up at full size, then timed `--reps` times and the median reported:
  - host call: host clock around the call (it returns with the result in host memory) and its device_ms counter;
  - device call: CUDA events around one sync=0 call on a user stream, queries already in HBM, capacity = the total.
The device call's offsets and indices must equal the host call's.  The card's name and power limit are read in the same
run.  One JSON line goes to --out.
    python scripts/radius_dev.py [--out profiles/radius_dev.jsonl] [--reps 5]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import petal_neighbors_b200 as pn  # noqa: E402
from petal_neighbors_b200 import synth  # noqa: E402


def card():
    """name and power limit of GPU 0, read in this run"""
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except Exception:   # noqa: BLE001
        power = "unknown"
    return name, power


def measure(label, pts, Q, r, reps):
    bt = pn.BallTree.euclidean(pts, device=0)
    if r is None:   # the median distance to the 50th neighbour of a sample
        r = np.float32(np.median(bt.query_batch(Q[:2000], 50)[1][:, -1]))
    nq = len(Q)
    # host-buffer call
    host_ms, dev_ms = [], []
    for i in range(reps + 1):
        t0 = time.perf_counter()
        ho, hi = bt.query_radius_batch(Q, r)
        if i:
            host_ms.append((time.perf_counter() - t0) * 1e3)
            dev_ms.append(bt.counters()["device_ms"])
    total = int(ho[-1])
    # device-resident call: queries in HBM, outputs sized to the total
    qd = torch.from_numpy(Q).cuda()
    offs = torch.empty(nq + 1, dtype=torch.int64, device="cuda")
    ind = torch.empty(max(total, 1), dtype=torch.int64, device="cuda")
    st = torch.cuda.Stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev_ms = []
    for i in range(reps + 1):
        e0.record(st)
        bt.query_radius_dev(qd.data_ptr(), nq, pts.shape[1], r, offs.data_ptr(), ind.data_ptr(), total,
                            stream=st.cuda_stream, sync=False)
        e1.record(st)
        st.synchronize()
        if i:
            ev_ms.append(e0.elapsed_time(e1))
    same = bool(np.array_equal(offs.cpu().numpy().view(np.uint64), ho) and
                np.array_equal(ind[:total].cpu().numpy().view(np.uint64), hi))
    med = lambda v: float(np.median(v))  # noqa: E731
    return {"shape": label, "n": len(pts), "d": pts.shape[1], "nq": nq, "radius": float(r), "total_hits": total,
            "hits_per_query": total / nq,
            "host_call_wall_ms": med(host_ms), "host_call_device_ms": med(dev_ms),
            "host_call_queries_per_s": nq / med(host_ms) * 1e3,
            "dev_call_event_ms": med(ev_ms), "dev_call_queries_per_s": nq / med(ev_ms) * 1e3,
            "dev_call_event_ms_all": ev_ms, "host_call_wall_ms_all": host_ms, "identical": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "radius_dev.jsonl"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the point and query counts (rehearsals)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    name, power = card()
    rows = []
    n, nq = int(10_000_000 * a.scale), int(1_000_000 * a.scale)
    rows.append(measure("C4 uniform 3-d", synth.uniform_torch(n, 3, 2, torch.float32).cpu().numpy(),
                        synth.uniform_torch(nq, 3, 3, torch.float32).cpu().numpy(), np.float32(0.01), a.reps))
    n, nq = int(4_000_000 * a.scale), int(1_000_000 * a.scale)
    rows.append(measure("clustered 16-d", synth.fast_gaussian_mixture(n, 16, 5, n_centers=1024, sigma=0.05),
                        synth.fast_gaussian_mixture(nq, 16, 6, n_centers=1024, sigma=0.05), None, a.reps))
    rec = {"gpu": name, "power_limit": power, "reps": a.reps, "shapes": rows}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        f.write(json.dumps(rec) + "\n")
    print(json.dumps(rec), flush=True)
    if not all(r["identical"] for r in rows):
        sys.exit("parity check FAILED: the device call's offsets or indices differ from the host call")
    print("parity ok: offsets and indices identical")


if __name__ == "__main__":
    main()
