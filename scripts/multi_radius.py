"""Radius search above one GPU: one GPU's BallTree.query_radius_batch against MultiGpuBallTree.query_radius_batch
(pn_multi_balltree_query_radius_f32) with the tree replicated and sharded by subtree, on 1 GPU and on the largest power of
two <= 8 of the box's GPUs.  Two shapes: C4 (10M x 3 f32, 1M queries, r = 0.01) and a 16-d clustered set whose radius is
the median distance to the 50th neighbour over a sample of queries (about 80 hits per query on average: the density is
skewed).  Every arm is warmed up once at full size, then timed (host clock around the call, which
returns with the result in host memory) `--reps` times; the median is reported with the per-rank statistics of the last
call.  Offsets and indices must be identical in every arm.  One JSON line per arm goes to --out.
    python scripts/multi_radius.py [--out profiles/multi_radius.jsonl] [--reps 3]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if os.environ.get("NCCL_DEBUG", "VERSION").upper() in ("VERSION", "WARN"):
    os.environ["NCCL_DEBUG"] = "NONE"
import torch  # noqa: E402
import petal_neighbors_b200 as pn  # noqa: E402
from petal_neighbors_b200 import parallel, synth  # noqa: E402


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


def timed(fn, reps):
    fn()   # warm-up at full size: every workspace and result buffer at its final size
    ts, out = [], None
    for _ in range(reps):
        out = None
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "multi_radius.jsonl"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the point and query counts (rehearsals)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    ng = torch.cuda.device_count()
    world = 1 << (min(ng, 8).bit_length() - 1)
    name, power = card()
    shapes = []
    n, nq = int(10_000_000 * a.scale), int(1_000_000 * a.scale)
    shapes.append(("C4 uniform 3-d", synth.uniform_torch(n, 3, 2, torch.float32).cpu().numpy(),
                   synth.uniform_torch(nq, 3, 3, torch.float32).cpu().numpy(), np.float32(0.01)))
    n, nq = int(4_000_000 * a.scale), int(1_000_000 * a.scale)
    pts = synth.fast_gaussian_mixture(n, 16, 5, n_centers=1024, sigma=0.05)
    Q = synth.fast_gaussian_mixture(nq, 16, 6, n_centers=1024, sigma=0.05)
    shapes.append(("clustered 16-d", pts, Q, None))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    ok = True
    with open(a.out, "w") as f:
        for label, pts, Q, r in shapes:
            n, d = pts.shape
            bt = pn.BallTree.euclidean(pts, device=0)
            if r is None:   # the median distance to the 50th neighbour of a sample
                r = np.float32(np.median(bt.query_batch(Q[:2000], 50)[1][:, -1]))
            arms = [("one_gpu_balltree", 1, None)]
            for w in sorted({1, world}):
                arms += [(f"replicate_{w}gpu", w, parallel.PN_SHARD_REPLICATE), (f"by_subtree_{w}gpu", w, parallel.PN_SHARD_BY_SUBTREE)]
            ref = None
            for arm, w, mode in arms:
                if mode is None:
                    h, stats = bt, None
                else:
                    h = parallel.MultiGpuBallTree(pts, list(range(w)), mode=mode)
                wall_ms, (offs, ind) = timed(lambda: h.query_radius_batch(Q, r), a.reps)
                stats = h.stats() if mode is not None else None
                if ref is None:
                    ref = (offs, ind)
                    same = True
                else:
                    same = bool(np.array_equal(offs, ref[0]) and np.array_equal(ind, ref[1]))
                ok &= same
                rec = {"shape": label, "n": n, "d": d, "nq": len(Q), "radius": float(r), "arm": arm, "n_gpus": w,
                       "wall_ms": wall_ms, "queries_per_s": len(Q) / wall_ms * 1e3, "total_hits": int(offs[-1]),
                       "hits_per_query": float(offs[-1]) / len(Q), "identical_to_one_gpu": same, "reps": a.reps,
                       "gpu": name, "power_limit": power, "gpus_on_box": ng, "per_rank": stats}
                f.write(json.dumps(rec) + "\n")
                f.flush()
                print(json.dumps({k: v for k, v in rec.items() if k != "per_rank"}), flush=True)
                del offs, ind
                if mode is not None:
                    h.close()
            del ref, bt
    if not ok:
        sys.exit("parity check FAILED: some arm's offsets or indices differ from the one-GPU BallTree")
    print("parity ok: offsets and indices identical in every arm")


if __name__ == "__main__":
    main()
