#!/usr/bin/env python
"""Batched normal estimation (row f6, csrc/normals.cu): time per call on the two workloads that need normals here.

  (a) ModelNet-shaped clouds: synth.make_clouds(512, 1024), i.e. both clouds of the registration job's 256 pairs;
      radius 0.2, max_nn 30, no orientation.
  (b) Scans: 8 raw synth.make_scan(400000) scans, grid-subsampled at 4.5 cm (grid_sub_sampling_many, the analytic normals
      averaged as features and renormalised, as tools/bench_scan.py does) and cut to a common N (~50k); radius 0.1,
      max_nn 30, camera = the room centre.
Per workload: ms per call by CUDA events over >= 20 warm calls and points/s; knn_indices(xyz, 30) timed the same way on the
same clouds; the mean neighbour count; the mean and 95th-percentile angle to the analytic normals (unsigned); for (b) the
share of normals whose sign disagrees with the analytic normal (which points into the room, towards the camera); the CPU
time per cloud of the numpy / scipy reference (tests/normals_oracle.py) as a yardstick; the card's name and power limit,
read in the same run.  One JSON line.

    python tools/bench_normals.py [--calls 20] [--profile out_dir]

--profile adds a separate torch.profiler run per workload and writes its per-kernel table to out_dir.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import normals_oracle                              # noqa: E402
import ri_b200                                     # noqa: E402
from ri_b200 import synth                          # noqa: E402

ROOM_CENTRE = [2.0, 1.5, 1.25]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def modelnet():
    c = synth.make_clouds(512, 1024, seed=2024)
    f = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return f(c[:, :3]), f(c[:, 3:]), 0.2, None


def scans(B=8, raw=400000, cell=0.045):
    clouds = [torch.from_numpy(np.ascontiguousarray(synth.make_scan(raw, seed=s).T)).cuda() for s in range(B)]
    subs = ri_b200.grid_sub_sampling_many([(r[:, :3].contiguous(), r[:, 3:].contiguous()) for r in clouds], grid_size=cell)
    n = min(p.shape[0] for p, _, _ in subs)
    xyz = torch.stack([p[:n].t() for p, _, _ in subs]).contiguous()
    nrm = torch.stack([torch.nn.functional.normalize(f[:n], dim=1).t() for _, f, _ in subs]).contiguous()
    return xyz, nrm, 0.1, torch.tensor(ROOM_CENTRE, device="cuda")


def timed(fn, calls):
    for _ in range(3):
        out = fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        out = fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls, out


def run(name, data, calls, profile_dir):
    xyz, truth, r, cam = data
    B, _, N = xyz.shape
    est = lambda: ri_b200.functional.estimate_normals(xyz, r, 30, camera=cam, return_counts=True)
    ms, (nrm, cnt) = timed(est, calls)
    ms_knn, _ = timed(lambda: ri_b200.functional.knn_indices(xyz, 30), calls)
    cos = (nrm * truth).sum(1)
    # atan2(|n x t|, |n.t|): no arccos amplification of the fp32 normals' rounding near 0 degrees
    ang = torch.rad2deg(torch.atan2(torch.linalg.cross(nrm, truth, dim=1).norm(dim=1), cos.abs())).flatten().cpu().numpy()
    row = {"workload": name, "clouds": B, "points_per_cloud": N, "radius": r, "max_nn": 30,
           "orientation": "camera at the room centre" if cam is not None else "none",
           "ms_per_call": ms, "points_per_s": B * N / (ms * 1e-3),
           "knn_indices_k30_ms": ms_knn, "normals_over_knn": ms / ms_knn,
           "mean_neighbours": float(cnt.float().mean()),
           "angle_to_analytic_deg_mean": float(ang.mean()), "angle_to_analytic_deg_p95": float(np.percentile(ang, 95)),
           "sign_disagrees_with_analytic": float((cos < 0).float().mean()) if cam is not None else None}
    # CPU yardstick: the numpy / scipy reference on one or two clouds of the same input
    k = 2 if N < 10000 else 1
    x = xyz[:k].cpu().numpy()
    t0 = time.time()
    for b in range(k):
        normals_oracle.estimate_normals(x[b].T, r, 30, camera=None if cam is None else np.asarray(ROOM_CENTRE))
    row["cpu_reference_ms_per_cloud"] = (time.time() - t0) * 1e3 / k
    if profile_dir:
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                est()
                ri_b200.functional.knn_indices(xyz, 30)
            torch.cuda.synchronize()
        with open(os.path.join(profile_dir, "normals_kernels_%s.txt" % name), "w") as f:
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=20))
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_normals.py measures the GPU kernels: no CUDA device")
    if a.profile:
        os.makedirs(a.profile, exist_ok=True)
    rows = [run("modelnet_512x1024", modelnet(), a.calls, a.profile), run("scan_8x50k", scans(), a.calls, a.profile)]
    print(json.dumps({"bench": "normals", "card": card(), "torch": torch.__version__, "calls_timed": a.calls,
                      "results": rows}))


if __name__ == "__main__":
    main()
