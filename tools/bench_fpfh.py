#!/usr/bin/env python
"""Batched FPFH descriptors (row f8, csrc/fpfh.cu): time per call on the two workloads that need descriptors here.

  (a) ModelNet-shaped clouds: synth.make_clouds(256, 1024) with their analytic normals; radius 0.25, max_nn 100 (the
      default of Open3D's compute_fpfh_feature in its global-registration tutorial).
  (b) Subsampled scans: 8 raw synth.make_scan(400000) scans, grid-subsampled at 4.5 cm (as tools/bench_normals.py does)
      and cut to a common N (~50k); radius 5 x 4.5 cm, max_nn 100 (Open3D's tutorial: 5 x the voxel size).
Per workload: ms per call by CUDA events over >= 20 warm calls; estimate_normals (max_nn 30; radius 0.1 for (a), 2 x the
cell for (b) as in Open3D's tutorial) timed the same way on the same clouds; points/s and pair features/s (sum of n - 1 over the
points, from the returned counts); bytes the list stages gather and write, from the shapes and the counts (the ring
search's candidate reads are not counted), and that over the time; the mean list length; the card's name and power limit,
read in the same run.  One JSON line.

    python tools/bench_fpfh.py [--calls 20] [--profile out_dir]

--profile adds a separate torch.profiler run per workload and writes its per-kernel table to out_dir.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ri_b200                                     # noqa: E402
from ri_b200 import synth                          # noqa: E402

CELL = 0.045


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def modelnet():
    c = synth.make_clouds(256, 1024, seed=2024)
    f = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return f(c[:, :3]), f(c[:, 3:]), 0.25, 0.1


def scans(B=8, raw=400000):
    clouds = [torch.from_numpy(np.ascontiguousarray(synth.make_scan(raw, seed=s).T)).cuda() for s in range(B)]
    subs = ri_b200.grid_sub_sampling_many([(r[:, :3].contiguous(), r[:, 3:].contiguous()) for r in clouds], grid_size=CELL)
    n = min(p.shape[0] for p, _, _ in subs)
    xyz = torch.stack([p[:n].t() for p, _, _ in subs]).contiguous()
    nrm = torch.stack([torch.nn.functional.normalize(f[:n], dim=1).t() for _, f, _ in subs]).contiguous()
    return xyz, nrm, 5 * CELL, 2 * CELL


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


def list_bytes(B, N, cnt):
    """Bytes the two list stages move, from the shapes and the list lengths n:
    search + SPFH: q's xyz + normal (24), per list entry its xyz + normal gathered (24) and its index written (4), the packed
    counts written (36); FPFH: q's packed counts and xyz (48), per entry after the first its index, xyz and packed counts
    (4 + 12 + 36), the 33 fp32 outputs (132)."""
    n = cnt.to(torch.float64)
    e = float(n.sum()); e1 = float((n - 1).clamp(min=0).sum())
    return B * N * (24 + 36 + 48 + 132) + e * 28 + e1 * 52


def run(name, data, calls, profile_dir):
    xyz, nrm, r, r_n = data
    B, _, N = xyz.shape
    fp = lambda: ri_b200.functional.compute_fpfh_feature(xyz, nrm, r, 100, return_counts=True)
    ms, (_, cnt) = timed(fp, calls)
    ms_n, _ = timed(lambda: ri_b200.functional.estimate_normals(xyz, r_n, 30), calls)
    pairs = float((cnt.to(torch.float64) - 1).clamp(min=0).sum())
    nbytes = list_bytes(B, N, cnt)
    row = {"workload": name, "clouds": B, "points_per_cloud": N, "radius": r, "max_nn": 100,
           "ms_per_call": ms, "points_per_s": B * N / (ms * 1e-3), "pair_features_per_s": pairs / (ms * 1e-3),
           "mean_list_length": float(cnt.float().mean()), "lists_at_max_nn": float((cnt == 100).float().mean()),
           "list_stage_bytes": nbytes, "list_stage_GB_per_s": nbytes / (ms * 1e-3) / 1e9,
           "estimate_normals_radius": r_n, "estimate_normals_max_nn30_ms": ms_n, "fpfh_over_normals": ms / ms_n}
    if profile_dir:
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                fp()
            torch.cuda.synchronize()
        with open(os.path.join(profile_dir, "fpfh_kernels_%s.txt" % name), "w") as f:
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=20))
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fpfh.py measures the GPU kernels: no CUDA device")
    if a.profile:
        os.makedirs(a.profile, exist_ok=True)
    rows = [run("modelnet_256x1024", modelnet(), a.calls, a.profile), run("scan_8x50k", scans(), a.calls, a.profile)]
    print(json.dumps({"bench": "fpfh", "card": card(), "torch": torch.__version__, "calls_timed": a.calls,
                      "results": rows}))


if __name__ == "__main__":
    main()
