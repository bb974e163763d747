#!/usr/bin/env python
"""Batched generalized ICP (row f9, csrc/icp.cu) beside point-to-point and point-to-plane ICP (row f5), on the two workloads
of tools/bench_icp.py with the same seeds and inputs:

  (a) ModelNet-shaped pairs: 256 pairs x 1024 points (synth.make_pairs(256, 1024, seed=2024)), init = GT perturbed by
      <= 5 degrees / <= 5 cm, max_correspondence_distance 0.05.
  (b) Scan pairs: 8 pairs of 50k-point ICL-NUIM-shaped scans (synth.make_scan), target = known SE(3) of the source + 5 mm
      noise, init 3 degrees / 3 cm off, max_correspondence_distance 0.1.
Methods: point_to_point, point_to_plane (target normals given), gicp (both clouds' normals given, epsilon 1e-3) and
gicp_xyz (no normals: the call estimates them from 20 neighbours, and that time is included).  Each runs with Open3D's
default criteria (1e-6 / 1e-6, max 30) and with a fixed 30 iterations (criteria 0).  Times are CUDA events over >= 20 warm
calls.  Beside them: the CPU time per pair of the numpy / scipy references (tests/icp_oracle.py, tests/gicp_oracle.py; for
gicp_xyz Open3D's no-normals path, covariances included), and the card's name and power limit read in the same run.

    python tools/bench_gicp.py [--calls 20] [--profile out_dir]

--profile adds a separate torch.profiler run of the fixed-iteration GICP calls per workload and writes the per-kernel table
to out_dir.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gicp_oracle                                 # noqa: E402
import icp_oracle                                  # noqa: E402
import ri_b200                                     # noqa: E402
from bench_icp import card, modelnet, pose_err, scans   # noqa: E402

METHODS = ("point_to_point", "point_to_plane", "gicp", "gicp_xyz")


def oracle(method, src, tgt, ns, nt, r, init, crit):
    kw = dict(init=init, max_iter=30, relative_fitness=crit, relative_rmse=crit)
    if method == "point_to_point":
        return icp_oracle.icp_point_to_point(src, tgt, r, **kw)
    if method == "point_to_plane":
        return icp_oracle.icp_point_to_plane(src, tgt, nt, r, **kw)
    if method == "gicp":
        return gicp_oracle.generalized_icp_normals(src, tgt, ns, nt, r, 1e-3, **kw)
    return gicp_oracle.generalized_icp(src, tgt, r, gicp_oracle.covariances_open3d_knn(src, 1e-3),
                                       gicp_oracle.covariances_open3d_knn(tgt, 1e-3), **kw)


def run(name, data, calls, profile_dir):
    src, tgt, nt, G, init, r = data
    ns = np.einsum('pni,pij->pnj', nt.astype(np.float64), G[:, :3, :3])   # source normals: the target's, rotated back
    P, n1 = src.shape[:2]
    f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()
    s, g, a, b, i0 = f32(src), f32(tgt), f32(ns), f32(nt), f32(init)
    reg = ri_b200.registration
    rows = []
    for method in METHODS:
        for crit in (1e-6, 0.0):
            kw = dict(init=i0, max_iter=30, relative_fitness=crit, relative_rmse=crit)
            if method in ("point_to_point", "point_to_plane"):
                call = lambda: reg.icp(s, g, r, estimation=method, tgt_normals=b, **kw)
            elif method == "gicp":
                call = lambda: reg.generalized_icp(s, g, r, src_normals=a, tgt_normals=b, **kw)
            else:
                call = lambda: reg.generalized_icp(s, g, r, **kw)
            for _ in range(3):
                res = call()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(calls):
                res = call()
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / calls
            it = res['iterations'].cpu().numpy()
            T = res['transformation'].cpu().numpy().astype(np.float64)
            err = np.array([pose_err(T[p], G[p]) for p in range(P)])
            launches = int(it.max()) + 1                         # evaluation launches that did work for some pair
            row = {"workload": name, "method": method, "criteria": crit, "pairs": P, "n1": n1, "n2": tgt.shape[1],
                   "max_corr_dist": r, "ms_per_call": ms, "us_per_iteration": ms * 1e3 / launches,
                   "iterations_mean": float(it.mean()), "iterations_max": int(it.max()),
                   "fitness_mean": float(res['fitness'].mean()),
                   "rre_deg_mean": float(err[:, 0].mean()), "rre_deg_max": float(err[:, 0].max()),
                   "rte_mean": float(err[:, 1].mean()), "rte_max": float(err[:, 1].max())}
            if crit == 1e-6:                                     # the CPU reference, on a few pairs of the same input
                k = min(P, 4 if n1 < 10000 else 1)
                t0 = time.time()
                for p in range(k):
                    oracle(method, src[p], tgt[p], ns[p], nt[p], r, init[p], crit)
                row["cpu_reference_ms_per_pair"] = (time.time() - t0) * 1e3 / k
            rows.append(row)
            if profile_dir and crit == 0.0 and method.startswith("gicp"):
                from torch.profiler import profile, ProfilerActivity
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(5):
                        call()
                    torch.cuda.synchronize()
                with open(os.path.join(profile_dir, "gicp_kernels_%s_%s.txt" % (name, method)), "w") as f:
                    f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=20))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_gicp.py measures the GPU kernels: no CUDA device")
    if a.profile:
        os.makedirs(a.profile, exist_ok=True)
    rng = np.random.default_rng(0)
    rows = run("modelnet_256x1024", modelnet(rng), a.calls, a.profile) + run("scan_8x50k", scans(rng), a.calls, a.profile)
    print(json.dumps({"bench": "gicp", "card": card(), "torch": torch.__version__, "calls_timed": a.calls,
                      "profiled": bool(a.profile), "results": rows}))


if __name__ == "__main__":
    main()
