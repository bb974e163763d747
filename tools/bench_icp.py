#!/usr/bin/env python
"""Batched ICP refinement (row f5, csrc/icp.cu): time per call on the two workloads ICP serves here.

  (a) ModelNet-shaped pairs: 256 pairs x 1024 points (synth.make_pairs(256, 1024, seed=2024)), init = GT perturbed by
      <= 5 degrees / <= 5 cm, max_correspondence_distance 0.05 — the refinement step after RANSAC in the registration job.
  (b) Scan pairs: 8 pairs of 50k-point ICL-NUIM-shaped scans (synth.make_scan), target = known SE(3) of the source + 5 mm
      noise, init 3 degrees / 3 cm off, max_correspondence_distance 0.1.
Each workload runs both estimations, with Open3D's default criteria (1e-6 / 1e-6, max 30) and with a fixed 30 iterations
(criteria 0).  Times are CUDA events over >= 20 warm calls.  Beside them: the CPU time per pair of the numpy / scipy oracle
(tests/icp_oracle.py), and the card's name and power limit read in the same run.

    python tools/bench_icp.py [--calls 20] [--profile out_dir]

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
import icp_oracle                                  # noqa: E402
import ri_b200                                     # noqa: E402
from ri_b200 import synth                          # noqa: E402


def pose(rng, deg, trans):
    ax = rng.standard_normal(3); ax /= np.linalg.norm(ax)
    a = np.deg2rad(deg)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    T = np.eye(4); T[:3, :3] = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    v = rng.standard_normal(3); T[:3, 3] = v / np.linalg.norm(v) * trans
    return T


def pose_err(T, G):
    """(degrees, distance); chord form of the rotation angle (no acos amplification of fp32 rounding)."""
    D = T[:3, :3] @ G[:3, :3].T
    return np.degrees(2 * np.arcsin(min(1.0, np.linalg.norm(D - np.eye(3)) / (2 * np.sqrt(2))))), np.linalg.norm(T[:3, 3] - G[:3, 3])


def modelnet(rng):
    src, tgt, R, t = synth.make_pairs(256, 1024, seed=2024)
    P = len(src)
    G = np.tile(np.eye(4), (P, 1, 1)); G[:, :3, :3] = R; G[:, :3, 3] = t
    init = np.stack([pose(rng, rng.uniform(0, 5), rng.uniform(0, 0.05)) @ G[p] for p in range(P)])
    pm = lambda a: np.ascontiguousarray(a.transpose(0, 2, 1))
    return pm(src[:, :3]), pm(tgt[:, :3]), pm(tgt[:, 3:]), G, init, 0.05


def scans(rng, P=8, N=50000):
    src, tgt, nrm, G, init = [], [], [], [], []
    for p in range(P):
        S = synth.make_scan(N, seed=100 + p)
        s = S[:3].T.astype(np.float64)
        g = pose(rng, 10.0, 0.2)
        src.append(s); G.append(g)
        tgt.append(s @ g[:3, :3].T + g[:3, 3] + rng.standard_normal(s.shape) * 0.005)
        nrm.append(S[3:].T @ g[:3, :3].T)
        init.append(pose(rng, 3.0, 0.03) @ g)
    return np.stack(src), np.stack(tgt), np.stack(nrm), np.stack(G), np.stack(init), 0.1


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def run(name, data, calls, profile_dir):
    src, tgt, nrm, G, init, r = data
    P, n1 = src.shape[:2]
    f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()
    s, g, n, i0 = f32(src), f32(tgt), f32(nrm), f32(init)
    rows = []
    for est in ("point_to_point", "point_to_plane"):
        for crit in (1e-6, 0.0):
            call = lambda: ri_b200.registration.icp(s, g, r, init=i0, estimation=est, tgt_normals=n, max_iter=30,
                                                    relative_fitness=crit, relative_rmse=crit)
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
            err0 = np.array([pose_err(init[p], G[p]) for p in range(P)])
            launches = int(it.max()) + 1                         # evaluation launches that did work for some pair
            # CPU oracle: the same algorithm in numpy fp64 + scipy's k-d tree, on a few pairs of the same input
            k = min(P, 4 if n1 < 10000 else 1)
            fn = icp_oracle.icp_point_to_point if est == "point_to_point" else icp_oracle.icp_point_to_plane
            t0 = time.time()
            for p in range(k):
                args = (src[p], tgt[p], r) if est == "point_to_point" else (src[p], tgt[p], nrm[p], r)
                fn(*args, init=init[p], max_iter=30, relative_fitness=crit, relative_rmse=crit)
            cpu_ms = (time.time() - t0) * 1e3 / k
            rows.append({"workload": name, "estimation": est, "criteria": crit, "pairs": P, "n1": n1, "n2": tgt.shape[1],
                         "max_corr_dist": r, "ms_per_call": ms, "pairs_per_s": P / (ms * 1e-3),
                         "us_per_iteration": ms * 1e3 / launches,
                         "queries_per_s": float((it + 1).sum()) * n1 / (ms * 1e-3),
                         "iterations_mean": float(it.mean()), "iterations_max": int(it.max()),
                         "fitness_mean": float(res['fitness'].mean()),
                         "rre_deg_init_mean": float(err0[:, 0].mean()), "rte_init_mean": float(err0[:, 1].mean()),
                         "rre_deg_mean": float(err[:, 0].mean()), "rre_deg_max": float(err[:, 0].max()),
                         "rte_mean": float(err[:, 1].mean()), "rte_max": float(err[:, 1].max()),
                         "cpu_reference_ms_per_pair": cpu_ms})
            if profile_dir and crit == 0.0:
                from torch.profiler import profile, ProfilerActivity
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(5):
                        call()
                    torch.cuda.synchronize()
                with open(os.path.join(profile_dir, "icp_kernels_%s_%s.txt" % (name, est)), "w") as f:
                    f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=20))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_icp.py measures the GPU kernels: no CUDA device")
    if a.profile:
        os.makedirs(a.profile, exist_ok=True)
    rng = np.random.default_rng(0)
    rows = run("modelnet_256x1024", modelnet(rng), a.calls, a.profile) + run("scan_8x50k", scans(rng), a.calls, a.profile)
    print(json.dumps({"bench": "icp", "card": card(), "torch": torch.__version__, "calls_timed": a.calls, "results": rows}))


if __name__ == "__main__":
    main()
