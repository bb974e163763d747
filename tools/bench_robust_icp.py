#!/usr/bin/env python
"""Robust kernels for batched point-to-plane and generalized ICP (row f11, csrc/icp.cu) on the two workloads of
tools/bench_icp.py (same seeds and inputs) and their outlier variants:

  modelnet_256x1024  256 ModelNet-shaped pairs x 1024 points, jitter sigma 1 cm, max_correspondence_distance 0.05.
  scan_8x50k         8 pairs of 50k-point scans (synth.make_scan), 5 mm noise, max_correspondence_distance 0.1.
  *_moved            the same, with the 30 % of each target's points nearest a random target point moved by r / 2 in a
                     random direction (the moved-furniture fixture of tests/test_robust_icp_oracle.py, applied per pair).
Methods: point_to_plane and gicp (both clouds' normals given, epsilon 1e-3), each with None (the plain estimator) and the
kernels l1, huber, cauchy, gm, tukey.  k follows from the workload's noise sigma: huber and cauchy sigma, gm sigma^2, tukey
4.685 sigma (the usual 95 %-efficiency constants); for gicp in whitened units, sigma / sqrt(2 epsilon) (the noise along a
shared normal).  Open3D's default criteria (1e-6 / 1e-6, max 30).  Times are CUDA events over >= 10 warm calls; the
card's name and power limit are read in the same run.

    python tools/bench_robust_icp.py [--calls 10] [--profile out_dir]

--profile runs only a torch.profiler pass (5 calls of each estimator, plain and tukey, per workload) and writes the
per-kernel tables to out_dir; take times from a run without it.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import ri_b200                                     # noqa: E402
from bench_icp import card, modelnet, pose_err, scans   # noqa: E402

EPS = 1e-3
KERNELS = (None, 'l1', 'huber', 'cauchy', 'gm', 'tukey')


def kernel_spec(name, sigma, gicp):
    if name is None or name == 'l1':
        return name
    s = sigma / np.sqrt(2 * EPS) if gicp else sigma
    return (name, {'huber': s, 'cauchy': s, 'gm': s * s, 'tukey': 4.685 * s}[name])


def moved(data, seed):
    """The outlier variant: per pair, the 30 % of target points nearest a random target point moved by r / 2."""
    src, tgt, nt, G, init, r = data
    rng = np.random.default_rng(seed)
    tgt = tgt.copy()
    for p in range(len(tgt)):
        c = tgt[p, rng.integers(tgt.shape[1])]
        idx = np.argsort(np.linalg.norm(tgt[p] - c, axis=1))[: int(0.3 * tgt.shape[1])]
        v = rng.standard_normal(3)
        tgt[p, idx] += v / np.linalg.norm(v) * 0.5 * r
    return src, tgt, nt, G, init, r


def workloads():
    rng = np.random.default_rng(0)
    mn, sc = modelnet(rng), scans(rng)
    return [("modelnet_256x1024", mn, 0.01), ("scan_8x50k", sc, 0.005),
            ("modelnet_256x1024_moved", moved(mn, 1), 0.01), ("scan_8x50k_moved", moved(sc, 2), 0.005)]


def calls_for(data):
    src, tgt, nt, G, init, r = data
    ns = np.einsum('pni,pij->pnj', nt.astype(np.float64), G[:, :3, :3])   # source normals: the target's, rotated back
    f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()
    s, g, a, b, i0 = f32(src), f32(tgt), f32(ns), f32(nt), f32(init)
    reg = ri_b200.registration

    def make(method, kernel):
        if method == "point_to_plane":
            return lambda: reg.icp(s, g, r, init=i0, estimation=method, tgt_normals=b, kernel=kernel)
        return lambda: reg.generalized_icp(s, g, r, init=i0, epsilon=EPS, src_normals=a, tgt_normals=b, kernel=kernel)
    return make


def run(name, data, sigma, calls):
    G = data[3]
    P = len(G)
    make = calls_for(data)
    rows = []
    for method in ("point_to_plane", "gicp"):
        for kname in KERNELS:
            spec = kernel_spec(kname, sigma, method == "gicp")
            call = make(method, spec)
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
            launches = int(it.max()) + 1                 # evaluation launches that did work for some pair
            rows.append({"workload": name, "method": method, "kernel": spec if spec is None or isinstance(spec, str)
                         else [spec[0], float(spec[1])], "pairs": P, "n1": int(data[0].shape[1]),
                         "max_corr_dist": data[5], "ms_per_call": ms, "us_per_iteration": ms * 1e3 / launches,
                         "iterations_mean": float(it.mean()), "iterations_max": int(it.max()),
                         "fitness_mean": float(res['fitness'].mean()),
                         "rre_deg_mean": float(err[:, 0].mean()), "rre_deg_max": float(err[:, 0].max()),
                         "rte_mean": float(err[:, 1].mean()), "rte_max": float(err[:, 1].max()),
                         "pairs_rre_over_1deg": int((err[:, 0] > 1.0).sum())})
    return rows


def profile(out_dir):
    from torch.profiler import profile as prof_ctx, ProfilerActivity
    for name, data, sigma in workloads():
        make = calls_for(data)
        for method in ("point_to_plane", "gicp"):
            for kname in (None, 'tukey'):
                call = make(method, kernel_spec(kname, sigma, method == "gicp"))
                call(); torch.cuda.synchronize()
                with prof_ctx(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(5):
                        call()
                    torch.cuda.synchronize()
                fn = "robust_icp_kernels_%s_%s_%s.txt" % (name, method, kname or "plain")
                with open(os.path.join(out_dir, fn), "w") as f:
                    f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=12))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_robust_icp.py measures the GPU kernels: no CUDA device")
    if a.profile:
        os.makedirs(a.profile, exist_ok=True)
        profile(a.profile)
        return
    rows = []
    for name, data, sigma in workloads():
        rows += run(name, data, sigma, a.calls)
    print(json.dumps({"bench": "robust_icp", "card": card(), "torch": torch.__version__, "calls_timed": a.calls,
                      "epsilon": EPS, "results": rows}))


if __name__ == "__main__":
    main()
