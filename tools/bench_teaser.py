#!/usr/bin/env python
"""Batched TEASER++ (row f10, csrc/teaser.cu): time per call next to RANSAC and FGR on the same matches.

Workloads are those of tools/bench_fgr.py, at 50 % and 95 % outlier matches:
  (a) 256 pairs x 1024 points (synth.make_pairs(256, 1024, seed=2024): 0.01 jitter per axis, clipped at 0.05), planted
      matches, noise_bound 0.05 (a match's noise exceeds it for about 2e-5 of the matches);
  (b) 8 pairs of ~20k-point ICL-NUIM-shaped scans, target = known SE(3) of the source + 5 mm noise per axis, every point
      matched, noise_bound 0.025 (5 sigma per axis).
--noise-scale multiplies both bounds, to show what an under-estimated bound costs the clique search.
All solvers run through estimate_poses with voxel_size 0.08 ('ransac' with 1000 hypotheses).  Times are CUDA events over
warm calls; the split into graph (graph, rank and permute kernels), clique and solve comes from torch.profiler in a run of
its own.  Beside the times: RRE / RTE of every solver against the ground truth, TEASER++'s clique sizes and the count of
pairs whose clique search ran out of its budget (exact = 0), and the card's name and power limit read in the same run.

    python tools/bench_teaser.py [--calls 5] [--max-clique-nodes N] [--noise-scale S]
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
from bench_fgr import VOXEL, card, errors, modelnet, scans, timed   # noqa: E402


def with_outliers(data, rng, outliers):
    """Re-draw the match partners of a bench_fgr workload at another outlier rate."""
    src, tgt, idx1, idx2, count, G = data
    P, n = idx1.shape
    idx2 = idx1.copy()
    bad = rng.random((P, n)) < outliers
    idx2[bad] = rng.integers(0, n, int(bad.sum()))
    return src, tgt, idx1, idx2, count, G


def split(call):
    """Device time per kernel group of one call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    call(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call(); torch.cuda.synchronize()
    out = {"graph": 0.0, "clique": 0.0, "solve": 0.0}
    for e in prof.key_averages():
        for k, names in (("graph", ("graph_kernel", "rank_kernel", "permute_kernel")), ("clique", ("clique_kernel",)),
                         ("solve", ("solve_kernel",))):
            if any(n in e.key for n in names):
                out[k] += e.device_time_total / 1e3
    return {k + "_ms": v for k, v in out.items()}


def run(name, data, noise_bound, outliers, calls, max_nodes):
    src, tgt, idx1, idx2, count, G = data
    P, n = src.shape[:2]
    d = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (src, tgt, idx1, idx2, count)]
    reg = ri_b200.registration
    row = {"workload": name, "pairs": P, "points": n, "matches_per_pair": int(count[0]), "outliers": outliers,
           "noise_bound": noise_bound}
    for func in ("teaserpp", "fgr", "ransac"):
        kw = {"noise_bound": noise_bound} if func == "teaserpp" else {}
        ms, (T, inl) = timed(lambda: reg.estimate_poses(*d, func=func, voxel_size=VOXEL, max_iter=1000, seed=1, **kw),
                             calls)
        rre, rte = errors(T.cpu().numpy().astype(np.float64), G)
        row[func] = {"ms_per_call": ms, "us_per_pair": ms * 1e3 / P, "rre_deg_mean": float(rre.mean()),
                     "rre_deg_max": float(rre.max()), "rte_mean": float(rte.mean()), "rte_max": float(rte.max()),
                     "inliers_mean": float(inl.float().mean())}
    one = lambda: reg.teaser(*d, noise_bound, inlier_dist=VOXEL, max_clique_nodes=max_nodes)
    r = one()
    size = r['clique_size'].cpu().numpy()
    row["teaserpp"].update(split(one))
    row["teaserpp"].update({"max_clique_nodes": max_nodes, "clique_size_min": int(size.min()),
                            "clique_size_mean": float(size.mean()), "clique_size_max": int(size.max()),
                            "pairs_not_exact": int((~r['clique_exact']).sum())})
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--max-clique-nodes", type=int, default=ri_b200.registration.MAX_CLIQUE_NODES)
    ap.add_argument("--noise-scale", type=float, default=1.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_teaser.py measures the GPU kernels: no CUDA device")
    rng = np.random.default_rng(0)
    mn, sc = modelnet(rng), scans(rng)
    rows = []
    for outliers in (0.5, 0.95):
        rows.append(run("modelnet_256x1024", with_outliers(mn, rng, outliers), 0.05 * a.noise_scale, outliers, a.calls,
                        a.max_clique_nodes))
        print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
        rows.append(run("scan_8x20k", with_outliers(sc, rng, outliers), 0.025 * a.noise_scale, outliers, a.calls,
                        a.max_clique_nodes))
        print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
    print(json.dumps({"bench": "teaser", "card": card(), "torch": torch.__version__, "calls_timed": a.calls,
                      "results": rows}))


if __name__ == "__main__":
    main()
