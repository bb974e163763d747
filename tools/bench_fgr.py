#!/usr/bin/env python
"""Batched Fast Global Registration (row f7, csrc/fgr.cu): time per call next to RANSAC on the same matches.

  (a) the registration job's shape: 256 pairs x 1024 points (synth.make_pairs(256, 1024, seed=2024)), planted matches
      (point i with its transformed copy) of which 50 % are replaced by random partners.
  (b) scan pairs: 8 pairs of ~20k-point ICL-NUIM-shaped scans (synth.make_scan), target = known SE(3) of the source + 5 mm
      noise, every point matched, 50 % of the matches replaced by random partners.
Both solvers run through estimate_poses with voxel_size 0.08: 'fgr' with Open3D's defaults and
maximum_correspondence_distance 0.04, 'ransac' with 1000 hypotheses.  Times are CUDA events over warm calls.  To place the
time, FGR is also timed with iteration_number 0 (tuple test, normalisation and inlier count only) and without the tuple
test.  Beside the times: RRE / RTE of both against the ground truth, the CPU time per pair of the fp64 replay
(tests/fgr_oracle.py), and the card's name and power limit read in the same run.

    python tools/bench_fgr.py [--calls 20]
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
import fgr_oracle                                  # noqa: E402
import ri_b200                                     # noqa: E402
from ri_b200 import synth                          # noqa: E402

VOXEL = 0.08


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def matches(rng, P, n, outliers):
    idx1 = np.tile(np.arange(n, dtype=np.int32), (P, 1))
    idx2 = idx1.copy()
    bad = rng.random((P, n)) < outliers
    idx2[bad] = rng.integers(0, n, int(bad.sum()))
    return idx1, idx2, np.full(P, n, np.int32)


def modelnet(rng):
    src, tgt, R, t = synth.make_pairs(256, 1024, seed=2024)
    P = len(src)
    G = np.tile(np.eye(4), (P, 1, 1)); G[:, :3, :3] = R; G[:, :3, 3] = t
    pm = lambda a: np.ascontiguousarray(a[:, :3].transpose(0, 2, 1))
    return (pm(src), pm(tgt)) + matches(rng, P, src.shape[2], 0.5) + (G,)


def scans(rng, P=8, N=20000):
    src, tgt, G = [], [], []
    for p in range(P):
        s = synth.make_scan(N, seed=200 + p)[:3].T.astype(np.float64)
        g = np.eye(4); g[:3, :3] = synth.random_rotations(rng, 1)[0]; g[:3, 3] = rng.uniform(-0.5, 0.5, 3)
        src.append(s); G.append(g)
        tgt.append(s @ g[:3, :3].T + g[:3, 3] + rng.standard_normal(s.shape) * 0.005)
    f = lambda x: np.ascontiguousarray(np.stack(x), dtype=np.float32)
    return (f(src), f(tgt)) + matches(rng, P, N, 0.5) + (np.stack(G),)


def errors(T, G):
    """(RRE degrees, RTE) per pair; chord form of the rotation angle."""
    D = np.einsum('pij,pkj->pik', T[:, :3, :3], G[:, :3, :3])
    rre = np.degrees(2 * np.arcsin(np.minimum(1.0, np.linalg.norm(D - np.eye(3), axis=(1, 2)) / (2 * np.sqrt(2)))))
    return rre, np.linalg.norm(T[:, :3, 3] - G[:, :3, 3], axis=1)


def timed(call, calls):
    for _ in range(3):
        out = call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        out = call()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls, out


def run(name, data, calls):
    src, tgt, idx1, idx2, count, G = data
    P, n = src.shape[:2]
    d = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (src, tgt, idx1, idx2, count)]
    reg = ri_b200.registration
    row = {"workload": name, "pairs": P, "points": n, "matches_per_pair": int(count[0]), "outliers": 0.5}
    for func in ("fgr", "ransac"):
        ms, (T, inl) = timed(lambda: reg.estimate_poses(*d, func=func, voxel_size=VOXEL, max_iter=1000, seed=1), calls)
        rre, rte = errors(T.cpu().numpy().astype(np.float64), G)
        row[func] = {"ms_per_call": ms, "us_per_pair": ms * 1e3 / P, "rre_deg_mean": float(rre.mean()),
                     "rre_deg_max": float(rre.max()), "rte_mean": float(rte.mean()), "rte_max": float(rte.max()),
                     "inliers_mean": float(inl.float().mean())}
    fgr = lambda **kw: reg.fgr(*d, maximum_correspondence_distance=0.5 * VOXEL, inlier_dist=VOXEL, seed=1, **kw)
    row["fgr"]["ms_iterations_0"] = timed(lambda: fgr(iteration_number=0), calls)[0]
    ms, r = timed(lambda: fgr(tuple_test=False), calls)
    row["fgr"]["ms_no_tuple_test"] = ms
    row["fgr"]["num_correspondences_mean"] = float(fgr()['num_correspondences'].float().mean())
    k = min(P, 4)
    t0 = time.time()
    for p in range(k):
        m = int(count[p])
        fgr_oracle.replay(src[p], tgt[p], src[p][idx1[p, :m]], tgt[p][idx2[p, :m]], seed=1, pair=p,
                          max_corr_dist=0.5 * VOXEL, inlier_dist=VOXEL)
    row["fgr"]["cpu_replay_ms_per_pair"] = (time.time() - t0) * 1e3 / k
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fgr.py measures the GPU kernels: no CUDA device")
    rng = np.random.default_rng(0)
    rows = [run("modelnet_256x1024", modelnet(rng), a.calls), run("scan_8x20k", scans(rng), a.calls)]
    print(json.dumps({"bench": "fgr", "card": card(), "torch": torch.__version__, "calls_timed": a.calls, "results": rows}))


if __name__ == "__main__":
    main()
