#!/usr/bin/env python
"""Batched ISS keypoints (row f13, csrc/iss.cu): time per call, keypoints per cloud, and what matching on keypoints instead
of every point does to the mutual matches and to the matcher / RANSAC time.

  (a) ModelNet-shaped pairs: synth.make_pairs(128, 1024) -> 256 clouds x 1024 points, automatic radii.
  (b) Scans: 8 synth.make_scan(50000) scans, explicit radii (0.1 m, 0.07 m).
  (c) Scans -> grid_sub_sampling_many(0.05) -> farthest_point_batch(4096) -> ISS (automatic radii); 4 pairs, the target a
      random rigid motion of the source scan plus 5 mm noise, each subsampled on its own.
For (a) and (c) both clouds of each pair get normals and FPFH on all their points; the mutual matches (matcher.mutual_nn)
are taken once over all points and once over the keypoints (functional.keypoint_batch), and each set gets its count, its
inlier ratio under the ground truth (|R a + t - b| < tau) and the time of the matcher and of RANSAC (1000 hypotheses).
Times by CUDA events over warm calls (median of 5 windows).  One scipy-oracle run (tests/iss_oracle.py) is timed for scale.
The card's name and power limit are read in the same run.  One JSON line at the end.

    python tools/bench_iss.py [--calls 10]
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
import ri_b200                                     # noqa: E402
from ri_b200 import synth                          # noqa: E402
import iss_oracle                                  # noqa: E402

F = ri_b200.functional


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn, calls):
    fn()
    torch.cuda.synchronize()
    wins = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            fn()
        b.record()
        torch.cuda.synchronize()
        wins.append(a.elapsed_time(b) / calls)
    return float(np.median(wins))


def kp_stats(count):
    c = count.cpu().numpy()
    return {"min": int(c.min()), "mean": round(float(c.mean()), 1), "max": int(c.max())}


def match_report(src_cm, tgt_cm, R, t, r_n, r_f, tau, calls):
    """src_cm / tgt_cm [P,3,N] pairs, R [P,3,3], t [P,3] (src -> tgt) -> matching on all points vs on ISS keypoints."""
    fs = F.compute_fpfh_feature(src_cm, F.estimate_normals(src_cm, r_n, 30), r_f, 100)
    ft = F.compute_fpfh_feature(tgt_cm, F.estimate_normals(tgt_cm, r_n, 30), r_f, 100)
    ks, cs = F.compute_iss_keypoints(src_cm)
    kt, ct = F.compute_iss_keypoints(tgt_cm)
    Rt = torch.as_tensor(R, dtype=torch.float32, device="cuda")
    tt = torch.as_tensor(t, dtype=torch.float32, device="cuda")
    out = {}
    for name in ("all_points", "keypoints"):
        if name == "all_points":
            ps, pt = src_cm.transpose(1, 2).contiguous(), tgt_cm.transpose(1, 2).contiguous()
            a, b = fs.transpose(1, 2).contiguous(), ft.transpose(1, 2).contiguous()
            rows = [ps.shape[1]] * len(ps)
        else:
            ps, a, _ = F.keypoint_batch(src_cm, ks, cs, fs)
            pt, b, _ = F.keypoint_batch(tgt_cm, kt, ct, ft)
            rows = cs.tolist()
        m = ri_b200.matcher.mutual_nn(a, b, point_major=True, want_dist=False)
        t_match = timed(lambda: ri_b200.matcher.mutual_nn(a, b, point_major=True, want_dist=False), calls)
        t_ransac = timed(lambda: ri_b200.registration.estimate_poses(ps, pt, m['idx1'], m['idx2'], m['count'],
                                                                     func='ransac', voxel_size=tau), max(1, calls // 5))
        cnt = m['count'].cpu().numpy()
        inl, tot = 0, 0
        for p in range(len(ps)):
            k = int(cnt[p])
            i1, i2 = m['idx1'][p, :k].long(), m['idx2'][p, :k].long()
            d = (ps[p, i1] @ Rt[p].T + tt[p] - pt[p, i2]).norm(dim=1)
            inl += int((d < tau).sum()); tot += k
        out[name] = {"rows_mean": round(float(np.mean(rows)), 1), "matches_mean": round(float(cnt.mean()), 1),
                     "inlier_ratio": round(inl / max(tot, 1), 4), "matcher_ms": round(t_match, 4),
                     "ransac_ms": round(t_ransac, 3)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    args = ap.parse_args()
    res = {"card": card(), "workloads": {}}

    # (a)
    src, tgt, R, t = synth.make_pairs(128, 1024, seed=2024)
    xyz = torch.from_numpy(np.ascontiguousarray(np.concatenate([src[:, :3], tgt[:, :3]]))).cuda()
    idx, cnt = F.compute_iss_keypoints(xyz)
    ms = timed(lambda: F.compute_iss_keypoints(xyz), args.calls)
    w = {"B": 256, "N": 1024, "radii": "auto", "ms_per_call": round(ms, 4), "keypoints": kp_stats(cnt)}
    w["matching"] = match_report(xyz[:128], xyz[128:], R, t, 0.15, 0.3, 0.05, args.calls)
    res["workloads"]["a_modelnet_256x1024_auto"] = w
    print("a", w, flush=True)

    # (b)
    scans = np.stack([synth.make_scan(50000, seed=s)[:3] for s in range(8)])
    xs = torch.from_numpy(scans).cuda()
    idx, cnt = F.compute_iss_keypoints(xs, 0.1, 0.07)
    ms = timed(lambda: F.compute_iss_keypoints(xs, 0.1, 0.07), args.calls)
    w = {"B": 8, "N": 50000, "radii": [0.1, 0.07], "ms_per_call": round(ms, 4), "keypoints": kp_stats(cnt)}
    res["workloads"]["b_scans_8x50000_explicit"] = w
    print("b", w, flush=True)

    # (c)
    rng = np.random.default_rng(7)
    Rc = synth.random_rotations(rng, 4)
    tc = rng.uniform(-1, 1, (4, 3))
    raw = [torch.from_numpy(scans[s].T.copy()).cuda() for s in range(4)]
    raw += [torch.from_numpy((scans[s].T.astype(np.float64) @ Rc[s].T + tc[s] +
                              rng.standard_normal((50000, 3)) * 0.005).astype(np.float32)).cuda() for s in range(4)]
    subs = ri_b200.grid_sub_sampling_many(raw, grid_size=0.05)
    pts, _, _ = ri_b200.farthest_point_batch(subs, 4096)
    xc = pts.transpose(1, 2).contiguous()
    idx, cnt = F.compute_iss_keypoints(xc)
    ms = timed(lambda: F.compute_iss_keypoints(xc), args.calls)
    w = {"B": 8, "N": 4096, "radii": "auto", "ms_per_call": round(ms, 4), "keypoints": kp_stats(cnt)}
    w["matching"] = match_report(xc[:4], xc[4:], Rc, tc, 0.15, 0.4, 0.1, args.calls)
    res["workloads"]["c_scans_gridsub_fps_8x4096_auto"] = w
    print("c", w, flush=True)

    # the scipy oracle, for scale
    t0 = time.perf_counter(); iss_oracle.iss(src[0, :3].T.copy()); t1 = time.perf_counter()
    iss_oracle.iss(scans[0].T.copy(), 0.1, 0.07); t2 = time.perf_counter()
    res["scipy_oracle_ms"] = {"one_1024_cloud_auto": round(1000 * (t1 - t0), 1), "one_50000_scan_explicit": round(1000 * (t2 - t1), 1)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
