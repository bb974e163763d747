#!/usr/bin/env python
"""Batched farthest point sampling (row f12, csrc/fps.cu): time per call against a torch fp64 loop of the same contract.

  (a) ModelNet-shaped clouds: synth.make_clouds(256, 1024) -> 512 samples (one CTA per cloud).
  (b) Scans: 8 raw synth.make_scan(400000) scans grid-subsampled at 4.5 cm (grid_sub_sampling_many, ragged, ~50k
      points each) -> 4096 samples (8-CTA clusters).
  (c) One scan at the largest N the kernel takes (131072 points, subsampled at 2 cm and cut to that size) -> 4096
      samples (one 16-CTA cluster).
  (d) Per-sample cost by cluster size: one cloud of N = 1024 .. 65536 uniform points -> 2048 samples, the launch picking
      1, 2, 4, 8, 8, 8 CTAs.
The baseline is the contract written as torch fp64 tensor ops, one sample at a time over the whole batch (torch.argmax
returns the first maximum); its indices must equal the kernel's, and the run fails otherwise.  Per workload: ms per call
by CUDA events over >= 10 warm calls (median and min / max of 5 windows), microseconds per sample, the baseline's ms per
call; the card's name and power limit, read in the same run.  One JSON line.

    python tools/bench_fps.py [--calls 10]
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def torch_fps(xyz, lengths, m):
    """The contract in torch fp64: every operation a separate kernel, so nothing is contracted."""
    B, _, N = xyz.shape
    p = xyz.double()
    valid = torch.arange(N, device=xyz.device)[None, :] < lengths.to(xyz.device)[:, None]
    dist = torch.where(valid, torch.full((B, N), float("inf"), dtype=torch.float64, device=xyz.device),
                       torch.zeros((B, N), dtype=torch.float64, device=xyz.device))
    s = torch.zeros(B, dtype=torch.long, device=xyz.device)
    out = torch.empty((B, m), dtype=torch.int32, device=xyz.device)
    ar = torch.arange(B, device=xyz.device)
    for k in range(m):
        out[:, k] = s
        if k == m - 1:
            break
        d = p - p[ar, :, s].unsqueeze(2)
        d = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        dist = torch.where(d < dist, d, dist)
        best, j = dist.max(1), torch.argmax(dist, 1)
        s = torch.where(best.values > 0, j, s)
    out[lengths.to(xyz.device) == 0] = -1
    return out


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
    return float(np.median(wins)), float(min(wins)), float(max(wins))


def padded(clouds):
    lens = [int(c.shape[0]) for c in clouds]
    xyz = torch.zeros((len(clouds), 3, max(lens)), device="cuda")
    for b, c in enumerate(clouds):
        xyz[b, :, :lens[b]] = c.t()
    return xyz, torch.tensor(lens, dtype=torch.int32)


def workloads():
    c = synth.make_clouds(256, 1024, seed=2024)
    yield "a_modelnet_256x1024_m512", torch.from_numpy(np.ascontiguousarray(c[:, :3])).cuda(), torch.full((256,), 1024, dtype=torch.int32), 512
    raw = [torch.from_numpy(np.ascontiguousarray(synth.make_scan(400000, seed=s).T)).cuda() for s in range(8)]
    subs = ri_b200.grid_sub_sampling_many([r[:, :3].contiguous() for r in raw], grid_size=0.045)
    xyz, lens = padded([p for p, _, _ in subs])
    yield "b_scans_8x%d-%d_m4096" % (int(lens.min()), int(lens.max())), xyz, lens, 4096
    big = ri_b200.grid_sub_sampling_many([torch.from_numpy(np.ascontiguousarray(synth.make_scan(1200000, seed=99).T[:, :3])).cuda()],
                                         grid_size=0.02)[0][0]
    assert big.shape[0] >= 131072, big.shape
    xyz, lens = padded([big[:131072]])
    yield "c_scan_1x131072_m4096", xyz, lens, 4096
    rng = np.random.default_rng(1)
    for N in (1024, 2048, 4096, 8192, 16384, 65536):
        xyz = torch.from_numpy(rng.uniform(-1, 1, (1, 3, N)).astype(np.float32)).cuda()
        yield "d_uniform_1x%d_m2048" % N, xyz, torch.tensor([N], dtype=torch.int32), 2048


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    args = ap.parse_args()
    res = {"card": card(), "workloads": {}}
    for name, xyz, lens, m in workloads():
        op = lambda: torch.ops.ri.furthest_point_sample(xyz, lens, m)
        got = op()
        want = torch_fps(xyz, lens, m)
        if not torch.equal(got, want):
            raise SystemExit("%s: kernel and torch baseline differ in %d clouds" % (name, int((got != want).any(1).sum())))
        med, lo, hi = timed(op, args.calls)
        base, _, _ = timed(lambda: torch_fps(xyz, lens, m), 1)
        res["workloads"][name] = {"B": int(xyz.shape[0]), "N": int(xyz.shape[2]), "m": m, "ms_per_call": round(med, 4),
                                  "ms_min": round(lo, 4), "ms_max": round(hi, 4), "us_per_sample": round(1000 * med / m, 3),
                                  "torch_fp64_ms_per_call": round(base, 2), "identical": True}
        print(name, res["workloads"][name], flush=True)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
