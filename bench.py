#!/usr/bin/env python
"""bench.py — feature-extractor front-end throughput (points/sec on 1024-point clouds) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload sph_dg|cu_dg|...] [--impl ours|reference] [--only]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

A "step" is one pass of the front end (SURVEY.md §8 rows a1-a10: k-NN -> fused gather+PPF; coordinate prologue ->
voxelize -> trilinear devoxelize -> DGCNN voxel-neighbour edge features) over one batch of 32 synthetic
ModelNet40-shaped clouds of 1024 points PER GPU (weak scaling: clouds are sharded by rank, no data-path collective; at
N > 1 every step's per-point voxel indices are all-gathered over NCCL inside the timed region — the result gather).

The line's own numbers are BASELINE.json configs[0] (sph_dg: spherical voxelization r = 32, C = 67 — the configuration the
north-star target is stated on).  The other BASELINE configurations are measured in the same run and reported under
`also`: configs[1] cu_dg, configs[4] the spherical resolution sweep r = 16 / 64, configs[2] the registration job
(front end on both clouds of a pair -> fixed random MLP -> tcgen05 mutual-NN matcher -> RANSAC -> metrics).

Every timed region runs exactly K = --steps steps between one pair of CUDA events (after a few untimed warm-up steps) and
`ms_per_step` is their mean; `timed_steps` = K.

`--dump-outputs DIR` writes what the headline's last timed step computed, the engine's output buffers a caller reads (ppf
[B,4,k,N], devox [B,C,N], edge [B,2C,N] in float32; the voxel indices ind [B,N] as float64), to DIR/<name>.npy.  Inputs
are seeded, so two builds run with the same arguments can be compared output for output.  bench_outputs/ in the repository
is git-ignored for this purpose.

Keys beyond the base contract:
  roofline      dominant HBM kernel (vox_fill: the dense [C, r^3] grid + count grid written exactly once), algorithmic
                bytes per launch / CUDA-event duration measured live, against MEASURED_PEAKS.json's HBM GB/s; the whole
                voxelize op, the devoxelizer and the whole step are quoted beside it
  cpu_baseline  the C oracle port (oracle/ri_oracle.c, OpenMP over clouds) timed on this box's host cores on a
                bounded sample of the same workload (rank 0, N=1 only)
  e2e           the same metric through the host-facing streaming call FrontEndPipeline.submit()/result(): every step
                copies its inputs pinned host -> device and its per-point outputs device -> pinned host; the copies of
                neighbouring steps overlap the compute (wall clock incl. the final drain)
`--impl reference` times the UNMODIFIED reference kernels (oracle/_ref, the reference's own CUDA backend recompiled
for sm_100a — the reference has no CPU implementation: every op CHECK_CUDAs) through the reference's op sequence on
the same workload with the same host<->device copies, one rank per GPU like the other arm; if that library is absent
it times the oracle port on the host.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "point-cloud-registration-based-on-rotation-invariant-feature_b200")
sys.path.insert(0, ROOT)

METRIC = "feature-extractor points/sec (1024-pt clouds)"
UNIT = "points/s"
WORKLOADS = {
    # BASELINE.json configs[0]: sph_dg classification front end; C = 3 + 64 channels into PVConv-1
    "sph_dg": dict(voxel_shape="spherical", B=32, N=1024, C=67, k=20, r=32,
                   name="sph_dg front end: 32 x 1024 pts with normals, k=20 KNN+PPF, spherical voxelize r=32 C=67, "
                        "spherical trilinear devox, DGCNN edge gather (BASELINE configs[0])"),
    # BASELINE.json configs[1]: cu_dg variant (cube voxelization + DGCNN), 32 x 1024 on 1 B200; C = 3 + 4 + 64
    "cu_dg": dict(voxel_shape="cube", B=32, N=1024, C=71, k=20, r=32,
                  name="cu_dg front end: 32 x 1024 pts with normals, k=20 KNN+PPF, cube voxelize r=32 C=71, "
                       "trilinear devox, DGCNN edge gather (BASELINE configs[1])"),
}
# BASELINE.json configs[4]: throughput sweep over the spherical resolution (4096 clouds x 1024 pts = 128 steps of 32 clouds)
for _r in (16, 64):
    WORKLOADS["sph_r%d" % _r] = dict(voxel_shape="spherical", B=32, N=1024, C=67, k=20, r=_r,
                                     name="sph_dg front end at spherical res %d: 32 x 1024 pts per step, k=20 KNN+PPF, C=67 "
                                          "(BASELINE configs[4] sweep)" % _r)
RING = 3            # independent input/output buffer sets cycled between timed steps (footprint > L2)
LANES = 2           # steps in flight (tools/tune_lanes.py: cu_dg 140 / 149 / 149 us per step with 2 / 3 / 4 in flight, sph_dg 121 throughout)
E2E_DEPTH = 4       # slots of the host-facing pipeline (tools/exp_e2e.py: 2 / 3 / 4 / 6 slots -> 0.578 / 0.579 / 0.547 / 0.552 ms per step)


def config_for(wl, world):
    """The `config` object: identical in both arms."""
    return {"workload": wl["name"], "clouds_per_gpu": wl["B"], "points_per_cloud": wl["N"], "k": wl["k"],
            "resolution": wl["r"], "channels": wl["C"], "voxel_shape": wl["voxel_shape"],
            "parallelism": "clouds sharded by rank (dp%d)" % world,
            "l2": "inputs larger than L2: %d independent batches cycled" % RING}


def load_by_path(name, filename):
    """Import one module of the package by file path (the reference arm must not load libri_b200.so)."""
    spec = importlib.util.spec_from_file_location(name, os.path.join(PKG, filename))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the benchmark runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.samples = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 6:
                try:
                    self.samples.append((time.time(), float(f[0]), float(f[1]), f[2:6]))
                except ValueError:
                    pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()

    def summary(self, windows):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "nvidia-smi unavailable"}
        inside = [s for s in self.samples if any(a <= s[0] <= b for a, b in windows)]
        note = "sampled inside the timed regions"
        if not inside:
            inside, note = self.samples, "no sample fell inside a timed region: whole-run samples"
        mhz = sorted(s[1] for s in inside)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in inside for n, v in zip(names, s[3]) if v.lower().startswith("active")})
        return {"sm_mhz": mhz[len(mhz) // 2], "sm_max_mhz": inside[0][2], "reasons": reasons,
                "samples": len(inside), "note": note}


def traffic_from_profile(key):
    """dram bytes per launch from the committed ncu capture (profiles/traffic.json), if one exists (else null)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(key)
    except Exception:
        return None


# ===================================================================================================== ours
class Harness:
    """Barrier + CUDA events + max over ranks around a callable that enqueues `steps` steps."""

    def __init__(self, torch, shard, dev, world):
        self.torch, self.shard, self.dev, self.world = torch, shard, dev, world
        self.windows = []

    def barrier(self):
        if self.world > 1:
            self.torch.distributed.barrier()

    def timed(self, body, steps, probe=3):
        """body(n) enqueues n steps.  Runs `probe` untimed steps, then times `steps` steps: returns (ms per step, steps)."""
        torch = self.torch
        def once(n):
            self.barrier(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.time()
            e0.record()
            body(n)
            e1.record()
            torch.cuda.synchronize(); self.barrier()
            return self.shard.max_over_ranks(e0.elapsed_time(e1), self.dev), (t0, time.time())
        once(max(probe, 1))
        ms, w = once(steps)
        self.windows.append(w)
        return ms / steps, steps


def measure_workload(key, args, ri_b200, H, rank, world, local, headline):
    import numpy as np
    torch = H.torch
    synth, shard = ri_b200.synth, ri_b200.shard
    wl = WORKLOADS[key]
    B, N, C, k, r = wl["B"], wl["N"], wl["C"], wl["k"], wl["r"]
    dev = H.dev
    engines, batches = [], []
    for q in range(RING):
        pts = synth.make_clouds(B, N, seed=1000 + 17 * rank + q)
        feats = synth.make_features(B, C, N, seed=1000 + 17 * rank + q)
        fe = ri_b200.FrontEnd(B, N, C, k=k, r=r, voxel_shape=wl["voxel_shape"], normalize=False, device=dev,
                              fuse_mean=args.fuse_mean_in_flight)
        fe.h_points.copy_(torch.from_numpy(pts)); fe.h_features.copy_(torch.from_numpy(feats))
        fe.load(fe.h_points, fe.h_features)
        engines.append(fe); batches.append((pts, feats))
    torch.cuda.synchronize()
    for i in range(max(args.warmup, RING)):
        engines[i % RING].forward()
    torch.cuda.synchronize()

    # ---- one step at a time (latency configuration: the mean fused into the prefix kernel)
    serial = []
    for q in range(RING):
        fe = ri_b200.FrontEnd(B, N, C, k=k, r=r, voxel_shape=wl["voxel_shape"], normalize=False, device=dev)
        fe.load(engines[q].h_points, engines[q].h_features); fe.forward(); serial.append(fe)
    torch.cuda.synchronize()
    ms_single, _ = H.timed(lambda n: [serial[i % RING].forward() for i in range(n)], args.steps)
    serial_fused_mean = bool(serial[0]._own_mean)
    del serial

    # ---- device-resident throughput (`value`): RING steps in flight (FrontEndLanes: engine q replays on its own launch
    #      stream, so the latency-bound prefix and the k-NN of one batch run under the grid write / devoxelize of
    #      another); every step is launched after the start event and has finished before the end event.  At N > 1 each
    #      step's voxel indices ([B,N] int32) are all-gathered over NCCL behind the step: the result gather.
    lanes = ri_b200.FrontEndLanes(engines, lanes=LANES)
    gathered = [torch.empty((world * B, N), dtype=torch.int32, device=dev) for _ in range(RING)] if world > 1 else None
    gather_stream = torch.cuda.Stream(device=dev) if world > 1 else None

    gather_done = [torch.cuda.Event() for _ in range(RING)] if world > 1 else None

    def lane_steps(n):
        lanes.begin()
        for i in range(n):
            q = i % RING
            if world > 1 and i >= RING:              # engine q's outputs are rewritten: its previous gather must have read them
                lanes.streams[i % lanes.lanes].wait_event(gather_done[q])
            lanes.forward(i)
            if world > 1:
                gather_stream.wait_event(lanes._done[q])
                with torch.cuda.stream(gather_stream):
                    torch.distributed.all_gather_into_tensor(gathered[q], engines[q].ind)
                    gather_done[q].record(gather_stream)
        lanes.end()
        if world > 1:
            torch.cuda.current_stream().wait_stream(gather_stream)
    lane_steps(max(args.warmup, RING))
    ms, timed_steps = H.timed(lane_steps, args.steps)
    if headline and args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, engines[(timed_steps - 1) % RING])
    pts_per_step = world * B * N
    value = pts_per_step / (ms * 1e-3)
    alg = engines[0].algorithmic_bytes()
    peak, peak_src = measured_peaks()
    step_gbs = alg["total"] / (ms * 1e-3) / 1e9
    out = {"workload": wl["name"], "value": value, "ms_per_step": ms, "timed_steps": timed_steps,
           "one_step_at_a_time": {"ms_per_step": ms_single, "value": pts_per_step / (ms_single * 1e-3),
                                  "mean_fused_into_prefix_kernel": serial_fused_mean},
           "whole_step": {"algorithmic_bytes": alg["total"], "achieved": step_gbs, "frac": step_gbs / peak}}

    # ---- end to end through the host-facing call (`e2e`): every step copies ITS inputs from pinned host memory to the
    #      device and ITS per-point outputs back to pinned host memory (ppf, devox, the feat - mean(cell) half of the
    #      edge features; the other half of that tensor is the caller's own input and is not shipped back); the
    #      streaming API overlaps the copies of neighbouring steps with the compute
    pipe = ri_b200.FrontEndPipeline(B, N, C, depth=E2E_DEPTH, k=k, r=r, voxel_shape=wl["voxel_shape"], normalize=False,
                                    device=dev, edge_echo=False)
    for q in range(E2E_DEPTH):
        pipe.slot(q).h_points.copy_(torch.from_numpy(batches[q % RING][0])); pipe.slot(q).h_features.copy_(torch.from_numpy(batches[q % RING][1]))
    for i in range(2 * E2E_DEPTH):
        pipe.submit(pipe.acquire())
    pipe.drain()

    def e2e_once(n):
        H.barrier(); torch.cuda.synchronize()
        t0 = time.time(); p0 = time.perf_counter()
        for i in range(n):
            pipe.submit(pipe.acquire())
        pipe.drain()
        torch.cuda.synchronize()
        el = shard.max_over_ranks((time.perf_counter() - p0) * 1e3, dev)
        H.barrier()
        return el, (t0, time.time())
    e2e_steps = args.steps
    ms_e2e, w = e2e_once(e2e_steps); H.windows.append(w)
    ms_e2e /= e2e_steps
    out["e2e"] = {"value": pts_per_step / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": pipe.slot(0).h2d_bytes,
                  "d2h_bytes_per_step": pipe.slot(0).d2h_bytes, "steps": e2e_steps, "ms_per_step": ms_e2e,
                  "api": "FrontEndPipeline.submit/result (%d slots: H2D, step and D2H of neighbouring steps overlap; one copy per direction and step); outputs " % E2E_DEPTH +
                         "ppf [B,4,k,N], devox [B,C,N], edge_rel [B,C,N]"}
    if headline:
        for i in range(3):
            engines[i % RING].run_staged()
        ms_sync, n_sync = H.timed(lambda n: [engines[i % RING].run_staged() for i in range(n)], args.steps)
        out["e2e"]["one_call_at_a_time"] = {"value": pts_per_step / (ms_sync * 1e-3), "ms_per_step": ms_sync,
                                            "api": "FrontEnd.run_staged() (full edge tensor [B,2C,N] shipped back)",
                                            "d2h_bytes_per_step": engines[0].d2h_bytes}
    del pipe

    # ---- the HBM kernels in isolation (CUDA events on the launching stream): vox_fill (the dense [C, r^3] grid + count
    #      grid written once), the devoxelizer, and the whole voxelize op (prefix + fill)
    L = ri_b200._lib.lib
    st = torch.cuda.current_stream().cuda_stream
    shape_id = 2 if wl["voxel_shape"] == "spherical" else 0

    def fill_only(i):
        fe = engines[i % RING]
        rc = L.ri_voxelize_fill_f32(B, C, N, r, 0, B, fe.grid.data_ptr(), fe.cnt.data_ptr(), fe._ws.data_ptr(), fe._ws_bytes, st)
        assert rc == 0

    def vox_op(i):
        fe = engines[i % RING]
        mean = fe._mean_buf if fe._own_mean else fe.points[:, :3, :].mean(2)
        rc = L.ri_vox_front_f32(fe.points.data_ptr(), 6, mean.data_ptr(), fe.features.data_ptr(), B, C, N, r, shape_id, 0.0,
                                fe._front_mode(fe._own_mean), fe.norm_coords.data_ptr(), fe._vox_coords.data_ptr(), fe.ind.data_ptr(),
                                fe.edge.data_ptr(), fe._ws.data_ptr(), fe._ws_bytes, st)
        assert rc == 0
        fill_only(i)
    for i in range(RING):
        vox_op(i)
    ms_fill, _ = H.timed(lambda n: [fill_only(i) for i in range(n)], args.steps)
    # the same launches with the writers of consecutive batches in flight (one stream per buffer set): ramp and tail of one
    # launch run under the next, which is how the step executes them
    fill_streams = [torch.cuda.Stream(device=dev) for _ in range(RING)]

    def fill_in_flight(n):
        cur = torch.cuda.current_stream()
        for s_ in fill_streams:
            s_.wait_stream(cur)
        for i in range(n):
            fe = engines[i % RING]
            rc = L.ri_voxelize_fill_f32(B, C, N, r, 0, B, fe.grid.data_ptr(), fe.cnt.data_ptr(), fe._ws.data_ptr(), fe._ws_bytes,
                                        fill_streams[i % RING].cuda_stream)
            assert rc == 0
        for s_ in fill_streams:
            cur.wait_stream(s_)
    ms_fill_flight, _ = H.timed(fill_in_flight, args.steps)
    ms_devox, _ = H.timed(lambda n: [engines[i % RING]._devox(0, B, st) for i in range(n)], args.steps)
    ms_vox, _ = H.timed(lambda n: [vox_op(i) for i in range(n)], args.steps)
    ms_knn, _ = H.timed(lambda n: [engines[i % RING]._knn() for i in range(n)], args.steps)
    fill_bytes = B * (4 * (r ** 3) + 4 * C * (r ** 3))
    fill_gbs = fill_bytes / (ms_fill * 1e-3) / 1e9
    vox_gbs = alg["voxelize"] / (ms_vox * 1e-3) / 1e9
    devox_gbs = alg["devox"] / (ms_devox * 1e-3) / 1e9
    step_traffic = traffic_from_profile(key + "_step_total")
    out["roofline"] = {
        "bound": "hbm", "kernel": "vox_fill (dense [C,r^3] grid + count grid, written once)",
        "achieved": fill_gbs, "peak": peak, "unit": "GB/s", "frac": fill_gbs / peak,
        "traffic": traffic_from_profile(key), "peak_source": peak_src,
        "algorithmic_bytes_per_launch": fill_bytes, "ms_per_launch": ms_fill,
        "launches_in_flight": {"what": "the same launches on %d streams (one per buffer set): what a launch costs when its ramp and tail "
                                       "run under its neighbours, as in the step" % RING,
                               "ms_per_launch": ms_fill_flight, "achieved": fill_bytes / (ms_fill_flight * 1e-3) / 1e9,
                               "frac": fill_bytes / (ms_fill_flight * 1e-3) / 1e9 / peak},
        "voxelize_op": {"kernels": ("vox_front (mean, prologue, cell sort, cell means, edge features) + vox_fill" if engines[0]._own_mean
                                    else "torch mean + vox_front (prologue, cell sort, cell means, edge features) + vox_fill"),
                        "algorithmic_bytes": alg["voxelize"], "ms": ms_vox, "achieved": vox_gbs, "frac": vox_gbs / peak},
        "devoxelize_op": {"algorithmic_bytes": alg["devox"], "ms": ms_devox, "achieved": devox_gbs, "frac": devox_gbs / peak,
                          "grid_bytes": B * 4 * C * r ** 3, "traffic": traffic_from_profile(key + "_devox")},
        "knn_op": {"kernel": "split + knn3_warp_kernel (one warp per query, exact threshold selection)", "ms": ms_knn},
        "whole_step": dict(out["whole_step"], dram_traffic=step_traffic,
                           dram_traffic_frac=(step_traffic / (ms * 1e-3) / 1e9 / peak) if step_traffic else None)}
    out["gpu_launches_per_step"] = engines[0].kernels_per_step
    out["_engine_meta"] = {"grid_chunks": engines[0].grid_chunks, "mean_in_flight_fused": bool(engines[0]._own_mean)}
    out["_batch0"] = batches[0]
    del lanes, engines
    torch.cuda.empty_cache()
    return out


def dump_outputs(out_dir, fe):
    """The outputs of engine `fe`'s last step as DIR/<name>.npy (float32 as computed; int32 indices as float64, exactly)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("ppf", fe.ppf), ("devox", fe.devox), ("edge", fe.edge), ("ind", fe.ind)):
        a = t.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def measure_registration(ri_b200, H, rank, world, steps):
    """BASELINE configs[2]: 256 source/target pairs x 1024 pts over the GPUs of the box = 256 / world pairs per GPU:
    front end on both clouds of every pair (k-NN + PPF) -> descriptors = a FIXED random two-layer MLP on each point's
    sorted-neighbour point-pair features (stand-in for the dense layers, which are out of scope; rigid-motion invariant like
    the real descriptor) -> tcgen05 mutual-NN matcher -> RANSAC + Horn refit -> RRE / RTE / RMSE -> one all-gather."""
    import numpy as np
    torch = H.torch
    synth, shard = ri_b200.synth, ri_b200.shard
    dev = H.dev
    PAIRS, N, k, Cd = 256, 1024, 20, 512
    lo, hi = shard.shard_range(PAIRS, rank, world)
    P = hi - lo
    src, tgt, R, t = synth.make_pairs(PAIRS, N, seed=2024)
    src, tgt, R, t = src[lo:hi], tgt[lo:hi], R[lo:hi], t[lo:hi]
    both = torch.from_numpy(np.concatenate([src, tgt], 0)).to(dev).contiguous()            # [2P,6,N]
    g = torch.Generator(device=dev); g.manual_seed(7)
    W1 = torch.randn((128, 4 * k), device=dev, generator=g) / (4 * k) ** 0.5
    W2 = torch.randn((Cd, 128), device=dev, generator=g) / 128 ** 0.5
    gt = torch.eye(4, device=dev)[None].repeat(P, 1, 1)
    gt[:, :3, :3] = torch.from_numpy(R).to(dev); gt[:, :3, 3] = torch.from_numpy(t).to(dev)
    p1 = both[:P, :3].transpose(1, 2).contiguous(); p2 = both[P:, :3].transpose(1, 2).contiguous()
    mm = ri_b200.matcher.MutualMatcher(P, Cd, N, N, device=dev, want_dist=False)     # the meter uses the indices only

    def step():
        xyz = both[:, :3].contiguous(); nrm = both[:, 3:].contiguous()
        _, _, ppf = torch.ops.ri.knn_ppf(xyz, nrm, k)                                       # [2P,4,k,N]
        # the stand-in for the (out-of-scope, stock cuBLAS) dense layers runs as those do in the reference's default
        # PyTorch configuration for convolutions: TF32 tensor cores (as fp32 SIMT GEMMs they were 1.8 of the job's 5.1 ms)
        tf32 = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        try:
            f = torch.tanh(torch.matmul(W1, ppf.reshape(2 * P, 4 * k, N)))                  # [2P,128,N]
            f = torch.matmul(W2, f)                                                         # [2P,512,N], contiguous as produced
            assert f.is_contiguous()
        finally:
            torch.backends.cuda.matmul.allow_tf32 = tf32
        m = mm(f[:P], f[P:])
        T, inl = ri_b200.registration.estimate_poses(p1, p2, m.idx1, m.idx2, m.count, func="ransac", seed=1)
        met = ri_b200.registration.registration_metrics(gt, T, p1)
        res = torch.cat([T.reshape(P, 16).double(), met, inl[:, None].double(), m.count[:, None].double()], 1)
        return shard.gather_clouds(res, PAIRS)
    try:
        full = None
        for _ in range(3):
            full = step()
        ms, n = H.timed(lambda n: [step() for _ in range(n)], steps, probe=2)
    except Exception as e:                                                                  # never take the headline down
        return {"error": repr(e)[:300]}
    full = full.cpu().numpy()
    return {"workload": "DeepGMR-shaped registration job (BASELINE configs[2]): %d pairs x %d pts, %d per GPU; front end (k-NN + PPF) "
                        "on both clouds -> fixed random MLP to %d-d descriptors -> mutual-NN matcher -> RANSAC + refit -> "
                        "metrics -> all_gather" % (PAIRS, N, P, Cd),
            "ms_per_job": ms, "pairs_per_s": PAIRS / (ms * 1e-3), "timed_jobs": n,
            "mean_mutual_matches": float(full[:, 20].mean()), "mean_inliers": float(full[:, 19].mean()),
            "rre_deg_median": float(np.median(full[:, 16])), "recall_rmse_lt_0.2": float((full[:, 18] < 0.2).mean())}


def measure_matcher(ri_b200, H, rank, world, steps):
    """The matcher alone (row a11): 32 pairs x 1024 x 1024 x 512 per GPU, descriptors resident in HBM."""
    torch = H.torch
    dev = H.dev
    MP, MC, Mn = 32, 512, 1024
    g = torch.Generator(device=dev); g.manual_seed(4242 + rank)
    d1 = torch.randn((MP, MC, Mn), device=dev, generator=g); d2 = torch.randn((MP, MC, Mn), device=dev, generator=g)
    mm = ri_b200.matcher.MutualMatcher(MP, MC, Mn, Mn, device=dev)
    for _ in range(3):
        mm(d1, d2)
    ms, n = H.timed(lambda n: [mm(d1, d2) for _ in range(n)], steps)
    mi = ri_b200.matcher.MutualMatcher(MP, MC, Mn, Mn, device=dev, want_dist=False)     # indices only, as the reference returns
    for _ in range(3):
        mi(d1, d2)
    same_idx = bool(torch.equal(mi.idx1, mm.idx1) and torch.equal(mi.idx2, mm.idx2) and torch.equal(mi.count, mm.count))
    ms_idx, _ = H.timed(lambda n: [mi(d1, d2) for _ in range(n)], steps)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    useful = world * 2.0 * MP * Mn * Mn * MC / (ms * 1e-3) / 1e12
    return {"workload": "mutual-NN matching, %d pairs x %d x %d x %d per GPU" % (MP, Mn, Mn, MC),
            "pairs_per_s": world * MP / (ms * 1e-3), "ms_per_call": ms, "timed_calls": n,
            "indices_only": {"what": "dist12 = NULL: (idx1, idx2) only, the reference method's return value; no distance re-evaluation",
                             "ms_per_call": ms_idx, "pairs_per_s": world * MP / (ms_idx * 1e-3), "same_matches": same_idx},
            "useful_tflops": useful, "issued_tf32_tflops": 3 * useful,
            "frac_of_bf16_sustained": (useful / world / peaks["bf16_tflops_sustained"]) if "bf16_tflops_sustained" in peaks else None,
            "note": "3xTF32 split precision on tcgen05: three tensor-core products per useful one (ceiling 1/6 of the bf16 "
                    "peak); includes the fp32 distance re-evaluation of the matches"}


def run_ours(args, rank, world, local):
    import torch
    import ri_b200
    from ri_b200 import shard

    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    numa = shard.bind_host_to_gpu(local)            # before any pinned allocation
    sampler = ClockSampler(local) if rank == 0 else None
    H = Harness(torch, shard, dev, world)

    head = measure_workload(args.workload, args, ri_b200, H, rank, world, local, headline=True)
    also = {}
    if not args.only:
        for key in ("cu_dg", "sph_dg", "sph_r16", "sph_r64"):
            if key == args.workload:
                continue
            m = measure_workload(key, args, ri_b200, H, rank, world, local, headline=False)
            m.pop("_batch0"); m.pop("_engine_meta")
            also[key] = m
        also["matcher"] = measure_matcher(ri_b200, H, rank, world, args.steps)
        also["registration_job"] = measure_registration(ri_b200, H, rank, world, args.steps)
    if rank != 0:
        return
    sampler.stop()
    wl = WORKLOADS[args.workload]
    meta = head.pop("_engine_meta")
    batch0 = head.pop("_batch0")
    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": head["ms_per_step"], "timed_steps": head["timed_steps"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_for(wl, world),
        "notes": {"cuda_graph": True, "steps_in_flight": LANES, "grid_chunks": meta["grid_chunks"],
                  "overlap": "k-NN/PPF branch on a side stream next to the grid writer and the devoxelizer; %d independent "
                             "batches in flight on %d launch streams, %d buffer sets cycled" % (LANES, LANES, RING),
                  "one_step_at_a_time": head["one_step_at_a_time"],
                  "result_gather": ("all_gather_into_tensor of every step's voxel indices [B,N] i32 over NCCL, inside the timed region"
                                    if world > 1 else "single GPU: nothing to gather"),
                  "host_numa_binding": numa,
                  "timed_region": "timed_steps = --steps steps between one pair of CUDA events"},
        "roofline": head["roofline"],
        "e2e": head["e2e"],
        "gpu_launches": head["gpu_launches_per_step"] * head["timed_steps"],
        "clocks": sampler.summary(H.windows),
        "also": also,
    }
    if world == 1:
        line["cpu_baseline"] = cpu_port_baseline(wl, batch0)
    print(json.dumps(line))


def cpu_port_step(wl, pts, feats, o):
    """The same front-end step with the C oracle port (OpenMP over clouds)."""
    import numpy as np
    B, N, C, k, r = pts.shape[0], wl["N"], wl["C"], wl["k"], wl["r"]
    xyz, nrm = np.ascontiguousarray(pts[:, :3]), np.ascontiguousarray(pts[:, 3:])
    _, idx = o.knn_one(xyz, xyz, k)
    gi = np.broadcast_to(idx.reshape(B, 1, k * N), (B, 3, k * N))
    o.ppf(np.broadcast_to(xyz[:, :, None, :], (B, 3, k, N)).reshape(B, 3, k * N), np.take_along_axis(xyz, gi, 2),
          np.broadcast_to(nrm[:, :, None, :], (B, 3, k, N)).reshape(B, 3, k * N), np.take_along_axis(nrm, gi, 2))
    if wl["voxel_shape"] == "spherical":
        avg, ind, nc = o.spherical_voxelization_module(feats, xyz, r)
        o.spherical_trilinear_devoxelize(nc, avg, ind, r)
    else:
        avg, ind, nc = o.voxelization_module(feats, xyz, r, normalize=False)
        o.trilinear_devoxelize(nc, avg, r)
    o.voxel_edge_gather(avg, feats, ind)


def cpu_port_baseline(wl, batch, reps=3):
    from oracle import cpu_oracle as o
    o.build()
    pts, feats = batch
    nb = min(pts.shape[0], 32)
    cpu_port_step(wl, pts[:2], feats[:2], o)              # warm-up (library load, page faults)
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        cpu_port_step(wl, pts[:nb], feats[:nb], o)
        best = min(best, time.perf_counter() - t0)
    return {"value": nb * wl["N"] / best, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
            "sample": "%d clouds x %d pts, best of %d passes of the C oracle port (OpenMP over clouds, %d threads)" %
                      (nb, wl["N"], reps, os.cpu_count())}


# ================================================================================================ reference
def run_reference(args, rank, world, local):
    """The reference arm, one rank per GPU like the other arm: every rank runs the reference's unmodified CUDA kernels on its
    own shard of the (world * B)-cloud job; value = all ranks' points / the slowest rank's time."""
    wl = WORKLOADS[args.workload]
    B, N, C, k, r = wl["B"], wl["N"], wl["C"], wl["k"], wl["r"]
    base = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_for(wl, world)}
    synth = load_by_path("ri_synth", "synth.py")
    pts = synth.make_clouds(B, N, seed=1000 + 17 * rank); feats = synth.make_features(B, C, N, seed=1000 + 17 * rank)

    ref = None
    torch = None
    try:
        import torch
        from oracle.build_ref import load_ref
        if torch.cuda.is_available():
            ref = load_ref()
    except Exception:
        ref = None

    if ref is None:                                       # no reference library on this box: the oracle port, rank 0 only
        if rank != 0:
            return
        cb = cpu_port_baseline(wl, (pts, feats), reps=max(1, min(args.steps, 3)))
        base.update({"n_gpus": 1, "value": cb["value"], "ms_per_step": B * N / cb["value"] * 1e3, "cpu_baseline": cb,
                     "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        print(json.dumps(base))
        return

    shard = load_by_path("ri_shard", "shard.py")          # torch-only helpers; the product library stays unloaded
    shard.init_from_env()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    numa = shard.bind_host_to_gpu(local)
    hp = torch.from_numpy(pts).pin_memory(); hf = torch.from_numpy(feats).pin_memory()
    out_h = {}

    def barrier():
        if world > 1:
            torch.distributed.barrier()

    def step(host):
        """Reference op sequence for the same front end, through the reference backend's own functions
        (bindings.cpp:13-56) and the torch glue the reference uses around them."""
        p = hp.to(dev, non_blocking=True) if host else d_p
        f = hf.to(dev, non_blocking=True) if host else d_f
        xyz = p[:, :3].contiguous(); nrm = p[:, 3:].contiguous()
        _, _, idx, _ = ref.knn_forward_cuda(xyz, xyz, k)                                   # bilateral API
        gi = idx.reshape(B, 1, k * N).expand(-1, 3, -1).long()
        c_xyz = xyz[:, :, None, :].expand(-1, -1, k, -1).reshape(B, 3, k * N).contiguous()
        c_n = nrm[:, :, None, :].expand(-1, -1, k, -1).reshape(B, 3, k * N).contiguous()
        ppf = ref.spherical_ppf_forward(torch.gather(xyz, 2, gi), c_xyz, torch.gather(nrm, 2, gi), c_n)
        nc = xyz - xyz.mean(2, keepdim=True)
        if wl["voxel_shape"] == "spherical":
            nc = nc / (nc.norm(dim=1, keepdim=True).max(dim=2, keepdim=True).values + 1e-20)
            avg, ind, cnt = ref.spherical_avg_voxelize_forward(f, nc.contiguous(), r)
            dv, _, _ = ref.spherical_trilinear_devoxelize_forward(r, True, nc.contiguous(), avg, ind)
        else:
            nc = torch.clamp((nc + 1) / 2.0 * r, 0, r - 1)
            avg, ind, cnt = ref.avg_voxelize_forward(f, torch.round(nc).to(torch.int32).contiguous(), r)
            dv, _, _ = ref.trilinear_devoxelize_forward(r, True, nc.contiguous(), avg)
        mask = ind == -1                                                                   # pvconv.py:68-90
        it = ind.clone(); it[mask] = 0
        centre = avg.gather(2, it.unsqueeze(1).expand(-1, C, -1).long())
        rel = f - centre
        rel[mask.unsqueeze(1).expand(-1, C, -1)] = 0
        edge = torch.cat((rel, f), 1)                                                      # what the next layer consumes
        if host:
            # the same three tensors the other arm ships back: ppf, devox, the relative half of the edge features
            for name, t in (("ppf", ppf), ("devox", dv), ("edge_rel", rel)):
                if name not in out_h:
                    out_h[name] = torch.empty(t.shape, dtype=t.dtype).pin_memory()
                out_h[name].copy_(t, non_blocking=True)
            torch.cuda.synchronize()
        return edge

    d_p, d_f = hp.to(dev), hf.to(dev)
    for _ in range(max(args.warmup, 3)):
        step(False)

    def timed_events(n):
        barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            step(False)
        e1.record(); torch.cuda.synchronize(); barrier()
        return shard.max_over_ranks(e0.elapsed_time(e1), dev)
    n1 = args.steps
    ms = timed_events(n1) / n1
    for _ in range(3):
        step(True)

    def timed_wall(n):
        barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n):
            step(True)
        el = shard.max_over_ranks((time.perf_counter() - t0) * 1e3, dev)
        barrier()
        return el
    n2 = args.steps
    ms2 = timed_wall(n2) / n2
    if world > 1:
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    value = world * B * N / (ms * 1e-3)
    base.update({
        "value": value, "ms_per_step": ms, "timed_steps": n1,
        "notes": {"host_numa_binding": numa},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 0, "kind": "reference",
                         "sample": "the reference's own CUDA kernels (oracle/_ref, unmodified sources recompiled for "
                                   "sm_100a) on the same B200s, one rank per GPU — the reference has no CPU implementation "
                                   "of this path"},
        "e2e": {"value": world * B * N / (ms2 * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": hp.numel() * 4 + hf.numel() * 4,
                "d2h_bytes_per_step": sum(t.numel() * 4 for t in out_h.values()), "steps": n2, "ms_per_step": ms2}})
    print(json.dumps(base))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="sph_dg")
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--only", action="store_true", help="measure only --workload (skip the `also` configurations)")
    ap.add_argument("--fuse-mean-in-flight", dest="fuse_mean_in_flight", action="store_true", default=True)
    ap.add_argument("--torch-mean-in-flight", dest="fuse_mean_in_flight", action="store_false")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the headline's last timed step to DIR/<name>.npy (bench_outputs/ is git-ignored)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world, local)
        return
    from ri_b200 import shard
    rank, world, local = shard.init_from_env()
    try:
        run_ours(args, rank, world, local)
    finally:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
