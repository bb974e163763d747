"""Registration back end on the GPU: descriptors -> mutual matches -> rigid pose -> ICP refinement -> RRE / RTE / RMSE,
whole batches of pairs per call (csrc/matcher.cu + csrc/pose.cu + csrc/fgr.cu + csrc/teaser.cu + csrc/icp.cu).

Mirrors the reference's meter `MeterModelNet40_registration` (/root/reference/datasets/deepgmr_mn40.py:98-244): same
constructor argument, same `update((feat1, feat2), (pt1, pt2, gt_trans))` / `compute()` contract, same thresholds
(:107-109), same result keys (:141).  The reference copies the descriptors to the host and calls Open3D / TEASER++ once
per pair (:121, :165-231); here `func='ransac'` runs the RANSAC configuration the reference hands to Open3D
(utils/open3d_func.py:43-49: voxel_size 0.08, edge-length similarity 0.9, max_iter 1000) on the GPU for all pairs at once,
`func='fgr'` Open3D's Fast Global Registration over the same matches (`fgr()`), `func='teaserpp'` TEASER++ with a known
scale (`teaser()`: maximum clique of the pairwise-consistency graph, GNC-TLS rotation, adaptive-voting translation), and
`func='kabsch'` the plain least squares over the mutual matches.  `icp()` / `evaluate_registration()` are Open3D's
registration_icp (point-to-point and point-to-plane) and evaluate_registration, batched over pairs; `register_pairs` and
the meter refine their pose with it when given `icp={...}`.  `generalized_icp()` is Open3D's registration_generalized_icp
(plane-to-plane, covariances from normals), a separate refinement after any of them: `generalized_icp(pt1, pt2, r, init=T)`.
Both point-to-plane `icp()` and `generalized_icp()` take Open3D's robust kernels (`kernel=('tukey', k)` and the like).
func='icp' raises in `estimate_poses`: ICP refines a pose, it does not estimate one from matches.
"""
import math
import time

import torch

from . import matcher, ops

__all__ = ['estimate_poses', 'fgr', 'teaser', 'registration_metrics', 'icp', 'generalized_icp', 'evaluate_registration',
           'register_pairs', 'MeterModelNet40_registration']


def estimate_poses(src, tgt, idx1, idx2, count, func='ransac', voxel_size=0.08, max_iter=1000, edge_similarity=0.9,
                   refine_iters=3, seed=0, noise_bound=None):
    """src [P,n1,3], tgt [P,n2,3] CUDA fp32; idx1/idx2/count: the mutual matches (matcher.mutual_nn).
    -> (T [P,4,4] fp32 mapping src onto tgt, inliers [P] int32).
    func='fgr' is fgr() with maximum_correspondence_distance = 0.5 * voxel_size (the value of Open3D's FGR tutorial) and
    inlier_dist = voxel_size, Open3D's other defaults, and `seed`; max_iter, edge_similarity and refine_iters are unused.
    func='teaserpp' is teaser() with `noise_bound` (required: it is in the clouds' units and has no unit-free default),
    inlier_dist = voxel_size and TEASER++'s other defaults; max_iter, edge_similarity, refine_iters and seed are unused.
    The other modes ignore noise_bound."""
    if func not in ('ransac', 'kabsch', 'fgr', 'teaserpp'):
        raise ValueError("func must be 'ransac', 'fgr', 'teaserpp' or 'kabsch' (ICP refines a pose: "
                         "icp() or register_pairs(..., icp={...}))")
    if func == 'fgr':
        r = fgr(src, tgt, idx1, idx2, count, maximum_correspondence_distance=0.5 * float(voxel_size), seed=seed,
                inlier_dist=float(voxel_size))
        return r['transformation'], r['inliers']
    if func == 'teaserpp':
        if noise_bound is None:
            raise ValueError("func='teaserpp' needs noise_bound (the bound on a match's noise, in the clouds' units)")
        r = teaser(src, tgt, idx1, idx2, count, noise_bound, inlier_dist=float(voxel_size))
        return r['transformation'], r['inliers']
    hyps = int(max_iter) if func == 'ransac' else 0
    return torch.ops.ri.pose_from_matches(src.float().contiguous(), tgt.float().contiguous(), idx1.contiguous(),
                                          idx2.contiguous(), count.contiguous(), hyps, float(voxel_size),
                                          float(edge_similarity), int(refine_iters), int(seed))


def _int64(seed):
    """A 64-bit seed as the signed integer a torch op argument holds (the library reads the same 64 bits unsigned)."""
    s = int(seed) & 0xFFFFFFFFFFFFFFFF
    return s - (1 << 64) if s >= 1 << 63 else s


def fgr(src, tgt, idx1, idx2, count, maximum_correspondence_distance=0.025, iteration_number=64, division_factor=1.4,
        use_absolute_scale=False, decrease_mu=True, tuple_test=True, tuple_scale=0.95, maximum_tuple_count=1000, seed=0,
        inlier_dist=None, return_correspondences=False):
    """Open3D's registration_fgr_based_on_feature_matching (FastGlobalRegistrationOption's names and defaults) for P pairs
    at once, over given matches: src [P,n1,3], tgt [P,n2,3] CUDA fp32; idx1/idx2 [P,ld], count [P] (matcher.mutual_nn).
    The tuple test samples with `seed`; inliers are counted within inlier_dist (default: maximum_correspondence_distance)
    under the returned pose, as in estimate_poses.  include/ri_b200.h (ri_fgr_f32) states the arithmetic.
    -> dict(transformation [P,4,4] fp32 src -> tgt, inliers [P] int32, num_correspondences [P] int32
    [, correspondences [P,L] int32: the list's match positions, -1 padded; L = 3 * maximum_tuple_count with the tuple
    test, else ld])."""
    if inlier_dist is None:
        inlier_dist = maximum_correspondence_distance
    T, inl, corr, ncorr = torch.ops.ri.fgr(src.float().contiguous(), tgt.float().contiguous(), idx1.contiguous(),
                                           idx2.contiguous(), count.contiguous(), float(maximum_correspondence_distance),
                                           int(iteration_number), float(division_factor), bool(use_absolute_scale),
                                           bool(decrease_mu), bool(tuple_test), float(tuple_scale),
                                           int(maximum_tuple_count), _int64(seed), float(inlier_dist))
    out = {'transformation': T, 'inliers': inl, 'num_correspondences': ncorr}
    if return_correspondences:
        if not tuple_test:                             # the list is the first ncorr matches
            pos = torch.arange(idx1.shape[1], dtype=torch.int32, device=ncorr.device).expand(idx1.shape[0], -1)
            corr = torch.where(pos < ncorr[:, None], pos, -1)
        out['correspondences'] = corr
    return out


# expand calls of the exact maximum-clique search per pair; no pair of tools/bench_teaser.py's workloads reaches it
# (profiles/r6_teaser.md)
MAX_CLIQUE_NODES = 100000


def teaser(src, tgt, idx1, idx2, count, noise_bound, cbar2=1.0, rotation_gnc_factor=1.4, rotation_max_iterations=100,
           rotation_cost_threshold=1e-12, max_clique_nodes=MAX_CLIQUE_NODES, inlier_dist=None, return_clique=False):
    """TEASER++ (RobustRegistrationSolver with a known scale: estimate_scaling=False) for P pairs at once, over given
    matches: src [P,n1,3], tgt [P,n2,3] CUDA fp32; idx1/idx2 [P,ld], count [P] (matcher.mutual_nn).  Options carry
    TEASER++'s names; noise_bound is in the clouds' units.  Pipeline: the pairwise-consistency graph (edge when two
    matches' lengths differ by at most 2 noise_bound sqrt(cbar2)), its maximum clique (deterministic branch and bound with
    a budget of max_clique_nodes expand calls; clique_exact says whether it finished), GNC-TLS rotation over the clique's
    chain TIMs, adaptive-voting translation.  Inliers are counted within inlier_dist (default: noise_bound) under the
    returned pose, as in estimate_poses.  include/ri_b200.h (ri_teaser_f32) states the arithmetic and DESIGN.md §8 the
    deltas from TEASER++.
    -> dict(transformation [P,4,4] fp32 src -> tgt, inliers [P] int32, clique_size [P] int32, clique_exact [P] bool
    [, clique [P,ld] int32: ascending match positions, -1 padded])."""
    if inlier_dist is None:
        inlier_dist = noise_bound
    T, inl, clique, size, exact = torch.ops.ri.teaser(src.float().contiguous(), tgt.float().contiguous(),
                                                      idx1.contiguous(), idx2.contiguous(), count.contiguous(),
                                                      float(noise_bound), float(cbar2), float(rotation_gnc_factor),
                                                      int(rotation_max_iterations), float(rotation_cost_threshold),
                                                      int(max_clique_nodes), float(inlier_dist))
    out = {'transformation': T, 'inliers': inl, 'clique_size': size, 'clique_exact': exact.bool()}
    if return_clique:
        out['clique'] = clique
    return out


def registration_metrics(gt_trans, est_trans, pts):
    """[P,4,4], [P,4,4], [P,n,3] -> [P,3] float64 (RRE in degrees, RTE, RMSE) — RE_TE_one_pair + the RMSE of update()."""
    return torch.ops.ri.registration_metrics(gt_trans.float().contiguous(), est_trans.float().contiguous(),
                                             pts.float().contiguous())


_ESTIMATIONS = ('point_to_point', 'point_to_plane')
_KERNELS_WITH_K = ('huber', 'cauchy', 'gm', 'tukey')


def _robust_loss(kernel):
    """A robust-kernel spec -> (loss index of ops.ROBUST_LOSSES, k), or None for None and 'l2' (the plain estimators).
    ValueError for anything else than 'l1' or (name, k) with name in _KERNELS_WITH_K and k finite and > 0."""
    if kernel is None or (isinstance(kernel, str) and kernel == 'l2'):
        return None
    if isinstance(kernel, str) and kernel == 'l1':
        return ops.ROBUST_LOSSES.index('l1'), 0.0
    if isinstance(kernel, (tuple, list)) and len(kernel) == 2 and isinstance(kernel[0], str) \
            and kernel[0] in _KERNELS_WITH_K:
        try:
            k = float(kernel[1])
        except (TypeError, ValueError):
            k = float('nan')
        if math.isfinite(k) and k > 0.0:
            return ops.ROBUST_LOSSES.index(kernel[0]), k
        raise ValueError("the %s kernel needs a finite k > 0, got %r" % (kernel[0], kernel[1]))
    raise ValueError("kernel must be None, 'l2', 'l1' or (name, k) with name one of %s, got %r" % (_KERNELS_WITH_K, kernel))


def icp(src, tgt, max_correspondence_distance, init=None, estimation='point_to_point', tgt_normals=None, max_iter=30,
        relative_fitness=1e-6, relative_rmse=1e-6, return_correspondences=False, kernel=None):
    """Open3D's registration_icp for P pairs at once.  src [P,n1,3], tgt [P,n2,3] CUDA fp32; init [P,4,4] (default identity);
    tgt_normals [P,n2,3] for estimation='point_to_plane'.  Stops a pair when both its fitness and its inlier RMSE change by
    less than the relative criteria (Open3D's ICPConvergenceCriteria), or after max_iter updates.
    kernel (point_to_plane only; Open3D's TransformationEstimationPointToPlane(loss)): None or 'l2' (the plain least
    squares), 'l1', or (name, k) with name 'huber', 'cauchy', 'gm' or 'tukey'.  Each correspondence's row of the update is
    weighted by w(r) of its point-to-plane residual r; k is in distance units (for 'gm' in squared distance units).
    include/ri_b200.h (ri_robust_icp_f32) states the weights and the deltas from Open3D.
    -> dict(transformation [P,4,4] fp32 src -> tgt, fitness [P] f64, inlier_rmse [P] f64, iterations [P] int32
    [, correspondences [P,n1] int32: target index or -1, under the returned transformation])."""
    if estimation not in _ESTIMATIONS:
        raise ValueError("estimation must be one of %s, got %r" % (_ESTIMATIONS, estimation))
    plane = estimation == 'point_to_plane'
    if kernel is not None and not plane:
        raise ValueError("a robust kernel needs estimation='point_to_plane' (Open3D's point-to-point takes none)")
    robust = _robust_loss(kernel)
    if plane and tgt_normals is None:
        raise ValueError("estimation='point_to_plane' needs tgt_normals")
    src = src.float().contiguous()
    if init is None:
        init = torch.eye(4, dtype=torch.float32, device=src.device).expand(src.shape[0], 4, 4)
    nrm = tgt_normals.float().contiguous() if plane else None
    if robust is not None:
        T, fit, rmse, iters, corr = torch.ops.ri.robust_icp(src, tgt.float().contiguous(), None, nrm,
                                                            init.float().contiguous(),
                                                            float(max_correspondence_distance), False, 1.0, robust[0],
                                                            robust[1], int(max_iter), float(relative_fitness),
                                                            float(relative_rmse), bool(return_correspondences))
    else:
        T, fit, rmse, iters, corr = torch.ops.ri.icp(src, tgt.float().contiguous(), nrm, init.float().contiguous(),
                                                     float(max_correspondence_distance), plane, int(max_iter),
                                                     float(relative_fitness), float(relative_rmse),
                                                     bool(return_correspondences))
    out = {'transformation': T, 'fitness': fit, 'inlier_rmse': rmse, 'iterations': iters}
    if return_correspondences:
        out['correspondences'] = corr
    return out


_icp = icp       # register_pairs() and the meter take an `icp` argument of their own


def generalized_icp(src, tgt, max_correspondence_distance, init=None, epsilon=1e-3, src_normals=None, tgt_normals=None,
                    max_iter=30, relative_fitness=1e-6, relative_rmse=1e-6, return_correspondences=False, kernel=None):
    """Open3D's registration_generalized_icp (plane-to-plane) for P pairs at once.  src [P,n1,3], tgt [P,n2,3] CUDA fp32;
    init [P,4,4] (default identity).  The loop, the stopping rule, fitness, inlier_rmse and the correspondences are icp()'s;
    the update minimises sum d^T (C_t + R C_s R^T)^-1 d over correspondences, d = T s - t, with the covariances
    C(n) = I - (1 - epsilon) n n^T built from unit normals (a zero or non-finite normal gives C = I).
    src_normals [P,n1,3] / tgt_normals [P,n2,3]: each cloud's normals in its own frame; a missing one is estimated with
    functional.estimate_normals(cloud, radius=inf, max_nn=20), i.e. from the 20 nearest neighbours (distance^2 < 10000;
    (0,0,1) with fewer than 3).  A normal's sign does not matter.
    Deltas from Open3D: M^-1 is used directly rather than its square root (equal up to rounding); every normal uses the
    exact covariance, where Open3D substitutes that of e1 for normals within about 8 degrees of -x (read from its source,
    not verified against a build); no caller-supplied covariance matrices.
    kernel: as in icp() (Open3D's TransformationEstimationForGeneralizedICP(epsilon, loss)).  Open3D's way: the residual is
    whitened, r = W d with W = (C_t + R C_s R^T)^-1/2, and each of its three rows weighted by w(r_k); so k is in whitened
    units (distance / sqrt(eigenvalue of C_t + R C_s R^T), e.g. distance / sqrt(2 epsilon) along a shared normal and
    distance / sqrt(2) across it; for 'gm' squared whitened units), and a robust result is not invariant to rotating both
    clouds together (the rows are the world axes).  None and 'l2' run the plain estimator.
    include/ri_b200.h (ri_generalized_icp_f32, ri_robust_icp_f32) states the arithmetic.
    -> dict(transformation [P,4,4] fp32 src -> tgt, fitness [P] f64, inlier_rmse [P] f64, iterations [P] int32
    [, correspondences [P,n1] int32: target index or -1, under the returned transformation])."""
    from .functional import estimate_normals
    src = src.float().contiguous()
    tgt = tgt.float().contiguous()
    if init is None:
        init = torch.eye(4, dtype=torch.float32, device=src.device).expand(src.shape[0], 4, 4)
    init = init.float().contiguous()
    src_normals = None if src_normals is None else src_normals.float().contiguous()
    tgt_normals = None if tgt_normals is None else tgt_normals.float().contiguous()
    robust = _robust_loss(kernel)
    ops.check_generalized_icp(src, tgt, src_normals, tgt_normals, init, max_correspondence_distance, epsilon, max_iter)
    estimate = lambda x: estimate_normals(x.transpose(1, 2), radius=float('inf'), max_nn=20).transpose(1, 2).contiguous()
    if src_normals is None:
        src_normals = estimate(src)
    if tgt_normals is None:
        tgt_normals = estimate(tgt)
    if robust is not None:
        T, fit, rmse, iters, corr = torch.ops.ri.robust_icp(src, tgt, src_normals, tgt_normals, init,
                                                            float(max_correspondence_distance), True, float(epsilon),
                                                            robust[0], robust[1], int(max_iter),
                                                            float(relative_fitness), float(relative_rmse),
                                                            bool(return_correspondences))
    else:
        T, fit, rmse, iters, corr = torch.ops.ri.generalized_icp(src, tgt, src_normals, tgt_normals, init,
                                                                 float(max_correspondence_distance), float(epsilon),
                                                                 int(max_iter), float(relative_fitness),
                                                                 float(relative_rmse), bool(return_correspondences))
    out = {'transformation': T, 'fitness': fit, 'inlier_rmse': rmse, 'iterations': iters}
    if return_correspondences:
        out['correspondences'] = corr
    return out


def evaluate_registration(src, tgt, max_correspondence_distance, T):
    """Open3D's evaluate_registration for P pairs: correspondences of src under T [P,4,4] within the distance, and
    -> dict(fitness [P] f64, inlier_rmse [P] f64, correspondences [P,n1] int32 (target index or -1))."""
    r = icp(src, tgt, max_correspondence_distance, init=T, max_iter=0, return_correspondences=True)
    return {'fitness': r['fitness'], 'inlier_rmse': r['inlier_rmse'], 'correspondences': r['correspondences']}


def register_pairs(feat1, feat2, pt1, pt2, func='ransac', icp=None, **kw):
    """feat1/feat2 [P,C,n] (the extractor's layout), pt1/pt2 [P,n,3], all CUDA -> (T [P,4,4], inliers [P], matches dict).
    icp: None, or a dict of `icp()` keyword arguments (max_correspondence_distance required) to refine the pose with."""
    m = matcher.mutual_nn(feat1, feat2, point_major=False, want_dist=False)      # the meter uses the matches only
    T, inl = estimate_poses(pt1, pt2, m['idx1'], m['idx2'], m['count'], func=func, **kw)
    if icp is not None:
        T = _icp(pt1, pt2, init=T, **icp)['transformation']
    return T, inl, m


class MeterModelNet40_registration:
    """Same state, thresholds and result keys as the reference meter (deepgmr_mn40.py:98-141)."""

    def __init__(self, func='ransac', device='cuda', icp=None, noise_bound=None):
        """func: 'ransac', 'fgr', 'teaserpp' or 'kabsch' (estimate_poses).  icp: None, or a dict of `icp()` keyword
        arguments; the estimated pose is then refined with it (inside reg_time).  noise_bound: required by 'teaserpp'."""
        if func == 'teaserpp' and noise_bound is None:
            raise ValueError("func='teaserpp' needs noise_bound (the bound on a match's noise, in the clouds' units)")
        self.rre = 0
        self.rte = 0
        self.num = 0
        self.succ = 0
        self.rmse = 0
        self.rmse_succ = 0
        self.reg_time = 0
        self.rot_thresh = 1e-05
        self.rmse_thresh = 0.2
        self.translate_thresh = 0.005
        self.func = func
        self.device = torch.device(device)
        self.icp = icp
        self.kw = {} if noise_bound is None else {'noise_bound': noise_bound}

    def update(self, output, target):
        """output = (feat1, feat2) [b,C,n]; target = (pt1 [b,n,3], pt2 [b,n,3], gt_trans [b,4,4]) — numpy or torch."""
        with torch.no_grad():
            dev = self.device
            feat1, feat2 = (torch.as_tensor(f, dtype=torch.float32).to(dev) for f in output)
            pt1, pt2, gt = (torch.as_tensor(t, dtype=torch.float32).to(dev) for t in target)
            torch.cuda.synchronize(dev)
            t0 = time.time()
            T, _, _ = register_pairs(feat1, feat2, pt1, pt2, func=self.func, icp=self.icp, **self.kw)
            torch.cuda.synchronize(dev)
            reg_time = time.time() - t0
            m = registration_metrics(gt, T, pt1).cpu()
            rre, rte, rmse = m[:, 0], m[:, 1], m[:, 2]
            b = pt1.shape[0]
            self.succ += int(((rre < self.rot_thresh) & (rte < self.translate_thresh)).sum())
            self.rmse_succ += int((rmse < self.rmse_thresh).sum())
            self.rre += float(rre.sum())
            self.rte += float(rte.sum())
            self.rmse += float(rmse.sum())
            self.reg_time += reg_time
            self.num += b

    def compute(self):
        return {'succ': self.succ / self.num, 'rre': self.rre / self.num, 'rte': self.rte / self.num,
                'rmse': self.rmse / self.num, 'reg_time': self.reg_time / self.num, 'rmse_succ': self.rmse_succ / self.num}
