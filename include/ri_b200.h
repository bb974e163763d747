/*
 * ri_b200.h — C ABI of libri_b200.so: the B200 (sm_100a) implementation of the data-parallel front end of the
 * rotation-invariant PVCNN feature extractor.
 *
 * This is the drop-in boundary.  Each entry point replaces one function of the reference's pybind11 module
 * `_multi_shape_pvcnn_backend` (/root/reference/PVCNN/modules/functional/src/bindings.cpp:13-56) or, for the
 * matcher and the edge gather, the Python block cited beside it.  INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference adds in PVCNN/modules/functional/backend.py.
 *
 * Conventions (all entry points):
 *   - plain device pointers + sizes; tensors are contiguous, channel-major [B, C, N] (points innermost), fp32 / int32;
 *   - the CALLER allocates every output and the workspace; nothing is allocated or freed inside;
 *   - the caller has made the right device current and passes its stream (`cudaStream_t` as void*); every kernel is
 *     enqueued on that stream and the call returns without synchronising;
 *   - return value: 0 on success, a positive cudaError_t if a launch failed, or a negative RI_ERR_* code for a bad
 *     argument.  Never calls exit() (the reference's CUDA_CHECK_ERRORS does, cuda_utils.cuh:28-37);
 *   - re-entrant and thread-safe: the only process-wide state is read-only after its first use — the environment knobs of
 *     DESIGN.md §11 (read once), the SM count per device, and the per-(kernel, device) record that a kernel's function
 *     attributes have been set (csrc/ri_common.cuh).  Several host threads may call into the library on several devices;
 *   - calls that share a WORKSPACE must be ordered on one stream (the workspace holds their intermediate tables).
 */
#ifndef RI_B200_H
#define RI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RI_OK 0
#define RI_ERR_BAD_ARG (-1)
#define RI_ERR_WORKSPACE (-2)
#define RI_ERR_UNSUPPORTED (-3)

/* ABI version of this header/library pair. */
int ri_abi_version(void);

/* Debug aid: a one-thread kernel that stores the device's nanosecond timer (%globaltimer) into *slot. */
int ri_debug_stamp(unsigned long long* slot, void* stream);

/* Debug aid for tests and tools: the environment knobs of DESIGN.md §11 are read once per process; this sets one of them
 * afterwards, by its variable name (e.g. "RI_DEVOX_STREAM", -1 = unset).  Not to be called while launches are in flight on
 * other threads.  RI_ERR_BAD_ARG for a name that cannot be changed at run time. */
int ri_debug_set_knob(const char* name, int value);

/* ---- k-nearest neighbours -------------------------------------------------------------------------------
 * One direction of knn_forward_cuda (knn/knn.cpp:6-25 -> KnnKernel knn/knn.cu:5-49): for each of the n points of
 * xyz1 [B,c,n] its k nearest (squared L2) among the m points of xyz2 [B,c,m].
 * dist1 [B,k,n] ascending along k, idx1 [B,k,n] indices into xyz2; unfilled slots are (10000.0f, 0).
 * Bit-exact against the reference incl. its tie rule (lower reference index first). */
int ri_knn_f32(const float* xyz1, const float* xyz2, int B, int c, int n, int m, int k,
               float* dist1, int* idx1, void* stream);

/* ri_knn_f32 through the one-thread-per-query kernel whatever the shape (ri_knn_f32 itself takes the warp-per-query
 * kernel of csrc/knn_warp.cu for c == 3, k <= 32, m <= 1024).  Same results bit for bit; exists for the tests. */
int ri_knn_thread_f32(const float* xyz1, const float* xyz2, int B, int c, int n, int m, int k,
                      float* dist1, int* idx1, void* stream);

/* knn_forward_cuda itself: both directions (knn/knn.cu:81-87). dist2/idx2 are [B,k,m]. */
int ri_knn_bilateral_f32(const float* xyz1, const float* xyz2, int B, int c, int n, int m, int k,
                         float* dist1, float* dist2, int* idx1, int* idx2, void* stream);

/* The same search for scan-sized clouds (~50k points, c == 3): uniform hash grid + ring expansion instead of the full
 * scan, results bit-identical to ri_knn_f32 (same distance expression, candidates ordered by (distance, index)).
 * k <= 32.  workspace >= ri_knn_grid_workspace_bytes(B, n, m) bytes, 16-byte aligned. */
size_t ri_knn_grid_workspace_bytes(int B, int n, int m);
int ri_knn_grid_f32(const float* xyz1, const float* xyz2, int B, int n, int m, int k,
                    float* dist1, int* idx1, void* workspace, size_t workspace_bytes, void* stream);

/* knn_backward_cuda (knn/knn.cpp:27-52 -> KnnGradKernel knn/knn.cu:52-78), both directions.
 * gradxyz1 [B,c,n] and gradxyz2 [B,c,m] are overwritten. */
int ri_knn_backward_f32(const float* xyz1, const float* xyz2, const float* graddist1, const float* graddist2,
                        const int* idx1, const int* idx2, int B, int c, int n, int m, int k,
                        float* gradxyz1, float* gradxyz2, void* stream);

/* ---- point-pair features --------------------------------------------------------------------------------
 * spherical_ppf_forward (spherical_ppf/ppf.cpp:17-36 -> spherical_ppf_kernel ppf.cu:19-92), backend argument
 * order: coords = the points, center = the centres (functional/ppf.py:22 swaps the user-facing order).
 * All inputs [B,3,L]; feat [B,4,L] = (angle(d,n_c), angle(d,n_p), angle(n_c,n_p), ||d||), d = center - coords. */
int ri_ppf_f32(const float* coords, const float* center, const float* normals, const float* center_normal,
               int B, int L, float* feat, void* stream);

/* Fused neighbour gather + PPF for k-NN neighbourhoods: xyz, normals [B,3,N], idx [B,k,N] -> out [B,4,k,N];
 * centre = point i, point = neighbour idx[b,s,i].  Equals ri_ppf_f32 on the gathered/expanded columns. */
int ri_ppf_gather_f32(const float* xyz, const float* normals, const int* idx, int B, int N, int k,
                      float* out, void* stream);

/* ---- coordinate prologue of the voxelization modules -----------------------------------------------------
 * Voxelization.forward (PVCNN/modules/voxelization.py:16-35) / Spherical_Voxelization.forward
 * (PVCNN/modules/spherical_vox.py:14-23) after the per-cloud mean: centre, scale, clamp/round or divide by the
 * largest radius, in one kernel.  points [B,pstride,N] (pstride 3 = xyz, 6 = xyz|normal), mean [B,3] (the caller's
 * `coords.mean(2)`: its summation order defines the bits).  shape: 0 cube normalize=False, 1 cube normalize=True,
 * 2 spherical.  Outputs: norm_coords [B,3,N] fp32 (always), vox_coords [B,3,N] i32 (shape 0/1), and optionally the
 * de-interleaved xyz / normals planes [B,3,N] (null to skip).  norm_mode selects the association of the 3-term
 * radius sum (1 = (x*x + y*y) + z*z without contraction, the one matching torch norm). */
int ri_vox_prologue_f32(const float* points, int pstride, const float* mean, int B, int N, int r,
                        int shape, float eps, int norm_mode,
                        float* xyz, float* normals, float* norm_coords, int* vox_coords, void* stream);

/* Fused self-query k-NN + PPF: ri_knn_f32(xyz, xyz) followed by ri_ppf_gather_f32, in one kernel and bit-identical to
 * that pair.  xyz / normals address [3,N] planes per cloud, cloud b at base + b * cloud_stride floats: 3N for two
 * contiguous [B,3,N] arrays, 6N (with normals = xyz + 3N) for the interleaved [B,6,N] input batch the models receive.
 * dist / idx [B,k,N] may both be null; ppf [B,4,k,N].  N <= 2048 and k <= 32, else RI_ERR_UNSUPPORTED. */
int ri_knn_ppf_f32(const float* xyz, const float* normals, long long cloud_stride, int B, int N, int k,
                   float* dist, int* idx, float* ppf, void* stream);

/* De-interleave points [B,6,N] (xyz | normal) into contiguous xyz [B,3,N] and normals [B,3,N] — the `.contiguous()`
 * copies of inputs[:, :3, :] / inputs[:, 3:, :] the reference's wrappers make (functional/knn.py:11-12,
 * functional/ppf.py:16-19) — and, optionally, the point-major packing packed [B,N,8] = (x,y,z,nx,ny,nz,0,0) (16-byte
 * aligned) that ri_ppf_gather_packed_f32 reads.  Any of the three outputs may be null; one launch. */
int ri_split_xyz_normals_f32(const float* points, int B, int N, float* xyz, float* normals, float* packed, void* stream);

/* ri_ppf_gather_f32 on the packed cloud: no shared memory, neighbours fetched as two 16-byte gathers.  Same values. */
int ri_ppf_gather_packed_f32(const float* packed, const int* idx, int B, int N, int k, float* out, void* stream);

/* ---- voxelization ---------------------------------------------------------------------------------------
 * spherical_avg_voxelize_forward (spherical_voxelization/spherical_vox.cpp:17-46) and avg_voxelize_forward
 * (voxelization/vox.cpp:17-43).  feat [B,C,N]; coords [B,3,N] (fp32 normalised Cartesian for the spherical
 * variant, int32 voxel coordinates for the cube variant) -> out [B,C,r^3], ind [B,N] (-1 = undefined point),
 * cnt [B,r^3].  All three outputs are fully overwritten (no pre-zeroing needed).
 * workspace >= ri_voxelize_workspace_bytes(B, C, N, r) bytes of device memory, 16-byte aligned (per-cloud cell tables
 * plus the compact table of cell means [B][C][<=N]). */
size_t ri_voxelize_workspace_bytes(int B, int C, int N, int r);
int ri_sph_voxelize_f32(const float* feat, const float* coords, int B, int C, int N, int r,
                        float* out, int* ind, int* cnt, void* workspace, size_t workspace_bytes, void* stream);
int ri_cube_voxelize_f32(const float* feat, const int* coords, int B, int C, int N, int r,
                         float* out, int* ind, int* cnt, void* workspace, size_t workspace_bytes, void* stream);

/* Fused voxelize + DGCNN edge features: same as above and additionally edge [B,2C,N] =
 * cat(feat - out[:, :, ind] (0 where ind == -1), feat), i.e. what ri_voxel_edge_gather_f32 would produce from `out`,
 * emitted in the same pass (the voxelizer already holds each point's cell mean; the dense grid is not re-read).
 * Replaces voxelize + PVCNN/modules/pvconv.py:68-90. */
int ri_sph_voxelize_edge_f32(const float* feat, const float* coords, int B, int C, int N, int r,
                             float* out, int* ind, int* cnt, float* edge,
                             void* workspace, size_t workspace_bytes, void* stream);
int ri_cube_voxelize_edge_f32(const float* feat, const int* coords, int B, int C, int N, int r,
                              float* out, int* ind, int* cnt, float* edge,
                              void* workspace, size_t workspace_bytes, void* stream);

/* Phase-by-phase form of the voxelizers, for schedules that overlap or pipeline the phases (the one-shot calls above run
 * the same three kernels back to back):
 *   prepare  ind [B,N] and the cell tables of ALL B clouds (one launch over the batch);
 *   means    the compact table of cell means of the clouds [b0, b1) and, when edge [B,2C,N] is non-null, their DGCNN edge
 *            features cat(feat - mean of own cell, feat) (pvconv.py:68-90);
 *   fill     out [B,C,r^3] / cnt [B,r^3] of the clouds [b0, b1) from the tables and means in the workspace.
 * out, cnt, edge are the whole-batch arrays; same workspace as the one-shot calls.  Returns RI_ERR_UNSUPPORTED when the
 * shape is outside the tiled path (N > 4096, r^3 % 4 != 0, outputs not 16-byte aligned): use the one-shot calls then. */
int ri_sph_voxelize_prepare_f32(const float* coords, int B, int C, int N, int r, int* ind,
                                void* workspace, size_t workspace_bytes, void* stream);
int ri_cube_voxelize_prepare_f32(const int* coords, int B, int C, int N, int r, int* ind,
                                 void* workspace, size_t workspace_bytes, void* stream);
int ri_voxelize_means_f32(const float* feat, int B, int C, int N, int r, int b0, int b1, float* edge,
                          void* workspace, size_t workspace_bytes, void* stream);
int ri_voxelize_fill_f32(int B, int C, int N, int r, int b0, int b1, float* out, int* cnt,
                         void* workspace, size_t workspace_bytes, void* stream);

/* The prefix of the voxel branch in one launch: ri_vox_prologue_f32 + ri_*_voxelize_prepare_f32 + ri_voxelize_means_f32
 * for all B clouds (bit-identical outputs); ri_voxelize_fill_f32 then completes the voxelization.  Arguments as
 * ri_vox_prologue_f32 plus feat [B,C,N]; outputs norm_coords [B,3,N], vox_coords [B,3,N] (cube shapes), ind [B,N],
 * edge [B,2C,N] (nullable) and the workspace tables.  N <= 1024 and the tiled-path conditions, else RI_ERR_UNSUPPORTED.
 * norm_mode flag bits: 0x100 = compute the per-cloud mean inside the kernel (torch's reduction order; written to `mean`);
 * 0x200 = `edge` is [B,C,N] and receives only the (feat - mean of the point's cell) half of the edge features — the
 * other half is the caller's own input. */
int ri_vox_front_f32(const float* points, int pstride, const float* mean, const float* feat,
                     int B, int C, int N, int r, int shape, float eps, int norm_mode,
                     float* norm_coords, int* vox_coords, int* ind, float* edge,
                     void* workspace, size_t workspace_bytes, void* stream);

/* avg_voxelize_backward == spherical_avg_voxelize_backward (vox.cpp:54-78, vox.cu:87-111):
 * grad_x [B,C,N] = grad_y[b,c,ind] / cnt (0 for undefined points); grad_x fully overwritten. */
int ri_voxelize_backward_f32(const float* grad_y, const int* ind, const int* cnt, int B, int C, int N, int s,
                             float* grad_x, void* stream);

/* ---- devoxelization -------------------------------------------------------------------------------------
 * trilinear_devoxelize_forward (interpolate/trilinear_devox.cpp:18-55): coords [B,3,N] in grid units [0,r-1],
 * feat [B,C,r^3] -> outs [B,C,N], inds [B,8,N], wgts [B,8,N] (all fully overwritten). */
int ri_trilinear_devox_f32(const float* coords, const float* feat, int B, int C, int N, int r,
                           float* outs, int* inds, float* wgts, void* stream);

/* spherical_trilinear_devoxelize_forward (interpolate/spherical_trilinear_devox.cpp:19-56), index quirks kept.
 * coords = normalised Cartesian coords, g_inds [B,N] = spherical cell of each point.
 * Requires r >= 4, else RI_ERR_UNSUPPORTED before any launch: the reference's corner rows are radians truncated to ints
 * (alpha row <= 6, beta row <= 3, gamma row always 0), so the highest corner index is r^2 + 7r + 4, which stays below r^3
 * only from r = 4 on. */
int ri_sph_trilinear_devox_f32(const float* coords, const float* feat, const int* g_inds, int B, int C, int N, int r,
                               float* outs, int* inds, float* wgts, void* stream);

/* trilinear_devoxelize_backward / spherical_trilinear_devoxelize_backward (trilinear_devox.cu:120-163,
 * spherical_trilinear_devox.cu:150-194): grad_x [B,C,s] fully overwritten; skip_undefined != 0 skips points whose
 * inds[b,0,i] == -1 (the spherical variant). */
int ri_devox_backward_f32(const float* grad_y, const int* inds, const float* wgts, int B, int C, int N, int s,
                          int skip_undefined, float* grad_x, void* stream);

/* ---- DGCNN voxel-neighbour edge features (PVCNN/modules/pvconv.py:68-90) --------------------------------
 * avg [B,C,s], feat [B,C,N], inds [B,N] -> out [B,2C,N] = cat(feat - avg[:, :, inds] (0 where inds == -1), feat). */
int ri_voxel_edge_gather_f32(const float* avg, const float* feat, const int* inds, int B, int C, int N, int s,
                             float* out, void* stream);

/* ---- ball query + grouping (SURVEY.md 8f row f1: the neighbourhood the shipped models use for local features) ----------
 * ball_query_forward (ball_query/ball_query.cpp:6-30 -> ball_query_kernel ball_query.cu:19-50): for each of the M centres
 * the first U points (in index order) with 1e-5 < d^2 < radius^2; the first hit fills the whole row, a centre without
 * neighbours keeps zeros.  centers [B,3,M], points [B,3,N] -> neighbors [B,M,U] int32, fully overwritten.  Bit-exact. */
int ri_ball_query_f32(const float* centers, const float* points, int B, int N, int M, float radius, int U,
                      int* neighbors, void* stream);

/* The 'ppf' local features of the shipped models from the neighbour indices, without materialising the grouped tensors:
 * PVCNN/models/pvcnn_classify.py:252-270 + PVCNN/modules/ball_query.py:16-35 (d = c - (p_nbr - c), |d|, three clamped acos
 * of torch-ordered dot products, fp32).  points_* [B,3,N], centers_* [B,3,M], neighbors [B,M,U] -> out [B,4,U,M]. */
int ri_local_ppf_f32(const float* points_coords, const float* points_normals, const float* centers_coords,
                     const float* centers_normals, const int* neighbors, int B, int N, int M, int U,
                     float* out, void* stream);

/* The whole local-feature branch of the shipped models (pvcnn_classify.py:61-67, 252-271) from the ball-query indices:
 * local point-pair features -> SharedMLP(4 -> 32 -> 64) in eval mode -> max over the neighbours, in one kernel (layer 2 on
 * tcgen05 as a 3xTF32 split product; nothing between the indices and the result leaves the SM).  w1 [32,4], b1 [32],
 * w2 [64,32], b2 [64]: the two 1x1 convolutions with their BatchNorm (running statistics) folded in.  neighbors [B,M,U];
 * out [B,64,M].  U == 128, C1 == 32, C2 == 64 (the shipped shape), else RI_ERR_UNSUPPORTED. */
int ri_local_ppf_mlp_max_f32(const float* points_coords, const float* points_normals, const float* centers_coords,
                             const float* centers_normals, const int* neighbors, int B, int N, int M, int U,
                             const float* w1, const float* b1, int C1, const float* w2, const float* b2, int C2,
                             float* out, void* stream);

/* grouping_forward / grouping_backward (grouping/grouping.cu:18-44, 58-84): out [B,C,M,U] = feat[b, c, idx[b, m, u]];
 * grad_x [B,C,N] += grad_y scattered through idx (float atomics, as the reference; grad_x is zeroed first). */
int ri_grouping_f32(const float* feat, const int* idx, int B, int C, int N, int M, int U, float* out, void* stream);
int ri_grouping_backward_f32(const float* grad_y, const int* idx, int B, int C, int N, int M, int U,
                             float* grad_x, void* stream);

/* ---- mutual-nearest-neighbour descriptor matching (datasets/deepgmr_mn40.py:232-244) ---------------------
 * find_correspondence_one_pair for P independent (source, target) pairs.
 * desc1, desc2: fp32 descriptors, channel-major [P,C,n1] / [P,C,n2] (what the feature extractor emits,
 * pvcnn_classify.py:345) when point_major == 0, or point-major [P,n1,C] / [P,n2,C] (the numpy layout the
 * reference's meter passes, deepgmr_mn40.py:121) when point_major != 0.
 *   diff[i,j] = |f1_i|^2 + |f2_j|^2 - 2 f1_i.f2_j           (3xTF32 split-precision tcgen05 contraction)
 *   corr12 [P,n1] = argmin_j diff, corr21 [P,n2] = argmin_i diff   (lowest index on ties, as np.argmin)
 *   dist12 [P,n1] = diff[i, corr12[i]] recomputed as an fp32 FMA chain; NULL = indices only (what the reference's
 *                   method returns): the re-evaluation pass over the descriptors is skipped
 *   idx1, idx2 [P,n1]: the mutual matches (corr21[corr12[i]] == i) in ascending i, count [P] of them, -1 beyond.
 * workspace >= ri_mutual_nn_workspace_bytes(P, C, n1, n2) bytes of device memory. */
size_t ri_mutual_nn_workspace_bytes(int P, int C, int n1, int n2);
int ri_mutual_nn_tf32x3(const float* desc1, const float* desc2, int P, int C, int n1, int n2, int point_major,
                        int* corr12, int* corr21, float* dist12, int* idx1, int* idx2, int* count,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- barycentre grid subsampling (SURVEY.md 8f row f2) ---------------------------------------------------------------
 * grid_subsampling() (cpp_wrappers/cpp_subsampling/grid_subsampling/grid_subsampling.cpp:4-106, called through
 * cpp_subsampling/wrapper.cpp:58-285 and utils/grid_subsampleing.py:3-21): one barycentre per occupied cell of edge dl.
 * points [N,3] row-major (the reference's numpy layout), features [N,fdim] or NULL, labels [N,ldim] or NULL ->
 * out_points [<=N,3], out_features [<=N,fdim], out_labels [<=N,ldim] (allocate for N cells), *out_count = number of cells
 * (DEVICE memory; no host synchronisation inside).  Cells come out in ascending cell index (the reference's order is an
 * unordered_map's); sums run in original point order, so barycentres and features are bit-identical to the reference;
 * label ties go to the smallest label.  workspace >= ri_grid_subsample_workspace_bytes(N). */
size_t ri_grid_subsample_workspace_bytes(int N);
int ri_grid_subsample_f32(const float* points, const float* features, const int* labels, int N, int fdim, int ldim,
                          float dl, float* out_points, float* out_features, int* out_labels, int* out_count,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---- correspondences -> rigid pose -> registration metrics (SURVEY.md 8f row f3) --------------------------------------
 * What follows the matcher in the reference's meter (datasets/deepgmr_mn40.py:104-139): the solve is delegated there to
 * Open3D RANSAC / FGR (utils/open3d_func.py:34-75) or TEASER++ (deepgmr_mn40.py:175-230) on the host, one pair at a time.
 * Here: RANSAC over the mutual matches with the configuration the reference hands to Open3D (3-point samples,
 * edge-length similarity 0.9, sample residual and validation distance = voxel_size, max_iter hypotheses, point-to-point
 * least squares without scale), all pairs in one launch, then Horn's closed-form refit on the inliers.
 * src [P,n1,3], tgt [P,n2,3] point-major fp32; idx1, idx2 [P,ld], count [P] as ri_mutual_nn_tf32x3 returns them;
 * hyps == 0: least squares over all matches (Kabsch).  T [P,4,4] row-major fp32 (src -> tgt), inliers [P].
 * Every match counts: min(count[p], ld) matches, any number (they are staged in shared memory 4096 at a time); sampling,
 * inlier counts, the refit and the Kabsch solve all run over all of them.
 * Sampler: hypothesis h < hyps of pair p uses matches (i0, i1, i2) = sample3(seed, p, h, M), M = the pair's match count:
 *   mix64 = the splitmix64 finaliser (x += 0x9E3779B97F4A7C15; x = (x ^ x>>30) * 0xBF58476D1CE4E5B9;
 *           x = (x ^ x>>27) * 0x94D049BB133111EB; x ^ x>>31), all uint64 with wrap-around;
 *   r0 = mix64(seed ^ (p << 32) ^ (uint32)h), r1 = mix64(r0), r2 = mix64(r1);
 *   i0 = r0 % M; i1 = r1 % (M-1), +1 if >= i0; i2 = r2 % (M-2), +1 if >= min(i0,i1), +1 more if then >= max(i0,i1).
 * The winner is the valid hypothesis with the most inliers, the lowest h on ties.
 * best: P * 8 bytes of scratch (may be NULL when hyps == 0).  With hyps > 0 it holds, after the call, the winner of each
 * pair as (inliers << 32) | (0xffffffff - h), or 0 when no hypothesis passed its checks.
 * inliers[p] is always the count under the returned T[p]; when no pose was found (fewer than 3 matches, or no valid
 * hypothesis) T[p] is the identity and inliers[p] is 0. */
int ri_pose_from_matches_f32(const float* src, const float* tgt, const int* idx1, const int* idx2, const int* count,
                             int P, int n1, int n2, int ld, int hyps, float inlier_dist, float edge_similarity,
                             int refine_iters, unsigned long long seed, float* T, int* inliers,
                             unsigned long long* best, void* stream);

/* RE_TE_one_pair (deepgmr_mn40.py:152-164) + the point RMSE of MeterModelNet40_registration.update (:121-126), fp64:
 * gt, est [P,4,4] row-major fp32, pts [P,n,3] -> out [P,3] double = (rotation error in degrees, translation error, rmse). */
int ri_registration_metrics_f32(const float* gt, const float* est, const float* pts, int P, int n, double* out,
                                void* stream);

/* ---- 'change_coords' rotation-invariant preprocessing (SURVEY.md 8f row f4) -------------------------------------------
 * The Python double loop of PVCNN_classifier.forward, rot_invariant_preprocess == 'change_coords'
 * (PVCNN/models/pvcnn_classify.py:153-184), as one kernel: per cloud a frame from the farthest point and the farthest
 * point not (anti)parallel to it (|cos| < 0.9), Gram-Schmidt, and the coordinates expressed in that frame.
 * coords [B,cstride,N] (cstride 3 or 6, first three planes used), mean [B,3] = torch's coords.mean(2), norm_mode as in
 * ri_vox_prologue_f32  ->  out [B,3,N], bases [B,3,3] (rows x, y, z; may be NULL), ok [B] (0 where the reference asserts). */
int ri_lrf_change_coords_f32(const float* coords, int cstride, const float* mean, int B, int N, int norm_mode,
                             float* out, float* bases, int* ok, void* stream);

/* ---- ICP refinement (SURVEY.md 8f, next row f5) -----------------------------------------------------------------------
 * Open3D's registration_icp (utils/open3d_func.py wraps it) for P independent pairs per call: T = init, then per iteration
 * correspondences under T (nearest target point with d^2 < max_corr_dist^2, ties to the lowest target index), an update U
 * (point-to-point: Horn's closed form, no scale; point-to-plane: Open3D's linearised 6x6 solve, identity when singular),
 * T = U T, until |d fitness| < rel_fitness and |d inlier_rmse| < rel_rmse or max_iter updates.  max_iter == 0 is Open3D's
 * evaluate_registration of init.
 * src [P,n1,3], tgt [P,n2,3], tgt_normals [P,n2,3] (point_to_plane != 0 only; may be NULL otherwise), init [P,4,4] row-major
 * (NULL = identity), fp32 point-major.  Outputs: T [P,4,4] fp32, fitness [P] and inlier_rmse [P] double, iters [P] int32
 * (updates applied), corr [P,n1] int32 = target index or -1 under the returned T (may be NULL).  Bit-reproducible; no host
 * synchronisation.  workspace >= ri_icp_workspace_bytes(P, n1, n2) bytes of device memory, 16-byte aligned. */
size_t ri_icp_workspace_bytes(int P, int n1, int n2);
int ri_icp_f32(const float* src, const float* tgt, const float* tgt_normals, const float* init, int P, int n1, int n2,
               float max_corr_dist, int point_to_plane, int max_iter, float rel_fitness, float rel_rmse,
               float* T, double* fitness, double* inlier_rmse, int* iters, int* corr,
               void* workspace, size_t workspace_bytes, void* stream);

/* ---- Generalized ICP (SURVEY.md 8f, row f9) ---------------------------------------------------------------------------
 * Open3D's registration_generalized_icp (Segal, Haehnel, Thrun, RSS 2009; plane-to-plane) for P independent pairs per call.
 * The loop, the correspondences, fitness, inlier_rmse, iters, corr and the fp64 accumulated T are exactly ri_icp_f32's
 * (T = init, evaluate; per iteration solve U, T = U T, re-evaluate; stop when |d fitness| < rel_fitness and
 * |d inlier_rmse| < rel_rmse or after max_iter updates; max_iter == 0 evaluates init).  Only the update differs:
 *   covariance  C(n) = I - (1 - epsilon) n^ n^T per point, n^ = n / |n| in fp64; a zero-length or non-finite normal gives
 *               C = I.  (Open3D's normals path, R_{e1->n} diag(eps,1,1) R_{e1->n}^T, and its no-normals path, the 20-NN
 *               covariance's SVD with singular values (1,1,eps), both build this matrix from the smallest-eigenvalue
 *               direction.)  The sign of a normal does not matter.
 *   term        for a correspondence (source s, target t): q = T s as in ri_icp_f32; a = R n^_s with R the rotation of the
 *               same fp32 T, evaluated in fp64; b = n^_t; M = C_t + R C_s R^T = 2I - (1 - epsilon)(a a^T + b b^T) (for
 *               0 < epsilon <= 1 its eigenvalues lie in [2 epsilon, 2]); d = q - t; J0 = [-[q]x, I3].
 *   update      H = sum J0^T M^-1 J0 and g = sum J0^T M^-1 d in fp64 with fixed-order reductions, M^-1 in closed form
 *               (adjugate over determinant); H x = -g by LDL^T, |det H| < 1e-6 or a non-finite x gives U = I (the
 *               point-to-plane rule); U = [Rz(x2) Ry(x1) Rx(x0) | x3 x4 x5].
 * Deltas from Open3D: (1) Open3D forms W = (M^-1)^(1/2) and sums (W J0)^T (W J0) and (W J0)^T (W d); with its default L2
 * kernel that equals H and g in exact arithmetic, so the two differ by rounding only.  (2) Open3D's GetRotationFromE1ToX
 * returns the identity when n.e1 < -0.99, so for normals within about 8 degrees of -x it uses the covariance of e1 instead of
 * that of n; here the exact formula is used for every normal (read from Open3D's GeneralizedICP.cpp, not verified against
 * a build of it).  (3) Caller-supplied covariance matrices are not supported (robust kernels: ri_robust_icp_f32).
 * src [P,n1,3], tgt [P,n2,3], src_normals [P,n1,3], tgt_normals [P,n2,3] (both required), init [P,4,4] row-major
 * (NULL = identity), fp32 point-major.  Outputs as ri_icp_f32.  Bit-reproducible (no float atomics); a pair's result does not
 * depend on the rest of the batch; max_iter + 6 launches, no host synchronisation, no allocation.
 * workspace >= ri_icp_workspace_bytes(P, n1, n2).  RI_ERR_BAD_ARG for n1 or n2 <= 0, max_corr_dist <= 0 or NaN,
 * epsilon <= 0 or not finite, max_iter < 0, or a NULL normals pointer. */
int ri_generalized_icp_f32(const float* src, const float* tgt, const float* src_normals, const float* tgt_normals,
                           const float* init, int P, int n1, int n2, float max_corr_dist, float epsilon, int max_iter,
                           float rel_fitness, float rel_rmse, float* T, double* fitness, double* inlier_rmse, int* iters,
                           int* corr, void* workspace, size_t workspace_bytes, void* stream);

/* ---- Robust kernels for point-to-plane and generalized ICP (SURVEY.md 8f, row f11) -------------------------------------
 * Open3D's TransformationEstimationPointToPlane(loss) and TransformationEstimationForGeneralizedICP(epsilon, loss).  The
 * loop, the correspondences, the stopping rule, fitness, inlier_rmse, iters, corr and the fp64 accumulated T are exactly
 * ri_icp_f32's; only the update's sums are weighted, in fp64, by w(r) = Open3D's RobustKernel::Weight (formulas recalled
 * from Open3D's RobustKernel.cpp, not verified against its source or a build), e = |r|:
 *   RI_LOSS_L2      1                                  RI_LOSS_CAUCHY  1 / (1 + (r/k)^2)
 *   RI_LOSS_L1      1 / e  (0 at e = 0, delta 1)       RI_LOSS_GM      k / (k + r^2)^2   (k in squared units, w(0) = 1/k)
 *   RI_LOSS_HUBER   k / max(e, k)                      RI_LOSS_TUKEY   (1 - (e/k)^2)^2 for e <= k, else 0
 *   point-to-plane (generalized == 0): r = (q - t).n_t, J = [q x n_t, n_t] with n_t as given (not normalised);
 *               H = sum w(r) J^T J, g = sum w(r) J^T r (w J_a first, then the same fma as ri_icp_f32: with w = 1 exactly the
 *               sums, and so every output, are bit-identical to ri_icp_f32's point-to-plane).
 *   generalized (!= 0): M as in ri_generalized_icp_f32, W = (M^-1)^(1/2) (principal root, closed form from the eigenvectors
 *               a +- b of M), r = W d, row k weighted by w(r_k): H = sum J0^T A J0, g = sum J0^T A d with
 *               A = W diag(w(r_0), w(r_1), w(r_2)) W (with L2, A = M^-1 up to rounding).  The rows are the world axes, so
 *               a robust result is not invariant to rotating both clouds together (as in Open3D).
 *   Then the point-to-plane solve: |det H| < 1e-6 or a non-finite x gives U = I.
 * Deltas from Open3D: (1) L1 gives w = 0 at r = 0 exactly, where Open3D's +inf makes the step non-finite (identity update).
 * (2) As in ri_icp_f32, the original source is transformed by the accumulated T.  (3) The 1e-6 determinant rule sees the
 * weighted H, so a kernel changes which systems count as singular (e.g. GM with a large k).
 * src, tgt, tgt_normals (required), src_normals (required and read when generalized != 0 only), init: as
 * ri_generalized_icp_f32.  Outputs as ri_icp_f32.  Bit-reproducible; a pair's result does not depend on the rest of the
 * batch.  workspace >= ri_icp_workspace_bytes(P, n1, n2).  RI_ERR_BAD_ARG for the argument errors of ri_icp_f32, a NULL
 * normals pointer, epsilon <= 0 or not finite (generalized), an unknown loss, or k <= 0 or not finite for Huber, Cauchy, GM
 * and Tukey. */
#define RI_LOSS_L2 0
#define RI_LOSS_L1 1
#define RI_LOSS_HUBER 2
#define RI_LOSS_CAUCHY 3
#define RI_LOSS_GM 4
#define RI_LOSS_TUKEY 5
int ri_robust_icp_f32(const float* src, const float* tgt, const float* src_normals, const float* tgt_normals,
                      const float* init, int P, int n1, int n2, float max_corr_dist, int generalized, float epsilon,
                      int loss, float k, int max_iter, float rel_fitness, float rel_rmse, float* T, double* fitness,
                      double* inlier_rmse, int* iters, int* corr, void* workspace, size_t workspace_bytes, void* stream);

/* ---- normal estimation for xyz-only clouds (SURVEY.md 8f, row f6) ----------------------------------------------------
 * Open3D's estimate_normals with KDTreeSearchParamHybrid(radius, max_nn) (the reference calls it on the host,
 * utils/open3d_func.py:77-83), B clouds per call.  xyz [B,3,N] fp32; radius > 0 (+inf = plain k-NN), 1 <= max_nn <= 32.
 * For each point q:
 *   neighbours  the max_nn smallest keys (d, index) among the points with d < min(r2, 10000), q itself included, where
 *               d = fma(dz,dz, fma(dy,dy, dx*dx)), d* = q - p in fp32, and r2 = radius * radius in fp32.  That is exactly
 *               the first max_nn entries of ri_knn_grid_f32(xyz, xyz, k = max_nn) whose distance is < min(r2, 10000).
 *               The radius cut is strict, as in ri_icp_f32 and ri_ball_query_f32;
 *   covariance  p - q in fp64, accumulated over that list in its (d, index) order; C = S2/n - mu mu^T (population);
 *   normal      unit eigenvector of the smallest eigenvalue of C (fp64 cyclic Jacobi, lowest index on equal eigenvalues),
 *               rounded to fp32; (0,0,1) when fewer than 3 neighbours or when trace(C) is not positive and finite;
 *   orientation camera [B,3]: flipped when n.(camera_b - q) < 0 (orient_normals_towards_camera_location); prior [B,3,N]:
 *               flipped when n.prior < 0 (Open3D's rule for a cloud that has normals); neither: the solver's sign
 *               (deterministic, not part of the contract).  At most one of camera / prior; the (0,0,1) default is
 *               oriented too.
 * Outputs normals [B,3,N] fp32 and, unless NULL, counts [B,N] int32 = neighbours used (q included).  No host
 * synchronisation; a cloud's result does not depend on the rest of the batch and is bit-reproducible.
 * workspace >= ri_knn_grid_workspace_bytes(B, N, N) bytes, 16-byte aligned.  RI_ERR_BAD_ARG for radius <= 0 or NaN,
 * max_nn <= 0 or both camera and prior; RI_ERR_UNSUPPORTED for max_nn > 32 or B > 65535. */
int ri_estimate_normals_f32(const float* xyz, int B, int N, float radius, int max_nn, const float* camera,
                            const float* prior, float* normals, int* counts, void* workspace, size_t workspace_bytes,
                            void* stream);

/* ---- Fast Global Registration (SURVEY.md 8f, row f7) -----------------------------------------------------------------
 * Open3D's registration_fgr_based_on_feature_matching (Zhou, Park, Koltun, ECCV 2016; the reference's alternative to RANSAC,
 * utils/open3d_func.py:50-62) over the mutual matches, P pairs in one launch.  src, tgt, idx1, idx2, count as in
 * ri_pose_from_matches_f32: pair p has M = min(count[p], ld) matches, match m pairs a_m = src[idx1[m]] with b_m = tgt[idx2[m]].
 *   tuple test  (tuple_test != 0; AdvancedMatching)  trial t = 0, 1, ... < 100 M draws r0 = mix64(seed ^ (p << 32) ^ (uint32)t),
 *               r1 = mix64(r0), r2 = mix64(r1) (mix64 as in ri_pose_from_matches_f32) and i_k = r_k % M, independently.
 *               Edge lengths |a_i0 - a_i1|, |a_i1 - a_i2|, |a_i2 - a_i0| (and the same over the b's) are computed in fp64 from
 *               the fp32 coordinates as sqrt((dx*dx + dy*dy) + dz*dz), each operation rounded (no contraction).  The trial is
 *               accepted when every edge has l_a * s < l_b && l_b < l_a / s, s = (double)tuple_scale.  The list is
 *               (i0, i1, i2) of each of the first max_tuples accepted trials, in trial order; fewer when the trials run out.
 *               tuple_test == 0: the list is the M matches in order.
 *   normalise   mu_s, mu_t = means of all n1 source / n2 target points (fp64); scale = the largest |x - mu| over both clouds;
 *               g = scale, par = 1 (use_absolute_scale == 0) or g = 1, par = scale; points are used as (x - mu) * (1 / g).
 *   GNC         (fp64) T' = I moves the normalised target onto the normalised source; per iteration it < iterations:
 *               par /= division_factor when decrease_mu && it % 4 == 0 && par > max_corr_dist; per correspondence q = T' q^,
 *               r = p^ - q, w = (par / (r.r + par))^2, rows r_x: J = (0, -q_z, q_y, -1, 0, 0), r_y: (q_z, 0, -q_x, 0, -1, 0),
 *               r_z: (-q_y, q_x, 0, 0, 0, -1); x = -(J^T W J)^-1 J^T W r (Delta = I when a pivot of the LDL^T factorisation is
 *               not positive or x is not finite); T' = [Rz(x2) Ry(x1) Rx(x0) | x3 x4 x5] T'.
 *   output      T[p] = inverse of [R' | mu_s - R' mu_t + g t'] (maps src onto tgt), rounded to fp32, row-major [4,4];
 *               inliers[p] = #{m < M : |R a_m + t - b_m|^2 < inlier_dist^2} under that fp32 T, with the arithmetic of
 *               ri_pose_from_matches_f32.  No pose (M < 3 or a list shorter than 10): T[p] = I and inliers[p] = 0.
 * corr [P, 3 * max_tuples] receives the list's match positions, -1 past its end; required when tuple_test != 0 (the list is
 * read back from it), may be NULL otherwise (and is not written).  ncorr [P] = the list's length (3 x accepted trials, or M).
 * No host synchronisation; a pair's result is bit-reproducible and does not depend on the rest of the batch.
 * RI_ERR_BAD_ARG for max_corr_dist <= 0, iterations < 0, division_factor <= 1, tuple_scale outside (0, 1], max_tuples < 1,
 * inlier_dist <= 0, or corr == NULL with tuple_test != 0; RI_ERR_UNSUPPORTED for 100 * ld >= 2^32 (the trial index is
 * 32-bit) or max_tuples > INT_MAX / 3. */
int ri_fgr_f32(const float* src, const float* tgt, const int* idx1, const int* idx2, const int* count,
               int P, int n1, int n2, int ld, float max_corr_dist, int iterations, float division_factor,
               int use_absolute_scale, int decrease_mu, int tuple_test, float tuple_scale, int max_tuples,
               unsigned long long seed, float inlier_dist, float* T, int* inliers, int* corr, int* ncorr,
               void* stream);

/* ---- TEASER++ with a known scale (SURVEY.md 8f, row f10) -------------------------------------------------------------
 * TEASER++ (Yang, Shi, Carlone, T-RO 2020; the reference's registration solver, deepgmr_mn40.py:175-230) over the mutual
 * matches, P pairs per call.  src, tgt, idx1, idx2, count as in ri_pose_from_matches_f32: pair p has M = min(count[p], ld)
 * matches a_m = src[idx1[m]], b_m = tgt[idx2[m]]; every match is a vertex.  tests/teaser_oracle.py replays every step.
 *   graph     edge (i, j), i != j, iff |l_a - l_b| <= beta, beta = 2 * noise_bound * sqrt(cbar2) (fp64, in that order);
 *             l = |u - v| in fp64 from the fp32 coordinates as sqrt((dx*dx + dy*dy) + dz*dz), each operation rounded (no
 *             contraction), |l_a - l_b| likewise: the graph is bit-exact.
 *   order     pi sorts the vertices by degree descending, then index ascending; "first" below means first in pi.
 *   clique    (a) for each of the first min(M, 64) vertices v of pi: C = {v}, cand = N(v); repeatedly add the first vertex of
 *             cand and intersect cand with its neighbourhood; best = the largest C, the earliest v on ties.  (b) Repeatedly
 *             remove every alive vertex whose alive-degree is below |best|.  (c) BBMC branch and bound over the alive
 *             vertices: expand(C, P) colours P greedily (each class takes, in pi order, every remaining vertex not adjacent
 *             to the class so far), then visits the vertices in reverse colouring order, returning when |C| + colour <=
 *             |best|; v with P & N(v) empty ends a clique C + {v}, which replaces best when strictly larger; otherwise
 *             expand(C + {v}, P & N(v)); then P -= {v}.  Each expand call costs one node; when a call would exceed
 *             max_clique_nodes the search stops, exact[p] = 0, and the best clique so far is kept (exact[p] = 1 otherwise).
 *   rotation  chain TIMs over the clique c(0) < ... < c(K-1): v_k = a_c(k+1) - a_c(k), w_k = b_c(k+1) - b_c(k), k + 1 taken
 *             mod K (fp64).  GNC-TLS with weights 1, c2 = beta^2, prev = 0: per iteration < max_iterations: R = Horn's
 *             rotation of S = sum wt_k v_k w_k^T (as ri_pose_from_matches_f32's refit), r2_k = |w_k - R v_k|^2; on the first
 *             iteration mu = 1 / (2 max r2 / c2 - 1), stop if mu <= 0; cost = sum wt_k r2_k (the weights before this update);
 *             wt = 0 if r2 >= (mu+1)/mu c2, 1 if r2 <= mu/(mu+1) c2, else sqrt(c2 mu (mu+1) / r2) - mu; mu *= gnc_factor;
 *             stop if |cost - prev| < cost_threshold; prev = cost.  R = I when max_iterations == 0.
 *   translation  per axis, x_k = b_c(k) - R a_c(k) (fp64), r = noise_bound * sqrt(cbar2): the events x_k - r (enter) and
 *             x_k + r (leave), ordered by value, then enter before leave, then k; after each event the consensus set S
 *             (when not empty) gives t = sum_S x / |S| and cost = sum_S (x - t)^2 + (K - |S|) r^2, sums in index order;
 *             the minimum cost wins, the earliest event on ties.
 *   output    T[p] = [R | t] rounded to fp32, row-major [4,4], maps src onto tgt; inliers[p] = #{m < M : |R a_m + t - b_m|^2
 *             < inlier_dist^2} under that fp32 T, with the arithmetic of ri_pose_from_matches_f32.  M < 3 or a clique of
 *             fewer than 3 vertices: T[p] = I and inliers[p] = 0.
 * clique [P,ld] (may be NULL) receives the clique as ascending match positions, -1 past its end; clique_size [P] and
 * exact [P] are required.  No host synchronisation, no float atomics: a pair's result is bit-reproducible and does not
 * depend on the rest of the batch.  workspace >= ri_teaser_workspace_bytes(P, ld) bytes (0 when P <= 0 or ld is outside
 * [1, 32768]), 256-byte aligned.  RI_ERR_BAD_ARG for a non-positive or non-finite noise_bound, cbar2 or inlier_dist,
 * gnc_factor <= 1, max_iterations < 0, max_clique_nodes < 1, or clique_size / exact NULL; RI_ERR_UNSUPPORTED for
 * ld > 32768 or P > 65535; RI_ERR_WORKSPACE for a missing or short workspace. */
size_t ri_teaser_workspace_bytes(int P, int ld);
int ri_teaser_f32(const float* src, const float* tgt, const int* idx1, const int* idx2, const int* count, int P, int n1,
                  int n2, int ld, float noise_bound, float cbar2, float gnc_factor, int max_iterations, float cost_threshold,
                  long long max_clique_nodes, float inlier_dist, float* T, int* inliers, int* clique, int* clique_size,
                  int* exact, void* workspace, size_t workspace_bytes, void* stream);

/* ---- FPFH descriptors (SURVEY.md 8f, row f8)-------------------------------------------------------------------------
 * Open3D's compute_fpfh_feature with KDTreeSearchParamHybrid(radius, max_nn) (Rusu, Blodow, Beetz, ICRA 2009;
 * pipelines/registration/Feature.cpp), B clouds per call.  xyz [B,3,N], normals [B,3,N] fp32 (used as given, not
 * renormalised); radius > 0 (+inf = plain k-NN), 1 <= max_nn <= 128.  For each point q:
 *   neighbours  the list of ri_estimate_normals_f32: the max_nn smallest keys (d, index) with d < min(r2, 10000), q included,
 *               d = fma(dz,dz, fma(dy,dy, dx*dx)), d* = q - p in fp32 — the first max_nn entries of the k-NN (ri_knn_f32,
 *               k = max_nn) whose distance passes the cut.  n = its length.  Nothing within the cap is dropped.
 *   pair        feature (f0, f1, f2) of (p1, n1) with (p2, n2), fp64 from the fp32 inputs, each operation rounded:
 *               dp = p2 - p1, L = |dp| (L == 0: (0,0,0)); a1 = n1.dp / L, a2 = n2.dp / L; if acos|a1| > acos|a2| swap n1
 *               and n2, negate dp, f2 = -a2, else f2 = a1; v = dp x n1' (|v| == 0: (0,0,0)), v /= |v|, w = n1' x v;
 *               f1 = v.n2', f0 = atan2(w.n2', n1'.n2').  Dot products are (x*x' + y*y') + z*z'.
 *   SPFH        n <= 1: zeros.  Otherwise the pair features of (q, n_q) with list positions k = 1 .. n-1 (position 0 is
 *               skipped whatever it holds) binned as b0 = floor(11 (f0 + pi) / (2 pi)), b1 = floor(11 (f1 + 1) * 0.5),
 *               b2 = floor(11 (f2 + 1) * 0.5), each clamped to [0, 10]; counts c_j over 3 x 11 bins;
 *               spfh_j = c_j * (100 / (n - 1)) in fp64 (Open3D adds 100 / (n - 1) c_j times: a few fp64 ulp apart).
 *   FPFH        n <= 1: zeros.  Otherwise for k = 1 .. n-1 in list order: w_k = |p_k - q|^2 in fp64 from the fp32
 *               coordinates (skipped when 0); val = spfh_j(p_k) / w_k is added to feat_j and to sum[j / 11]; then
 *               fpfh_j = feat_j * (sum != 0 ? 100 / sum : 0) + spfh_j(q), rounded to fp32.  An exact duplicate of q with a
 *               lower index sorts before q, so q meets itself at a later position: pair feature (0,0,0), weight skipped.
 * Outputs fpfh [B,33,N] fp32; unless NULL, spfh [B,33,N] fp32 (c = round(spfh * (n - 1) / 100) recovers the counts) and
 * counts [B,N] int32 = n.  No host synchronisation, no float atomics: a cloud's result does not depend on the rest of the
 * batch and is bit-reproducible.  workspace >= ri_fpfh_workspace_bytes(B, N, max_nn) bytes (the grid, the lists and the
 * packed bin counts), 16-byte aligned.  RI_ERR_BAD_ARG for radius <= 0 or NaN or max_nn <= 0; RI_ERR_UNSUPPORTED for
 * max_nn > 128 or B > 65535. */
size_t ri_fpfh_workspace_bytes(int B, int N, int max_nn);
int ri_compute_fpfh_f32(const float* xyz, const float* normals, int B, int N, float radius, int max_nn, float* fpfh,
                        float* spfh, int* counts, void* workspace, size_t workspace_bytes, void* stream);

/* ---- farthest point sampling over variable-length clouds (SURVEY.md 8f, row f12) -------------------------------------
 * The reference's furthest_point_sampling (backend name; F.furthest_point_sample) and Open3D's farthest_point_down_sample,
 * B clouds per call.  xyz [B,3,N] fp32; lengths [B] int32 (device) or NULL: cloud b uses its first n_b = lengths[b]
 * points, 0 <= n_b <= N (values outside are clamped), NULL means n_b = N; m >= 1.  Per cloud, with dist[i] = +inf for
 * i < n_b and s = 0:
 *   for k in 0 .. m-1:  idx[b,k] = s;  q = s;  best = 0
 *                       for i in 0 .. n_b-1 ascending:  d = (dx*dx + dy*dy) + dz*dz in fp64, dx = (double)x_i - (double)x_q,
 *                                                       each operation rounded (no contraction)
 *                                                       dist[i] = d < dist[i] ? d : dist[i]
 *                                                       if dist[i] > best: best = dist[i], s = i
 * So the lowest index wins ties, s is unchanged when every dist is 0 (once every distinct point is taken, or m > n_b, the
 * last index repeats), a duplicate of a taken point is never taken, and n_b = 0 gives all -1.  Non-finite coordinates
 * follow the rule literally (a NaN point keeps dist = +inf; once taken it repeats).  tests/fps_oracle.py replays it.
 * Deltas.  Open3D (recalled, unverified): the same loop from index 0 with fp64 distances, std::min and a strict > from
 * max_dist = 0, but it raises when num_samples > n, and Eigen's squaredNorm may sum in another order, so near-ties can
 * split differently.  The reference kernel (not checked here, unverified): fp32 distances, ties broken in its reduction
 * tree's order and, if it follows pointnet2, points with |p|^2 <= 1e-3 skipped; no parity with it is claimed.
 * Output idx [B,m] int32.  Points past n_b are never read.  No float atomics, no workspace, no host synchronisation: a
 * cloud's result is bit-reproducible and does not depend on the rest of the batch or on its padding.  RI_ERR_BAD_ARG for
 * B < 0, N < 0, m < 1 or a NULL pointer; RI_ERR_UNSUPPORTED for N > RI_FPS_MAX_POINTS, or N > 65536 on a device that
 * cannot schedule a 16-CTA cluster (clouds up to 65536 points run on portable clusters of at most 8 CTAs). */
#define RI_FPS_MAX_POINTS 131072
int ri_furthest_point_sample_f32(const float* xyz, const int* lengths, int B, int N, int m, int* idx, void* stream);

/* ---- ISS keypoints (SURVEY.md 8f, row f13) ---------------------------------------------------------------------------
 * Intrinsic Shape Signatures (Zhong, ICCV Workshops 2009) as Open3D's geometry::keypoint::ComputeISSKeypoints computes
 * them, B clouds per call.  xyz [B,3,N] fp32; gamma a HOST pointer to {gamma_21, gamma_32} in fp64 (read during the call:
 * Open3D's thresholds are doubles).  tests/iss_oracle.py replays every step.
 *   distance    d(q,p) = fma(dz,dz, fma(dy,dy, dx*dx)), d* = q - p in fp32 (the expression of ri_estimate_normals_f32);
 *               N_r(q) = {p : d(q,p) < r*r}, r*r rounded to fp32, q itself included.  A point with a non-finite coordinate
 *               is nobody's neighbour, has s = 0 and is never a keypoint.
 *   radii       salient_radius == 0 or non_max_radius == 0: both come from the resolution res_b = the mean, over the
 *               cloud's finite points, of sqrt((double)d) to the nearest other point (the second key of the k = 2 list:
 *               0 for a duplicate), summed in fp64 in a fixed order; r_s = (float)(6 res_b), r_nm = (float)(4 res_b).
 *               Computed on the device per cloud.  A cloud with fewer than 2 finite points gets radii 0 and no keypoints.
 *               Otherwise both radii must be finite and > 0.
 *   saliency    s(q) = 0 unless |N_rs(q)| >= min_neighbors; C = the population covariance of N_rs(q) from p - q in fp64,
 *               summed in an order that depends on the cloud alone; C is not skipped (skipped: every |C_ij| <= 1e-12
 *               (Eigen's isZero()), an entry not finite, or trace(C) not positive); its eigenvalues e1 >= e2 >= e3 (fp64
 *               Jacobi on C / trace(C), scaled back) pass e2 / e1 < gamma_21 && e3 / e2 < gamma_32 (fp64 divisions, a NaN
 *               ratio fails).  Then s(q) = e3.
 *   keypoint    s(q) > 0, |N_rnm(q)| >= min_neighbors, and no p in N_rnm(q) has s(p) > s(q) (ties keep both points, as
 *               Open3D's IsLocalMaxima).
 * Outputs idx [B,N] int32: row b holds the keypoints in ascending index in idx[b, 0:count[b]], -1 after them (the convention
 * of the matcher's idx1 / count); count [B] int32; unless NULL, saliency [B,N] fp64 = s and radii [B,2] fp32 = (r_s, r_nm)
 * as used.  No float atomics, no host synchronisation: a cloud's result is bit-reproducible and does not depend on the
 * rest of the batch.
 * Deltas from Open3D (read from its source, not verified against a build): the keypoints come back as indices in ascending
 * order (Open3D pushes them in an unspecified OpenMP order and returns a point cloud); the radius cut is strict; the moments
 * are centred on q instead of raw cumulants (differs by rounding only); a cloud with fewer than 2 (finite) points and
 * automatic radii has no keypoints (Open3D reads out of bounds there) and non-finite points are skipped in the resolution.
 * workspace >= ri_iss_workspace_bytes(B, N) bytes (0 when B <= 0), 256-byte aligned.  RI_ERR_BAD_ARG for B < 0, N < 0, a
 * radius that is negative or not finite, a NULL gamma, gamma_21 or gamma_32 not > 0, min_neighbors < 1, or a NULL
 * idx / count / xyz that the call would use; RI_ERR_UNSUPPORTED for B > 65535 or B * N > INT_MAX; RI_ERR_WORKSPACE for a missing, misaligned
 * or short workspace.  Every check happens before any launch. */
size_t ri_iss_workspace_bytes(int B, int N);
int ri_iss_keypoints_f32(const float* xyz, int B, int N, float salient_radius, float non_max_radius, const double* gamma,
                         int min_neighbors, int* idx, int* count, double* saliency, float* radii, void* workspace,
                         size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RI_B200_H */
