// pose.cu — correspondences -> rigid pose -> registration metrics on the GPU, sm_100a  (SURVEY.md §8 row f3).
//
// In the reference this step leaves the GPU: the meter copies the descriptors to the host, matches them with numpy
// (datasets/deepgmr_mn40.py:232-244, row a11 — csrc/matcher.cu here) and hands the matches to a third-party solver, one
// pair at a time: Open3D RANSAC / FGR (utils/open3d_func.py:34-75) or TEASER++ (deepgmr_mn40.py:175-230), then scores
// the estimate with RE_TE_one_pair (deepgmr_mn40.py:152-164) and a point RMSE (:121-126).  Open3D and TEASER++ are
// not part of the reference tree (un-vendored, versions unpinned), so there is no arithmetic to be bit-exact with; what
// is kept is the CONTRACT of the RANSAC configuration the reference passes to Open3D (open3d_func.py:43-49):
//   * 3-point minimal samples drawn from the feature correspondences (here: the mutual matches of row a11),
//   * hypothesis pruning by edge-length similarity 0.9 (CorrespondenceCheckerBasedOnEdgeLength) and by the residual of
//     the sample itself (CorrespondenceCheckerBasedOnDistance(voxel_size)),
//   * validation = number of correspondences within `voxel_size` of their partner, `max_iter` hypotheses,
//   * point-to-point least squares (TransformationEstimationPointToPoint(False): rotation + translation, no scale),
// and the metric formulas, which are restated exactly (fp64).
//
// Kernels
//   pose_ransac_kernel   grid (hypothesis blocks, pairs).  The pair's matched coordinates are staged in shared memory
//                        once per CTA; one thread = one hypothesis: counter-based RNG -> 3 distinct matches -> checks ->
//                        rotation from the two triangles' orthonormal frames -> inlier count over all matches -> 64-bit
//                        atomicMax of (inliers << 32 | ~hypothesis id)  (deterministic: lowest id wins ties).
//   pose_refine_kernel   one CTA per pair: rebuilds the winning hypothesis from its id, then `iters` rounds of
//                        {inlier set under the current pose -> centroids and 3x3 cross-covariance by block reduction in
//                        fp64 -> Horn's closed form: the unit quaternion maximising q^T N q, found by cyclic Jacobi
//                        sweeps on the symmetric 4x4 N -> R, t}.  Writes T [4,4] (row-major, fp32) and the inlier count.
//   pose_metrics_kernel  one CTA per pair: RRE (degrees), RTE, RMSE exactly as the reference's meter computes them.
#include "ri_common.cuh"
#include "rigid.cuh"
#include "matches.cuh"

namespace {

constexpr int kHypThreads = 128;
constexpr int kRefThreads = 256;
constexpr int kMaxMatches = 4096;        // matched coordinates staged per pair at a time: 6 floats each (96 KB); more
                                         // matches are processed in chunks of this size

// three distinct indices in [0, M), M >= 3, from (seed, pair, hypothesis)
__device__ __forceinline__ void sample3(uint64_t seed, int pair, int hyp, int M, int& i0, int& i1, int& i2)
{
    const uint64_t r0 = mix64(seed ^ ((uint64_t)pair << 32) ^ (uint64_t)(uint32_t)hyp);
    const uint64_t r1 = mix64(r0), r2 = mix64(r1);
    i0 = (int)(r0 % (uint64_t)M);
    i1 = (int)(r1 % (uint64_t)(M - 1)); if (i1 >= i0) ++i1;
    i2 = (int)(r2 % (uint64_t)(M - 2));
    const int lo = min(i0, i1), hi = max(i0, i1);
    if (i2 >= lo) ++i2;
    if (i2 >= hi) ++i2;
}

__device__ __forceinline__ float3 f3sub(float3 a, float3 b) { return make_float3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float f3dot(float3 a, float3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ float3 f3cross(float3 a, float3 b)
{
    return make_float3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ float3 f3scale(float3 a, float s) { return make_float3(a.x * s, a.y * s, a.z * s); }

// orthonormal frame of a triangle; false if (nearly) degenerate
__device__ __forceinline__ bool tri_frame(float3 p0, float3 p1, float3 p2, float3& e1, float3& e2, float3& e3)
{
    const float3 u = f3sub(p1, p0), v = f3sub(p2, p0);
    const float nu = sqrtf(f3dot(u, u));
    if (!(nu > 1e-6f)) return false;
    e1 = f3scale(u, 1.0f / nu);
    const float3 w = f3sub(v, f3scale(e1, f3dot(v, e1)));
    const float nw = sqrtf(f3dot(w, w));
    if (!(nw > 1e-6f)) return false;
    e2 = f3scale(w, 1.0f / nw);
    e3 = f3cross(e1, e2);
    return true;
}

// stage matches [base, base + kMaxMatches) of [0, M) into A, Bm (the whole pair when M <= kMaxMatches); returns their number
__device__ __forceinline__ int stage_matches(const PairMatches& pm, int base, int M, float3* A, float3* Bm)
{
    const int len = min(M - base, kMaxMatches);
    for (int m = threadIdx.x; m < len; m += blockDim.x) pm.load(base + m, A[m], Bm[m]);
    __syncthreads();
    return len;
}

// hypothesis of one minimal sample: checks of open3d_func.py:46-48, rotation from the two triangle frames
__device__ __forceinline__ bool hypothesis(float3 a0, float3 a1, float3 a2, float3 b0, float3 b1, float3 b2, float edge_sim,
                                           float thresh, Rt& T)
{
    // edge-length similarity: every edge of the source triangle within [sim, 1/sim] of the target's
    const float ea[3] = {sqrtf(f3dot(f3sub(a0, a1), f3sub(a0, a1))), sqrtf(f3dot(f3sub(a1, a2), f3sub(a1, a2))),
                         sqrtf(f3dot(f3sub(a2, a0), f3sub(a2, a0)))};
    const float eb[3] = {sqrtf(f3dot(f3sub(b0, b1), f3sub(b0, b1))), sqrtf(f3dot(f3sub(b1, b2), f3sub(b1, b2))),
                         sqrtf(f3dot(f3sub(b2, b0), f3sub(b2, b0)))};
#pragma unroll
    for (int e = 0; e < 3; ++e)
        if (!(ea[e] >= eb[e] * edge_sim && eb[e] >= ea[e] * edge_sim)) return false;
    float3 s1, s2, s3, t1, t2, t3;
    if (!tri_frame(a0, a1, a2, s1, s2, s3) || !tri_frame(b0, b1, b2, t1, t2, t3)) return false;
    // R = [t1 t2 t3] [s1 s2 s3]^T
    T.r[0] = t1.x * s1.x + t2.x * s2.x + t3.x * s3.x; T.r[1] = t1.x * s1.y + t2.x * s2.y + t3.x * s3.y; T.r[2] = t1.x * s1.z + t2.x * s2.z + t3.x * s3.z;
    T.r[3] = t1.y * s1.x + t2.y * s2.x + t3.y * s3.x; T.r[4] = t1.y * s1.y + t2.y * s2.y + t3.y * s3.y; T.r[5] = t1.y * s1.z + t2.y * s2.z + t3.y * s3.z;
    T.r[6] = t1.z * s1.x + t2.z * s2.x + t3.z * s3.x; T.r[7] = t1.z * s1.y + t2.z * s2.y + t3.z * s3.y; T.r[8] = t1.z * s1.z + t2.z * s2.z + t3.z * s3.z;
    const float3 ca = f3scale(make_float3(a0.x + a1.x + a2.x, a0.y + a1.y + a2.y, a0.z + a1.z + a2.z), 1.0f / 3.0f);
    const float3 cb = f3scale(make_float3(b0.x + b1.x + b2.x, b0.y + b1.y + b2.y, b0.z + b1.z + b2.z), 1.0f / 3.0f);
    T.t[0] = cb.x - (T.r[0] * ca.x + T.r[1] * ca.y + T.r[2] * ca.z);
    T.t[1] = cb.y - (T.r[3] * ca.x + T.r[4] * ca.y + T.r[5] * ca.z);
    T.t[2] = cb.z - (T.r[6] * ca.x + T.r[7] * ca.y + T.r[8] * ca.z);
    // the sample itself must agree with the hypothesis
    const float t2h = thresh * thresh;
    const float3 as[3] = {a0, a1, a2}, bs[3] = {b0, b1, b2};
#pragma unroll
    for (int e = 0; e < 3; ++e) {
        const float dx = T.r[0] * as[e].x + T.r[1] * as[e].y + T.r[2] * as[e].z + T.t[0] - bs[e].x;
        const float dy = T.r[3] * as[e].x + T.r[4] * as[e].y + T.r[5] * as[e].z + T.t[1] - bs[e].y;
        const float dz = T.r[6] * as[e].x + T.r[7] * as[e].y + T.r[8] * as[e].z + T.t[2] - bs[e].z;
        if (!(dx * dx + dy * dy + dz * dz < t2h)) return false;
    }
    return true;
}

// hypothesis h of pair p: its sample3 triple, read from shared memory when the whole pair is staged, else from global
__device__ __forceinline__ bool sample_hypothesis(const PairMatches& pm, const float3* A, const float3* Bm, int M,
                                                  unsigned long long seed, int p, int h, float edge_sim, float thresh, Rt& T)
{
    int i0, i1, i2;
    sample3(seed, p, h, M, i0, i1, i2);
    float3 a0, a1, a2, b0, b1, b2;
    if (M <= kMaxMatches) { a0 = A[i0]; a1 = A[i1]; a2 = A[i2]; b0 = Bm[i0]; b1 = Bm[i1]; b2 = Bm[i2]; }
    else { pm.load(i0, a0, b0); pm.load(i1, a1, b1); pm.load(i2, a2, b2); }
    return hypothesis(a0, a1, a2, b0, b1, b2, edge_sim, thresh, T);
}

// one block-strided pass over all M matches of the pair: f(a, b) for each.  `staged` is the base of the chunk held in
// A / Bm; with M <= kMaxMatches that is the whole pair and nothing is restaged, otherwise the pass walks the chunks in
// order and every thread of the block takes part in each restaging barrier.
template <class F>
__device__ __forceinline__ void for_each_match(const PairMatches& pm, int M, int& staged, float3* A, float3* Bm, F f)
{
    for (int base = 0; base < M; base += kMaxMatches) {
        if (base != staged) { __syncthreads(); stage_matches(pm, base, M, A, Bm); staged = base; }
        const int len = min(M - base, kMaxMatches);
        for (int m = threadIdx.x; m < len; m += blockDim.x) f(A[m], Bm[m]);
    }
}

__global__ void __launch_bounds__(kHypThreads)
pose_ransac_kernel(const float* __restrict__ src, const float* __restrict__ tgt, const int* __restrict__ idx1,
                   const int* __restrict__ idx2, const int* __restrict__ count, int n1, int n2, int ld, int hyps,
                   float thresh, float edge_sim, unsigned long long seed, unsigned long long* __restrict__ best)
{
    extern __shared__ float3 pose_smem[];
    const int p = blockIdx.y;
    float3* A = pose_smem;
    float3* Bm = pose_smem + min(ld, kMaxMatches);
    const PairMatches pm(src, tgt, idx1, idx2, p, n1, n2, ld);
    const int M = match_count(count, p, ld);
    int len = stage_matches(pm, 0, M, A, Bm);
    const int h = blockIdx.x * kHypThreads + threadIdx.x;
    if (M < 3) return;                                   // uniform over the block
    Rt T;
    const bool valid = h < hyps && sample_hypothesis(pm, A, Bm, M, seed, p, h, edge_sim, thresh, T);
    const float t2h = thresh * thresh;
    int n = 0;
    for (int base = 0;;) {                               // every thread walks the chunks: the barriers are block-wide
        if (valid)
            for (int m = 0; m < len; ++m) n += inlier(T, A[m], Bm[m], t2h) ? 1 : 0;
        base += kMaxMatches;
        if (base >= M) break;
        __syncthreads();
        len = stage_matches(pm, base, M, A, Bm);
    }
    if (valid) atomicMax(best + p, ((unsigned long long)(unsigned)n << 32) | (unsigned long long)(0xffffffffu - (unsigned)h));
}

// use_all != 0: plain least squares over ALL matches (the Kabsch solve alone; no RANSAC seed needed)
__global__ void __launch_bounds__(kRefThreads)
pose_refine_kernel(const float* __restrict__ src, const float* __restrict__ tgt, const int* __restrict__ idx1,
                   const int* __restrict__ idx2, const int* __restrict__ count, int n1, int n2, int ld,
                   float thresh, float edge_sim, unsigned long long seed, const unsigned long long* __restrict__ best,
                   int iters, int use_all, float* __restrict__ T_out, int* __restrict__ inliers_out)
{
    extern __shared__ float3 pose_smem[];
    __shared__ double red[(kRefThreads / 32) * 9];
    __shared__ Rt Tcur;
    __shared__ int ok, posed;
    __shared__ double cen[6];
    const int p = blockIdx.x;
    float3* A = pose_smem;
    float3* Bm = pose_smem + min(ld, kMaxMatches);
    const PairMatches pm(src, tgt, idx1, idx2, p, n1, n2, ld);
    const int M = match_count(count, p, ld);
    stage_matches(pm, 0, M, A, Bm);
    int staged = 0;
    const float t2h = thresh * thresh;
    if (threadIdx.x == 0) {
        ok = 0;
#pragma unroll
        for (int i = 0; i < 9; ++i) Tcur.r[i] = (i % 4 == 0) ? 1.f : 0.f;
        Tcur.t[0] = Tcur.t[1] = Tcur.t[2] = 0.f;
        if (M >= 3) {
            if (use_all) ok = 1;
            else {
                const unsigned long long key = best[p];
                if (key != 0ull) {
                    const int h = (int)(0xffffffffu - (unsigned)(key & 0xffffffffull));
                    Rt T;
                    if (sample_hypothesis(pm, A, Bm, M, seed, p, h, edge_sim, thresh, T)) { Tcur = T; ok = 1; }
                }
            }
        }
        posed = ok;                                      // a pose exists; ok may still drop during the refit
    }
    __syncthreads();
    for (int it = 0; it < iters && ok; ++it) {
        const Rt T = Tcur;
        double s[7] = {0, 0, 0, 0, 0, 0, 0};
        for_each_match(pm, M, staged, A, Bm, [&](float3 a, float3 b) {
            if (use_all || inlier(T, a, b, t2h)) {
                s[0] += 1.0; s[1] += a.x; s[2] += a.y; s[3] += a.z; s[4] += b.x; s[5] += b.y; s[6] += b.z;
            }
        });
        block_sum<7>(s, red);
        if (threadIdx.x == 0) {
            if (s[0] < 3.0) ok = 0;
            else for (int i = 0; i < 6; ++i) cen[i] = s[1 + i] / s[0];
        }
        __syncthreads();
        if (!ok) break;
        double h9[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        const double cax = cen[0], cay = cen[1], caz = cen[2], cbx = cen[3], cby = cen[4], cbz = cen[5];
        for_each_match(pm, M, staged, A, Bm, [&](float3 a, float3 b) {
            if (use_all || inlier(T, a, b, t2h)) {
                const double ax = a.x - cax, ay = a.y - cay, az = a.z - caz;
                const double bx = b.x - cbx, by = b.y - cby, bz = b.z - cbz;
                h9[0] += ax * bx; h9[1] += ax * by; h9[2] += ax * bz;
                h9[3] += ay * bx; h9[4] += ay * by; h9[5] += ay * bz;
                h9[6] += az * bx; h9[7] += az * by; h9[8] += az * bz;
            }
        });
        block_sum<9>(h9, red);
        if (threadIdx.x == 0) {
            double R[9];
            horn_rotation(h9, R);
#pragma unroll
            for (int i = 0; i < 9; ++i) Tcur.r[i] = (float)R[i];
            Tcur.t[0] = (float)(cbx - (R[0] * cax + R[1] * cay + R[2] * caz));
            Tcur.t[1] = (float)(cby - (R[3] * cax + R[4] * cay + R[5] * caz));
            Tcur.t[2] = (float)(cbz - (R[6] * cax + R[7] * cay + R[8] * caz));
        }
        __syncthreads();
    }
    // final inlier count under the returned pose (also when a refit round fell below 3 inliers and kept the pose
    // that round was evaluated under); no pose at all -> identity, 0 inliers
    const Rt T = Tcur;
    double c1[1] = {0};
    for_each_match(pm, M, staged, A, Bm, [&](float3 a, float3 b) { c1[0] += inlier(T, a, b, t2h) ? 1.0 : 0.0; });
    block_sum<1>(c1, red);
    if (threadIdx.x == 0) {
        float* O = T_out + (size_t)p * 16;
        O[0] = T.r[0]; O[1] = T.r[1]; O[2] = T.r[2]; O[3] = T.t[0];
        O[4] = T.r[3]; O[5] = T.r[4]; O[6] = T.r[5]; O[7] = T.t[1];
        O[8] = T.r[6]; O[9] = T.r[7]; O[10] = T.r[8]; O[11] = T.t[2];
        O[12] = 0.f; O[13] = 0.f; O[14] = 0.f; O[15] = 1.f;
        inliers_out[p] = posed ? (int)c1[0] : 0;
    }
}

// RE_TE_one_pair (deepgmr_mn40.py:152-164) and the point RMSE of MeterModelNet40_registration.update (:121-126):
//   A = (trace(gt_R^T est_R) - 1) / 2 clamped to [-1, 1];  rre = degrees(|acos(A)|);  rte = |gt_t - est_t|;
//   rmse = mean_i | (pts_i est_R^T + est_t) - (pts_i gt_R^T + gt_t) |
__global__ void __launch_bounds__(kRefThreads)
pose_metrics_kernel(const float* __restrict__ gt, const float* __restrict__ est, const float* __restrict__ pts, int n,
                    double* __restrict__ out)
{
    __shared__ double red[(kRefThreads / 32) * 1];
    const int p = blockIdx.x;
    const float* G = gt + (size_t)p * 16;
    const float* E = est + (size_t)p * 16;
    const float* X = pts + (size_t)p * n * 3;
    double s[1] = {0};
    for (int i = threadIdx.x; i < n; i += kRefThreads) {
        const double x = X[3 * i], y = X[3 * i + 1], z = X[3 * i + 2];
        const double dx = (E[0] * x + E[1] * y + E[2] * z + E[3]) - (G[0] * x + G[1] * y + G[2] * z + G[3]);
        const double dy = (E[4] * x + E[5] * y + E[6] * z + E[7]) - (G[4] * x + G[5] * y + G[6] * z + G[7]);
        const double dz = (E[8] * x + E[9] * y + E[10] * z + E[11]) - (G[8] * x + G[9] * y + G[10] * z + G[11]);
        s[0] += sqrt(dx * dx + dy * dy + dz * dz);
    }
    block_sum<1>(s, red);
    if (threadIdx.x == 0) {
        double tr = 0.0;                                       // trace(gt_R^T est_R) = sum_ij G_ij E_ij
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) tr += (double)G[4 * i + j] * (double)E[4 * i + j];
        double a = (tr - 1.0) / 2.0;
        a = a > 1.0 ? 1.0 : (a < -1.0 ? -1.0 : a);
        const double tx = (double)G[3] - E[3], ty = (double)G[7] - E[7], tz = (double)G[11] - E[11];
        out[3 * p + 0] = fabs(acos(a)) * (180.0 / 3.14159265358979323846);
        out[3 * p + 1] = sqrt(tx * tx + ty * ty + tz * tz);
        out[3 * p + 2] = n > 0 ? s[0] / n : 0.0;
    }
}

}  // namespace

// src [P,n1,3], tgt [P,n2,3] point-major fp32 (the (b,n,3) arrays the reference's meter receives); idx1 / idx2 [P,ld] and
// count [P]: the mutual matches as ri_mutual_nn_tf32x3 returns them (ld = n1).  hyps = 0 skips RANSAC and solves the least
// squares over all matches (Kabsch).  T [P,4,4] row-major fp32 maps src onto tgt; inliers [P].  best [P] uint64 scratch.
extern "C" int ri_pose_from_matches_f32(const float* src, const float* tgt, const int* idx1, const int* idx2, const int* count,
                                        int P, int n1, int n2, int ld, int hyps, float inlier_dist, float edge_similarity,
                                        int refine_iters, unsigned long long seed, float* T, int* inliers,
                                        unsigned long long* best, void* stream)
{
    if (P < 0 || n1 <= 0 || n2 <= 0 || ld <= 0 || hyps < 0 || refine_iters < 1 || !(inlier_dist > 0.f)) return RI_ERR_BAD_ARG;
    if (P > 65535) return RI_ERR_UNSUPPORTED;
    if (P == 0) return RI_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int cap = ld < kMaxMatches ? ld : kMaxMatches;
    const size_t smem = (size_t)cap * 2 * sizeof(float3);
    cudaError_t e;
    RI_KERNEL_SETUP(pose_ransac_kernel, true, -1);
    RI_KERNEL_SETUP(pose_refine_kernel, true, -1);
    if (hyps > 0) {
        if (best == nullptr) return RI_ERR_WORKSPACE;
        e = cudaMemsetAsync(best, 0, (size_t)P * sizeof(unsigned long long), st);
        if (e != cudaSuccess) return (int)e;
        dim3 grid((hyps + kHypThreads - 1) / kHypThreads, P);
        pose_ransac_kernel<<<grid, kHypThreads, smem, st>>>(src, tgt, idx1, idx2, count, n1, n2, ld, hyps, inlier_dist,
                                                            edge_similarity, seed, best);
        RI_LAUNCH_CHECK();
    }
    pose_refine_kernel<<<P, kRefThreads, smem, st>>>(src, tgt, idx1, idx2, count, n1, n2, ld, inlier_dist, edge_similarity,
                                                     seed, best, hyps > 0 ? refine_iters : 1, hyps > 0 ? 0 : 1, T, inliers);
    RI_LAUNCH_CHECK();
    return RI_OK;
}

// gt, est [P,4,4] row-major fp32, pts [P,n,3] -> out [P,3] fp64 = (rre degrees, rte, rmse)
extern "C" int ri_registration_metrics_f32(const float* gt, const float* est, const float* pts, int P, int n, double* out,
                                           void* stream)
{
    if (P < 0 || n < 0) return RI_ERR_BAD_ARG;
    if (P == 0) return RI_OK;
    pose_metrics_kernel<<<P, kRefThreads, 0, (cudaStream_t)stream>>>(gt, est, pts, n, out);
    RI_LAUNCH_CHECK();
    return RI_OK;
}
