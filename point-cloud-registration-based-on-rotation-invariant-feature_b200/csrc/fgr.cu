// fgr.cu — Fast Global Registration (Zhou, Park, Koltun, ECCV 2016) over the mutual matches, P pairs per launch, sm_100a
// (SURVEY.md §8 row f7).
//
// The reference's meter can hand its matches to Open3D's registration_fgr_based_on_feature_matching instead of RANSAC
// (utils/open3d_func.py:50-62).  Open3D is not part of the reference tree, so what is kept is the contract of that solver,
// restated in include/ri_b200.h (ri_fgr_f32) and DESIGN.md §8:
//   * the tuple test of AdvancedMatching: 100 M random 3-match trials, accepted when all three edge lengths agree within
//     tuple_scale; the first max_tuples accepted trials, in trial order, form the correspondence list;
//   * NormalizePointCloud: both clouds centred on their means and divided by the largest centred norm (or not divided,
//     with use_absolute_scale, where that norm starts the GNC parameter instead);
//   * OptimizePairwiseRegistration: `iterations` Gauss-Newton steps of the Geman-McClure objective with graduated
//     non-convexity, moving the normalised target onto the normalised source;
//   * GetInvTransformationOriginalScale: back to original units and inverted, so T maps src onto tgt.
//
// Kernel
//   fgr_kernel  one CTA per pair.  Tuple test: the block evaluates kChunk trials at a time (kTrialsPerThread consecutive
//               trials per thread), then an ordered block scan over the accept counts gives every accepted trial its rank,
//               so the list is the sequential loop's.  The edge lengths and their comparisons are spelled with __d*_rn
//               intrinsics (no contraction), so the list is bit-exact.  Means and scale by block reductions in fp64.  The
//               list's matched coordinates are staged in shared memory up to kStage entries; later entries are gathered
//               from global memory in every iteration.  Each GNC iteration accumulates the moments of J^T J and J^T r in
//               fp64 per thread, reduces them in a fixed order (block_sum), and thread 0 solves the 6x6 system and composes
//               T' in shared memory.  No float atomics: a pair's result is bit-reproducible and independent of the batch.
#include "ri_common.cuh"
#include "rigid.cuh"
#include "matches.cuh"

#include <limits.h>

namespace {

constexpr int kThreads = 256;
constexpr int kTrialsPerThread = 4;
constexpr int kChunk = kThreads * kTrialsPerThread;
constexpr int kStage = 3072;     // list entries staged in shared memory (a, b: 24 bytes each, 72 KB), the default list of
                                 // 3 x 1000 tuples; entries past it are read through the match lists in every iteration
constexpr int kMinCorr = 10;     // OptimizePairwiseRegistration returns the identity for fewer correspondences

struct FgrParams {
    double max_corr_dist, division_factor, tuple_scale;
    int iterations, use_absolute_scale, decrease_mu, tuple_test, max_tuples;
};

__device__ __forceinline__ bool edge_ok(double la, double lb, double s)
{
    return __dmul_rn(la, s) < lb && lb < __ddiv_rn(la, s);
}

// trial t of pair p: three independent match positions (a repeated one gives a zero edge, which fails the strict test)
__device__ __forceinline__ bool tuple_trial(const PairMatches& pm, unsigned long long seed, int p, uint32_t t, int M,
                                            double s, int& i0, int& i1, int& i2)
{
    const uint64_t r0 = mix64(seed ^ ((uint64_t)p << 32) ^ (uint64_t)t);
    const uint64_t r1 = mix64(r0), r2 = mix64(r1);
    i0 = (int)(r0 % (uint64_t)M);
    i1 = (int)(r1 % (uint64_t)M);
    i2 = (int)(r2 % (uint64_t)M);
    float3 a0, a1, a2, b0, b1, b2;
    pm.load(i0, a0, b0); pm.load(i1, a1, b1); pm.load(i2, a2, b2);
    return edge_ok(edge_len(a0, a1), edge_len(b0, b1), s) && edge_ok(edge_len(a1, a2), edge_len(b1, b2), s) &&
           edge_ok(edge_len(a2, a0), edge_len(b2, b0), s);
}

__global__ void __launch_bounds__(kThreads, 2)
fgr_kernel(const float* __restrict__ src, const float* __restrict__ tgt, const int* __restrict__ idx1,
           const int* __restrict__ idx2, const int* __restrict__ count, int n1, int n2, int ld, FgrParams o,
           unsigned long long seed, float inlier_dist, int stage_cap, float* __restrict__ T_out,
           int* __restrict__ inliers_out, int* corr, int* __restrict__ ncorr_out)
{
    extern __shared__ float3 fgr_smem[];
    __shared__ double red[(kThreads / 32) * 16];
    __shared__ int wsum[kThreads / 32];
    __shared__ double mu[6], norm[3];            // mu_s, mu_t; g, 1/g, par_0
    __shared__ double Tp[12];                    // T' (target -> source, normalised units): R row-major, then t
    __shared__ Rt Tf;
    const int p = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float3* A = fgr_smem;
    float3* Bm = fgr_smem + stage_cap;
    const PairMatches pm(src, tgt, idx1, idx2, p, n1, n2, ld);
    const int M = match_count(count, p, ld);
    int* C = o.tuple_test ? corr + (size_t)p * 3 * o.max_tuples : nullptr;

    // ---- 1. the correspondence list: the first max_tuples accepted trials (positions into the matches), or all M matches
    int L = M;
    if (o.tuple_test) {
        int acc = 0;                                             // accepted tuples so far (uniform over the block)
        const uint64_t trials = M >= 3 ? 100ull * (uint64_t)M : 0;  // with M < 3 every trial repeats an index: none passes
        for (uint64_t base = 0; acc < o.max_tuples && base < trials; base += kChunk) {
            int id[kTrialsPerThread][3];
            unsigned ok = 0;
            int n = 0;
#pragma unroll
            for (int k = 0; k < kTrialsPerThread; ++k) {
                const uint64_t t = base + (uint64_t)(tid * kTrialsPerThread + k);
                if (t < trials && tuple_trial(pm, seed, p, (uint32_t)t, M, o.tuple_scale, id[k][0], id[k][1], id[k][2])) {
                    ok |= 1u << k;
                    ++n;
                }
            }
            int incl = n;                                        // inclusive scan of the accept counts, in trial order
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += v;
            }
            if (lane == 31) wsum[warp] = incl;
            __syncthreads();
            int before = 0, total = 0;
#pragma unroll
            for (int w = 0; w < kThreads / 32; ++w) {
                const int v = wsum[w];
                before += w < warp ? v : 0;
                total += v;
            }
            int rank = acc + before + incl - n;
#pragma unroll
            for (int k = 0; k < kTrialsPerThread; ++k)
                if (ok >> k & 1u) {
                    if (rank < o.max_tuples) {
                        C[3 * (size_t)rank] = id[k][0]; C[3 * (size_t)rank + 1] = id[k][1]; C[3 * (size_t)rank + 2] = id[k][2];
                    }
                    ++rank;
                }
            acc = min(acc + total, o.max_tuples);
            __syncthreads();                                     // wsum is rewritten by the next chunk
        }
        L = 3 * acc;
        for (size_t k = (size_t)L + tid; k < 3 * (size_t)o.max_tuples; k += kThreads) C[k] = -1;
        __syncthreads();                                         // the list is read back by every thread below
    }
    const bool posed = M >= 3 && L >= kMinCorr;

    // ---- 2. NormalizePointCloud: means of all points, scale = the largest centred norm of either cloud (fp64)
    if (posed) {
        const float* S = src + (size_t)p * n1 * 3;
        const float* G = tgt + (size_t)p * n2 * 3;
        double s6[6] = {0, 0, 0, 0, 0, 0};
        for (int i = tid; i < n1; i += kThreads) { s6[0] += S[3 * i]; s6[1] += S[3 * i + 1]; s6[2] += S[3 * i + 2]; }
        for (int i = tid; i < n2; i += kThreads) { s6[3] += G[3 * i]; s6[4] += G[3 * i + 1]; s6[5] += G[3 * i + 2]; }
        block_sum<6>(s6, red);
        if (tid == 0) {
            mu[0] = s6[0] / n1; mu[1] = s6[1] / n1; mu[2] = s6[2] / n1;
            mu[3] = s6[3] / n2; mu[4] = s6[4] / n2; mu[5] = s6[5] / n2;
        }
        __syncthreads();
        double m2 = 0.0;
        for (int i = tid; i < n1; i += kThreads) {
            const double dx = S[3 * i] - mu[0], dy = S[3 * i + 1] - mu[1], dz = S[3 * i + 2] - mu[2];
            m2 = fmax(m2, dx * dx + dy * dy + dz * dz);
        }
        for (int i = tid; i < n2; i += kThreads) {
            const double dx = G[3 * i] - mu[3], dy = G[3 * i + 1] - mu[4], dz = G[3 * i + 2] - mu[5];
            m2 = fmax(m2, dx * dx + dy * dy + dz * dz);
        }
        m2 = block_max(m2, red);
        if (tid == 0) {
            const double scale = sqrt(m2);
            norm[0] = o.use_absolute_scale ? 1.0 : scale;
            norm[1] = 1.0 / norm[0];
            norm[2] = o.use_absolute_scale ? scale : 1.0;
#pragma unroll
            for (int i = 0; i < 12; ++i) Tp[i] = (i == 0 || i == 4 || i == 8) ? 1.0 : 0.0;
        }
        // ---- 3. stage the list's matched coordinates
        const int ns = min(L, stage_cap);
        for (int k = tid; k < ns; k += kThreads) pm.load(C ? C[k] : k, A[k], Bm[k]);
        __syncthreads();
    }

    // ---- 4. OptimizePairwiseRegistration: GNC over the list, T' moves the normalised target onto the normalised source
    if (posed) {
        const int ns = min(L, stage_cap);
        const double msx = mu[0], msy = mu[1], msz = mu[2], mtx = mu[3], mty = mu[4], mtz = mu[5], ig = norm[1];
        double par = norm[2];
        for (int it = 0; it < o.iterations; ++it) {
            if (o.decrease_mu && it % 4 == 0 && par > o.max_corr_dist) par /= o.division_factor;
            const double R0 = Tp[0], R1 = Tp[1], R2 = Tp[2], R3 = Tp[3], R4 = Tp[4], R5 = Tp[5], R6 = Tp[6], R7 = Tp[7],
                         R8 = Tp[8], t0 = Tp[9], t1 = Tp[10], t2 = Tp[11];
            // the distinct sums of w * (J^T J, J^T r) over the three residual rows of every correspondence:
            // w; w q; w (qy^2+qz^2), w (qx^2+qz^2), w (qx^2+qy^2); w qx qy, w qx qz, w qy qz; w (q x r); w r
            double s[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) s[i] = 0.0;
            for (int k = tid; k < L; k += kThreads) {
                float3 a, b;
                if (k < ns) { a = A[k]; b = Bm[k]; }
                else pm.load(C ? C[k] : k, a, b);
                const double px = (a.x - msx) * ig, py = (a.y - msy) * ig, pz = (a.z - msz) * ig;
                const double hx = (b.x - mtx) * ig, hy = (b.y - mty) * ig, hz = (b.z - mtz) * ig;
                const double qx = R0 * hx + R1 * hy + R2 * hz + t0;
                const double qy = R3 * hx + R4 * hy + R5 * hz + t1;
                const double qz = R6 * hx + R7 * hy + R8 * hz + t2;
                const double rx = px - qx, ry = py - qy, rz = pz - qz;
                const double u = par / (rx * rx + ry * ry + rz * rz + par), w = u * u;
                const double wx = w * qx, wy = w * qy, wz = w * qz;
                s[0] += w; s[1] += wx; s[2] += wy; s[3] += wz;
                s[4] += wy * qy + wz * qz; s[5] += wx * qx + wz * qz; s[6] += wx * qx + wy * qy;
                s[7] += wx * qy; s[8] += wx * qz; s[9] += wy * qz;
                s[10] += wz * ry - wy * rz; s[11] += wx * rz - wz * rx; s[12] += wy * rx - wx * ry;
                s[13] += w * rx; s[14] += w * ry; s[15] += w * rz;
            }
            block_sum<16>(s, red);
            if (tid == 0) {
                // rows r_x: J = (0, -qz, qy, -1, 0, 0), r_y: (qz, 0, -qx, 0, -1, 0), r_z: (-qy, qx, 0, 0, 0, -1)
                const double up[21] = {s[4], -s[7], -s[8], 0.0, -s[3], s[2],
                                       s[5], -s[9], s[3], 0.0, -s[1],
                                       s[6], -s[2], s[1], 0.0,
                                       s[0], 0.0, 0.0,
                                       s[0], 0.0,
                                       s[0]};
                const double rhs[6] = {-s[10], -s[11], -s[12], s[13], s[14], s[15]};     // -J^T r
                double x[6];
                if (ldlt_solve6(up, rhs, x, 0.0)) {
                    const double ca = cos(x[0]), sa = sin(x[0]), cb = cos(x[1]), sb = sin(x[1]), cg = cos(x[2]), sg = sin(x[2]);
                    // Rz(x2) Ry(x1) Rx(x0), then T' = [D | x3..5] T'
                    const double D[9] = {cg * cb, cg * sb * sa - sg * ca, cg * sb * ca + sg * sa,
                                         sg * cb, sg * sb * sa + cg * ca, sg * sb * ca - cg * sa,
                                         -sb, cb * sa, cb * ca};
                    double Tc[12];
#pragma unroll
                    for (int i = 0; i < 12; ++i) Tc[i] = Tp[i];
#pragma unroll
                    for (int i = 0; i < 3; ++i) {
#pragma unroll
                        for (int j = 0; j < 3; ++j)
                            Tp[3 * i + j] = D[3 * i] * Tc[j] + D[3 * i + 1] * Tc[3 + j] + D[3 * i + 2] * Tc[6 + j];
                        Tp[9 + i] = D[3 * i] * Tc[9] + D[3 * i + 1] * Tc[10] + D[3 * i + 2] * Tc[11] + x[3 + i];
                    }
                }
            }
            __syncthreads();
        }
    }

    // ---- 5. GetInvTransformationOriginalScale: T_tgt->src = [R' | mu_s - R' mu_t + g t'], returned inverted, in fp32
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 9; ++i) Tf.r[i] = (i % 4 == 0) ? 1.f : 0.f;
        Tf.t[0] = Tf.t[1] = Tf.t[2] = 0.f;
        if (posed) {
            const double g = norm[0];
            double c[3];
#pragma unroll
            for (int i = 0; i < 3; ++i)
                c[i] = mu[i] - (Tp[3 * i] * mu[3] + Tp[3 * i + 1] * mu[4] + Tp[3 * i + 2] * mu[5]) + g * Tp[9 + i];
#pragma unroll
            for (int i = 0; i < 3; ++i) {
#pragma unroll
                for (int j = 0; j < 3; ++j) Tf.r[3 * i + j] = (float)Tp[3 * j + i];
                Tf.t[i] = (float)-(Tp[i] * c[0] + Tp[3 + i] * c[1] + Tp[6 + i] * c[2]);
            }
        }
    }
    __syncthreads();
    const Rt T = Tf;
    double c1[1] = {0};
    if (posed) {
        const float t2h = inlier_dist * inlier_dist;
        for (int m = tid; m < M; m += kThreads) {
            float3 a, b;
            pm.load(m, a, b);
            c1[0] += inlier(T, a, b, t2h) ? 1.0 : 0.0;
        }
    }
    block_sum<1>(c1, red);
    if (tid == 0) {
        float* O = T_out + (size_t)p * 16;
        O[0] = T.r[0]; O[1] = T.r[1]; O[2] = T.r[2]; O[3] = T.t[0];
        O[4] = T.r[3]; O[5] = T.r[4]; O[6] = T.r[5]; O[7] = T.t[1];
        O[8] = T.r[6]; O[9] = T.r[7]; O[10] = T.r[8]; O[11] = T.t[2];
        O[12] = 0.f; O[13] = 0.f; O[14] = 0.f; O[15] = 1.f;
        inliers_out[p] = posed ? (int)c1[0] : 0;
        ncorr_out[p] = L;
    }
}

}  // namespace

extern "C" int ri_fgr_f32(const float* src, const float* tgt, const int* idx1, const int* idx2, const int* count, int P,
                          int n1, int n2, int ld, float max_corr_dist, int iterations, float division_factor,
                          int use_absolute_scale, int decrease_mu, int tuple_test, float tuple_scale, int max_tuples,
                          unsigned long long seed, float inlier_dist, float* T, int* inliers, int* corr, int* ncorr,
                          void* stream)
{
    if (P < 0 || n1 <= 0 || n2 <= 0 || ld <= 0 || !(max_corr_dist > 0.f) || iterations < 0 || !(division_factor > 1.f) ||
        !(tuple_scale > 0.f && tuple_scale <= 1.f) || max_tuples < 1 || !(inlier_dist > 0.f))
        return RI_ERR_BAD_ARG;
    if (tuple_test && corr == nullptr) return RI_ERR_BAD_ARG;
    if (100ull * (unsigned long long)ld >= (1ull << 32) || max_tuples > INT_MAX / 3) return RI_ERR_UNSUPPORTED;
    if (P == 0) return RI_OK;
    const long long list_max = tuple_test ? 3ll * (long long)(max_tuples < 100ll * ld ? max_tuples : 100ll * ld) : ld;
    const int cap = (int)(list_max < kStage ? list_max : kStage);
    const size_t smem = (size_t)cap * 2 * sizeof(float3);
    RI_KERNEL_SETUP(fgr_kernel, true, -1);
    const FgrParams o{(double)max_corr_dist, (double)division_factor, (double)tuple_scale, iterations,
                      use_absolute_scale ? 1 : 0, decrease_mu ? 1 : 0, tuple_test ? 1 : 0, max_tuples};
    fgr_kernel<<<P, kThreads, smem, (cudaStream_t)stream>>>(src, tgt, idx1, idx2, count, n1, n2, ld, o, seed, inlier_dist,
                                                            cap, T, inliers, tuple_test ? corr : nullptr, ncorr);
    RI_LAUNCH_CHECK();
    return RI_OK;
}
