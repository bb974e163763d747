// icp.cu — batched ICP refinement (point-to-point, point-to-plane and generalized / plane-to-plane) and registration
// evaluation, sm_100a (SURVEY.md §8f rows f5, f9 and f11).
//
// Open3D's registration_icp / evaluate_registration (the reference reaches them through utils/open3d_func.py), for P
// independent (source, target) pairs per call, with Open3D's loop per pair:
//   T = init; res = evaluate(T)
//   for i in range(max_iter):
//       U = solve(res.correspondences); T = U T; prev, res = res, evaluate(T)
//       if |prev.fitness - res.fitness| < rel_fitness and |prev.rmse - res.rmse| < rel_rmse: break
//   -> T, res.fitness, res.inlier_rmse, iterations (= updates applied), res.correspondences
//
// Correspondence: q = T s in fp32 from the fp32 rounding of T; the nearest target point with d^2 < r^2 (strict, as the RANSAC
// inlier test of pose.cu), d^2 = fma(dz,dz, fma(dy,dy, dx*dx)), d = q - t; equal distances go to the lowest target index
// (the k-NN tie rule).  fitness = |C| / n1, inlier_rmse = sqrt(sum d^2 / |C|), both 0 when C is empty.
// Point-to-point: Horn's quaternion on (q_i, t_i), no scale (the optimum of Open3D's Umeyama).  Point-to-plane: Open3D's
// linearisation r_i = (q_i - t_i).n_i, J_i = [q_i x n_i, n_i], J^T J x = -J^T r in fp64; |det J^T J| < 1e-6 or a non-finite
// x gives the identity update; U = Rz(x2) Ry(x1) Rx(x0) with translation x3..5 (TransformVector6dToMatrix4d).
// Generalized ICP (row f9, Open3D's registration_generalized_icp): covariances C(n) = I - (1 - eps) n^ n^T from unit normals
// (C = I for a zero-length or non-finite normal); per correspondence a = R n^_s (R the rotation of the fp32 T that moved the
// point, in fp64), b = n^_t, M = C_t + R C_s R^T = 2I - (1 - eps)(a a^T + b b^T), d = q - t, J0 = [-[q]x, I3];
// H = sum J0^T M^-1 J0, g = sum J0^T M^-1 d in fp64, then the point-to-plane solve and composition above on (H, g).
// Robust kernels (row f11, Open3D's RobustKernel of TransformationEstimationPointToPlane / ForGeneralizedICP): the same loop
// with every residual row weighted by w(r) (robust_weight).  Point-to-plane: w of the scalar residual multiplies J^T J and
// J r.  Generalized: W = (M^-1)^(1/2) in closed form, r = W d, row k weighted by w(r_k); H and g are the sums above with M^-1
// replaced by A = W diag(w) W.
//
// One deliberate difference from Open3D: Open3D transforms its copy of the source incrementally (s <- U s every
// iteration); here every iteration transforms the ORIGINAL source by the accumulated T, which is kept in fp64 on the device.
// The two agree up to rounding; this form does not accumulate fp32 error in the source over the iterations.
//
// Kernels (one call: 4 + (max_iter + 1) + 1 launches, no host synchronisation, no allocation)
//   icp_setup      one CTA per pair: bounding box of the target -> uniform grid (grid_g cells per axis as knn_grid.cu,
//                  <= 64, cell edge >= r / 2 so that a radius query touches at most 5 cells per axis); pair state
//                  (T = init in fp64, done flag, ticket) initialised; cell histogram cleared.
//   icp_bin<0/1>   histogram of the target's cells, then counting-sort scatter: float4 (x, y, z, index) in cell order,
//                  normals in the same order.  (Order inside a cell is not fixed; nothing depends on it: the selection key
//                  is (distance, index).)
//   icp_scan       exclusive scan of the histogram.
//   icp_iter       grid (source tiles, P), once per iteration (one instantiation per estimator, plus a robust one each for
//                  point-to-plane and generalized ICP that takes the loss and its parameter as launch arguments).  A CTA of
//                  a converged pair exits at once.  Otherwise each
//                  thread runs a radius-bounded 1-NN for its source points over the cells the query ball can touch,
//                  accumulates count, sum d^2 and the solver's moments in fp64 (15 for point-to-point: sum q, sum t,
//                  sum q t^T; 27 for point-to-plane and generalized ICP: the upper triangle of H and g), the CTA reduces them in a
//                  fixed order into partials[P][tiles][K].  The last CTA of the pair (threadfence + atomic ticket, reset
//                  afterwards) sums the partials in tile order, computes fitness / rmse, applies the convergence test
//                  against the previous iteration's values, and either marks the pair done or solves U and sets T = U T.
//                  No float atomics anywhere: a call is bit-reproducible.
//   icp_final      T (fp32), fitness, rmse (fp64), iterations (int32).
#include "ri_common.cuh"
#include "rigid.cuh"
#include "ri_b200.h"

namespace {

constexpr int kMaxG = 64;
constexpr int kSetupThreads = 1024;
constexpr int kThreads = 256;
constexpr int kPerThread = 2;
constexpr int kTile = kThreads * kPerThread;      // source points per CTA
constexpr int kKMax = 29;                         // count, sum d^2, 27 point-to-plane / generalized moments
constexpr int kKPoint = 17;                       // count, sum d^2, 15 point-to-point moments

enum Estimator : int { kPointToPoint = 0, kPointToPlane = 1, kGeneralized = 2 };

struct GridHdr {               // per pair, 16 ints at the head of its grid slab
    float ox, oy, oz, h, inv_h;
    int gx, gy, gz;
    int pad[8];
};

struct PairState {             // per pair, 128 bytes
    double T[12];              // 3x4 row-major, fp64
    double fitness, rmse;      // of the last evaluation
    int done, iters, ticket, pad;
};

__host__ __device__ inline int grid_g(int m)
{
    int g = 1;
    while ((long long)(g + 1) * (g + 1) * (g + 1) * 2 <= (long long)(m > 0 ? m : 1) && g < kMaxG) ++g;   // ~cbrt(m/2)
    return g;
}

struct IcpWs {                 // byte offsets into the workspace; the grid slab offsets are int32 indices inside one slab
    size_t state, partials, grids, total;
    int tiles, cells_max, hdr, start, cur, sorted, normals, stride;
};
__host__ __device__ inline IcpWs icp_ws_layout(int P, int n1, int n2)
{
    IcpWs w;
    w.tiles = (n1 + kTile - 1) / kTile;
    const int g = grid_g(n2);
    w.cells_max = g * g * g;
    int o = 0;
    w.hdr = o; o += 16;
    w.start = o; o += w.cells_max + 1;
    w.cur = o; o += w.cells_max;
    o = (o + 3) / 4 * 4;
    w.sorted = o; o += 4 * n2;                                      // float4 (x, y, z, index)
    w.normals = o; o += 4 * n2;                                     // float4 (nx, ny, nz, 0)
    w.stride = o;
    w.state = 0;
    w.partials = (size_t)P * sizeof(PairState);
    w.grids = (w.partials + (size_t)P * w.tiles * kKMax * sizeof(double) + 255) / 256 * 256;   // float4 slabs: 16-byte aligned
    w.total = w.grids + (size_t)P * w.stride * sizeof(int);
    return w;
}

__global__ void __launch_bounds__(kSetupThreads)
icp_setup_kernel(const float* __restrict__ tgt, const float* __restrict__ init, int P, int n1, int n2, float r,
                 unsigned char* __restrict__ ws)
{
    __shared__ float smin[3][kSetupThreads / 32], smax[3][kSetupThreads / 32];
    const int p = blockIdx.x, tid = threadIdx.x;
    const IcpWs L = icp_ws_layout(P, n1, n2);
    int* W = reinterpret_cast<int*>(ws + L.grids) + (size_t)p * L.stride;
    const float* X = tgt + (size_t)p * n2 * 3;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int j = tid; j < n2; j += kSetupThreads)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = X[3 * (size_t)j + a];
            lo[a] = fminf(lo[a], v); hi[a] = fmaxf(hi[a], v);
        }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
        if ((tid & 31) == 0) { smin[a][tid >> 5] = lo[a]; smax[a][tid >> 5] = hi[a]; }
    }
    __syncthreads();
    if (tid == 0) {
        GridHdr H;
        float e[3];
        for (int a = 0; a < 3; ++a) {
            float l = smin[a][0], h = smax[a][0];
            for (int w = 1; w < kSetupThreads / 32; ++w) { l = fminf(l, smin[a][w]); h = fmaxf(h, smax[a][w]); }
            if (!(l <= h)) { l = 0.f; h = 0.f; }               // NaN cloud
            (a == 0 ? H.ox : a == 1 ? H.oy : H.oz) = l;
            e[a] = h - l;
        }
        const int g = grid_g(n2);
        const float emax = fmaxf(e[0], fmaxf(e[1], e[2]));
        H.h = fmaxf(emax / (float)g, 0.5f * r);                 // >= r/2: a query ball spans at most 5 cells per axis
        H.inv_h = 1.0f / H.h;
        H.gx = min(g, (int)(e[0] * H.inv_h) + 1);
        H.gy = min(g, (int)(e[1] * H.inv_h) + 1);
        H.gz = min(g, (int)(e[2] * H.inv_h) + 1);
        *reinterpret_cast<GridHdr*>(W + L.hdr) = H;
        PairState* S = reinterpret_cast<PairState*>(ws + L.state) + p;
        for (int k = 0; k < 12; ++k)
            S->T[k] = init ? (double)init[(size_t)p * 16 + k] : (k % 5 == 0 ? 1.0 : 0.0);
        S->fitness = 0.0; S->rmse = 0.0;
        S->done = 0; S->iters = 0; S->ticket = 0;
    }
    for (int c = tid; c < L.cells_max; c += kSetupThreads) W[L.cur + c] = 0;
}

__device__ __forceinline__ int cell_of(const GridHdr& H, float x, float y, float z)
{
    const int cx = min(max((int)floorf((x - H.ox) * H.inv_h), 0), H.gx - 1);
    const int cy = min(max((int)floorf((y - H.oy) * H.inv_h), 0), H.gy - 1);
    const int cz = min(max((int)floorf((z - H.oz) * H.inv_h), 0), H.gz - 1);
    return (cx * H.gy + cy) * H.gz + cz;
}

// PASS 0: histogram into cur; PASS 1: scatter through start + atomic cursor
template <int PASS>
__global__ void __launch_bounds__(256)
icp_bin_kernel(const float* __restrict__ tgt, const float* __restrict__ nrm, int P, int n1, int n2,
               unsigned char* __restrict__ ws)
{
    const int p = blockIdx.y, t = blockIdx.x * 256 + threadIdx.x;
    if (t >= n2) return;
    const IcpWs L = icp_ws_layout(P, n1, n2);
    int* W = reinterpret_cast<int*>(ws + L.grids) + (size_t)p * L.stride;
    const GridHdr H = *reinterpret_cast<const GridHdr*>(W + L.hdr);
    const float* X = tgt + ((size_t)p * n2 + t) * 3;
    const float x = X[0], y = X[1], z = X[2];
    const int c = cell_of(H, x, y, z);
    if (PASS == 0) {
        atomicAdd(W + L.cur + c, 1);
    } else {
        const int pos = W[L.start + c] + atomicAdd(W + L.cur + c, 1);
        reinterpret_cast<float4*>(W + L.sorted)[pos] = make_float4(x, y, z, __int_as_float(t));
        if (nrm) {
            const float* Nv = nrm + ((size_t)p * n2 + t) * 3;
            reinterpret_cast<float4*>(W + L.normals)[pos] = make_float4(Nv[0], Nv[1], Nv[2], 0.f);
        }
    }
}

// exclusive scan of a pair's histogram; the cursors are reset to 0 for the scatter pass
__global__ void __launch_bounds__(1024)
icp_scan_kernel(int P, int n1, int n2, unsigned char* __restrict__ ws)
{
    __shared__ int swarp[32];
    __shared__ int scarry, stotal;
    const int p = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const IcpWs L = icp_ws_layout(P, n1, n2);
    int* W = reinterpret_cast<int*>(ws + L.grids) + (size_t)p * L.stride;
    int* cur = W + L.cur;
    int* start = W + L.start;
    if (tid == 0) scarry = 0;
    __syncthreads();
    for (int c0 = 0; c0 < L.cells_max; c0 += 1024) {
        const int c = c0 + tid;
        const int v = c < L.cells_max ? cur[c] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) swarp[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            const int w = swarp[lane];
            int wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += t;
            }
            swarp[lane] = wi - w;
            if (lane == 31) stotal = wi;
        }
        __syncthreads();
        if (c < L.cells_max) { start[c] = scarry + swarp[wid] + incl - v; cur[c] = 0; }
        __syncthreads();
        if (tid == 0) scarry += stotal;
        __syncthreads();
    }
    if (tid == 0) start[L.cells_max] = scarry;
}

// Cell range [lo, hi] of one axis that a ball of radius r around coordinate x can touch; false when it misses the grid.
// In cell units (u = (x - o) / h) the exact range is [floor(u - r/h), floor(u + r/h)].  Every rounded quantity involved
// (u, r/h, the cell coordinate a target point was binned with) is within a few ulps of a value of magnitude <= g + r/h
// <= 66 whenever the ball reaches the grid, i.e. within 1e-4 cells; the 1e-3-cell widening on each side therefore cannot
// drop a cell that holds a point within r.  Far outside the grid the widening may admit an extra cell: harmless, the
// distance test decides.
__device__ __forceinline__ bool axis_range(float x, float o, float inv_h, float rc, int g, int& lo, int& hi)
{
    const float u = (x - o) * inv_h;
    const float a = floorf(u - rc - 1e-3f), b = floorf(u + rc + 1e-3f);
    if (!(b >= 0.f) || !(a <= (float)(g - 1))) return false;
    lo = a < 0.f ? 0 : (int)a;
    hi = b > (float)(g - 1) ? g - 1 : (int)b;
    return true;
}

// n / |n| in fp64; the zero vector (which makes C(n) = I) for a zero-length or non-finite n.  -n gives exactly -(n / |n|).
__device__ __forceinline__ void unit_or_zero(float x, float y, float z, double u[3])
{
    const double dx = x, dy = y, dz = z;
    const double l2 = dx * dx + dy * dy + dz * dz;
    if (!(l2 > 0.0 && isfinite(l2))) {                 // explicit zeros: a NaN or infinite component times 0 is NaN
        u[0] = 0.0; u[1] = 0.0; u[2] = 0.0;
        return;
    }
    const double s = 1.0 / sqrt(l2);
    u[0] = dx * s; u[1] = dy * s; u[2] = dz * s;
}

// The linearised 6x6 step shared by point-to-plane and generalized ICP, on the reduced 29-slot moments m (m[2..22]: the upper
// triangle of H in row order, m[23..28]: g): H x = -g with the 1e-6 determinant rule of ldlt_solve6, then
// U = [Rz(x2) Ry(x1) Rx(x0) | x3..5]; U is left unchanged (the identity) when the solve fails.  b and x are the caller's
// scratch: local arrays of an inlined callee are allocated ahead of the caller's, which reorders the accumulators' registers.
__device__ __forceinline__ void linearised_update(const double* m, double b[6], double x[6], double U[12])
{
#pragma unroll
    for (int a = 0; a < 6; ++a) b[a] = -m[23 + a];
    if (ldlt_solve6(m + 2, b, x, 1e-6)) {
        const double ca = cos(x[0]), sa = sin(x[0]), cb = cos(x[1]), sb = sin(x[1]), cg = cos(x[2]), sg = sin(x[2]);
        // Rz(x2) Ry(x1) Rx(x0)
        U[0] = cg * cb; U[1] = cg * sb * sa - sg * ca; U[2] = cg * sb * ca + sg * sa; U[3] = x[3];
        U[4] = sg * cb; U[5] = sg * sb * sa + cg * ca; U[6] = sg * sb * ca - cg * sa; U[7] = x[4];
        U[8] = -sb;     U[9] = cb * sa;                U[10] = cb * ca;               U[11] = x[5];
    }
}

// One generalized-ICP correspondence into acc[2..28]: q = T s (fp32), t its target point, ns the source normal (caller's
// frame), nt the target normal, Tf the fp32 T that moved s, c = 1 - eps.  M^-1 is the adjugate of the symmetric M over its
// determinant (eigenvalues of M in [2 min(eps, 1), 2 max(eps, 1)]: never singular).  With u_k = e_k x q (J0's k-th
// column) the moments are H_kl = u_k.M^-1 u_l, H_k(3+l) = (M^-1 u_k)_l, H_(3+k)(3+l) = M^-1_kl, g_k = (M^-1 u_k).d,
// g_(3+k) = (M^-1 d)_k.
__device__ __forceinline__ void gicp_moments(const float* Tf, double qx, double qy, double qz, double tx, double ty,
                                             double tz, const float* ns, float4 nt, double c, double* acc)
{
    double n[3], a[3], b[3];
    unit_or_zero(ns[0], ns[1], ns[2], n);
    unit_or_zero(nt.x, nt.y, nt.z, b);
#pragma unroll
    for (int k = 0; k < 3; ++k)
        a[k] = (double)Tf[4 * k] * n[0] + (double)Tf[4 * k + 1] * n[1] + (double)Tf[4 * k + 2] * n[2];
    const double m00 = 2.0 - c * (a[0] * a[0] + b[0] * b[0]), m11 = 2.0 - c * (a[1] * a[1] + b[1] * b[1]);
    const double m22 = 2.0 - c * (a[2] * a[2] + b[2] * b[2]);
    const double m01 = -c * (a[0] * a[1] + b[0] * b[1]), m02 = -c * (a[0] * a[2] + b[0] * b[2]);
    const double m12 = -c * (a[1] * a[2] + b[1] * b[2]);
    double i00 = m11 * m22 - m12 * m12, i01 = m02 * m12 - m01 * m22, i02 = m01 * m12 - m02 * m11;
    double i11 = m00 * m22 - m02 * m02, i12 = m01 * m02 - m00 * m12, i22 = m00 * m11 - m01 * m01;
    const double inv = 1.0 / (m00 * i00 + m01 * i01 + m02 * i02);
    i00 *= inv; i01 *= inv; i02 *= inv; i11 *= inv; i12 *= inv; i22 *= inv;
    const double dx = qx - tx, dy = qy - ty, dz = qz - tz;
    // w_k = M^-1 u_k with u_0 = (0, -qz, qy), u_1 = (qz, 0, -qx), u_2 = (-qy, qx, 0)
    const double w0[3] = {i02 * qy - i01 * qz, i12 * qy - i11 * qz, i22 * qy - i12 * qz};
    const double w1[3] = {i00 * qz - i02 * qx, i01 * qz - i12 * qx, i02 * qz - i22 * qx};
    const double w2[3] = {i01 * qx - i00 * qy, i11 * qx - i01 * qy, i12 * qx - i02 * qy};
    acc[2] += w0[2] * qy - w0[1] * qz;                  // H_00 = u_0.w_0
    acc[3] += w1[2] * qy - w1[1] * qz;                  // H_01 = u_0.w_1
    acc[4] += w2[2] * qy - w2[1] * qz;                  // H_02 = u_0.w_2
    acc[5] += w0[0]; acc[6] += w0[1]; acc[7] += w0[2];
    acc[8] += w1[0] * qz - w1[2] * qx;                  // H_11 = u_1.w_1
    acc[9] += w2[0] * qz - w2[2] * qx;                  // H_12 = u_1.w_2
    acc[10] += w1[0]; acc[11] += w1[1]; acc[12] += w1[2];
    acc[13] += w2[1] * qx - w2[0] * qy;                 // H_22 = u_2.w_2
    acc[14] += w2[0]; acc[15] += w2[1]; acc[16] += w2[2];
    acc[17] += i00; acc[18] += i01; acc[19] += i02;
    acc[20] += i11; acc[21] += i12;
    acc[22] += i22;
    acc[23] += w0[0] * dx + w0[1] * dy + w0[2] * dz;
    acc[24] += w1[0] * dx + w1[1] * dy + w1[2] * dz;
    acc[25] += w2[0] * dx + w2[1] * dy + w2[2] * dz;
    acc[26] += i00 * dx + i01 * dy + i02 * dz;
    acc[27] += i01 * dx + i11 * dy + i12 * dz;
    acc[28] += i02 * dx + i12 * dy + i22 * dz;
}

// Open3D's RobustKernel::Weight(r) in fp64 (RI_LOSS_*; k > 0 for Huber, Cauchy, GM and Tukey), with e = |r|:
// L2 1; L1 1/e (0 at e = 0, where Open3D's +inf would make the step non-finite); Huber k / max(e, k);
// Cauchy 1 / (1 + (r/k)^2); GM k / (k + r^2)^2 (k in squared-residual units); Tukey (1 - (e/k)^2)^2 for e <= k, else 0.
__device__ __forceinline__ double robust_weight(int loss, double k, double r)
{
    const double e = fabs(r);
    switch (loss) {
    case RI_LOSS_L1: return e > 0.0 ? 1.0 / e : 0.0;
    case RI_LOSS_HUBER: return k / fmax(e, k);
    case RI_LOSS_CAUCHY: { const double u = r / k; return 1.0 / (1.0 + u * u); }
    case RI_LOSS_GM: { const double s = k + r * r; return k / (s * s); }
    case RI_LOSS_TUKEY: { if (!(e <= k)) return 0.0; const double u = e / k, v = 1.0 - u * u; return v * v; }
    default: return 1.0;
    }
}

// One robust generalized-ICP correspondence into acc[2..28] (arguments as gicp_moments, eps = 1 - c).  W = (M^-1)^(1/2) in
// closed form: M = 2I - c (a a^T + b b^T) has the eigenvalue 2 off span{a, b}; for unit a and b, u+- = a +- b are
// eigenvectors with lambda+- = 2 - c (1 +- a.b), so W = 2^-1/2 I + sum (lambda+-^-1/2 - 2^-1/2) u u^T / |u|^2 (a zero u has
// lambda = 2 and is skipped); with one of a, b zero and u the other, W = 2^-1/2 I + ((2 - c)^-1/2 - 2^-1/2) u u^T.
// r = W d, w_k = robust_weight(r_k), A = W diag(w) W; the moments are gicp_moments' with A in place of M^-1.
__device__ __forceinline__ void robust_gicp_moments(const float* Tf, double qx, double qy, double qz, double tx, double ty,
                                                    double tz, const float* ns, float4 nt, double c, int loss, double kp,
                                                    double* acc)
{
    constexpr double kR2 = 0.70710678118654752440;     // 2^-1/2
    double n[3], a[3], b[3];
    unit_or_zero(ns[0], ns[1], ns[2], n);
    unit_or_zero(nt.x, nt.y, nt.z, b);
#pragma unroll
    for (int k = 0; k < 3; ++k)
        a[k] = (double)Tf[4 * k] * n[0] + (double)Tf[4 * k + 1] * n[1] + (double)Tf[4 * k + 2] * n[2];
    const bool za = n[0] == 0.0 && n[1] == 0.0 && n[2] == 0.0, zb = b[0] == 0.0 && b[1] == 0.0 && b[2] == 0.0;
    double w00 = kR2, w01 = 0.0, w02 = 0.0, w11 = kR2, w12 = 0.0, w22 = kR2;     // W, symmetric
    auto add = [&](double u0, double u1, double u2, double f) {                   // W += f u u^T
        w00 += f * u0 * u0; w01 += f * u0 * u1; w02 += f * u0 * u2;
        w11 += f * u1 * u1; w12 += f * u1 * u2; w22 += f * u2 * u2;
    };
    if (!za && !zb) {
        const double s = a[0] * b[0] + a[1] * b[1] + a[2] * b[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const double sg = h == 0 ? 1.0 : -1.0;
            const double u0 = a[0] + sg * b[0], u1 = a[1] + sg * b[1], u2 = a[2] + sg * b[2];
            const double uu = u0 * u0 + u1 * u1 + u2 * u2;
            if (uu > 0.0) add(u0, u1, u2, (1.0 / sqrt(2.0 - c * (1.0 + sg * s)) - kR2) / uu);
        }
    } else if (!(za && zb)) {
        const double* u = za ? b : a;
        add(u[0], u[1], u[2], 1.0 / sqrt(2.0 - c) - kR2);
    }
    const double dx = qx - tx, dy = qy - ty, dz = qz - tz;
    const double v0 = robust_weight(loss, kp, w00 * dx + w01 * dy + w02 * dz);
    const double v1 = robust_weight(loss, kp, w01 * dx + w11 * dy + w12 * dz);
    const double v2 = robust_weight(loss, kp, w02 * dx + w12 * dy + w22 * dz);
    // A = W diag(v) W
    const double i00 = v0 * w00 * w00 + v1 * w01 * w01 + v2 * w02 * w02;
    const double i01 = v0 * w00 * w01 + v1 * w01 * w11 + v2 * w02 * w12;
    const double i02 = v0 * w00 * w02 + v1 * w01 * w12 + v2 * w02 * w22;
    const double i11 = v0 * w01 * w01 + v1 * w11 * w11 + v2 * w12 * w12;
    const double i12 = v0 * w01 * w02 + v1 * w11 * w12 + v2 * w12 * w22;
    const double i22 = v0 * w02 * w02 + v1 * w12 * w12 + v2 * w22 * w22;
    const double w0[3] = {i02 * qy - i01 * qz, i12 * qy - i11 * qz, i22 * qy - i12 * qz};
    const double w1[3] = {i00 * qz - i02 * qx, i01 * qz - i12 * qx, i02 * qz - i22 * qx};
    const double w2[3] = {i01 * qx - i00 * qy, i11 * qx - i01 * qy, i12 * qx - i02 * qy};
    acc[2] += w0[2] * qy - w0[1] * qz;
    acc[3] += w1[2] * qy - w1[1] * qz;
    acc[4] += w2[2] * qy - w2[1] * qz;
    acc[5] += w0[0]; acc[6] += w0[1]; acc[7] += w0[2];
    acc[8] += w1[0] * qz - w1[2] * qx;
    acc[9] += w2[0] * qz - w2[2] * qx;
    acc[10] += w1[0]; acc[11] += w1[1]; acc[12] += w1[2];
    acc[13] += w2[1] * qx - w2[0] * qy;
    acc[14] += w2[0]; acc[15] += w2[1]; acc[16] += w2[2];
    acc[17] += i00; acc[18] += i01; acc[19] += i02;
    acc[20] += i11; acc[21] += i12;
    acc[22] += i22;
    acc[23] += w0[0] * dx + w0[1] * dy + w0[2] * dz;
    acc[24] += w1[0] * dx + w1[1] * dy + w1[2] * dz;
    acc[25] += w2[0] * dx + w2[1] * dy + w2[2] * dz;
    acc[26] += i00 * dx + i01 * dy + i02 * dz;
    acc[27] += i01 * dx + i11 * dy + i12 * dz;
    acc[28] += i02 * dx + i12 * dy + i22 * dz;
}

// EST = kPointToPoint / kPointToPlane / kGeneralized.  src_nrm [P,n1,3] and eps are read by kGeneralized only; ROBUST
// (point-to-plane and generalized only) weights each residual row with robust_weight(loss, kp, .).
template <int EST, bool ROBUST>
__global__ void __launch_bounds__(kThreads)
icp_iter_kernel(const float* __restrict__ src, int P, int n1, int n2, float r, int it, int max_iter, float rel_fitness,
                float rel_rmse, int* __restrict__ corr, unsigned char* __restrict__ ws, const float* __restrict__ src_nrm,
                float eps, int loss, float kp)
{
    static_assert(!ROBUST || EST != kPointToPoint, "point-to-point takes no robust kernel");
    constexpr bool PLANE = EST != kPointToPoint;       // the 27-moment layout and the linearised solve
    constexpr int K = PLANE ? kKMax : kKPoint;
    __shared__ double red[(kThreads / 32) * K];
    __shared__ double tot[K];
    __shared__ float Tf[12];
    __shared__ int s_flag;
    const int p = blockIdx.y, tile = blockIdx.x, tid = threadIdx.x;
    const IcpWs L = icp_ws_layout(P, n1, n2);
    PairState* S = reinterpret_cast<PairState*>(ws + L.state) + p;
    if (tid == 0) {
        s_flag = S->done;
        for (int k = 0; k < 12; ++k) Tf[k] = (float)S->T[k];
    }
    __syncthreads();
    if (s_flag) return;

    const int* W = reinterpret_cast<const int*>(ws + L.grids) + (size_t)p * L.stride;
    const GridHdr H = *reinterpret_cast<const GridHdr*>(W + L.hdr);
    const int* start = W + L.start;
    const float4* Pt = reinterpret_cast<const float4*>(W + L.sorted);
    const float4* Nt = reinterpret_cast<const float4*>(W + L.normals);
    const float r2 = __fmul_rn(r, r);
    const float rc = r * H.inv_h;

    double acc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = 0.0;

#pragma unroll 1
    for (int s = 0; s < kPerThread; ++s) {
        const int i = tile * kTile + s * kThreads + tid;
        if (i >= n1) break;
        const float* Sv = src + ((size_t)p * n1 + i) * 3;
        const float sx = Sv[0], sy = Sv[1], sz = Sv[2];
        const float qx = __fadd_rn(__fmaf_rn(Tf[2], sz, __fmaf_rn(Tf[1], sy, __fmul_rn(Tf[0], sx))), Tf[3]);
        const float qy = __fadd_rn(__fmaf_rn(Tf[6], sz, __fmaf_rn(Tf[5], sy, __fmul_rn(Tf[4], sx))), Tf[7]);
        const float qz = __fadd_rn(__fmaf_rn(Tf[10], sz, __fmaf_rn(Tf[9], sy, __fmul_rn(Tf[8], sx))), Tf[11]);
        float best = r2;
        int bj = -1, bp = -1;
        int x0, x1, y0, y1, z0, z1;
        if (isfinite(qx) && isfinite(qy) && isfinite(qz) &&
            axis_range(qx, H.ox, H.inv_h, rc, H.gx, x0, x1) && axis_range(qy, H.oy, H.inv_h, rc, H.gy, y0, y1) &&
            axis_range(qz, H.oz, H.inv_h, rc, H.gz, z0, z1)) {
            for (int x = x0; x <= x1; ++x)
                for (int y = y0; y <= y1; ++y) {
                    const int base = (x * H.gy + y) * H.gz;
                    const int p0 = __ldg(start + base + z0), p1 = __ldg(start + base + z1 + 1);
                    for (int q = p0; q < p1; ++q) {
                        const float4 c = __ldg(Pt + q);
                        const float dx = __fsub_rn(qx, c.x), dy = __fsub_rn(qy, c.y), dz = __fsub_rn(qz, c.z);
                        const float d = __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
                        const int j = __float_as_int(c.w);
                        if (d < best || (d == best && j < bj)) { best = d; bj = j; bp = q; }
                    }
                }
        }
        if (corr) corr[(size_t)p * n1 + i] = bj;
        if (bj < 0) continue;
        const float4 c = __ldg(Pt + bp);
        const double dqx = qx, dqy = qy, dqz = qz, tx = c.x, ty = c.y, tz = c.z;
        acc[0] += 1.0;
        acc[1] += (double)best;
        if (!PLANE) {
            acc[2] += dqx; acc[3] += dqy; acc[4] += dqz;
            acc[5] += tx; acc[6] += ty; acc[7] += tz;
            acc[8] += dqx * tx; acc[9] += dqx * ty; acc[10] += dqx * tz;
            acc[11] += dqy * tx; acc[12] += dqy * ty; acc[13] += dqy * tz;
            acc[14] += dqz * tx; acc[15] += dqz * ty; acc[16] += dqz * tz;
        } else if (EST == kPointToPlane) {
            const float4 nv = __ldg(Nt + bp);
            const double nx = nv.x, ny = nv.y, nz = nv.z;
            const double res = (dqx - tx) * nx + (dqy - ty) * ny + (dqz - tz) * nz;
            const double J[6] = {dqy * nz - dqz * ny, dqz * nx - dqx * nz, dqx * ny - dqy * nx, nx, ny, nz};
            int k = 2;
            if (ROBUST) {      // w J_a, then the same fma as below: w = 1 gives bit-identical sums
                const double w = robust_weight(loss, (double)kp, res);
#pragma unroll
                for (int a = 0; a < 6; ++a) {
                    const double wJ = w * J[a];
#pragma unroll
                    for (int b = a; b < 6; ++b) acc[k++] += wJ * J[b];
                    acc[23 + a] += wJ * res;
                }
            } else {
#pragma unroll
                for (int a = 0; a < 6; ++a)
#pragma unroll
                    for (int b = a; b < 6; ++b) acc[k++] += J[a] * J[b];
#pragma unroll
                for (int a = 0; a < 6; ++a) acc[23 + a] += J[a] * res;
            }
        } else if (ROBUST) {
            robust_gicp_moments(Tf, dqx, dqy, dqz, tx, ty, tz, src_nrm + ((size_t)p * n1 + i) * 3, __ldg(Nt + bp),
                                1.0 - (double)eps, loss, (double)kp, acc);
        } else {
            gicp_moments(Tf, dqx, dqy, dqz, tx, ty, tz, src_nrm + ((size_t)p * n1 + i) * 3, __ldg(Nt + bp),
                         1.0 - (double)eps, acc);
        }
    }

    block_sum<K>(acc, red);
    double* part = reinterpret_cast<double*>(ws + L.partials) + (size_t)p * L.tiles * kKMax;
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) part[(size_t)tile * kKMax + k] = acc[k];
        __threadfence();
        s_flag = atomicAdd(&S->ticket, 1) == L.tiles - 1;
    }
    __syncthreads();
    if (!s_flag) return;

    // ---- last CTA of the pair: partials in tile order -> fitness, rmse, convergence, update
    __threadfence();
    if (tid < K) {
        double v = 0.0;
        for (int t = 0; t < L.tiles; ++t) v += __ldcg(part + (size_t)t * kKMax + tid);
        tot[tid] = v;
    }
    __syncthreads();
    if (tid != 0) return;
    S->ticket = 0;
    const double cnt = tot[0];
    const double fitness = cnt / (double)n1;
    const double rmse = cnt > 0.0 ? sqrt(tot[1] / cnt) : 0.0;
    const bool converged = it > 0 && fabs(S->fitness - fitness) < (double)rel_fitness &&
                           fabs(S->rmse - rmse) < (double)rel_rmse;
    S->fitness = fitness;
    S->rmse = rmse;
    if (converged || it == max_iter) {
        S->done = 1;
        S->iters = it;
        return;
    }
    double U[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
    if (!PLANE) {
        if (cnt > 0.0) {
            const double inv = 1.0 / cnt;
            const double cq[3] = {tot[2] * inv, tot[3] * inv, tot[4] * inv};
            const double ct[3] = {tot[5] * inv, tot[6] * inv, tot[7] * inv};
            double Hm[9], R[9];
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int b = 0; b < 3; ++b) Hm[3 * a + b] = tot[8 + 3 * a + b] - cnt * cq[a] * ct[b];
            horn_rotation(Hm, R);
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                U[4 * a + 0] = R[3 * a + 0]; U[4 * a + 1] = R[3 * a + 1]; U[4 * a + 2] = R[3 * a + 2];
                U[4 * a + 3] = ct[a] - (R[3 * a] * cq[0] + R[3 * a + 1] * cq[1] + R[3 * a + 2] * cq[2]);
            }
        }
    } else {
        double b[6], x[6];
        linearised_update(tot, b, x, U);
    }
    double Tn[12];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c)
            Tn[4 * a + c] = U[4 * a] * S->T[c] + U[4 * a + 1] * S->T[4 + c] + U[4 * a + 2] * S->T[8 + c] + (c == 3 ? U[4 * a + 3] : 0.0);
#pragma unroll
    for (int k = 0; k < 12; ++k) S->T[k] = Tn[k];
}

__global__ void icp_final_kernel(int P, int n1, int n2, const unsigned char* __restrict__ ws, float* __restrict__ T,
                                 double* __restrict__ fitness, double* __restrict__ rmse, int* __restrict__ iters)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const IcpWs L = icp_ws_layout(P, n1, n2);
    const PairState* S = reinterpret_cast<const PairState*>(ws + L.state) + p;
    float* O = T + (size_t)p * 16;
    for (int k = 0; k < 12; ++k) O[k] = (float)S->T[k];
    O[12] = 0.f; O[13] = 0.f; O[14] = 0.f; O[15] = 1.f;
    fitness[p] = S->fitness;
    rmse[p] = S->rmse;
    iters[p] = S->iters;
}

// The launch sequence of one call, after the arguments have been checked (P > 0): setup, binning, max_iter + 1 iteration
// launches, final.  nrm: target normals binned with the grid (NULL for point-to-point).  loss >= 0 selects the robust
// instantiation of est (point-to-plane or generalized) with parameter kp; -1 the plain one.
int icp_launch(int est, int loss, float kp, const float* src, const float* tgt, const float* nrm, const float* src_nrm,
               const float* init, int P, int n1, int n2, float max_corr_dist, float eps, int max_iter, float rel_fitness,
               float rel_rmse, float* T, double* fitness, double* inlier_rmse, int* iters, int* corr, void* workspace,
               size_t workspace_bytes, void* stream)
{
    if (P > 65535) return RI_ERR_UNSUPPORTED;
    if (P == 0) return RI_OK;
    const IcpWs L = icp_ws_layout(P, n1, n2);
    if (L.tiles > 65535) return RI_ERR_UNSUPPORTED;
    if (workspace == nullptr || ((uintptr_t)workspace & 15) != 0 || workspace_bytes < L.total) return RI_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
    icp_setup_kernel<<<P, kSetupThreads, 0, st>>>(tgt, init, P, n1, n2, max_corr_dist, ws);
    RI_LAUNCH_CHECK();
    const dim3 gb((n2 + 255) / 256, P);
    icp_bin_kernel<0><<<gb, 256, 0, st>>>(tgt, nrm, P, n1, n2, ws);
    RI_LAUNCH_CHECK();
    icp_scan_kernel<<<P, 1024, 0, st>>>(P, n1, n2, ws);
    RI_LAUNCH_CHECK();
    icp_bin_kernel<1><<<gb, 256, 0, st>>>(tgt, nrm, P, n1, n2, ws);
    RI_LAUNCH_CHECK();
    const dim3 gi(L.tiles, P);
    const bool robust = loss >= 0;
    for (int it = 0; it <= max_iter; ++it) {
        if (est == kGeneralized && robust)
            icp_iter_kernel<kGeneralized, true><<<gi, kThreads, 0, st>>>(src, P, n1, n2, max_corr_dist, it, max_iter,
                                                                         rel_fitness, rel_rmse, corr, ws, src_nrm, eps,
                                                                         loss, kp);
        else if (est == kGeneralized)
            icp_iter_kernel<kGeneralized, false><<<gi, kThreads, 0, st>>>(src, P, n1, n2, max_corr_dist, it, max_iter,
                                                                          rel_fitness, rel_rmse, corr, ws, src_nrm, eps,
                                                                          0, 0.f);
        else if (est == kPointToPlane && robust)
            icp_iter_kernel<kPointToPlane, true><<<gi, kThreads, 0, st>>>(src, P, n1, n2, max_corr_dist, it, max_iter,
                                                                          rel_fitness, rel_rmse, corr, ws, nullptr, 0.f,
                                                                          loss, kp);
        else if (est == kPointToPlane)
            icp_iter_kernel<kPointToPlane, false><<<gi, kThreads, 0, st>>>(src, P, n1, n2, max_corr_dist, it, max_iter,
                                                                           rel_fitness, rel_rmse, corr, ws, nullptr, 0.f,
                                                                           0, 0.f);
        else
            icp_iter_kernel<kPointToPoint, false><<<gi, kThreads, 0, st>>>(src, P, n1, n2, max_corr_dist, it, max_iter,
                                                                           rel_fitness, rel_rmse, corr, ws, nullptr, 0.f,
                                                                           0, 0.f);
        RI_LAUNCH_CHECK();
    }
    icp_final_kernel<<<(P + 127) / 128, 128, 0, st>>>(P, n1, n2, ws, T, fitness, inlier_rmse, iters);
    RI_LAUNCH_CHECK();
    return RI_OK;
}

}  // namespace

extern "C" size_t ri_icp_workspace_bytes(int P, int n1, int n2)
{
    if (P <= 0 || n1 <= 0 || n2 <= 0) return 16;
    return icp_ws_layout(P, n1, n2).total;
}

// src [P,n1,3], tgt [P,n2,3], tgt_normals [P,n2,3] (point-to-plane only), init [P,4,4] row-major (NULL = identity), all fp32
// point-major.  -> T [P,4,4] fp32, fitness [P], inlier_rmse [P] fp64, iters [P] int32, corr [P,n1] (target index or -1 under
// the returned T; NULL = not written).
extern "C" int ri_icp_f32(const float* src, const float* tgt, const float* tgt_normals, const float* init, int P, int n1,
                          int n2, float max_corr_dist, int point_to_plane, int max_iter, float rel_fitness, float rel_rmse,
                          float* T, double* fitness, double* inlier_rmse, int* iters, int* corr, void* workspace,
                          size_t workspace_bytes, void* stream)
{
    if (P < 0 || n1 <= 0 || n2 <= 0 || !(max_corr_dist > 0.f) || max_iter < 0) return RI_ERR_BAD_ARG;
    if (point_to_plane && tgt_normals == nullptr) return RI_ERR_BAD_ARG;
    return icp_launch(point_to_plane ? kPointToPlane : kPointToPoint, -1, 0.f, src, tgt,
                      point_to_plane ? tgt_normals : nullptr, nullptr, init, P, n1, n2, max_corr_dist, 0.f, max_iter,
                      rel_fitness, rel_rmse, T, fitness, inlier_rmse, iters, corr, workspace, workspace_bytes, stream);
}

// ri_icp_f32 with the generalized (plane-to-plane) estimator: src_normals [P,n1,3] and tgt_normals [P,n2,3] fp32 point-major
// (both required; used through n / |n|), eps the covariances' smallest eigenvalue (finite, > 0).
extern "C" int ri_generalized_icp_f32(const float* src, const float* tgt, const float* src_normals,
                                      const float* tgt_normals, const float* init, int P, int n1, int n2,
                                      float max_corr_dist, float epsilon, int max_iter, float rel_fitness,
                                      float rel_rmse, float* T, double* fitness, double* inlier_rmse, int* iters,
                                      int* corr, void* workspace, size_t workspace_bytes, void* stream)
{
    if (P < 0 || n1 <= 0 || n2 <= 0 || !(max_corr_dist > 0.f) || max_iter < 0) return RI_ERR_BAD_ARG;
    if (!(epsilon > 0.f) || !isfinite(epsilon) || src_normals == nullptr || tgt_normals == nullptr) return RI_ERR_BAD_ARG;
    return icp_launch(kGeneralized, -1, 0.f, src, tgt, tgt_normals, src_normals, init, P, n1, n2, max_corr_dist, epsilon,
                      max_iter, rel_fitness, rel_rmse, T, fitness, inlier_rmse, iters, corr, workspace, workspace_bytes,
                      stream);
}

// ri_icp_f32 (point-to-plane) or ri_generalized_icp_f32 (generalized != 0) with a robust kernel: loss RI_LOSS_*, k its
// parameter (finite, > 0; read by Huber, Cauchy, GM and Tukey only).  src_normals is read when generalized only.
extern "C" int ri_robust_icp_f32(const float* src, const float* tgt, const float* src_normals, const float* tgt_normals,
                                 const float* init, int P, int n1, int n2, float max_corr_dist, int generalized,
                                 float epsilon, int loss, float k, int max_iter, float rel_fitness, float rel_rmse,
                                 float* T, double* fitness, double* inlier_rmse, int* iters, int* corr, void* workspace,
                                 size_t workspace_bytes, void* stream)
{
    if (P < 0 || n1 <= 0 || n2 <= 0 || !(max_corr_dist > 0.f) || max_iter < 0) return RI_ERR_BAD_ARG;
    if (loss < RI_LOSS_L2 || loss > RI_LOSS_TUKEY) return RI_ERR_BAD_ARG;
    if (loss >= RI_LOSS_HUBER && !(k > 0.f && isfinite(k))) return RI_ERR_BAD_ARG;
    if (tgt_normals == nullptr) return RI_ERR_BAD_ARG;
    if (generalized && (!(epsilon > 0.f) || !isfinite(epsilon) || src_normals == nullptr)) return RI_ERR_BAD_ARG;
    return icp_launch(generalized ? kGeneralized : kPointToPlane, loss, k, src, tgt, tgt_normals,
                      generalized ? src_normals : nullptr, init, P, n1, n2, max_corr_dist, generalized ? epsilon : 0.f,
                      max_iter, rel_fitness, rel_rmse, T, fitness, inlier_rmse, iters, corr, workspace, workspace_bytes,
                      stream);
}
