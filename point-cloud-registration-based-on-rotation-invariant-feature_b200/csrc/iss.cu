// iss.cu — Intrinsic Shape Signatures keypoints (Zhong, ICCV Workshops 2009; Open3D's compute_iss_keypoints), a batch of B
// dense clouds per call, sm_100a.  include/ri_b200.h (ri_iss_keypoints_f32) states the contract; the tests replay it in
// numpy (iss_oracle).
//
// Pipeline per call:
//   1. grid      the uniform grid of grid.cuh (setup, histogram, scan), then a STABLE placement: one radix sort
//                (radix.cuh) of (cloud, cell) keys over the batch's points in index order, so each cell lists its points
//                in ascending index.  grid_bin_kernel<1> places them in atomic order, and a covariance summed in that
//                order would not be reproducible;
//   2. nn        (automatic radii only) per point the distance to the nearest other point, sqrt((double)d);
//   3. radii     one CTA per cloud: the mean of those distances in a fixed fp64 reduction order, r_s = 6 res,
//                r_nm = 4 res (or the explicit radii);
//   4. saliency  one thread per point: the ring search of normals.cu with a pure radius exit, fp64 moments of p - q in
//                the visiting order (rings, cells, ascending index: a function of the cloud alone), eigenvalues by the
//                Jacobi sweeps of eig3.cuh;
//   5. suppress  one thread per point: the radius-r_nm search, non-maximum suppression on the saliency;
//   6. compact   one CTA per cloud: keypoint indices in ascending order, -1 after them.
// No float atomics and no allocation: a cloud's result is bit-reproducible and does not depend on the rest of the batch.
#include "eig3.cuh"
#include "grid.cuh"
#include "radix.cuh"

namespace {

constexpr int kIssThreads = 128;
constexpr int kCtaThreads = 1024;

struct IssWs {                 // byte offsets into the workspace
    size_t grid, keys_a, keys_b, vals_a, vals_b, hist, nn, sal, radii, flags, total;
};

inline size_t al256(size_t x) { return (x + 255) / 256 * 256; }

inline IssWs iss_ws_layout(int B, int N)
{
    const size_t n = (size_t)B * N;
    IssWs w;
    size_t o = 0;
    w.grid = o; o = al256(o + (size_t)B * grid_ws_layout(N, N).stride * sizeof(int));
    w.keys_a = o; o = al256(o + n * sizeof(unsigned long long));
    w.keys_b = o; o = al256(o + n * sizeof(unsigned long long));
    w.vals_a = o; o = al256(o + n * sizeof(int));
    w.vals_b = o; o = al256(o + n * sizeof(int));
    w.hist = o; o = al256(o + ri_radix::hist_bytes((long long)n));
    w.nn = o; o = al256(o + n * sizeof(double));
    w.sal = o; o = al256(o + n * sizeof(double));
    w.radii = o; o = al256(o + (size_t)B * 2 * sizeof(float));
    w.flags = o; o = al256(o + n);
    w.total = o;
    return w;
}

// Visits every point p of the cloud with d(q, p) < lim (q itself included) in ring order: rings R = 0, 1, ... around q's
// cell, cells in (x, y, z) order within a ring, points in the cell's order.  f(d, j, p) returns true to stop early; it may
// lower lim (the nearest-point search does).  The exit is the ring bound of normals.cu: every unvisited cell lies at
// least sqrt(bound) away.
template <class F>
__device__ __forceinline__ void ring_visit(const GridHdr& H, const int* __restrict__ start, const float4* __restrict__ P,
                                           float qx, float qy, float qz, float& lim, F&& f)
{
    int cx, cy, cz;
    cell_of(H, qx, qy, qz, cx, cy, cz);
    const int rmax = max(max(cx, H.gx - 1 - cx), max(max(cy, H.gy - 1 - cy), max(cz, H.gz - 1 - cz)));
    for (int R = 0; R <= rmax; ++R) {
        const int x0 = max(cx - R, 0), x1 = min(cx + R, H.gx - 1);
        const int y0 = max(cy - R, 0), y1 = min(cy + R, H.gy - 1);
        for (int x = x0; x <= x1; ++x) {
            const bool xface = (x == cx - R) || (x == cx + R);
            for (int y = y0; y <= y1; ++y) {
                const bool face = xface || (y == cy - R) || (y == cy + R);
                const int nseg = (face || R == 0) ? 1 : 2;
                for (int sgi = 0; sgi < nseg; ++sgi) {
                    int z0, z1;
                    if (face || R == 0) { z0 = max(cz - R, 0); z1 = min(cz + R, H.gz - 1); }
                    else { z0 = z1 = (sgi == 0 ? cz - R : cz + R); if (z0 < 0 || z0 >= H.gz) continue; }
                    const int base = (x * H.gy + y) * H.gz;
                    const int p0 = __ldg(start + base + z0), p1 = __ldg(start + base + z1 + 1);
                    for (int p = p0; p < p1; ++p) {
                        const float4 r = __ldg(P + p);
                        const float dx = __fsub_rn(qx, r.x), dy = __fsub_rn(qy, r.y), dz = __fsub_rn(qz, r.z);
                        const float d = __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
                        if (d < lim && f(d, __float_as_int(r.w), r)) return;
                    }
                }
            }
        }
        float lb = INFINITY;
        if (cx - R > 0) lb = fminf(lb, qx - (H.ox + (float)(cx - R) * H.h));
        if (cx + R < H.gx - 1) lb = fminf(lb, (H.ox + (float)(cx + R + 1) * H.h) - qx);
        if (cy - R > 0) lb = fminf(lb, qy - (H.oy + (float)(cy - R) * H.h));
        if (cy + R < H.gy - 1) lb = fminf(lb, (H.oy + (float)(cy + R + 1) * H.h) - qy);
        if (cz - R > 0) lb = fminf(lb, qz - (H.oz + (float)(cz - R) * H.h));
        if (cz + R < H.gz - 1) lb = fminf(lb, (H.oz + (float)(cz + R + 1) * H.h) - qz);
        lb = fmaxf(lb - 1e-3f * H.h, 0.f);
        if (lb * lb * 0.999f >= lim) break;
    }
}

__device__ __forceinline__ bool finite3(float x, float y, float z) { return isfinite(x) && isfinite(y) && isfinite(z); }

// (cloud, cell) key and global point index of every point, in index order: the input of the stable sort
__global__ void __launch_bounds__(256)
iss_key_kernel(const float* __restrict__ xyz, int N, const int* __restrict__ ws, unsigned long long* __restrict__ keys,
               int* __restrict__ vals)
{
    const int b = blockIdx.y, t = blockIdx.x * 256 + threadIdx.x;
    if (t >= N) return;
    const GridWs L = grid_ws_layout(N, N);
    const GridHdr H = *reinterpret_cast<const GridHdr*>(ws + (size_t)b * L.stride + L.hdr);
    const float* X = xyz + (size_t)b * 3 * N;
    int cx, cy, cz;
    const int c = cell_of(H, X[t], X[t + N], X[t + 2 * (size_t)N], cx, cy, cz);
    const size_t g = (size_t)b * N + t;
    keys[g] = (unsigned long long)b * L.cells_max + c;
    vals[g] = (int)g;
}

// sorted position i -> the cloud's cell-ordered float4 list (cloud b owns positions [b N, (b+1) N)); the per-point
// kernels take their queries in that order too
__global__ void __launch_bounds__(256)
iss_place_kernel(const float* __restrict__ xyz, int B, int N, const int* __restrict__ vals, int* __restrict__ ws)
{
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= (long long)B * N) return;
    const int g = vals[i], b = g / N, t = g - b * N;
    const int pos = (int)(i - (long long)b * N);
    const GridWs L = grid_ws_layout(N, N);
    int* W = ws + (size_t)b * L.stride;
    const float* X = xyz + (size_t)b * 3 * N;
    reinterpret_cast<float4*>(W + L.sorted)[pos] = make_float4(X[t], X[t + N], X[t + 2 * (size_t)N], __int_as_float(t));
}

// distance to the nearest other point (the second key of the k = 2 list), -1 for a point that has none or is not finite
__global__ void __launch_bounds__(kIssThreads, 1)
iss_nn_kernel(int N, const int* __restrict__ ws, double* __restrict__ nn)
{
    const int b = blockIdx.y, t = blockIdx.x * kIssThreads + threadIdx.x;
    if (t >= N) return;
    const GridWs L = grid_ws_layout(N, N);
    const int* W = ws + (size_t)b * L.stride;
    const GridHdr H = *reinterpret_cast<const GridHdr*>(W + L.hdr);
    const float4 q = reinterpret_cast<const float4*>(W + L.sorted)[t];
    const int qi = __float_as_int(q.w);
    float best = INFINITY;
    if (finite3(q.x, q.y, q.z))
        ring_visit(H, W + L.rstart, reinterpret_cast<const float4*>(W + L.sorted), q.x, q.y, q.z, best,
                   [&](float d, int j, float4) { if (j != qi) best = d; return false; });
    nn[(size_t)b * N + qi] = best < INFINITY ? sqrt((double)best) : -1.0;
}

// One CTA per cloud: res = mean of the nn distances (fixed order: a strided fp64 sum per thread, then a fixed tree),
// radii = (6 res, 4 res) rounded to fp32; or the explicit radii.  A cloud with no counted distance gets radii 0.
__global__ void __launch_bounds__(kCtaThreads)
iss_radii_kernel(int N, int automatic, float rs, float rnm, const double* __restrict__ nn, float* __restrict__ radii,
                 float* __restrict__ radii_out)
{
    __shared__ double ssum[kCtaThreads];
    __shared__ int scnt[kCtaThreads];
    const int b = blockIdx.x, tid = threadIdx.x;
    if (automatic) {
        double s = 0.0;
        int c = 0;
        for (int i = tid; i < N; i += kCtaThreads) {
            const double v = nn[(size_t)b * N + i];
            if (v >= 0.0) { s += v; ++c; }
        }
        ssum[tid] = s; scnt[tid] = c;
        __syncthreads();
        for (int h = kCtaThreads / 2; h > 0; h >>= 1) {
            if (tid < h) { ssum[tid] += ssum[tid + h]; scnt[tid] += scnt[tid + h]; }
            __syncthreads();
        }
        const double res = scnt[0] > 0 ? ssum[0] / (double)scnt[0] : 0.0;
        rs = (float)(6.0 * res);
        rnm = (float)(4.0 * res);
    }
    if (tid == 0) {
        radii[2 * b] = rs; radii[2 * b + 1] = rnm;
        if (radii_out != nullptr) { radii_out[2 * b] = rs; radii_out[2 * b + 1] = rnm; }
    }
}

__global__ void __launch_bounds__(kIssThreads, 1)
iss_saliency_kernel(int N, int min_nn, double gamma_21, double gamma_32, const int* __restrict__ ws,
                    const float* __restrict__ radii, double* __restrict__ sal)
{
    const int b = blockIdx.y, t = blockIdx.x * kIssThreads + threadIdx.x;
    if (t >= N) return;
    const GridWs L = grid_ws_layout(N, N);
    const int* W = ws + (size_t)b * L.stride;
    const GridHdr H = *reinterpret_cast<const GridHdr*>(W + L.hdr);
    const float4 q = reinterpret_cast<const float4*>(W + L.sorted)[t];
    const int qi = __float_as_int(q.w);
    const float r = radii[2 * b];
    float lim = __fmul_rn(r, r);
    double s = 0.0;
    if (finite3(q.x, q.y, q.z)) {
        int cnt = 0;
        double s1x = 0, s1y = 0, s1z = 0, sxx = 0, sxy = 0, sxz = 0, syy = 0, syz = 0, szz = 0;
        ring_visit(H, W + L.rstart, reinterpret_cast<const float4*>(W + L.sorted), q.x, q.y, q.z, lim,
                   [&](float, int, float4 p) {
                       const double ex = (double)p.x - (double)q.x;
                       const double ey = (double)p.y - (double)q.y;
                       const double ez = (double)p.z - (double)q.z;
                       s1x += ex; s1y += ey; s1z += ez;
                       sxx = fma(ex, ex, sxx); sxy = fma(ex, ey, sxy); sxz = fma(ex, ez, sxz);
                       syy = fma(ey, ey, syy); syz = fma(ey, ez, syz); szz = fma(ez, ez, szz);
                       ++cnt;
                       return false;
                   });
        if (cnt >= min_nn) {
            const double inv = 1.0 / (double)cnt;
            const double mx = s1x * inv, my = s1y * inv, mz = s1z * inv;
            const double c[6] = {sxx * inv - mx * mx, sxy * inv - mx * my, sxz * inv - mx * mz,
                                 syy * inv - my * my, syz * inv - my * mz, szz * inv - mz * mz};
            bool zero = true, fin = true;
#pragma unroll
            for (int e = 0; e < 6; ++e) { zero = zero && fabs(c[e]) <= 1e-12; fin = fin && isfinite(c[e]); }
            const double tr = c[0] + c[3] + c[5];
            if (!zero && fin && tr > 0.0 && isfinite(tr)) {
                const double it = 1.0 / tr;              // unit trace: the Jacobi thresholds are relative
                double a[3][3], v[3][3];
                a[0][0] = c[0] * it; a[0][1] = c[1] * it; a[0][2] = c[2] * it;
                a[1][1] = c[3] * it; a[1][2] = c[4] * it; a[2][2] = c[5] * it;
                a[1][0] = a[0][1]; a[2][0] = a[0][2]; a[2][1] = a[1][2];
                jacobi3(a, v);
                double e1 = a[0][0] * tr, e2 = a[1][1] * tr, e3 = a[2][2] * tr, x;
                if (e1 < e2) { x = e1; e1 = e2; e2 = x; }
                if (e2 < e3) { x = e2; e2 = e3; e3 = x; }
                if (e1 < e2) { x = e1; e1 = e2; e2 = x; }
                if (e2 / e1 < gamma_21 && e3 / e2 < gamma_32) s = e3;
            }
        }
    }
    sal[(size_t)b * N + qi] = s;
}

__global__ void __launch_bounds__(kIssThreads, 1)
iss_suppress_kernel(int N, int min_nn, const int* __restrict__ ws, const float* __restrict__ radii,
                    const double* __restrict__ sal, unsigned char* __restrict__ flags)
{
    const int b = blockIdx.y, t = blockIdx.x * kIssThreads + threadIdx.x;
    if (t >= N) return;
    const GridWs L = grid_ws_layout(N, N);
    const int* W = ws + (size_t)b * L.stride;
    const GridHdr H = *reinterpret_cast<const GridHdr*>(W + L.hdr);
    const float4 q = reinterpret_cast<const float4*>(W + L.sorted)[t];
    const int qi = __float_as_int(q.w);
    const double* S = sal + (size_t)b * N;
    const double sq = S[qi];
    bool keep = false;
    if (sq > 0.0) {                                      // s > 0 implies q is finite
        const float r = radii[2 * b + 1];
        float lim = __fmul_rn(r, r);
        int cnt = 0;
        bool beaten = false;
        ring_visit(H, W + L.rstart, reinterpret_cast<const float4*>(W + L.sorted), q.x, q.y, q.z, lim,
                   [&](float, int j, float4) {
                       ++cnt;
                       beaten = __ldg(S + j) > sq;
                       return beaten;
                   });
        keep = !beaten && cnt >= min_nn;
    }
    flags[(size_t)b * N + qi] = keep ? 1 : 0;
}

// One CTA per cloud: the flagged indices in ascending order, -1 after them; count[b].
__global__ void __launch_bounds__(kCtaThreads)
iss_compact_kernel(int N, const unsigned char* __restrict__ flags, int* __restrict__ idx, int* __restrict__ count)
{
    __shared__ int swarp[kCtaThreads / 32];
    __shared__ int stotal;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned char* F = flags + (size_t)b * N;
    int* I = idx + (size_t)b * N;
    int base = 0;
    for (int c0 = 0; c0 < N; c0 += kCtaThreads) {
        const int i = c0 + tid;
        const bool f = i < N && F[i] != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        if (lane == 0) swarp[wid] = __popc(bal);
        __syncthreads();
        if (wid == 0) {
            const int w = swarp[lane];
            int incl = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += up;
            }
            swarp[lane] = incl - w;
            if (lane == 31) stotal = incl;
        }
        __syncthreads();
        if (f) I[base + swarp[wid] + __popc(bal & ((1u << lane) - 1u))] = i;
        base += stotal;
        __syncthreads();
    }
    for (int i = base + tid; i < N; i += kCtaThreads) I[i] = -1;
    if (tid == 0) count[b] = base;
}

}  // namespace

extern "C" size_t ri_iss_workspace_bytes(int B, int N)
{
    if (B <= 0 || N < 0) return 0;
    return iss_ws_layout(B, N).total;
}

extern "C" int ri_iss_keypoints_f32(const float* xyz, int B, int N, float salient_radius, float non_max_radius,
                                    const double* gamma, int min_neighbors, int* idx, int* count, double* saliency,
                                    float* radii, void* workspace, size_t workspace_bytes, void* stream)
{
    if (gamma == nullptr) return RI_ERR_BAD_ARG;
    const double gamma_21 = gamma[0], gamma_32 = gamma[1];
    if (B < 0 || N < 0 || !(gamma_21 > 0.0) || !(gamma_32 > 0.0) || min_neighbors < 1) return RI_ERR_BAD_ARG;
    if (!(salient_radius >= 0.f) || !isfinite(salient_radius) || !(non_max_radius >= 0.f) || !isfinite(non_max_radius))
        return RI_ERR_BAD_ARG;
    if (B > 0 && (count == nullptr || (N > 0 && (idx == nullptr || xyz == nullptr)))) return RI_ERR_BAD_ARG;
    if (B > 65535 || (long long)B * N > 0x7FFFFFFFLL) return RI_ERR_UNSUPPORTED;
    if (B == 0) return RI_OK;
    const IssWs V = iss_ws_layout(B, N);
    if (workspace == nullptr || ((uintptr_t)workspace & 255) != 0 || workspace_bytes < V.total) return RI_ERR_WORKSPACE;
    const int automatic = salient_radius == 0.f || non_max_radius == 0.f;
    cudaStream_t st = (cudaStream_t)stream;
    char* base = reinterpret_cast<char*>(workspace);
    int* ws = reinterpret_cast<int*>(base + V.grid);
    double* nn = reinterpret_cast<double*>(base + V.nn);
    double* sal = saliency != nullptr ? saliency : reinterpret_cast<double*>(base + V.sal);
    float* rad = reinterpret_cast<float*>(base + V.radii);
    unsigned char* flags = reinterpret_cast<unsigned char*>(base + V.flags);

    if (N > 0) {
        grid_setup_kernel<<<B, kSetupThreads, 0, st>>>(xyz, N, N, ws);
        RI_LAUNCH_CHECK();
        const dim3 gb((N + 255) / 256, B);
        grid_bin_kernel<0><<<gb, 256, 0, st>>>(xyz, xyz, N, N, ws);
        RI_LAUNCH_CHECK();
        grid_scan_kernel<<<dim3(B, 2), 1024, 0, st>>>(N, N, ws);
        RI_LAUNCH_CHECK();
        auto* ka = reinterpret_cast<unsigned long long*>(base + V.keys_a);
        auto* kb = reinterpret_cast<unsigned long long*>(base + V.keys_b);
        int* va = reinterpret_cast<int*>(base + V.vals_a);
        int* vb = reinterpret_cast<int*>(base + V.vals_b);
        iss_key_kernel<<<gb, 256, 0, st>>>(xyz, N, ws, ka, va);
        RI_LAUNCH_CHECK();
        const unsigned long long maxkey = (unsigned long long)B * grid_ws_layout(N, N).cells_max - 1;
        const int bits = 64 - __builtin_clzll(maxkey | 1ull);
        const int rc = ri_radix::sort_pairs<unsigned long long>(ka, kb, va, vb, B * N, bits, nullptr,
                                                                 reinterpret_cast<int*>(base + V.hist), st);
        if (rc != RI_OK) return rc;
        const int* sorted = (ri_radix::passes_for_bits(bits) & 1) ? vb : va;
        iss_place_kernel<<<(unsigned)(((long long)B * N + 255) / 256), 256, 0, st>>>(xyz, B, N, sorted, ws);
        RI_LAUNCH_CHECK();
        if (automatic) {
            iss_nn_kernel<<<dim3((N + kIssThreads - 1) / kIssThreads, B), kIssThreads, 0, st>>>(N, ws, nn);
            RI_LAUNCH_CHECK();
        }
    }
    iss_radii_kernel<<<B, kCtaThreads, 0, st>>>(N, automatic, salient_radius, non_max_radius, nn, rad, radii);
    RI_LAUNCH_CHECK();
    if (N > 0) {
        const dim3 gq((N + kIssThreads - 1) / kIssThreads, B);
        iss_saliency_kernel<<<gq, kIssThreads, 0, st>>>(N, min_neighbors, gamma_21, gamma_32, ws, rad, sal);
        RI_LAUNCH_CHECK();
        iss_suppress_kernel<<<gq, kIssThreads, 0, st>>>(N, min_neighbors, ws, rad, sal, flags);
        RI_LAUNCH_CHECK();
    }
    iss_compact_kernel<<<B, kCtaThreads, 0, st>>>(N, flags, idx, count);
    RI_LAUNCH_CHECK();
    return RI_OK;
}
