// normals.cu — per-point normal estimation for xyz-only clouds (Open3D's estimate_normals with KDTreeSearchParamHybrid),
// a batch of B clouds per call, sm_100a.
//
// For each point q of a cloud xyz [3,N]:
//   neighbours  the max_nn smallest keys (d, index) among the points with d < min(radius^2, 10000), q itself included,
//               d = fma(dz,dz, fma(dy,dy, dx*dx)), d* = q - p in fp32 — exactly the first max_nn entries of the k-NN
//               (csrc/knn_grid.cu, same grid, same expression, same keys) whose distance passes the cut;
//   covariance  p - q in fp64 (exact), summed over that list in its (d, index) order, C = S2/n - mu mu^T (Open3D's
//               population covariance, centred on q for conditioning);
//   normal      unit eigenvector of the smallest eigenvalue of C by fp64 cyclic Jacobi sweeps (lowest index on equal
//               eigenvalues), rounded to fp32; (0,0,1) for fewer than 3 neighbours or a trace that is not positive and
//               finite;
//   orientation flipped when n.(camera_b - q) < 0 or n.prior < 0 (at most one of the two), the default included.
//
// Pipeline per call: the grid build of grid.cuh over the batch (setup, histogram, scan, scatter: 4 launches), then
// normals_query_kernel: one thread per point in cell order, the ring search of grid_query_kernel with a second exit (every
// unvisited cell is at least radius away), then the fp64 epilogue in registers.  No atomics after the scatter, so a point's
// result depends only on its cloud and is bit-reproducible.
#include "eig3.cuh"
#include "grid.cuh"

namespace {

// Smallest-eigenvalue eigenvector of the symmetric 3x3 c (c00 c01 c02 c11 c12 c22), scaled to unit trace by the caller.
// Cyclic Jacobi of csrc/eig3.cuh, fp64.
__device__ __forceinline__ void smallest_eigvec3(const double c[6], double& nx, double& ny, double& nz)
{
    double a[3][3], v[3][3];
    a[0][0] = c[0]; a[0][1] = c[1]; a[0][2] = c[2];
    a[1][1] = c[3]; a[1][2] = c[4]; a[2][2] = c[5];
    a[1][0] = c[1]; a[2][0] = c[2]; a[2][1] = c[4];
    jacobi3(a, v);
    double lo = a[0][0];                                // strict '<': the lowest index wins a tie
    nx = v[0][0]; ny = v[1][0]; nz = v[2][0];
#pragma unroll
    for (int i = 1; i < 3; ++i)
        if (a[i][i] < lo) { lo = a[i][i]; nx = v[0][i]; ny = v[1][i]; nz = v[2][i]; }
    const double nn = sqrt(nx * nx + ny * ny + nz * nz);
    nx /= nn; ny /= nn; nz /= nn;
}

// minBlocks = 1 lets ptxas keep the top-k and the fp64 epilogue in registers at every KCAP (its default budget spills).
template <int KCAP>
__global__ void __launch_bounds__(128, 1)
normals_query_kernel(const float* __restrict__ xyz, int n, int max_nn, float lim, const float* __restrict__ camera,
                     const float* __restrict__ prior, const int* __restrict__ ws, float* __restrict__ normals,
                     int* __restrict__ counts)
{
    const int b = blockIdx.y;
    const GridWs L = grid_ws_layout(n, n);
    const int* W = ws + (size_t)b * L.stride;
    const GridHdr H = *reinterpret_cast<const GridHdr*>(W + L.hdr);
    const int t = blockIdx.x * 128 + threadIdx.x;
    if (t >= n) return;
    const int qi = W[L.qorder + t];
    const float* X = xyz + (size_t)b * 3 * n;
    const float qx = X[qi], qy = X[qi + n], qz = X[qi + 2 * (size_t)n];
    int cx, cy, cz;
    cell_of(H, qx, qy, qz, cx, cy, cz);
    const int* start = W + L.rstart;
    const float4* P = reinterpret_cast<const float4*>(W + L.sorted);

    KeyTopK<KCAP> top;
    top.init();
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
                        const int j = __float_as_int(r.w);
                        if (d < lim && KeyTopK<KCAP>::before(d, j, top.d[KCAP - 1], top.j[KCAP - 1]))
                            top.insert(d, j);
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
        const float bound = lb * lb * 0.999f;
        // the last key is strictly inside, or nothing unvisited can pass the radius cut (the exit radius search adds)
        if (top.d[KCAP - 1] < bound || bound >= lim) break;
    }

    // epilogue: fp64 moments of p - q over the list in (d, index) order
    int cnt = 0;
    double s1x = 0, s1y = 0, s1z = 0, sxx = 0, sxy = 0, sxz = 0, syy = 0, syz = 0, szz = 0;
#pragma unroll
    for (int s = 0; s < KCAP; ++s)
        if (s < max_nn && top.d[s] < lim) {
            const int j = top.j[s];
            const double ex = (double)__ldg(X + j) - (double)qx;
            const double ey = (double)__ldg(X + j + n) - (double)qy;
            const double ez = (double)__ldg(X + j + 2 * (size_t)n) - (double)qz;
            s1x += ex; s1y += ey; s1z += ez;
            sxx = fma(ex, ex, sxx); sxy = fma(ex, ey, sxy); sxz = fma(ex, ez, sxz);
            syy = fma(ey, ey, syy); syz = fma(ey, ez, syz); szz = fma(ez, ez, szz);
            ++cnt;
        }
    double nx = 0.0, ny = 0.0, nz = 1.0;
    if (cnt >= 3) {
        const double inv = 1.0 / (double)cnt;
        const double mx = s1x * inv, my = s1y * inv, mz = s1z * inv;
        double c[6] = {sxx * inv - mx * mx, sxy * inv - mx * my, sxz * inv - mx * mz,
                       syy * inv - my * my, syz * inv - my * mz, szz * inv - mz * mz};
        const double tr = c[0] + c[3] + c[5];
        if (tr > 0.0 && isfinite(tr)) {
            const double it = 1.0 / tr;                  // unit trace: the Jacobi thresholds are relative
#pragma unroll
            for (int e = 0; e < 6; ++e) c[e] *= it;
            smallest_eigvec3(c, nx, ny, nz);
        }
    }
    double dot = 0.0;
    if (camera != nullptr)
        dot = nx * ((double)camera[3 * b] - (double)qx) + ny * ((double)camera[3 * b + 1] - (double)qy) +
              nz * ((double)camera[3 * b + 2] - (double)qz);
    else if (prior != nullptr) {
        const float* Pr = prior + (size_t)b * 3 * n;
        dot = nx * (double)Pr[qi] + ny * (double)Pr[qi + n] + nz * (double)Pr[qi + 2 * (size_t)n];
    }
    if (dot < 0.0) { nx = -nx; ny = -ny; nz = -nz; }
    float* O = normals + (size_t)b * 3 * n + qi;
    O[0] = (float)nx; O[n] = (float)ny; O[2 * (size_t)n] = (float)nz;
    if (counts != nullptr) counts[(size_t)b * n + qi] = cnt;
}

}  // namespace

extern "C" int ri_estimate_normals_f32(const float* xyz, int B, int N, float radius, int max_nn, const float* camera,
                                       const float* prior, float* normals, int* counts, void* workspace,
                                       size_t workspace_bytes, void* stream)
{
    if (B < 0 || N < 0 || !(radius > 0.f) || max_nn <= 0 || (camera != nullptr && prior != nullptr)) return RI_ERR_BAD_ARG;
    if (max_nn > 32 || B > 65535) return RI_ERR_UNSUPPORTED;
    if (B == 0 || N == 0) return RI_OK;
    if (workspace == nullptr || ((uintptr_t)workspace & 15) != 0 ||
        workspace_bytes < (size_t)B * grid_ws_layout(N, N).stride * sizeof(int)) return RI_ERR_WORKSPACE;
    const float r2 = radius * radius;                   // fp32, +inf for an infinite radius
    const float lim = r2 < kUndefDist ? r2 : kUndefDist;
    cudaStream_t st = (cudaStream_t)stream;
    int* ws = reinterpret_cast<int*>(workspace);
    grid_setup_kernel<<<B, kSetupThreads, 0, st>>>(xyz, N, N, ws);
    RI_LAUNCH_CHECK();
    dim3 gb((N + 255) / 256, B);
    grid_bin_kernel<0><<<gb, 256, 0, st>>>(xyz, xyz, N, N, ws);
    RI_LAUNCH_CHECK();
    grid_scan_kernel<<<dim3(B, 2), 1024, 0, st>>>(N, N, ws);
    RI_LAUNCH_CHECK();
    grid_bin_kernel<1><<<gb, 256, 0, st>>>(xyz, xyz, N, N, ws);
    RI_LAUNCH_CHECK();
    dim3 gq((N + 127) / 128, B);
    if (max_nn <= 8) normals_query_kernel<8><<<gq, 128, 0, st>>>(xyz, N, max_nn, lim, camera, prior, ws, normals, counts);
    else if (max_nn <= 16) normals_query_kernel<16><<<gq, 128, 0, st>>>(xyz, N, max_nn, lim, camera, prior, ws, normals, counts);
    else if (max_nn <= 20) normals_query_kernel<20><<<gq, 128, 0, st>>>(xyz, N, max_nn, lim, camera, prior, ws, normals, counts);
    else normals_query_kernel<32><<<gq, 128, 0, st>>>(xyz, N, max_nn, lim, camera, prior, ws, normals, counts);
    RI_LAUNCH_CHECK();
    return RI_OK;
}
