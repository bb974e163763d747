// knn_grid.cu — k-nearest neighbours through a uniform hash grid, for scan-sized clouds (~50k points), sm_100a.
//
// Same contract as knn.cu / the reference's KnnKernel (/root/reference/PVCNN/modules/functional/src/knn/knn.cu:5-49,
// knn.cpp:6-25): dist [B,k,n] ascending, idx [B,k,n], slots (10000.0f, 0) when fewer than k references lie within
// d^2 < 10000, equal distances ordered by ascending reference index.  The reference scans all m references per query
// (O(n m k) with its list in global memory — seconds for a 50k-point scan); here each query looks only at the cells
// around it, and the result is still BIT-IDENTICAL to the brute-force scan because
//   * every candidate distance is the same expression  fma(dz,dz, fma(dy,dy, dx*dx)),  d* = query - reference;
//   * the k best are selected by the lexicographic key (distance, reference index), which is exactly "first k of a
//     stable sort by distance" — the order candidates are met in no longer matters;
//   * the search stops only when the k-th key is strictly below a conservative lower bound of every unvisited cell.
//
// Pipeline per call (all clouds of the batch in each launch; the first four kernels and KeyTopK live in grid.cuh, shared
// with csrc/normals.cu):
//   grid_setup    one CTA per cloud: bounding box of the references -> cubic cells, G = round(cbrt(m/2)) <= 64 per axis
//                 (about 16 points per occupied cell on surface-like scans); clears the cell histograms.
//   grid_count    cell of every reference / query (queries clamped into the grid), integer histogram.
//   grid_scan     per cloud exclusive scan of both histograms.
//   grid_scatter  counting sort: references -> float4 (x, y, z, original index) in cell order; queries -> order list.
//   grid_query    one thread per query IN CELL ORDER (a warp's queries share their neighbourhood, so the candidate
//                 loads are broadcast/L1 hits and the warp does not diverge much); sorted top-k in registers;
//                 Chebyshev rings of cells, z-runs of a ring are contiguous in the sorted array.
#include "grid.cuh"

namespace {

template <int KCAP>
__global__ void __launch_bounds__(128)
grid_query_kernel(const float* __restrict__ queries, int n, int m, int k, const int* __restrict__ ws,
                  float* __restrict__ dist, int* __restrict__ idx)
{
    const int b = blockIdx.y;
    const GridWs L = grid_ws_layout(n, m);
    const int* W = ws + (size_t)b * L.stride;
    const GridHdr H = *reinterpret_cast<const GridHdr*>(W + L.hdr);
    const int t = blockIdx.x * 128 + threadIdx.x;
    if (t >= n) return;
    const int qi = W[L.qorder + t];
    const float* Q = queries + (size_t)b * 3 * n;
    const float qx = Q[qi], qy = Q[qi + n], qz = Q[qi + 2 * (size_t)n];
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
                // on a face of the ring the whole z-run belongs to it; inside, only the two end cells do
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
                        if (d < kUndefDist && KeyTopK<KCAP>::before(d, j, top.d[KCAP - 1], top.j[KCAP - 1]))
                            top.insert(d, j);
                    }
                }
            }
        }
        // lower bound of the distance to anything outside the visited block (faces on the grid border: nothing beyond)
        float lb = INFINITY;
        if (cx - R > 0) lb = fminf(lb, qx - (H.ox + (float)(cx - R) * H.h));
        if (cx + R < H.gx - 1) lb = fminf(lb, (H.ox + (float)(cx + R + 1) * H.h) - qx);
        if (cy - R > 0) lb = fminf(lb, qy - (H.oy + (float)(cy - R) * H.h));
        if (cy + R < H.gy - 1) lb = fminf(lb, (H.oy + (float)(cy + R + 1) * H.h) - qy);
        if (cz - R > 0) lb = fminf(lb, qz - (H.oz + (float)(cz - R) * H.h));
        if (cz + R < H.gz - 1) lb = fminf(lb, (H.oz + (float)(cz + R + 1) * H.h) - qz);
        lb = fmaxf(lb - 1e-3f * H.h, 0.f);                      // cell assignment and the bound itself are rounded
        const float bound = lb * lb * 0.999f;
        if (top.d[KCAP - 1] < bound || bound >= kUndefDist) break;   // k-th key strictly inside, or nothing insertable left
    }
    float* od = dist + (size_t)b * k * n + qi;
    int* oi = idx + (size_t)b * k * n + qi;
#pragma unroll
    for (int s = 0; s < KCAP; ++s)
        if (s < k) { od[(size_t)s * n] = top.d[s]; oi[(size_t)s * n] = top.j[s]; }
}

}  // namespace

extern "C" size_t ri_knn_grid_workspace_bytes(int B, int n, int m)
{
    if (B <= 0 || n < 0 || m < 0) return 16;
    return (size_t)B * grid_ws_layout(n, m).stride * sizeof(int) + 16;
}

extern "C" int ri_knn_grid_f32(const float* xyz1, const float* xyz2, int B, int n, int m, int k,
                               float* dist1, int* idx1, void* workspace, size_t workspace_bytes, void* stream)
{
    if (B < 0 || n < 0 || m < 0 || k <= 0) return RI_ERR_BAD_ARG;
    if (k > 32 || B > 65535) return RI_ERR_UNSUPPORTED;
    if (B == 0 || n == 0) return RI_OK;
    if (workspace == nullptr || ((uintptr_t)workspace & 15) != 0 ||
        workspace_bytes < (size_t)B * grid_ws_layout(n, m).stride * sizeof(int)) return RI_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    int* ws = reinterpret_cast<int*>(workspace);
    grid_setup_kernel<<<B, kSetupThreads, 0, st>>>(xyz2, m, n, ws);
    RI_LAUNCH_CHECK();
    const int big = n > m ? n : m;
    dim3 gb((big + 255) / 256, B);
    grid_bin_kernel<0><<<gb, 256, 0, st>>>(xyz1, xyz2, n, m, ws);
    RI_LAUNCH_CHECK();
    grid_scan_kernel<<<dim3(B, 2), 1024, 0, st>>>(n, m, ws);
    RI_LAUNCH_CHECK();
    grid_bin_kernel<1><<<gb, 256, 0, st>>>(xyz1, xyz2, n, m, ws);
    RI_LAUNCH_CHECK();
    dim3 gq((n + 127) / 128, B);
    if (k <= 8) grid_query_kernel<8><<<gq, 128, 0, st>>>(xyz1, n, m, k, ws, dist1, idx1);
    else if (k <= 16) grid_query_kernel<16><<<gq, 128, 0, st>>>(xyz1, n, m, k, ws, dist1, idx1);
    else if (k <= 20) grid_query_kernel<20><<<gq, 128, 0, st>>>(xyz1, n, m, k, ws, dist1, idx1);
    else grid_query_kernel<32><<<gq, 128, 0, st>>>(xyz1, n, m, k, ws, dist1, idx1);
    RI_LAUNCH_CHECK();
    return RI_OK;
}
