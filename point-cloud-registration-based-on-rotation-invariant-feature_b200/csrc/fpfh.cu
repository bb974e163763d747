// fpfh.cu — Fast Point Feature Histograms (Rusu, Blodow, Beetz, ICRA 2009) of xyz + normal clouds, Open3D's
// compute_fpfh_feature with KDTreeSearchParamHybrid, a batch of B clouds per call, sm_100a.  The contract is restated in
// include/ri_b200.h (ri_compute_fpfh_f32) and DESIGN.md §8 (row f8).
//
// For each point q of a cloud xyz [3,N], normals [3,N]:
//   neighbours  the max_nn (<= 128) smallest keys (d, index) among the points with d < min(radius^2, 10000), q included,
//               d = fma(dz,dz, fma(dy,dy, dx*dx)), d* = q - p in fp32: the rule of csrc/normals.cu, so the list is the
//               first max_nn entries of the k-NN whose distance passes the cut;
//   SPFH        the pair features of (q, n_q) with each list entry after position 0, binned 3 x 11, as counts;
//   FPFH        the SPFH of the list entries weighted by 1 / |p - q|^2 and normalised per group, plus q's own SPFH.
//
// Pipeline per call: the grid build of grid.cuh (4 launches), then
//   fpfh_spfh_kernel  one warp per point in cell order.  The ring search of normals_query_kernel, but with an exact
//                     streaming top-k in shared memory instead of the register top-k: passing (d bits << 32 | index) keys
//                     are appended to a per-warp buffer of kBuf keys; when it would overflow, a warp bitonic sort keeps the
//                     best max_nn, and the max_nn-th key prunes later candidates.  The ring stops when max_nn buffered keys
//                     are strictly inside the bound of the unvisited cells, or when that bound reaches the radius cut.  The
//                     lanes then compute the pair features of the sorted list and count the bins (integer shared atomics).
//                     It writes the list (int32) and the packed counts (33 bytes + n in one byte, 9 words) per point.
//   fpfh_kernel       one thread per point: gathers the neighbours' packed counts in list order and accumulates in fp64.
// No float atomics: every sum is in a fixed order, so a point's result depends only on its cloud and is bit-reproducible.
#include "grid.cuh"

namespace {

constexpr int kFpfhMaxNN = 128;
constexpr int kBuf = 256;              // keys per warp: after a compaction at most 128 remain, so a 32-key round always fits
constexpr int kWarps = 4;              // warps (points) per CTA of the search kernel
constexpr int kPackWords = 9;          // 33 count bytes + n
constexpr unsigned long long kNoKey = ~0ull;

struct FpfhWs {                        // byte offsets inside the workspace
    size_t grid, lists, packed, total;
};
__host__ __device__ inline FpfhWs fpfh_ws_layout(int B, int N, int max_nn)
{
    FpfhWs w;
    w.grid = 0;
    w.lists = (size_t)B * grid_ws_layout(N, N).stride * sizeof(int);
    w.packed = w.lists + ((size_t)B * N * max_nn * sizeof(int) + 15) / 16 * 16;
    w.total = w.packed + ((size_t)B * N * kPackWords * sizeof(int) + 15) / 16 * 16;
    return w;
}

// Ascending bitonic sort of the warp's kBuf keys in shared memory.
__device__ __forceinline__ void warp_sort(unsigned long long* buf, int lane)
{
    __syncwarp();
    for (int k = 2; k <= kBuf; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int i = lane; i < kBuf / 2; i += 32) {
                const int lo = 2 * j * (i / j) + (i % j), hi = lo + j;
                const unsigned long long a = buf[lo], b = buf[hi];
                if ((a > b) == ((lo & k) == 0)) { buf[lo] = b; buf[hi] = a; }
            }
            __syncwarp();
        }
}

// Sort the first cnt keys (the rest padded) and keep the best min(cnt, keep); returns the new count.
__device__ __forceinline__ int warp_compact(unsigned long long* buf, int cnt, int keep, int lane)
{
    __syncwarp();
    for (int s = cnt + lane; s < kBuf; s += 32) buf[s] = kNoKey;
    warp_sort(buf, lane);
    return min(cnt, keep);
}

__device__ __forceinline__ double dot3(double ax, double ay, double az, double bx, double by, double bz)
{
    return __dadd_rn(__dadd_rn(__dmul_rn(ax, bx), __dmul_rn(ay, by)), __dmul_rn(az, bz));
}

// Open3D's ComputePairFeatures of (p1, n1) with (p2, n2) in fp64, each operation rounded (no contraction) -> bins.
__device__ __forceinline__ void pair_feature_bins(double p1x, double p1y, double p1z, double n1x, double n1y, double n1z,
                                                  double p2x, double p2y, double p2z, double n2x, double n2y, double n2z,
                                                  int& b0, int& b1, int& b2)
{
    double f0 = 0.0, f1 = 0.0, f2 = 0.0;
    double dx = __dsub_rn(p2x, p1x), dy = __dsub_rn(p2y, p1y), dz = __dsub_rn(p2z, p1z);
    const double L = __dsqrt_rn(dot3(dx, dy, dz, dx, dy, dz));
    if (L != 0.0) {
        const double a1 = __ddiv_rn(dot3(n1x, n1y, n1z, dx, dy, dz), L);
        const double a2 = __ddiv_rn(dot3(n2x, n2y, n2z, dx, dy, dz), L);
        double ux = n1x, uy = n1y, uz = n1z, sx = n2x, sy = n2y, sz = n2z;     // n1', n2'
        if (acos(fabs(a1)) > acos(fabs(a2))) {
            ux = n2x; uy = n2y; uz = n2z; sx = n1x; sy = n1y; sz = n1z;
            dx = -dx; dy = -dy; dz = -dz;
            f2 = -a2;
        } else {
            f2 = a1;
        }
        double vx = __dsub_rn(__dmul_rn(dy, uz), __dmul_rn(dz, uy));         // v = dp x n1'
        double vy = __dsub_rn(__dmul_rn(dz, ux), __dmul_rn(dx, uz));
        double vz = __dsub_rn(__dmul_rn(dx, uy), __dmul_rn(dy, ux));
        const double vn = __dsqrt_rn(dot3(vx, vy, vz, vx, vy, vz));
        if (vn != 0.0) {
            vx = __ddiv_rn(vx, vn); vy = __ddiv_rn(vy, vn); vz = __ddiv_rn(vz, vn);
            const double wx = __dsub_rn(__dmul_rn(uy, vz), __dmul_rn(uz, vy)); // w = n1' x v
            const double wy = __dsub_rn(__dmul_rn(uz, vx), __dmul_rn(ux, vz));
            const double wz = __dsub_rn(__dmul_rn(ux, vy), __dmul_rn(uy, vx));
            f1 = dot3(vx, vy, vz, sx, sy, sz);
            f0 = atan2(dot3(wx, wy, wz, sx, sy, sz), dot3(ux, uy, uz, sx, sy, sz));
        } else {
            f2 = 0.0;
        }
    }
    b0 = (int)floor(__ddiv_rn(__dmul_rn(11.0, __dadd_rn(f0, RI_PI)), __dmul_rn(2.0, RI_PI)));
    b1 = (int)floor(__dmul_rn(__dmul_rn(11.0, __dadd_rn(f1, 1.0)), 0.5));
    b2 = (int)floor(__dmul_rn(__dmul_rn(11.0, __dadd_rn(f2, 1.0)), 0.5));
    b0 = min(max(b0, 0), 10); b1 = min(max(b1, 0), 10); b2 = min(max(b2, 0), 10);
}

__device__ __forceinline__ double count_of(const unsigned* w, int j) { return (double)((w[j >> 2] >> (8 * (j & 3))) & 0xffu); }

// minBlocks = 4 (16 warps an SM) keeps ptxas from the 64-register budget that spills around the libdevice acos / atan2.
__global__ void __launch_bounds__(kWarps * 32, 4)
fpfh_spfh_kernel(const float* __restrict__ xyz, const float* __restrict__ normals, int n, int max_nn, float lim,
                 const int* __restrict__ ws, int* __restrict__ lists, unsigned* __restrict__ packed,
                 float* __restrict__ spfh, int* __restrict__ counts)
{
    __shared__ unsigned long long sbuf[kWarps][kBuf];
    __shared__ int shist[kWarps][33];
    const int b = blockIdx.y, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const GridWs L = grid_ws_layout(n, n);
    const int* W = ws + (size_t)b * L.stride;
    const GridHdr H = *reinterpret_cast<const GridHdr*>(W + L.hdr);
    const int t = blockIdx.x * kWarps + wid;
    if (t >= n) return;                                 // warp-uniform
    unsigned long long* buf = sbuf[wid];
    int* hist = shist[wid];
    const int qi = W[L.qorder + t];
    const float* X = xyz + (size_t)b * 3 * n;
    const float* Nm = normals + (size_t)b * 3 * n;
    const float qx = X[qi], qy = X[qi + n], qz = X[qi + 2 * (size_t)n];
    int cx, cy, cz;
    cell_of(H, qx, qy, qz, cx, cy, cz);
    const int* start = W + L.rstart;
    const float4* P = reinterpret_cast<const float4*>(W + L.sorted);
    const unsigned lt = (1u << lane) - 1u;

    int cnt = 0;
    unsigned long long thr = kNoKey;                    // the max_nn-th key once known: later keys must sort before it
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
                    for (int pb = p0; pb < p1; pb += 32) {
                        const int p = pb + lane;
                        unsigned long long key = kNoKey;
                        bool pass = false;
                        if (p < p1) {
                            const float4 r = __ldg(P + p);
                            const float dx = __fsub_rn(qx, r.x), dy = __fsub_rn(qy, r.y), dz = __fsub_rn(qz, r.z);
                            const float d = __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
                            key = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)__float_as_int(r.w);
                            pass = d < lim && key < thr;
                        }
                        unsigned m = __ballot_sync(0xffffffffu, pass);
                        if (m == 0u) continue;
                        if (cnt + __popc(m) > kBuf) {           // compaction: cnt > kBuf - 32 >= max_nn, so max_nn remain
                            cnt = warp_compact(buf, cnt, max_nn, lane);
                            thr = buf[max_nn - 1];
                            pass = pass && key < thr;
                            m = __ballot_sync(0xffffffffu, pass);
                        }
                        if (pass) buf[cnt + __popc(m & lt)] = key;
                        cnt += __popc(m);
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
        if (bound >= lim) break;                        // nothing unvisited can pass the radius cut
        __syncwarp();
        int inside = 0;                                 // buffered keys strictly inside the bound
        for (int s = lane; s < cnt; s += 32) inside += __uint_as_float((unsigned)(buf[s] >> 32)) < bound;
        if (__reduce_add_sync(0xffffffffu, inside) >= max_nn) break;
    }
    const int nl = warp_compact(buf, cnt, max_nn, lane);

    // the list, and the binned pair features of (q, n_q) with list positions 1 .. nl-1
    int* lst = lists + ((size_t)b * n + qi) * max_nn;
    for (int s = lane; s < 33; s += 32) hist[s] = 0;
    const double q0 = qx, q1 = qy, q2 = qz;
    const double m0 = Nm[qi], m1 = Nm[qi + n], m2 = Nm[qi + 2 * (size_t)n];
    __syncwarp();
    for (int s = lane; s < nl; s += 32) {
        const int j = (int)(unsigned)(buf[s] & 0xffffffffull);
        lst[s] = j;
        if (s == 0) continue;
        int b0, b1, b2;
        pair_feature_bins(q0, q1, q2, m0, m1, m2, (double)__ldg(X + j), (double)__ldg(X + j + n),
                          (double)__ldg(X + j + 2 * (size_t)n), (double)__ldg(Nm + j), (double)__ldg(Nm + j + n),
                          (double)__ldg(Nm + j + 2 * (size_t)n), b0, b1, b2);
        atomicAdd(hist + b0, 1); atomicAdd(hist + 11 + b1, 1); atomicAdd(hist + 22 + b2, 1);
    }
    __syncwarp();
    if (lane < kPackWords) {
        unsigned w = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int j = 4 * lane + e;
            const unsigned v = j < 33 ? (unsigned)hist[j] : (j == 33 ? (unsigned)nl : 0u);
            w |= v << (8 * e);
        }
        packed[((size_t)b * n + qi) * kPackWords + lane] = w;
    }
    if (spfh != nullptr) {
        const double incr = nl > 1 ? __ddiv_rn(100.0, (double)(nl - 1)) : 0.0;
        for (int j = lane; j < 33; j += 32)
            spfh[((size_t)b * 33 + j) * n + qi] = (float)__dmul_rn((double)hist[j], incr);
    }
    if (counts != nullptr && lane == 0) counts[(size_t)b * n + qi] = nl;
}

// minBlocks = 2 leaves ptxas room for the 33 fp64 accumulators without spilling.
__global__ void __launch_bounds__(128, 2)
fpfh_kernel(const float* __restrict__ xyz, int n, int max_nn, const int* __restrict__ lists,
            const unsigned* __restrict__ packed, float* __restrict__ fpfh)
{
    const int b = blockIdx.y;
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= n) return;
    const float* X = xyz + (size_t)b * 3 * n;
    const unsigned* PK = packed + (size_t)b * n * kPackWords;
    unsigned own[kPackWords];
#pragma unroll
    for (int e = 0; e < kPackWords; ++e) own[e] = PK[(size_t)i * kPackWords + e];
    const int nq = (int)(own[8] >> 8) & 0xff;
    float* O = fpfh + (size_t)b * 33 * n + i;
    if (nq <= 1) {
#pragma unroll
        for (int j = 0; j < 33; ++j) O[(size_t)j * n] = 0.f;
        return;
    }
    const double qx = X[i], qy = X[i + n], qz = X[i + 2 * (size_t)n];
    const int* lst = lists + ((size_t)b * n + i) * max_nn;
    double feat[33], sum[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int j = 0; j < 33; ++j) feat[j] = 0.0;
    for (int k = 1; k < nq; ++k) {
        const int p = __ldg(lst + k);
        const double dx = __dsub_rn((double)__ldg(X + p), qx), dy = __dsub_rn((double)__ldg(X + p + n), qy);
        const double dz = __dsub_rn((double)__ldg(X + p + 2 * (size_t)n), qz);
        const double w = dot3(dx, dy, dz, dx, dy, dz);
        if (w == 0.0) continue;
        unsigned c[kPackWords];
#pragma unroll
        for (int e = 0; e < kPackWords; ++e) c[e] = __ldg(PK + (size_t)p * kPackWords + e);
        const int np = (int)(c[8] >> 8) & 0xff;
        if (np <= 1) continue;                          // an all-zero SPFH adds +0 everywhere
        const double incr = __ddiv_rn(100.0, (double)(np - 1));
#pragma unroll
        for (int j = 0; j < 33; ++j) {
            const double val = __ddiv_rn(__dmul_rn(count_of(c, j), incr), w);
            feat[j] = __dadd_rn(feat[j], val);
            sum[j / 11] = __dadd_rn(sum[j / 11], val);
        }
    }
    const double incr = __ddiv_rn(100.0, (double)(nq - 1));
#pragma unroll
    for (int g = 0; g < 3; ++g) sum[g] = sum[g] != 0.0 ? __ddiv_rn(100.0, sum[g]) : 0.0;
#pragma unroll
    for (int j = 0; j < 33; ++j)
        O[(size_t)j * n] = (float)__dadd_rn(__dmul_rn(feat[j], sum[j / 11]), __dmul_rn(count_of(own, j), incr));
}

}  // namespace

extern "C" size_t ri_fpfh_workspace_bytes(int B, int N, int max_nn)
{
    if (B <= 0 || N <= 0 || max_nn <= 0 || max_nn > kFpfhMaxNN) return 16;
    return fpfh_ws_layout(B, N, max_nn).total + 16;
}

extern "C" int ri_compute_fpfh_f32(const float* xyz, const float* normals, int B, int N, float radius, int max_nn,
                                   float* fpfh, float* spfh, int* counts, void* workspace, size_t workspace_bytes,
                                   void* stream)
{
    if (B < 0 || N < 0 || !(radius > 0.f) || max_nn <= 0) return RI_ERR_BAD_ARG;
    if (max_nn > kFpfhMaxNN || B > 65535) return RI_ERR_UNSUPPORTED;
    if (B == 0 || N == 0) return RI_OK;
    const FpfhWs F = fpfh_ws_layout(B, N, max_nn);
    if (workspace == nullptr || ((uintptr_t)workspace & 15) != 0 || workspace_bytes < F.total) return RI_ERR_WORKSPACE;
    const float r2 = radius * radius;                   // fp32, +inf for an infinite radius
    const float lim = r2 < kUndefDist ? r2 : kUndefDist;
    cudaStream_t st = (cudaStream_t)stream;
    char* base = reinterpret_cast<char*>(workspace);
    int* ws = reinterpret_cast<int*>(base + F.grid);
    int* lists = reinterpret_cast<int*>(base + F.lists);
    unsigned* packed = reinterpret_cast<unsigned*>(base + F.packed);
    grid_setup_kernel<<<B, kSetupThreads, 0, st>>>(xyz, N, N, ws);
    RI_LAUNCH_CHECK();
    dim3 gb((N + 255) / 256, B);
    grid_bin_kernel<0><<<gb, 256, 0, st>>>(xyz, xyz, N, N, ws);
    RI_LAUNCH_CHECK();
    grid_scan_kernel<<<dim3(B, 2), 1024, 0, st>>>(N, N, ws);
    RI_LAUNCH_CHECK();
    grid_bin_kernel<1><<<gb, 256, 0, st>>>(xyz, xyz, N, N, ws);
    RI_LAUNCH_CHECK();
    fpfh_spfh_kernel<<<dim3((N + kWarps - 1) / kWarps, B), kWarps * 32, 0, st>>>(xyz, normals, N, max_nn, lim, ws, lists,
                                                                                packed, spfh, counts);
    RI_LAUNCH_CHECK();
    fpfh_kernel<<<dim3((N + 127) / 128, B), 128, 0, st>>>(xyz, N, max_nn, lists, packed, fpfh);
    RI_LAUNCH_CHECK();
    return RI_OK;
}
