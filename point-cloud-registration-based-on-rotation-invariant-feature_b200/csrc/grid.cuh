// grid.cuh — the uniform hash grid over a batch of clouds shared by csrc/knn_grid.cu (k-NN) and csrc/normals.cu (normal
// estimation): per-cloud workspace layout, bounding-box setup, counting-sort binning of references and queries, and the
// register top-k of (distance, index) keys.  See knn_grid.cu for the search built on it.
#pragma once
#include "ri_common.cuh"

namespace {

constexpr float kUndefDist = 10000.0f;
constexpr int kMaxG = 64;
constexpr int kSetupThreads = 1024;

struct GridHdr {               // per cloud, 16 ints at the head of its workspace slab
    float ox, oy, oz, h, inv_h;
    int gx, gy, gz;
    int pad[8];
};

__host__ __device__ inline int grid_g(int m)
{
    int g = 1;
    while ((long long)(g + 1) * (g + 1) * (g + 1) * 2 <= (long long)(m > 0 ? m : 1) && g < kMaxG) ++g;   // ~cbrt(m/2)
    return g;
}

struct GridWs {                // int32 offsets inside one cloud's slab
    int hdr, rstart, rcur, qstart, qcur, qorder, sorted, stride, cells_max;
};
__host__ __device__ inline GridWs grid_ws_layout(int n, int m)
{
    GridWs w;
    const int g = grid_g(m);
    w.cells_max = g * g * g;
    int o = 0;
    w.hdr = o; o += 16;
    w.rstart = o; o += w.cells_max + 1;
    w.rcur = o; o += w.cells_max;
    w.qstart = o; o += w.cells_max + 1;
    w.qcur = o; o += w.cells_max;
    w.qorder = o; o += n;
    o = (o + 3) / 4 * 4;
    w.sorted = o; o += 4 * m;                                   // float4 per reference
    w.stride = (o + 3) / 4 * 4;
    return w;
}

__device__ __forceinline__ int cell_of(const GridHdr& H, float x, float y, float z, int& cx, int& cy, int& cz)
{
    cx = min(max((int)floorf((x - H.ox) * H.inv_h), 0), H.gx - 1);
    cy = min(max((int)floorf((y - H.oy) * H.inv_h), 0), H.gy - 1);
    cz = min(max((int)floorf((z - H.oz) * H.inv_h), 0), H.gz - 1);
    return (cx * H.gy + cy) * H.gz + cz;
}

__global__ void __launch_bounds__(kSetupThreads)
grid_setup_kernel(const float* __restrict__ refs, int m, int n, int* __restrict__ ws)
{
    __shared__ float smin[3][kSetupThreads / 32], smax[3][kSetupThreads / 32];
    const int b = blockIdx.x, tid = threadIdx.x;
    const GridWs L = grid_ws_layout(n, m);
    int* W = ws + (size_t)b * L.stride;
    const float* R = refs + (size_t)b * 3 * m;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int j = tid; j < m; j += kSetupThreads)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = R[j + (size_t)a * m];
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
            if (!(l <= h)) { l = 0.f; h = 0.f; }               // empty or NaN cloud
            (a == 0 ? H.ox : a == 1 ? H.oy : H.oz) = l;
            e[a] = h - l;
        }
        const int g = grid_g(m);
        const float emax = fmaxf(e[0], fmaxf(e[1], e[2]));
        H.h = emax > 0.f ? emax / (float)g : 1.0f;
        H.inv_h = 1.0f / H.h;
        H.gx = min(g, (int)(e[0] * H.inv_h) + 1);
        H.gy = min(g, (int)(e[1] * H.inv_h) + 1);
        H.gz = min(g, (int)(e[2] * H.inv_h) + 1);
        *reinterpret_cast<GridHdr*>(W + L.hdr) = H;
    }
    for (int c = tid; c < L.cells_max; c += kSetupThreads) { W[L.rcur + c] = 0; W[L.qcur + c] = 0; }
}

// pass 0: histogram into *cur; pass 1: scatter using *start + atomic cursor
template <int PASS>
__global__ void __launch_bounds__(256)
grid_bin_kernel(const float* __restrict__ queries, const float* __restrict__ refs, int n, int m, int* __restrict__ ws)
{
    const int b = blockIdx.y;
    const GridWs L = grid_ws_layout(n, m);
    int* W = ws + (size_t)b * L.stride;
    const GridHdr H = *reinterpret_cast<const GridHdr*>(W + L.hdr);
    const int t = blockIdx.x * 256 + threadIdx.x;
    int cx, cy, cz;
    if (t < m) {
        const float* R = refs + (size_t)b * 3 * m;
        const float x = R[t], y = R[t + m], z = R[t + 2 * (size_t)m];
        const int c = cell_of(H, x, y, z, cx, cy, cz);
        if (PASS == 0) atomicAdd(W + L.rcur + c, 1);
        else {
            const int pos = W[L.rstart + c] + atomicAdd(W + L.rcur + c, 1);
            reinterpret_cast<float4*>(W + L.sorted)[pos] = make_float4(x, y, z, __int_as_float(t));
        }
    }
    if (t < n) {
        const float* Q = queries + (size_t)b * 3 * n;
        const int c = cell_of(H, Q[t], Q[t + n], Q[t + 2 * (size_t)n], cx, cy, cz);
        if (PASS == 0) atomicAdd(W + L.qcur + c, 1);
        else W[L.qorder + W[L.qstart + c] + atomicAdd(W + L.qcur + c, 1)] = t;
    }
}

// exclusive scan of the two histograms of a cloud; the cursors are reset to 0 for the scatter pass
__global__ void __launch_bounds__(1024)
grid_scan_kernel(int n, int m, int* __restrict__ ws)
{
    __shared__ int swarp[32];
    __shared__ int scarry, stotal;
    const int b = blockIdx.x, which = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const GridWs L = grid_ws_layout(n, m);
    int* W = ws + (size_t)b * L.stride;
    int* cur = W + (which ? L.qcur : L.rcur);
    int* start = W + (which ? L.qstart : L.rstart);
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
            swarp[lane] = wi - w;                               // exclusive offset of each warp
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

template <int KCAP>
struct KeyTopK {
    float d[KCAP];
    int j[KCAP];
    __device__ __forceinline__ void init()
    {
#pragma unroll
        for (int q = 0; q < KCAP; ++q) { d[q] = kUndefDist; j[q] = 0; }
    }
    static __device__ __forceinline__ bool before(float x, int xi, float y, int yi)
    {
        return x < y || (x == y && xi < yi);
    }
    // caller guarantees x < 10000 (so it sorts before every sentinel slot) and (x, idx) before slot KCAP-1
    __device__ __forceinline__ void insert(float x, int idx)
    {
#pragma unroll
        for (int q = KCAP - 1; q > 0; --q) {
            const bool up = before(x, idx, d[q - 1], j[q - 1]);
            const bool here = before(x, idx, d[q], j[q]);
            d[q] = up ? d[q - 1] : (here ? x : d[q]);
            j[q] = up ? j[q - 1] : (here ? idx : j[q]);
        }
        const bool first = before(x, idx, d[0], j[0]);
        d[0] = first ? x : d[0];
        j[0] = first ? idx : j[0];
    }
};

}  // namespace
