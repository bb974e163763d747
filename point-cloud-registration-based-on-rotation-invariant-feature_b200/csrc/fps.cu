// fps.cu — batched farthest point sampling over variable-length clouds (SURVEY.md 8f, row f12; include/ri_b200.h states
// the contract).  FPS is m dependent arg-max reductions over n points: its cost is the latency of one sample, repeated.
//
// One cluster of C CTAs per cloud (C in {1, 2, 4, 8, 16}, chosen from N and B).  CTA `rank` owns the contiguous slice
// [rank * P, rank * P + P) of the cloud, P = kPPT * blockDim.x; thread t holds the points rank * P + t + j * blockDim.x,
// j < kPPT, in registers (xyz fp32, dist fp64) and a copy of the slice's xyz in shared memory, from which the CTA's
// candidate's coordinates are read.  Per sample:
//   1. every thread updates its dist and keeps its best (dist bits, index): dist >= 0 or +inf, never NaN or -0, so the
//      uint64 order of the bits is the fp64 order, and points are visited in ascending index with a strict >, so the
//      lowest index wins ties;
//   2. the warp reduces with redux.sync (max of the high word, max of the low word among the lanes that hold it, min of
//      the index among the lanes that hold both), lane 0 writes a per-warp slot;
//   3. C == 1: __syncthreads, then every warp reduces the per-warp slots itself.  C > 1: __syncthreads, warp 0 reduces
//      the per-warp slots and writes the CTA's candidate (with its coordinates) into cta_slot[k & 1], one
//      barrier.cluster arrive / wait, then every warp reads the C slots over DSMEM and computes the same winner.
//      The winner's coordinates travel with it in the slot.
// Why one cluster barrier per sample is enough: CTA r writes cta_slot[k & 1] only at samples k, k + 2, ...; a remote reader
// of sample k reads it between barrier k and its own arrival at barrier k + 1, and CTA r cannot pass barrier k + 1 (and so
// cannot reach sample k + 2) before every CTA has arrived there.  Sample k + 1 writes the other slot.  The per-warp slots
// of the C == 1 form are double-buffered by the same argument with __syncthreads; in the C > 1 form they are read by
// warp 0 before it arrives at the cluster barrier, which every warp passes before sample k + 1 writes them again.  The
// first remote read follows barrier 0 (every CTA of the cluster is running); a last barrier keeps each CTA's shared memory
// alive until the other CTAs have read it.
// When the winner's distance is 0 no later sample can change s (dist only decreases): the cluster stops and rank 0 writes
// the remaining indices.  No float atomics, no workspace, no host synchronisation.
#include "ri_common.cuh"
#include "ri_b200.h"

#include <limits.h>

namespace {

constexpr int kPPT = 16;                          // points per thread
constexpr int kMaxThreads = 512;                  // threads per CTA (kPPT * 512 = 8192 points per CTA)
constexpr int kMaxWarps = kMaxThreads / 32;
constexpr int kMaxPointsPerCta = kPPT * kMaxThreads;
constexpr int kMaxClusterPortable = 8;
constexpr int kMaxCluster = 16;
static_assert(RI_FPS_MAX_POINTS == kMaxCluster * kMaxPointsPerCta, "the header's limit is what 16-CTA clusters hold");
constexpr unsigned kFull = 0xffffffffu;

struct alignas(16) Slot {                         // one candidate: fp64 distance bits, index, coordinates
    unsigned long long bits;
    int idx;
    float x, y, z;
    int pad[1];
};

__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// One cluster barrier that orders shared memory only.  barrier.cluster.arrive.release orders global memory too and compiles
// to MEMBAR.ALL.GPU; the exchange here is through shared memory, so the release / acquire fences are restricted to it
// (MEMBAR.ALL.CTA).
__device__ __forceinline__ void cluster_sync_shared()
{
    asm volatile("fence.release.sync_restrict::shared::cta.cluster;" ::: "memory");
    asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
    asm volatile("fence.acquire.sync_restrict::shared::cluster.cluster;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ Slot ld_slot_cluster(uint32_t addr)
{
    uint32_t a, b, c, d, e, f;
    asm volatile("ld.shared::cluster.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr) : "memory");
    asm volatile("ld.shared::cluster.v2.u32 {%0, %1}, [%2];" : "=r"(e), "=r"(f) : "r"(addr + 16) : "memory");
    Slot s;
    s.bits = ((unsigned long long)b << 32) | a;
    s.idx = (int)c;
    s.x = __uint_as_float(d);
    s.y = __uint_as_float(e);
    s.z = __uint_as_float(f);
    return s;
}

// Arg-max over the lanes of a warp: the largest bits, the lowest index among equal bits.  Every lane gets the result.
__device__ __forceinline__ void warp_argmax(unsigned long long& bits, int& idx)
{
    const unsigned hi = __reduce_max_sync(kFull, (unsigned)(bits >> 32));
    const unsigned lo = __reduce_max_sync(kFull, (unsigned)(bits >> 32) == hi ? (unsigned)bits : 0u);
    const unsigned long long best = ((unsigned long long)hi << 32) | lo;
    idx = (int)__reduce_min_sync(kFull, bits == best ? (unsigned)idx : (unsigned)INT_MAX);
    bits = best;
}

// The coordinates held by the lane whose (bits, idx) equals the warp's arg-max (lowest such lane).
__device__ __forceinline__ void warp_bcast_winner(bool mine, float& x, float& y, float& z)
{
    const unsigned who = __ballot_sync(kFull, mine);
    const int src = who ? __ffs(who) - 1 : 0;
    x = __shfl_sync(kFull, x, src);
    y = __shfl_sync(kFull, y, src);
    z = __shfl_sync(kFull, z, src);
}

__global__ void __launch_bounds__(kMaxThreads, 1)
fps_kernel(const float* __restrict__ xyz, const int* __restrict__ lengths, int N, int m, int C, int* __restrict__ out)
{
    extern __shared__ float s_xyz[];                       // [3][P]: the slice's x, y, z
    __shared__ Slot warp_slot[2][kMaxWarps];
    __shared__ Slot cta_slot[2];

    const int T = blockDim.x, t = threadIdx.x, lane = t & 31, warp = t >> 5, nwarps = T >> 5;
    const int P = kPPT * T;
    const int rank = C > 1 ? (int)cluster_ctarank() : 0;
    const int b = blockIdx.x / C;
    const int base = rank * P;
    int n = lengths ? lengths[b] : N;
    n = n < 0 ? 0 : (n > N ? N : n);
    int* o = out + (size_t)b * m;
    if (n == 0) {                                          // uniform over the cluster: no barrier, no remote access
        if (rank == 0)
            for (int k = t; k < m; k += T) o[k] = -1;
        return;
    }
    const float* X = xyz + (size_t)b * 3 * N;
    float* sx_ = s_xyz;
    float* sy_ = s_xyz + P;
    float* sz_ = s_xyz + 2 * P;

    float px[kPPT], py[kPPT], pz[kPPT];
    double dist[kPPT];
#pragma unroll
    for (int j = 0; j < kPPT; ++j) {
        const int i = base + t + j * T;
        const bool valid = i < n;                          // points past n_b are never read and never selected
        px[j] = valid ? X[i] : 0.0f;
        py[j] = valid ? X[N + i] : 0.0f;
        pz[j] = valid ? X[2 * N + i] : 0.0f;
        dist[j] = valid ? __longlong_as_double(0x7ff0000000000000ll) : 0.0;
        sx_[t + j * T] = px[j];
        sy_[t + j * T] = py[j];
        sz_[t + j * T] = pz[j];
    }
    __syncthreads();                                       // lane 0 of each warp reads any point of the slice
    // s = 0; its coordinates from global memory (the first sample precedes any exchange)
    int s = 0;
    float cx = X[0], cy = X[N], cz = X[2 * N];

    for (int k = 0;; ++k) {
        if (rank == 0 && t == 0) o[k] = s;
        if (k == m - 1) break;
        const double qx = (double)cx, qy = (double)cy, qz = (double)cz;
        unsigned long long bb = 0ull;
        int bj = -1;
#pragma unroll
        for (int j = 0; j < kPPT; ++j) {
            const double dx = __dsub_rn((double)px[j], qx);
            const double dy = __dsub_rn((double)py[j], qy);
            const double dz = __dsub_rn((double)pz[j], qz);
            const double d = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
            dist[j] = d < dist[j] ? d : dist[j];
            const unsigned long long db = (unsigned long long)__double_as_longlong(dist[j]);
            if (db > bb) { bb = db; bj = j; }
        }
        int bi = bj < 0 ? INT_MAX : base + t + bj * T;
        warp_argmax(bb, bi);
        const int buf = k & 1;
        if (lane == 0) {
            Slot w;
            w.bits = bb;
            w.idx = bi;
            if (bi != INT_MAX) { w.x = sx_[bi - base]; w.y = sy_[bi - base]; w.z = sz_[bi - base]; }
            else { w.x = w.y = w.z = 0.0f; }
            warp_slot[buf][warp] = w;
        }
        __syncthreads();

        Slot c;
        if (C == 1) {
            c = lane < nwarps ? warp_slot[buf][lane] : Slot{0ull, INT_MAX, 0.0f, 0.0f, 0.0f, {0}};
        } else {
            if (warp == 0) {
                Slot w = lane < nwarps ? warp_slot[buf][lane] : Slot{0ull, INT_MAX, 0.0f, 0.0f, 0.0f, {0}};
                unsigned long long wb = w.bits;
                int wi = w.idx;
                warp_argmax(wb, wi);
                warp_bcast_winner(w.bits == wb && w.idx == wi, w.x, w.y, w.z);
                if (lane == 0) { w.bits = wb; w.idx = wi; cta_slot[buf] = w; }
            }
            cluster_sync_shared();
            c = lane < C ? ld_slot_cluster(mapa_shared(ri_smem_u32(&cta_slot[buf]), (uint32_t)lane))
                         : Slot{0ull, INT_MAX, 0.0f, 0.0f, 0.0f, {0}};
        }
        unsigned long long wb = c.bits;
        int wi = c.idx;
        warp_argmax(wb, wi);
        warp_bcast_winner(c.bits == wb && c.idx == wi, c.x, c.y, c.z);
        if (wb == 0ull) {                                  // every dist is 0: s never changes again
            if (rank == 0)
                for (int r = k + 1 + t; r < m; r += T) o[r] = s;
            break;
        }
        s = wi;
        cx = c.x; cy = c.y; cz = c.z;
    }
    if (C > 1) {                                           // no CTA leaves while another may still read its slots
        cluster_sync_shared();
    }
}

}  // namespace

// Cluster size: the fewest CTAs whose slices hold N points, then doubled while the cloud still gives each CTA at least
// 1024 points, the batch still fits the SMs once, and the cluster stays portable (<= 8).  ModelNet-shaped clouds
// (N = 1024) run one CTA per cloud.
static int fps_cluster_size(int B, int N)
{
    int C = 1;
    while ((long long)C * kMaxPointsPerCta < N) C *= 2;
    const long long sms = ri_num_sms();
    while (2 * C <= kMaxClusterPortable && N / (2 * C) >= 1024 && (long long)B * 2 * C <= sms) C *= 2;
    return C;
}

extern "C" int ri_furthest_point_sample_f32(const float* xyz, const int* lengths, int B, int N, int m, int* idx,
                                            void* stream)
{
    if (B < 0 || N < 0 || m < 1 || (B > 0 && (xyz == nullptr || idx == nullptr))) return RI_ERR_BAD_ARG;
    if (N > RI_FPS_MAX_POINTS) return RI_ERR_UNSUPPORTED;
    if (B == 0) return RI_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (N == 0) {                                          // every cloud is empty
        cudaError_t e = cudaMemsetAsync(idx, 0xff, (size_t)B * m * sizeof(int), st);
        return e == cudaSuccess ? RI_OK : (int)e;
    }
    const int C = fps_cluster_size(B, N);
    if ((long long)B * C > INT_MAX) return RI_ERR_UNSUPPORTED;
    const int per_cta = (N + C - 1) / C;
    int T = ((per_cta + kPPT - 1) / kPPT + 31) / 32 * 32;
    if (T > kMaxThreads) T = kMaxThreads;
    const size_t smem = (size_t)3 * kPPT * T * sizeof(float);

    RI_KERNEL_SETUP(fps_kernel, true, -1);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(B * C));
    cfg.blockDim = dim3((unsigned)T);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (C > kMaxClusterPortable) {
        cudaError_t e = cudaFuncSetAttribute(fps_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (e != cudaSuccess) return (int)e;
        int clusters = 0;
        e = cudaOccupancyMaxActiveClusters(&clusters, fps_kernel, &cfg);
        if (e != cudaSuccess || clusters < 1) {
            cudaGetLastError();
            return RI_ERR_UNSUPPORTED;                     // no 16-CTA cluster of this size fits the device
        }
    }
    cudaError_t e = cudaLaunchKernelEx(&cfg, fps_kernel, xyz, lengths, N, m, C, idx);
    if (e != cudaSuccess) return (int)e;
    RI_LAUNCH_CHECK();
    return RI_OK;
}
