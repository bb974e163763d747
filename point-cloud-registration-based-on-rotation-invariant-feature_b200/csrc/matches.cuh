// matches.cuh — how the pose solvers read the mutual matches, shared by csrc/pose.cu (RANSAC, Kabsch), csrc/fgr.cu (FGR) and
// csrc/teaser.cu (TEASER++):
// the splitmix64 finaliser their samplers hash with, the gather of a pair's matched coordinates, the clamped match count,
// the fp64 edge length and the inlier test, so that every mode reads the same matches and its inlier count means the same thing.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace {

__device__ __forceinline__ uint64_t mix64(uint64_t x)          // splitmix64 finaliser
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

struct Rt { float r[9]; float t[3]; };

// the matched coordinates of pair p, read through the match lists: a(m) = src[idx1[m]], b(m) = tgt[idx2[m]]
struct PairMatches {
    const float* S; const float* Tg; const int* i1; const int* i2; int n1, n2;
    __device__ __forceinline__ PairMatches(const float* src, const float* tgt, const int* idx1, const int* idx2, int p,
                                           int n1_, int n2_, int ld)
        : S(src + (size_t)p * n1_ * 3), Tg(tgt + (size_t)p * n2_ * 3), i1(idx1 + (size_t)p * ld), i2(idx2 + (size_t)p * ld),
          n1(n1_), n2(n2_) {}
    __device__ __forceinline__ void load(int m, float3& a, float3& b) const
    {
        int i = i1[m], j = i2[m];
        i = i < 0 ? 0 : (i >= n1 ? n1 - 1 : i);
        j = j < 0 ? 0 : (j >= n2 ? n2 - 1 : j);
        a = make_float3(S[3 * i], S[3 * i + 1], S[3 * i + 2]);
        b = make_float3(Tg[3 * j], Tg[3 * j + 1], Tg[3 * j + 2]);
    }
};

// number of matches of pair p: count[p] clamped to [0, ld].  Every match is used.
__device__ __forceinline__ int match_count(const int* __restrict__ count, int p, int ld)
{
    const int M = count[p];
    return M < 0 ? 0 : (M > ld ? ld : M);
}

// |u - v| in fp64 from fp32 coordinates, in the fixed order sqrt((dx*dx + dy*dy) + dz*dz), without contraction
__device__ __forceinline__ double edge_len(float3 u, float3 v)
{
    const double dx = __dsub_rn((double)u.x, (double)v.x);
    const double dy = __dsub_rn((double)u.y, (double)v.y);
    const double dz = __dsub_rn((double)u.z, (double)v.z);
    return __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
}

__device__ __forceinline__ bool inlier(const Rt& T, float3 a, float3 b, float t2h)
{
    const float dx = T.r[0] * a.x + T.r[1] * a.y + T.r[2] * a.z + T.t[0] - b.x;
    const float dy = T.r[3] * a.x + T.r[4] * a.y + T.r[5] * a.z + T.t[1] - b.y;
    const float dz = T.r[6] * a.x + T.r[7] * a.y + T.r[8] * a.z + T.t[2] - b.z;
    return dx * dx + dy * dy + dz * dz < t2h;
}

}  // namespace
