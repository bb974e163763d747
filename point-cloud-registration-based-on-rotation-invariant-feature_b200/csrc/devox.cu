// devox.cu — cube and spherical trilinear devoxelization + the DGCNN voxel-neighbour edge gather, sm_100a.
//
// Replaces  trilinear_devoxelize_kernel            (/root/reference/PVCNN/modules/functional/src/interpolate/
//                                                   trilinear_devox.cu:22-106, host trilinear_devox.cpp:18-55)
//           spherical_trilinear_devoxelize_kernel  (.../interpolate/spherical_trilinear_devox.cu:23-136,
//                                                   host spherical_trilinear_devox.cpp:19-56)
//           the torch gather/sub/mask/cat block of PVConv.forward (/root/reference/PVCNN/modules/pvconv.py:68-90).
//
// The spherical variant keeps the reference's index quirks on purpose (integer `grid_gama / r` == 0, radian
// values truncated to ints and used as grid rows/columns, residuals not normalised by the cell size): they are
// what the shipped weights were trained against.
//
// Launch shape: grid = (point tiles, channel groups, clouds) — a 1024-point, 64-channel cloud becomes 64 CTAs
// instead of the reference's single 512-thread CTA, and each thread keeps 8 channels x 8 corners = 64 independent
// gathers in flight.  Lanes of a warp are consecutive points, so outs/inds/wgts stores are fully coalesced.
// The 8-term sum uses the reference's contraction order (001 mul, then fma 000,010,011,100,101,110,111), so outs
// is bit-identical given identical inputs.
#include "ri_common.cuh"

namespace {

constexpr int kDevoxThreads = 128;
constexpr int kDevoxChans = 8;

__device__ __forceinline__ float devox_sum(const float* __restrict__ f, const int (&id)[8], const float (&w)[8])
{
    float acc = __fmul_rn(w[1], __ldg(f + id[1]));
    acc = __fmaf_rn(w[0], __ldg(f + id[0]), acc);
    acc = __fmaf_rn(w[2], __ldg(f + id[2]), acc);
    acc = __fmaf_rn(w[3], __ldg(f + id[3]), acc);
    acc = __fmaf_rn(w[4], __ldg(f + id[4]), acc);
    acc = __fmaf_rn(w[5], __ldg(f + id[5]), acc);
    acc = __fmaf_rn(w[6], __ldg(f + id[6]), acc);
    acc = __fmaf_rn(w[7], __ldg(f + id[7]), acc);
    return acc;
}

// SPH == false: coords are grid-unit coordinates in [0, r-1] (Voxelization.forward's norm_coords).
// SPH == true : coords are the normalised Cartesian coords, g_inds the spherical cell of each point.
template <bool SPH, int CH>
__global__ void __launch_bounds__(kDevoxThreads)
devox_kernel(const float* __restrict__ coords, const float* __restrict__ feat, const int* __restrict__ g_inds,
             int C, int N, int r, float* __restrict__ outs, int* __restrict__ inds, float* __restrict__ wgts)
{
    // Clouds are walked in DESCENDING order: when the grid was produced just before by a kernel that wrote clouds
    // in ascending order (the voxelizer, a Conv3d), the highest-numbered clouds are the ones still resident in L2.
    const int b = (int)gridDim.z - 1 - (int)blockIdx.z;
    const int i = blockIdx.x * kDevoxThreads + threadIdx.x;
    if (i >= N) return;
    const int r2 = r * r;
    const size_t s = (size_t)r2 * r;
    const float* X = coords + (size_t)b * 3 * N;
    const bool writer = blockIdx.y == 0;         // channel group 0 also emits inds / wgts
    int id[8]; float w[8];
    bool defined = true;
    int first_ind = 0;                           // what inds[0,i] holds for an undefined point

    if (SPH) {
        const int pos = g_inds[(size_t)b * N + i];
        float g = 0.f, a = 0.f, be = 0.f;
        if (pos == -1) { defined = false; first_ind = -1; }                         // :42-47
        else if (!ri_sph_coords(X[i], X[i + N], X[i + 2 * (size_t)N], r, g, a, be)) defined = false;   // :54,:59
        if (defined) {
            const int gg = pos / r2;
            const int ga = (pos - gg * r2) / r;
            const int gb = pos - gg * r2 - ga * r;
            const float g_lo = (float)(gg / r);                                                         // :71
            const float a_lo = __double2float_rn(__ddiv_rn(__dmul_rn(__dmul_rn(RI_PI, 2.0), (double)ga), (double)r));  // :72
            const float b_lo = __double2float_rn(__ddiv_rn(__dmul_rn(RI_PI, (double)gb), (double)r));   // :73
            ri_corners(__fsub_rn(g, g_lo), __fsub_rn(a, a_lo), __fsub_rn(be, b_lo),
                       (int)g_lo, (int)a_lo, (int)b_lo, r, r2, id, w);
        }
    } else {
        const float x = X[i], y = X[i + N], z = X[i + 2 * (size_t)N];
        const float xl = floorf(x), yl = floorf(y), zl = floorf(z);
        ri_corners(__fsub_rn(x, xl), __fsub_rn(y, yl), __fsub_rn(z, zl), (int)xl, (int)yl, (int)zl, r, r2, id, w);
    }

    if (writer) {
        int* I = inds + (size_t)b * 8 * N + i;
        float* Wt = wgts + (size_t)b * 8 * N + i;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            I[(size_t)q * N] = defined ? id[q] : (q == 0 ? first_ind : 0);
            Wt[(size_t)q * N] = defined ? w[q] : 0.f;
        }
    }
    const int c0 = blockIdx.y * CH;
    const int c1 = min(C, c0 + CH);
    float* O = outs + (size_t)b * C * N + i;
    if (!defined) {
        for (int c = c0; c < c1; ++c) O[(size_t)c * N] = 0.f;       // the reference leaves its zero-fill
        return;
    }
    const float* F = feat + (size_t)b * C * s;
    float v[CH];                                  // CH channels x 8 corners of independent gathers in flight
    if (c1 - c0 == CH) {
#pragma unroll
        for (int u = 0; u < CH; ++u) v[u] = devox_sum(F + (size_t)(c0 + u) * s, id, w);
#pragma unroll
        for (int u = 0; u < CH; ++u) O[(size_t)(c0 + u) * N] = v[u];
    } else {                                      // last group of the cloud: clamp the plane, store what exists
#pragma unroll
        for (int u = 0; u < CH; ++u) v[u] = devox_sum(F + (size_t)min(c0 + u, c1 - 1) * s, id, w);
#pragma unroll
        for (int u = 0; u < CH; ++u)
            if (c0 + u < c1) O[(size_t)(c0 + u) * N] = v[u];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Streaming cube devoxelizer.  At r = 32, N = 1024 the 8 corners of a cloud's points touch about every 32-byte sector
// of a 128 KB channel plane, so the gather form above effectively reads the whole grid through L1 as a miss buffer —
// its speed follows the L1 size, which forces it into a different L1/shared-memory split from the rest of the step
// (ri_common.cuh, carveout note).  This form reads the grid the way the grid writer writes it: a persistent CTA per
// SM streams x-slab ranges of its planes into a shared-memory ring with cp.async.bulk (TMA engine, mbarrier
// complete_tx) and the points gather their corners from shared memory.  No L1 dependence, one carveout family for
// the whole step, reads are sequential 64 KB bursts, every grid byte is read exactly once.
//
//   work unit  plane (cloud b, channel c); every CTA owns a contiguous range of planes, so it meets at most a few
//              clouds and computes a cloud's corner data (base corner, 3 high-offset bits, 8 weights per point, in
//              registers) once per cloud;
//   tile       TS consecutive x-slabs of a plane, NO halo: the reference's 8-term chain visits the four low-x corners
//              first (001 mul, fma 000, 010, 011) and the four high-x corners after (100, 101, 110, 111), so a point adds
//              its low half when the tile holding slab floor(x) passes and continues the same chain with its high half
//              when the tile holding slab floor(x)+1 passes (the same tile or the next one) — the accumulator lives
//              in a register across tiles, the order of operations is untouched: bit-identical to devox_kernel;
//   warps      8 consumer warps (P = ceil(N/256) points per thread) + 1 producer warp; full[] barriers carry the TMA
//              byte counts, empty[] barriers get one arrival per consumer warp, so warps drift freely and the
//              producer refills a slot as soon as the last warp has left it.
constexpr int kSdThreads = 256;                     // consumer threads
constexpr int kSdWarps = kSdThreads / 32;
constexpr int kSdMaxRing = 8;
// registers: min-CTAs 2 caps the kernel at 112 registers per thread (288 threads: 32 K of the SM's 64 K), so that a CTA of
// the voxel branch's prefix kernel (512 threads x 64 registers) of ANOTHER batch in flight fits on the SM next to it
constexpr int kSdMinCtas = 2;
constexpr uint32_t kSdTileBytesDefault = 64u << 10;   // measured: 8 / 16 / 32 / 64 KB tiles -> 154 / 91 / 58 / 56 us (B200, 32 x 71 planes)
constexpr uint32_t kSdRingBytesDefault = 128u << 10;   // leaves room for k-NN CTAs on the same SM

__device__ __forceinline__ void sd_mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void sd_mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void sd_mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void sd_mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" :: "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void sd_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

template <int P>
__global__ void __launch_bounds__(kSdThreads + 32, kSdMinCtas)
devox_stream_kernel(const float* __restrict__ coords, const float* __restrict__ feat, int B, int C, int N, int r,
                    int TS, int nt, uint32_t slot_bytes, int R,
                    float* __restrict__ outs, int* __restrict__ inds, float* __restrict__ wgts, int dbg_skip)
{
    extern __shared__ __align__(128) unsigned char sd_smem[];
    __shared__ __align__(8) uint64_t full[kSdMaxRing];
    __shared__ __align__(8) uint64_t empty[kSdMaxRing];
    const int tid = threadIdx.x;
    const int r2 = r * r;
    const size_t s = (size_t)r2 * r;
    const long long planes = (long long)B * C;
    // contiguous, balanced plane range of this CTA
    const int p0 = (int)(planes * blockIdx.x / gridDim.x), p1 = (int)(planes * (blockIdx.x + 1) / gridDim.x);
    const int my_tiles = (p1 - p0) * nt;

    if (tid == 0) {
        for (int i = 0; i < R; ++i) { sd_mbar_init(ri_smem_u32(&full[i]), 1); sd_mbar_init(ri_smem_u32(&empty[i]), kSdWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (tid >= kSdThreads) {
        // ---------------------------------------------------------------- producer warp (one lane issues)
        if (tid == kSdThreads) {
            int slot = 0; uint32_t round = 0;
            for (int n = 0; n < my_tiles; ++n) {
                const int pl = p0 + n / nt, t = n - (n / nt) * nt;
                const int x0 = t * TS;
                const int nsl = min(r, x0 + TS) - x0;
                const uint32_t bytes = (uint32_t)nsl * (uint32_t)r2 * 4u;
                const float* src = feat + (size_t)pl * s + (size_t)x0 * r2;
                if (round > 0) sd_mbar_wait(ri_smem_u32(&empty[slot]), (round - 1) & 1);
                const uint32_t bar = ri_smem_u32(&full[slot]);
                sd_mbar_expect_tx(bar, bytes);
                sd_bulk_g2s(ri_smem_u32(sd_smem + (size_t)slot * slot_bytes), src, bytes, bar);
                if (++slot == R) { slot = 0; ++round; }
            }
        }
        return;
    }

    // -------------------------------------------------------------------- consumers
    const int lane = tid & 31;
    int id0[P], tl[P];          // id0: base corner | high-offset bits << 28;  tl: tile of the low half | tile of the high half << 8
    float w[P][8];
    int cur_b = -1;
    int slot = 0; uint32_t round = 0;
    for (int pl = p0; pl < p1; ++pl) {
        const int b = pl / C, c = pl - b * C;
        if (b != cur_b) {
            cur_b = b;
            const float* X = coords + (size_t)b * 3 * N;
#pragma unroll
            for (int p = 0; p < P; ++p) {
                const int i = tid + p * kSdThreads;
                tl[p] = 0xffff;                    // no point: matches no tile
                id0[p] = 0;
                if (i < N) {
                    const float x = X[i], y = X[i + N], z = X[i + 2 * (size_t)N];
                    const float xl = floorf(x), yl = floorf(y), zl = floorf(z);
                    int id[8];
                    ri_corners(__fsub_rn(x, xl), __fsub_rn(y, yl), __fsub_rn(z, zl), (int)xl, (int)yl, (int)zl, r, r2, id, w[p]);
                    const int hbits = (id[1] != id[0] ? 1 : 0) | (id[2] != id[0] ? 2 : 0) | (id[4] != id[0] ? 4 : 0);
                    const int xi = (int)xl, yi = (int)yl, zi = (int)zl;
                    const int xh = xi + ((hbits >> 2) & 1);
                    const bool inside = xi >= 0 && yi >= 0 && zi >= 0 && xh < r &&
                                        yi + ((hbits >> 1) & 1) < r && zi + (hbits & 1) < r;
                    tl[p] = inside ? ((xi / TS) | ((xh / TS) << 8)) : 0xfefe;   // 0xfefe: outside the grid, global path
                    id0[p] = id[0] | (hbits << 28);
                }
            }
        }
        if (c == 0) {
            // the CTA that owns a cloud's first plane also emits inds / wgts
#pragma unroll
            for (int p = 0; p < P; ++p) {
                const int i = tid + p * kSdThreads;
                if (i < N) {
                    const int base = id0[p] & 0x0fffffff;
                    const int hc = (id0[p] >> 28) & 1, hb = ((id0[p] >> 29) & 1) * r, ha = ((id0[p] >> 30) & 1) * r2;
                    int* I = inds + (size_t)b * 8 * N + i;
                    float* Wt = wgts + (size_t)b * 8 * N + i;
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        I[(size_t)u * N] = base + ((u & 1) ? hc : 0) + ((u & 2) ? hb : 0) + ((u & 4) ? ha : 0);
                        Wt[(size_t)u * N] = w[p][u];
                    }
                }
            }
        }
        float acc[P];
#pragma unroll
        for (int p = 0; p < P; ++p) acc[p] = 0.f;
        for (int t = 0; t < nt; ++t) {
            sd_mbar_wait(ri_smem_u32(&full[slot]), round & 1);
            const float* tile = reinterpret_cast<const float*>(sd_smem + (size_t)slot * slot_bytes);
            const int tile_base = t * TS * r2;
#pragma unroll
            for (int p = 0; p < P; ++p) {
                if (dbg_skip) break;
                const int base = (id0[p] & 0x0fffffff) - tile_base;
                const int hc = (id0[p] >> 28) & 1, hb = ((id0[p] >> 29) & 1) * r, ha = ((id0[p] >> 30) & 1) * r2;
                if ((tl[p] & 0xff) == t) {
                    const float* f = tile + base;
                    float a = __fmul_rn(w[p][1], f[hc]);
                    a = __fmaf_rn(w[p][0], f[0], a);
                    a = __fmaf_rn(w[p][2], f[hb], a);
                    acc[p] = __fmaf_rn(w[p][3], f[hb + hc], a);
                }
                if ((tl[p] >> 8) == t) {
                    const float* f = tile + base + ha;
                    float a = __fmaf_rn(w[p][4], f[0], acc[p]);
                    a = __fmaf_rn(w[p][5], f[hc], a);
                    a = __fmaf_rn(w[p][6], f[hb], a);
                    acc[p] = __fmaf_rn(w[p][7], f[hb + hc], a);
                }
            }
            __syncwarp();
            if (lane == 0) sd_mbar_arrive(ri_smem_u32(&empty[slot]));
            if (++slot == R) { slot = 0; ++round; }
        }
        const float* F = feat + (size_t)pl * s;
        float* O = outs + (size_t)pl * N;
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const int i = tid + p * kSdThreads;
            if (tl[p] == 0xfefe) {                             // outside the grid: what the gather form would read
                const int base = id0[p] & 0x0fffffff;
                int id[8]; float ww[8];
                const int hc = (id0[p] >> 28) & 1, hb = ((id0[p] >> 29) & 1) * r, ha = ((id0[p] >> 30) & 1) * r2;
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    long long v = (long long)base + ((u & 1) ? hc : 0) + ((u & 2) ? hb : 0) + ((u & 4) ? ha : 0);
                    v = v < 0 ? 0 : (v >= (long long)s ? (long long)s - 1 : v);
                    id[u] = (int)v; ww[u] = w[p][u];
                }
                acc[p] = devox_sum(F, id, ww);
            }
            if (i < N) O[i] = acc[p];
        }
    }
}

// host-side geometry of the streaming form; returns false when it does not apply
struct SdPlan { int TS, nt, R; uint32_t slot_bytes; };
static bool sd_plan(const float* feat, int C, int N, int r, SdPlan& pl)
{
    // RI_DEVOX_STREAM=0 forces the gather form, =1 takes the streaming form wherever it is able to run (tests compare
    // the two); unset: streaming where a whole plane is not much more than what the gathers would move
    const RiEnv& env = ri_env();
    const int mode = env.devox_stream >= 0 ? env.devox_stream + 1 : 0;
    if (mode == 1) return false;
    if (C < 1 || N < 1 || N > kSdThreads * 8 || (r & 1) || r < 2) return false;
    if (((uintptr_t)feat & 15) != 0) return false;
    const size_t slab = (size_t)r * r * 4, plane = slab * r;
    uint32_t tile_bytes = kSdTileBytesDefault, ring_bytes = kSdRingBytesDefault;
    if (env.devox_tile_kb >= 1 && env.devox_tile_kb <= 96) tile_bytes = (uint32_t)env.devox_tile_kb << 10;
    if (env.devox_ring_kb >= 2 && env.devox_ring_kb <= 208) ring_bytes = (uint32_t)env.devox_ring_kb << 10;
    if (slab > tile_bytes) return false;
    if (plane / 4 >= (1u << 28)) return false;      // base index is packed into 28 bits
    // the gather form moves ~128 B per point and plane; stream only where a whole plane is not much more than that
    if (mode != 2 && plane > (size_t)256 * N) return false;
    int TS = (int)(tile_bytes / slab);
    if (TS > r) TS = r;
    pl.TS = TS;
    pl.nt = (r + TS - 1) / TS;
    if (pl.nt > 250) return false;                  // tile numbers are packed into 8 bits
    pl.slot_bytes = (uint32_t)((TS * slab + 127) & ~(size_t)127);
    int R = (int)(ring_bytes / pl.slot_bytes);
    pl.R = R > kSdMaxRing ? kSdMaxRing : R;
    return pl.R >= 2;
}

template <int P>
static int sd_launch(const SdPlan& pl, const float* coords, const float* feat, int B, int C, int N, int r,
                     float* outs, int* inds, float* wgts, cudaStream_t st)
{
    auto kern = devox_stream_kernel<P>;
    size_t smem = (size_t)pl.R * pl.slot_bytes;
    const RiEnv& env = ri_env();
    if (env.devox_pad_kb >= 0 && env.devox_pad_kb <= 64) smem += (size_t)env.devox_pad_kb << 10;
    RI_KERNEL_SETUP(kern, true, ri_step_carveout_percent());
    const long long planes = (long long)B * C;
    const int grid = planes < ri_num_sms() ? (int)planes : ri_num_sms();
    kern<<<grid, kSdThreads + 32, smem, st>>>(coords, feat, B, C, N, r, pl.TS, pl.nt, pl.slot_bytes, pl.R, outs, inds, wgts,
                                              env.devox_dbg_skip);
    RI_LAUNCH_CHECK();
    return RI_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Sector-compacting devoxelizer (both grids; N <= 1024 points per cloud).  What the 8 corners of a cloud's points touch
// is a SMALL part of a channel plane and it is the same part in every plane: measured on the bench clouds
// (tools/exp_devox_sectors.py) 26.5 % of the 32-byte sectors of a plane on the cube grid at r = 32 (8 % at r = 64), 0.4 % on
// the spherical grid.  Streaming whole planes (devox_stream_kernel) reads 3.8x what is needed; gathering per point
// (devox_kernel) asks L2 for every sector ~4 times (as many points share it) through uncoalesced 4-byte loads.  Here a CTA
// = (cloud, group of planes):
//   once   corner cells + weights of its points (registers); a bit per touched sector in a shared-memory bitmap, ranked by a
//          prefix sum over the words -> the sorted list of the cloud's U distinct sectors and, per corner, its slot in it;
//   per plane  the U sectors are copied global -> shared memory, 32 bytes each, by cp.async (every needed DRAM sector is
//          read exactly once, as a whole, and nothing else is), double-buffered against the previous plane's arithmetic;
//          the points then take their 8 corners from the compact buffer and run the reference's 8-term chain.
// Same corner indices, weights and sums as devox_kernel, bit for bit.  A cloud with more distinct sectors than the buffer
// holds (kDsCap) runs the chain on global loads instead.
constexpr int kDsThreads = 256;
constexpr int kDsPts = 4;                            // points per thread: N <= 1024
constexpr int kDsCap = 3072;                         // sectors the plane buffer holds (96 KB): two planes of <= 1536, or one
constexpr int kDsMaxWords = 2048;                    // bitmap words: r^3 / 8 sectors <= 65536

template <bool SPH>
__global__ void __launch_bounds__(kDsThreads, 2)
devox_sectors_kernel(const float* __restrict__ coords, const float* __restrict__ feat, const int* __restrict__ g_inds,
                     int C, int N, int r, int group, int nwords,
                     float* __restrict__ outs, int* __restrict__ inds, float* __restrict__ wgts)
{
    extern __shared__ __align__(128) unsigned char ds_smem[];
    float* buf = reinterpret_cast<float*>(ds_smem);                          // [kDsCap * 8] floats: one plane, or two halves
    unsigned short* slist = reinterpret_cast<unsigned short*>(buf + kDsCap * 8);   // [kDsCap] sector ids, ascending
    unsigned* bitmap = reinterpret_cast<unsigned*>(slist + kDsCap);          // [nwords]
    int* prefix = reinterpret_cast<int*>(bitmap + nwords);                   // [nwords] sectors before this word
    __shared__ int swarp[kDsThreads / 32];
    __shared__ int s_total;

    const int b = (int)gridDim.y - 1 - (int)blockIdx.y;                      // last-written clouds first (still in L2)
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int r2 = r * r;
    const size_t s = (size_t)r2 * r;
    const float* X = coords + (size_t)b * 3 * N;
    const bool writer = blockIdx.x == 0;                                     // plane group 0 also emits inds / wgts

    for (int w = tid; w < nwords; w += kDsThreads) bitmap[w] = 0u;
    __syncthreads();

    int id[kDsPts][8];
    float wt[kDsPts][8];
    bool defined[kDsPts];
#pragma unroll
    for (int q = 0; q < kDsPts; ++q) {
        const int i = tid + q * kDsThreads;
        defined[q] = false;
        if (i >= N) continue;
        defined[q] = true;
        int first_ind = 0;
        if (SPH) {
            const int pos = g_inds[(size_t)b * N + i];
            float g = 0.f, a = 0.f, be = 0.f;
            if (pos == -1) { defined[q] = false; first_ind = -1; }
            else if (!ri_sph_coords(X[i], X[i + N], X[i + 2 * (size_t)N], r, g, a, be)) defined[q] = false;
            if (defined[q]) {
                const int gg = pos / r2;
                const int ga = (pos - gg * r2) / r;
                const int gb = pos - gg * r2 - ga * r;
                const float g_lo = (float)(gg / r);
                const float a_lo = __double2float_rn(__ddiv_rn(__dmul_rn(__dmul_rn(RI_PI, 2.0), (double)ga), (double)r));
                const float b_lo = __double2float_rn(__ddiv_rn(__dmul_rn(RI_PI, (double)gb), (double)r));
                ri_corners(__fsub_rn(g, g_lo), __fsub_rn(a, a_lo), __fsub_rn(be, b_lo),
                           (int)g_lo, (int)a_lo, (int)b_lo, r, r2, id[q], wt[q]);
            }
        } else {
            const float x = X[i], y = X[i + N], z = X[i + 2 * (size_t)N];
            const float xl = floorf(x), yl = floorf(y), zl = floorf(z);
            ri_corners(__fsub_rn(x, xl), __fsub_rn(y, yl), __fsub_rn(z, zl), (int)xl, (int)yl, (int)zl, r, r2, id[q], wt[q]);
        }
        if (writer) {
            int* I = inds + (size_t)b * 8 * N + i;
            float* Wt = wgts + (size_t)b * 8 * N + i;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                I[(size_t)c * N] = defined[q] ? id[q][c] : (c == 0 ? first_ind : 0);
                Wt[(size_t)c * N] = defined[q] ? wt[q][c] : 0.f;
            }
        }
        if (defined[q]) {
#pragma unroll
            for (int c = 0; c < 8; ++c) atomicOr(&bitmap[id[q][c] >> 8], 1u << ((id[q][c] >> 3) & 31));
        }
    }
    __syncthreads();
    // ---- rank the touched sectors: exclusive prefix sum of the words' popcounts
    {
        const int per = (nwords + kDsThreads - 1) / kDsThreads;              // consecutive words per thread
        const int w0 = tid * per, w1 = min(nwords, w0 + per);
        int sum = 0;
        for (int w = w0; w < w1; ++w) sum += __popc(bitmap[w]);
        int inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) swarp[wid] = inc;
        __syncthreads();
        if (wid == 0) {
            const int v = lane < kDsThreads / 32 ? swarp[lane] : 0;
            int wi = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += t;
            }
            if (lane < kDsThreads / 32) swarp[lane] = wi - v;
            if (lane == kDsThreads / 32 - 1) s_total = wi;
        }
        __syncthreads();
        int run = swarp[wid] + inc - sum;
        for (int w = w0; w < w1; ++w) { prefix[w] = run; run += __popc(bitmap[w]); }
    }
    __syncthreads();
    const int U = s_total;
    const bool compact = U <= kDsCap;
    // ---- the sorted sector list, and every corner's float offset in a plane buffer
    unsigned short off[kDsPts][8];
    if (compact) {
        for (int w = tid; w < nwords; w += kDsThreads) {
            unsigned m = bitmap[w];
            int k2 = prefix[w];
            while (m) { const int bit = __ffs(m) - 1; m &= m - 1; slist[k2++] = (unsigned short)(w * 32 + bit); }
        }
#pragma unroll
        for (int q = 0; q < kDsPts; ++q) {
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                off[q][c] = 0;
                if (defined[q]) {
                    const int sec = id[q][c] >> 3, w = sec >> 5;
                    const int slot = prefix[w] + __popc(bitmap[w] & ((1u << (sec & 31)) - 1u));
                    off[q][c] = (unsigned short)(slot * 8 + (id[q][c] & 7));
                }
            }
        }
    }
    __syncthreads();

    const int c0 = blockIdx.x * group, c1 = min(C, c0 + group);
    const float* F = feat + (size_t)b * C * s;
    float* O = outs + (size_t)b * C * N;
    auto fetch = [&](int c, float* dst) {                                    // the cloud's sectors of plane c -> dst
        const float* src = F + (size_t)c * s;
        for (int j = tid; j < 2 * U; j += kDsThreads) {                      // two 16-byte halves per sector
            const int sec = slist[j >> 1], h = j & 1;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                         :: "r"(ri_smem_u32(dst + (j >> 1) * 8 + h * 4)), "l"(src + (size_t)sec * 8 + h * 4) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (compact) {
        // a cloud whose sectors fill at most half of the buffer runs two planes deep (the next plane's copies fly under this
        // plane's arithmetic); a larger one plane at a time (the other CTA of the SM fills the gaps)
        const int nbuf = U <= kDsCap / 2 ? 2 : 1;
        const int half = kDsCap / 2 * 8;
        if (nbuf == 2 && c0 < c1) fetch(c0, buf);
        for (int c = c0; c < c1; ++c) {
            float* cur = buf + (nbuf == 2 ? ((c - c0) & 1) * half : 0);
            if (nbuf == 2) {
                if (c + 1 < c1) { fetch(c + 1, buf + ((c + 1 - c0) & 1) * half); asm volatile("cp.async.wait_group 1;" ::: "memory"); }
                else asm volatile("cp.async.wait_group 0;" ::: "memory");
            } else {
                fetch(c, cur);
                asm volatile("cp.async.wait_group 0;" ::: "memory");
            }
            __syncthreads();
#pragma unroll
            for (int q = 0; q < kDsPts; ++q) {
                const int i = tid + q * kDsThreads;
                if (i >= N) continue;
                float acc = 0.f;                                             // the reference leaves its zero-fill for undefined points
                if (defined[q]) {
                    acc = __fmul_rn(wt[q][1], cur[off[q][1]]);
                    acc = __fmaf_rn(wt[q][0], cur[off[q][0]], acc);
                    acc = __fmaf_rn(wt[q][2], cur[off[q][2]], acc);
                    acc = __fmaf_rn(wt[q][3], cur[off[q][3]], acc);
                    acc = __fmaf_rn(wt[q][4], cur[off[q][4]], acc);
                    acc = __fmaf_rn(wt[q][5], cur[off[q][5]], acc);
                    acc = __fmaf_rn(wt[q][6], cur[off[q][6]], acc);
                    acc = __fmaf_rn(wt[q][7], cur[off[q][7]], acc);
                }
                O[(size_t)c * N + i] = acc;
            }
            __syncthreads();                                                 // `cur` is refilled next
        }
    } else {
        for (int c = c0; c < c1; ++c) {
#pragma unroll
            for (int q = 0; q < kDsPts; ++q) {
                const int i = tid + q * kDsThreads;
                if (i >= N) continue;
                O[(size_t)c * N + i] = defined[q] ? devox_sum(F + (size_t)c * s, id[q], wt[q]) : 0.f;
            }
        }
    }
}

template <bool SPH>
static int ds_launch(const float* coords, const float* feat, const int* g_inds, int B, int C, int N, int r,
                     float* outs, int* inds, float* wgts, cudaStream_t st)
{
    const long long s = (long long)r * r * r;
    const int nwords = (int)((s / 8 + 31) / 32);
    // planes per CTA: enough CTAs for two per SM, at least 4 planes each so the per-cloud setup is amortised
    int group = (int)(((long long)B * C + 2LL * ri_num_sms() - 1) / (2LL * ri_num_sms()));
    if (group < 4) group = 4;
    if (group > C) group = C > 0 ? C : 1;
    const int groups = C > 0 ? (C + group - 1) / group : 1;
    const size_t smem = (size_t)kDsCap * 32 + (size_t)kDsCap * 2 + (size_t)nwords * 8;
    auto kern = devox_sectors_kernel<SPH>;
    RI_KERNEL_SETUP(kern, true, ri_step_carveout_percent());
    kern<<<dim3(groups, B), kDsThreads, smem, st>>>(coords, feat, g_inds, C, N, r, group, nwords, outs, inds, wgts);
    RI_LAUNCH_CHECK();
    return RI_OK;
}

// out[b, c, i]     = inds[b,i] == -1 ? 0 : feat[b,c,i] - avg[b,c,inds[b,i]]
// out[b, C + c, i] = feat[b,c,i]                                                    (pvconv.py:68-90)
constexpr int kEdgeThreads = 128;
constexpr int kEdgeChans = 8;
__global__ void __launch_bounds__(kEdgeThreads)
edge_gather_kernel(const float* __restrict__ avg, const float* __restrict__ feat, const int* __restrict__ inds,
                   int C, int N, int s, float* __restrict__ out)
{
    const int b = blockIdx.z;
    const int i = blockIdx.x * kEdgeThreads + threadIdx.x;
    if (i >= N) return;
    const int id = inds[(size_t)b * N + i];
    const bool undef = id == -1;
    const int idc = undef ? 0 : id;
    const int c0 = blockIdx.y * kEdgeChans, c1 = min(C, c0 + kEdgeChans);
    const float* A = avg + (size_t)b * C * s + idc;
    const float* F = feat + (size_t)b * C * N + i;
    float* O = out + (size_t)b * 2 * C * N + i;
    float f[kEdgeChans], a[kEdgeChans];
#pragma unroll
    for (int u = 0; u < kEdgeChans; ++u) {
        const int c = c0 + u;
        if (c < c1) { f[u] = F[(size_t)c * N]; a[u] = __ldg(A + (size_t)c * s); }
    }
#pragma unroll
    for (int u = 0; u < kEdgeChans; ++u) {
        const int c = c0 + u;
        if (c < c1) {
            O[(size_t)c * N] = undef ? 0.f : __fsub_rn(f[u], a[u]);
            O[(size_t)(C + c) * N] = f[u];
        }
    }
}

template <bool SPH>
int devox_impl(const float* coords, const float* feat, const int* g_inds, int B, int C, int N, int r,
               float* outs, int* inds, float* wgts, cudaStream_t st)
{
    if (B < 0 || C < 0 || N < 0 || r <= 0 || r > 1024) return RI_ERR_BAD_ARG;
    if ((long long)r * r * r > 0x7fffffffLL || B > 65535) return RI_ERR_UNSUPPORTED;
    if (B == 0 || N == 0) return RI_OK;
    {
        // sector-compacting form: N <= 1024 points, r^3 a multiple of 8 with at most 65536 sectors per plane, 32-byte
        // aligned planes.  RI_DEVOX_STREAM = 0 / 1 still forces the gather / streaming forms (tests, experiments).
        const long long s = (long long)r * r * r;
        // (the spherical grid keeps the per-point gather form: its index quirks fold a cloud's corners onto ~17 sectors of a
        // plane, there is nothing to compact — 21 us against 27)
        if (!SPH && ri_env().devox_stream < 0 && N <= kDsThreads * kDsPts && s % 8 == 0 && s / 8 <= 32LL * kDsMaxWords &&
            ((uintptr_t)feat & 31) == 0)
            return ds_launch<SPH>(coords, feat, g_inds, B, C, N, r, outs, inds, wgts, st);
    }
    if (!SPH) {
        SdPlan pl;
        if ((long long)B * C < 0x7fffffffLL && sd_plan(feat, C, N, r, pl)) {
            const int P = (N + kSdThreads - 1) / kSdThreads;
            if (P <= 4) return sd_launch<4>(pl, coords, feat, B, C, N, r, outs, inds, wgts, st);
            return sd_launch<8>(pl, coords, feat, B, C, N, r, outs, inds, wgts, st);
        }
    }
    // 8 channels per CTA.  Every CTA of a point tile recomputes the tile's corner cells and weights (a third of the kernel's
    // instructions on the spherical grid), but more channels per CTA measured slower: 18.5 / 22.5 / 24.6 us with 8 / 12 / 16
    // (spherical, 32 x 1024 x 67, r = 32) — the registers of the extra gathers in flight cost more occupancy than the
    // recomputation costs issue slots.
    const int groups = C > 0 ? (C + kDevoxChans - 1) / kDevoxChans : 1;   // one group still writes inds/wgts
    dim3 grid((N + kDevoxThreads - 1) / kDevoxThreads, groups, B);
    devox_kernel<SPH, kDevoxChans><<<grid, kDevoxThreads, 0, st>>>(coords, feat, g_inds, C, N, r, outs, inds, wgts);
    RI_LAUNCH_CHECK();
    return RI_OK;
}

}  // namespace

extern "C" int ri_trilinear_devox_f32(const float* coords, const float* feat, int B, int C, int N, int r,
                                      float* outs, int* inds, float* wgts, void* stream)
{
    return devox_impl<false>(coords, feat, nullptr, B, C, N, r, outs, inds, wgts, (cudaStream_t)stream);
}

extern "C" int ri_sph_trilinear_devox_f32(const float* coords, const float* feat, const int* g_inds,
                                          int B, int C, int N, int r, float* outs, int* inds, float* wgts, void* stream)
{
    // The reference's corner rows are radians truncated to ints (a_lo <= 6, b_lo <= 3) and the gamma row is always 0, so
    // the highest corner index is r^2 + 7r + 4: inside the r^3 grid only for r >= 4.  Smaller grids would read (forward)
    // and atomically add (backward) past the end of every channel plane.
    if (r > 0 && r < 4) return RI_ERR_UNSUPPORTED;
    if (g_inds == nullptr) return RI_ERR_BAD_ARG;
    return devox_impl<true>(coords, feat, g_inds, B, C, N, r, outs, inds, wgts, (cudaStream_t)stream);
}

extern "C" int ri_voxel_edge_gather_f32(const float* avg, const float* feat, const int* inds,
                                        int B, int C, int N, int s, float* out, void* stream)
{
    if (B < 0 || C < 0 || N < 0 || s <= 0) return RI_ERR_BAD_ARG;
    if (B > 65535) return RI_ERR_UNSUPPORTED;
    if (B == 0 || N == 0 || C == 0) return RI_OK;
    dim3 grid((N + kEdgeThreads - 1) / kEdgeThreads, (C + kEdgeChans - 1) / kEdgeChans, B);
    edge_gather_kernel<<<grid, kEdgeThreads, 0, (cudaStream_t)stream>>>(avg, feat, inds, C, N, s, out);
    RI_LAUNCH_CHECK();
    return RI_OK;
}
