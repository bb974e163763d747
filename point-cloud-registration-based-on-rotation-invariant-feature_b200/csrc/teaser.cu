// teaser.cu — TEASER++ (Yang, Shi, Carlone, T-RO 2020) with a known scale over the mutual matches, P pairs per call, sm_100a
// (SURVEY.md §8 row f10).
//
// The reference's registration script hands its matches to teaserpp_python (deepgmr_mn40.py:175-230).  TEASER++ is not part
// of the reference tree; what is kept is its pipeline for a known scale, restated in include/ri_b200.h (ri_teaser_f32) and
// DESIGN.md §8: the pairwise-consistency graph, a maximum clique of it, GNC-TLS rotation over the clique's chain TIMs and
// adaptive-voting translation.  The fp64 replay in tests/ (teaser_oracle) repeats every step.
//
// Kernels (in launch order)
//   teaser_graph_kernel    one warp per match i: each lane produces whole 32-bit words of row i of the graph (the fp64 edge
//                          test of matches.cuh::edge_len) and the warp's popcounts give deg(i).  Written unpermuted into
//                          the region that later holds the search stack.
//   teaser_rank_kernel     one thread per match: its rank in the order pi (deg descending, index ascending) by counting.
//   teaser_permute_kernel  one thread per word of the rank-space adjacency: bit (r, c) = graph(pi(r), pi(c)).  In rank space
//                          "the first vertex in pi order" of a set is its lowest set bit.
//   teaser_clique_kernel   one CTA per pair.  The eight warps split the 64 greedy starts of the heuristic incumbent; all
//                          threads peel; warp 0 runs the branch and bound (BBMC: greedy colouring in rank order, vertices
//                          visited in reverse colouring order) sequentially with an explicit stack of candidate bitsets in
//                          the workspace.  The colouring of a level is recomputed when the search returns to it, so the
//                          stack holds one bitset per level and no colour lists.  Every expand call costs one node; at
//                          max_clique_nodes the search stops with exact = 0.
//   teaser_solve_kernel    one CTA per pair: the chain TIMs, the GNC-TLS loop (fixed-order block_sum reductions, thread 0
//                          runs Horn's step), three adaptive-voting sweeps (every candidate evaluated with sums in index
//                          order), the inlier count.
// No float atomics (integer atomics only set bits), no host synchronisation, no allocation: a pair's result is
// bit-reproducible and does not depend on the rest of the batch.
#include "ri_common.cuh"
#include "rigid.cuh"
#include "matches.cuh"

namespace {

constexpr int kMaxLd = 1 << 15;      // ld limit: W <= 1024 words per bitset row, 128 MB of adjacency per pair at most
constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kStarts = 64;          // greedy starts of the heuristic incumbent

struct TeaserParams {
    double beta, c2, range, gnc_factor, cost_threshold;
    int max_iterations;
    long long max_nodes;
    float inlier_dist;
};

// per-pair regions of the workspace, each region [P][...] and 256-byte aligned
struct Layout {
    size_t adj, stk, deg, perm, lvl_i, lvl_v, list_v, list_c, best, cliq, tim, wt, xs, total;
    __host__ __device__ Layout(int P, int ld)
    {
        const size_t W = (size_t)(ld + 31) / 32, L = (size_t)ld, Pn = (size_t)P;
        size_t o = 0;
        auto take = [&](size_t bytes) { const size_t at = o; o += (bytes + 255) / 256 * 256; return at; };
        adj = take(Pn * L * W * 4);
        stk = take(Pn * (L + 1) * W * 4);
        deg = take(Pn * L * 4);
        perm = take(Pn * L * 4);
        lvl_i = take(Pn * (L + 1) * 4);
        lvl_v = take(Pn * (L + 1) * 4);
        list_v = take(Pn * L * 4);
        list_c = take(Pn * L * 4);
        best = take(Pn * L * 4);
        cliq = take(Pn * L * 4);
        tim = take(Pn * L * 6 * 8);
        wt = take(Pn * L * 8);
        xs = take(Pn * L * 8);
        total = o;
    }
};

template <typename T>
__device__ __forceinline__ T* region(void* ws, size_t off, int p, size_t per_pair)
{
    return reinterpret_cast<T*>(static_cast<char*>(ws) + off) + (size_t)p * per_pair;
}

// ---------------------------------------------------------------------------------------------- graph, order, relabelling
__global__ void __launch_bounds__(kThreads)
teaser_graph_kernel(const float* __restrict__ src, const float* __restrict__ tgt, const int* __restrict__ idx1,
                    const int* __restrict__ idx2, const int* __restrict__ count, int n1, int n2, int ld, double beta,
                    void* ws, Layout lay)
{
    const int p = blockIdx.y, lane = threadIdx.x & 31;
    const int i = blockIdx.x * kWarps + (threadIdx.x >> 5);
    const int M = match_count(count, p, ld);
    if (i >= M) return;
    const int W = (ld + 31) / 32;
    uint32_t* g0 = region<uint32_t>(ws, lay.stk, p, (size_t)(ld + 1) * W) + (size_t)i * W;   // unpermuted row i
    const PairMatches pm(src, tgt, idx1, idx2, p, n1, n2, ld);
    float3 ai, bi;
    pm.load(i, ai, bi);
    int deg = 0;
    for (int w = lane; w < W; w += 32) {
        uint32_t word = 0;
        const int j0 = w * 32, j1 = min(j0 + 32, M);
        for (int j = j0; j < j1; ++j) {
            if (j == i) continue;
            float3 aj, bj;
            pm.load(j, aj, bj);
            if (fabs(__dsub_rn(edge_len(ai, aj), edge_len(bi, bj))) <= beta) word |= 1u << (j - j0);
        }
        g0[w] = word;
        deg += __popc(word);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) deg += __shfl_down_sync(0xffffffffu, deg, o);
    if (lane == 0) region<int>(ws, lay.deg, p, ld)[i] = deg;
}

__global__ void __launch_bounds__(kThreads)
teaser_rank_kernel(const int* __restrict__ count, int ld, void* ws, Layout lay)
{
    __shared__ int tile[kThreads];
    const int p = blockIdx.y, v = blockIdx.x * kThreads + threadIdx.x;
    const int M = match_count(count, p, ld);
    if (blockIdx.x * kThreads >= M) return;                         // uniform over the block
    const int* deg = region<int>(ws, lay.deg, p, ld);
    const int dv = v < M ? deg[v] : 0;
    int rank = 0;
    for (int base = 0; base < M; base += kThreads) {
        __syncthreads();
        if (base + threadIdx.x < M) tile[threadIdx.x] = deg[base + threadIdx.x];
        __syncthreads();
        const int n = min(kThreads, M - base);
        for (int k = 0; k < n; ++k) {
            const int du = tile[k], u = base + k;
            rank += (du > dv || (du == dv && u < v)) ? 1 : 0;
        }
    }
    if (v < M) region<int>(ws, lay.perm, p, ld)[rank] = v;
}

__global__ void __launch_bounds__(kThreads)
teaser_permute_kernel(const int* __restrict__ count, int ld, void* ws, Layout lay)
{
    const int p = blockIdx.y, W = (ld + 31) / 32;
    const long long t = (long long)blockIdx.x * kThreads + threadIdx.x;
    const int M = match_count(count, p, ld);
    if (t >= (long long)M * W) return;
    const int r = (int)(t / W), w = (int)(t % W);
    const int* perm = region<int>(ws, lay.perm, p, ld);
    const uint32_t* g0 = region<uint32_t>(ws, lay.stk, p, (size_t)(ld + 1) * W) + (size_t)perm[r] * W;
    uint32_t word = 0;
    const int c1 = min(w * 32 + 32, M);
    for (int c = w * 32; c < c1; ++c) {
        const int u = perm[c];
        word |= ((g0[u >> 5] >> (u & 31)) & 1u) << (c & 31);
    }
    region<uint32_t>(ws, lay.adj, p, (size_t)ld * W)[(size_t)r * W + w] = word;
}

// ---------------------------------------------------------------------------------------------- maximum clique
// lowest set bit of s at word index >= from, -1 if none; the same value in every lane of the warp
__device__ __forceinline__ int first_bit(const uint32_t* s, int from, int W, int lane)
{
    for (int w0 = from; w0 < W; w0 += 32) {
        const int w = w0 + lane;
        const uint32_t x = w < W ? s[w] : 0u;
        const unsigned bal = __ballot_sync(0xffffffffu, x != 0u);
        if (bal) {
            const int l = __ffs(bal) - 1;
            const uint32_t xw = __shfl_sync(0xffffffffu, x, l);
            return (w0 + l) * 32 + __ffs(xw) - 1;
        }
    }
    return -1;
}

// greedy clique from rank s: C = {s}, cand = N(s); repeatedly add the lowest rank of cand and intersect.  Its size; with
// `out`, lane 0 writes the members in the order they are added.
__device__ int greedy_clique(const uint32_t* adj, int W, int s, uint32_t* cand, int lane, int* out)
{
    const uint32_t* rs = adj + (size_t)s * W;
    for (int w = lane; w < W; w += 32) cand[w] = rs[w];
    __syncwarp();
    if (out && lane == 0) out[0] = s;
    int size = 1, from = 0;
    for (;;) {
        const int u = first_bit(cand, from, W, lane);
        if (u < 0) break;
        if (out && lane == 0) out[size] = u;
        ++size;
        from = u >> 5;                                  // every later member ranks above u
        const uint32_t* ru = adj + (size_t)u * W;
        for (int w = from + lane; w < W; w += 32) cand[w] &= ru[w];
        __syncwarp();
    }
    return size;
}

// BBMC greedy colouring of the set Pe: colour classes built in rank order, each class taking the lowest remaining vertex
// not adjacent to the class so far.  lane 0 writes vertex / colour in colouring order; returns their number.
__device__ int colour(const uint32_t* adj, int W, const uint32_t* Pe, uint32_t* U, uint32_t* Q, int lane, int* lv, int* lc)
{
    for (int w = lane; w < W; w += 32) U[w] = Pe[w];
    __syncwarp();
    int m = 0, k = 0, ufrom = 0;
    for (;;) {
        int v = first_bit(U, ufrom, W, lane);
        if (v < 0) break;
        ufrom = v >> 5;
        ++k;
        for (int w = ufrom + lane; w < W; w += 32) Q[w] = U[w];
        __syncwarp();
        while (v >= 0) {
            if (lane == 0) { lv[m] = v; lc[m] = k; }
            ++m;
            const int vw = v >> 5;
            const uint32_t vb = 1u << (v & 31);
            const uint32_t* rv = adj + (size_t)v * W;
            for (int w = vw + lane; w < W; w += 32) {
                Q[w] &= ~rv[w] & (w == vw ? ~vb : ~0u);
                if (w == vw) U[w] &= ~vb;
            }
            __syncwarp();
            v = first_bit(Q, vw, W, lane);
        }
    }
    __syncwarp();
    return m;
}

__global__ void __launch_bounds__(kThreads)
teaser_clique_kernel(const int* __restrict__ count, int ld, long long max_nodes, void* ws, Layout lay, int* clique_out,
                     int* __restrict__ clique_size, int* __restrict__ exact_out)
{
    extern __shared__ uint32_t tz_smem[];
    __shared__ int red_size[kWarps], red_start[kWarps], s_best, s_start, s_exact;
    const int p = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int W = (ld + 31) / 32;
    uint32_t* Pc = tz_smem;                 // the current level's candidates (first: the alive set)
    uint32_t* U = Pc + W;
    uint32_t* Q = U + W;
    uint32_t* cand = Q + W + (size_t)warp * W;
    const int M = match_count(count, p, ld);
    const uint32_t* adj = region<uint32_t>(ws, lay.adj, p, (size_t)ld * W);
    uint32_t* stk = region<uint32_t>(ws, lay.stk, p, (size_t)(ld + 1) * W);
    int* best = region<int>(ws, lay.best, p, ld);

    // ---- 1. heuristic incumbent: the largest greedy clique from the first min(M, 64) ranks, the earliest on ties
    int bsz = 0, bst = -1;
    for (int s = warp; s < min(M, kStarts); s += kWarps) {
        const int size = greedy_clique(adj, W, s, cand, lane, nullptr);
        if (size > bsz) { bsz = size; bst = s; }
    }
    if (lane == 0) { red_size[warp] = bsz; red_start[warp] = bst; }
    __syncthreads();
    if (tid == 0) {
        int b = 0, s = -1;
        for (int w = 0; w < kWarps; ++w)
            if (red_size[w] > b || (red_size[w] == b && b > 0 && red_start[w] < s)) { b = red_size[w]; s = red_start[w]; }
        s_best = b; s_start = s; s_exact = 1;
    }
    __syncthreads();
    if (warp == 0 && s_start >= 0) greedy_clique(adj, W, s_start, cand, lane, best);

    // ---- 2. peeling: drop every alive vertex whose alive-degree is below |best| until none is
    int bsize = s_best;
    for (int w = tid; w < W; w += kThreads) {
        const int lo = w * 32;
        Pc[w] = lo + 32 <= M ? 0xffffffffu : (lo >= M ? 0u : (1u << (M - lo)) - 1u);
    }
    for (;;) {
        for (int w = tid; w < W; w += kThreads) Q[w] = 0u;
        __syncthreads();
        int dropped = 0;
        for (int v = tid; v < M; v += kThreads) {
            if (!(Pc[v >> 5] >> (v & 31) & 1u)) continue;
            const uint32_t* rv = adj + (size_t)v * W;
            int d = 0;
            for (int w = 0; w < W; ++w) d += __popc(rv[w] & Pc[w]);
            if (d < bsize) { atomicOr(&Q[v >> 5], 1u << (v & 31)); dropped = 1; }
        }
        if (!__syncthreads_or(dropped)) break;
        for (int w = tid; w < W; w += kThreads) Pc[w] &= ~Q[w];
        __syncthreads();
    }

    // ---- 3. branch and bound (warp 0): stack level d holds its entry set in stk + d*W, the path and the resume position
    if (warp == 0 && M > 0) {
        int* lvl_i = region<int>(ws, lay.lvl_i, p, ld + 1);
        int* lvl_v = region<int>(ws, lay.lvl_v, p, ld + 1);
        int* lv = region<int>(ws, lay.list_v, p, ld);
        int* lc = region<int>(ws, lay.list_c, p, ld);
        for (int w = lane; w < W; w += 32) stk[w] = Pc[w];
        __syncwarp();
        long long nodes = 1;                               // the root call
        int d = 0;
        int i = colour(adj, W, stk, U, Q, lane, lv, lc) - 1;
        for (;;) {
            if (i < 0 || d + lc[i] <= bsize) {             // bound: return to the parent level
                if (d == 0) break;
                --d;
                const uint32_t* Pe = stk + (size_t)d * W;
                const int m = colour(adj, W, Pe, U, Q, lane, lv, lc);
                i = lvl_i[d];
                for (int w = lane; w < W; w += 32) Pc[w] = Pe[w];
                __syncwarp();
                for (int j = i + lane; j < m; j += 32) atomicAnd(&Pc[lv[j] >> 5], ~(1u << (lv[j] & 31)));
                __syncwarp();
                --i;
                continue;
            }
            const int v = lv[i];
            uint32_t* Pn = stk + (size_t)(d + 1) * W;
            const uint32_t* rv = adj + (size_t)v * W;
            bool any = false;
            for (int w = lane; w < W; w += 32) {
                const uint32_t x = Pc[w] & rv[w];
                Pn[w] = x;
                any |= x != 0u;
            }
            if (!__any_sync(0xffffffffu, any)) {           // C + {v} is maximal
                if (d + 1 > bsize) {
                    for (int j = lane; j < d; j += 32) best[j] = lvl_v[j];
                    if (lane == 0) best[d] = v;
                    bsize = d + 1;
                }
                if (lane == (v >> 5) % 32) Pc[v >> 5] &= ~(1u << (v & 31));
                __syncwarp();
                --i;
                continue;
            }
            if (nodes == max_nodes) { if (lane == 0) s_exact = 0; break; }
            ++nodes;
            if (lane == 0) { lvl_v[d] = v; lvl_i[d] = i; }
            ++d;
            __syncwarp();
            i = colour(adj, W, Pn, U, Q, lane, lv, lc) - 1;
            for (int w = lane; w < W; w += 32) Pc[w] = Pn[w];
            __syncwarp();
        }
        if (lane == 0) s_best = bsize;
    }
    __syncthreads();

    // ---- 4. the clique as ascending match positions
    bsize = s_best;
    const int* perm = region<int>(ws, lay.perm, p, ld);
    for (int w = tid; w < W; w += kThreads) Q[w] = 0u;
    __syncthreads();
    for (int k = tid; k < bsize; k += kThreads) {
        const int v = perm[best[k]];
        atomicOr(&Q[v >> 5], 1u << (v & 31));
    }
    __syncthreads();
    int* cq = region<int>(ws, lay.cliq, p, ld);
    int* co = clique_out ? clique_out + (size_t)p * ld : nullptr;
    if (warp == 0) {
        int base = 0;
        for (int w0 = 0; w0 < W; w0 += 32) {
            const int w = w0 + lane;
            uint32_t x = w < W ? Q[w] : 0u;
            const int c = __popc(x);
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += y;
            }
            int pos = base + incl - c;
            while (x) {
                const int v = w * 32 + __ffs(x) - 1;
                x &= x - 1u;
                cq[pos] = v;
                if (co) co[pos] = v;
                ++pos;
            }
            base += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
    if (co)
        for (int k = bsize + tid; k < ld; k += kThreads) co[k] = -1;
    if (tid == 0) {
        clique_size[p] = bsize;
        exact_out[p] = s_exact;
    }
}

// ---------------------------------------------------------------------------------------------- rotation, translation
// sweep event e < 2K of the intervals [x_k - r, x_k + r]: (value, type 0 enter / 1 leave, index); key order lexicographic
__device__ __forceinline__ bool key_le(double v1, int t1, int i1, double v2, int t2, int i2)
{
    return v1 < v2 || (v1 == v2 && (t1 < t2 || (t1 == t2 && i1 <= i2)));
}

__global__ void __launch_bounds__(kThreads)
teaser_solve_kernel(const float* __restrict__ src, const float* __restrict__ tgt, const int* __restrict__ idx1,
                    const int* __restrict__ idx2, const int* __restrict__ count, int n1, int n2, int ld, TeaserParams o,
                    void* ws, Layout lay, const int* __restrict__ clique_size, float* __restrict__ T_out,
                    int* __restrict__ inliers_out)
{
    __shared__ double red[(kThreads / 32) * 9];
    __shared__ double Rs[9], s_mu, s_prev, s_t[3];
    __shared__ double c_cost[kThreads], c_val[kThreads], c_est[kThreads];
    __shared__ int c_key[kThreads], s_stop;
    __shared__ Rt Tf;
    const int p = blockIdx.x, tid = threadIdx.x;
    const PairMatches pm(src, tgt, idx1, idx2, p, n1, n2, ld);
    const int M = match_count(count, p, ld);
    const int K = clique_size[p];
    const bool posed = M >= 3 && K >= 3;
    if (posed) {
        const int* cl = region<int>(ws, lay.cliq, p, ld);
        double* tim = region<double>(ws, lay.tim, p, (size_t)ld * 6);
        double* wt = region<double>(ws, lay.wt, p, ld);
        double* xs = region<double>(ws, lay.xs, p, ld);
        // ---- chain TIMs v_k = a_{c(k+1)} - a_{c(k)}, w_k = b_{c(k+1)} - b_{c(k)}, the last wrapping to the first
        for (int k = tid; k < K; k += kThreads) {
            float3 a0, b0, a1, b1;
            pm.load(cl[k], a0, b0);
            pm.load(cl[k + 1 == K ? 0 : k + 1], a1, b1);
            double* t = tim + 6 * (size_t)k;
            t[0] = (double)a1.x - a0.x; t[1] = (double)a1.y - a0.y; t[2] = (double)a1.z - a0.z;
            t[3] = (double)b1.x - b0.x; t[4] = (double)b1.y - b0.y; t[5] = (double)b1.z - b0.z;
            wt[k] = 1.0;
        }
        if (tid == 0) {
#pragma unroll
            for (int i = 0; i < 9; ++i) Rs[i] = (i % 4 == 0) ? 1.0 : 0.0;
            s_mu = 1.0; s_prev = 0.0;
        }
        __syncthreads();
        // ---- GNC-TLS: R = Horn(sum w v w^T); weights in closed form; mu grows by gnc_factor
        for (int it = 0; it < o.max_iterations; ++it) {
            double S[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
            for (int k = tid; k < K; k += kThreads) {
                const double* t = tim + 6 * (size_t)k;
                const double w = wt[k];
#pragma unroll
                for (int i = 0; i < 3; ++i)
#pragma unroll
                    for (int j = 0; j < 3; ++j) S[3 * i + j] += w * t[i] * t[3 + j];
            }
            block_sum<9>(S, red);
            if (tid == 0) horn_rotation(S, Rs);
            __syncthreads();
            double R[9];
#pragma unroll
            for (int i = 0; i < 9; ++i) R[i] = Rs[i];
            double rmax = 0.0;
            for (int k = tid; k < K; k += kThreads) {
                const double* t = tim + 6 * (size_t)k;
                const double dx = t[3] - (R[0] * t[0] + R[1] * t[1] + R[2] * t[2]);
                const double dy = t[4] - (R[3] * t[0] + R[4] * t[1] + R[5] * t[2]);
                const double dz = t[5] - (R[6] * t[0] + R[7] * t[1] + R[8] * t[2]);
                xs[k] = dx * dx + dy * dy + dz * dz;
                rmax = fmax(rmax, xs[k]);
            }
            if (it == 0) {
                rmax = block_max(rmax, red);
                if (tid == 0) {
                    s_mu = 1.0 / (2.0 * rmax / o.c2 - 1.0);
                    s_stop = !(s_mu > 0.0);
                }
                __syncthreads();
                if (s_stop) break;
            }
            const double mu = s_mu;
            const double th1 = (mu + 1.0) / mu * o.c2, th2 = mu / (mu + 1.0) * o.c2;
            double cost[1] = {0.0};
            for (int k = tid; k < K; k += kThreads) {
                const double r2 = xs[k];
                cost[0] += wt[k] * r2;
                wt[k] = r2 >= th1 ? 0.0 : (r2 <= th2 ? 1.0 : sqrt(o.c2 * mu * (mu + 1.0) / r2) - mu);
            }
            block_sum<1>(cost, red);
            if (tid == 0) {
                const double diff = fabs(cost[0] - s_prev);
                s_mu = mu * o.gnc_factor;
                s_prev = cost[0];
                s_stop = diff < o.cost_threshold;
            }
            __syncthreads();
            if (s_stop) break;
        }
        double R[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) R[i] = Rs[i];
        // ---- adaptive voting per axis over x_k = b_k - R a_k: every candidate's consensus set summed in index order
        const double r = o.range, r2 = o.range * o.range;
        for (int ax = 0; ax < 3; ++ax) {
            __syncthreads();                                    // xs is rewritten
            for (int k = tid; k < K; k += kThreads) {
                float3 a, b;
                pm.load(cl[k], a, b);
                const double bx = ax == 0 ? b.x : (ax == 1 ? b.y : b.z);
                xs[k] = bx - (R[3 * ax] * a.x + R[3 * ax + 1] * a.y + R[3 * ax + 2] * a.z);
            }
            __syncthreads();
            double bcost = 0.0, bval = 0.0, best_est = 0.0;
            int bkey = -1;
            for (int e = tid; e < 2 * K; e += kThreads) {
                const int ty = e >= K, ie = ty ? e - K : e;
                const double ve = ty ? __dadd_rn(xs[ie], r) : __dsub_rn(xs[ie], r);
                int n = 0;
                double s = 0.0;
                for (int j = 0; j < K; ++j) {
                    const double x = xs[j];
                    if (key_le(__dsub_rn(x, r), 0, j, ve, ty, ie) && !key_le(__dadd_rn(x, r), 1, j, ve, ty, ie)) {
                        ++n;
                        s += x;
                    }
                }
                if (n == 0) continue;
                const double est = s / n;
                double q = 0.0;
                for (int j = 0; j < K; ++j) {
                    const double x = xs[j];
                    if (key_le(__dsub_rn(x, r), 0, j, ve, ty, ie) && !key_le(__dadd_rn(x, r), 1, j, ve, ty, ie))
                        q += (x - est) * (x - est);
                }
                const double cost = q + (double)(K - n) * r2;
                const int key = ty * K + ie;
                if (bkey < 0 || cost < bcost ||
                    (cost == bcost && key_le(ve, ty, ie, bval, bkey >= K, bkey >= K ? bkey - K : bkey))) {
                    bcost = cost; bval = ve; bkey = key; best_est = est;
                }
            }
            c_cost[tid] = bcost; c_val[tid] = bval; c_key[tid] = bkey; c_est[tid] = best_est;
            __syncthreads();
            if (tid == 0) {
                int b = -1;
                for (int k = 0; k < kThreads; ++k) {
                    if (c_key[k] < 0) continue;
                    if (b < 0 || c_cost[k] < c_cost[b] ||
                        (c_cost[k] == c_cost[b] && key_le(c_val[k], c_key[k] >= K, c_key[k] >= K ? c_key[k] - K : c_key[k],
                                                          c_val[b], c_key[b] >= K, c_key[b] >= K ? c_key[b] - K : c_key[b])))
                        b = k;
                }
                s_t[ax] = c_est[b];
            }
        }
    }
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 9; ++i) Tf.r[i] = posed ? (float)Rs[i] : ((i % 4 == 0) ? 1.f : 0.f);
#pragma unroll
        for (int i = 0; i < 3; ++i) Tf.t[i] = posed ? (float)s_t[i] : 0.f;
    }
    __syncthreads();
    const Rt T = Tf;
    double c1[1] = {0};
    if (posed) {
        const float t2h = o.inlier_dist * o.inlier_dist;
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
    }
}

}  // namespace

extern "C" size_t ri_teaser_workspace_bytes(int P, int ld)
{
    if (P <= 0 || ld <= 0 || ld > kMaxLd) return 0;
    return Layout(P, ld).total;
}

extern "C" int ri_teaser_f32(const float* src, const float* tgt, const int* idx1, const int* idx2, const int* count, int P,
                             int n1, int n2, int ld, float noise_bound, float cbar2, float gnc_factor, int max_iterations,
                             float cost_threshold, long long max_clique_nodes, float inlier_dist, float* T, int* inliers,
                             int* clique, int* clique_size, int* exact, void* workspace, size_t workspace_bytes,
                             void* stream)
{
    if (P < 0 || n1 <= 0 || n2 <= 0 || ld <= 0 || !(noise_bound > 0.f) || !isfinite(noise_bound) || !(cbar2 > 0.f) ||
        !isfinite(cbar2) || !(inlier_dist > 0.f) || !isfinite(inlier_dist) || !(gnc_factor > 1.f) || max_iterations < 0 ||
        max_clique_nodes < 1 || clique_size == nullptr || exact == nullptr)
        return RI_ERR_BAD_ARG;
    if (ld > kMaxLd || P > 65535) return RI_ERR_UNSUPPORTED;
    if (P == 0) return RI_OK;
    const Layout lay(P, ld);
    if (workspace == nullptr || workspace_bytes < lay.total) return RI_ERR_WORKSPACE;
    const cudaStream_t s = (cudaStream_t)stream;
    const int W = (ld + 31) / 32;
    const double beta = 2.0 * (double)noise_bound * sqrt((double)cbar2);
    teaser_graph_kernel<<<dim3((ld + kWarps - 1) / kWarps, P), kThreads, 0, s>>>(src, tgt, idx1, idx2, count, n1, n2, ld,
                                                                                 beta, workspace, lay);
    RI_LAUNCH_CHECK();
    teaser_rank_kernel<<<dim3((ld + kThreads - 1) / kThreads, P), kThreads, 0, s>>>(count, ld, workspace, lay);
    RI_LAUNCH_CHECK();
    const long long words = (long long)ld * W;
    teaser_permute_kernel<<<dim3((unsigned)((words + kThreads - 1) / kThreads), P), kThreads, 0, s>>>(count, ld, workspace,
                                                                                                      lay);
    RI_LAUNCH_CHECK();
    const size_t smem = (size_t)(3 + kWarps) * W * sizeof(uint32_t);
    teaser_clique_kernel<<<P, kThreads, smem, s>>>(count, ld, max_clique_nodes, workspace, lay, clique, clique_size, exact);
    RI_LAUNCH_CHECK();
    const TeaserParams o{beta, beta * beta, (double)noise_bound * sqrt((double)cbar2), (double)gnc_factor,
                         (double)cost_threshold, max_iterations, max_clique_nodes, inlier_dist};
    teaser_solve_kernel<<<P, kThreads, 0, s>>>(src, tgt, idx1, idx2, count, n1, n2, ld, o, workspace, lay, clique_size, T,
                                               inliers);
    RI_LAUNCH_CHECK();
    return RI_OK;
}
