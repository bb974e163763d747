// rigid.cuh — fp64 rigid-transform solvers and the block reduction shared by csrc/pose.cu, csrc/icp.cu, csrc/fgr.cu
// and csrc/teaser.cu.
#pragma once
#include <cuda_runtime.h>

namespace {

// ---- Horn's closed form: unit quaternion of the rotation that best maps the centred a's onto the centred b's,
//      S[3*i + j] = sum a_i b_j.  Largest eigenvector of the symmetric 4x4 N by cyclic Jacobi sweeps (fp64).
__device__ void horn_rotation(const double S[9], double R[9])
{
    double a[4][4], v[4][4];
    const double Sxx = S[0], Sxy = S[1], Sxz = S[2], Syx = S[3], Syy = S[4], Syz = S[5], Szx = S[6], Szy = S[7], Szz = S[8];
    a[0][0] = Sxx + Syy + Szz; a[0][1] = Syz - Szy; a[0][2] = Szx - Sxz; a[0][3] = Sxy - Syx;
    a[1][1] = Sxx - Syy - Szz; a[1][2] = Sxy + Syx; a[1][3] = Szx + Sxz;
    a[2][2] = -Sxx + Syy - Szz; a[2][3] = Syz + Szy;
    a[3][3] = -Sxx - Syy + Szz;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { if (j < i) a[i][j] = a[j][i]; v[i][j] = i == j ? 1.0 : 0.0; }
    for (int sweep = 0; sweep < 12; ++sweep) {
        double off = 0.0;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = i + 1; j < 4; ++j) off += a[i][j] * a[i][j];
        if (off < 1e-30) break;
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int q = p + 1; q < 4; ++q) {
                const double apq = a[p][q];
                if (fabs(apq) < 1e-300) continue;
                const double theta = (a[q][q] - a[p][p]) / (2.0 * apq);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
                for (int k = 0; k < 4; ++k) {               // A <- A J (columns p, q)
                    const double akp = a[k][p], akq = a[k][q];
                    a[k][p] = c * akp - s * akq; a[k][q] = s * akp + c * akq;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {               // A <- J^T A (rows p, q)
                    const double apk = a[p][k], aqk = a[q][k];
                    a[p][k] = c * apk - s * aqk; a[q][k] = s * apk + c * aqk;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const double vkp = v[k][p], vkq = v[k][q];
                    v[k][p] = c * vkp - s * vkq; v[k][q] = s * vkp + c * vkq;
                }
            }
    }
    int best = 0;
#pragma unroll
    for (int i = 1; i < 4; ++i) if (a[i][i] > a[best][best]) best = i;
    double qw = 0, qx = 0, qy = 0, qz = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) if (i == best) { qw = v[0][i]; qx = v[1][i]; qy = v[2][i]; qz = v[3][i]; }
    const double nq = sqrt(qw * qw + qx * qx + qy * qy + qz * qz);
    qw /= nq; qx /= nq; qy /= nq; qz /= nq;
    R[0] = 1 - 2 * (qy * qy + qz * qz); R[1] = 2 * (qx * qy - qz * qw); R[2] = 2 * (qx * qz + qy * qw);
    R[3] = 2 * (qx * qy + qz * qw); R[4] = 1 - 2 * (qx * qx + qz * qz); R[5] = 2 * (qy * qz - qx * qw);
    R[6] = 2 * (qx * qz - qy * qw); R[7] = 2 * (qy * qz + qx * qw); R[8] = 1 - 2 * (qx * qx + qy * qy);
}

// block-wide sum of NV doubles per thread; result valid in thread 0
template <int NV>
__device__ void block_sum(double (&v)[NV], double* red)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int k = 0; k < NV; ++k)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], o);
    __syncthreads();
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < NV; ++k) red[warp * NV + k] = v[k];
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < nw; ++w)
#pragma unroll
            for (int k = 0; k < NV; ++k) v[k] += red[w * NV + k];
}

// block-wide maximum of one double per thread; result valid in thread 0
__device__ __forceinline__ double block_max(double v, double* red)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_down_sync(0xffffffffu, v, o));
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < nw; ++w) v = fmax(v, red[w]);
    return v;
}

// Solves A x = b for the symmetric 6x6 A given by its 21 upper-triangle entries in row order (A00 A01 .. A05 A11 .. A55),
// by an LDL^T factorisation without pivoting (A = J^T J is positive semi-definite).  det = prod(D) = det(A).  Returns false
// when the factorisation or the solution is not finite, and
//   min_det > 0:  when |det| < min_det.  ICP passes 1e-6: Open3D's SolveLinearSystemPSD rejects the same systems, and its
//                 caller (SolveJacobianSystemAndObtainExtrinsicMatrix) then returns the identity;
//   min_det <= 0: when a pivot D[j] is not positive, i.e. A is not numerically positive definite (FGR: where an LLT
//                 factorisation would break down).
__device__ bool ldlt_solve6(const double up[21], const double b[6], double x[6], double min_det)
{
    double L[6][6], D[6];
    double A[6][6];
    int k = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = i; j < 6; ++j) { A[i][j] = up[k]; A[j][i] = up[k]; ++k; }
    double det = 1.0;
    bool pd = true;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        double d = A[j][j];
#pragma unroll
        for (int m = 0; m < j; ++m) d -= L[j][m] * L[j][m] * D[m];
        D[j] = d;
        det *= d;
        pd = pd && d > 0.0;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            double s = A[i][j];
#pragma unroll
            for (int m = 0; m < j; ++m) s -= L[i][m] * L[j][m] * D[m];
            L[i][j] = s / d;
        }
    }
    if ((min_det > 0.0 ? !(fabs(det) >= min_det) : !pd) || !isfinite(det)) return false;
    double y[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {                      // L y = b
        double s = b[i];
#pragma unroll
        for (int m = 0; m < i; ++m) s -= L[i][m] * y[m];
        y[i] = s;
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {                     // D L^T x = y
        double s = y[i] / D[i];
#pragma unroll
        for (int m = i + 1; m < 6; ++m) s -= L[m][i] * x[m];
        x[i] = s;
    }
    bool ok = true;
#pragma unroll
    for (int i = 0; i < 6; ++i) ok = ok && isfinite(x[i]);
    return ok;
}

}  // namespace
