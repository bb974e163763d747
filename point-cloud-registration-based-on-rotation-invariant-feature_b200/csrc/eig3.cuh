// eig3.cuh — fp64 cyclic Jacobi sweeps on a symmetric 3x3 matrix, shared by csrc/normals.cu (the eigenvector of the
// smallest eigenvalue) and csrc/iss.cu (the three eigenvalues).  The caller scales the matrix to unit trace: the
// thresholds below are absolute.
#pragma once

namespace {

// On return the diagonal of a holds the eigenvalues (unsorted) and column i of v the eigenvector of a[i][i].
// Cyclic Jacobi as horn_rotation (csrc/rigid.cuh).
__device__ __forceinline__ void jacobi3(double a[3][3], double v[3][3])
{
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) v[i][j] = i == j ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 12; ++sweep) {
        const double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2];
        if (off < 1e-30) break;
#pragma unroll
        for (int p = 0; p < 2; ++p)
#pragma unroll
            for (int q = p + 1; q < 3; ++q) {
                const double apq = a[p][q];
                if (fabs(apq) < 1e-300) continue;
                const double theta = (a[q][q] - a[p][p]) / (2.0 * apq);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
#pragma unroll
                for (int k = 0; k < 3; ++k) {               // A <- A J (columns p, q)
                    const double akp = a[k][p], akq = a[k][q];
                    a[k][p] = cs * akp - sn * akq; a[k][q] = sn * akp + cs * akq;
                }
#pragma unroll
                for (int k = 0; k < 3; ++k) {               // A <- J^T A (rows p, q)
                    const double apk = a[p][k], aqk = a[q][k];
                    a[p][k] = cs * apk - sn * aqk; a[q][k] = sn * apk + cs * aqk;
                }
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const double vkp = v[k][p], vkq = v[k][q];
                    v[k][p] = cs * vkp - sn * vkq; v[k][q] = sn * vkp + cs * vkq;
                }
            }
    }
}

}  // namespace
