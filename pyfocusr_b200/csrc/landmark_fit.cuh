// vtkLandmarkTransform (Horn 1987, unit quaternions; rigid body or similarity) on the device, shared by the ICP
// iterations (K10, icp.cu) and the Procrustes fits of the shape model (K13, shape.cu), so both fit bit for bit alike.
// The numpy restatement is oracle/icp_port.py::landmark_transform.
#pragma once
#include <cuda_runtime.h>

namespace fb {

constexpr int FIT_THREADS = 256;  // threads of a CTA that runs landmark_fit_block

// fixed-tree block sum (blockDim.x a power of two <= 1024); every thread gets the total
__device__ __forceinline__ double fit_block_sum(double v, double* red) {
  const int t = threadIdx.x;
  __syncthreads();
  red[t] = v;
  __syncthreads();
  for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
    if (t < s) red[t] += red[t + s];
    __syncthreads();
  }
  return red[0];
}

// The 4x4 matrix (row-major, column vectors) taking point set a onto point set b, from M = {sum (a - ca)(b - cb)^T
// row-major, sum |a - ca|^2, sum |b - cb|^2} and the centroids ca, cb of nb points: Horn's 4x4 matrix, its dominant
// eigenvector by cyclic Jacobi, rotation (times sqrt(sb / sa) for a similarity), translation cb - R ca.  A single point
// or a set whose points coincide gives the identity rotation plus that translation.
__device__ __forceinline__ void horn_matrix(const double* M, const double* ca, const double* cb, int nb, int similarity,
                                            double* Lm) {
  double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  const double sa = M[9], sb = M[10];
  if (nb > 1 && sa != 0.0 && sb != 0.0) {
    double N[4][4], V[4][4];
    N[0][0] = M[0] + M[4] + M[8];
    N[1][1] = M[0] - M[4] - M[8];
    N[2][2] = -M[0] + M[4] - M[8];
    N[3][3] = -M[0] - M[4] + M[8];
    N[0][1] = N[1][0] = M[5] - M[7];
    N[0][2] = N[2][0] = M[6] - M[2];
    N[0][3] = N[3][0] = M[1] - M[3];
    N[1][2] = N[2][1] = M[1] + M[3];
    N[1][3] = N[3][1] = M[6] + M[2];
    N[2][3] = N[3][2] = M[5] + M[7];
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) V[i][j] = i == j ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 60; ++sweep) {  // cyclic Jacobi
      double off = 0.0, diag = 0.0;
      for (int i = 0; i < 4; ++i) {
        diag += N[i][i] * N[i][i];
        for (int j = i + 1; j < 4; ++j) off += N[i][j] * N[i][j];
      }
      if (off <= 1e-32 * diag || off == 0.0) break;
      for (int p = 0; p < 3; ++p)
        for (int q = p + 1; q < 4; ++q) {
          if (N[p][q] == 0.0) continue;
          const double theta = (N[q][q] - N[p][p]) / (2.0 * N[p][q]);
          const double tt = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
          const double c = 1.0 / sqrt(tt * tt + 1.0), sn = tt * c;
          for (int k = 0; k < 4; ++k) {
            const double nkp = N[k][p], nkq = N[k][q];
            N[k][p] = c * nkp - sn * nkq;
            N[k][q] = sn * nkp + c * nkq;
          }
          for (int k = 0; k < 4; ++k) {
            const double npk = N[p][k], nqk = N[q][k];
            N[p][k] = c * npk - sn * nqk;
            N[q][k] = sn * npk + c * nqk;
          }
          for (int k = 0; k < 4; ++k) {
            const double vkp = V[k][p], vkq = V[k][q];
            V[k][p] = c * vkp - sn * vkq;
            V[k][q] = sn * vkp + c * vkq;
          }
        }
    }
    int top = 0;
    for (int i = 1; i < 4; ++i)
      if (N[i][i] > N[top][top]) top = i;
    const double w = V[0][top], x = V[1][top], y = V[2][top], z = V[3][top];
    const double ww = w * w, wx = w * x, wy = w * y, wz = w * z, xx = x * x, yy = y * y, zz = z * z, xy = x * y, xz = x * z, yz = y * z;
    R[0] = ww + xx - yy - zz;
    R[3] = 2.0 * (wz + xy);
    R[6] = 2.0 * (-wy + xz);
    R[1] = 2.0 * (-wz + xy);
    R[4] = ww - xx + yy - zz;
    R[7] = 2.0 * (wx + yz);
    R[2] = 2.0 * (wy + xz);
    R[5] = 2.0 * (-wx + yz);
    R[8] = ww - xx - yy + zz;
    if (similarity) {
      const double sc = sqrt(sb / sa);
      for (int i = 0; i < 9; ++i) R[i] *= sc;
    }
  }
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) Lm[4 * r + c] = R[3 * r + c];
    Lm[4 * r + 3] = cb[r] - (R[3 * r] * ca[0] + R[3 * r + 1] * ca[1] + R[3 * r + 2] * ca[2]);
  }
  Lm[12] = Lm[13] = Lm[14] = 0.0;
  Lm[15] = 1.0;
}

// The landmark transform of a [nb][3] -> b [nb][3] by one CTA of FIT_THREADS threads (`red`: FIT_THREADS doubles of
// shared memory), every sum a fixed tree: returns true in thread 0, which then holds the matrix in Lm, and false in the
// others.  Every thread must call it.
__device__ __forceinline__ bool landmark_fit_block(const double* __restrict__ a, const double* __restrict__ b, int nb,
                                                   int similarity, double* red, double* Lm) {
  const int t = threadIdx.x;
  double s[6] = {0, 0, 0, 0, 0, 0};
  for (int i = t; i < nb; i += FIT_THREADS)
    for (int d = 0; d < 3; ++d) {
      s[d] += a[3 * i + d];
      s[3 + d] += b[3 * i + d];
    }
  double ca[3], cb[3];
  for (int d = 0; d < 3; ++d) {
    ca[d] = fit_block_sum(s[d], red) / nb;
    cb[d] = fit_block_sum(s[3 + d], red) / nb;
  }
  double m[11] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};  // M row-major, sa, sb
  for (int i = t; i < nb; i += FIT_THREADS) {
    double x[3], y[3];
    for (int d = 0; d < 3; ++d) {
      x[d] = a[3 * i + d] - ca[d];
      y[d] = b[3 * i + d] - cb[d];
    }
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) m[3 * r + c] += x[r] * y[c];
    m[9] += x[0] * x[0] + x[1] * x[1] + x[2] * x[2];
    m[10] += y[0] * y[0] + y[1] * y[1] + y[2] * y[2];
  }
  double M[11];
  for (int k = 0; k < 11; ++k) M[k] = fit_block_sum(m[k], red);
  if (t != 0) return false;
  horn_matrix(M, ca, cb, nb, similarity, Lm);
  return true;
}

}  // namespace fb
