// 30-bit Morton codes of points in a box cut into 1024^3 cells: the locality order of the pruned KNN (knn_pruned.cu)
// and of the ICP target tiles and landmark groups (icp.cu).
#pragma once

namespace fb {

__device__ __forceinline__ unsigned spread10(unsigned v) {  // 10 bits -> every third bit
  v &= 0x3ffu;
  v = (v | (v << 16)) & 0x030000ffu;
  v = (v | (v << 8)) & 0x0300f00fu;
  v = (v | (v << 4)) & 0x030c30c3u;
  v = (v | (v << 2)) & 0x09249249u;
  return v;
}

// first min(dim, 3) coordinates of p, relative to lo and scaled by inv (= 1024 / extent, 0 for a flat axis)
__device__ __forceinline__ unsigned morton3(const double* p, int dim, const double* lo, const double* inv) {
  unsigned key = 0;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    unsigned q = 0;
    if (c < dim) {
      double t = (p[c] - lo[c]) * inv[c];
      t = fmin(fmax(t, 0.0), 1023.0);
      q = (unsigned)t;
    }
    key |= spread10(q) << c;
  }
  return key;
}

}  // namespace fb
