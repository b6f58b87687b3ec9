// K10  ICP pre-alignment -- the reference's default `icp_register_first=True` (focusr.py:106-131 ->
// vtk_functions.py:12-37: vtkIterativeClosestPointTransform with a rigid-body / similarity
// vtkLandmarkTransform, 100 iterations, StartByMatchingCentroids; SURVEY.md section 8f-4).  VTK is an absent,
// unpinned dependency: the algorithm is the one of VTK 9 as restated in oracle/icp_port.py.
//
// Batched: every (fixed, moving) pair of a call is aligned by the same launches, and the single-pair entry point
// focusr_icp is the one-pair case of the same code.  Everything runs on the device with no synchronisation inside
// the loop: the accumulated 4x4 matrices, the per-iteration landmark transforms and the landmark positions live in HBM.
// Set-up, once per call:
//   k_icp_plan        per-pair sizes (landmark step and count, tiles, landmark groups) and their prefix sums.
//   k_icp_start       one 1024-thread CTA per pair: accumulated matrix = centroid match or identity.
//   k_icp_bbox/_keys  Morton code of every fixed-mesh triangle centroid (in that mesh's box) and of every landmark's
//                     source point (in the moving mesh's box); one CUB segmented radix sort orders both, per pair.
//   k_icp_fill/_tile_boxes  the sorted triangles' 9 coordinates stored contiguously with their original index, cut
//                     into tiles of ICP_TILE with a padded axis-aligned box each; the landmark order = groups of 32.
// Per iteration:
//   k_icp_closest     closest point ON THE FIXED SURFACE for every landmark: one warp per group of up to 32
//                     Morton-adjacent landmarks of one pair, over all pairs in one grid.  The bound is seeded with the
//                     previous winner (first iteration: the best triangle of the landmark's home tile); the warp then
//                     visits only the tiles whose box lies within the largest bound of its group.  Its lanes load a
//                     tile's triangles (one each) and evaluate, one landmark after the other, the landmarks whose own
//                     bound reaches the tile's box; a triangle is evaluated (Ericson's region test) unless its own box
//                     is STRICTLY beyond the landmark's best distance known.  Boxes are padded and their distances rounded down, so
//                     every triangle that can attain the minimum is evaluated: the winner is the lexicographic minimum
//                     of (d^2, original triangle index) over all triangles, bit-for-bit that of a brute-force scan,
//                     whatever the tiling or grouping.  The closest point is recomputed from the winner.
//   k_icp_fit         one 256-thread CTA per pair: centroids, M = sum a b^T, Horn's 4x4 matrix, its dominant
//                     eigenvector by cyclic Jacobi in one thread, rotation (+ scale), translation; acc <- L * acc.
//   k_icp_move        landmarks <- L landmarks.
// End: moved points = acc * moving points (k_icp_apply).
#include <limits.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include <cub/device/device_segmented_radix_sort.cuh>

#include "closest_point.cuh"
#include "common.cuh"
#include "landmark_fit.cuh"
#include "morton.cuh"

namespace fb {

// Triangles per target tile, measured at 128 pairs of 15 212-vertex / 30 420-triangle meshes, 100 iterations x 1000
// landmarks (tools/batch_icp_bench.py, B200 at 1000 W, profiles/r3_batch_icp_bench.json): 32 per tile 45.5 ms,
// 64 per tile 57.2 ms, identical matrices.
#ifndef FB_ICP_TILE
#define FB_ICP_TILE 32
#endif
constexpr int ICP_TILE = FB_ICP_TILE;
// Landmarks per group (one warp): 32 when the batch has enough groups to fill the GPU, fewer for small calls (a single
// pair: 1000 landmarks = 31 warps of 32) so that more warps share the search; the result does not depend on it.
constexpr int ICP_GROUPS[4] = {32, 16, 8, 4};
constexpr int ICP_WARPS = 4;   // groups per CTA of k_icp_closest
// The keys are Morton << 32 | index, written in index order: a stable radix sort of the 30 Morton bits alone gives the
// order of the whole keys.  CUB's segmented RADIX sort is used because it never waits for the device (its segmented merge
// sort reads segment sizes back to the host for batches of more than 500 segments).
constexpr int ICP_SORT_BITS[2] = {32, 62};
constexpr int ICP_BOX = 8;     // doubles per (pair, mesh) box record: lo[3], 1024 / extent[3], pad, 0

__device__ __forceinline__ P3 xform(const double* __restrict__ m, P3 p) {  // 4x4 row-major, column vectors
  return P3{m[0] * p.x + m[1] * p.y + m[2] * p.z + m[3], m[4] * p.x + m[5] * p.y + m[6] * p.z + m[7],
            m[8] * p.x + m[9] * p.y + m[10] * p.z + m[11]};
}

// one (fixed, moving) pair; point indices are rows of the call's fixed / moving point arrays
struct IcpPair {
  int fp0, fnp;  // fixed mesh: first point, point count
  int ft0, fnt;  // fixed mesh: first triangle, triangle count
  int mp0, mnp;  // moving mesh: first point, point count
  int step, nb;  // every step-th moving point is a landmark; nb landmarks
};

// Per-pair sizes and their exclusive prefix sums [P + 1]: landmarks, landmark groups, sorted triangles, tiles.  One
// CTA, chunks of 1024 pairs with a carry.  mesh_off == nullptr: one pair given by the scalars (focusr_icp).
__global__ void __launch_bounds__(1024)
k_icp_plan(const int* __restrict__ mesh_off, const int* __restrict__ tri_off, const int* __restrict__ fixed_mesh,
           const int* __restrict__ moving_mesh, int P, int one_fnp, int one_fnt, int one_mnp, int max_landmarks,
           int group, int n_sorted_tris, IcpPair* __restrict__ pairs, int* __restrict__ off_lm, int* __restrict__ off_grp,
           int* __restrict__ off_tri, int* __restrict__ off_tile, int* __restrict__ sort_begin, int* __restrict__ sort_end) {
  __shared__ int s[4][1024];
  __shared__ int carry[4];
  const int t = threadIdx.x;
  if (t < 4) carry[t] = 0;
  int* const out[4] = {off_lm, off_grp, off_tri, off_tile};
  for (int c0 = 0; c0 < P; c0 += 1024) {
    const int p = c0 + t;
    int v[4] = {0, 0, 0, 0};
    if (p < P) {
      IcpPair pr;
      if (mesh_off == nullptr) {
        pr.fp0 = 0, pr.fnp = one_fnp, pr.ft0 = 0, pr.fnt = one_fnt, pr.mp0 = 0, pr.mnp = one_mnp;
      } else {
        const int f = fixed_mesh[p], m = moving_mesh[p];
        pr.fp0 = mesh_off[f], pr.fnp = mesh_off[f + 1] - mesh_off[f];
        pr.ft0 = tri_off[f], pr.fnt = tri_off[f + 1] - tri_off[f];
        pr.mp0 = mesh_off[m], pr.mnp = mesh_off[m + 1] - mesh_off[m];
      }
      // vtkIterativeClosestPointTransform::InternalUpdate: every step-th source point is a landmark
      pr.step = pr.mnp > max_landmarks ? pr.mnp / max_landmarks : 1;
      pr.nb = pr.mnp / pr.step;
      pairs[p] = pr;
      v[0] = pr.nb;
      v[1] = (pr.nb + group - 1) / group;
      v[2] = pr.fnt;
      v[3] = (pr.fnt + ICP_TILE - 1) / ICP_TILE;
    }
    __syncthreads();
    for (int k = 0; k < 4; ++k) s[k][t] = v[k];
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {  // inclusive scan
      int x[4] = {0, 0, 0, 0};
      if (t >= d)
        for (int k = 0; k < 4; ++k) x[k] = s[k][t - d];
      __syncthreads();
      for (int k = 0; k < 4; ++k) s[k][t] += x[k];
      __syncthreads();
    }
    if (p < P) {
      int e[4];
      for (int k = 0; k < 4; ++k) {
        e[k] = carry[k] + s[k][t] - v[k];
        out[k][p] = e[k];
      }
      // segments of the one sort: the triangles of every pair, then the landmarks of every pair
      sort_begin[p] = e[2];
      sort_end[p] = e[2] + v[2];
      sort_begin[P + p] = n_sorted_tris + e[0];
      sort_end[P + p] = n_sorted_tris + e[0] + v[0];
    }
    __syncthreads();
    if (t < 4) carry[t] += s[t][1023];
  }
  __syncthreads();
  if (t < 4) out[t][P] = carry[t];
}

// acc = translation(fixed centroid - moving centroid) or identity; one CTA per pair
__global__ void __launch_bounds__(1024) k_icp_start(const IcpPair* __restrict__ pairs, const double* __restrict__ fixed_pts,
                                                   const double* __restrict__ moving_pts, int match, double* __restrict__ acc_all) {
  __shared__ double red[1024];
  const IcpPair pr = pairs[blockIdx.x];
  const double* src = moving_pts + 3 * (size_t)pr.mp0;
  const double* tgt = fixed_pts + 3 * (size_t)pr.fp0;
  const int ns = pr.mnp, nt = pr.fnp;
  double* acc = acc_all + 16 * (size_t)blockIdx.x;
  double s[3] = {0, 0, 0}, g[3] = {0, 0, 0};
  if (match) {
    for (int i = threadIdx.x; i < ns; i += 1024)
      for (int d = 0; d < 3; ++d) s[d] += src[3 * (size_t)i + d];
    for (int i = threadIdx.x; i < nt; i += 1024)
      for (int d = 0; d < 3; ++d) g[d] += tgt[3 * (size_t)i + d];
  }
  double tr[3];
  for (int d = 0; d < 3; ++d) {
    const double a = fit_block_sum(s[d], red), b = fit_block_sum(g[d], red);
    tr[d] = match ? b / nt - a / ns : 0.0;
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < 16; ++i) acc[i] = (i % 5 == 0) ? 1.0 : 0.0;
    acc[3] = tr[0];
    acc[7] = tr[1];
    acc[11] = tr[2];
  }
}

// grid (P, 2): y = 0 the fixed mesh's points (+ the box padding of its tiles), y = 1 the moving mesh's
__global__ void __launch_bounds__(256) k_icp_bbox(const IcpPair* __restrict__ pairs, const double* __restrict__ fixed_pts,
                                                 const double* __restrict__ moving_pts, double* __restrict__ box) {
  const IcpPair pr = pairs[blockIdx.x];
  const int which = blockIdx.y;
  const double* pts = which == 0 ? fixed_pts + 3 * (size_t)pr.fp0 : moving_pts + 3 * (size_t)pr.mp0;
  const int n = which == 0 ? pr.fnp : pr.mnp;
  double mn[3] = {1e300, 1e300, 1e300}, mx[3] = {-1e300, -1e300, -1e300};
  for (int i = threadIdx.x; i < n; i += 256)
    for (int c = 0; c < 3; ++c) {
      const double v = pts[3 * (size_t)i + c];
      mn[c] = fmin(mn[c], v);
      mx[c] = fmax(mx[c], v);
    }
  __shared__ double smn[3][256], smx[3][256];
  for (int c = 0; c < 3; ++c) {
    smn[c][threadIdx.x] = mn[c];
    smx[c][threadIdx.x] = mx[c];
  }
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o)
      for (int c = 0; c < 3; ++c) {
        smn[c][threadIdx.x] = fmin(smn[c][threadIdx.x], smn[c][threadIdx.x + o]);
        smx[c][threadIdx.x] = fmax(smx[c][threadIdx.x], smx[c][threadIdx.x + o]);
      }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    double* b = box + ICP_BOX * (2 * (size_t)blockIdx.x + which);
    double mag = 0.0;
    for (int c = 0; c < 3; ++c) {
      const double ext = smx[c][0] - smn[c][0];
      b[c] = smn[c][0];
      b[3 + c] = (ext > 0.0 && ext < 1e300) ? 1024.0 / ext : 0.0;
      mag = fmax(mag, fmax(fabs(smn[c][0]), fabs(smx[c][0])) + ext);
    }
    // Tile and triangle boxes are widened by this much: far more than the rounding error of a computed closest point
    // (a few ulps of the coordinates), far less than the distances that decide a pruning.
    b[6] = 1e-9 * mag;
    b[7] = 0.0;
  }
}

// keys (Morton << 32 | local index) of the fixed triangles' centroids and of the landmarks' source points
__global__ void __launch_bounds__(256)
k_icp_keys(const IcpPair* __restrict__ pairs, const int* __restrict__ off_lm, const int* __restrict__ off_tri,
           const double* __restrict__ fixed_pts, const int* __restrict__ tris, const double* __restrict__ moving_pts,
           const double* __restrict__ box, int n_sorted_tris, unsigned long long* __restrict__ keys) {
  const int p = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  const IcpPair pr = pairs[p];
  const double* fb = box + ICP_BOX * (2 * (size_t)p);
  const double* mb = fb + ICP_BOX;
  if (i < pr.fnt) {
    const int* tr = tris + 3 * (size_t)(pr.ft0 + i);
    const P3 a = p3(fixed_pts, tr[0]), b = p3(fixed_pts, tr[1]), c = p3(fixed_pts, tr[2]);
    const P3 m = (a + b + c) * (1.0 / 3.0);
    const double q[3] = {m.x, m.y, m.z};
    keys[off_tri[p] + i] = ((unsigned long long)morton3(q, 3, fb, fb + 3) << 32) | (unsigned)i;
  }
  if (i < pr.nb) {
    const double* q = moving_pts + 3 * ((size_t)pr.mp0 + (size_t)i * pr.step);
    keys[n_sorted_tris + off_lm[p] + i] = ((unsigned long long)morton3(q, 3, mb, mb + 3) << 32) | (unsigned)i;
  }
}

// sorted triangles -> contiguous vertex coordinates + original (mesh-local) index; sorted landmarks -> group order
__global__ void __launch_bounds__(256)
k_icp_fill(const IcpPair* __restrict__ pairs, const int* __restrict__ off_lm, const int* __restrict__ off_tri,
           const double* __restrict__ fixed_pts, const int* __restrict__ tris, const unsigned long long* __restrict__ keys,
           int n_sorted_tris, double* __restrict__ tv, int* __restrict__ tid, int* __restrict__ perm) {
  const int p = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  const IcpPair pr = pairs[p];
  if (i < pr.fnt) {
    const size_t pos = (size_t)off_tri[p] + i;
    const int orig = (int)(keys[pos] & 0xffffffffu);
    const int* tr = tris + 3 * (size_t)(pr.ft0 + orig);
    for (int v = 0; v < 3; ++v)
      for (int c = 0; c < 3; ++c) tv[9 * pos + 3 * v + c] = fixed_pts[3 * (size_t)tr[v] + c];
    tid[pos] = orig;
  }
  if (i < pr.nb) perm[off_lm[p] + i] = (int)(keys[(size_t)n_sorted_tris + off_lm[p] + i] & 0xffffffffu);
}

__global__ void __launch_bounds__(128)
k_icp_tile_boxes(const IcpPair* __restrict__ pairs, const int* __restrict__ off_tri, const int* __restrict__ off_tile,
                 const double* __restrict__ box, const double* __restrict__ tv, const unsigned long long* __restrict__ keys,
                 double* __restrict__ tile_lo, double* __restrict__ tile_hi, unsigned* __restrict__ tile_key) {
  const int p = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
  const int t0 = off_tile[p];
  if (j >= off_tile[p + 1] - t0) return;
  const IcpPair pr = pairs[p];
  const double pad = box[ICP_BOX * (2 * (size_t)p) + 6];
  const size_t r0 = (size_t)off_tri[p] + (size_t)j * ICP_TILE, r1 = (size_t)off_tri[p] + min(pr.fnt, (j + 1) * ICP_TILE);
  double mn[3] = {1e300, 1e300, 1e300}, mx[3] = {-1e300, -1e300, -1e300};
  for (size_t r = r0; r < r1; ++r)
    for (int v = 0; v < 3; ++v)
      for (int c = 0; c < 3; ++c) {
        const double x = tv[9 * r + 3 * v + c];
        mn[c] = fmin(mn[c], x);
        mx[c] = fmax(mx[c], x);
      }
  for (int c = 0; c < 3; ++c) {
    tile_lo[3 * (size_t)(t0 + j) + c] = mn[c] - pad;
    tile_hi[3 * (size_t)(t0 + j) + c] = mx[c] + pad;
  }
  tile_key[t0 + j] = (unsigned)(keys[r0] >> 32);
}

__global__ void k_icp_init_landmarks(const IcpPair* __restrict__ pairs, const int* __restrict__ off_lm,
                                     const double* __restrict__ moving_pts, const double* __restrict__ acc_all,
                                     double* __restrict__ a_all) {
  const int p = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  const IcpPair pr = pairs[p];
  if (i >= pr.nb) return;
  const double* src = moving_pts + 3 * (size_t)pr.mp0;
  double* a = a_all + 3 * (size_t)off_lm[p];
  const P3 q = xform(acc_all + 16 * (size_t)p, p3(src, (long long)i * pr.step));
  a[3 * i] = q.x;
  a[3 * i + 1] = q.y;
  a[3 * i + 2] = q.z;
}

// (landmark, triangle) closest-point evaluations of k_icp_closest since the last reset; counted only in builds with
// -DFB_ICP_COUNT (tools/batch_icp_bench.py), read through focusr_profile_get_kind(5, ...)
__device__ unsigned long long g_icp_evals = 0ull;

unsigned long long icp_evals_read_and_maybe_reset(bool reset) {
  unsigned long long v = 0ull;
  cudaMemcpyFromSymbol(&v, g_icp_evals, sizeof(v));
  if (reset) {
    const unsigned long long z = 0ull;
    cudaMemcpyToSymbol(g_icp_evals, &z, sizeof(z));
  }
  return v;
}

__global__ void __launch_bounds__(32 * ICP_WARPS)
k_icp_closest(const IcpPair* __restrict__ pairs, int P, const int* __restrict__ off_lm, const int* __restrict__ off_grp,
              const int* __restrict__ off_tri, const int* __restrict__ off_tile, int group, int n_groups,
              const double* __restrict__ box,
              const double* __restrict__ tv, const int* __restrict__ tid, const double* __restrict__ tile_lo,
              const double* __restrict__ tile_hi, const unsigned* __restrict__ tile_key, const int* __restrict__ perm,
              const double* __restrict__ a, int have_prev, int* __restrict__ winner, double* __restrict__ closest) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int g = blockIdx.x * ICP_WARPS + (threadIdx.x >> 5);
  if (g >= n_groups) return;  // the whole warp
  int p = 0;
  {  // the pair of this group: every pair has at least one group
    int hi = P - 1;
    while (p < hi) {
      const int mid = (p + hi + 1) >> 1;
      if (off_grp[mid] <= g)
        p = mid;
      else
        hi = mid - 1;
    }
  }
  const IcpPair pr = pairs[p];
  const int lm0 = off_lm[p], s0 = off_tri[p], t0 = off_tile[p], ntiles = off_tile[p + 1] - t0;
  const double* fbox = box + ICP_BOX * (2 * (size_t)p);
  const double pad = fbox[6];
  const int slot = (g - off_grp[p]) * group + lane;
  const bool valid = lane < group && slot < pr.nb;
  const int li = lm0 + (valid ? perm[lm0 + slot] : 0);
  const P3 q = p3(a, li);
  // Seed of the bound (squared): the previous winner, or the best triangle of the landmark's home tile (the tile whose
  // Morton range holds the landmark).  It is a bound only: those triangles are met again in the scan below.
  double bound = INFINITY;
  int best_pos = s0;
  if (valid) {
    if (have_prev) {
      best_pos = winner[li];
      const double* v = tv + 9 * (size_t)best_pos;
      const P3 d = q - closest_on_triangle(q, P3{v[0], v[1], v[2]}, P3{v[3], v[4], v[5]}, P3{v[6], v[7], v[8]});
      bound = dot3(d, d);
    } else {
      const double qa[3] = {q.x, q.y, q.z};
      const unsigned key = morton3(qa, 3, fbox, fbox + 3);
      int lo = 0, hi = ntiles - 1;
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (tile_key[t0 + mid] <= key)
          lo = mid;
        else
          hi = mid - 1;
      }
      const int r0 = s0 + lo * ICP_TILE, r1 = s0 + min(pr.fnt, (lo + 1) * ICP_TILE);
      best_pos = r0;
      for (int r = r0; r < r1; ++r) {
        const double* v = tv + 9 * (size_t)r;
        const P3 d = q - closest_on_triangle(q, P3{v[0], v[1], v[2]}, P3{v[3], v[4], v[5]}, P3{v[6], v[7], v[8]});
        bound = fmin(bound, dot3(d, d));
      }
    }
  }
  // bounding box of the group's landmarks
  double glo[3] = {valid ? q.x : INFINITY, valid ? q.y : INFINITY, valid ? q.z : INFINITY};
  double ghi[3] = {valid ? q.x : -INFINITY, valid ? q.y : -INFINITY, valid ? q.z : -INFINITY};
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      glo[c] = fmin(glo[c], __shfl_xor_sync(full, glo[c], o));
      ghi[c] = fmax(ghi[c], __shfl_xor_sync(full, ghi[c], o));
    }
  double best = INFINITY;
  int best_id = INT_MAX;
  unsigned n_eval = 0;
  // Tiles are walked in chunks of 32, lane k holding the box of tile c0 + k; the next chunk's boxes are loaded while
  // this one is walked.
  double blo[3] = {INFINITY, INFINITY, INFINITY}, bhi[3] = {-INFINITY, -INFINITY, -INFINITY};
  if (lane < ntiles)
    for (int c = 0; c < 3; ++c) {
      blo[c] = tile_lo[3 * (size_t)(t0 + lane) + c];
      bhi[c] = tile_hi[3 * (size_t)(t0 + lane) + c];
    }
  for (int c0 = 0; c0 < ntiles; c0 += 32) {
    double nlo[3] = {INFINITY, INFINITY, INFINITY}, nhi[3] = {-INFINITY, -INFINITY, -INFINITY};
    if (c0 + 32 + lane < ntiles)
      for (int c = 0; c < 3; ++c) {
        nlo[c] = tile_lo[3 * (size_t)(t0 + c0 + 32 + lane) + c];
        nhi[c] = tile_hi[3 * (size_t)(t0 + c0 + 32 + lane) + c];
      }
    // A tile can matter to the group only if its box lies within the largest bound of the group (the distance between
    // the tile's box and the group's box is a lower bound of every landmark's distance to the tile's triangles).
    double rmax = valid ? fmin(bound, best) : -INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rmax = fmax(rmax, __shfl_xor_sync(full, rmax, o));
    bool flag = false;
    if (c0 + lane < ntiles) {
      double s = 0.0;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const double gg = fmax(fmax(blo[c] - ghi[c], glo[c] - bhi[c]), 0.0);
        s += gg * gg;
      }
      flag = s * (1.0 - 1e-12) <= rmax;
    }
    unsigned mask = __ballot_sync(full, flag);
    while (mask) {  // uniform over the warp
      const int k = __ffs(mask) - 1, j = c0 + k;
      mask &= mask - 1;
      double tl[3], th[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        tl[c] = __shfl_sync(full, blo[c], k);
        th[c] = __shfl_sync(full, bhi[c], k);
      }
      const bool need = valid && box_lb(q, tl, th) <= fmin(bound, best);
      const unsigned need_mask = __ballot_sync(full, need);
      if (!need_mask) continue;
      // lane r holds triangle r of the tile (one coalesced load); the warp evaluates the landmarks that need the tile one
      // after the other, each against all its triangles at once, and reduces (d^2, original index) to that landmark
      const int rt = s0 + j * ICP_TILE, cnt = min(ICP_TILE, pr.fnt - j * ICP_TILE);
      for (int sl = 0; sl < cnt; sl += 32) {  // slices of 32 triangles
        const int r0 = rt + sl;
        const bool have = sl + lane < cnt;
        P3 A{0, 0, 0}, B{0, 0, 0}, C{0, 0, 0};
        int id = INT_MAX;
        if (have) {
          const double* v = tv + 9 * (size_t)(r0 + lane);
          A = P3{v[0], v[1], v[2]}, B = P3{v[3], v[4], v[5]}, C = P3{v[6], v[7], v[8]};
          id = tid[r0 + lane];
        }
        const double lo[3] = {fmin(A.x, fmin(B.x, C.x)) - pad, fmin(A.y, fmin(B.y, C.y)) - pad, fmin(A.z, fmin(B.z, C.z)) - pad};
        const double hi[3] = {fmax(A.x, fmax(B.x, C.x)) + pad, fmax(A.y, fmax(B.y, C.y)) + pad, fmax(A.z, fmax(B.z, C.z)) + pad};
        unsigned nmask = need_mask;
        while (nmask) {
          const int l = __ffs(nmask) - 1;
          nmask &= nmask - 1;
          const P3 ql{__shfl_sync(full, q.x, l), __shfl_sync(full, q.y, l), __shfl_sync(full, q.z, l)};
          const double lim = __shfl_sync(full, fmin(bound, best), l);
          double d2 = INFINITY;
          int did = INT_MAX, dr = lane;
          if (have && !(box_lb(ql, lo, hi) > lim)) {  // strictly beyond: cannot attain the minimum
            ++n_eval;
            const P3 d = ql - closest_on_triangle(ql, A, B, C);
            d2 = dot3(d, d);
            did = id;
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            const double od = __shfl_xor_sync(full, d2, o);
            const int oi = __shfl_xor_sync(full, did, o), orr = __shfl_xor_sync(full, dr, o);
            if (od < d2 || (od == d2 && oi < did)) {
              d2 = od;
              did = oi;
              dr = orr;
            }
          }
          if (lane == l && (d2 < best || (d2 == best && did < best_id))) {
            best = d2;
            best_id = did;
            best_pos = r0 + dr;
          }
        }
      }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      blo[c] = nlo[c];
      bhi[c] = nhi[c];
    }
  }
#ifdef FB_ICP_COUNT
  {
    unsigned tot = n_eval;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(full, tot, o);
    if (lane == 0 && tot) atomicAdd(&g_icp_evals, (unsigned long long)tot);
  }
#else
  (void)n_eval;
#endif
  if (valid) {
    const double* v = tv + 9 * (size_t)best_pos;
    const P3 c = closest_on_triangle(q, P3{v[0], v[1], v[2]}, P3{v[3], v[4], v[5]}, P3{v[6], v[7], v[8]});
    closest[3 * (size_t)li] = c.x;
    closest[3 * (size_t)li + 1] = c.y;
    closest[3 * (size_t)li + 2] = c.z;
    winner[li] = best_pos;
  }
}

// vtkLandmarkTransform (rigid body / similarity) of a -> b, then acc <- L * acc; one CTA per pair
__global__ void __launch_bounds__(FIT_THREADS) k_icp_fit(const int* __restrict__ off_lm, const double* __restrict__ a_all,
                                                        const double* __restrict__ b_all, int similarity, double* __restrict__ L_all,
                                                        double* __restrict__ acc_all) {
  __shared__ double red[FIT_THREADS];
  const int l0 = off_lm[blockIdx.x], nb = off_lm[blockIdx.x + 1] - l0;
  double* L = L_all + 16 * (size_t)blockIdx.x;
  double* acc = acc_all + 16 * (size_t)blockIdx.x;
  double Lm[16];
  if (!landmark_fit_block(a_all + 3 * (size_t)l0, b_all + 3 * (size_t)l0, nb, similarity, red, Lm)) return;
  double old[16], nw[16];
  for (int i = 0; i < 16; ++i) old[i] = acc[i];
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) {
      double v = 0.0;
      for (int k = 0; k < 4; ++k) v += Lm[4 * r + k] * old[4 * k + c];
      nw[4 * r + c] = v;
    }
  for (int i = 0; i < 16; ++i) {
    acc[i] = nw[i];
    L[i] = Lm[i];
  }
}

// landmarks <- L landmarks, per pair
__global__ void k_icp_move(const int* __restrict__ off_lm, const double* __restrict__ L_all, double* __restrict__ a_all) {
  const int p = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  const int l0 = off_lm[p];
  if (i >= off_lm[p + 1] - l0) return;
  double* a = a_all + 3 * (size_t)l0;
  const P3 q = xform(L_all + 16 * (size_t)p, p3(a, i));
  a[3 * (size_t)i] = q.x;
  a[3 * (size_t)i + 1] = q.y;
  a[3 * (size_t)i + 2] = q.z;
}

// out rows of every moving mesh = acc * moving points
__global__ void k_icp_apply(const IcpPair* __restrict__ pairs, const double* __restrict__ moving_pts,
                            const double* __restrict__ acc_all, double* __restrict__ out) {
  const int p = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  const IcpPair pr = pairs[p];
  if (i >= pr.mnp) return;
  const size_t r = (size_t)pr.mp0 + i;
  const P3 q = xform(acc_all + 16 * (size_t)p, p3(moving_pts, (long long)r));
  out[3 * r] = q.x;
  out[3 * r + 1] = q.y;
  out[3 * r + 2] = q.z;
}

// sizes of one call, from the host copies
struct IcpSizes {
  int P = 0;
  long long n_tris = 0, n_lm = 0, n_tiles = 0, n_groups[4] = {0, 0, 0, 0};  // groups for each of ICP_GROUPS
  int max_fnt = 0, max_nb = 0, max_mnp = 0, max_tiles = 0;
};

struct IcpWs {
  IcpPair* pairs;
  int *off_lm, *off_grp, *off_tri, *off_tile, *sort_begin, *sort_end;
  unsigned long long *keys_in, *keys_out;
  void* sort_tmp;
  size_t sort_tmp_bytes;
  double *box, *tv, *tile_lo, *tile_hi, *mats, *a, *cl;
  int *tid, *perm, *winner;
  unsigned* tile_key;
};

static size_t icp_sort_tmp_bytes(const IcpSizes& s) {
  size_t bytes = 0;
  cub::DeviceSegmentedRadixSort::SortKeys(nullptr, bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                          (int)(s.n_tris + s.n_lm), 2 * s.P, (const int*)nullptr, (const int*)nullptr,
                                          ICP_SORT_BITS[0], ICP_SORT_BITS[1]);
  return bytes;
}

static IcpWs icp_carve(Carver& cv, const IcpSizes& s) {
  IcpWs w;
  const size_t P = (size_t)s.P, items = (size_t)(s.n_tris + s.n_lm);
  w.pairs = cv.take<IcpPair>(P);
  w.off_lm = cv.take<int>(P + 1);
  w.off_grp = cv.take<int>(P + 1);
  w.off_tri = cv.take<int>(P + 1);
  w.off_tile = cv.take<int>(P + 1);
  w.sort_begin = cv.take<int>(2 * P);
  w.sort_end = cv.take<int>(2 * P);
  w.keys_in = cv.take<unsigned long long>(items);
  w.keys_out = cv.take<unsigned long long>(items);
  w.sort_tmp_bytes = icp_sort_tmp_bytes(s);
  w.sort_tmp = cv.take<char>(w.sort_tmp_bytes);
  w.box = cv.take<double>(2 * ICP_BOX * P);
  w.tv = cv.take<double>(9 * (size_t)s.n_tris);
  w.tid = cv.take<int>((size_t)s.n_tris);
  w.tile_lo = cv.take<double>(3 * (size_t)s.n_tiles);
  w.tile_hi = cv.take<double>(3 * (size_t)s.n_tiles);
  w.tile_key = cv.take<unsigned>((size_t)s.n_tiles);
  w.mats = cv.take<double>(32 * P);  // acc[P][16], L[P][16]
  w.perm = cv.take<int>((size_t)s.n_lm);
  w.a = cv.take<double>(3 * (size_t)s.n_lm);
  w.cl = cv.take<double>(3 * (size_t)s.n_lm);
  w.winner = cv.take<int>((size_t)s.n_lm);
  return w;
}

static size_t icp_bytes(const IcpSizes& s) {
  Carver cv(nullptr, 0);
  icp_carve(cv, s);
  return cv.used + 256;
}

static void icp_add_pair(IcpSizes& s, int fnt, int mnp, int max_landmarks) {
  const int step = mnp > max_landmarks ? mnp / max_landmarks : 1, nb = mnp / step;
  const int tiles = (fnt + ICP_TILE - 1) / ICP_TILE;
  s.P += 1;
  s.n_tris += fnt;
  s.n_lm += nb;
  s.n_tiles += tiles;
  for (int k = 0; k < 4; ++k) s.n_groups[k] += (nb + ICP_GROUPS[k] - 1) / ICP_GROUPS[k];
  s.max_fnt = std::max(s.max_fnt, fnt);
  s.max_nb = std::max(s.max_nb, nb);
  s.max_mnp = std::max(s.max_mnp, mnp);
  s.max_tiles = std::max(s.max_tiles, tiles);
}

// the batch's sizes; a message in *why when the description is not valid
static bool icp_batch_sizes(const int* mesh_off_host, const int* tri_off_host, int n_meshes, const int* fixed_host,
                            const int* moving_host, int n_pairs, int max_landmarks, IcpSizes& s, const char** why) {
  *why = nullptr;
  if (!mesh_off_host || !tri_off_host || !fixed_host || !moving_host || n_meshes <= 0 || n_pairs <= 0 || max_landmarks <= 0) {
    *why = "icp_batch: empty batch, missing host offsets or bad landmark count";
    return false;
  }
  if (n_pairs > 65535) {  // the pair is the grid's y index of the per-pair launches
    *why = "icp_batch: at most 65535 pairs per call";
    return false;
  }
  std::vector<char> moving_seen(n_meshes, 0);
  for (int p = 0; p < n_pairs; ++p) {
    const int f = fixed_host[p], m = moving_host[p];
    if (f < 0 || f >= n_meshes || m < 0 || m >= n_meshes) {
      *why = "icp_batch: mesh index out of range";
      return false;
    }
    if (moving_seen[m]) {
      *why = "icp_batch: a mesh is the moving mesh of more than one pair";
      return false;
    }
    moving_seen[m] = 1;
    const int fnt = tri_off_host[f + 1] - tri_off_host[f];
    const int fnp = mesh_off_host[f + 1] - mesh_off_host[f], mnp = mesh_off_host[m + 1] - mesh_off_host[m];
    if (fnt <= 0) {
      *why = "icp_batch: a fixed mesh has no triangles";
      return false;
    }
    if (fnp <= 0 || mnp <= 0) {
      *why = "icp_batch: empty mesh";
      return false;
    }
    icp_add_pair(s, fnt, mnp, max_landmarks);
  }
  return true;
}

// the whole registration of every pair; descriptions either from the batch arrays or (mesh_off == nullptr) one pair
static int icp_run(const IcpSizes& s, void* workspace, size_t workspace_bytes, const double* fixed_pts, const int* tris,
                   const double* moving_pts, const int* mesh_off, const int* tri_off, const int* fixed_mesh,
                   const int* moving_mesh, int one_fnp, int one_fnt, int one_mnp, int max_landmarks, int max_iterations,
                   int similarity, int match, double* matrices, double* moved, cudaStream_t stream) {
  Carver cv(workspace, workspace_bytes);
  IcpWs w = icp_carve(cv, s);
  if (!cv.ok()) {
    set_error("icp: workspace too small (%zu < %zu)", workspace_bytes, cv.used);
    return FB_ERR_WORKSPACE;
  }
  const int P = s.P, n_sorted_tris = (int)s.n_tris;
  int gk = 0;  // the largest group that still gives about 8 warps per SM, else the smallest
  while (gk < 3 && s.n_groups[gk] < 8LL * sm_count()) ++gk;
  const int group = ICP_GROUPS[gk], n_groups = (int)s.n_groups[gk];
  double *acc = w.mats, *L = w.mats + 16 * (size_t)P;
  k_icp_plan<<<1, 1024, 0, stream>>>(mesh_off, tri_off, fixed_mesh, moving_mesh, P, one_fnp, one_fnt, one_mnp, max_landmarks,
                                     group, n_sorted_tris, w.pairs, w.off_lm, w.off_grp, w.off_tri, w.off_tile, w.sort_begin,
                                     w.sort_end);
  k_icp_start<<<P, 1024, 0, stream>>>(w.pairs, fixed_pts, moving_pts, match, acc);
  k_icp_bbox<<<dim3(P, 2), 256, 0, stream>>>(w.pairs, fixed_pts, moving_pts, w.box);
  const dim3 g_items(div_up(std::max(s.max_fnt, s.max_nb), 256), P);
  k_icp_keys<<<g_items, 256, 0, stream>>>(w.pairs, w.off_lm, w.off_tri, fixed_pts, tris, moving_pts, w.box, n_sorted_tris, w.keys_in);
  FB_COUNT_LAUNCH(5);
  size_t tmp = w.sort_tmp_bytes;
  FB_CUDA(cub::DeviceSegmentedRadixSort::SortKeys(w.sort_tmp, tmp, (const unsigned long long*)w.keys_in, w.keys_out,
                                                  (int)(s.n_tris + s.n_lm), 2 * P, (const int*)w.sort_begin,
                                                  (const int*)w.sort_end, ICP_SORT_BITS[0], ICP_SORT_BITS[1], stream));
  k_icp_fill<<<g_items, 256, 0, stream>>>(w.pairs, w.off_lm, w.off_tri, fixed_pts, tris, w.keys_out, n_sorted_tris, w.tv,
                                          w.tid, w.perm);
  k_icp_tile_boxes<<<dim3(div_up(s.max_tiles, 128), P), 128, 0, stream>>>(w.pairs, w.off_tri, w.off_tile, w.box, w.tv,
                                                                          w.keys_out, w.tile_lo, w.tile_hi, w.tile_key);
  const dim3 g_lm(div_up(s.max_nb, 256), P);
  k_icp_init_landmarks<<<g_lm, 256, 0, stream>>>(w.pairs, w.off_lm, moving_pts, acc, w.a);
  FB_COUNT_LAUNCH(3);
  for (int it = 0; it < max_iterations; ++it) {
    k_icp_closest<<<div_up(n_groups, ICP_WARPS), 32 * ICP_WARPS, 0, stream>>>(
        w.pairs, P, w.off_lm, w.off_grp, w.off_tri, w.off_tile, group, n_groups, w.box, w.tv, w.tid, w.tile_lo, w.tile_hi,
        w.tile_key, w.perm, w.a, it > 0 ? 1 : 0, w.winner, w.cl);
    k_icp_fit<<<P, FIT_THREADS, 0, stream>>>(w.off_lm, w.a, w.cl, similarity ? 1 : 0, L, acc);
    FB_COUNT_LAUNCH(2);
    if (it + 1 >= max_iterations) break;
    k_icp_move<<<g_lm, 256, 0, stream>>>(w.off_lm, L, w.a);
    FB_COUNT_LAUNCH(1);
  }
  if (matrices) FB_CUDA(cudaMemcpyAsync(matrices, acc, sizeof(double) * 16 * (size_t)P, cudaMemcpyDeviceToDevice, stream));
  if (moved) {
    k_icp_apply<<<dim3(div_up(s.max_mnp, 256), P), 256, 0, stream>>>(w.pairs, moving_pts, acc, moved);
    FB_COUNT_LAUNCH(1);
  }
  FB_LAUNCH_CHECK();
  return FB_OK;
}

}  // namespace fb

using namespace fb;

extern "C" {

size_t focusr_icp_workspace_bytes(int n_source_points, int n_target_tris) {
  if (n_source_points <= 0 || n_target_tris <= 0) return 0;
  IcpSizes s;
  icp_add_pair(s, n_target_tris, n_source_points, n_source_points);  // at most every source point is a landmark
  return icp_bytes(s);
}

int focusr_icp(const double* target_points, int n_target_points, const int* target_tris, int n_target_tris,
               const double* source_points, int n_source_points, int max_landmarks, int max_iterations, int similarity,
               int start_by_matching_centroids, double* matrix_out, double* transformed_out, void* workspace,
               size_t workspace_bytes, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_target_points > 0 && n_target_tris > 0 && n_source_points > 0, "icp: empty mesh");
  FB_REQUIRE(max_landmarks > 0 && max_iterations >= 0, "icp: bad iteration or landmark count");
  const size_t need = focusr_icp_workspace_bytes(n_source_points, n_target_tris);
  if (need > workspace_bytes) {
    set_error("icp: workspace too small (%zu < %zu)", workspace_bytes, need);
    return FB_ERR_WORKSPACE;
  }
  // focusr_icp_workspace_bytes sized the workspace for every source point as a landmark; the call needs at most that
  IcpSizes s;
  icp_add_pair(s, n_target_tris, n_source_points, max_landmarks);
  return icp_run(s, workspace, workspace_bytes, target_points, target_tris, source_points, nullptr, nullptr, nullptr,
                 nullptr, n_target_points, n_target_tris, n_source_points, max_landmarks, max_iterations, similarity,
                 start_by_matching_centroids, matrix_out, transformed_out, stream);
}

size_t focusr_icp_batch_workspace_bytes(const int* mesh_off_host, const int* tri_off_host, int n_meshes,
                                        const int* fixed_mesh_host, const int* moving_mesh_host, int n_pairs,
                                        int max_landmarks) {
  IcpSizes s;
  const char* why;
  if (!icp_batch_sizes(mesh_off_host, tri_off_host, n_meshes, fixed_mesh_host, moving_mesh_host, n_pairs, max_landmarks, s, &why))
    return 0;
  return icp_bytes(s);
}

int focusr_icp_batch(const double* points, int n_points, const int* tris, const int* mesh_off, const int* mesh_off_host,
                     const int* tri_off, const int* tri_off_host, int n_meshes, const int* fixed_mesh,
                     const int* moving_mesh, const int* fixed_mesh_host, const int* moving_mesh_host, int n_pairs,
                     int max_landmarks, int max_iterations, int similarity, int start_by_matching_centroids,
                     double* matrices, double* moved_points, void* workspace, size_t workspace_bytes,
                     focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(max_iterations >= 0, "icp_batch: bad iteration count");
  FB_REQUIRE(points && tris && mesh_off && tri_off && fixed_mesh && moving_mesh, "icp_batch: missing device array");
  FB_REQUIRE(moved_points == nullptr || moved_points != points, "icp_batch: moved_points must not alias points");
  IcpSizes s;
  const char* why;
  if (!icp_batch_sizes(mesh_off_host, tri_off_host, n_meshes, fixed_mesh_host, moving_mesh_host, n_pairs, max_landmarks, s, &why)) {
    set_error("%s", why);
    return FB_ERR_ARG;
  }
  FB_REQUIRE(mesh_off_host[n_meshes] <= n_points, "icp_batch: mesh offsets exceed n_points");
  const size_t need = icp_bytes(s);
  if (need > workspace_bytes) {
    set_error("icp_batch: workspace too small (%zu < %zu)", workspace_bytes, need);
    return FB_ERR_WORKSPACE;
  }
  // rows of meshes that do not move are copied unchanged; the moving meshes' rows are overwritten below
  if (moved_points) FB_CUDA(cudaMemcpyAsync(moved_points, points, sizeof(double) * 3 * (size_t)n_points, cudaMemcpyDeviceToDevice, stream));
  return icp_run(s, workspace, workspace_bytes, points, tris, points, mesh_off, tri_off, fixed_mesh, moving_mesh, 0, 0, 0,
                 max_landmarks, max_iterations, similarity, start_by_matching_centroids, matrices, moved_points, stream);
}

}  // extern "C"
