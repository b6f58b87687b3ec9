// K14  Closest points on triangle surfaces, for whole meshes of queries at once: the surface distances that say how well
// a registered source fits its target (and the target its source), per vertex and, per pair, as means, ASSD and
// Hausdorff distance.  The reference has no such measure in use (its test.py get_all_pairwise_surface_errors is dead
// code, SURVEY.md section 2).
//
// Surfaces use the batch layout (triangles with global vertex ids into one point array; surface m = points
// surf_point_off[m] .. [m+1], triangles surf_tri_off[m] .. [m+1]); query segment s is searched against surface
// surf_of_segment[s], so a surface may serve several segments, one or none.  The winner of a query is the lexicographic
// minimum of (d^2, local triangle index) over every triangle of its surface, each scored by Ericson's region test
// (closest_point.cuh, the arithmetic of ICP's search) with the edge rule for collapsed triangles.
//
// Brute force (no workspace): one thread per query scans its surface's triangles in index order.
// Pruned (with a workspace), the search of ICP's k_icp_closest for whole meshes of queries:
//   k_sf_plan       one CTA: which surfaces are mapped, their tiles and the segments' query groups (prefix sums), and
//                   the segments of the one sort (every mapped surface's triangles, then every segment's queries).
//   k_sf_bbox       per mapped surface: its points' box (the Morton frame) and the padding of its tile boxes.
//   k_sf_keys       Morton code (in the surface's box) of every mapped triangle's centroid and of every query; one CUB
//                   segmented radix sort orders both without reading a size back to the host.
//   k_sf_fill / k_sf_tile_boxes  sorted triangles stored as 9 contiguous coordinates with their local index, cut into
//                   tiles of 32 with a padded box each; the queries' sorted order = groups of up to 32 per warp.
//   k_sf_closest    one warp per group: the bound of each query starts from the best triangle of its home tile (the tile
//                   whose Morton range holds the query); the warp visits only the tiles whose box lies within the largest
//                   bound of its group and evaluates a triangle unless its padded box is STRICTLY beyond the query's best
//                   distance known.  Every triangle that can attain the minimum is evaluated, so the result is bit for
//                   bit that of the brute force, whatever the tiling, grouping or batch.
// Each mapped surface is sorted and tiled once per call, whatever number of segments it serves.
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

constexpr int SF_TILE = 32;                     // triangles per tile: lane r of a warp holds triangle r of a tile
constexpr int SF_GROUPS[4] = {32, 16, 8, 4};    // queries per warp: the largest that gives about 8 warps per SM
constexpr int SF_WARPS = 4;                     // groups per CTA of k_sf_closest
constexpr int SF_SORT_BITS[2] = {32, 62};       // keys = Morton << 32 | local index, written in index order
constexpr int SF_BOX = 8;                       // doubles per surface box record: lo[3], 1024 / extent[3], pad, 0
constexpr int SF_STATS_THREADS = 256;

// the last m in [0, n) with off[m] <= i (off non-decreasing, off[0] <= i): the segment of item i, empty ones skipped
__device__ __forceinline__ int seg_of(const int* __restrict__ off, int n, long long i) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (off[mid] <= i)
      lo = mid;
    else
      hi = mid - 1;
  }
  return lo;
}

// exclusive prefix sum out[0..n] of value(i), i < n, by one 1024-thread CTA in chunks with a carry
template <class F>
__device__ void block_scan_1024(int n, F value, int* __restrict__ out, int* s, int* carry) {
  const int t = threadIdx.x;
  if (t == 0) *carry = 0;
  for (int c0 = 0; c0 < n; c0 += 1024) {
    const int v = c0 + t < n ? value(c0 + t) : 0;
    __syncthreads();
    s[t] = v;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {  // inclusive scan
      const int x = t >= d ? s[t - d] : 0;
      __syncthreads();
      s[t] += x;
      __syncthreads();
    }
    if (c0 + t < n) out[c0 + t] = *carry + s[t] - v;
    __syncthreads();
    if (t == 0) *carry += s[1023];
  }
  __syncthreads();
  if (t == 0) out[n] = *carry;
}

__global__ void __launch_bounds__(1024)
k_sf_plan(const int* __restrict__ tri_off, int n_surf, const int* __restrict__ query_off, int n_seg,
          const int* __restrict__ surf_of_seg, int group, int t0, int q0, int n_tris, int* __restrict__ used,
          int* __restrict__ off_tile, int* __restrict__ off_grp, int* __restrict__ sort_begin, int* __restrict__ sort_end) {
  __shared__ int s[1024];
  __shared__ int carry;
  for (int m = threadIdx.x; m < n_surf; m += 1024) used[m] = 0;
  __syncthreads();
  for (int k = threadIdx.x; k < n_seg; k += 1024) used[surf_of_seg[k]] = 1;  // same value from every writer
  __syncthreads();
  for (int m = threadIdx.x; m < n_surf; m += 1024) {  // a surface no segment maps is neither sorted nor tiled
    sort_begin[m] = tri_off[m] - t0;
    sort_end[m] = (used[m] ? tri_off[m + 1] : tri_off[m]) - t0;
  }
  for (int k = threadIdx.x; k < n_seg; k += 1024) {
    sort_begin[n_surf + k] = n_tris + query_off[k] - q0;
    sort_end[n_surf + k] = n_tris + query_off[k + 1] - q0;
  }
  block_scan_1024(n_surf, [&](int m) { return used[m] ? (tri_off[m + 1] - tri_off[m] + SF_TILE - 1) / SF_TILE : 0; },
                  off_tile, s, &carry);
  block_scan_1024(n_seg, [&](int k) { return (query_off[k + 1] - query_off[k] + group - 1) / group; }, off_grp, s, &carry);
}

// one CTA per surface: the box of its points (Morton frame) and the padding of its tile and triangle boxes
__global__ void __launch_bounds__(256) k_sf_bbox(const int* __restrict__ used, const double* __restrict__ pts,
                                                const int* __restrict__ point_off, double* __restrict__ box) {
  const int m = blockIdx.x;
  if (!used[m]) return;
  const int p0 = point_off[m], n = point_off[m + 1] - p0;
  double mn[3] = {1e300, 1e300, 1e300}, mx[3] = {-1e300, -1e300, -1e300};
  for (int i = threadIdx.x; i < n; i += 256)
    for (int c = 0; c < 3; ++c) {
      const double v = pts[3 * ((size_t)p0 + i) + c];
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
    double* b = box + SF_BOX * (size_t)m;
    double mag = 0.0;
    for (int c = 0; c < 3; ++c) {
      const double ext = smx[c][0] - smn[c][0];
      b[c] = smn[c][0];
      b[3 + c] = (ext > 0.0 && ext < 1e300) ? 1024.0 / ext : 0.0;
      mag = fmax(mag, fmax(fabs(smn[c][0]), fabs(smx[c][0])) + ext);
    }
    // as in ICP: far more than the rounding error of a computed closest point, far less than a pruning distance
    b[6] = 1e-9 * mag;
    b[7] = 0.0;
  }
}

// keys (Morton << 32 | local index) of every mapped triangle's centroid, then of every query, in its surface's box
__global__ void __launch_bounds__(256)
k_sf_keys(const int* __restrict__ used, const double* __restrict__ pts, const int* __restrict__ tris,
          const int* __restrict__ tri_off, int n_surf, const double* __restrict__ queries, const int* __restrict__ query_off,
          int n_seg, const int* __restrict__ surf_of_seg, const double* __restrict__ box, int t0, int q0, int n_tris,
          int n_items, unsigned long long* __restrict__ keys) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_items) return;
  if (i < n_tris) {
    const int m = seg_of(tri_off, n_surf, (long long)t0 + i);
    if (!used[m]) return;
    const int* tr = tris + 3 * ((size_t)t0 + i);
    const P3 c = (p3(pts, tr[0]) + p3(pts, tr[1]) + p3(pts, tr[2])) * (1.0 / 3.0);
    const double q[3] = {c.x, c.y, c.z};
    const double* b = box + SF_BOX * (size_t)m;
    keys[i] = ((unsigned long long)morton3(q, 3, b, b + 3) << 32) | (unsigned)(t0 + i - tri_off[m]);
  } else {
    const int j = q0 + i - n_tris, s = seg_of(query_off, n_seg, j);
    const double* b = box + SF_BOX * (size_t)surf_of_seg[s];
    keys[i] = ((unsigned long long)morton3(queries + 3 * (size_t)j, 3, b, b + 3) << 32) | (unsigned)(j - query_off[s]);
  }
}

// sorted triangles -> contiguous vertex coordinates + local index; sorted queries -> their local index in group order
__global__ void __launch_bounds__(256)
k_sf_fill(const int* __restrict__ used, const double* __restrict__ pts, const int* __restrict__ tris,
          const int* __restrict__ tri_off, int n_surf, const unsigned long long* __restrict__ keys, int t0, int n_tris,
          int n_items, double* __restrict__ tv, int* __restrict__ tid, int* __restrict__ perm) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_items) return;
  const int local = (int)(keys[i] & 0xffffffffu);
  if (i >= n_tris) {
    perm[i - n_tris] = local;
    return;
  }
  const int m = seg_of(tri_off, n_surf, (long long)t0 + i);
  if (!used[m]) return;
  const int* tr = tris + 3 * ((size_t)tri_off[m] + local);
  for (int v = 0; v < 3; ++v)
    for (int c = 0; c < 3; ++c) tv[9 * (size_t)i + 3 * v + c] = pts[3 * (size_t)tr[v] + c];
  tid[i] = local;
}

__global__ void __launch_bounds__(128)
k_sf_tile_boxes(const int* __restrict__ tri_off, const int* __restrict__ off_tile, int n_surf, int n_tiles, int t0,
                const double* __restrict__ box, const double* __restrict__ tv, const unsigned long long* __restrict__ keys,
                double* __restrict__ tile_lo, double* __restrict__ tile_hi, unsigned* __restrict__ tile_key) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_tiles) return;
  const int m = seg_of(off_tile, n_surf, j), jj = j - off_tile[m];
  const double pad = box[SF_BOX * (size_t)m + 6];
  const size_t s0 = (size_t)(tri_off[m] - t0), r0 = s0 + (size_t)jj * SF_TILE;
  const size_t r1 = s0 + (size_t)min(tri_off[m + 1] - tri_off[m], (jj + 1) * SF_TILE);
  double mn[3] = {1e300, 1e300, 1e300}, mx[3] = {-1e300, -1e300, -1e300};
  for (size_t r = r0; r < r1; ++r)
    for (int v = 0; v < 3; ++v)
      for (int c = 0; c < 3; ++c) {
        const double x = tv[9 * r + 3 * v + c];
        mn[c] = fmin(mn[c], x);
        mx[c] = fmax(mx[c], x);
      }
  for (int c = 0; c < 3; ++c) {
    tile_lo[3 * (size_t)j + c] = mn[c] - pad;
    tile_hi[3 * (size_t)j + c] = mx[c] + pad;
  }
  tile_key[j] = (unsigned)(keys[r0] >> 32);
}

// (query, triangle) closest-point evaluations of k_sf_closest since the last reset, the home-tile seed included; counted
// only in builds with -DFB_SURFACE_COUNT (tools/surface_distance_bench.py), read through focusr_profile_get_kind(6, ...)
__device__ unsigned long long g_surface_evals = 0ull;

unsigned long long surface_evals_read_and_maybe_reset(bool reset) {
  unsigned long long v = 0ull;
  cudaMemcpyFromSymbol(&v, g_surface_evals, sizeof(v));
  if (reset) {
    const unsigned long long z = 0ull;
    cudaMemcpyToSymbol(g_surface_evals, &z, sizeof(z));
  }
  return v;
}

// the outputs of query qi from the winning triangle: the closest point recomputed from it (the same arithmetic that
// scored it), its local index and the distance
__device__ __forceinline__ void sf_write(P3 q, P3 a, P3 b, P3 c, int tri, long long qi, double* __restrict__ closest_out,
                                         int* __restrict__ tri_out, double* __restrict__ dist_out) {
  const P3 cl = closest_on_triangle_t<true>(q, a, b, c);
  const P3 d = q - cl;
  if (closest_out) {
    closest_out[3 * qi] = cl.x;
    closest_out[3 * qi + 1] = cl.y;
    closest_out[3 * qi + 2] = cl.z;
  }
  if (tri_out) tri_out[qi] = tri;
  if (dist_out) dist_out[qi] = sqrt(dot3(d, d));
}

__global__ void __launch_bounds__(256)
k_sf_brute(const double* __restrict__ pts, const int* __restrict__ tris, const int* __restrict__ tri_off,
           const double* __restrict__ queries, const int* __restrict__ query_off, int n_seg, const int* __restrict__ surf_of_seg,
           int q0, int n_queries, double* __restrict__ closest_out, int* __restrict__ tri_out, double* __restrict__ dist_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_queries) return;
  const long long qi = (long long)q0 + i;
  const int m = surf_of_seg[seg_of(query_off, n_seg, qi)];
  const P3 q = p3(queries, qi);
  const int f0 = tri_off[m], f1 = tri_off[m + 1];
  double best = INFINITY;
  int win = f0;
  for (int f = f0; f < f1; ++f) {  // index order: a tie keeps the lower index
    const int* tr = tris + 3 * (size_t)f;
    const P3 d = q - closest_on_triangle_t<true>(q, p3(pts, tr[0]), p3(pts, tr[1]), p3(pts, tr[2]));
    const double d2 = dot3(d, d);
    if (d2 < best) {
      best = d2;
      win = f;
    }
  }
  const int* tr = tris + 3 * (size_t)win;
  sf_write(q, p3(pts, tr[0]), p3(pts, tr[1]), p3(pts, tr[2]), win - f0, qi, closest_out, tri_out, dist_out);
}

__global__ void __launch_bounds__(32 * SF_WARPS)
k_sf_closest(const int* __restrict__ tri_off, const int* __restrict__ query_off, int n_seg,
             const int* __restrict__ surf_of_seg, const int* __restrict__ off_tile, const int* __restrict__ off_grp,
             int group, int n_groups, int t0, int q0, const double* __restrict__ box, const double* __restrict__ tv,
             const int* __restrict__ tid, const double* __restrict__ tile_lo, const double* __restrict__ tile_hi,
             const unsigned* __restrict__ tile_key, const int* __restrict__ perm, const double* __restrict__ queries,
             double* __restrict__ closest_out, int* __restrict__ tri_out, double* __restrict__ dist_out) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int g = blockIdx.x * SF_WARPS + (threadIdx.x >> 5);
  if (g >= n_groups) return;  // the whole warp
  const int s = seg_of(off_grp, n_seg, g), m = surf_of_seg[s];
  const int qs = query_off[s], nq = query_off[s + 1] - qs;
  const int s0 = tri_off[m] - t0, nt = tri_off[m + 1] - tri_off[m];
  const int tt0 = off_tile[m], ntiles = off_tile[m + 1] - tt0;
  const double* sbox = box + SF_BOX * (size_t)m;
  const double pad = sbox[6];
  const int slot = (g - off_grp[s]) * group + lane;
  const bool valid = lane < group && slot < nq;
  const long long qi = (long long)qs + (valid ? perm[qs - q0 + slot] : 0);
  const P3 q = p3(queries, qi);
  unsigned n_eval = 0;
  // Seed of the bound (squared): the best triangle of the query's home tile.  It is a bound only: those triangles are
  // met again in the walk below.
  double bound = INFINITY;
  int best_pos = s0;
  if (valid) {
    const double qa[3] = {q.x, q.y, q.z};
    const unsigned key = morton3(qa, 3, sbox, sbox + 3);
    int lo = 0, hi = ntiles - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (tile_key[tt0 + mid] <= key)
        lo = mid;
      else
        hi = mid - 1;
    }
    const int r0 = s0 + lo * SF_TILE, r1 = s0 + min(nt, (lo + 1) * SF_TILE);
    for (int r = r0; r < r1; ++r) {
      const double* v = tv + 9 * (size_t)r;
      const P3 d = q - closest_on_triangle_t<true>(q, P3{v[0], v[1], v[2]}, P3{v[3], v[4], v[5]}, P3{v[6], v[7], v[8]});
      bound = fmin(bound, dot3(d, d));
    }
    n_eval += r1 - r0;
  }
  // bounding box of the group's queries
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
  // tiles in chunks of 32, lane k holding the box of tile c0 + k; the next chunk's boxes load while this one is walked
  double blo[3] = {INFINITY, INFINITY, INFINITY}, bhi[3] = {-INFINITY, -INFINITY, -INFINITY};
  if (lane < ntiles)
    for (int c = 0; c < 3; ++c) {
      blo[c] = tile_lo[3 * (size_t)(tt0 + lane) + c];
      bhi[c] = tile_hi[3 * (size_t)(tt0 + lane) + c];
    }
  for (int c0 = 0; c0 < ntiles; c0 += 32) {
    double nlo[3] = {INFINITY, INFINITY, INFINITY}, nhi[3] = {-INFINITY, -INFINITY, -INFINITY};
    if (c0 + 32 + lane < ntiles)
      for (int c = 0; c < 3; ++c) {
        nlo[c] = tile_lo[3 * (size_t)(tt0 + c0 + 32 + lane) + c];
        nhi[c] = tile_hi[3 * (size_t)(tt0 + c0 + 32 + lane) + c];
      }
    // a tile can matter to the group only if its box lies within the largest bound of the group
    double rmax = valid ? fmin(bound, best) : -INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rmax = fmax(rmax, __shfl_xor_sync(full, rmax, o));
    bool flag = false;
    if (c0 + lane < ntiles) {
      double sq = 0.0;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const double gg = fmax(fmax(blo[c] - ghi[c], glo[c] - bhi[c]), 0.0);
        sq += gg * gg;
      }
      flag = sq * (1.0 - 1e-12) <= rmax;
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
      // lane r holds triangle r of the tile (one coalesced load); the warp evaluates the queries that need the tile one
      // after the other, each against all its triangles at once, and reduces (d^2, local index) to that query
      const int r0 = s0 + j * SF_TILE, cnt = min(SF_TILE, nt - j * SF_TILE);
      const bool have = lane < cnt;
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
          const P3 d = ql - closest_on_triangle_t<true>(ql, A, B, C);
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
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      blo[c] = nlo[c];
      bhi[c] = nhi[c];
    }
  }
#ifdef FB_SURFACE_COUNT
  {
    unsigned tot = n_eval;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(full, tot, o);
    if (lane == 0 && tot) atomicAdd(&g_surface_evals, (unsigned long long)tot);
  }
#else
  (void)n_eval;
#endif
  if (valid) {
    const double* v = tv + 9 * (size_t)best_pos;
    sf_write(q, P3{v[0], v[1], v[2]}, P3{v[3], v[4], v[5]}, P3{v[6], v[7], v[8]}, tid[best_pos], qi, closest_out, tri_out,
             dist_out);
  }
}

// fixed-tree block maximum (blockDim.x a power of two); every thread gets the result
__device__ __forceinline__ double block_max(double v, double* red) {
  const int t = threadIdx.x;
  __syncthreads();
  red[t] = v;
  __syncthreads();
  for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
    if (t < s) red[t] = fmax(red[t], red[t + s]);
    __syncthreads();
  }
  return red[0];
}

// one CTA per pair: {mean a->b, max a->b, mean b->a, max b->a, ASSD, Hausdorff}
__global__ void __launch_bounds__(SF_STATS_THREADS)
k_sf_stats(const double* __restrict__ a_dist, const int* __restrict__ a_off, const double* __restrict__ b_dist,
           const int* __restrict__ b_off, double* __restrict__ stats) {
  __shared__ double red[SF_STATS_THREADS];
  const int p = blockIdx.x;
  double sum[2], mx[2];
  int n[2];
  for (int side = 0; side < 2; ++side) {
    const double* d = side == 0 ? a_dist : b_dist;
    const int* off = side == 0 ? a_off : b_off;
    const int i0 = off[p];
    n[side] = off[p + 1] - i0;
    double s = 0.0, m = -INFINITY;
    for (int i = threadIdx.x; i < n[side]; i += SF_STATS_THREADS) {
      const double v = d[(size_t)i0 + i];
      s += v;
      m = fmax(m, v);
    }
    sum[side] = fit_block_sum(s, red);
    mx[side] = block_max(m, red);
  }
  if (threadIdx.x == 0) {
    double* o = stats + 6 * (size_t)p;
    o[0] = sum[0] / n[0];
    o[1] = n[0] ? mx[0] : NAN;
    o[2] = sum[1] / n[1];
    o[3] = n[1] ? mx[1] : NAN;
    o[4] = (sum[0] + sum[1]) / (n[0] + n[1]);
    o[5] = (n[0] && n[1]) ? fmax(mx[0], mx[1]) : NAN;
  }
}

// sizes of one call, from the host copies
struct SfSizes {
  int n_surf = 0, n_seg = 0, t0 = 0, q0 = 0;
  long long n_tris = 0, n_queries = 0, n_tiles = 0, n_groups[4] = {0, 0, 0, 0};
};

static bool monotone(const int* off, int n) {
  if (off[0] < 0) return false;
  for (int i = 0; i < n; ++i)
    if (off[i + 1] < off[i]) return false;
  return true;
}

// the call's sizes; a message in *why when the description is not valid
static bool sf_sizes(const int* point_off, const int* tri_off, int n_surf, const int* query_off, int n_seg,
                     const int* surf_of_seg, SfSizes& s, const char** why) {
  *why = nullptr;
  if (!point_off || !tri_off || !query_off || !surf_of_seg || n_surf <= 0 || n_seg <= 0) {
    *why = "closest_points: no surface or no segment, or a missing host array";
    return false;
  }
  if (!monotone(point_off, n_surf) || !monotone(tri_off, n_surf) || !monotone(query_off, n_seg)) {
    *why = "closest_points: point, triangle or query offsets are negative or not monotone";
    return false;
  }
  s.n_surf = n_surf;
  s.n_seg = n_seg;
  s.t0 = tri_off[0];
  s.q0 = query_off[0];
  s.n_tris = (long long)tri_off[n_surf] - tri_off[0];
  s.n_queries = (long long)query_off[n_seg] - query_off[0];
  if (s.n_tris + s.n_queries > INT_MAX) {
    *why = "closest_points: more than 2^31 - 1 triangles and queries in one call";
    return false;
  }
  std::vector<char> mapped(n_surf, 0);
  for (int k = 0; k < n_seg; ++k) {
    const int m = surf_of_seg[k];
    if (m < 0 || m >= n_surf) {
      *why = "closest_points: a segment's surface index is out of range";
      return false;
    }
    if (tri_off[m + 1] == tri_off[m]) {
      *why = "closest_points: a surface that a segment maps to has no triangles";
      return false;
    }
    mapped[m] = 1;
    const long long nq = (long long)query_off[k + 1] - query_off[k];
    for (int g = 0; g < 4; ++g) s.n_groups[g] += (nq + SF_GROUPS[g] - 1) / SF_GROUPS[g];
  }
  for (int m = 0; m < n_surf; ++m)
    if (mapped[m]) s.n_tiles += (tri_off[m + 1] - tri_off[m] + SF_TILE - 1) / SF_TILE;
  return true;
}

struct SfWs {
  int *used, *off_tile, *off_grp, *sort_begin, *sort_end, *tid, *perm;
  unsigned long long *keys_in, *keys_out;
  void* sort_tmp;
  size_t sort_tmp_bytes;
  double *box, *tv, *tile_lo, *tile_hi;
  unsigned* tile_key;
};

static SfWs sf_carve(Carver& cv, const SfSizes& s) {
  SfWs w;
  const size_t items = (size_t)(s.n_tris + s.n_queries);
  w.used = cv.take<int>(s.n_surf);
  w.off_tile = cv.take<int>(s.n_surf + 1);
  w.off_grp = cv.take<int>(s.n_seg + 1);
  w.sort_begin = cv.take<int>(s.n_surf + s.n_seg);
  w.sort_end = cv.take<int>(s.n_surf + s.n_seg);
  w.keys_in = cv.take<unsigned long long>(items);
  w.keys_out = cv.take<unsigned long long>(items);
  w.sort_tmp_bytes = 0;
  cub::DeviceSegmentedRadixSort::SortKeys(nullptr, w.sort_tmp_bytes, (const unsigned long long*)nullptr,
                                          (unsigned long long*)nullptr, (int)items, s.n_surf + s.n_seg, (const int*)nullptr,
                                          (const int*)nullptr, SF_SORT_BITS[0], SF_SORT_BITS[1]);
  w.sort_tmp = cv.take<char>(w.sort_tmp_bytes);
  w.box = cv.take<double>(SF_BOX * (size_t)s.n_surf);
  w.tv = cv.take<double>(9 * (size_t)s.n_tris);
  w.tid = cv.take<int>((size_t)s.n_tris);
  w.tile_lo = cv.take<double>(3 * (size_t)s.n_tiles);
  w.tile_hi = cv.take<double>(3 * (size_t)s.n_tiles);
  w.tile_key = cv.take<unsigned>((size_t)s.n_tiles);
  w.perm = cv.take<int>((size_t)s.n_queries);
  return w;
}

static size_t sf_bytes(const SfSizes& s) {
  Carver cv(nullptr, 0);
  sf_carve(cv, s);
  return cv.used + 256;
}

}  // namespace fb

using namespace fb;

extern "C" {

size_t focusr_closest_points_workspace_bytes(const int* surf_point_off_host, const int* surf_tri_off_host, int n_surfaces,
                                             const int* query_off_host, int n_segments, const int* surf_of_segment_host) {
  SfSizes s;
  const char* why;
  if (!sf_sizes(surf_point_off_host, surf_tri_off_host, n_surfaces, query_off_host, n_segments, surf_of_segment_host, s, &why))
    return 0;
  return sf_bytes(s);
}

int focusr_closest_points(const double* surf_points, const int* tris, const int* surf_point_off, const int* surf_tri_off,
                          const int* surf_point_off_host, const int* surf_tri_off_host, int n_surfaces,
                          const double* queries, const int* query_off, const int* query_off_host, int n_segments,
                          const int* surf_of_segment, const int* surf_of_segment_host, double* closest_out, int* tri_out,
                          double* dist_out, void* workspace, size_t workspace_bytes, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  SfSizes s;
  const char* why;
  if (!sf_sizes(surf_point_off_host, surf_tri_off_host, n_surfaces, query_off_host, n_segments, surf_of_segment_host, s, &why)) {
    set_error("%s", why);
    return FB_ERR_ARG;
  }
  FB_REQUIRE(surf_points && tris && surf_point_off && surf_tri_off && query_off && surf_of_segment,
             "closest_points: missing device array");
  FB_REQUIRE(s.n_queries == 0 || queries, "closest_points: missing queries");
  if (s.n_queries == 0) return FB_OK;
  const int n_items = (int)(s.n_tris + s.n_queries), n_tris = (int)s.n_tris, nq = (int)s.n_queries;
  if (workspace == nullptr) {
    k_sf_brute<<<div_up(nq, 256), 256, 0, stream>>>(surf_points, tris, surf_tri_off, queries, query_off, n_segments,
                                                    surf_of_segment, s.q0, nq, closest_out, tri_out, dist_out);
    FB_COUNT_LAUNCH(1);
    FB_LAUNCH_CHECK();
    return FB_OK;
  }
  Carver cv(workspace, workspace_bytes);
  SfWs w = sf_carve(cv, s);
  if (!cv.ok()) {
    set_error("closest_points: workspace too small (%zu < %zu)", workspace_bytes, cv.used);
    return FB_ERR_WORKSPACE;
  }
  int gk = 0;  // the largest group that still gives about 8 warps per SM, else the smallest
  while (gk < 3 && s.n_groups[gk] < 8LL * sm_count()) ++gk;
  const int group = SF_GROUPS[gk], n_groups = (int)s.n_groups[gk];
  k_sf_plan<<<1, 1024, 0, stream>>>(surf_tri_off, n_surfaces, query_off, n_segments, surf_of_segment, group, s.t0, s.q0,
                                    n_tris, w.used, w.off_tile, w.off_grp, w.sort_begin, w.sort_end);
  k_sf_bbox<<<n_surfaces, 256, 0, stream>>>(w.used, surf_points, surf_point_off, w.box);
  k_sf_keys<<<div_up(n_items, 256), 256, 0, stream>>>(w.used, surf_points, tris, surf_tri_off, n_surfaces, queries, query_off,
                                                      n_segments, surf_of_segment, w.box, s.t0, s.q0, n_tris, n_items,
                                                      w.keys_in);
  FB_COUNT_LAUNCH(3);
  size_t tmp = w.sort_tmp_bytes;
  FB_CUDA(cub::DeviceSegmentedRadixSort::SortKeys(w.sort_tmp, tmp, (const unsigned long long*)w.keys_in, w.keys_out, n_items,
                                                  n_surfaces + n_segments, (const int*)w.sort_begin, (const int*)w.sort_end,
                                                  SF_SORT_BITS[0], SF_SORT_BITS[1], stream));
  k_sf_fill<<<div_up(n_items, 256), 256, 0, stream>>>(w.used, surf_points, tris, surf_tri_off, n_surfaces, w.keys_out, s.t0,
                                                      n_tris, n_items, w.tv, w.tid, w.perm);
  k_sf_tile_boxes<<<div_up(std::max(s.n_tiles, 1LL), 128), 128, 0, stream>>>(surf_tri_off, w.off_tile, n_surfaces,
                                                                              (int)s.n_tiles, s.t0, w.box, w.tv, w.keys_out,
                                                                              w.tile_lo, w.tile_hi, w.tile_key);
  k_sf_closest<<<div_up(n_groups, SF_WARPS), 32 * SF_WARPS, 0, stream>>>(
      surf_tri_off, query_off, n_segments, surf_of_segment, w.off_tile, w.off_grp, group, n_groups, s.t0, s.q0, w.box, w.tv,
      w.tid, w.tile_lo, w.tile_hi, w.tile_key, w.perm, queries, closest_out, tri_out, dist_out);
  FB_COUNT_LAUNCH(3);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

int focusr_surface_distance_stats(const double* a_dist, const int* a_off, const double* b_dist, const int* b_off, int n_pairs,
                                  double* stats_out, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_pairs > 0, "surface_distance_stats: no pairs");
  FB_REQUIRE(a_dist && a_off && b_dist && b_off && stats_out, "surface_distance_stats: missing device array");
  k_sf_stats<<<n_pairs, SF_STATS_THREADS, 0, stream>>>(a_dist, a_off, b_dist, b_off, stats_out);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

}  // extern "C"
