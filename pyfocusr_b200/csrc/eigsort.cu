// K3: eigenvector normalisation (reference graph.py:254-257), eigsort's cost matrices
// (eigsort.py:34-41, 162-233), the flip + reorder of eigsort.py:108-122 and the spectral
// coordinates of focusr.py:492-508.
//
// The expensive part of eigsort in the reference is 2 n^2 calls of scipy.stats.wasserstein_distance
// on 5000-sample columns (each call sorts both inputs).  Only 3n distinct columns exist
// (target_i, source_j, -source_j after the log shift), so they are sorted once each -- one CTA,
// bitonic network in shared memory -- and every (i, j, flip) distance is then a merged-CDF
// integral evaluated in parallel with one binary search per sample (same definition as
// scipy/stats/_stats_py.py `_cdf_distance`, p = 1).  c_lambda, min(c, c_f), the n x n assignment
// and the flip list are O(n^2..n^3) with n <= ~70 and stay on the host (pyfocusr_b200/eigsort.py).
#include <float.h>
#include <limits.h>

#include <algorithm>
#include <cub/device/device_segmented_radix_sort.cuh>
#include <vector>

#include "common.cuh"
#include "eigsort_decide.h"
#include "knn.cuh"
#include "rowops.h"

namespace fb {

// ---------------------------------------------------------------------------------------------
// B2: per (mesh, column): v <- (v - min) / (max - min) - 0.5
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_normalize_cols(double* __restrict__ vecs, int ld, const int* __restrict__ mesh_off,
                 const int* __restrict__ n_cols) {
  const int mesh = blockIdx.y, j = blockIdx.x;
  if (j >= n_cols[mesh]) return;
  const int r0 = mesh_off[mesh], r1 = mesh_off[mesh + 1];
  double mn = DBL_MAX, mx = -DBL_MAX;
  for (int r = r0 + threadIdx.x; r < r1; r += blockDim.x) {
    const double v = vecs[(size_t)r * ld + j];
    mn = fmin(mn, v);
    mx = fmax(mx, v);
  }
  __shared__ double smn[256], smx[256];
  smn[threadIdx.x] = mn;
  smx[threadIdx.x] = mx;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      smn[threadIdx.x] = fmin(smn[threadIdx.x], smn[threadIdx.x + o]);
      smx[threadIdx.x] = fmax(smx[threadIdx.x], smx[threadIdx.x + o]);
    }
    __syncthreads();
  }
  mn = smn[0];
  const double ptp = FB_SUB(smx[0], mn);
  for (int r = r0 + threadIdx.x; r < r1; r += blockDim.x) {
    const double v = vecs[(size_t)r * ld + j];
    vecs[(size_t)r * ld + j] = FB_SUB(FB_DIV(FB_SUB(v, mn), ptp), 0.5);
  }
}

// C5: new[:, dst[t]] = sign[t] * old[:, src[t]]  (eigsort.py:108-122: flip, then fancy-index copy)
constexpr int MAX_MOVES = 96;
__global__ void __launch_bounds__(128)
k_flip_permute(double* __restrict__ vecs, int ld, const int* __restrict__ mesh_off, const int* __restrict__ dst,
               const int* __restrict__ src, const int* __restrict__ sign, int n_moves) {
  const int mesh = blockIdx.y;
  const int r = mesh_off[mesh] + blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= mesh_off[mesh + 1]) return;
  double tmp[MAX_MOVES];
  double* row = vecs + (size_t)r * ld;
  for (int t = 0; t < n_moves; ++t) {
    const double v = row[src[mesh * n_moves + t]];
    tmp[t] = sign[mesh * n_moves + t] < 0 ? FB_MUL(v, -1.0) : v;
  }
  for (int t = 0; t < n_moves; ++t) row[dst[mesh * n_moves + t]] = tmp[t];
}

// D1: out[i][u] = vecs[i][u] * weights[mesh][u]
__global__ void k_spectral_coords(const double* __restrict__ vecs, int ld, const int* __restrict__ mesh_off,
                                  const double* __restrict__ weights, int ns, double* __restrict__ out,
                                  int max_rows) {
  const int mesh = blockIdx.y;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int nrows = mesh_off[mesh + 1] - mesh_off[mesh];
  if (t >= (long long)nrows * ns) return;
  const int r = mesh_off[mesh] + (int)(t / ns), u = (int)(t % ns);
  out[(size_t)r * ns + u] = FB_MUL(vecs[(size_t)r * ld + u], weights[mesh * ns + u]);
}

// ---------------------------------------------------------------------------------------------
// eigsort costs.  Pair p's samples: target idx_t[off_t[p] .. off_t[p+1]), source idx_s[off_s[p] .. off_s[p+1]) (local
// row ids).  Its 3n sorted columns are stored from n * off_t[p] + 2n * off_s[p] on: n target columns of n_t samples,
// then 2n source columns (source_j, -source_j) of n_s samples.
// ---------------------------------------------------------------------------------------------
struct SampleCol {  // column c of pair p in the sorted-column storage
  long long start;  // first element
  int cnt;          // samples
};
__device__ __forceinline__ SampleCol sample_col(const int* __restrict__ off_t, const int* __restrict__ off_s, int n,
                                                int pair, int c) {
  const int t0 = off_t[pair], s0 = off_s[pair];
  const int n_t = off_t[pair + 1] - t0, n_s = off_s[pair + 1] - s0;
  const long long base = (long long)n * t0 + 2LL * n * s0;
  if (c < n) return {base + (long long)c * n_t, n_t};
  return {base + (long long)n * n_t + (long long)(c - n) * n_s, n_s};
}

// C1: sampled xyz normalised per axis to [0,1] over the sample (graph.py:269-272).
// grid (2, n_pairs): blockIdx.x = 0 target, 1 source.  out_t / out_s [samples][3] in the sample layout
__global__ void __launch_bounds__(256)
k_sample_points(const double* __restrict__ points, const int* __restrict__ mesh_off,
                const int* __restrict__ t_mesh, const int* __restrict__ s_mesh,
                const long long* __restrict__ idx_t, const long long* __restrict__ idx_s,
                const int* __restrict__ off_t, const int* __restrict__ off_s,
                double* __restrict__ out_t, double* __restrict__ out_s) {
  const int pair = blockIdx.y, side = blockIdx.x;
  const int mesh = side == 0 ? t_mesh[pair] : s_mesh[pair];
  const int* off = side == 0 ? off_t : off_s;
  const int s0 = off[pair], n = off[pair + 1] - s0;
  const long long* idx = (side == 0 ? idx_t : idx_s) + s0;
  const size_t base = mesh_off[mesh];
  double mn[3] = {DBL_MAX, DBL_MAX, DBL_MAX}, mx[3] = {-DBL_MAX, -DBL_MAX, -DBL_MAX};
  for (int s = threadIdx.x; s < n; s += blockDim.x)
    for (int a = 0; a < 3; ++a) {
      const double v = points[3 * (base + idx[s]) + a];
      mn[a] = fmin(mn[a], v);
      mx[a] = fmax(mx[a], v);
    }
  __shared__ double smn[3][256], smx[3][256];
  for (int a = 0; a < 3; ++a) {
    smn[a][threadIdx.x] = mn[a];
    smx[a][threadIdx.x] = mx[a];
  }
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o)
      for (int a = 0; a < 3; ++a) {
        smn[a][threadIdx.x] = fmin(smn[a][threadIdx.x], smn[a][threadIdx.x + o]);
        smx[a][threadIdx.x] = fmax(smx[a][threadIdx.x], smx[a][threadIdx.x + o]);
      }
    __syncthreads();
  }
  double* dstp = (side == 0 ? out_t : out_s) + 3 * (size_t)s0;
  for (int s = threadIdx.x; s < n; s += blockDim.x)
    for (int a = 0; a < 3; ++a) {
      const double v = points[3 * (base + idx[s]) + a];
      dstp[3 * (size_t)s + a] = FB_DIV(FB_SUB(v, smn[a][0]), FB_SUB(smx[a][0], smn[a][0]));
    }
}

__global__ void k_linear_offsets(int* off, int n, int stride) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) off[p] = p * stride;
}

// C3 step 1, the key of sample s of column c of pair p (c < n: target_i; c < 2n: source_j; else: -source_j): the
// log shift of eigsort.py:183-188, log(v + 0.5 + eps) with eps = machine epsilon.  NaN cannot be ordered: it becomes
// +inf and sorts last.  The shift never yields -0.0, so every sort orders these keys into the same array.
__device__ __forceinline__ double logcol_key(const double* __restrict__ vecs, int ld, size_t base,
                                             const long long* __restrict__ idx, int s, int c, int n) {
  const int col = c < n ? c : (c < 2 * n ? c - n : c - 2 * n);
  const double e = vecs[(base + idx[s]) * ld + col];
  const double v = log(FB_ADD(FB_ADD(c >= 2 * n ? -e : e, 0.5), 2.220446049250313e-16));
  return v != v ? __longlong_as_double(0x7ff0000000000000LL) : v;
}

// The mesh base row and sample indices of column c of pair p.
__device__ __forceinline__ const long long* col_samples(const int* __restrict__ mesh_off, const int* __restrict__ t_mesh,
                                                        const int* __restrict__ s_mesh, const long long* __restrict__ idx_t,
                                                        const long long* __restrict__ idx_s, const int* __restrict__ off_t,
                                                        const int* __restrict__ off_s, int n, int pair, int c, size_t& base) {
  const bool is_t = c < n;
  base = mesh_off[is_t ? t_mesh[pair] : s_mesh[pair]];
  return is_t ? idx_t + off_t[pair] : idx_s + off_s[pair];
}

// C3 step 1 while every column fits in shared memory (<= EIGSORT_SMEM_SORT_MAX samples): the keys of one column per CTA,
// bitonic-sorted over the column's count padded to a power of two.  Dynamic shared memory is sized for the batch's
// largest column.
constexpr int EIGSORT_SMEM_SORT_MAX = 16384;
__global__ void __launch_bounds__(512)
k_sorted_logcols(const double* __restrict__ vecs, int ld, const int* __restrict__ mesh_off,
                 const int* __restrict__ t_mesh, const int* __restrict__ s_mesh,
                 const long long* __restrict__ idx_t, const long long* __restrict__ idx_s,
                 const int* __restrict__ off_t, const int* __restrict__ off_s, int n, double* __restrict__ sorted) {
  extern __shared__ double sh[];
  const int pair = blockIdx.y, c = blockIdx.x;
  const SampleCol sc = sample_col(off_t, off_s, n, pair, c);
  size_t base;
  const long long* idx = col_samples(mesh_off, t_mesh, s_mesh, idx_t, idx_s, off_t, off_s, n, pair, c, base);
  int p2 = 1;
  while (p2 < sc.cnt) p2 <<= 1;
  for (int s = threadIdx.x; s < p2; s += blockDim.x)
    sh[s] = s < sc.cnt ? logcol_key(vecs, ld, base, idx, s, c, n) : __longlong_as_double(0x7ff0000000000000LL);
  __syncthreads();
  for (int k = 2; k <= p2; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < p2; t += blockDim.x) {
        const int ixj = t ^ j;
        if (ixj > t) {
          const double a = sh[t], b = sh[ixj];
          const bool up = (t & k) == 0;
          if ((a > b) == up) {
            sh[t] = b;
            sh[ixj] = a;
          }
        }
      }
      __syncthreads();
    }
  double* dstp = sorted + sc.start;
  for (int s = threadIdx.x; s < sc.cnt; s += blockDim.x) dstp[s] = sh[s];
}

// C3 step 1 above EIGSORT_SMEM_SORT_MAX samples: the unsorted keys of every column in the sorted-column layout, and the
// (pair, column) segments of the global segmented sort.  grid (div_up(largest column, 256), 3n, n_pairs)
__global__ void __launch_bounds__(256)
k_logcol_keys(const double* __restrict__ vecs, int ld, const int* __restrict__ mesh_off,
              const int* __restrict__ t_mesh, const int* __restrict__ s_mesh,
              const long long* __restrict__ idx_t, const long long* __restrict__ idx_s,
              const int* __restrict__ off_t, const int* __restrict__ off_s, int n, double* __restrict__ keys,
              int* __restrict__ seg_begin, int* __restrict__ seg_end) {
  const int pair = blockIdx.z, c = blockIdx.y;
  const SampleCol sc = sample_col(off_t, off_s, n, pair, c);
  size_t base;
  const long long* idx = col_samples(mesh_off, t_mesh, s_mesh, idx_t, idx_s, off_t, off_s, n, pair, c, base);
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < sc.cnt) keys[sc.start + s] = logcol_key(vecs, ld, base, idx, s, c, n);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    seg_begin[(size_t)pair * 3 * n + c] = (int)sc.start;
    seg_end[(size_t)pair * 3 * n + c] = (int)(sc.start + sc.cnt);
  }
}

__device__ __forceinline__ int lower_bound_d(const double* a, int n, double x) {  // first a[i] >= x
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] < x)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}
__device__ __forceinline__ int upper_bound_d(const double* a, int n, double x) {  // first a[i] > x
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] <= x)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

// C3 step 2: W1(u, v) = sum over the merged sorted values of |F_u - F_v| * gap  (scipy
// _cdf_distance with p=1).  grid (n*n, 2, n_pairs): blockIdx.x = i*n+j, blockIdx.y = flip.
__global__ void __launch_bounds__(256)
k_wasserstein(const double* __restrict__ sorted, const int* __restrict__ off_t, const int* __restrict__ off_s, int n,
              double* __restrict__ c_hist, double* __restrict__ c_hist_f) {
  const int pair = blockIdx.z, flip = blockIdx.y, i = blockIdx.x / n, j = blockIdx.x % n;
  const SampleCol cu = sample_col(off_t, off_s, n, pair, i), cv = sample_col(off_t, off_s, n, pair, (flip ? 2 * n : n) + j);
  const double* u = sorted + cu.start;
  const double* v = sorted + cv.start;
  const int n_t = cu.cnt, n_s = cv.cnt;
  const double inf = __longlong_as_double(0x7ff0000000000000LL);
  double acc = 0.0;
  for (int t = threadIdx.x; t < n_t + n_s; t += blockDim.x) {
    double x, nxt, fu, fv;
    if (t < n_t) {
      x = u[t];
      const int lb = lower_bound_d(v, n_s, x);
      nxt = fmin(t + 1 < n_t ? u[t + 1] : inf, lb < n_s ? v[lb] : inf);
      fu = (double)(t + 1) / (double)n_t;
      fv = (double)lb / (double)n_s;
    } else {
      const int c = t - n_t;
      x = v[c];
      const int ub = upper_bound_d(u, n_t, x);
      nxt = fmin(c + 1 < n_s ? v[c + 1] : inf, ub < n_t ? u[ub] : inf);
      fu = (double)ub / (double)n_t;
      fv = (double)(c + 1) / (double)n_s;
    }
    if (nxt < inf && nxt > x) acc += fabs(fu - fv) * (nxt - x);
  }
  __shared__ double red[256];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) (flip ? c_hist_f : c_hist)[(size_t)pair * n * n + i * n + j] = red[0];
}

// C4: c_spatial[i][j] = sqrt(sum_r (s_j[nn[r]] - t_i[r])^2) / n_t, flipped: (-s_j[nn[r]] - t_i[r]); n_t = the pair's
// target samples.  nn follows the target-sample layout, its indices local to the pair's source samples.
__global__ void __launch_bounds__(128)
k_spatial(const double* __restrict__ vecs, int ld, const int* __restrict__ mesh_off,
          const int* __restrict__ t_mesh, const int* __restrict__ s_mesh, const long long* __restrict__ idx_t,
          const long long* __restrict__ idx_s, const int* __restrict__ off_t, const int* __restrict__ off_s,
          const long long* __restrict__ nn, int n, double* __restrict__ c_spatial, double* __restrict__ c_spatial_f) {
  const int pair = blockIdx.y, i = blockIdx.x / n, j = blockIdx.x % n;
  const size_t bt = mesh_off[t_mesh[pair]], bs = mesh_off[s_mesh[pair]];
  const int t0 = off_t[pair], n_t = off_t[pair + 1] - t0;
  const long long* it = idx_t + t0;
  const long long* is = idx_s + off_s[pair];
  const long long* nnp = nn + t0;
  double a = 0.0, af = 0.0;
  for (int r = threadIdx.x; r < n_t; r += blockDim.x) {
    const double tv = vecs[(bt + it[r]) * ld + i];
    const double sv = vecs[(bs + is[nnp[r]]) * ld + j];
    const double d = sv - tv, df = -sv - tv;
    a += d * d;
    af += df * df;
  }
  __shared__ double r0[128], r1[128];
  r0[threadIdx.x] = a;
  r1[threadIdx.x] = af;
  __syncthreads();
  for (int o = 64; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      r0[threadIdx.x] += r0[threadIdx.x + o];
      r1[threadIdx.x] += r1[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    c_spatial[(size_t)pair * n * n + i * n + j] = sqrt(r0[0]) / (double)n_t;
    c_spatial_f[(size_t)pair * n * n + i * n + j] = sqrt(r1[0]) / (double)n_t;
  }
}

// sizes of one eigsort cost call, from the host copies of the sample offsets
struct EigsortSizes {
  long long tot_t = 0, tot_s = 0, n_keys = 0;  // target / source samples, elements of the sorted columns
  int max_t = 0, max_s = 0;                     // largest pair
  bool global_sort = false;                     // some column holds more than EIGSORT_SMEM_SORT_MAX samples
};

static bool eigsort_sizes(const int* off_t, const int* off_s, int n_pairs, int n, EigsortSizes& z, const char** why) {
  if (!off_t || !off_s || n_pairs <= 0 || n <= 0) {
    *why = "eigsort_costs: no pairs, no features or missing host offsets";
    return false;
  }
  if (n_pairs > 65535 || (long long)n * n > 65535) {
    *why = "eigsort_costs: grid too large";
    return false;
  }
  if (off_t[0] != 0 || off_s[0] != 0) {
    *why = "eigsort_costs: sample offsets must start at 0";
    return false;
  }
  for (int p = 0; p < n_pairs; ++p) {
    const int ct = off_t[p + 1] - off_t[p], cs = off_s[p + 1] - off_s[p];
    if (ct <= 0 || cs <= 0) {
      *why = "eigsort_costs: every pair needs at least one target and one source sample (offsets must increase)";
      return false;
    }
    z.max_t = std::max(z.max_t, ct);
    z.max_s = std::max(z.max_s, cs);
  }
  z.tot_t = off_t[n_pairs];
  z.tot_s = off_s[n_pairs];
  z.n_keys = (long long)n * z.tot_t + 2LL * n * z.tot_s;
  z.global_sort = std::max(z.max_t, z.max_s) > EIGSORT_SMEM_SORT_MAX;
  if (z.global_sort && z.n_keys > INT_MAX) {
    *why = "eigsort_costs: more than 2^31 - 1 sorted-column elements in one call";
    return false;
  }
  return true;
}

static size_t eigsort_sort_tmp_bytes(const EigsortSizes& z, int n_segments) {
  size_t bytes = 0;
  cub::DeviceSegmentedRadixSort::SortKeys(nullptr, bytes, (const double*)nullptr, (double*)nullptr, (int)z.n_keys, n_segments,
                                          (const int*)nullptr, (const int*)nullptr);
  return bytes;
}

struct EigsortWs {
  double *pts_t, *pts_s, *sorted, *keys = nullptr;
  int *seg_begin = nullptr, *seg_end = nullptr;
  void* sort_tmp = nullptr;
  size_t sort_tmp_bytes = 0, knn_bytes;
  char* knn_ws;
};

static EigsortWs eigsort_carve(Carver& cv, const EigsortSizes& z, int n_pairs, int n) {
  EigsortWs w;
  w.pts_t = cv.take<double>((size_t)z.tot_t * 3);
  w.pts_s = cv.take<double>((size_t)z.tot_s * 3);
  w.sorted = cv.take<double>((size_t)z.n_keys);
  w.knn_bytes = knn_pruned_workspace_bytes(z.tot_s, z.tot_t, n_pairs, 3);
  w.knn_ws = cv.take<char>(w.knn_bytes);
  if (z.global_sort) {
    const int n_segments = 3 * n * n_pairs;
    w.keys = cv.take<double>((size_t)z.n_keys);
    w.seg_begin = cv.take<int>(n_segments);
    w.seg_end = cv.take<int>(n_segments);
    w.sort_tmp_bytes = eigsort_sort_tmp_bytes(z, n_segments);
    w.sort_tmp = cv.take<char>(w.sort_tmp_bytes);
  }
  return w;
}

// The uniform layout: pair p's samples are idx_t[p * n_samp_t ..] and idx_s[p * n_samp_s ..]
static std::vector<int> linear_offsets(int n_pairs, int stride) {
  std::vector<int> off((size_t)std::max(n_pairs, 0) + 1);
  for (size_t p = 0; p < off.size(); ++p) off[p] = (int)p * stride;
  return off;
}

}  // namespace fb

using namespace fb;

extern "C" {

int focusr_normalize_columns(double* vecs, int n_points, int ld, const int* mesh_point_off, int n_meshes,
                             const int* n_cols, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_points > 0 && ld > 0 && n_meshes > 0, "normalize_columns: empty");
  dim3 grid(ld, n_meshes);
  k_normalize_cols<<<grid, 256, 0, stream>>>(vecs, ld, mesh_point_off, n_cols);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

int focusr_flip_permute_columns(double* vecs, int n_points, int ld, const int* mesh_point_off, int n_meshes,
                                int max_mesh_points, const int* dst, const int* src, const int* sign,
                                int n_moves, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_moves >= 0 && n_moves <= MAX_MOVES, "flip_permute: at most %d columns", MAX_MOVES);
  if (n_moves == 0) return FB_OK;
  dim3 grid(div_up(max_mesh_points, 128), n_meshes);
  k_flip_permute<<<grid, 128, 0, stream>>>(vecs, ld, mesh_point_off, dst, src, sign, n_moves);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

int focusr_spectral_coords(const double* vecs, int n_points, int ld, const int* mesh_point_off, int n_meshes,
                           int max_mesh_points, const double* weights, int ns, double* out,
                           focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(ns >= 1 && ns <= ld, "spectral_coords: need 1 <= ns <= ld");
  dim3 grid(div_up((long long)max_mesh_points * ns, 256), n_meshes);
  k_spectral_coords<<<grid, 256, 0, stream>>>(vecs, ld, mesh_point_off, weights, ns, out, max_mesh_points);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

// C2, C5, D1 on the device: one thread per pair runs eigsort_decide_pair (eigsort_decide.h) and writes the column moves
// of BOTH meshes of the pair (identity for the reference graph) and their spectral weights.
__global__ void __launch_bounds__(64)
k_eigsort_decide(const double* __restrict__ eig_vals, int ldv, const int* __restrict__ n_found, const int* __restrict__ t_mesh,
                 const int* __restrict__ s_mesh, int n_pairs, const double* __restrict__ c_hist,
                 const double* __restrict__ c_hist_f, const double* __restrict__ c_spatial,
                 const double* __restrict__ c_spatial_f, int n, int ns, int target_as_reference, int weighted,
                 double* __restrict__ q_out, int* __restrict__ dst, int* __restrict__ src, int* __restrict__ sign,
                 double* __restrict__ weights, double* __restrict__ scratch, int* __restrict__ status) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pairs) return;
  const int mt = t_mesh[p], ms = s_mesh[p];
  const size_t nn = (size_t)n * n;
  int d[LSAP_MAX], s[LSAP_MAX], g[LSAP_MAX];
  double w[LSAP_MAX];
  const int rc = eigsort_decide_pair(eig_vals + (size_t)mt * ldv, n_found[mt], eig_vals + (size_t)ms * ldv, n_found[ms],
                                     c_hist + p * nn, c_hist_f + p * nn, c_spatial + p * nn, c_spatial_f + p * nn, n, ns,
                                     target_as_reference != 0, weighted != 0, q_out + (size_t)p * n, d, s, g, w,
                                     scratch + (size_t)p * 2 * nn);
  if (rc != 0) atomicExch(status, 1);
  const int moved = target_as_reference ? ms : mt, fixed = target_as_reference ? mt : ms;
  for (int k = 0; k < n; ++k) {
    dst[(size_t)moved * n + k] = rc == 0 ? d[k] : k;
    src[(size_t)moved * n + k] = rc == 0 ? s[k] : k;
    sign[(size_t)moved * n + k] = rc == 0 ? g[k] : 1;
    dst[(size_t)fixed * n + k] = k;
    src[(size_t)fixed * n + k] = k;
    sign[(size_t)fixed * n + k] = 1;
  }
  for (int k = 0; k < ns; ++k) weights[(size_t)mt * ns + k] = weights[(size_t)ms * ns + k] = rc == 0 ? w[k] : 1.0;
}

size_t focusr_eigsort_ragged_workspace_bytes(const int* samp_off_t_host, const int* samp_off_s_host, int n_pairs,
                                             int n_features) {
  EigsortSizes z;
  const char* why;
  if (!eigsort_sizes(samp_off_t_host, samp_off_s_host, n_pairs, n_features, z, &why)) return 0;
  Carver cv(nullptr, 0);
  eigsort_carve(cv, z, n_pairs, n_features);
  return cv.used + 1024;
}

int focusr_eigsort_costs_ragged(const double* vecs, int ld, const double* points, const int* mesh_point_off,
                                const int* t_mesh, const int* s_mesh, int n_pairs, const long long* idx_t,
                                const long long* idx_s, const int* samp_off_t, const int* samp_off_s,
                                const int* samp_off_t_host, const int* samp_off_s_host, int n_features, double* c_hist,
                                double* c_hist_f, double* c_spatial, double* c_spatial_f, long long* nn_idx,
                                void* workspace, size_t workspace_bytes, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_features > 0 && n_features <= ld, "eigsort_costs: need 1 <= n_features <= ld");
  EigsortSizes z;
  const char* why;
  if (!eigsort_sizes(samp_off_t_host, samp_off_s_host, n_pairs, n_features, z, &why)) {
    set_error("%s", why);
    return FB_ERR_ARG;
  }
  const int n = n_features;
  Carver cv(workspace, workspace_bytes);
  const EigsortWs w = eigsort_carve(cv, z, n_pairs, n);
  if (!cv.ok()) {
    set_error("eigsort_costs: workspace too small (%zu < %zu)", workspace_bytes, cv.used);
    return FB_ERR_WORKSPACE;
  }
  k_sample_points<<<dim3(2, n_pairs), 256, 0, stream>>>(points, mesh_point_off, t_mesh, s_mesh, idx_t, idx_s, samp_off_t,
                                                        samp_off_s, w.pts_t, w.pts_s);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  // nearest sampled source point of every sampled target point (eigsort.py:203-204)
  int rc;
  if (knn_pruned_applicable(z.max_s, z.max_t, 3, 1))
    rc = launch_knn_pruned(w.pts_s, 3, samp_off_s, w.pts_t, 3, samp_off_t, n_pairs, z.max_s, z.max_t, z.tot_s, z.tot_t, 3,
                           1, nn_idx, nullptr, w.knn_ws, w.knn_bytes, stream);
  else
    rc = launch_knn(w.pts_s, 3, samp_off_s, w.pts_t, 3, samp_off_t, n_pairs, z.max_t, 3, 1, nn_idx, nullptr, stream);
  if (rc) return rc;
  if (!z.global_sort) {
    int p2 = 1;
    while (p2 < std::max(z.max_t, z.max_s)) p2 <<= 1;
    const size_t smem = sizeof(double) * (size_t)p2;
    // the opt-in is per device and per function: set whenever it is needed (cheap), never cached process-wide
    if (smem > 48 * 1024) FB_CUDA(cudaFuncSetAttribute(k_sorted_logcols, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_sorted_logcols<<<dim3(3 * n, n_pairs), 512, smem, stream>>>(vecs, ld, mesh_point_off, t_mesh, s_mesh, idx_t, idx_s,
                                                                  samp_off_t, samp_off_s, n, w.sorted);
    FB_COUNT_LAUNCH(1);
  } else {
    const dim3 grid(div_up(std::max(z.max_t, z.max_s), 256), 3 * n, n_pairs);
    k_logcol_keys<<<grid, 256, 0, stream>>>(vecs, ld, mesh_point_off, t_mesh, s_mesh, idx_t, idx_s, samp_off_t, samp_off_s, n,
                                            w.keys, w.seg_begin, w.seg_end);
    FB_COUNT_LAUNCH(1);
    FB_LAUNCH_CHECK();
    size_t tmp = w.sort_tmp_bytes;
    FB_CUDA(cub::DeviceSegmentedRadixSort::SortKeys(w.sort_tmp, tmp, (const double*)w.keys, w.sorted, (int)z.n_keys,
                                                    3 * n * n_pairs, (const int*)w.seg_begin, (const int*)w.seg_end, 0,
                                                    (int)(8 * sizeof(double)), stream));
  }
  k_wasserstein<<<dim3(n * n, 2, n_pairs), 256, 0, stream>>>(w.sorted, samp_off_t, samp_off_s, n, c_hist, c_hist_f);
  k_spatial<<<dim3(n * n, n_pairs), 128, 0, stream>>>(vecs, ld, mesh_point_off, t_mesh, s_mesh, idx_t, idx_s, samp_off_t,
                                                      samp_off_s, nn_idx, n, c_spatial, c_spatial_f);
  FB_COUNT_LAUNCH(2);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

size_t focusr_eigsort_workspace_bytes(int n_pairs, int n_samp_t, int n_samp_s, int n_features) {
  if (n_pairs <= 0 || (long long)n_pairs * std::max(n_samp_t, n_samp_s) > INT_MAX) return 0;
  const std::vector<int> ot = linear_offsets(n_pairs, n_samp_t), os = linear_offsets(n_pairs, n_samp_s);
  const size_t ragged = focusr_eigsort_ragged_workspace_bytes(ot.data(), os.data(), n_pairs, n_features);
  return ragged ? 2 * align_up(sizeof(int) * ((size_t)n_pairs + 1)) + ragged : 0;
}

int focusr_eigsort_costs(const double* vecs, int ld, const double* points, const int* mesh_point_off,
                         const int* t_mesh, const int* s_mesh, int n_pairs, const long long* idx_t,
                         const long long* idx_s, int n_samp_t, int n_samp_s, int n_features, double* c_hist,
                         double* c_hist_f, double* c_spatial, double* c_spatial_f, long long* nn_idx,
                         void* workspace, size_t workspace_bytes, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_pairs > 0 && n_samp_t > 0 && n_samp_s > 0 && n_features > 0 && n_features <= ld,
             "eigsort_costs: bad sizes");
  FB_REQUIRE((long long)n_pairs * std::max(n_samp_t, n_samp_s) <= INT_MAX, "eigsort_costs: more than 2^31 - 1 samples");
  Carver cv(workspace, workspace_bytes);
  int* off_t = cv.take<int>((size_t)n_pairs + 1);
  int* off_s = cv.take<int>((size_t)n_pairs + 1);
  cv.used = align_up(cv.used);
  if (!cv.ok()) {
    set_error("eigsort_costs: workspace too small (%zu < %zu)", workspace_bytes, cv.used);
    return FB_ERR_WORKSPACE;
  }
  k_linear_offsets<<<div_up(n_pairs + 1, 256), 256, 0, stream>>>(off_t, n_pairs + 1, n_samp_t);
  k_linear_offsets<<<div_up(n_pairs + 1, 256), 256, 0, stream>>>(off_s, n_pairs + 1, n_samp_s);
  FB_COUNT_LAUNCH(2);
  FB_LAUNCH_CHECK();
  const std::vector<int> ot = linear_offsets(n_pairs, n_samp_t), os = linear_offsets(n_pairs, n_samp_s);
  return focusr_eigsort_costs_ragged(vecs, ld, points, mesh_point_off, t_mesh, s_mesh, n_pairs, idx_t, idx_s, off_t, off_s,
                                     ot.data(), os.data(), n_features, c_hist, c_hist_f, c_spatial, c_spatial_f, nn_idx,
                                     cv.base + cv.used, workspace_bytes - cv.used, stream_);
}

size_t focusr_eigsort_decide_workspace_bytes(int n_pairs, int n_features) {
  return sizeof(double) * 2 * (size_t)n_pairs * n_features * n_features + 256;
}

int focusr_eigsort_decide(const double* eig_vals, int ldv, const int* n_found, const int* t_mesh, const int* s_mesh,
                          int n_pairs, const double* c_hist, const double* c_hist_f, const double* c_spatial,
                          const double* c_spatial_f, int n_features, int ns, int target_as_reference, int weighted,
                          double* q_out, int* dst, int* src, int* sign, double* weights, int* status, void* workspace,
                          size_t workspace_bytes, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_pairs > 0 && n_features >= 1 && n_features <= LSAP_MAX && ns >= 1 && ns <= n_features && n_features <= ldv,
             "eigsort_decide: need 1 <= ns <= n_features <= %d", LSAP_MAX);
  FB_REQUIRE(workspace_bytes >= focusr_eigsort_decide_workspace_bytes(n_pairs, n_features), "eigsort_decide: workspace too small");
  FB_CUDA(cudaMemsetAsync(status, 0, sizeof(int), stream));
  k_eigsort_decide<<<div_up(n_pairs, 64), 64, 0, stream>>>(eig_vals, ldv, n_found, t_mesh, s_mesh, n_pairs, c_hist, c_hist_f,
                                                           c_spatial, c_spatial_f, n_features, ns, target_as_reference, weighted,
                                                           q_out, dst, src, sign, weights, static_cast<double*>(workspace), status);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}
}
