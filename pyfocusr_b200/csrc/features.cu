// K12  Node features of a batch: the per-mesh reductions of Graph.norm_node_features (graph.py:121-142) with the edge
// points of graph.py:166-175, and the extended correspondence coordinates of focusr.py:218-295.  Every result equals
// numpy's bit for bit:
//   - np.sum / np.mean / np.std on a contiguous float64 array use numpy's pairwise summation: fewer than 8 elements
//     are added left to right; a block of 8..128 elements uses 8 interleaved accumulators combined as
//     ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the remainder left to right; a longer run splits at
//     n2 = n/2 - (n/2) % 8 and the halves' sums are added.  pw_sum restates that tree: the leaves (64..128 elements
//     each) are summed in parallel, one thread per leaf, and one thread adds them up in the tree's shape.
//   - std = sqrt(pw((x - mean) * (x - mean)) / n) with the square rounded before it is added (__dmul_rn / __dadd_rn:
//     no FMA contraction anywhere a product meets a sum).
//   - min / max / ptp are exact; a NaN anywhere gives NaN, as np.min / np.max do.
// One CTA per (mesh, feature column) or per mesh; no floating-point atomics, so nothing depends on the batch.
#include <cmath>

#include "common.cuh"

namespace fb {

constexpr int NF_THREADS = 256;
constexpr int PW_BLOCK = 128;  // numpy's PW_BLOCKSIZE
constexpr int PW_LEAF_MIN = 64;  // every leaf of a run longer than 128 holds at least 64 elements (n2 >= 64)

// min / max that propagate NaN (np.minimum / np.maximum)
__device__ __forceinline__ double nmin(double a, double b) { return (a < b || isnan(a)) ? a : b; }
__device__ __forceinline__ double nmax(double a, double b) { return (a > b || isnan(a)) ? a : b; }

// numpy's sum of a run of n <= 128 elements v(b) .. v(b + n - 1)
template <class V>
__device__ double pw_leaf(const V& v, int b, int n) {
  if (n < 8) {
    double res = -0.0;
    for (int i = 0; i < n; ++i) res = __dadd_rn(res, v(b + i));
    return res;
  }
  double r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = v(b + j);
  int i = 8;
  for (; i < n - (n % 8); i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], v(b + i + j));
  }
  double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
  for (; i < n; ++i) res = __dadd_rn(res, v(b + i));
  return res;
}

__device__ __forceinline__ int pw_split(int m) { return m / 2 - (m / 2) % 8; }

// the leaf of numpy's pairwise tree over [0, n) that holds position p: [*lb, *lb + *lm)
__device__ __forceinline__ void pw_find_leaf(int n, int p, int* lb, int* lm) {
  int b = 0, m = n;
  while (m > PW_BLOCK) {
    const int n2 = pw_split(m);
    if (p < b + n2) {
      m = n2;
    } else {
      b += n2;
      m -= n2;
    }
  }
  *lb = b;
  *lm = m;
}

// numpy's pairwise sum of v(0) .. v(n - 1), returned to every thread of the CTA.  `slot` holds one double per 64
// positions (the leaf sums, indexed by the window their leaf starts in: at most one leaf starts in a window).
template <class V>
__device__ double pw_sum(const V& v, int n, double* __restrict__ slot, double* s_bcast) {
  if (n <= PW_BLOCK) {
    if (threadIdx.x == 0) *s_bcast = pw_leaf(v, 0, n);
    __syncthreads();
    const double r = *s_bcast;
    __syncthreads();
    return r;
  }
  const int n_win = (n + PW_LEAF_MIN - 1) / PW_LEAF_MIN;
  for (int w = threadIdx.x; w < n_win; w += blockDim.x) {
    const int p = w * PW_LEAF_MIN;
    int lb, lm;
    pw_find_leaf(n, p, &lb, &lm);
    if (lb != p) {  // the leaf holding p started in an earlier window; the next one may start in this window
      const int nb = lb + lm;
      if (nb >= n || nb >= p + PW_LEAF_MIN) continue;
      pw_find_leaf(n, nb, &lb, &lm);
    }
    slot[w] = pw_leaf(v, lb, lm);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    // post-order walk of the tree: a frame is a run (b, m); state 0 = nothing summed, 1 = left half summed
    int sb[32], sm[32], st[32];
    double left[32];
    int top = 0;
    sb[0] = 0;
    sm[0] = n;
    st[0] = 0;
    double ret = 0.0;
    for (;;) {
      const int b = sb[top], m = sm[top];
      if (m <= PW_BLOCK || st[top] == 2) {
        if (m <= PW_BLOCK) ret = slot[b / PW_LEAF_MIN];
        else ret = __dadd_rn(left[top], ret);
        if (top == 0) break;
        --top;
        continue;
      }
      const int n2 = pw_split(m);
      if (st[top] == 0) {
        st[top] = 1;
        ++top;
        sb[top] = b;
        sm[top] = n2;
        st[top] = 0;
      } else {
        left[top] = ret;
        st[top] = 2;
        ++top;
        sb[top] = b + n2;
        sm[top] = m - n2;
        st[top] = 0;
      }
    }
    *s_bcast = ret;
  }
  __syncthreads();
  const double r = *s_bcast;
  __syncthreads();
  return r;
}

// CTA-wide NaN-propagating min and max; every thread gets the result
__device__ void block_min_max(double& mn, double& mx, double* s_red) {
  for (int o = 16; o > 0; o >>= 1) {
    mn = nmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = nmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if ((threadIdx.x & 31) == 0) {
    s_red[w] = mn;
    s_red[32 + w] = mx;
  }
  __syncthreads();
  mn = s_red[0];
  mx = s_red[32];
  for (int i = 1; i < nw; ++i) {
    mn = nmin(mn, s_red[i]);
    mx = nmax(mx, s_red[32 + i]);
  }
  __syncthreads();
}

// mean_pts_scale_range = np.mean(np.ptp(points, axis=0)) and the per-axis minimum of one mesh's points
__device__ double mesh_scale_range(const double* __restrict__ pts, int n, double* pmin, double* s_red) {
  double ptp[3];
  for (int a = 0; a < 3; ++a) {
    double mn = INFINITY, mx = -INFINITY;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const double x = pts[3 * (size_t)i + a];
      mn = nmin(mn, x);
      mx = nmax(mx, x);
    }
    block_min_max(mn, mx, s_red);
    pmin[a] = mn;
    ptp[a] = __dsub_rn(mx, mn);
  }
  return __ddiv_rn(__dadd_rn(__dadd_rn(ptp[0], ptp[1]), ptp[2]), 3.0);
}

struct ColView {
  const double* p;
  int ld;
  __device__ __forceinline__ double operator()(int i) const { return p[(size_t)i * ld]; }
};
struct SqDevView {
  const double* p;
  int ld;
  double mean;
  __device__ __forceinline__ double operator()(int i) const {
    const double d = __dsub_rn(p[(size_t)i * ld], mean);
    return __dmul_rn(d, d);
  }
};


// The value of feature column c of one mesh after graph.py:123-128 (z-score, then the cap), before the 0-1 range
struct ZView {
  const double* x;
  int ld, norm_std, has_cap;
  double mean, sd, cap;
  __device__ __forceinline__ double operator()(int i) const {
    double y = x[(size_t)i * ld];
    if (norm_std) {
      y = __ddiv_rn(__dsub_rn(y, mean), sd);
      if (has_cap) {  // f[f > cap] = cap, then f[f < -cap] = -cap
        if (y > cap) y = cap;
        if (y < -cap) y = -cap;
      }
    }
    return y;
  }
};

// grid (n_meshes, n_features): graph.py:121-142 for one column of one mesh, then its edge-point column (graph.py:166-175)
__global__ void __launch_bounds__(NF_THREADS)
k_node_features(const double* __restrict__ raw, const double* __restrict__ points, const int* __restrict__ mesh_off, int f,
                size_t slots_per_col, int norm_std, int has_cap, double cap, int norm_0_1, double* __restrict__ slots,
                double* __restrict__ out, double* __restrict__ edge_points) {
  __shared__ double s_red[64];
  __shared__ double s_bcast;
  const int m = blockIdx.x, c = blockIdx.y;
  const int base = mesh_off[m], n = mesh_off[m + 1] - base;
  if (n <= 0) return;
  const double* x = raw + (size_t)base * f + c;
  double* slot = slots + (size_t)c * slots_per_col + (size_t)m + (size_t)(base / PW_LEAF_MIN);  // focusr_node_features
  ZView z{x, f, norm_std, has_cap, 0.0, 1.0, cap};
  if (norm_std) {
    z.mean = __ddiv_rn(pw_sum(ColView{x, f}, n, slot, &s_bcast), (double)n);
    z.sd = __dsqrt_rn(__ddiv_rn(pw_sum(SqDevView{x, f, z.mean}, n, slot, &s_bcast), (double)n));
  }
  double lo = 0.0, ptp = 1.0;
  if (norm_0_1) {
    double mn = INFINITY, mx = -INFINITY;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const double y = z(i);
      mn = nmin(mn, y);
      mx = nmax(mx, y);
    }
    block_min_max(mn, mx, s_red);
    lo = mn;
    ptp = __dsub_rn(mx, mn);
  }
  double scale = 0.0, pmin[3];
  if (edge_points) scale = mesh_scale_range(points + 3 * (size_t)base, n, pmin, s_red);
  const int ld_e = 3 + f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    double y = z(i);
    if (norm_0_1) y = __ddiv_rn(__dsub_rn(y, lo), ptp);
    out[(size_t)(base + i) * f + c] = y;
    if (edge_points) {
      double* e = edge_points + (size_t)(base + i) * ld_e;
      e[3 + c] = __dmul_rn(y, scale);
      if (c == 0) {
        const double* p = points + 3 * (size_t)(base + i);
        e[0] = p[0];
        e[1] = p[1];
        e[2] = p[2];
      }
    }
  }
}

// grid n_meshes: focusr.py:218-295 for one mesh -- out = [spectral | smoothed features rescaled to the spectral range |
// normed or raw xyz]
__global__ void __launch_bounds__(NF_THREADS)
k_feature_coords(const double* __restrict__ spectral, int ns, const double* __restrict__ smoothed, int f,
                 const double* __restrict__ points, const int* __restrict__ mesh_off, int include_points, int norm_physical,
                 double* __restrict__ out) {
  __shared__ double s_red[64];
  const int m = blockIdx.x;
  const int base = mesh_off[m], n = mesh_off[m + 1] - base;
  if (n <= 0) return;
  const int ld = ns + f + (include_points ? 3 : 0);
  double scale = 1.0, pmin[3] = {0.0, 0.0, 0.0};
  if (include_points) scale = mesh_scale_range(points + 3 * (size_t)base, n, pmin, s_red);
  const bool mul = include_points && !norm_physical;  // focusr.py:289-295: every column so far times the xyz range
  const double* sp = spectral + (size_t)base * ns;
  double* o = out + (size_t)base * ld;
  const long long n_sp = (long long)n * ns;
  for (long long t = threadIdx.x; t < n_sp; t += blockDim.x) {
    const int i = (int)(t / ns), u = (int)(t - (long long)i * ns);
    const double v = sp[t];
    o[(size_t)i * ld + u] = mul ? __dmul_rn(v, scale) : v;
  }
  if (f > 0) {
    double mn = INFINITY, mx = -INFINITY;  // np.ptp(coords) over all ns columns
    for (long long t = threadIdx.x; t < n_sp; t += blockDim.x) {
      mn = nmin(mn, sp[t]);
      mx = nmax(mx, sp[t]);
    }
    block_min_max(mn, mx, s_red);
    const double range = __dsub_rn(mx, mn);
    for (int k = 0; k < f; ++k) {
      const double* g = smoothed + (size_t)base * f + k;
      double gmn = INFINITY, unused = -INFINITY;
      for (int i = threadIdx.x; i < n; i += blockDim.x) gmn = nmin(gmn, g[(size_t)i * f]);
      block_min_max(gmn, unused, s_red);
      double unused2 = INFINITY, gmx = -INFINITY;  // max of g - min(g)
      for (int i = threadIdx.x; i < n; i += blockDim.x) gmx = nmax(gmx, __dsub_rn(g[(size_t)i * f], gmn));
      block_min_max(unused2, gmx, s_red);
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double v = __dmul_rn(range, __ddiv_rn(__dsub_rn(g[(size_t)i * f], gmn), gmx));
        if (mul) v = __dmul_rn(v, scale);
        o[(size_t)i * ld + ns + k] = v;
      }
    }
  }
  if (include_points) {
    for (int t = threadIdx.x; t < 3 * n; t += blockDim.x) {
      const int i = t / 3, a = t - 3 * i;
      const double p = points[3 * (size_t)base + t];
      o[(size_t)i * ld + ns + f + a] = norm_physical ? __ddiv_rn(__dsub_rn(p, pmin[a]), scale) : p;
    }
  }
}

}  // namespace fb

using namespace fb;

extern "C" {

size_t focusr_node_features_workspace_bytes(int n_points, int n_meshes, int n_features) {
  if (n_points <= 0 || n_meshes <= 0 || n_features <= 0) return 0;
  const size_t slots_per_col = (size_t)n_meshes + (size_t)n_points / PW_LEAF_MIN + 1;
  return slots_per_col * (size_t)n_features * sizeof(double) + 256;
}

int focusr_node_features(const double* raw, const double* points, int n_points, const int* mesh_point_off, int n_meshes,
                         int n_features, int norm_std, int has_cap, double cap, int norm_0_1, double* features_out,
                         double* edge_points, void* workspace, size_t workspace_bytes, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_points > 0 && n_meshes > 0 && n_features > 0, "node_features: bad sizes");
  FB_REQUIRE(n_features <= 61, "node_features: at most 61 features (edge points of at most 64 coordinates)");
  FB_REQUIRE(raw && features_out && mesh_point_off && (points || !edge_points), "node_features: null argument");
  const size_t need = focusr_node_features_workspace_bytes(n_points, n_meshes, n_features);
  if (need > workspace_bytes || !workspace) {
    set_error("node_features: workspace too small (%zu < %zu)", workspace_bytes, need);
    return FB_ERR_WORKSPACE;
  }
  const size_t slots_per_col = (size_t)n_meshes + (size_t)n_points / PW_LEAF_MIN + 1;
  k_node_features<<<dim3(n_meshes, n_features), NF_THREADS, 0, stream>>>(raw, points, mesh_point_off, n_features, slots_per_col,
                                                                       norm_std != 0, has_cap != 0, cap, norm_0_1 != 0,
                                                                       (double*)workspace, features_out, edge_points);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

int focusr_feature_coords(const double* spectral, int ns, const double* smoothed_features, int n_features,
                          const double* points, int n_points, const int* mesh_point_off, int n_meshes, int include_points,
                          int norm_physical_and_spectral, double* out, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_points > 0 && n_meshes > 0 && ns >= 1 && n_features >= 0, "feature_coords: bad sizes");
  FB_REQUIRE(spectral && out && mesh_point_off && (smoothed_features || n_features == 0) && (points || !include_points),
             "feature_coords: null argument");
  k_feature_coords<<<n_meshes, NF_THREADS, 0, stream>>>(spectral, ns, smoothed_features, n_features, points, mesh_point_off,
                                                        include_points != 0, norm_physical_and_spectral != 0, out);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

}  // extern "C"
