// K4: exact fp64 k-nearest neighbours, tiled brute force.  Replaces scipy cKDTree build + query
// (reference focusr.py:351-353 k=1, focusr.py:409-413 k=3 in a Python loop per point,
// eigsort.py:203-204) and the k=3 inverse-distance weighting of focusr.py:415-426.
//
// One thread owns one query (coordinates and its running top-k in registers); a CTA of 256 queries
// streams the reference set through shared memory in tiles, every thread reading the same
// reference (a broadcast, conflict-free).  Squared distances are accumulated as
// ((q0-r0)^2 + (q1-r1)^2) + ... with separate multiply and add, i.e. exactly numpy's / cKDTree's
// direct-difference arithmetic (never |q|^2+|r|^2-2qr: cancellation would change near-ties,
// SURVEY.md section 7.3-7); a strict `<` while scanning references in ascending order gives the
// lower index on ties.  At these shapes (AI ~ 2000 flop/B) the kernel is FP64-ALU-bound, not
// HBM-bound: DESIGN.md reports it against the FP64 pipe, with queries/s.
#include "common.cuh"
#include "knn.cuh"
#include "rowops.h"

namespace fb {

constexpr int KNN_THREADS = 256;
constexpr int KNN_TILE = 512;   // references per shared-memory tile
constexpr int KNN_MAX_DIM = 32;
constexpr int KNN_MAX_K = 8;

template <int D, int K>
__global__ void __launch_bounds__(KNN_THREADS)
k_knn(const double* __restrict__ refs, int ld_refs, const int* __restrict__ ref_off,
      const int* __restrict__ ref_seg, const double* __restrict__ queries, int ld_queries,
      const int* __restrict__ query_off, int dim_rt, int k_rt, long long* __restrict__ idx, double* __restrict__ dist) {
  extern __shared__ double tile[];  // [KNN_TILE][dim]
  const int dim = D > 0 ? D : dim_rt;
  const int kk = K > 0 ? K : k_rt;
  constexpr int DM = D > 0 ? D : KNN_MAX_DIM;
  constexpr int KM = K > 0 ? K : KNN_MAX_K;
  const int seg = blockIdx.y;
  const int q0 = query_off[seg] + blockIdx.x * KNN_THREADS;
  const int q1 = query_off[seg + 1];
  if (q0 >= q1) return;
  const int rseg = ref_seg ? ref_seg[seg] : seg;
  const int rbeg = ref_off[rseg], rend = ref_off[rseg + 1];
  const int q = q0 + threadIdx.x;
  const bool valid = q < q1;
  double qc[DM];
#pragma unroll
  for (int c = 0; c < DM; ++c) qc[c] = (valid && c < dim) ? queries[(size_t)q * ld_queries + c] : 0.0;
  double best[KM];
  int besti[KM];
#pragma unroll
  for (int j = 0; j < KM; ++j) {
    best[j] = __longlong_as_double(0x7ff0000000000000LL);  // +inf
    besti[j] = -1;
  }
  for (int t0 = rbeg; t0 < rend; t0 += KNN_TILE) {
    const int tn = min(KNN_TILE, rend - t0);
    __syncthreads();
    for (int e = threadIdx.x; e < tn * dim; e += KNN_THREADS) {
      const int r = e / dim, c = e - r * dim;
      tile[e] = refs[(size_t)(t0 + r) * ld_refs + c];
    }
    __syncthreads();
    if (valid) {
      for (int r = 0; r < tn; ++r) {
        const double* rp = tile + r * dim;
        double d2 = 0.0;
#pragma unroll
        for (int c = 0; c < DM; ++c)
          if (c < dim) {
            const double df = FB_SUB(qc[c], rp[c]);
            d2 = FB_ADD(d2, FB_MUL(df, df));
          }
        // insertion into the ascending top-k, all register indices static (strict <: the
        // earlier = lower reference index wins ties); slots >= kk stay at +inf and never match
#pragma unroll
        for (int j = KM - 1; j >= 0; --j) {
          if (j < kk) {
            if (j > 0 && d2 < best[j - 1]) {
              best[j] = best[j - 1];
              besti[j] = besti[j - 1];
            } else if (d2 < best[j]) {
              best[j] = d2;
              besti[j] = t0 + r - rbeg;
            }
          }
        }
      }
    }
  }
  if (valid) {
    for (int j = 0; j < kk; ++j) {
      idx[(size_t)q * kk + j] = besti[j];
      if (dist) dist[(size_t)q * kk + j] = FB_SQRT(best[j]);
    }
  }
}

int launch_knn(const double* refs, int ld_refs, const int* ref_off, const double* queries, int ld_queries,
               const int* query_off, int n_segments, int max_queries, int dim, int k, long long* idx,
               double* dist, cudaStream_t stream, const int* ref_seg) {
  if (!(dim >= 1 && dim <= KNN_MAX_DIM && k >= 1 && k <= KNN_MAX_K && n_segments > 0 && max_queries > 0)) {
    set_error("knn: need 1 <= dim <= %d, 1 <= k <= %d (got dim=%d k=%d)", KNN_MAX_DIM, KNN_MAX_K, dim, k);
    return FB_ERR_ARG;
  }
  dim3 grid(div_up(max_queries, KNN_THREADS), n_segments);
  const size_t smem = sizeof(double) * KNN_TILE * dim;
  if (smem > 48 * 1024) {
    // per device and per function: set on every call that needs it (cheap), never cached process-wide
    const int cap = (int)(sizeof(double) * KNN_TILE * KNN_MAX_DIM);
    FB_CUDA(cudaFuncSetAttribute(k_knn<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    FB_CUDA(cudaFuncSetAttribute(k_knn<0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    FB_CUDA(cudaFuncSetAttribute(k_knn<0, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
  }
#define FB_KNN(DD, KK) \
  k_knn<DD, KK><<<grid, KNN_THREADS, smem, stream>>>(refs, ld_refs, ref_off, ref_seg, queries, ld_queries, query_off, dim, \
                                                     k, idx, dist)
  if (dim == 3 && k == 1)
    FB_KNN(3, 1);
  else if (dim == 3 && k == 3)
    FB_KNN(3, 3);
  else if (k == 1)
    FB_KNN(0, 1);
  else if (k == 3)
    FB_KNN(0, 3);
  else
    FB_KNN(0, 0);
#undef FB_KNN
  FB_COUNT_LAUNCH(1);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("knn: launch failed: %s", cudaGetErrorString(e));
    return FB_ERR_CUDA;
  }
  return FB_OK;
}

// focusr.py:415-426.  numpy: weighting = 1/d; sum(points[idx]*w, axis=0) / sum(w), both left to right.
__global__ void k_weighted_positions(const long long* __restrict__ idx3, const double* __restrict__ dist3,
                                     const double* __restrict__ target_points, const int* __restrict__ point_base,
                                     int n, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long base = point_base ? point_base[i] : 0;
  const double d0 = dist3[3 * (size_t)i], d1 = dist3[3 * (size_t)i + 1], d2 = dist3[3 * (size_t)i + 2];
  const long long i0 = idx3[3 * (size_t)i] + base, i1 = idx3[3 * (size_t)i + 1] + base, i2 = idx3[3 * (size_t)i + 2] + base;
  double r[3];
  if (d0 == 0.0 || d1 == 0.0 || d2 == 0.0) {
    const long long c = d0 == 0.0 ? i0 : (d1 == 0.0 ? i1 : i2);  // first coincident neighbour
    for (int a = 0; a < 3; ++a) r[a] = target_points[3 * c + a];
  } else {
    const double w0 = FB_DIV(1.0, d0), w1 = FB_DIV(1.0, d1), w2 = FB_DIV(1.0, d2);
    const double den = FB_ADD(FB_ADD(w0, w1), w2);
    for (int a = 0; a < 3; ++a) {
      const double num = FB_ADD(FB_ADD(FB_MUL(target_points[3 * i0 + a], w0), FB_MUL(target_points[3 * i1 + a], w1)),
                                FB_MUL(target_points[3 * i2 + a], w2));
      r[a] = FB_DIV(num, den);
    }
  }
  for (int a = 0; a < 3; ++a) out[3 * (size_t)i + a] = r[a];
}

}  // namespace fb

namespace fb {
// out[q][r] = sqrt(sum_d (a_q[d] - b_r[d])^2), sequential sum without FMA (scipy cdist's arithmetic)
__global__ void k_cdist(const double* __restrict__ a, int na, const double* __restrict__ b, int nb, int dim, double* __restrict__ out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x, q = blockIdx.y;
  if (r >= nb) return;
  const double* pa = a + (size_t)q * dim;
  const double* pb = b + (size_t)r * dim;
  const double d0 = FB_SUB(pa[0], pb[0]);
  double s = FB_MUL(d0, d0);
  for (int c = 1; c < dim; ++c) {
    const double d = FB_SUB(pa[c], pb[c]);
    s = FB_ADD(s, FB_MUL(d, d));
  }
  out[(size_t)q * nb + r] = sqrt(s);
}
}  // namespace fb

using namespace fb;

extern "C" {

int focusr_cdist(const double* a, int n_a, const double* b, int n_b, int dim, double* out, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_a > 0 && n_b > 0 && dim > 0 && n_a <= 65535, "cdist: bad sizes (at most 65535 rows)");
  dim3 grid(div_up(n_b, 256), n_a);
  k_cdist<<<grid, 256, 0, stream>>>(a, n_a, b, n_b, dim, out);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

size_t focusr_knn_workspace_bytes(int n_refs_total, int n_queries_total, int n_segments, int dim) {
  return knn_pruned_workspace_bytes(n_refs_total, n_queries_total, n_segments, dim);
}

int focusr_knn(const double* refs, int ld_refs, const int* ref_off, int n_refs_total, int max_refs_per_segment,
               const double* queries, int ld_queries, const int* query_off, int n_queries_total,
               int max_queries_per_segment, int n_segments, int dim, int k, long long* idx, double* dist,
               void* workspace, size_t workspace_bytes, focusr_stream_t stream) {
  FB_REQUIRE(n_segments > 0 && n_refs_total > 0 && n_queries_total > 0, "knn: empty input");
  if (workspace != nullptr && knn_pruned_applicable(max_refs_per_segment, max_queries_per_segment, dim, k))
    return launch_knn_pruned(refs, ld_refs, ref_off, queries, ld_queries, query_off, n_segments,
                             max_refs_per_segment, max_queries_per_segment, n_refs_total, n_queries_total, dim, k,
                             idx, dist, workspace, workspace_bytes, (cudaStream_t)stream);
  return launch_knn(refs, ld_refs, ref_off, queries, ld_queries, query_off, n_segments,
                    max_queries_per_segment, dim, k, idx, dist, (cudaStream_t)stream);
}

size_t focusr_knn_mapped_workspace_bytes(int n_refs_total, int n_queries_total, int n_ref_segments, int dim) {
  return knn_pruned_workspace_bytes(n_refs_total, n_queries_total, n_ref_segments, dim);
}

int focusr_knn_mapped(const double* refs, int ld_refs, const int* ref_off, int n_refs_total, int n_ref_segments,
                      int max_refs_per_segment, const double* queries, int ld_queries, const int* query_off,
                      int n_queries_total, int max_queries_per_segment, int n_query_segments, const int* ref_seg,
                      const int* ref_seg_host, int dim, int k, long long* idx, double* dist, void* workspace,
                      size_t workspace_bytes, focusr_stream_t stream) {
  FB_REQUIRE(n_ref_segments > 0 && n_query_segments > 0 && n_refs_total > 0 && n_queries_total > 0, "knn_mapped: empty input");
  FB_REQUIRE(ref_seg != nullptr && ref_seg_host != nullptr, "knn_mapped: ref_seg and its host copy are required");
  for (int s = 0; s < n_query_segments; ++s)
    FB_REQUIRE(ref_seg_host[s] >= 0 && ref_seg_host[s] < n_ref_segments,
               "knn_mapped: query segment %d maps to reference segment %d, outside [0, %d)", s, ref_seg_host[s],
               n_ref_segments);
  if (workspace != nullptr && knn_pruned_applicable(max_refs_per_segment, max_queries_per_segment, dim, k))
    return launch_knn_pruned(refs, ld_refs, ref_off, queries, ld_queries, query_off, n_query_segments,
                             max_refs_per_segment, max_queries_per_segment, n_refs_total, n_queries_total, dim, k,
                             idx, dist, workspace, workspace_bytes, (cudaStream_t)stream, n_ref_segments, ref_seg);
  return launch_knn(refs, ld_refs, ref_off, queries, ld_queries, query_off, n_query_segments,
                    max_queries_per_segment, dim, k, idx, dist, (cudaStream_t)stream, ref_seg);
}

int focusr_weighted_positions(const long long* idx3, const double* dist3, const double* target_points,
                              const int* point_base, int n_queries, double* out, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_queries > 0, "weighted_positions: empty");
  k_weighted_positions<<<div_up(n_queries, 256), 256, 0, stream>>>(idx3, dist3, target_points, point_base,
                                                                   n_queries, out);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}
}
