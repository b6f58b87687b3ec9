// K4, pruned variant: the same exact fp64 k-NN as knn.cu (identical distance arithmetic, identical
// tie rule: lower ORIGINAL index wins), but references and queries of every segment are first put
// in Morton order, references are cut into tiles of 128 with a bounding box, and a query skips a
// tile whose box is farther than its current k-th best.  Every reference is either scanned with
// the exact arithmetic or excluded by a (safely rounded-down) lower bound, so the result is
// bit-identical to brute force; only the number of FP64 distance evaluations drops (the brute
// force kernel is FP64-pipe-bound, profiles/r1_summary.md).
//
// Per segment (<= 16384 points a side): one CTA sorts 64-bit (morton << 32 | index) keys with a
// bitonic network in shared memory -- the "sort" of north_star's sort/segment-reduce vocabulary --
// and writes the permuted reference coordinates and tile boxes.
//
// Mapped form (focusr_knn_mapped): query segment s searches reference segment ref_seg[s], so several query segments
// can share one reference segment.  Each reference segment is boxed, sorted and tiled once, in a box of its own
// references; the queries of s are keyed in the box of ref_seg[s].  ref_seg = NULL is the identity map (focusr_knn),
// whose box is that of the segment's references and queries, as before.
#include <limits.h>

#include "common.cuh"
#include "knn.cuh"
#include "morton.cuh"
#include "rowops.h"

namespace fb {

// Tile sizes, measured at bench shape (128 segments of 15 212 x 15 212, d = 3; tools/knn_ab.sh, gpurun_out/r2g_knn_ab.log),
// k = 1 / k = 3 in ms, distance evaluations per query in brackets:
//   references per tile x queries per CTA   128 x 128: 2.76 / 4.33 (359 / 440)     64 x 128: 2.59 / 3.90 (209 / 261)
//   64 x 64: 2.12 / 3.21 (189 / 244)   128 x 64: 2.39 / 3.79   32 x 64: 2.50 / 3.48 (109 / 145)   256 x 128: 3.63 / 5.65
// Smaller reference tiles prune more but cost a box test and a barrier each; fewer queries per CTA shrink the union of
// tiles the CTA has to stage.
#ifndef FB_PK_TR
#define FB_PK_TR 64
#endif
#ifndef FB_PK_TQ
#define FB_PK_TQ 64
#endif
constexpr int PK_TR = FB_PK_TR;  // references per tile (A/B builds: tools/knn_ab.sh)
constexpr int PK_TQ = FB_PK_TQ;  // queries per CTA
constexpr int PK_SORT_MAX = 16384;
constexpr int PK_MAX_DIM = 32;

// bounding box of refs U queries of each segment over the first min(dim,3) coordinates (refs alone: query_off = NULL)
__global__ void __launch_bounds__(256)
k_pk_bbox(const double* __restrict__ refs, int ldr, const int* __restrict__ ref_off,
          const double* __restrict__ queries, int ldq, const int* __restrict__ query_off, int dim,
          double* __restrict__ seg_lo, double* __restrict__ seg_inv) {
  const int seg = blockIdx.x;
  double mn[3] = {1e300, 1e300, 1e300}, mx[3] = {-1e300, -1e300, -1e300};
  const int nd = dim < 3 ? dim : 3;
  for (int r = ref_off[seg] + threadIdx.x; r < ref_off[seg + 1]; r += blockDim.x)
    for (int c = 0; c < nd; ++c) {
      const double v = refs[(size_t)r * ldr + c];
      mn[c] = fmin(mn[c], v);
      mx[c] = fmax(mx[c], v);
    }
  if (query_off)
    for (int r = query_off[seg] + threadIdx.x; r < query_off[seg + 1]; r += blockDim.x)
      for (int c = 0; c < nd; ++c) {
        const double v = queries[(size_t)r * ldq + c];
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
  if (threadIdx.x < 3) {
    const int c = threadIdx.x;
    const double ext = smx[c][0] - smn[c][0];
    seg_lo[3 * seg + c] = smn[c][0];
    seg_inv[3 * seg + c] = (ext > 0.0 && ext < 1e300) ? 1024.0 / ext : 0.0;
  }
}

// grid (max(reference, query segments), 2): y = 0 sorts the references of reference segment x, y = 1 the queries of
// query segment x, keyed in the box of the reference segment they search (ref_seg[x], or x when ref_seg is NULL).
__global__ void __launch_bounds__(1024)
k_pk_sort(const double* __restrict__ refs, int ldr, const int* __restrict__ ref_off, int n_ref_segments,
          const double* __restrict__ queries, int ldq, const int* __restrict__ query_off, int n_query_segments,
          const int* __restrict__ ref_seg, int dim, const double* __restrict__ seg_lo, const double* __restrict__ seg_inv,
          int p2,
          double* __restrict__ refs_sorted, int* __restrict__ ref_orig, int* __restrict__ q_orig,
          unsigned* __restrict__ q_key, double* __restrict__ tile_lo, double* __restrict__ tile_hi,
          unsigned* __restrict__ tile_key) {
  extern __shared__ unsigned long long keys[];
  const int seg = blockIdx.x, which = blockIdx.y;
  if (seg >= (which == 0 ? n_ref_segments : n_query_segments)) return;
  const int box = (which == 1 && ref_seg) ? ref_seg[seg] : seg;
  const double* src = which == 0 ? refs : queries;
  const int ld = which == 0 ? ldr : ldq;
  const int base = which == 0 ? ref_off[seg] : query_off[seg];
  const int n = (which == 0 ? ref_off[seg + 1] : query_off[seg + 1]) - base;
  const double lo[3] = {seg_lo[3 * box], seg_lo[3 * box + 1], seg_lo[3 * box + 2]};
  const double inv[3] = {seg_inv[3 * box], seg_inv[3 * box + 1], seg_inv[3 * box + 2]};
  for (int e = threadIdx.x; e < p2; e += blockDim.x) {
    unsigned long long k = ~0ull;
    if (e < n) k = ((unsigned long long)morton3(src + (size_t)(base + e) * ld, dim, lo, inv) << 32) | (unsigned)e;
    keys[e] = k;
  }
  __syncthreads();
  for (int k = 2; k <= p2; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < p2; t += blockDim.x) {
        const int ixj = t ^ j;
        if (ixj > t) {
          const unsigned long long a = keys[t], b = keys[ixj];
          if ((a > b) == ((t & k) == 0)) {
            keys[t] = b;
            keys[ixj] = a;
          }
        }
      }
      __syncthreads();
    }
  if (which == 1) {
    for (int pos = threadIdx.x; pos < n; pos += blockDim.x) {
      q_orig[base + pos] = (int)(keys[pos] & 0xffffffffu);
      q_key[base + pos] = (unsigned)(keys[pos] >> 32);
    }
    return;
  }
  for (long long t = threadIdx.x; t < (long long)n * dim; t += blockDim.x) {
    const int pos = (int)(t / dim), c = (int)(t % dim);
    const int orig = (int)(keys[pos] & 0xffffffffu);
    refs_sorted[(size_t)(base + pos) * dim + c] = src[(size_t)(base + orig) * ld + c];
  }
  for (int pos = threadIdx.x; pos < n; pos += blockDim.x) ref_orig[base + pos] = (int)(keys[pos] & 0xffffffffu);
  __syncthreads();  // refs_sorted of this segment is complete and visible to the block
  const int ntiles = (n + PK_TR - 1) / PK_TR;
  const int tbase = base / PK_TR + seg;
  for (int t = threadIdx.x; t < ntiles * dim; t += blockDim.x) {
    const int tile = t / dim, c = t % dim;
    const int r0 = tile * PK_TR, r1 = min(n, r0 + PK_TR);
    double mn = 1e300, mx = -1e300;
    for (int r = r0; r < r1; ++r) {
      const double v = refs_sorted[(size_t)(base + r) * dim + c];
      mn = fmin(mn, v);
      mx = fmax(mx, v);
    }
    tile_lo[(size_t)(tbase + tile) * dim + c] = mn;
    tile_hi[(size_t)(tbase + tile) * dim + c] = mx;
    if (c == 0) tile_key[tbase + tile] = (unsigned)(keys[r0] >> 32);
  }
}

// qc[c] with a run-time c (the query coordinates live in registers: a select chain for the small fixed dimensions)
template <int DM>
__device__ __forceinline__ double qc_at(const double (&qc)[DM], int c) {
  double v = qc[0];
#pragma unroll
  for (int i = 1; i < DM; ++i)
    if (i == c) v = qc[i];
  return v;
}

__device__ __forceinline__ bool lex_lt(double d2, int id, double bd, int bi) {
  return d2 < bd || (d2 == bd && id < bi);
}

// live profile: (query, reference) distance evaluations of the pruned search since the last reset (one atomic per warp
// at kernel end), so that bench.py can state the KNN's rate as a fraction of the FP64 instruction peak
__device__ unsigned long long g_pk_evals = 0ull;

unsigned long long pk_evals_read_and_maybe_reset(bool reset) {
  unsigned long long v = 0ull;
  cudaMemcpyFromSymbol(&v, g_pk_evals, sizeof(v));
  if (reset) {
    const unsigned long long z = 0ull;
    cudaMemcpyToSymbol(g_pk_evals, &z, sizeof(z));
  }
  return v;
}

// grid (query blocks, query segments): query segment blockIdx.y searches reference segment ref_seg[blockIdx.y] (MAP)
// or reference segment blockIdx.y.  MAP is a template parameter so that the identity map of focusr_knn keeps its
// register count (a loaded segment index stays live where blockIdx.y is re-read: +8 registers at d = 3).
template <int D, int K, bool MAP>
__global__ void __launch_bounds__(PK_TQ)
k_pk_search(const double* __restrict__ refs_sorted, const int* __restrict__ ref_orig, const int* __restrict__ ref_off,
            const int* __restrict__ ref_seg, const double* __restrict__ queries, int ldq, const int* __restrict__ query_off,
            const int* __restrict__ q_orig, const unsigned* __restrict__ q_key, const double* __restrict__ tile_lo,
            const double* __restrict__ tile_hi, const unsigned* __restrict__ tile_key, int dim_rt, int k_rt,
            long long* __restrict__ idx, double* __restrict__ dist) {
  extern __shared__ double tile[];  // [PK_TR][dim] coordinates, then PK_TR original indices
  const int dim = D > 0 ? D : dim_rt;
  const int kk = K > 0 ? K : k_rt;
  constexpr int DM = D > 0 ? D : PK_MAX_DIM;
  constexpr int KM = K > 0 ? K : 8;
  int* tile_idx = reinterpret_cast<int*>(tile + PK_TR * dim);
  __shared__ int s_j0;
  __shared__ unsigned char s_flag[PK_SORT_MAX / PK_TR];         // tiles of the segment that can matter to this CTA
  __shared__ double s_red[2 * PK_MAX_DIM + 1][PK_TQ / 32];      // per-warp partials: query bounding box, largest k-th best
  const int seg = blockIdx.y;
  const int qbase = query_off[seg];
  const int q0 = qbase + blockIdx.x * PK_TQ, qend = query_off[seg + 1];
  if (q0 >= qend) return;
  const int rseg = MAP ? ref_seg[seg] : seg;
  const int rbase = ref_off[rseg], nr = ref_off[rseg + 1] - rbase;
  const int ntiles = (nr + PK_TR - 1) / PK_TR;
  const int tbase = rbase / PK_TR + rseg;
  const int pos = q0 + threadIdx.x;
  const bool valid = pos < qend;
  const int qo = valid ? q_orig[pos] : 0;
  double qc[DM];
#pragma unroll
  for (int c = 0; c < DM; ++c) qc[c] = (valid && c < dim) ? queries[(size_t)(qbase + qo) * ldq + c] : 0.0;
  double best[KM];
  int besti[KM];
#pragma unroll
  for (int j = 0; j < KM; ++j) {
    best[j] = __longlong_as_double(0x7ff0000000000000LL);
    besti[j] = INT_MAX;
  }
  if (threadIdx.x == 0) {
    // reference tile whose Morton range holds the middle query of this CTA
    const unsigned key = q_key[q0 + (min(qend, q0 + PK_TQ) - q0) / 2];
    int lo = 0, hi = ntiles - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (tile_key[tbase + mid] <= key)
        lo = mid;
      else
        hi = mid - 1;
    }
    s_j0 = lo;
  }
  __syncthreads();
  int left = s_j0, right = s_j0 + 1;
  unsigned n_eval = 0;
  for (int t = 0; t < ntiles; ++t) {
    int j;
    if ((((t & 1) == 0) && left >= 0) || right >= ntiles)
      j = left--;
    else
      j = right++;
    if (t == 1) {
      // The home tile has been scanned: every query of the CTA holds a k-th best.  A tile can only matter to a query
      // whose box distance to it is <= that query's k-th best, hence only if the distance between the tile's box and the
      // bounding box of ALL queries of the CTA (a lower bound of every such distance; every floating-point step below
      // is monotone, so it is one in rounded arithmetic too) is <= the LARGEST k-th best of the CTA.  One thread per
      // tile marks those tiles; the loop then visits only them (~8 of ~120 on a 15k-vertex surface) instead of paying
      // a box test per thread and a barrier for every tile of the segment.
      double rmax = valid ? best[kk - 1] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) rmax = fmax(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
      if ((threadIdx.x & 31) == 0) s_red[2 * PK_MAX_DIM][threadIdx.x >> 5] = rmax;
      for (int c = 0; c < dim; ++c) {
        double lo = valid ? qc_at(qc, c) : __longlong_as_double(0x7ff0000000000000LL);
        double hi = valid ? qc_at(qc, c) : __longlong_as_double(0xfff0000000000000LL);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
          hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if ((threadIdx.x & 31) == 0) {
          s_red[2 * c][threadIdx.x >> 5] = lo;
          s_red[2 * c + 1][threadIdx.x >> 5] = hi;
        }
      }
      __syncthreads();
      constexpr int NW = PK_TQ / 32;
      double r2 = s_red[2 * PK_MAX_DIM][0];
#pragma unroll
      for (int w = 1; w < NW; ++w) r2 = fmax(r2, s_red[2 * PK_MAX_DIM][w]);
      for (int jt = threadIdx.x; jt < ntiles; jt += PK_TQ) {
        double lbb = 0.0;
        for (int c = 0; c < dim; ++c) {
          double qlo = s_red[2 * c][0], qhi = s_red[2 * c + 1][0];
#pragma unroll
          for (int w = 1; w < NW; ++w) {
            qlo = fmin(qlo, s_red[2 * c][w]);
            qhi = fmax(qhi, s_red[2 * c + 1][w]);
          }
          const double g = fmax(fmax(tile_lo[(size_t)(tbase + jt) * dim + c] - qhi, qlo - tile_hi[(size_t)(tbase + jt) * dim + c]), 0.0);
          lbb += g * g;
        }
        lbb *= (1.0 - 1e-12);
        s_flag[jt] = lbb <= r2 ? 1 : 0;
      }
      __syncthreads();
    }
    if (t >= 1 && !s_flag[j]) continue;   // uniform over the CTA
    // squared distance from the query to the tile's box, rounded down so it never exceeds the
    // distance the exact arithmetic below would compute for any reference inside the box
    double lb = 0.0;
    const double* blo = tile_lo + (size_t)(tbase + j) * dim;
    const double* bhi = tile_hi + (size_t)(tbase + j) * dim;
#pragma unroll
    for (int c = 0; c < DM; ++c)
      if (c < dim) {
        const double g = fmax(fmax(blo[c] - qc[c], qc[c] - bhi[c]), 0.0);
        lb += g * g;
      }
    lb *= (1.0 - 1e-12);
    const bool need = valid && lb <= best[kk - 1];
    if (!__syncthreads_or(need)) continue;
    const int r0 = j * PK_TR, cnt = min(PK_TR, nr - r0);
    for (int e = threadIdx.x; e < cnt * dim; e += PK_TQ) tile[e] = refs_sorted[(size_t)(rbase + r0) * dim + e];
    for (int e = threadIdx.x; e < cnt; e += PK_TQ) tile_idx[e] = ref_orig[rbase + r0 + e];
    __syncthreads();
    if (need) {
      n_eval += cnt;
      for (int r = 0; r < cnt; ++r) {
        const double* rp = tile + r * dim;
        double d2 = 0.0;
#pragma unroll
        for (int c = 0; c < DM; ++c)
          if (c < dim) {
            const double df = FB_SUB(qc[c], rp[c]);
            d2 = FB_ADD(d2, FB_MUL(df, df));
          }
        if (!lex_lt(d2, tile_idx[r], best[kk - 1], besti[kk - 1])) continue;
        const int id = tile_idx[r];
#pragma unroll
        for (int jj = KM - 1; jj >= 0; --jj) {
          if (jj < kk) {
            if (jj > 0 && lex_lt(d2, id, best[jj - 1], besti[jj - 1])) {
              best[jj] = best[jj - 1];
              besti[jj] = besti[jj - 1];
            } else if (lex_lt(d2, id, best[jj], besti[jj])) {
              best[jj] = d2;
              besti[jj] = id;
            }
          }
        }
      }
    }
    __syncthreads();  // everyone is done with the tile before the next load overwrites it
  }
  {  // profile counter: one atomic per warp
    unsigned tot = n_eval;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
    if ((threadIdx.x & 31) == 0 && tot) atomicAdd(&g_pk_evals, (unsigned long long)tot);
  }
  if (valid) {
    const size_t o = (size_t)(qbase + qo) * kk;
    for (int j = 0; j < kk; ++j) {
      idx[o + j] = besti[j] == INT_MAX ? -1 : besti[j];
      if (dist) dist[o + j] = FB_SQRT(best[j]);
    }
  }
}

static int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

size_t knn_pruned_workspace_bytes(long long n_refs, long long n_queries, int n_segments, int dim) {
  const size_t tiles = (size_t)(n_refs / PK_TR) + n_segments + 1;
  size_t b = 0;
  b += align_up(sizeof(double) * 6 * (size_t)n_segments);
  b += align_up(sizeof(double) * (size_t)n_refs * dim);
  b += align_up(sizeof(int) * (size_t)n_refs);
  b += align_up(sizeof(int) * (size_t)n_queries) * 2;
  b += align_up(sizeof(double) * tiles * dim) * 2;
  b += align_up(sizeof(unsigned) * tiles);
  return b + 1024;
}

bool knn_pruned_applicable(int max_refs, int max_queries, int dim, int k) {
  return max_refs <= PK_SORT_MAX && max_queries <= PK_SORT_MAX && dim <= PK_MAX_DIM && k <= 8 && max_refs >= 4 * PK_TR;
}

int launch_knn_pruned(const double* refs, int ld_refs, const int* ref_off, const double* queries, int ld_queries,
                      const int* query_off, int n_segments, int max_refs, int max_queries, long long n_refs,
                      long long n_queries, int dim, int k, long long* idx, double* dist, void* workspace,
                      size_t workspace_bytes, cudaStream_t stream, int n_ref_segments, const int* ref_seg) {
  if (!ref_seg) n_ref_segments = n_segments;
  Carver cv(workspace, workspace_bytes);
  const size_t tiles = (size_t)(n_refs / PK_TR) + n_ref_segments + 1;
  double* seg_lo = cv.take<double>(3 * (size_t)n_ref_segments);
  double* seg_inv = cv.take<double>(3 * (size_t)n_ref_segments);
  double* refs_sorted = cv.take<double>((size_t)n_refs * dim);
  int* ref_orig = cv.take<int>((size_t)n_refs);
  int* q_orig = cv.take<int>((size_t)n_queries);
  unsigned* q_key = cv.take<unsigned>((size_t)n_queries);
  double* tile_lo = cv.take<double>(tiles * dim);
  double* tile_hi = cv.take<double>(tiles * dim);
  unsigned* tile_key = cv.take<unsigned>(tiles);
  if (!cv.ok()) {
    set_error("knn: workspace too small (%zu < %zu)", workspace_bytes, cv.used);
    return FB_ERR_WORKSPACE;
  }
  k_pk_bbox<<<n_ref_segments, 256, 0, stream>>>(refs, ld_refs, ref_off, queries, ld_queries, ref_seg ? nullptr : query_off,
                                                dim, seg_lo, seg_inv);
  const int p2 = next_pow2(max_refs > max_queries ? max_refs : max_queries);
  const size_t sort_smem = sizeof(unsigned long long) * (size_t)p2;
  // the opt-in is per device and per function: set whenever it is needed (cheap), never cached process-wide
  if (sort_smem > 48 * 1024) FB_CUDA(cudaFuncSetAttribute(k_pk_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_smem));
  k_pk_sort<<<dim3(n_ref_segments > n_segments ? n_ref_segments : n_segments, 2), 1024, sort_smem, stream>>>(
      refs, ld_refs, ref_off, n_ref_segments, queries, ld_queries, query_off, n_segments, ref_seg, dim, seg_lo, seg_inv,
      p2, refs_sorted, ref_orig, q_orig, q_key, tile_lo, tile_hi, tile_key);
  dim3 grid(div_up(max_queries, PK_TQ), n_segments);
  const size_t smem = sizeof(double) * PK_TR * dim + sizeof(int) * PK_TR;
#define FB_PK(DD, KK)                                                                                               \
  do {                                                                                                              \
    if (ref_seg)                                                                                                    \
      k_pk_search<DD, KK, true><<<grid, PK_TQ, smem, stream>>>(refs_sorted, ref_orig, ref_off, ref_seg, queries,      \
                                                               ld_queries, query_off, q_orig, q_key, tile_lo, tile_hi, \
                                                               tile_key, dim, k, idx, dist);                          \
    else                                                                                                            \
      k_pk_search<DD, KK, false><<<grid, PK_TQ, smem, stream>>>(refs_sorted, ref_orig, ref_off, nullptr, queries,    \
                                                                ld_queries, query_off, q_orig, q_key, tile_lo,        \
                                                                tile_hi, tile_key, dim, k, idx, dist);                \
  } while (0)
  if (dim == 3 && k == 1)
    FB_PK(3, 1);
  else if (dim == 3 && k == 3)
    FB_PK(3, 3);
  else if (k == 1)
    FB_PK(0, 1);
  else if (k == 3)
    FB_PK(0, 3);
  else
    FB_PK(0, 0);
#undef FB_PK
  FB_COUNT_LAUNCH(3);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("knn (pruned): launch failed: %s", cudaGetErrorString(e));
    return FB_ERR_CUDA;
  }
  return FB_OK;
}

}  // namespace fb
