// K2: smallest-k eigenpairs of the mesh Laplacian on the B200 -- the CUDA backend of the block
// solver in chfsi_driver.hpp.  Replaces scipy's shift-invert ARPACK + SuperLU call
// (reference graph.py:357-389) with factorisation-free Chebyshev-filtered subspace iteration.
//
// Kernels in this file (the CSR SpMM of the filter itself is in spmm.cu):
//   k_gram    tall-skinny Gram pair G = X^T g X, H = X^T h Z per mesh with FP64 tensor-core
//             DMMA (mma.sync.m8n8k4.f64: tcgen05 has no f64 kind, SURVEY.md section 7.3-8);
//   k_rr_sym  one warp (or CTA) per mesh: Cholesky + congruence + round-robin Jacobi in shared memory;
//   k_rotate  X <- X W (DMMA) fused with the residual norms ||L x - theta x||;
//   k_write_pairs  unit-norm, sign-fixed eigenvectors into the caller's [n_points][ldv] block.
// All reductions use fixed trees / fixed chunk order: results are bit-reproducible run to run.
#include <mutex>
#include <vector>

#include "chfsi_driver.hpp"
#include "nonsym_small.h"
#include "common.cuh"
#include "nccl_dyn.h"
#include "rowops.h"
#include "sell.cuh"
#include "spmm.cuh"

namespace fb {

unsigned long long pk_evals_read_and_maybe_reset(bool reset);  // knn_pruned.cu

constexpr int GRAM_ROWS = 1024;  // rows per CTA (8 warps x 128 rows)
constexpr int GRAM_THREADS = 256;

__device__ __forceinline__ long long dkey(double v) {
  const long long b = __double_as_longlong(v);
  return b >= 0 ? b : (b ^ 0x7fffffffffffffffLL);
}
__device__ __forceinline__ double dkey_inv(long long k) {
  return __longlong_as_double(k >= 0 ? k : (k ^ 0x7fffffffffffffffLL));
}

__global__ void k_bbox_init(long long* lo, long long* hi, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    lo[i] = 0x7fffffffffffffffLL;
    hi[i] = (long long)0x8000000000000000ULL;
  }
}

__global__ void __launch_bounds__(256)
k_bbox(const double* __restrict__ points, const int* __restrict__ mesh_off, long long* lo, long long* hi) {
  const int mesh = blockIdx.y;
  const int r0 = mesh_off[mesh] + blockIdx.x * GRAM_ROWS;
  const int r1 = min(mesh_off[mesh + 1], r0 + GRAM_ROWS);
  long long mn[3] = {0x7fffffffffffffffLL, 0x7fffffffffffffffLL, 0x7fffffffffffffffLL};
  long long mx[3] = {(long long)0x8000000000000000ULL, (long long)0x8000000000000000ULL, (long long)0x8000000000000000ULL};
  for (int r = r0 + threadIdx.x; r < r1; r += blockDim.x)
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const long long k = dkey(points[3 * (size_t)r + a]);
      mn[a] = min(mn[a], k);
      mx[a] = max(mx[a], k);
    }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn[a] = min(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
      mx[a] = max(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
    }
    if ((threadIdx.x & 31) == 0 && r0 < r1) {
      atomicMin(&lo[3 * mesh + a], mn[a]);
      atomicMax(&hi[3 * mesh + a], mx[a]);
    }
  }
}

template <int B>
__global__ void __launch_bounds__(256)
k_init_block(const double* __restrict__ points, const double* __restrict__ degree,
             const int* __restrict__ mesh_off, const long long* __restrict__ lo,
             const long long* __restrict__ hi, double* __restrict__ x, long long row_base) {
  const int mesh = blockIdx.y;
  const int m0 = mesh_off[mesh];
  const int r0 = m0 + blockIdx.x * GRAM_ROWS;
  const int r1 = min(mesh_off[mesh + 1], r0 + GRAM_ROWS);
  if (r0 >= r1) return;
  double c[3], scale = 0.0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double l = dkey_inv(lo[3 * mesh + a]), h = dkey_inv(hi[3 * mesh + a]);
    c[a] = 0.5 * (l + h);
    scale = fmax(scale, 0.5 * (h - l));
  }
  if (!(scale > 0.0)) scale = 1.0;
  for (long long t = threadIdx.x; t < (long long)(r1 - r0) * B; t += blockDim.x) {
    const int r = r0 + (int)(t / B), col = (int)(t % B);
    double v = 0.0;
    if (degree[r] != 0.0) {  // zero-degree rows stay pinned at 0 (exact null vectors, handled analytically)
      const double px = (points[3 * (size_t)r] - c[0]) / scale;
      const double py = (points[3 * (size_t)r + 1] - c[1]) / scale;
      const double pz = (points[3 * (size_t)r + 2] - c[2]) / scale;
      v = start_block_value(col, px, py, pz, (uint32_t)(r - m0 + row_base), 1u);
    }
    x[(size_t)r * B + col] = v;
  }
}

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

// G[p][q] = sum_r X[r][p] g_r X[r][q],  H[p][q] = sum_r X[r][p] h_r Z[r][q]  per (mesh, chunk).
// blockIdx.z picks a group of QT column tiles (8 columns each) so the accumulators fit registers.
// As an MMA: D(8x8) += A(8x4) B(4x8) with A[p][r'] = X[r+r'][p], B[r'][q] = g X[r+r'][q]; for
// m8n8k4 lane l holds A[l>>2][l&3], B[l&3][l>>2] and D[l>>2][2*(l&3)+{0,1}].
template <int B, int QT>
__global__ void __launch_bounds__(GRAM_THREADS)
k_gram(const double* __restrict__ x, const double* __restrict__ z, const double* __restrict__ degree,
       const double* __restrict__ degree_inv, const int* __restrict__ mesh_off, int sym,
       double* __restrict__ partial, int chunks_max) {
  constexpr int PT = B / 8;
  const int mesh = blockIdx.y, chunk = blockIdx.x, q0 = blockIdx.z * QT;
  const int r0 = mesh_off[mesh] + chunk * GRAM_ROWS;
  const int r1 = min(mesh_off[mesh + 1], r0 + GRAM_ROWS);
  if (r0 >= r1) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rr = lane & 3, cc = lane >> 2;
  double accg[PT][QT][2], acch[PT][QT][2];
#pragma unroll
  for (int a = 0; a < PT; ++a)
#pragma unroll
    for (int b = 0; b < QT; ++b) accg[a][b][0] = accg[a][b][1] = acch[a][b][0] = acch[a][b][1] = 0.0;
  const int w0 = r0 + warp * (GRAM_ROWS / 8);
  const int w1 = min(r1, w0 + GRAM_ROWS / 8);
  for (int r = w0; r < w1; r += 4) {
    const int row = r + rr;
    const bool valid = row < w1;
    double gw = 0.0, hw = 0.0;
    if (valid) {
      gw = sym ? degree[row] + 1e-8 : 1.0;
      hw = sym ? 1.0 : degree_inv[row];
    }
    double xs[PT], xq[QT], zq[QT];
#pragma unroll
    for (int t = 0; t < PT; ++t) xs[t] = valid ? x[(size_t)row * B + 8 * t + cc] : 0.0;
#pragma unroll
    for (int t = 0; t < QT; ++t) {
      const bool qv = valid && (q0 + t) < PT;
      xq[t] = qv ? x[(size_t)row * B + 8 * (q0 + t) + cc] * gw : 0.0;
      zq[t] = qv ? z[(size_t)row * B + 8 * (q0 + t) + cc] * hw : 0.0;
    }
#pragma unroll
    for (int a = 0; a < PT; ++a)
#pragma unroll
      for (int b = 0; b < QT; ++b) {
        dmma884(accg[a][b][0], accg[a][b][1], xs[a], xq[b]);
        dmma884(acch[a][b][0], acch[a][b][1], xs[a], zq[b]);
      }
  }
  // deterministic cross-warp reduction: warps add their tiles in warp order
  __shared__ double red[2][B][QT * 8];
  for (int w = 0; w < GRAM_THREADS / 32; ++w) {
    if (warp == w) {
#pragma unroll
      for (int a = 0; a < PT; ++a)
#pragma unroll
        for (int b = 0; b < QT; ++b)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int p = 8 * a + cc, q = 8 * b + 2 * rr + e;
            if (w == 0) {
              red[0][p][q] = accg[a][b][e];
              red[1][p][q] = acch[a][b][e];
            } else {
              red[0][p][q] += accg[a][b][e];
              red[1][p][q] += acch[a][b][e];
            }
          }
    }
    __syncthreads();
  }
  double* dst = partial + ((size_t)mesh * chunks_max + chunk) * 2 * B * B;
  for (int t = threadIdx.x; t < 2 * B * QT * 8; t += GRAM_THREADS) {
    const int mat = t / (B * QT * 8), rem = t % (B * QT * 8);
    const int p = rem / (QT * 8), ql = rem % (QT * 8);
    const int q = 8 * q0 + ql;
    if (q < B) dst[(size_t)mat * B * B + p * B + q] = red[mat][p][ql];
  }
}

// The same Gram pair for WIDE blocks (b >= 64: BASELINE.json configs[4], k up to 64).  There the contraction is bound
// by the FP64 tensor pipe (4 N b^2 flop against 16 b N bytes: 24 flop/B at b = 96), and k_gram above -- operands straight
// from global memory, 14 loads per 24 DMMA, every X tile re-read by each of the b/8 column groups -- kept that pipe only
// 35% busy (profiles/r1_summary.md).  Here a CTA stages 16 rows of X and Z at a time in shared memory (row stride b + 4
// doubles: the 4 rows x 8 columns of a fragment load fall into distinct banks), the next stage is already in flight in
// registers while the current one is multiplied, and the 8 warps split the output tiles 4 (p) x 2 (q) so that nothing
// has to be reduced across warps: every warp writes its own tiles of the (mesh, chunk) partial.  blockIdx.z cuts the q
// tiles in three so that one 100k-vertex mesh (98 chunks) still fills the 148 SMs twice.
constexpr int GW_R = 16;   // rows per stage
constexpr int GW_ZS = 3;   // q-tile groups (grid.z)
template <int B>
__global__ void __launch_bounds__(GRAM_THREADS, 2)
k_gram_wide(const double* __restrict__ x, const double* __restrict__ z, const double* __restrict__ degree,
            const double* __restrict__ degree_inv, const int* __restrict__ mesh_off, int sym,
            double* __restrict__ partial, int chunks_max) {
  constexpr int PT = B / 8, QZ = (PT + GW_ZS - 1) / GW_ZS, PW = (PT + 3) / 4, QW = (QZ + 1) / 2;
  constexpr int LD = B + 4;
  constexpr int V2 = GW_R * B / 2, NV = (V2 + GRAM_THREADS - 1) / GRAM_THREADS;
  __shared__ __align__(16) double sx[GW_R][LD];
  __shared__ __align__(16) double sz[GW_R][LD];
  __shared__ double sg[GW_R], sh[GW_R];
  const int mesh = blockIdx.y, chunk = blockIdx.x;
  const int r0 = mesh_off[mesh] + chunk * GRAM_ROWS;
  const int r1 = min(mesh_off[mesh + 1], r0 + GRAM_ROWS);
  if (r0 >= r1) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rr = lane & 3, cc = lane >> 2;
  const int p_first = (warp >> 1) * PW;
  const int q_first = blockIdx.z * QZ + (warp & 1) * QW;
  const int q_lim = min(PT, ((int)blockIdx.z + 1) * QZ);
  double accg[PW][QW][2], acch[PW][QW][2];
#pragma unroll
  for (int a = 0; a < PW; ++a)
#pragma unroll
    for (int b = 0; b < QW; ++b) accg[a][b][0] = accg[a][b][1] = acch[a][b][0] = acch[a][b][1] = 0.0;
  double2 px[NV], pz[NV];
  double pg = 0.0, ph = 0.0;
  auto fetch = [&](int rs) {
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int e = (int)threadIdx.x + v * GRAM_THREADS;
      px[v] = make_double2(0.0, 0.0);
      pz[v] = make_double2(0.0, 0.0);
      if (e < V2) {
        const int row = rs + (2 * e) / B, col = (2 * e) % B;
        if (row < r1) {
          px[v] = __ldg(reinterpret_cast<const double2*>(x + (size_t)row * B + col));
          pz[v] = __ldg(reinterpret_cast<const double2*>(z + (size_t)row * B + col));
        }
      }
    }
    pg = ph = 0.0;
    if ((int)threadIdx.x < GW_R && rs + (int)threadIdx.x < r1) {
      const int row = rs + (int)threadIdx.x;
      pg = sym ? degree[row] + 1e-8 : 1.0;
      ph = sym ? 1.0 : degree_inv[row];
    }
  };
  fetch(r0);
  for (int rs = r0; rs < r1; rs += GW_R) {
    __syncthreads();  // the previous stage has been consumed
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int e = (int)threadIdx.x + v * GRAM_THREADS;
      if (e < V2) {
        const int lr = (2 * e) / B, col = (2 * e) % B;
        *reinterpret_cast<double2*>(&sx[lr][col]) = px[v];
        *reinterpret_cast<double2*>(&sz[lr][col]) = pz[v];
      }
    }
    if ((int)threadIdx.x < GW_R) {
      sg[threadIdx.x] = pg;
      sh[threadIdx.x] = ph;
    }
    __syncthreads();
    if (rs + GW_R < r1) fetch(rs + GW_R);  // in flight while this stage is multiplied
#pragma unroll
    for (int kk = 0; kk < GW_R; kk += 4) {
      const int lr = kk + rr;
      const double gw = sg[lr], hw = sh[lr];
      double a[PW], bg[QW], bh[QW];
#pragma unroll
      for (int t = 0; t < PW; ++t) a[t] = (p_first + t < PT) ? sx[lr][8 * (p_first + t) + cc] : 0.0;
#pragma unroll
      for (int t = 0; t < QW; ++t) {
        const bool ok = q_first + t < q_lim;
        bg[t] = ok ? sx[lr][8 * (q_first + t) + cc] * gw : 0.0;
        bh[t] = ok ? sz[lr][8 * (q_first + t) + cc] * hw : 0.0;
      }
#pragma unroll
      for (int t = 0; t < PW; ++t)
#pragma unroll
        for (int u = 0; u < QW; ++u) {
          dmma884(accg[t][u][0], accg[t][u][1], a[t], bg[u]);
          dmma884(acch[t][u][0], acch[t][u][1], a[t], bh[u]);
        }
    }
  }
  double* dst = partial + ((size_t)mesh * chunks_max + chunk) * 2 * B * B;
#pragma unroll
  for (int t = 0; t < PW; ++t)
#pragma unroll
    for (int u = 0; u < QW; ++u) {
      if (p_first + t >= PT || q_first + u >= q_lim) continue;
      const int p = 8 * (p_first + t) + cc, q = 8 * (q_first + u) + 2 * rr;
      *reinterpret_cast<double2*>(dst + (size_t)p * B + q) = make_double2(accg[t][u][0], accg[t][u][1]);
      *reinterpret_cast<double2*>(dst + (size_t)B * B + (size_t)p * B + q) = make_double2(acch[t][u][0], acch[t][u][1]);
    }
}

// One warp (NT = 32, many small meshes in flight) or one CTA (NT = 256, large blocks) per mesh: sum
// the chunk partials in chunk order, then the b x b Rayleigh-Ritz step in shared memory
// (Cholesky, congruence, round-robin Jacobi: dense_small.h).
template <int NT>
__global__ void __launch_bounds__(NT)
k_rr_sym(const double* __restrict__ partial, int chunks_max, const int* __restrict__ mesh_off, int B,
         double* __restrict__ w_out, double* __restrict__ theta_out, int* __restrict__ info) {
  extern __shared__ double sm[];
  double* g = sm;
  double* h = g + B * B;
  double* y = h + B * B;
  double* th = y + B * B;
  double* rot = th + B;
  double* red = rot + (B + 2);
  int* rank = reinterpret_cast<int*>(red + NT);
  int* pq = rank + B;
  const int mesh = blockIdx.x, tid = threadIdx.x;
  const int nchunks = (mesh_off[mesh + 1] - mesh_off[mesh] + GRAM_ROWS - 1) / GRAM_ROWS;
  const double* src = partial + (size_t)mesh * chunks_max * 2 * B * B;
  for (int e = tid; e < B * B; e += NT) {
    double sg = 0.0, sh = 0.0;
    for (int c = 0; c < nchunks; ++c) {
      sg += src[(size_t)c * 2 * B * B + e];
      sh += src[(size_t)c * 2 * B * B + B * B + e];
    }
    g[e] = sg;
    h[e] = sh;
  }
  __syncthreads();
  int rc;
  if (NT == 32) {
    WarpPar par{tid};
    rc = rayleigh_ritz_sym(g, h, y, w_out + (size_t)mesh * B * B, th, rank, rot, pq, B, par);
  } else {
    BlockPar par{red};
    rc = rayleigh_ritz_sym(g, h, y, w_out + (size_t)mesh * B * B, th, rank, rot, pq, B, par);
  }
  __syncthreads();
  for (int j = tid; j < B; j += NT) theta_out[(size_t)mesh * B + j] = th[j];
  if (tid == 0) info[mesh] = rc;
}

// Non-symmetric adjacency (open / non-manifold meshes): the general b x b Rayleigh-Ritz step, one CTA per mesh, all in
// shared memory (nonsym_small.h has the algorithm; 48 b^2 bytes + scratch, hence b <= 64).  The Cholesky factor is parked
// in `g_save` (global) while its shared-memory space holds the back-substituted vectors.
constexpr int RRN_THREADS = 128;
static size_t rr_nonsym_smem_bytes(int B) {
  return sizeof(double) * 2 * (size_t)B * B + sizeof(Cd) * 2 * (size_t)B * B + nonsym_small_scratch_bytes(B) +
         sizeof(double) * RRN_THREADS;
}
__global__ void __launch_bounds__(RRN_THREADS)
k_rr_nonsym(const double* __restrict__ partial, int chunks_max, const int* __restrict__ mesh_off, int B, int M,
            const double* __restrict__ cut, double* __restrict__ g_save, double* __restrict__ w_out,
            double* __restrict__ theta_out, int* __restrict__ info) {
  extern __shared__ double sm[];
  double* g = sm;
  double* h = g + B * B;
  Cd* Hc = reinterpret_cast<Cd*>(h + B * B);
  Cd* Qc = Hc + B * B;
  unsigned char* scratch = reinterpret_cast<unsigned char*>(Qc + B * B);
  double* red = reinterpret_cast<double*>(scratch + nonsym_small_scratch_bytes(B));
  const int mesh = blockIdx.x, tid = threadIdx.x;
  const int nchunks = (mesh_off[mesh + 1] - mesh_off[mesh] + GRAM_ROWS - 1) / GRAM_ROWS;
  const double* src = partial + (size_t)mesh * chunks_max * 2 * B * B;
  for (int e = tid; e < B * B; e += RRN_THREADS) {
    double sg = 0.0, sh = 0.0;
    for (int c = 0; c < nchunks; ++c) {
      sg += src[(size_t)c * 2 * B * B + e];
      sh += src[(size_t)c * 2 * B * B + B * B + e];
    }
    g[e] = sg;
    h[e] = sh;
  }
  __syncthreads();
  BlockPar par{red};
  const int rc = rr_nonsym_small(g, h, Hc, Qc, g_save + (size_t)mesh * B * B, B, cut[mesh], w_out + (size_t)mesh * B * B,
                                 theta_out + (size_t)mesh * B, info + M + mesh, scratch, par);
  if (tid == 0) info[mesh] = rc;
}

// Non-symmetric path: only the chunk reduction happens on the device; the host does the rest.
__global__ void k_reduce_gh(const double* __restrict__ partial, int chunks_max,
                            const int* __restrict__ mesh_off, int B, double* __restrict__ g_out,
                            double* __restrict__ h_out) {
  const int mesh = blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B * B) return;
  const int nchunks = (mesh_off[mesh + 1] - mesh_off[mesh] + GRAM_ROWS - 1) / GRAM_ROWS;
  const double* src = partial + (size_t)mesh * chunks_max * 2 * B * B;
  double sg = 0.0, sh = 0.0;
  for (int c = 0; c < nchunks; ++c) {
    sg += src[(size_t)c * 2 * B * B + e];
    sh += src[(size_t)c * 2 * B * B + B * B + e];
  }
  g_out[(size_t)mesh * B * B + e] = sg;
  h_out[(size_t)mesh * B * B + e] = sh;
}

// X <- X W in place, Z' = Z W kept in registers, residual sums of dinv*Z' - theta*X' and X'^2.
// D(8 rows x 8 cols) += A(8x4) B(4x8): A[r'][k'] = X[r+r'][k+k'] (lane: r' = l>>2, k' = l&3),
// B[k'][j'] = W[k+k'][j+j'] (lane: k' = l&3, j' = l>>2), D lane: row l>>2, cols 2*(l&3)+{0,1}.
template <int B>
__global__ void __launch_bounds__(GRAM_THREADS)
k_rotate(double* __restrict__ x, const double* __restrict__ z, const double* __restrict__ w,
         const double* __restrict__ theta, const double* __restrict__ degree_inv,
         const int* __restrict__ mesh_off, double* __restrict__ partial_res, int chunks_max,
         float* __restrict__ r_out) {  // r_out != null: the residual block dinv Z' - X' theta, rounded to fp32
  constexpr int WS = (B % 16 == 0) ? B + 8 : B;  // row stride of W in smem: 2-wavefront fragment reads
  constexpr int KS = B / 4, JT = B / 8;
  extern __shared__ double sm[];
  double* ws = sm;                          // [B][WS]
  double* acc = ws + B * WS;                // [8 warps][2][B]
  const int mesh = blockIdx.y, chunk = blockIdx.x;
  const int r0 = mesh_off[mesh] + chunk * GRAM_ROWS;
  const int r1 = min(mesh_off[mesh + 1], r0 + GRAM_ROWS);
  if (r0 >= r1) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = threadIdx.x; t < B * B; t += GRAM_THREADS) ws[(t / B) * WS + (t % B)] = w[(size_t)mesh * B * B + t];
  for (int t = threadIdx.x; t < 8 * 2 * B; t += GRAM_THREADS) acc[t] = 0.0;
  __syncthreads();
  const int kq = lane & 3, rq = lane >> 2;
  double* my_num = acc + (warp * 2 + 0) * B;
  double* my_den = acc + (warp * 2 + 1) * B;
  const int w0 = r0 + warp * (GRAM_ROWS / 8);
  const int w1 = min(r1, w0 + GRAM_ROWS / 8);
  for (int rb = w0; rb < w1; rb += 8) {
    const int row = rb + rq;
    const bool valid = row < w1;
    double xa[KS], za[KS];
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      xa[ks] = valid ? x[(size_t)row * B + 4 * ks + kq] : 0.0;
      za[ks] = valid ? z[(size_t)row * B + 4 * ks + kq] : 0.0;
    }
    const double di = valid ? degree_inv[row] : 0.0;
#pragma unroll
    for (int tj = 0; tj < JT; ++tj) {
      double cx0 = 0.0, cx1 = 0.0, cz0 = 0.0, cz1 = 0.0;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const double bf = ws[(4 * ks + kq) * WS + 8 * tj + rq];
        dmma884(cx0, cx1, xa[ks], bf);
        dmma884(cz0, cz1, za[ks], bf);
      }
      const int c0 = 8 * tj + 2 * kq;
      if (valid) *reinterpret_cast<double2*>(x + (size_t)row * B + c0) = make_double2(cx0, cx1);
      const double t0 = theta[(size_t)mesh * B + c0], t1 = theta[(size_t)mesh * B + c0 + 1];
      const double e0 = di * cz0 - t0 * cx0, e1 = di * cz1 - t1 * cx1;
      if (r_out && valid) *reinterpret_cast<float2*>(r_out + (size_t)row * B + c0) = make_float2((float)e0, (float)e1);
      double n0 = e0 * e0, n1 = e1 * e1, d0 = cx0 * cx0, d1 = cx1 * cx1;
      // sum over the 8 rows of the tile (lanes with equal l&3), fixed tree
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) {
        n0 += __shfl_xor_sync(0xffffffffu, n0, o);
        n1 += __shfl_xor_sync(0xffffffffu, n1, o);
        d0 += __shfl_xor_sync(0xffffffffu, d0, o);
        d1 += __shfl_xor_sync(0xffffffffu, d1, o);
      }
      if (rq == 0) {
        my_num[c0] += n0;
        my_num[c0 + 1] += n1;
        my_den[c0] += d0;
        my_den[c0 + 1] += d1;
      }
    }
    __syncwarp();
  }
  __syncthreads();
  double* dst = partial_res + ((size_t)mesh * chunks_max + chunk) * 2 * B;
  for (int t = threadIdx.x; t < 2 * B; t += GRAM_THREADS) {
    double s = 0.0;
    for (int wv = 0; wv < 8; ++wv) s += acc[(wv * 2 + t / B) * B + (t % B)];
    dst[t] = s;
  }
}

__global__ void k_residual(const double* __restrict__ partial_res, int chunks_max,
                           const int* __restrict__ mesh_off, int B, double* __restrict__ res) {
  const int mesh = blockIdx.x;
  const int nchunks = (mesh_off[mesh + 1] - mesh_off[mesh] + GRAM_ROWS - 1) / GRAM_ROWS;
  for (int j = threadIdx.x; j < B; j += blockDim.x) {
    double n = 0.0, d = 0.0;
    for (int c = 0; c < nchunks; ++c) {
      n += partial_res[((size_t)mesh * chunks_max + c) * 2 * B + j];
      d += partial_res[((size_t)mesh * chunks_max + c) * 2 * B + B + j];
    }
    res[(size_t)mesh * B + j] = sqrt(n / d);
  }
}

// Output of a converged mesh: column j of eig_vecs = X[:, sel[j]] / ||.||_2, sign such that the
// entry of largest magnitude (lowest row on ties) is positive; eig_vals[j] = theta[sel[j]].
__global__ void __launch_bounds__(256)
k_write_pairs(const double* __restrict__ x, const double* __restrict__ theta, int B,
              const int* __restrict__ mesh_off, const int* __restrict__ flags,
              const int* __restrict__ sel, const int* __restrict__ n_out, double* __restrict__ eig_vals,
              double* __restrict__ eig_vecs, int ldv, int mesh_base) {
  const int mesh = blockIdx.y, j = blockIdx.x;
  if (!flags[mesh] || j >= n_out[mesh]) return;
  const int c = sel[(size_t)mesh * B + j];
  const int r0 = mesh_off[mesh], r1 = mesh_off[mesh + 1];
  double ss = 0.0, best = -1.0, bestv = 0.0;
  int besti = 0x7fffffff;
  for (int r = r0 + threadIdx.x; r < r1; r += blockDim.x) {
    const double v = x[(size_t)r * B + c];
    ss += v * v;
    const double a = fabs(v);
    if (a > best) {
      best = a;
      bestv = v;
      besti = r;
    }
  }
  __shared__ double s_ss[256], s_best[256], s_bestv[256];
  __shared__ int s_besti[256];
  s_ss[threadIdx.x] = ss;
  s_best[threadIdx.x] = best;
  s_bestv[threadIdx.x] = bestv;
  s_besti[threadIdx.x] = besti;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      s_ss[threadIdx.x] += s_ss[threadIdx.x + o];
      const double ob = s_best[threadIdx.x + o];
      const int oi = s_besti[threadIdx.x + o];
      if (ob > s_best[threadIdx.x] || (ob == s_best[threadIdx.x] && oi < s_besti[threadIdx.x])) {
        s_best[threadIdx.x] = ob;
        s_bestv[threadIdx.x] = s_bestv[threadIdx.x + o];
        s_besti[threadIdx.x] = oi;
      }
    }
    __syncthreads();
  }
  const double scale = (s_bestv[0] < 0.0 ? -1.0 : 1.0) / sqrt(s_ss[0]);
  for (int r = r0 + threadIdx.x; r < r1; r += blockDim.x)
    eig_vecs[(size_t)r * ldv + j] = x[(size_t)r * B + c] * scale;
  if (threadIdx.x == 0) eig_vals[(size_t)(mesh_base + mesh) * ldv + j] = theta[(size_t)mesh * B + c];
}

// ---------------------------------------------------------------------------------------------
// pinned host staging (grow-only, process lifetime)
// ---------------------------------------------------------------------------------------------
struct PinnedPool {
  void* p = nullptr;
  size_t cap = 0;
  void* get(size_t bytes) {
    if (bytes > cap) {
      if (p) cudaFreeHost(p);
      p = nullptr;
      cap = 0;
      if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
      cap = bytes;
    }
    return p;
  }
};
static thread_local PinnedPool g_pin_small, g_pin_tables, g_pin_cut;

// Live profile of the dominant kernel (the Chebyshev SpMM step): CUDA events bracket every
// filter() on the launching stream; the elapsed time is collected at the next synchronisation the
// driver performs anyway.  bench.py turns {ms, launches, algorithmic bytes} into the roofline line.
// fp32 filter passes (chfsi_driver.hpp, k_filter_sell in sell.cu): a pass may run in fp32 if it is meant to leave every residual
// above this value.  The fp32 floor measured on 15k-vertex meshes is ~5e-7 (a pass aimed lower stalls there).
constexpr double LOWP_FLOOR = 1.4e-6;
// A sized plain-fp32 pass aims here (lands at ~0.7 of its aim): low enough for the fp32 correction form to reach 1e-10
// from it with its rounding noise (2.3e-5 of the starting residual, chfsi_driver.hpp) well below the tolerance.
constexpr double LOWP_AIM = 1.5e-6;

// The sized pass aims at SIZED_PASS_LAND * tol.  The prediction (residual / amplification of the slowest wanted pair) is
// pessimistic by a steady factor: aimed at 0.2 / 0.35 / 0.5 tol, batches of 15k-vertex meshes land at 0.13 / 0.24 / 0.35 tol
// with 282 / 274 / 269 filter steps.  A miss costs one more (short) pass, never accuracy.
constexpr double SIZED_PASS_LAND = 0.4;

// Totals are shared (solves may run on several host threads, one stream each); the event pair and the pending
// bracket belong to the calling thread.
struct FilterTotals {
  std::mutex mu;
  double ms = 0.0, launches = 0.0, bytes = 0.0;
};
struct FilterProfile {
  FilterTotals* tot;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  bool pending = false;
  double pending_launches = 0.0, pending_bytes = 0.0;
  explicit FilterProfile(FilterTotals* t) : tot(t) {}
  void begin(cudaStream_t s) {
    if (!e0) {
      cudaEventCreate(&e0);
      cudaEventCreate(&e1);
    }
    collect();
    cudaEventRecord(e0, s);
  }
  void end(cudaStream_t s, double n_launches, double n_bytes) {
    cudaEventRecord(e1, s);
    pending = true;
    pending_launches = n_launches;
    pending_bytes = n_bytes;
  }
  void collect() {  // call only after the stream has been synchronised past e1
    if (!pending) return;
    float t = 0.f;
    if (cudaEventSynchronize(e1) == cudaSuccess && cudaEventElapsedTime(&t, e0, e1) == cudaSuccess) {
      std::lock_guard<std::mutex> lock(tot->mu);
      tot->ms += t;
      tot->launches += pending_launches;
      tot->bytes += pending_bytes;
    }
    pending = false;
  }
};
static FilterTotals g_totals[3];  // fp64 steps (k_spmm<b,.,0>), fp32 steps (k_filter_sell modes 0-2), fp32 correction steps (modes 3-4)
static thread_local FilterProfile g_filter_profile(&g_totals[0]);
static thread_local FilterProfile g_filter_profile_lowp(&g_totals[1]);
static thread_local FilterProfile g_filter_profile_corr(&g_totals[2]);

// Tuning record: blocking the filter over groups of meshes that fit the 126 MB L2 (all steps of a table chunk on one group
// before the next) was measured on B200 at 128 pairs: off 641 pairs/s, 64 MB groups 548, 32 MB 341 -- groups that fit L2
// are < 1 wave of CTAs and the kernel turns latency-bound -- and removed.
template <int B>
struct GramCfg {
  static constexpr int QT = (B <= 32) ? B / 8 : (B <= 64 ? 2 : 1);
};


// ---------------------------------------------------------------------------------------------
// row-partitioned solve across GPUs (SURVEY.md section 8e-ii): one mesh, rank r owns a contiguous
// block of rows; vector blocks carry n_ghost extra rows (copies of the neighbours' boundary rows,
// grouped by owner rank) refreshed by one grouped ncclSend/ncclRecv before every SpMM.
// ---------------------------------------------------------------------------------------------
struct DistCtx {
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1;
  long long row_base = 0;          // global index of local row 0
  int n_loc = 0, n_ghost = 0, n_send = 0;
  const int* send_idx = nullptr;   // device [n_send]: local rows to ship, grouped by destination rank
  const int* send_counts = nullptr;  // host [world]
  const int* recv_counts = nullptr;  // host [world]
  double* sendbuf = nullptr;       // device [n_send][B]
  double* small = nullptr;         // device scratch for all-reduced small blocks
  int* fake_off = nullptr;         // device {0, 1}: lets the chunk-summing kernels read one chunk
  // --- P2P mode: halo fused into the SpMM, vector blocks live in an IPC-shared region ---
  bool p2p = false;
  double* blocks = nullptr;              // this rank's three [rows_cap][B] blocks inside the shared region
  size_t block_stride = 0;               // doubles between consecutive blocks
  const double* const* peer_blocks = nullptr;  // device [3][world]: block k of rank p
  unsigned long long* flags = nullptr;   // this rank's flag slots (one 128-byte line per peer)
  unsigned long long* const* peer_flags = nullptr;  // device [world]: flag array of rank p
  const int* ghost_peer = nullptr;       // device [n_ghost]
  const int* ghost_row = nullptr;        // device [n_ghost]
  int* dev_err = nullptr;                // device flag raised by a barrier time-out
  unsigned long long epoch = 0;
  // --- fp32 filter passes as ONE persistent cooperative kernel per pass (sell.cu: k_filter_persist) ---
  bool lowp = false;                     // P2P mode + SELL copy of the local rows built
  int rows_cap = 0;                      // rows of a block in the shared region (identical on every rank)
  int ghost_base = 0;                    // first ghost row of an fp32 view (= largest n_local of any rank)
  const int* push_row = nullptr;         // device [n_push], sorted: local rows some peer gathers
  const int* push_dst = nullptr;         // device [n_push]: (peer << 24) | ghost slot on that peer
  int n_push = 0;
  const float* const* peer_views = nullptr;  // device [6][world]: fp32 view 2 * block + half of rank p
  unsigned* counter = nullptr;           // arrivals of this GPU's CTAs at the in-kernel barrier
  unsigned long long* timing = nullptr;  // {ns at barriers, ns working, steps} of CTA 0 of the persistent kernels
};
static double g_persist_timing[4] = {0.0, 0.0, 0.0, 0.0};  // last row-partitioned solve of this process (profile kind 3)
static ncclComm_t g_dist_comm = nullptr;
static int g_dist_rank = 0, g_dist_world = 1;

__global__ void k_pack_rows(const double* __restrict__ x, const int* __restrict__ idx, int n, int B,
                            double* __restrict__ out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * B) return;
  const int i = (int)(t / B), c = (int)(t % B);
  out[t] = x[(size_t)idx[i] * B + c];
}

__global__ void k_sum_chunks(const double* __restrict__ partial, int nchunks, int len, double* __restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= len) return;
  double s = 0.0;
  for (int c = 0; c < nchunks; ++c) s += partial[(size_t)c * len + e];
  out[e] = s;
}

// per selected column: {sum of squares, max |v|, v at that entry, global row of that entry}
__global__ void __launch_bounds__(256)
k_colstats_local(const double* __restrict__ x, int B, int n_rows, const int* __restrict__ sel, int n_out,
                 long long row_base, double* __restrict__ stats) {
  const int j = blockIdx.x;
  if (j >= n_out) return;
  const int c = sel[j];
  double ss = 0.0, best = -1.0, bestv = 0.0;
  long long besti = 0x7fffffffffffffffLL;
  for (int r = threadIdx.x; r < n_rows; r += blockDim.x) {
    const double v = x[(size_t)r * B + c];
    ss += v * v;
    const double a = fabs(v);
    if (a > best) {
      best = a;
      bestv = v;
      besti = r + row_base;
    }
  }
  __shared__ double s_ss[256], s_best[256], s_bestv[256];
  __shared__ long long s_besti[256];
  s_ss[threadIdx.x] = ss;
  s_best[threadIdx.x] = best;
  s_bestv[threadIdx.x] = bestv;
  s_besti[threadIdx.x] = besti;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      s_ss[threadIdx.x] += s_ss[threadIdx.x + o];
      const double ob = s_best[threadIdx.x + o];
      const long long oi = s_besti[threadIdx.x + o];
      if (ob > s_best[threadIdx.x] || (ob == s_best[threadIdx.x] && oi < s_besti[threadIdx.x])) {
        s_best[threadIdx.x] = ob;
        s_bestv[threadIdx.x] = s_bestv[threadIdx.x + o];
        s_besti[threadIdx.x] = oi;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    stats[4 * j + 0] = s_ss[0];
    stats[4 * j + 1] = s_best[0];
    stats[4 * j + 2] = s_bestv[0];
    stats[4 * j + 3] = (double)s_besti[0];  // exact below 2^53
  }
}

// gathered [world][B][4] stats -> normalise local rows: unit 2-norm, largest-magnitude entry positive
__global__ void __launch_bounds__(256)
k_write_scaled(const double* __restrict__ x, const double* __restrict__ theta, int B, int n_rows,
               const int* __restrict__ sel, int n_out, const double* __restrict__ gathered, int world,
               double* __restrict__ eig_vals, double* __restrict__ eig_vecs, int ldv) {
  const int j = blockIdx.x;
  if (j >= n_out) return;
  const int c = sel[j];
  double ss = 0.0, best = -1.0, bestv = 0.0, besti = 1e300;
  for (int r = 0; r < world; ++r) {
    const double* st = gathered + ((size_t)r * B + j) * 4;
    ss += st[0];
    if (st[1] > best || (st[1] == best && st[3] < besti)) {
      best = st[1];
      bestv = st[2];
      besti = st[3];
    }
  }
  const double scale = (bestv < 0.0 ? -1.0 : 1.0) / sqrt(ss);
  for (int r = threadIdx.x; r < n_rows; r += blockDim.x) eig_vecs[(size_t)r * ldv + j] = x[(size_t)r * B + c] * scale;
  if (threadIdx.x == 0) eig_vals[j] = theta[c];
}


// Inter-GPU barrier through flags in peer memory: lane p publishes `epoch` into slot `rank` of rank
// p's flag array (st.release.sys over NVLink) and waits until rank p has published the same epoch
// here.  Kernels of different ranks run on different GPUs, so the spin always makes progress; a
// generous cycle budget turns a lost peer into an error instead of a hang.
__global__ void k_peer_barrier(unsigned long long* my_flags, unsigned long long* const* peer_flags, int rank,
                               int world, unsigned long long epoch, int* err) {
  const int p = threadIdx.x;
  if (p >= world || p == rank) return;
  __threadfence_system();
  unsigned long long* dst = peer_flags[p] + (size_t)rank * 16;  // 16 x 8 B = one 128-byte line per slot
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(epoch) : "memory");
  const unsigned long long* src = my_flags + (size_t)p * 16;
  const long long t0 = clock64();
  for (;;) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(src) : "memory");
    if (v >= epoch) break;
    if (clock64() - t0 > 20000000000LL) {  // ~10 s at 1.9 GHz
      atomicExch(err, 1);
      break;
    }
  }
}

struct PeerShared {
  void* base = nullptr;
  size_t bytes = 0;
  int world = 0, rank = 0;
  std::vector<void*> peer;
};
static PeerShared g_shared;
constexpr size_t PEER_FLAG_BYTES = 128;

// Per-column tables of a correction pass, steps [s0, s0 + len) of `deg`: thread (mesh, column j) runs the three-term
// coefficient recurrence of corr_table_column (chfsi_driver.hpp) from step 0 and stores its slice as floats
// [mesh][len][B]; thread 0 of a mesh also writes the centre of the filter interval.  ab = {a[M], beta[M]}.
__global__ void k_corr_tables(const double* __restrict__ theta, const double* __restrict__ ab, int M, int B, int deg, int s0,
                              int len, float* __restrict__ alpha_c, float* __restrict__ gamma_c, double* __restrict__ center) {
  const int m = blockIdx.x, j = threadIdx.x;
  if (j >= B) return;
  const double a = ab[m], beta = ab[M + m];
  if (j == 0) center[m] = 0.5 * (beta + a);
  float* al = alpha_c + (size_t)m * len * B + j;
  float* ga = gamma_c + (size_t)m * len * B + j;
  corr_table_column(a, theta[(size_t)m * B + j], beta, min(deg, s0 + len), [&](int s, double av, double gv) {
    if (s >= s0) {
      al[(size_t)(s - s0) * B] = (float)av;
      ga[(size_t)(s - s0) * B] = (float)gv;
    }
  });
}

static void launch_corr_tables(const double* theta, const double* ab, int M, int B, int deg, int s0, int len, float* alpha_c,
                               float* gamma_c, double* center, cudaStream_t stream) {
  k_corr_tables<<<M, 96, 0, stream>>>(theta, ab, M, B, deg, s0, len, alpha_c, gamma_c, center);
  FB_COUNT_LAUNCH(1);
}

struct CudaBackend {
  // graph of this run (rows are the run's meshes; pointers are global, offsets select the run)
  SpmmGraph g;
  const double* points;
  const int* off_host;   // [M+1] global row offsets of the run's meshes
  const int* info_host;  // [M][FOCUSR_MESH_INFO_INTS]
  int M, B, mesh_base;
  bool sym;
  cudaStream_t stream;
  // workspace
  double *X, *Y, *Xn, *partial, *partial_res, *W, *theta, *res, *G, *H, *alpha, *gamma, *center, *corr_ab;
  long long *lo, *hi;
  int *flags, *sel, *n_out, *rr_info;
  int chunks_max, table_cap;
  // outputs
  double* eig_vals;
  double* eig_vecs;
  int ldv;
  int err = FB_OK;
  DistCtx* dist = nullptr;  // row-partitioned multi-GPU solve (one mesh); null = everything is local
  bool mixed = true;        // fp32 filter passes allowed (focusr_eigs_options.mixed_precision)
  FilterTuning tune;        // kernel form of the fp32 filter steps
  bool nonsym_device = true;  // non-symmetric Rayleigh-Ritz on the device (focusr_eigs_options.nonsym_device)
  SellF32 sell;             // SELL-64 fp32 copy of the matrix (tune.format == 0)

  int n_meshes() const { return M; }
  int block() const { return B; }
  bool symmetric() const { return sym; }
  int zero_rows(int m) const { return info_host[FOCUSR_MESH_INFO_INTS * m + 2]; }
  // fp32 filter passes: local solves only (the peer-shared blocks of the row-partitioned solve are fp64)
  // fp32 filter passes: batches on one GPU, and the row-partitioned solve in P2P mode (fp32 views of the peer-shared blocks)
  bool lowp_available() const { return (dist == nullptr || dist->lowp) && mixed && sell.entries != nullptr; }

  // fp32 view number `half` (0 or 1) of an fp64 block, indexed by global row like the block itself
  float* f32_view(double* blk, int half) const {
    if (dist) return reinterpret_cast<float*>(blk) + (size_t)half * dist->rows_cap * B;  // same offset on every rank
    const size_t shift = (size_t)off_host[0] * B;
    const size_t rows = (size_t)(off_host[M] - off_host[0]);
    return reinterpret_cast<float*>(blk + shift) + (size_t)half * rows * B - shift;
  }

  void fail(cudaError_t e, const char* what) {
    if (e != cudaSuccess && err == FB_OK) {
      set_error("eigs: %s -> %s", what, cudaGetErrorString(e));
      err = FB_ERR_CUDA;
    }
  }
  void check(const char* what) { fail(cudaGetLastError(), what); }
  void nccl_check(int rc, const char* what) {
    if (rc != NCCL_SUCCESS && err == FB_OK) {
      set_error("eigs (dist): %s -> %s", what, nccl_api().GetErrorString(rc));
      err = FB_ERR_CUDA;
    }
  }
  // refresh the ghost rows of a [n_loc + n_ghost][B] block from their owners
  void halo_exchange(double* x) {
    if (!dist || dist->world == 1) return;
    if (dist->p2p) {  // nothing moves: peers read the rows in place; only order the steps
      ++dist->epoch;
      k_peer_barrier<<<1, 32, 0, stream>>>(dist->flags, dist->peer_flags, dist->rank, dist->world, dist->epoch, dist->dev_err);
      FB_COUNT_LAUNCH(1);
      return;
    }
    NcclApi& api = nccl_api();
    if (dist->n_send > 0) {
      k_pack_rows<<<div_up((long long)dist->n_send * B, 256), 256, 0, stream>>>(x, dist->send_idx, dist->n_send, B, dist->sendbuf);
      FB_COUNT_LAUNCH(1);
    }
    nccl_check(api.GroupStart(), "group start");
    size_t so = 0, ro = 0;
    for (int p = 0; p < dist->world; ++p) {
      const int sc = dist->send_counts[p], rcnt = dist->recv_counts[p];
      if (p != dist->rank) {
        if (sc > 0) nccl_check(api.Send(dist->sendbuf + so * B, (size_t)sc * B, NCCL_FLOAT64, p, dist->comm, stream), "send");
        if (rcnt > 0)
          nccl_check(api.Recv(x + ((size_t)dist->n_loc + ro) * B, (size_t)rcnt * B, NCCL_FLOAT64, p, dist->comm, stream), "recv");
      }
      so += sc;
      ro += rcnt;
    }
    nccl_check(api.GroupEnd(), "group end");
  }
  int block_index(const double* ptr) const { return (int)((ptr - dist->blocks) / (ptrdiff_t)dist->block_stride); }
  int view_id(const double* blk, int half) const { return 2 * block_index(blk) + half; }
  // one chunk of steps [s0, s0 + len) of a `deg`-step pass as one persistent kernel; views rotate by len afterwards
  void persist_chunk(bool corr, int s0, int len, int deg, int (&v)[3], const void* al, const void* ga) {
    fail(cudaMemsetAsync(dist->counter, 0, sizeof(unsigned), stream), "zero barrier counter");
    PersistArgs a{};
    a.entries = sell.entries;
    a.slice_ptr = sell.slice_ptr;
    a.ddi = sell.ddi;
    a.n_loc = dist->n_loc;
    a.ghost_base = dist->ghost_base;
    a.push_row = dist->push_row;
    a.push_dst = dist->push_dst;
    a.n_push = dist->n_push;
    a.push_first = (!corr && s0 == 0) ? 1 : 0;   // plain pass: the fp32 copy of X still lacks its ghost rows
    a.peer_views = dist->peer_views;
    a.world = dist->world;
    a.rank = dist->rank;
    a.v_prev = v[0];
    a.v_cur = v[1];
    a.v_next = v[2];
    a.r = f32_view(Y, 0);
    a.x = X;
    a.alpha = al;
    a.gamma = ga;
    a.center = center;
    a.s0 = s0;
    a.len = len;
    a.deg = deg;
    a.prefetch = tune.prefetch;
    a.counter = dist->counter;
    a.my_flags = dist->flags;
    a.peer_flags = dist->peer_flags;
    a.epoch0 = dist->epoch;
    a.err = dist->dev_err;
    a.timing = dist->timing;
    if (launch_filter_persist(corr, B, a, stream) != FB_OK && err == FB_OK) err = FB_ERR_CUDA;
    dist->epoch += (unsigned long long)len;
    for (int i = 0; i < len % 3; ++i) {
      const int t = v[0];
      v[0] = v[1];
      v[1] = v[2];
      v[2] = t;
    }
  }
  void spmm(int mode, const SpmmGraph& gg, const double* y, const double* x_prev, double* out, const double* al,
            const double* ga, const double* ce, int step, int n_steps) {
    if (dist && dist->p2p && dist->world > 1)
      launch_spmm_p2p(mode, B, gg, dist->n_loc, y, dist->peer_blocks + (size_t)block_index(y) * dist->world,
                      dist->ghost_peer, dist->ghost_row, x_prev, out, al, ga, ce, step, n_steps, stream);
    else
      launch_spmm(mode, B, gg, y, x_prev, out, al, ga, ce, step, n_steps, stream);
  }
  void all_reduce(void* buf, size_t count, int dtype, int op, const char* what) {
    if (!dist || dist->world == 1) return;
    nccl_check(nccl_api().AllReduce(buf, buf, count, dtype, op, dist->comm, stream), what);
  }

  template <int BB>
  void init_block_t() {
    dim3 grid(chunks_max, M);
    k_init_block<BB><<<grid, 256, 0, stream>>>(points, g.degree, g.mesh_off, lo, hi, X, dist ? dist->row_base : 0LL);
  }
  template <int BB>
  void gram_t() {
    if constexpr (BB >= 64) {
      dim3 grid(chunks_max, M, GW_ZS);
      k_gram_wide<BB><<<grid, GRAM_THREADS, 0, stream>>>(X, Xn, g.degree, g.degree_inv, g.mesh_off, sym ? 1 : 0, partial,
                                                         chunks_max);
    } else {
      constexpr int QT = GramCfg<BB>::QT;
      dim3 grid(chunks_max, M, (BB / 8 + QT - 1) / QT);
      k_gram<BB, QT><<<grid, GRAM_THREADS, 0, stream>>>(X, Xn, g.degree, g.degree_inv, g.mesh_off, sym ? 1 : 0,
                                                        partial, chunks_max);
    }
  }
  template <int BB>
  void rotate_t() {
    constexpr int WS = (BB % 16 == 0) ? BB + 8 : BB;
    const size_t smem = sizeof(double) * ((size_t)BB * WS + 16 * BB);
    // the attribute is per device and per function: set on every call (cheap), never cached process-wide
    fail(cudaFuncSetAttribute(k_rotate<BB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "smem opt-in (rotate)");
    dim3 grid(chunks_max, M);
    // the fp32 residual block goes to the first half of Y (dead between filters), where filter_correction reads it
    k_rotate<BB><<<grid, GRAM_THREADS, smem, stream>>>(X, Xn, W, theta, g.degree_inv, g.mesh_off, partial_res, chunks_max,
                                                       lowp_available() ? f32_view(Y, 0) : nullptr);
  }
#define FB_DISPATCH_B(fn)                \
  switch (B) {                           \
    case 8: fn<8>(); break;              \
    case 16: fn<16>(); break;            \
    case 24: fn<24>(); break;            \
    case 32: fn<32>(); break;            \
    case 40: fn<40>(); break;            \
    case 48: fn<48>(); break;            \
    case 56: fn<56>(); break;            \
    case 64: fn<64>(); break;            \
    case 72: fn<72>(); break;            \
    case 80: fn<80>(); break;            \
    case 88: fn<88>(); break;            \
    case 96: fn<96>(); break;            \
    default: break;                      \
  }

  void init_block() {
    k_bbox_init<<<div_up(3 * M, 256), 256, 0, stream>>>(lo, hi, 3 * M);
    dim3 grid(chunks_max, M);
    k_bbox<<<grid, 256, 0, stream>>>(points, g.mesh_off, lo, hi);
    all_reduce(lo, 3 * (size_t)M, NCCL_INT64, NCCL_MIN, "bbox min");
    all_reduce(hi, 3 * (size_t)M, NCCL_INT64, NCCL_MAX, "bbox max");
    FB_DISPATCH_B(init_block_t)
    FB_COUNT_LAUNCH(3);
    check("init_block");
  }
  void apply_DmA() {  // Z (stored in Xn) = (D - A) X
    halo_exchange(X);
    spmm(1, g, X, X, Xn, nullptr, nullptr, nullptr, 0, 0);
    check("apply_DmA");
  }
  void gram() {
    FB_DISPATCH_B(gram_t)
    FB_COUNT_LAUNCH(1);
    if (dist) {  // local chunk sums -> [2][B][B], then the sum over ranks
      const int nchunks = div_up(off_host[1] - off_host[0], GRAM_ROWS);
      k_sum_chunks<<<div_up(2 * B * B, 256), 256, 0, stream>>>(partial, nchunks, 2 * B * B, dist->small);
      FB_COUNT_LAUNCH(1);
      all_reduce(dist->small, 2 * (size_t)B * B, NCCL_FLOAT64, NCCL_SUM, "gram all-reduce");
    }
    check("gram");
  }
  int rr_sym() {
    // one warp per mesh while the matrices are small or the meshes many; a whole CTA per mesh otherwise
    const bool wide = B > 32 || (B > 16 && M < 64);
    const int nt = wide ? 256 : 32;
    const size_t smem = sizeof(double) * ((size_t)3 * B * B + B + (B + 2) + nt) + sizeof(int) * (2 * B + 2);
    if (smem > 48 * 1024) {  // per device and per function: set on every call that needs it, never cached process-wide
      if (wide)
        fail(cudaFuncSetAttribute(k_rr_sym<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "smem opt-in (rr_sym)");
      else
        fail(cudaFuncSetAttribute(k_rr_sym<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "smem opt-in (rr_sym)");
    }
    const double* src = dist ? dist->small : partial;
    const int cm = dist ? 1 : chunks_max;
    const int* offs = dist ? dist->fake_off : g.mesh_off;
    if (wide)
      k_rr_sym<256><<<M, 256, smem, stream>>>(src, cm, offs, B, W, theta, rr_info);
    else
      k_rr_sym<32><<<M, 32, smem, stream>>>(src, cm, offs, B, W, theta, rr_info);
    FB_COUNT_LAUNCH(1);
    check("rr_sym");
    return 0;
  }
  // non-symmetric Rayleigh-Ritz on the device (b <= 64); `cut` [M] from the driver.  W, theta stay on the device; the
  // return codes and n_low come back with get_nonsym_info after the residuals.
  bool rr_nonsym_device(const double* cut_host) {
    if (B > 64 || !nonsym_device) return false;
    const size_t smem = rr_nonsym_smem_bytes(B);
    double* pin = (double*)g_pin_cut.get(sizeof(double) * (size_t)M);  // its own pool: the tables of the filter that is
                                                                        // still running are staged in the other ones
    if (!pin) {
      fail(cudaErrorMemoryAllocation, "pinned staging (cut)");
      return true;
    }
    memcpy(pin, cut_host, sizeof(double) * (size_t)M);
    fail(cudaMemcpyAsync(corr_ab, pin, sizeof(double) * (size_t)M, cudaMemcpyHostToDevice, stream), "H2D cut");
    if (smem > 48 * 1024)
      fail(cudaFuncSetAttribute(k_rr_nonsym, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "smem opt-in (rr_nonsym)");
    const double* src = dist ? dist->small : partial;
    const int cm = dist ? 1 : chunks_max;
    const int* offs = dist ? dist->fake_off : g.mesh_off;
    k_rr_nonsym<<<M, RRN_THREADS, smem, stream>>>(src, cm, offs, B, M, corr_ab, G, W, theta, rr_info);
    FB_COUNT_LAUNCH(1);
    check("rr_nonsym");
    return true;
  }
  void get_nonsym_info(int* rc_out, int* n_low_out) {
    int* pin = (int*)g_pin_small.get(sizeof(int) * 2 * (size_t)M);
    if (!pin) {
      fail(cudaErrorMemoryAllocation, "pinned staging");
      return;
    }
    fail(cudaMemcpyAsync(pin, rr_info, sizeof(int) * 2 * (size_t)M, cudaMemcpyDeviceToHost, stream), "D2H rr info");
    fail(cudaStreamSynchronize(stream), "sync after rr info");
    memcpy(rc_out, pin, sizeof(int) * (size_t)M);
    memcpy(n_low_out, pin + M, sizeof(int) * (size_t)M);
  }
  void get_GH(double* gh, double* hh) {
    dim3 grid(div_up(B * B, 256), M);
    k_reduce_gh<<<grid, 256, 0, stream>>>(partial, chunks_max, g.mesh_off, B, G, H);
    FB_COUNT_LAUNCH(1);
    check("reduce_gh");
    const size_t bytes = sizeof(double) * (size_t)M * B * B;
    fail(cudaMemcpyAsync(gh, G, bytes, cudaMemcpyDeviceToHost, stream), "D2H G");
    fail(cudaMemcpyAsync(hh, H, bytes, cudaMemcpyDeviceToHost, stream), "D2H H");
    fail(cudaStreamSynchronize(stream), "sync after G/H");
  }
  void set_W_theta(const double* wv, const double* th) {
    // pageable host memory: the copy is staged by the runtime before the call returns
    fail(cudaMemcpyAsync(W, wv, sizeof(double) * (size_t)M * B * B, cudaMemcpyHostToDevice, stream), "H2D W");
    fail(cudaMemcpyAsync(theta, th, sizeof(double) * (size_t)M * B, cudaMemcpyHostToDevice, stream), "H2D theta");
  }
  void rotate_and_residual() {
    FB_DISPATCH_B(rotate_t)
    if (dist) {
      const int nchunks = div_up(off_host[1] - off_host[0], GRAM_ROWS);
      k_sum_chunks<<<div_up(2 * B, 256), 256, 0, stream>>>(partial_res, nchunks, 2 * B, dist->small);
      all_reduce(dist->small, 2 * (size_t)B, NCCL_FLOAT64, NCCL_SUM, "residual all-reduce");
      k_residual<<<M, 128, 0, stream>>>(dist->small, 1, dist->fake_off, B, res);
      FB_COUNT_LAUNCH(1);
    } else {
      k_residual<<<M, 128, 0, stream>>>(partial_res, chunks_max, g.mesh_off, B, res);
    }
    FB_COUNT_LAUNCH(2);
    check("rotate");
  }
  void get_theta_res(double* th, double* rs) {
    const size_t bytes = sizeof(double) * (size_t)M * B;
    double* pin = (double*)g_pin_small.get(2 * bytes);
    if (!pin) {
      fail(cudaErrorMemoryAllocation, "pinned staging");
      return;
    }
    fail(cudaMemcpyAsync(pin, theta, bytes, cudaMemcpyDeviceToHost, stream), "D2H theta");
    fail(cudaMemcpyAsync(pin + (size_t)M * B, res, bytes, cudaMemcpyDeviceToHost, stream), "D2H res");
    fail(cudaStreamSynchronize(stream), "sync after theta/res");
    memcpy(th, pin, bytes);
    memcpy(rs, pin + (size_t)M * B, bytes);
  }
  // one fp32 filter step on the sliced-ELL copy of the matrix (sell.cu has the modes)
  void lowp_step(int mode, const void* y, const float* x_prev, const float* r, void* out, float* y_copy, const void* al,
                 const void* ga, int step, int n_steps, bool has_prev) {
    launch_filter_sell(mode, B, sell, g.mesh_off, g.n_meshes, g.max_mesh_rows, y, x_prev, r, out, y_copy, al, ga, center,
                       step, n_steps, has_prev, tune, stream);
  }
  void filter(int deg, const double* al, const double* ga, const double* ce, bool lowp) {
    lowp = lowp && lowp_available() && deg >= 3;
    // tables are uploaded in chunks of table_cap steps; pinned staging holds every chunk of this
    // filter until the next synchronisation (get_theta_res of the next outer iteration)
    const size_t total = (size_t)M * deg;
    double* pin = (double*)g_pin_tables.get(sizeof(double) * (2 * total + M));
    if (!pin) {
      fail(cudaErrorMemoryAllocation, "pinned tables");
      return;
    }
    double* pc = pin + 2 * total;
    memcpy(pc, ce, sizeof(double) * M);
    fail(cudaMemcpyAsync(center, pc, sizeof(double) * M, cudaMemcpyHostToDevice, stream), "H2D center");
    double* cur = X;   // Y_k
    double* prev = Y;  // Y_{k-1} (unused at step 0)
    double* next = Xn;
    size_t pin_off = 0;
    // algorithmic bytes of one step over the run: matrix once (int32 col + fp64 weight per entry,
    // row_ptr), degree + 1/degree~, and three passes over the [rows][B] block (DESIGN.md)
    const double rows = (double)(off_host[M] - off_host[0]);
    double nnz = 0.0;
    for (int m = 0; m < M; ++m) nnz += info_host[FOCUSR_MESH_INFO_INTS * m];
    // fp32 passes read the fp32 copy of the matrix (4 + 4 bytes per entry, 8 bytes of (d, 1/d~) per row)
    const double step_bytes = lowp ? 8.0 * nnz + 4.0 * rows + 8.0 * rows + 12.0 * (double)B * rows
                                   : 12.0 * nnz + 4.0 * rows + 16.0 * rows + 24.0 * (double)B * rows;
    FilterProfile& prof = lowp ? g_filter_profile_lowp : g_filter_profile;
    prof.begin(stream);
    // fp32 pass: the three fp32 blocks live in the two fp64 blocks that are free during a filter (Y: two of
    // them, Xn: one); the first step reads X (fp64) and the last one writes X, so X holds the result again.
    float* f_cur = f32_view(Y, 0);
    float* f_prev = f32_view(Y, 1);
    float* f_next = f32_view(Xn, 0);
    int dist_views[3] = {0, 0, 0};
    for (int s0 = 0; s0 < deg; s0 += table_cap) {
      const int len = std::min(table_cap, deg - s0);
      double* pa = pin + pin_off;
      double* pg = pa + (size_t)M * len;
      pin_off += 2 * (size_t)M * len;
      for (int m = 0; m < M; ++m) {
        memcpy(pa + (size_t)m * len, al + (size_t)m * deg + s0, sizeof(double) * len);
        memcpy(pg + (size_t)m * len, ga + (size_t)m * deg + s0, sizeof(double) * len);
      }
      fail(cudaMemcpyAsync(alpha, pa, sizeof(double) * (size_t)M * len, cudaMemcpyHostToDevice, stream), "H2D alpha");
      fail(cudaMemcpyAsync(gamma, pg, sizeof(double) * (size_t)M * len, cudaMemcpyHostToDevice, stream), "H2D gamma");
      if (lowp && dist) {
        // row-partitioned: the fp32 copy of X goes to view (Y,1) first, then every step has the same form
        if (s0 == 0) {
          block_to_f32(X, f32_view(Y, 1), (long long)dist->n_loc * B, stream);
          dist_views[0] = view_id(Xn, 0);
          dist_views[1] = view_id(Y, 1);
          dist_views[2] = view_id(Y, 0);
        }
        persist_chunk(false, s0, len, deg, dist_views, alpha, gamma);
        continue;
      }
      if (lowp) {
        for (int s = 0; s < len; ++s) {
          const int gs = s0 + s;
          if (gs == 0) {  // X (fp64) -> f_cur, fp32 copy of X -> f_prev
            lowp_step(1, X, nullptr, nullptr, f_cur, f_prev, alpha, gamma, s, len, false);
          } else {
            const bool last = gs == deg - 1;
            lowp_step(last ? 2 : 0, f_cur, f_prev, nullptr, last ? (void*)X : (void*)f_next, nullptr, alpha, gamma, s, len,
                      true);
            float* t = f_prev;
            f_prev = f_cur;
            f_cur = f_next;
            f_next = t;
          }
        }
        continue;
      }
      for (int s = 0; s < len; ++s) {
        halo_exchange(cur);
        spmm(0, g, cur, prev, next, alpha, gamma, center, s, len);
        double* t = prev;
        prev = cur;
        cur = next;
        next = t;
      }
    }
    prof.end(stream, (double)deg, (double)deg * step_bytes);
    if (!lowp) {  // rotate names so that X is the filtered block again
      double* nx = cur;
      double* ny = prev;
      double* nn = next;
      X = nx;
      Y = ny;
      Xn = nn;
    }
    check("filter");
  }
  // fp32 correction pass (chfsi_driver.hpp): X += z_deg, z_{k+1} = alpha_kj ((L - c) z_k + r_j) - gamma_kj z_{k-1}, z_0 = 0.
  // r (fp32) was left in the first half of Y by the last rotate_and_residual; the three z blocks live in the second
  // half of Y and the two halves of Xn.  The per-column tables [M][len][B] (float) are built on the device from the
  // Ritz values of that Rayleigh-Ritz step (k_corr_tables): the host hands over 2 M numbers.
  void filter_correction(int deg, const double* a_m, const double* beta_m) {
    // the device tables (alpha, gamma: M * table_cap doubles each) hold M * cap_c * B floats
    const int cap_c = std::max(1, (int)((size_t)table_cap * 2 / B));
    double* pin = (double*)g_pin_tables.get(sizeof(double) * 2 * (size_t)M);
    if (!pin) {
      fail(cudaErrorMemoryAllocation, "pinned tables");
      return;
    }
    memcpy(pin, a_m, sizeof(double) * M);
    memcpy(pin + M, beta_m, sizeof(double) * M);
    fail(cudaMemcpyAsync(corr_ab, pin, sizeof(double) * 2 * (size_t)M, cudaMemcpyHostToDevice, stream), "H2D filter edges");
    const float* r = f32_view(Y, 0);
    float* z_cur = f32_view(Y, 1);
    float* z_prev = f32_view(Xn, 0);
    float* z_next = f32_view(Xn, 1);
    const double rows = (double)(off_host[M] - off_host[0]);
    double nnz = 0.0;
    for (int m = 0; m < M; ++m) nnz += info_host[FOCUSR_MESH_INFO_INTS * m];
    const double step_bytes = 8.0 * nnz + 4.0 * rows + 8.0 * rows + 16.0 * (double)B * rows;
    float* d_al = reinterpret_cast<float*>(alpha);
    float* d_ga = reinterpret_cast<float*>(gamma);
    // first chunk of tables before the timed bracket (its launches are the filter steps only)
    launch_corr_tables(theta, corr_ab, M, B, deg, 0, std::min(cap_c, deg), d_al, d_ga, center, stream);
    g_filter_profile_corr.begin(stream);
    // (row-partitioned: the ghost rows of the view are zeroed too)
    fail(cudaMemsetAsync(z_cur + (size_t)off_host[0] * B, 0, sizeof(float) * (size_t)(dist ? dist->rows_cap : rows) * B, stream),
         "zero z");
    int dist_views[3] = {0, 0, 0};
    if (dist) {
      dist_views[0] = view_id(Xn, 0);
      dist_views[1] = view_id(Y, 1);
      dist_views[2] = view_id(Xn, 1);
    }
    for (int s0 = 0; s0 < deg; s0 += cap_c) {
      const int len = std::min(cap_c, deg - s0);
      if (s0 > 0) launch_corr_tables(theta, corr_ab, M, B, deg, s0, len, d_al, d_ga, center, stream);
      if (dist) {
        persist_chunk(true, s0, len, deg, dist_views, d_al, d_ga);
        continue;
      }
      for (int s = 0; s < len; ++s) {
        const int gs = s0 + s;
        const bool last = gs == deg - 1;
        lowp_step(last ? 4 : 3, z_cur, z_prev, r, last ? (void*)X : (void*)z_next, nullptr, d_al, d_ga, s, len, gs > 0);
        float* t = z_prev;
        z_prev = z_cur;
        z_cur = z_next;
        z_next = t;
      }
    }
    g_filter_profile_corr.end(stream, (double)deg, (double)deg * step_bytes);
    check("filter_correction");
  }
  void finalize(const int* fl, const int* sl, const int* no) {
    fail(cudaMemcpyAsync(flags, fl, sizeof(int) * M, cudaMemcpyHostToDevice, stream), "H2D flags");
    fail(cudaMemcpyAsync(sel, sl, sizeof(int) * (size_t)M * B, cudaMemcpyHostToDevice, stream), "H2D sel");
    fail(cudaMemcpyAsync(n_out, no, sizeof(int) * M, cudaMemcpyHostToDevice, stream), "H2D n_out");
    if (dist) {
      const int cnt = no[0];
      double* stats = dist->small;                        // [B][4] local
      double* gathered = dist->small + 4 * (size_t)B;     // [world][B][4]
      k_colstats_local<<<std::max(cnt, 1), 256, 0, stream>>>(X, B, dist->n_loc, sel, cnt, dist->row_base, stats);
      if (dist->world > 1)
        nccl_check(nccl_api().AllGather(stats, gathered, 4 * (size_t)B, NCCL_FLOAT64, dist->comm, stream), "stats all-gather");
      else
        fail(cudaMemcpyAsync(gathered, stats, sizeof(double) * 4 * B, cudaMemcpyDeviceToDevice, stream), "stats copy");
      k_write_scaled<<<std::max(cnt, 1), 256, 0, stream>>>(X, theta, B, dist->n_loc, sel, cnt, gathered, dist->world,
                                                           eig_vals, eig_vecs, ldv);
      FB_COUNT_LAUNCH(1);
    } else {
      dim3 grid(std::min(B, ldv), M);
      k_write_pairs<<<grid, 256, 0, stream>>>(X, theta, B, g.mesh_off, flags, sel, n_out, eig_vals, eig_vecs, ldv, mesh_base);
    }
    FB_COUNT_LAUNCH(1);
    check("write_pairs");
    // the host arrays are reused by the driver right after this call returns
    fail(cudaStreamSynchronize(stream), "sync after finalize");
  }
};

static size_t eigs_ws_layout(int n_rows, int n_meshes, int max_mesh_rows, int B, CudaBackend* be, void* ws, size_t ws_bytes) {
  Carver cv(ws, ws_bytes);
  const int chunks_max = div_up(max_mesh_rows, GRAM_ROWS);
  const int table_cap = std::max(64, std::min(8192, (1 << 20) / std::max(1, n_meshes)));
  double* X = cv.take<double>((size_t)n_rows * B);
  double* Y = cv.take<double>((size_t)n_rows * B);
  double* Xn = cv.take<double>((size_t)n_rows * B);
  double* partial = cv.take<double>((size_t)n_meshes * chunks_max * 2 * B * B);
  double* partial_res = cv.take<double>((size_t)n_meshes * chunks_max * 2 * B);
  double* W = cv.take<double>((size_t)n_meshes * B * B);
  double* G = cv.take<double>((size_t)n_meshes * B * B);
  double* H = cv.take<double>((size_t)n_meshes * B * B);
  double* theta = cv.take<double>((size_t)n_meshes * B);
  double* res = cv.take<double>((size_t)n_meshes * B);
  double* alpha = cv.take<double>((size_t)n_meshes * table_cap);
  double* gamma = cv.take<double>((size_t)n_meshes * table_cap);
  double* center = cv.take<double>((size_t)n_meshes);
  double* corr_ab = cv.take<double>((size_t)2 * n_meshes);
  long long* lo = cv.take<long long>((size_t)3 * n_meshes);
  long long* hi = cv.take<long long>((size_t)3 * n_meshes);
  int* flags = cv.take<int>((size_t)n_meshes);
  int* sel = cv.take<int>((size_t)n_meshes * B);
  int* n_out = cv.take<int>((size_t)n_meshes);
  int* rr_info = cv.take<int>((size_t)2 * n_meshes);  // return code per mesh; n_low per mesh (non-symmetric path)
  int* off = cv.take<int>((size_t)n_meshes + 1);
  if (be) {
    be->X = X; be->Y = Y; be->Xn = Xn; be->partial = partial; be->partial_res = partial_res;
    be->W = W; be->G = G; be->H = H; be->theta = theta; be->res = res; be->alpha = alpha;
    be->gamma = gamma; be->center = center; be->corr_ab = corr_ab; be->lo = lo; be->hi = hi; be->flags = flags;
    be->sel = sel; be->n_out = n_out; be->rr_info = rr_info; be->g.mesh_off = off;
    be->chunks_max = chunks_max; be->table_cap = table_cap;
  }
  return cv.used + 256;
}

}  // namespace fb

using namespace fb;

extern "C" {

void focusr_profile_reset(void) {
  pk_evals_read_and_maybe_reset(true);
  g_filter_profile.collect();
  g_filter_profile_lowp.collect();
  g_filter_profile_corr.collect();
  for (FilterTotals& t : g_totals) {
    std::lock_guard<std::mutex> lock(t.mu);
    t.ms = t.launches = t.bytes = 0.0;
  }
}

void focusr_profile_get_kind(int kind, double* out4_host) {
  if (kind == 4) {  // pruned KNN: (query, reference) distance evaluations since the last reset (synchronises the device)
    cudaDeviceSynchronize();
    out4_host[0] = (double)pk_evals_read_and_maybe_reset(false);
    out4_host[1] = out4_host[2] = out4_host[3] = 0.0;
    return;
  }
  if (kind == 3) {  // persistent filter kernels of the last row-partitioned solve: CTA 0's {ns at barriers, ns working, steps}
    for (int i = 0; i < 4; ++i) out4_host[i] = g_persist_timing[i];
    return;
  }
  g_filter_profile.collect();
  g_filter_profile_lowp.collect();
  g_filter_profile_corr.collect();
  FilterTotals& t = g_totals[kind == 0 ? 0 : (kind == 1 ? 1 : 2)];
  std::lock_guard<std::mutex> lock(t.mu);
  out4_host[0] = t.ms;
  out4_host[1] = t.launches;
  out4_host[2] = t.bytes;
  out4_host[3] = 0.0;
}

void focusr_profile_get(double* out4_host) { focusr_profile_get_kind(0, out4_host); }

size_t focusr_eigs_workspace_bytes(int n_points, int n_meshes, int max_mesh_points, int block_size) {
  return eigs_ws_layout(n_points, n_meshes, max_mesh_points, block_size, nullptr, nullptr, 0);
}

// room for the fp32 copy of the matrix at the end of the workspace: (degree, 1/degree~) per row and the SELL-64 packed
// entries (8 bytes per padded entry) with their slice tables.  focusr_eigs_smallest runs its fp32 filter passes only if
// the workspace it is given has this room.
struct F32Layout {
  float2* ddi;
  int2* entries;
  int *all_mesh_off, *mesh_slice_off, *slice_ptr, *slice_cnt, *scan_tmp;
  size_t bytes;
};
static F32Layout f32_layout(long long sell_entries, int n_points, int n_meshes, void* base) {
  Carver cv(base, (size_t)-1);
  F32Layout l;
  const size_t n_slices = (size_t)n_points / SELL_ROWS + (size_t)n_meshes + 1;
  l.ddi = cv.take<float2>((size_t)n_points);
  l.all_mesh_off = cv.take<int>((size_t)n_meshes + 1);  // device copy of every mesh offset (the SELL build spans the batch)
  l.mesh_slice_off = cv.take<int>((size_t)n_meshes + 1);
  l.slice_ptr = cv.take<int>(n_slices + 1);
  l.slice_cnt = cv.take<int>(n_slices + 1);
  l.scan_tmp = cv.take<int>(scan_tmp_ints((int)n_slices + 1));
  l.entries = cv.take<int2>((size_t)std::max(sell_entries, 1LL));
  l.bytes = cv.used + 512;
  return l;
}

size_t focusr_eigs_workspace_bytes_mixed(int n_points, long long sell_entries_cap, int n_meshes, int max_mesh_points,
                                         int block_size) {
  return eigs_ws_layout(n_points, n_meshes, max_mesh_points, block_size, nullptr, nullptr, 0) +
         f32_layout(sell_entries_cap, n_points, n_meshes, nullptr).bytes;
}

void focusr_eigs_default_options(focusr_eigs_options* o) {
  o->mixed_precision = 1;
  o->filter_policy = 3;
  o->filter_prefetch = 1;
  o->filter_min_blocks = 8;
  o->filter_pdl = 2;
  o->nonsym_device = 1;
  for (int& r : o->reserved) r = 0;
}

int focusr_eigs_block_size(int k, int n_k_needed, int k_buffer, int max_one_way, int max_zero_rows) {
  // pinned pairs needed if the null space is {constant} + zero rows
  int k_cur = k;
  const int z = max_zero_rows + 1;
  while (k_cur - (z < k_cur ? z : k_cur) < n_k_needed) k_cur += k_buffer + n_k_needed;
  const int kp = k_cur - max_zero_rows > 1 ? k_cur - max_zero_rows : 1;
  int b = kp + (kp / 2 > 8 ? kp / 2 : 8);
  if (max_one_way > 0) b += 8 + 2 * (max_one_way < 8 ? max_one_way : 8);
  b = (b + 7) / 8 * 8;
  if (b < 16) b = 16;
  if (b > 96) b = 96;
  return b;
}

int focusr_eigs_smallest(const int* row_ptr, const int* cols, const double* weights, const double* degree,
                         const double* degree_inv, const double* points, int n_points,
                         const int* mesh_point_off_host, int n_meshes, const int* mesh_info_host, int k,
                         int n_k_needed, int k_buffer, double min_eig_val, double tol, int max_outer,
                         int block_size, double spectrum_upper_bound, double* eig_vals, double* eig_vecs,
                         int ldv, int* result_i_host,
                         double* result_d_host, void* workspace, size_t workspace_bytes,
                         const focusr_eigs_options* options, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  focusr_eigs_options opt;
  focusr_eigs_default_options(&opt);
  if (options) opt = *options;
  FB_REQUIRE(n_points > 0 && n_meshes > 0 && k >= 1 && n_k_needed >= 1 && ldv >= 1, "eigs: bad sizes");
  FB_REQUIRE(mesh_point_off_host[0] == 0 && mesh_point_off_host[n_meshes] == n_points,
             "eigs: mesh offsets must cover [0, n_points)");
  int max_oneway = 0, max_zero = 0, max_rows = 0;
  for (int m = 0; m < n_meshes; ++m) {
    max_oneway = std::max(max_oneway, mesh_info_host[FOCUSR_MESH_INFO_INTS * m + 1]);
    max_zero = std::max(max_zero, mesh_info_host[FOCUSR_MESH_INFO_INTS * m + 2]);
    max_rows = std::max(max_rows, mesh_point_off_host[m + 1] - mesh_point_off_host[m]);
    FB_REQUIRE(mesh_info_host[FOCUSR_MESH_INFO_INTS * m + 3] == 0,
               "eigs: mesh %d has %d non-finite edge weights (zero-length edges, graph.py:177-178)", m,
               mesh_info_host[FOCUSR_MESH_INFO_INTS * m + 3]);
  }
  const int B = block_size > 0 ? block_size
                               : focusr_eigs_block_size(k, n_k_needed, k_buffer, max_oneway, max_zero);
  FB_REQUIRE(spmm_block_supported(B), "eigs: block size %d unsupported (multiples of 8 up to 96)", B);
  FB_REQUIRE(max_rows > B, "eigs: a mesh has fewer vertices (%d) than the block size (%d)", max_rows, B);

  SolveParams p;
  p.k0 = k;
  p.n_needed = n_k_needed;
  p.k_buffer = k_buffer;
  p.min_eig = min_eig_val;
  p.tol = tol > 0.0 ? tol : 1e-10;
  p.max_outer = max_outer > 0 ? max_outer : 60;
  p.amp_target = 1e3;
  p.max_degree = 16384;
  // Gershgorin bound of the random-walk Laplacian: |L_ii| + sum_j |L_ij| = 2 d / (d + 1e-8) < 2
  p.beta = spectrum_upper_bound > 0.0 ? spectrum_upper_bound : 2.0;
  p.ldv = ldv;
  // 0: probe the top of the spectrum and filter only up to it; > 0: trust the caller; < 0: Gershgorin as is
  p.probe_degree = spectrum_upper_bound == 0.0 ? 10 : 0;
  p.land = SIZED_PASS_LAND;
  p.lowp_floor = LOWP_FLOOR;
  p.lowp_aim = LOWP_AIM;

  // fp32 copy of the matrix for the fp32 filter passes, at the end of the workspace if it has the room
  // (focusr_eigs_workspace_bytes_mixed); without it every pass is fp64
  F32Layout f32{};
  bool have_f32 = false;
  size_t ws_main = workspace_bytes;
  FilterTuning tune;
  tune.policy = opt.filter_policy;
  tune.prefetch = opt.filter_prefetch;
  tune.min_blocks = opt.filter_min_blocks;
  tune.pdl = opt.filter_pdl;
  {
    const long long sell_cap = sell_entries_cap(mesh_point_off_host, mesh_info_host, n_meshes, 0);
    const size_t extra = f32_layout(sell_cap, n_points, n_meshes, nullptr).bytes;
    const size_t base = eigs_ws_layout(n_points, n_meshes, max_rows, B, nullptr, nullptr, 0);
    if (opt.mixed_precision != 0 && workspace_bytes >= base + extra) {
      ws_main = workspace_bytes - extra;
      char* tail = reinterpret_cast<char*>(workspace) + ws_main;
      tail += (256 - (reinterpret_cast<uintptr_t>(tail) & 255)) & 255;
      f32 = f32_layout(sell_cap, n_points, n_meshes, tail);
      have_f32 = true;
      FB_CUDA(cudaMemcpyAsync(f32.all_mesh_off, mesh_point_off_host, sizeof(int) * ((size_t)n_meshes + 1), cudaMemcpyHostToDevice,
                              stream));
      const int rc = sell_build_f32(row_ptr, cols, weights, degree, degree_inv, f32.all_mesh_off, mesh_point_off_host, n_meshes,
                                    n_points, f32.mesh_slice_off, f32.slice_ptr, f32.entries, f32.ddi, f32.slice_cnt,
                                    f32.scan_tmp, stream);
      if (rc) return rc;
    }
  }
  // contiguous runs of meshes with the same symmetry class are solved as one batch
  int rc_all = FB_OK;
  std::vector<MeshResult> results(n_meshes);
  int m0 = 0;
  while (m0 < n_meshes) {
    const bool sym = mesh_info_host[FOCUSR_MESH_INFO_INTS * m0 + 1] == 0;
    int m1 = m0 + 1;
    while (m1 < n_meshes && (mesh_info_host[FOCUSR_MESH_INFO_INTS * m1 + 1] == 0) == sym) ++m1;
    const int M = m1 - m0;
    CudaBackend be;
    be.g = SpmmGraph{row_ptr, cols, weights, degree, degree_inv, nullptr, M, 0};
    be.mixed = opt.mixed_precision != 0;
    be.tune = tune;
    be.nonsym_device = opt.nonsym_device != 0;
    if (have_f32) {
      be.sell.entries = f32.entries;
      be.sell.slice_ptr = f32.slice_ptr;
      be.sell.mesh_slice_off = f32.mesh_slice_off + m0;
      be.sell.ddi = f32.ddi;
    }
    int run_max = 0;
    for (int m = m0; m < m1; ++m)
      run_max = std::max(run_max, mesh_point_off_host[m + 1] - mesh_point_off_host[m]);
    be.g.max_mesh_rows = run_max;
    const int run_rows = mesh_point_off_host[m1] - mesh_point_off_host[m0];
    const size_t need = eigs_ws_layout(run_rows, M, run_max, B, &be, workspace, ws_main);
    if (need > ws_main) {
      set_error("eigs: workspace too small (%zu < %zu)", ws_main, need);
      return FB_ERR_WORKSPACE;
    }
    // X/Y/Xn index rows globally: shift the base so that row r of the batch maps into the run's block
    const size_t shift = (size_t)mesh_point_off_host[m0] * B;
    be.X -= shift;
    be.Y -= shift;
    be.Xn -= shift;
    be.points = points;
    be.off_host = mesh_point_off_host + m0;
    be.info_host = mesh_info_host + FOCUSR_MESH_INFO_INTS * m0;
    be.M = M;
    be.B = B;
    be.mesh_base = m0;
    be.sym = sym;
    be.stream = stream;
    be.eig_vals = eig_vals;
    be.eig_vecs = eig_vecs;
    be.ldv = ldv;
    FB_CUDA(cudaMemcpyAsync(const_cast<int*>(be.g.mesh_off), mesh_point_off_host + m0, sizeof(int) * (M + 1),
                            cudaMemcpyHostToDevice, stream));
    const int rc = chfsi_solve(be, p, results.data() + m0);
    if (be.err != FB_OK) return be.err;
    FB_CUDA(cudaStreamSynchronize(stream));
    g_filter_profile.collect();
    g_filter_profile_lowp.collect();
    g_filter_profile_corr.collect();
    for (int m = m0; m < m1; ++m) {
      int* ri = result_i_host + 8 * m;
      ri[0] = results[m].status;
      ri[1] = results[m].n_out;
      ri[2] = results[m].k_final;
      ri[3] = results[m].outer_iters;
      ri[4] = results[m].total_degree;
      ri[5] = B;
      ri[6] = sym ? 1 : 0;
      ri[7] = results[m].lowp_degree;
      result_d_host[2 * m] = results[m].max_residual;
      result_d_host[2 * m + 1] = results[m].beta;
    }
    rc_all = std::max(rc_all, rc);
    m0 = m1;
  }
  if (rc_all != FB_OK)
    set_error("eigs: solver status %d (1 not converged, 2 block too small, 3 breakdown, 4 ldv too small); "
              "see result_i_host", rc_all);
  return rc_all;
}

// ---------------------------------------------------------------------------------------------
// row-partitioned multi-GPU solve
// ---------------------------------------------------------------------------------------------
int focusr_dist_unique_id(char* out128_host) {
  NcclApi& api = nccl_api();
  FB_REQUIRE(api.ok, "dist: libnccl.so.2 could not be loaded");
  ncclUniqueId id;
  const int rc = api.GetUniqueId(&id);
  FB_REQUIRE(rc == NCCL_SUCCESS, "dist: ncclGetUniqueId -> %s", api.GetErrorString(rc));
  memcpy(out128_host, id.internal, 128);
  return FB_OK;
}

int focusr_dist_init(const char* id128_host, int rank, int world) {
  NcclApi& api = nccl_api();
  FB_REQUIRE(api.ok, "dist: libnccl.so.2 could not be loaded");
  FB_REQUIRE(world >= 1 && rank >= 0 && rank < world, "dist: bad rank %d / world %d", rank, world);
  if (g_dist_comm) {
    api.CommDestroy(g_dist_comm);
    g_dist_comm = nullptr;
  }
  ncclUniqueId id;
  memcpy(id.internal, id128_host, 128);
  const int rc = api.CommInitRank(&g_dist_comm, world, id, rank);
  FB_REQUIRE(rc == NCCL_SUCCESS, "dist: ncclCommInitRank -> %s", api.GetErrorString(rc));
  g_dist_rank = rank;
  g_dist_world = world;
  return FB_OK;
}

int focusr_dist_finalize(void) {
  if (g_dist_comm) {
    nccl_api().CommDestroy(g_dist_comm);
    g_dist_comm = nullptr;
  }
  g_dist_world = 1;
  g_dist_rank = 0;
  return FB_OK;
}


// ---- IPC-shared region for the P2P-fused halo: [flags: world x 128 B][3 x rows_cap x B doubles] ----
static size_t shared_flag_bytes(int world) { return align_up((size_t)world * PEER_FLAG_BYTES); }

size_t focusr_dist_shared_bytes(int rows_cap, int block_size, int world) {
  return shared_flag_bytes(world) + 3 * align_up(sizeof(double) * (size_t)rows_cap * block_size);
}

int focusr_dist_shared_alloc(size_t bytes, char* handle64_host) {
  if (g_shared.base) {
    for (int p = 0; p < (int)g_shared.peer.size(); ++p)
      if (g_shared.peer[p] && p != g_shared.rank) cudaIpcCloseMemHandle(g_shared.peer[p]);
    cudaFree(g_shared.base);
    g_shared = PeerShared();
  }
  FB_CUDA(cudaMalloc(&g_shared.base, bytes));
  FB_CUDA(cudaMemset(g_shared.base, 0, bytes));
  g_shared.bytes = bytes;
  cudaIpcMemHandle_t h;
  FB_CUDA(cudaIpcGetMemHandle(&h, g_shared.base));
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(handle64_host, &h, 64);
  FB_CUDA(cudaDeviceSynchronize());
  return FB_OK;
}

int focusr_dist_shared_open(const char* handles_host, int rank, int world) {
  FB_REQUIRE(g_shared.base != nullptr, "dist_shared_open: allocate first");
  g_shared.peer.assign(world, nullptr);
  g_shared.world = world;
  g_shared.rank = rank;
  for (int p = 0; p < world; ++p) {
    if (p == rank) {
      g_shared.peer[p] = g_shared.base;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles_host + (size_t)p * 64, 64);
    FB_CUDA(cudaIpcOpenMemHandle(&g_shared.peer[p], h, cudaIpcMemLazyEnablePeerAccess));
  }
  return FB_OK;
}

int focusr_dist_shared_free(void) {
  if (g_shared.base) {
    for (int p = 0; p < (int)g_shared.peer.size(); ++p)
      if (g_shared.peer[p] && p != g_shared.rank) cudaIpcCloseMemHandle(g_shared.peer[p]);
    cudaFree(g_shared.base);
  }
  g_shared = PeerShared();
  return FB_OK;
}
static unsigned long long g_peer_epoch = 0;

static size_t dist_extra_layout(int n_send, int B, int world, DistCtx* d, Carver& cv) {
  double* sendbuf = cv.take<double>((size_t)std::max(n_send, 1) * B);
  const size_t small_n = std::max((size_t)2 * B * B, (size_t)4 * B * (world + 1));
  double* small = cv.take<double>(small_n);
  int* fake_off = cv.take<int>(2);
  const double** peer_blocks = cv.take<const double*>((size_t)3 * world);
  unsigned long long** peer_flags = cv.take<unsigned long long*>((size_t)world);
  int* dev_err = cv.take<int>(2);
  const float** peer_views = cv.take<const float*>((size_t)6 * world);
  unsigned* counter = cv.take<unsigned>(4);
  unsigned long long* timing = cv.take<unsigned long long>(4);
  if (d) {
    d->timing = timing;
    d->sendbuf = sendbuf;
    d->small = small;
    d->fake_off = fake_off;
    d->peer_blocks = peer_blocks;
    d->peer_flags = peer_flags;
    d->dev_err = dev_err;
    d->peer_views = peer_views;
    d->counter = counter;
  }
  return cv.used + 256;
}

static long long dist_sell_cap(int n_local, int max_row_entries) {
  return (long long)div_up(n_local, SELL_ROWS) * SELL_ROWS * (long long)std::max(max_row_entries, 1);
}

size_t focusr_eigs_dist_workspace_bytes(int n_local, int n_ghost, int n_send, int max_row_entries, int block_size, int world) {
  const size_t base = eigs_ws_layout(n_local + n_ghost, 1, n_local, block_size, nullptr, nullptr, 0);
  Carver cv(nullptr, 0);
  return align_up(base) + align_up(dist_extra_layout(n_send, block_size, world, nullptr, cv)) +
         f32_layout(dist_sell_cap(n_local, max_row_entries), n_local, 1, nullptr).bytes + 1024;
}

int focusr_eigs_smallest_dist(const int* row_ptr, const int* cols_local, const double* weights,
                              const double* degree, const double* degree_inv, const double* points,
                              int n_local, int n_ghost, long long row_begin_global, long long nnz_local,
                              const int* send_idx, int n_send, const int* send_counts_host,
                              const int* recv_counts_host, const int* ghost_peer, const int* ghost_row,
                              int ghost_base, const int* push_row, const int* push_dst, int n_push,
                              int use_p2p, int rows_cap, int n_zero_rows_global, int max_row_entries, int k,
                              int n_k_needed, int k_buffer, double min_eig_val, double tol, int max_outer,
                              int block_size, double spectrum_upper_bound, double* eig_vals, double* eig_vecs,
                              int ldv, int* result_i_host, double* result_d_host, void* workspace,
                              size_t workspace_bytes, const focusr_eigs_options* options, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  focusr_eigs_options opt;
  focusr_eigs_default_options(&opt);
  if (options) opt = *options;
  FB_REQUIRE(n_local > 0 && k >= 1 && n_k_needed >= 1 && ldv >= 1, "eigs_dist: bad sizes");
  FB_REQUIRE(g_dist_world == 1 || g_dist_comm != nullptr, "eigs_dist: call focusr_dist_init first");
  const int world = g_dist_world;
  const int B = block_size > 0 ? block_size : focusr_eigs_block_size(k, n_k_needed, k_buffer, 0, n_zero_rows_global);
  FB_REQUIRE(spmm_block_supported(B), "eigs_dist: block size %d unsupported", B);
  FB_REQUIRE(n_local > B, "eigs_dist: fewer local rows (%d) than the block size (%d)", n_local, B);
  SolveParams p;
  p.k0 = k;
  p.n_needed = n_k_needed;
  p.k_buffer = k_buffer;
  p.min_eig = min_eig_val;
  p.tol = tol > 0.0 ? tol : 1e-10;
  p.max_outer = max_outer > 0 ? max_outer : 60;
  p.amp_target = 1e3;
  p.max_degree = 16384;
  p.beta = spectrum_upper_bound > 0.0 ? spectrum_upper_bound : 2.0;
  p.ldv = ldv;
  // 0: probe the top of the spectrum and filter only up to it; > 0: trust the caller; < 0: Gershgorin as is
  p.probe_degree = spectrum_upper_bound == 0.0 ? 10 : 0;
  p.land = SIZED_PASS_LAND;
  p.lowp_floor = LOWP_FLOOR;
  p.lowp_aim = LOWP_AIM;

  DistCtx d;
  d.comm = g_dist_comm;
  d.rank = g_dist_rank;
  d.world = world;
  d.row_base = row_begin_global;
  d.n_loc = n_local;
  d.n_ghost = n_ghost;
  d.n_send = n_send;
  d.send_idx = send_idx;
  d.send_counts = send_counts_host;
  d.recv_counts = recv_counts_host;

  CudaBackend be;
  be.g = SpmmGraph{row_ptr, cols_local, weights, degree, degree_inv, nullptr, 1, n_local};
  const size_t base = eigs_ws_layout(n_local + n_ghost, 1, n_local, B, &be, workspace, workspace_bytes);
  Carver cv((char*)workspace + align_up(base), workspace_bytes > align_up(base) ? workspace_bytes - align_up(base) : 0);
  const size_t extra = align_up(dist_extra_layout(n_send, B, world, &d, cv));
  const long long sell_cap = dist_sell_cap(n_local, max_row_entries);
  const size_t f32_bytes = f32_layout(sell_cap, n_local, 1, nullptr).bytes;
  if (align_up(base) + extra + f32_bytes > workspace_bytes) {
    set_error("eigs_dist: workspace too small (%zu < %zu)", workspace_bytes, align_up(base) + extra + f32_bytes);
    return FB_ERR_WORKSPACE;
  }
  const F32Layout f32 = f32_layout(sell_cap, n_local, 1, (char*)workspace + align_up(base) + extra);
  const int off_host[2] = {0, n_local};
  const int info_host[FOCUSR_MESH_INFO_INTS] = {(int)nnz_local, 0, n_zero_rows_global, 0, 0, 0, 0, 0};
  const int fake[2] = {0, 1};
  be.points = points;
  be.off_host = off_host;
  be.info_host = info_host;
  be.M = 1;
  be.B = B;
  be.mesh_base = 0;
  be.sym = true;
  be.stream = stream;
  be.eig_vals = eig_vals;
  be.eig_vecs = eig_vecs;
  be.ldv = ldv;
  be.dist = &d;
  std::vector<const double*> pb_host;
  std::vector<const float*> pv_host;
  std::vector<unsigned long long*> pf_host;
  if (use_p2p && world > 1) {
    FB_REQUIRE(g_shared.base != nullptr && g_shared.world == world && (int)g_shared.peer.size() == world,
               "eigs_dist: P2P mode needs focusr_dist_shared_alloc/open first");
    FB_REQUIRE(ghost_base >= n_local && rows_cap >= ghost_base + n_ghost &&
                   focusr_dist_shared_bytes(rows_cap, B, world) <= g_shared.bytes,
               "eigs_dist: shared region too small for rows_cap=%d (ghost rows from %d, %d of them) block=%d", rows_cap,
               ghost_base, n_ghost, B);
    const size_t stride = align_up(sizeof(double) * (size_t)rows_cap * B) / sizeof(double);
    d.p2p = true;
    d.block_stride = stride;
    d.blocks = reinterpret_cast<double*>((char*)g_shared.base + shared_flag_bytes(world));
    d.flags = reinterpret_cast<unsigned long long*>(g_shared.base);
    d.ghost_peer = ghost_peer;
    d.ghost_row = ghost_row;
    d.epoch = g_peer_epoch;
    pb_host.resize((size_t)3 * world);
    pf_host.resize(world);
    for (int p = 0; p < world; ++p) {
      pf_host[p] = reinterpret_cast<unsigned long long*>(g_shared.peer[p]);
      for (int kb = 0; kb < 3; ++kb)
        pb_host[(size_t)kb * world + p] =
            reinterpret_cast<const double*>((char*)g_shared.peer[p] + shared_flag_bytes(world)) + (size_t)kb * stride;
    }
    FB_CUDA(cudaMemcpyAsync(const_cast<const double**>(d.peer_blocks), pb_host.data(), sizeof(double*) * 3 * world,
                            cudaMemcpyHostToDevice, stream));
    FB_CUDA(cudaMemcpyAsync(const_cast<unsigned long long**>(d.peer_flags), pf_host.data(), sizeof(void*) * world,
                            cudaMemcpyHostToDevice, stream));
    FB_CUDA(cudaMemsetAsync(d.dev_err, 0, sizeof(int) * 2, stream));
    FB_CUDA(cudaMemsetAsync(d.timing, 0, sizeof(unsigned long long) * 4, stream));
    be.X = d.blocks;
    be.Y = d.blocks + stride;
    be.Xn = d.blocks + 2 * stride;
    // fp32 views of the shared blocks: view 2 * block + half of rank p starts half * rows_cap * B floats into block `block`
    d.rows_cap = rows_cap;
    pv_host.resize((size_t)6 * world);
    for (int p = 0; p < world; ++p)
      for (int kb = 0; kb < 3; ++kb)
        for (int half = 0; half < 2; ++half)
          pv_host[(size_t)(2 * kb + half) * world + p] =
              reinterpret_cast<const float*>(pb_host[(size_t)kb * world + p]) + (size_t)half * rows_cap * B;
    FB_CUDA(cudaMemcpyAsync(const_cast<const float**>(d.peer_views), pv_host.data(), sizeof(float*) * 6 * world,
                            cudaMemcpyHostToDevice, stream));
  }
  FB_CUDA(cudaMemcpyAsync(const_cast<int*>(be.g.mesh_off), off_host, sizeof(off_host), cudaMemcpyHostToDevice, stream));
  FB_CUDA(cudaMemcpyAsync(d.fake_off, fake, sizeof(fake), cudaMemcpyHostToDevice, stream));
  // ghost rows of all three blocks start defined (the first exchange overwrites them)
  const size_t ext_rows = d.p2p ? (size_t)n_local : (size_t)(n_local + n_ghost);
  FB_CUDA(cudaMemsetAsync(be.X, 0, sizeof(double) * ext_rows * B, stream));
  FB_CUDA(cudaMemsetAsync(be.Y, 0, sizeof(double) * ext_rows * B, stream));
  FB_CUDA(cudaMemsetAsync(be.Xn, 0, sizeof(double) * ext_rows * B, stream));
  // fp32 filter passes: SELL copy of the local rows, remote columns encoded for the in-kernel peer gather.  P2P mode
  // only (the fp32 views live in the peer-shared blocks); the ncclSend/ncclRecv path keeps the fp64 steps.
  be.mixed = opt.mixed_precision != 0;
  be.nonsym_device = opt.nonsym_device != 0;
  be.tune.policy = opt.filter_policy;
  be.tune.prefetch = opt.filter_prefetch;
  be.tune.min_blocks = opt.filter_min_blocks;
  be.tune.pdl = opt.filter_pdl;
  if (d.p2p && be.mixed && max_row_entries > 0 && rows_cap < (1 << 24) && world <= 128) {
    const int rcs = sell_build_f32(row_ptr, cols_local, weights, degree, degree_inv, be.g.mesh_off, off_host, 1, n_local,
                                   f32.mesh_slice_off, f32.slice_ptr, f32.entries, f32.ddi, f32.slice_cnt, f32.scan_tmp,
                                   stream);
    if (rcs) return rcs;
    const int rcg = sell_remap_ghosts(f32.entries, sell_cap, f32.slice_ptr, div_up(n_local, SELL_ROWS), n_local, ghost_base,
                                      stream);
    if (rcg) return rcg;
    be.sell.entries = f32.entries;
    be.sell.slice_ptr = f32.slice_ptr;
    be.sell.mesh_slice_off = f32.mesh_slice_off;
    be.sell.ddi = f32.ddi;
    d.lowp = true;
    d.ghost_base = ghost_base;
    d.push_row = push_row;
    d.push_dst = push_dst;
    d.n_push = n_push;
  }
  FB_CUDA(cudaStreamSynchronize(stream));  // off_host / fake live on this stack frame
  MeshResult r;
  const int rc = chfsi_solve(be, p, &r);
  if (d.p2p) {
    // peers may still be reading this rank's blocks in their last step: leave together
    be.halo_exchange(be.X);
    g_peer_epoch = d.epoch;
    int herr[2] = {0, 0};
    unsigned long long tim[4] = {0, 0, 0, 0};
    cudaMemcpyAsync(herr, d.dev_err, sizeof(herr), cudaMemcpyDeviceToHost, stream);
    cudaMemcpyAsync(tim, d.timing, sizeof(tim), cudaMemcpyDeviceToHost, stream);
    cudaStreamSynchronize(stream);
    for (int i = 0; i < 4; ++i) g_persist_timing[i] = (double)tim[i];
    if (herr[0] != 0) {
      set_error("eigs_dist: a peer did not reach the inter-GPU barrier (time-out)");
      return FB_ERR_CUDA;
    }
  }
  if (be.err != FB_OK) return be.err;
  FB_CUDA(cudaStreamSynchronize(stream));
  g_filter_profile.collect();
  g_filter_profile_lowp.collect();
  g_filter_profile_corr.collect();
  result_i_host[0] = r.status;
  result_i_host[1] = r.n_out;
  result_i_host[2] = r.k_final;
  result_i_host[3] = r.outer_iters;
  result_i_host[4] = r.total_degree;
  result_i_host[5] = B;
  result_i_host[6] = r.lowp_degree;  // filter steps that ran in fp32 (0: every step fp64)
  result_i_host[7] = world;
  result_d_host[0] = r.max_residual;
  result_d_host[1] = r.beta;
  if (rc != FB_OK) set_error("eigs_dist: solver status %d", rc);
  return rc;
}
}
