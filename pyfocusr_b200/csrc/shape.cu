// K13  Statistical shape models: generalized Procrustes analysis (GPA) and PCA of P configurations [P][N][3], every
// configuration being the N points of one template located on one subject.  Every sum has a fixed order and there are
// no floating-point atomics, so two runs give the same bits.
//   k_procrustes_fit   one FIT_THREADS CTA per configuration: vtkLandmarkTransform of the configuration onto the shared
//                      reference (landmark_fit.cuh, the fit of the ICP iterations), then aligned = matrix * configuration.
//                      A configuration's fit reads only that configuration and the reference: it does not depend on the
//                      batch it is in.
//   k_shape_mean_sum   raw mean of the aligned configurations, summed in p order, divided by P.
//   k_procrustes_mean  one CTA: the raw mean's fit onto the GPA reference, applied, and the RMS change against the
//                      previous mean.
//   k_shape_gram       partial Gram matrices of D = aligned - mean viewed as [P][3N] on the FP64 tensor pipe
//                      (mma.sync m8n8k4): one CTA per (32 x 32 block of the upper triangle, chunk of 3N); its 4 warps take
//                      a quarter of the chunk each and are added in warp order; k_shape_gram_sum adds the chunks in order
//                      and writes both triangles from the same sum, so G is exactly symmetric.
//   k_shape_modes      D^T W for a [P][K] matrix W, summed in p order.
#include <cmath>

#include "common.cuh"
#include "landmark_fit.cuh"

namespace fb {

constexpr int GRAM_BLK = 32;                           // configurations per side of a Gram block
constexpr int GRAM_WARPS = 4;
constexpr int GRAM_STEPS = 64;                         // k-steps of 4 per warp and chunk
constexpr int GRAM_CHUNK = GRAM_WARPS * GRAM_STEPS * 4;  // entries of 3N per CTA: 1024
constexpr int MODES_COLS = 8;                          // modes per thread of k_shape_modes

__device__ __forceinline__ void dmma884s(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ void apply_matrix(const double* m, const double* p, double* q) {  // 4x4 row-major
  const double x = p[0], y = p[1], z = p[2];
  q[0] = m[0] * x + m[1] * y + m[2] * z + m[3];
  q[1] = m[4] * x + m[5] * y + m[6] * z + m[7];
  q[2] = m[8] * x + m[9] * y + m[10] * z + m[11];
}

__global__ void __launch_bounds__(FIT_THREADS)
k_procrustes_fit(const double* __restrict__ configs, int N, const double* __restrict__ reference, int similarity,
                 double* __restrict__ mats, double* __restrict__ aligned) {
  __shared__ double red[FIT_THREADS];
  __shared__ double Ls[16];
  const size_t base = 3 * (size_t)N * blockIdx.x;
  double Lm[16];
  if (landmark_fit_block(configs + base, reference, N, similarity, red, Lm))
    for (int i = 0; i < 16; ++i) {
      mats[16 * (size_t)blockIdx.x + i] = Lm[i];
      Ls[i] = Lm[i];
    }
  if (aligned == nullptr) return;
  __syncthreads();
  for (int i = threadIdx.x; i < N; i += FIT_THREADS) apply_matrix(Ls, configs + base + 3 * (size_t)i, aligned + base + 3 * (size_t)i);
}

__global__ void __launch_bounds__(256)
k_shape_mean_sum(const double* __restrict__ aligned, int P, long long n3, double* __restrict__ raw) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n3) return;
  double s = 0.0;
  for (int p = 0; p < P; ++p) s += aligned[(size_t)p * n3 + j];
  raw[j] = s / P;
}

__global__ void __launch_bounds__(FIT_THREADS)
k_procrustes_mean(const double* __restrict__ raw, int N, const double* __restrict__ reference, int similarity,
                  const double* prev, double* mean_out, double* __restrict__ change_out) {
  __shared__ double red[FIT_THREADS];
  __shared__ double Ls[16];
  double Lm[16];
  if (landmark_fit_block(raw, reference, N, similarity, red, Lm))
    for (int i = 0; i < 16; ++i) Ls[i] = Lm[i];
  __syncthreads();
  double s = 0.0;
  for (int i = threadIdx.x; i < N; i += FIT_THREADS) {  // point i is read and written by this thread alone
    double q[3];
    apply_matrix(Ls, raw + 3 * (size_t)i, q);
    for (int d = 0; d < 3; ++d) {
      const double e = q[d] - prev[3 * (size_t)i + d];
      s += e * e;
      mean_out[3 * (size_t)i + d] = q[d];
    }
  }
  const double total = fit_block_sum(s, red);
  if (threadIdx.x == 0) *change_out = sqrt(total / N);
}

// block pair bp of the upper triangle (row-major over bi <= bj) of nb x nb blocks
__device__ __forceinline__ void gram_block_pair(int bp, int nb, int& bi, int& bj) {
  bi = 0;
  while (bp >= nb - bi) {
    bp -= nb - bi;
    ++bi;
  }
  bj = bi + bp;
}

// DMMA m8n8k4: lane l holds A[l>>2][l&3] and B[l&3][l>>2] and accumulates D[l>>2][2(l&3)+{0,1}].  With A = D rows of
// block bi and B = D rows of block bj (both over the same 4 entries of 3N) the tile is a block of D D^T.
__global__ void __launch_bounds__(32 * GRAM_WARPS)
k_shape_gram(const double* __restrict__ aligned, const double* __restrict__ mean, int P, long long n3, int nb,
             double* __restrict__ partial) {
  __shared__ double red[GRAM_WARPS][GRAM_BLK * GRAM_BLK];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, kq = lane & 3, cc = lane >> 2;
  int bi, bj;
  gram_block_pair(blockIdx.x, nb, bi, bj);
  const long long r0 = (long long)blockIdx.y * GRAM_CHUNK + (long long)warp * GRAM_STEPS * 4;
  const double* ra[4];
  const double* rb[4];
  bool oka[4], okb[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int pa = GRAM_BLK * bi + 8 * t + cc, pb = GRAM_BLK * bj + 8 * t + cc;
    oka[t] = pa < P;
    okb[t] = pb < P;
    ra[t] = aligned + (size_t)(oka[t] ? pa : 0) * n3;
    rb[t] = aligned + (size_t)(okb[t] ? pb : 0) * n3;
  }
  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  for (int s = 0; s < GRAM_STEPS; ++s) {
    const long long r = r0 + 4 * s + kq;
    const bool okr = r < n3;
    const double mu = okr ? mean[r] : 0.0;
    double a[4], b[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      a[t] = (okr && oka[t]) ? ra[t][r] - mu : 0.0;
      b[t] = (okr && okb[t]) ? rb[t][r] - mu : 0.0;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dmma884s(acc[i][j][0], acc[i][j][1], a[i], b[j]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      double* o = &red[warp][(8 * i + cc) * GRAM_BLK + 8 * j + 2 * kq];
      o[0] = acc[i][j][0];
      o[1] = acc[i][j][1];
    }
  __syncthreads();
  double* out = partial + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * (GRAM_BLK * GRAM_BLK);
  for (int e = threadIdx.x; e < GRAM_BLK * GRAM_BLK; e += 32 * GRAM_WARPS)
    out[e] = ((red[0][e] + red[1][e]) + red[2][e]) + red[3][e];
}

__global__ void __launch_bounds__(256)
k_shape_gram_sum(const double* __restrict__ partial, int P, int nb, int n_bp, int chunks, double* __restrict__ gram) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= (long long)P * P) return;
  const int p = (int)(k / P), q = (int)(k % P);
  const int a = min(p, q), b = max(p, q);  // both triangles from the entry of the upper one
  const int bi = a / GRAM_BLK, bj = b / GRAM_BLK;
  const int bp = bi * nb - bi * (bi - 1) / 2 + (bj - bi);
  const int e = (a % GRAM_BLK) * GRAM_BLK + b % GRAM_BLK;
  double s = 0.0;
  for (int c = 0; c < chunks; ++c) s += partial[((size_t)c * n_bp + bp) * (GRAM_BLK * GRAM_BLK) + e];
  gram[k] = s;
}

// modes[k][r] = sum_p (aligned[p][r] - mean[r]) W[p][k] for MODES_COLS modes per thread
__global__ void __launch_bounds__(256)
k_shape_modes(const double* __restrict__ aligned, const double* __restrict__ mean, int P, long long n3,
              const double* __restrict__ W, int K, double* __restrict__ modes) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int k0 = blockIdx.y * MODES_COLS;
  if (r >= n3) return;
  const double mu = mean[r];
  double acc[MODES_COLS];
#pragma unroll
  for (int j = 0; j < MODES_COLS; ++j) acc[j] = 0.0;
  for (int p = 0; p < P; ++p) {
    const double d = aligned[(size_t)p * n3 + r] - mu;
#pragma unroll
    for (int j = 0; j < MODES_COLS; ++j)
      if (k0 + j < K) acc[j] += d * W[(size_t)p * K + k0 + j];
  }
#pragma unroll
  for (int j = 0; j < MODES_COLS; ++j)
    if (k0 + j < K) modes[(size_t)(k0 + j) * n3 + r] = acc[j];
}

static int gram_blocks(int P) { return div_up(P, GRAM_BLK); }
static int gram_chunks(int N) { return div_up(3LL * N, GRAM_CHUNK); }

}  // namespace fb

using namespace fb;

extern "C" {

int focusr_procrustes_fit(const double* configs, int n_configs, int n_points, const double* reference, int similarity,
                          double* mats_out, double* aligned_out, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_configs > 0 && n_points > 0, "procrustes_fit: empty input (%d configurations of %d points)", n_configs, n_points);
  FB_REQUIRE(configs && reference && mats_out, "procrustes_fit: missing device array");
  FB_REQUIRE(aligned_out != configs || aligned_out == nullptr, "procrustes_fit: aligned_out must not alias configs");
  FB_REQUIRE(3LL * n_points < INT32_MAX, "procrustes_fit: at most %d points", INT32_MAX / 3);
  k_procrustes_fit<<<n_configs, FIT_THREADS, 0, stream>>>(configs, n_points, reference, similarity ? 1 : 0, mats_out,
                                                           aligned_out);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

size_t focusr_procrustes_mean_workspace_bytes(int n_points) {
  if (n_points <= 0) return 0;
  return align_up(sizeof(double) * 3 * (size_t)n_points) + 256;
}

int focusr_procrustes_mean(const double* aligned, int n_configs, int n_points, const double* reference, int similarity,
                           const double* prev_mean, double* mean_out, double* change_out, void* workspace,
                           size_t workspace_bytes, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_configs > 0 && n_points > 0, "procrustes_mean: empty input (%d configurations of %d points)", n_configs, n_points);
  FB_REQUIRE(aligned && reference && prev_mean && mean_out && change_out, "procrustes_mean: missing device array");
  FB_REQUIRE(3LL * n_points < INT32_MAX, "procrustes_mean: at most %d points", INT32_MAX / 3);
  Carver cv(workspace, workspace_bytes);
  double* raw = cv.take<double>(3 * (size_t)n_points);
  if (!cv.ok()) {
    set_error("procrustes_mean: workspace too small (%zu < %zu)", workspace_bytes, cv.used);
    return FB_ERR_WORKSPACE;
  }
  const long long n3 = 3LL * n_points;
  k_shape_mean_sum<<<div_up(n3, 256), 256, 0, stream>>>(aligned, n_configs, n3, raw);
  k_procrustes_mean<<<1, FIT_THREADS, 0, stream>>>(raw, n_points, reference, similarity ? 1 : 0, prev_mean, mean_out,
                                                   change_out);
  FB_COUNT_LAUNCH(2);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

size_t focusr_shape_gram_workspace_bytes(int n_configs, int n_points) {
  if (n_configs <= 0 || n_points <= 0) return 0;
  const size_t nb = (size_t)gram_blocks(n_configs), n_bp = nb * (nb + 1) / 2;
  return align_up(sizeof(double) * (size_t)gram_chunks(n_points) * n_bp * GRAM_BLK * GRAM_BLK) + 256;
}

int focusr_shape_gram(const double* aligned, const double* mean, int n_configs, int n_points, double* gram_out,
                      void* workspace, size_t workspace_bytes, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_configs > 0 && n_points > 0, "shape_gram: empty input (%d configurations of %d points)", n_configs, n_points);
  FB_REQUIRE(aligned && mean && gram_out, "shape_gram: missing device array");
  const int nb = gram_blocks(n_configs), n_bp = nb * (nb + 1) / 2, chunks = gram_chunks(n_points);
  FB_REQUIRE(chunks <= 65535, "shape_gram: at most %d points", 65535 * (GRAM_CHUNK / 3));
  Carver cv(workspace, workspace_bytes);
  double* partial = cv.take<double>((size_t)chunks * n_bp * GRAM_BLK * GRAM_BLK);
  if (!cv.ok()) {
    set_error("shape_gram: workspace too small (%zu < %zu)", workspace_bytes, cv.used);
    return FB_ERR_WORKSPACE;
  }
  k_shape_gram<<<dim3(n_bp, chunks), 32 * GRAM_WARPS, 0, stream>>>(aligned, mean, n_configs, 3LL * n_points, nb, partial);
  k_shape_gram_sum<<<div_up((long long)n_configs * n_configs, 256), 256, 0, stream>>>(partial, n_configs, nb, n_bp, chunks,
                                                                                       gram_out);
  FB_COUNT_LAUNCH(2);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

int focusr_shape_modes(const double* aligned, const double* mean, int n_configs, int n_points, const double* weights,
                       int n_modes, double* modes_out, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(n_configs > 0 && n_points > 0 && n_modes > 0, "shape_modes: empty input (%d configurations of %d points, %d modes)",
             n_configs, n_points, n_modes);
  FB_REQUIRE(aligned && mean && weights && modes_out, "shape_modes: missing device array");
  FB_REQUIRE(div_up(n_modes, MODES_COLS) <= 65535, "shape_modes: too many modes (%d)", n_modes);
  const long long n3 = 3LL * n_points;
  k_shape_modes<<<dim3(div_up(n3, 256), div_up(n_modes, MODES_COLS)), 256, 0, stream>>>(aligned, mean, n_configs, n3, weights,
                                                                                        n_modes, modes_out);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

}  // extern "C"
