// Test-only entry points into the eigensolver's kernels, one step at a time (tests/test_gpu_kernels.py).
//
// k_gram, k_gram_wide, k_reduce_gh, k_rotate and k_residual are internal to eigs.cu, so this file includes it; the
// library is linked from this object and the product's other objects (not eigs.o) with -Bsymbolic, so that nothing in
// it binds to a libfocusr_b200.so that is already loaded in the process.  The wrappers take device pointers and the
// caller's stream, allocate nothing and launch exactly what the solver launches: launch_filter_sell / launch_spmm with
// explicit arguments, and the Gram and rotation steps through CudaBackend's own dispatch.
#include "../../pyfocusr_b200/csrc/eigs.cu"

using namespace fb;

extern "C" {

const char* probe_last_error(void) { return focusr_last_error(); }

long long probe_sell_entries_cap(const int* off_host, const int* info_host, int n_meshes) {
  return sell_entries_cap(off_host, info_host, n_meshes, 0);
}

int probe_scan_tmp_ints(int n) { return (int)scan_tmp_ints(n); }

// sell_build_f32: slice_ptr [n_slices + 1], entries, ddi [n_rows], mesh_slice_off [n_meshes + 1]
int probe_sell_build(const int* row_ptr, const int* cols, const double* weights, const double* degree, const double* degree_inv,
                     const int* mesh_off, const int* off_host, int n_meshes, int n_rows, int* mesh_slice_off, int* slice_ptr,
                     int2* entries, float2* ddi, int* slice_cnt, int* scan_tmp, void* stream) {
  const int rc = sell_build_f32(row_ptr, cols, weights, degree, degree_inv, mesh_off, off_host, n_meshes, n_rows,
                                mesh_slice_off, slice_ptr, entries, ddi, slice_cnt, scan_tmp, (cudaStream_t)stream);
  if (rc) return rc;
  FB_LAUNCH_CHECK();
  return FB_OK;
}

// one k_filter_sell step (modes 0..4, sell.cu) with an explicit FilterTuning
int probe_filter_sell(int mode, int b, const int2* entries, const int* slice_ptr, const int* mesh_slice_off, const float2* ddi,
                      const int* mesh_off, int n_meshes, int max_mesh_rows, const void* y, const float* x_prev, const float* r,
                      void* out, float* y_copy, const void* alpha, const void* gamma, const double* center, int step,
                      int n_steps, int has_prev, int policy, int prefetch, int pdl, int min_blocks, void* stream) {
  FB_REQUIRE(mode >= 0 && mode <= 4, "probe_filter_sell: mode %d", mode);
  SellF32 m;
  m.entries = entries;
  m.slice_ptr = slice_ptr;
  m.mesh_slice_off = mesh_slice_off;
  m.ddi = ddi;
  FilterTuning tune;
  tune.policy = policy;
  tune.prefetch = prefetch;
  tune.pdl = pdl;
  tune.min_blocks = min_blocks;
  const int rc = launch_filter_sell(mode, b, m, mesh_off, n_meshes, max_mesh_rows, y, x_prev, r, out, y_copy, alpha, gamma,
                                    center, step, n_steps, has_prev != 0, tune, (cudaStream_t)stream);
  if (rc) return rc;
  FB_LAUNCH_CHECK();
  return FB_OK;
}

// one fp64 k_spmm launch (modes 0..2, spmm.cuh)
int probe_spmm(int mode, int b, const int* row_ptr, const int* cols, const double* weights, const double* degree,
               const double* degree_inv, const int* mesh_off, int n_meshes, int max_mesh_rows, const double* y,
               const double* x_prev, double* out, const double* alpha, const double* gamma, const double* center, int step,
               int n_steps, void* stream) {
  FB_REQUIRE(mode >= 0 && mode <= 2, "probe_spmm: mode %d", mode);
  SpmmGraph g{row_ptr, cols, weights, degree, degree_inv, mesh_off, n_meshes, max_mesh_rows};
  const int rc = launch_spmm(mode, b, g, y, x_prev, out, alpha, gamma, center, step, n_steps, (cudaStream_t)stream);
  if (rc) return rc;
  FB_LAUNCH_CHECK();
  return FB_OK;
}

// a backend that holds only what the Gram and rotation steps read
static CudaBackend probe_backend(int b, int n_meshes, const int* off_host, const double* degree, const double* degree_inv,
                                 const int* mesh_off, int chunks_max, void* stream) {
  CudaBackend be{};
  be.g = SpmmGraph{nullptr, nullptr, nullptr, degree, degree_inv, mesh_off, n_meshes, 0};
  be.off_host = off_host;
  be.M = n_meshes;
  be.B = b;
  be.chunks_max = chunks_max;
  be.stream = (cudaStream_t)stream;
  return be;
}

static bool probe_block_ok(int b) { return b >= 8 && b <= 96 && b % 8 == 0; }

// Gram pair of every mesh: CudaBackend::gram (k_gram for b < 64, k_gram_wide for b >= 64) into partial
// [n_meshes][chunks_max][2][b][b], then k_reduce_gh into G, H [n_meshes][b][b].  chunks_max = max_m ceil(rows_m / 1024).
int probe_gram(int b, int sym, const double* x, const double* z, const double* degree, const double* degree_inv,
               const int* mesh_off, const int* off_host, int n_meshes, int chunks_max, double* partial, double* g_out,
               double* h_out, void* stream) {
  FB_REQUIRE(probe_block_ok(b), "probe_gram: block size %d", b);
  CudaBackend be = probe_backend(b, n_meshes, off_host, degree, degree_inv, mesh_off, chunks_max, stream);
  be.sym = sym != 0;
  be.X = const_cast<double*>(x);
  be.Xn = const_cast<double*>(z);
  be.partial = partial;
  be.gram();
  if (be.err) return be.err;
  dim3 grid(div_up(b * b, 256), n_meshes);
  k_reduce_gh<<<grid, 256, 0, be.stream>>>(partial, chunks_max, mesh_off, b, g_out, h_out);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

// X <- X W and Z W per mesh with the residual sums (CudaBackend::rotate_and_residual: k_rotate, then k_residual):
// x [rows][b] is rotated in place, res [n_meshes][b] = ||dinv Z W - theta X W|| / ||X W|| per column, r_out [rows][b]
// the fp32 residual block dinv Z W - X W theta.  off_host[0] must be 0 (r_out is indexed by global row).
int probe_rotate(int b, double* x, const double* z, const double* w, const double* theta, const double* degree_inv,
                 const int* mesh_off, const int* off_host, int n_meshes, int chunks_max, double* partial_res, double* res,
                 float* r_out, void* stream) {
  FB_REQUIRE(probe_block_ok(b), "probe_rotate: block size %d", b);
  FB_REQUIRE(off_host[0] == 0, "probe_rotate: the first mesh must start at row 0");
  CudaBackend be = probe_backend(b, n_meshes, off_host, nullptr, degree_inv, mesh_off, chunks_max, stream);
  be.X = x;
  be.Xn = const_cast<double*>(z);
  be.W = const_cast<double*>(w);
  be.theta = const_cast<double*>(theta);
  be.partial_res = partial_res;
  be.res = res;
  // rotate_t writes the fp32 residual block to f32_view(Y, 0) when fp32 filter passes are available: with
  // off_host[0] == 0 that view starts at Y itself
  be.mixed = true;
  be.sell.entries = reinterpret_cast<const int2*>(r_out);
  be.Y = reinterpret_cast<double*>(r_out);
  be.rotate_and_residual();
  return be.err;
}

}  // extern "C"
