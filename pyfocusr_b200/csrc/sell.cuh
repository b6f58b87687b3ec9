// internal interface of sell.cu: sliced-ELL (SELL-64) copies of the adjacency for the two HBM-bound hot loops
// (the fp32 Chebyshev filter steps of the eigensolver and the smoothing passes of Graph.mean_filter_graph).
#pragma once
#include <cuda_runtime.h>

namespace fb {

constexpr int SELL_ROWS = 64;  // rows per slice = rows one CTA pass of the filter kernels covers

// fp32 copy of the adjacency in SELL-64 form.  Slice s covers 64 consecutive rows of ONE mesh (a mesh starts a new
// slice); its k-th entries lie together: entry k of row r (0..63) at slice_ptr[s] + k * 64 + r, an 8-byte
// {column, weight as float bits} pair, so a pass of the kernel reads one coalesced 512-byte line per k and needs no
// row pointer (the dependent chain row_ptr -> entry -> gather loses its first link, and the trip count is uniform
// over the CTA pass).  Rows shorter than the slice width are padded with {first row of the slice, 0.0f}.
struct SellF32 {
  const int2* entries = nullptr;
  const int* slice_ptr = nullptr;       // device [n_slices + 1], multiples of 64
  const int* mesh_slice_off = nullptr;  // device [n_meshes + 1]: first slice of every mesh of the RUN
  const float2* ddi = nullptr;          // [n_rows] (degree, 1/(degree + 1e-8)), indexed by global row
};

// exact upper bound of the entry count of the SELL copies from the per-mesh facts of focusr_laplacian_build
// (mesh_info[m][4] = longest row): sum over meshes of ceil(rows / 64) * 64 * longest row
long long sell_entries_cap(const int* mesh_point_off_host, const int* mesh_info_host, int n_meshes, int extra_per_row);
int sell_slice_count(const int* mesh_point_off_host, int n_meshes);

// builds the fp32 SELL copy of meshes [0, n_meshes) given by mesh_off (device) / mesh_point_off_host.
// slice_cnt / scan_tmp: scratch of n_slices + 1 ints / scan_tmp_ints(n_slices + 1) ints.
int sell_build_f32(const int* row_ptr, const int* cols, const double* weights, const double* degree,
                   const double* degree_inv, const int* mesh_off, const int* mesh_point_off_host, int n_meshes,
                   int n_rows, int* mesh_slice_off, int* slice_ptr, int2* entries, float2* ddi, int* slice_cnt,
                   int* scan_tmp, cudaStream_t stream);

// per-call tuning of the filter-step kernels (focusr_eigs_options in the C ABI)
struct FilterTuning {
  int policy = 3;    // bit 1 = no L1 allocation + L2 evict_first on the single-use streams (entries, z_prev, r, stores);
                     // bit 0 = L2 evict_last on the gathered block; default both
  int prefetch = 1;  // ask L2 early for the CTA's streams
  int min_blocks = 8;  // resident CTAs per SM the b = 16 kernels are compiled for (8, 6 or 5)
  int pdl = 2;       // 0 = plain launches, 1 = programmatic dependent launch, 2 = + the prefetch of the streams the previous
                     // step does not write is issued before the dependency wait
};

// One Chebyshev filter step on the SELL copy.  mode: 0 plain fp32 step (y, x_prev, out fp32), 1 first step of a pass (y
// fp64 -> out fp32, y_copy = fp32 copy of y), 2 last step (out fp64), 3 correction step (z, z_prev, r -> z_next; per-column
// float tables), 4 last correction step (x += z_next in fp64).
int launch_filter_sell(int mode, int b, const SellF32& m, const int* mesh_off, int n_meshes, int max_mesh_rows,
                       const void* y, const float* x_prev, const float* r, void* out, float* y_copy,
                       const void* alpha, const void* gamma, const double* center, int step, int n_steps, bool has_prev,
                       const FilterTuning& tune, cudaStream_t stream);

// ---- row-partitioned solve: all steps of a filter pass in one persistent cooperative kernel per GPU (sell.cu) ----
struct PersistArgs {
  const int2* entries;       // SELL copy of the LOCAL rows; ghost columns point at the views' ghost rows (sell_remap_ghosts)
  const int* slice_ptr;
  const float2* ddi;
  int n_loc;
  int n_units, units_per_cta;              // filled by the launcher (units = CTA passes of 256 / TPR rows)
  int ghost_base;                          // first ghost row of a view (same on every rank)
  const int* push_row;                     // push list, sorted by row: local rows some peer gathers ...
  const int* push_dst;                     // ... and where they go: (peer << 24) | ghost slot on that peer
  int n_push;
  int push_first;                          // the view gathered by the first step still needs its ghost rows filled
  const float* const* peer_views;          // device [6][world]: fp32 view v (= 2 * block + half) of rank p's blocks
  int world, rank;
  int v_prev, v_cur, v_next;               // views at the first step of this launch
  const float* r;                          // correction form: the fp32 residual block (local)
  double* x;                               // fp64 block the last step writes (plain) or updates (correction)
  const void* alpha;                       // this launch's tables: double [len] (plain) or float [len][B] (correction)
  const void* gamma;
  const double* center;
  int s0, len, deg;                        // first step, steps of this launch, steps of the pass
  int prefetch;                            // L2 prefetch of the next unit's streams (pays when the rank's rows exceed L2)
  unsigned* counter;                       // zeroed before the launch: arrivals of this GPU's CTAs
  unsigned long long* my_flags;            // one 128-byte line per rank
  unsigned long long* const* peer_flags;   // device [world]
  unsigned long long epoch0;               // step s of the launch publishes epoch0 + 1 + s
  int* err;
  unsigned long long* timing;              // nullable: {ns at barriers, ns working, steps} of CTA 0 are added here
};
int launch_filter_persist(bool corr, int b, const PersistArgs& a, cudaStream_t stream);
int sell_remap_ghosts(int2* entries, long long n_entries_cap, const int* slice_ptr, int n_slices, int n_loc, int ghost_base,
                      cudaStream_t stream);
int block_to_f32(const double* x, float* out, long long n, cudaStream_t stream);

}  // namespace fb
