/* libfocusr_b200 -- C ABI of the B200 (sm_100a) spectral-correspondence hot path of PyFOCUSR.
 *
 * The reference (gattia/pyfocusr) has no FFI: its boundary is the Python class API
 * (pyfocusr/focusr.py:22-69, pyfocusr/graph.py:18-34, pyfocusr/eigsort.py:9-22).  The Python
 * drop-in classes in pyfocusr_b200/ keep that API and bind the entry points below with ctypes
 * (pyfocusr_b200/_lib.py); each entry point names the reference code it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it except
 *     focusr_laplacian_build (validates triangle indices) and focusr_eigs_smallest (reads Ritz
 *     values back to drive the outer loop), which synchronise it;
 *   - the library never allocates device memory: callers pass workspaces sized by the matching
 *     *_workspace_bytes() function (PyTorch's caching allocator owns all HBM);
 *   - return value 0 = success; otherwise an error code and focusr_last_error() describes it;
 *   - dense matrices are row-major; eigenvector / feature blocks are [n_points][ld];
 *   - a "batch" is a set of meshes concatenated into one block-diagonal graph: vertex ids in
 *     `tris` are global, `mesh_point_off[m] .. mesh_point_off[m+1]` are mesh m's rows.
 */
#ifndef FOCUSR_B200_H
#define FOCUSR_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* focusr_stream_t;

/* ints per mesh in `mesh_info`: {nnz(A), one-way entries (A_ij stored, A_ji not), zero-degree rows, non-finite
 * weights, longest row, 0, 0, 0} */
#define FOCUSR_MESH_INFO_INTS 8

const char* focusr_last_error(void);
int focusr_version(void);
/* kernels launched by this library since load (bench.py's `gpu_launches`) */
unsigned long long focusr_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * K1  Laplacian assembly.  Replaces Graph.get_weighted_adjacency_matrix (graph.py:148-178: the
 * Python loop over cells x edges filling a lil_matrix), get_degree_matrix (graph.py:216-219).
 * Output: canonical CSR of the weighted adjacency A (columns ascending, duplicates collapsed),
 * degree d = A.sum(axis=1) (sequential ascending-column sum, bit-identical to scipy) and
 * 1/(d+1e-8).  `cols`/`weights` need capacity 3*n_tris.  `mesh_info` is [n_meshes][FOCUSR_MESH_INFO_INTS] int
 * (layout above).
 * `points` is [n_points][point_dim]: point_dim = 3 (xyz) by default, or 3 + f when
 * include_features_in_adj_matrix appends f range-scaled node features to the position
 * (graph.py:166-175); the edge weight is 1/||p1 - p2|| over all point_dim coordinates.
 * ------------------------------------------------------------------------------------------- */
size_t focusr_laplacian_workspace_bytes(int n_points, int n_tris);
int focusr_laplacian_build(const double* points, int point_dim, const int* tris, int n_points, int n_tris,
                           const int* mesh_point_off, int n_meshes, int* row_ptr, int* cols,
                           double* weights, double* degree, double* degree_inv, int* mesh_info,
                           void* workspace, size_t workspace_bytes, focusr_stream_t stream);

/* L = D~^-1 (D - A) as CSR with sorted columns and explicit zeros dropped, i.e. what
 * Graph.get_laplacian_matrix (graph.py:221-226) produces after sort_indices().  The solver does
 * not need it (it applies L from A, d, 1/(d+1e-8)); it exists for Graph.laplacian_matrix.
 * `l_cols`/`l_vals` need capacity nnz(A) + n_points. */
int focusr_laplacian_csr(const int* row_ptr, const int* cols, const double* weights,
                         const double* degree, const double* degree_inv, int n_points,
                         int* l_row_ptr, int* l_cols, double* l_vals, void* workspace,
                         size_t workspace_bytes, focusr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * K5  Graph.mean_filter_graph (graph.py:320-354): values <- M^iterations values with
 * M = diag(1/(1+d)) (A + I), for rows [row_begin, row_end) of the batch graph, which must be whole meshes
 * (values are indexed by global row; values_in is not modified; the result lands in values_out).
 * Accumulation order and rounding reproduce scipy's CSR product bit-for-bit (descending columns, multiply
 * then add).  The passes are chained by programmatic dependent launch.  The workspace holds the two ping-pong
 * iterates (not needed for a single iteration).
 * ------------------------------------------------------------------------------------------- */
size_t focusr_mean_filter_workspace_bytes(int n_rows, int n_cols);
int focusr_mean_filter(const int* row_ptr, const int* cols, const double* weights,
                       const double* degree, int row_begin, int row_end, const double* values_in,
                       double* values_out, int n_cols, int iterations, void* workspace,
                       size_t workspace_bytes, focusr_stream_t stream);

/* out[i][:] = in[idx[i]][:]  (focusr.py:387 `smoothed_target_coords[corresponding_idx, :]`;
 * focusr.py:429-431 nearest-neighbour positions).  `idx_base[i]` (nullable) is added to idx[i]. */
int focusr_gather_rows(const double* in, const long long* idx, const int* idx_base, int n_rows,
                       int n_cols, double* out, focusr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * K2  recursive_eig (graph.py:357-389) = scipy eigs(L, k, sigma=1e-10, which="LM", ncv=4k) +
 * retry while fewer than n_k_needed eigenvalues exceed min_eig_val.  Returns, per mesh, the
 * eigenpairs with eigenvalue > min_eig_val among the k_final smallest, ascending, eigenvectors
 * with unit 2-norm and the largest-magnitude entry positive.  SYNCHRONISES the stream (once per
 * outer iteration).  `mesh_info_host` is focusr_laplacian_build's mesh_info copied to the host.
 * result_i_host [n_meshes][8]: {status, n_found, k_final, outer_iterations, total_filter_degree,
 * block_size, symmetric, filter steps that ran in fp32 (of the total, plus the probe's)};
 * result_d_host [n_meshes][2]: {max_residual, upper edge of the filter interval}.
 * Mixed precision (symmetric adjacencies): a filter pass that is meant to leave residuals above the fp32 floor
 * (1.4e-6) runs with fp32 vector blocks (k_filter_sell on a sliced-ELL fp32 copy of the matrix, 47% fewer bytes per
 * step); a pass that lands lower runs in fp32 CORRECTION form: only z = p(L) x - x is iterated in fp32, driven by the fp64 residual of the
 * Ritz pairs, so rounding is relative to the error of x, and x += z is fp64 (34% fewer bytes per step).
 * Rayleigh-Ritz and every residual that is tested are fp64, so the returned pairs meet `tol` in fp64 either way.
 * options->mixed_precision = 0 keeps every pass in fp64.
 * status: 0 ok, 1 not converged, 2 block too small, 3 numerical breakdown, 4 ldv too small.
 * `spectrum_upper_bound`: > 0 = filter up to this caller-guaranteed bound; 0 = start from the
 * Gershgorin bound 2 and, for symmetric adjacencies, tighten it per mesh with a 10-step probe of the
 * top of the spectrum (triangle meshes sit near 1.5; the degree scales with sqrt of the bound; an
 * underestimate is detected and reverts to 2); < 0 = Gershgorin bound as is.
 * ------------------------------------------------------------------------------------------- */
size_t focusr_eigs_workspace_bytes(int n_points, int n_meshes, int max_mesh_points, int block_size);
/* The same plus room for the fp32 copy of the matrix that the fp32 filter passes read (sliced-ELL: 8 bytes per padded
 * entry, `sell_entries_cap` of them = focusr_sell_entries_cap(...); 8 bytes per row); focusr_eigs_smallest takes fp32
 * passes only when the workspace it is given is at least this large. */
long long focusr_sell_entries_cap(const int* mesh_point_off_host, const int* mesh_info_host, int n_meshes);
size_t focusr_eigs_workspace_bytes_mixed(int n_points, long long sell_entries_cap, int n_meshes,
                                         int max_mesh_points, int block_size);
/* Per-call options of the eigensolver (NULL = defaults; no process-wide state).  filter_* select the kernel form of
 * the fp32 filter steps and exist for A/B measurements (csrc/sell.cu has the record). */
typedef struct focusr_eigs_options {
  int mixed_precision;   /* 1 (default): fp32 filter passes for symmetric adjacencies; 0: every pass fp64 */
  int filter_policy;     /* fp32 filter steps: bit 1 = no L1 allocation + L2 evict_first on the single-use streams,
                            bit 0 = L2 evict_last on the gathered block; default 3 = both */
  int filter_prefetch;   /* 1 (default): the CTA asks L2 early for the lines it will stream */
  int filter_min_blocks; /* resident CTAs per SM the b = 16 kernels are compiled for: 8 (default), 6 or 5 */
  int filter_pdl;        /* 2 (default): steps chained by programmatic dependent launch, constant streams prefetched
                            before the dependency wait; 1: the same, prefetch after the wait; 0: plain launches */
  int nonsym_device;     /* 1 (default): the b x b general Rayleigh-Ritz step of non-symmetric adjacencies (open /
                            non-manifold meshes) runs on the device, one CTA per mesh (b <= 64); 0: on the host */
  int reserved[10];
} focusr_eigs_options;
void focusr_eigs_default_options(focusr_eigs_options* options);
int focusr_eigs_block_size(int k, int n_k_needed, int k_buffer, int max_one_way, int max_zero_rows);
int focusr_eigs_smallest(const int* row_ptr, const int* cols, const double* weights,
                         const double* degree, const double* degree_inv, const double* points,
                         int n_points, const int* mesh_point_off_host, int n_meshes,
                         const int* mesh_info_host, int k, int n_k_needed, int k_buffer,
                         double min_eig_val, double tol, int max_outer, int block_size,
                         double spectrum_upper_bound,
                         double* eig_vals, double* eig_vecs, int ldv, int* result_i_host,
                         double* result_d_host, void* workspace, size_t workspace_bytes,
                         const focusr_eigs_options* options, focusr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * K2, row-partitioned across GPUs (BASELINE.json configs[3]; SURVEY.md section 8e-ii): ONE mesh,
 * rank r owns the contiguous rows [row_begin_global, row_begin_global + n_local) of the symmetric
 * adjacency.  `cols_local` are remapped columns: j in the local block -> j - row_begin_global,
 * remote j -> n_local + (position of j in the rank's sorted ghost list, which is grouped by owner).
 * Before every SpMM the ghost rows of the vector block are refreshed by one grouped
 * ncclSend/ncclRecv of the boundary rows (`send_idx`: device list of local rows to ship, grouped by
 * destination; `send_counts_host` / `recv_counts_host` [world]); Gram blocks, residual sums, the
 * bounding box and the eigenvector norms are all-reduced.  NCCL is resolved at run time from the
 * already-loaded libnccl.so.2; the library creates its own communicator from a 128-byte unique id
 * (rank 0: focusr_dist_unique_id, broadcast by the caller, then focusr_dist_init on every rank).
 * Every rank runs the same driver and sees identical Ritz values, so all control decisions agree.
 * Outputs: eig_vals [ldv] (identical on all ranks), eig_vecs [n_local][ldv] (this rank's rows).
 *
 * P2P mode (use_p2p = 1): the halo is FUSED into the SpMM.  Every rank keeps its three vector blocks
 * in a region shared through CUDA IPC (focusr_dist_shared_alloc -> 64-byte handle, exchanged by the
 * caller, focusr_dist_shared_open) and the kernel gathers a remote column straight from the owning
 * rank's HBM over NVLink (ghost g lives at row ghost_row[g] of rank ghost_peer[g]); no pack / send /
 * receive, no ghost copies, and the steps are ordered by a flag barrier in peer memory instead of a
 * collective.  `rows_cap` = rows of a block in the shared region (identical layout on every rank).
 * In P2P mode the filter passes take the fp32 forms of the single-GPU solver (plain fp32 blocks, then the correction
 * form) on fp32 views of the shared blocks, and ALL steps of a pass run in ONE persistent cooperative kernel per GPU
 * (k_filter_persist): every fp32 view carries ghost rows from row `ghost_base` on (= the largest n_local of any rank;
 * `rows_cap` >= ghost_base + the largest n_ghost), a rank PUSHES the rows its peers gather into their ghost rows with
 * posted NVLink stores as soon as it has written them (`push_row` [n_push] sorted local rows, `push_dst` [n_push] =
 * (peer << 24) | ghost slot on that peer), and the steps are separated by an in-kernel barrier (local arrival counter +
 * one flag line per peer) -- no launch, no collective and no host involvement per step.  `max_row_entries` = longest
 * local row (sizes the sliced-ELL copy).  result_i_host = {status, n_found, k_final, outer_iterations, total_filter_degree, block_size,
 * filter steps that ran in fp32, world}.
 * ------------------------------------------------------------------------------------------- */
size_t focusr_dist_shared_bytes(int rows_cap, int block_size, int world);
int focusr_dist_shared_alloc(size_t bytes, char* handle64_host);
int focusr_dist_shared_open(const char* handles_host, int rank, int world);
int focusr_dist_shared_free(void);
int focusr_dist_unique_id(char* out128_host);
int focusr_dist_init(const char* id128_host, int rank, int world);
int focusr_dist_finalize(void);
size_t focusr_eigs_dist_workspace_bytes(int n_local, int n_ghost, int n_send, int max_row_entries,
                                        int block_size, int world);
int focusr_eigs_smallest_dist(const int* row_ptr, const int* cols_local, const double* weights,
                              const double* degree, const double* degree_inv, const double* points,
                              int n_local, int n_ghost, long long row_begin_global, long long nnz_local,
                              const int* send_idx, int n_send, const int* send_counts_host,
                              const int* recv_counts_host, const int* ghost_peer, const int* ghost_row,
                              int ghost_base, const int* push_row, const int* push_dst, int n_push,
                              int use_p2p, int rows_cap, int n_zero_rows_global, int max_row_entries,
                              int k, int n_k_needed, int k_buffer, double min_eig_val, double tol,
                              int max_outer, int block_size, double spectrum_upper_bound,
                              double* eig_vals, double* eig_vecs, int ldv, int* result_i_host,
                              double* result_d_host, void* workspace, size_t workspace_bytes,
                              const focusr_eigs_options* options, focusr_stream_t stream);

/* Live profile of the dominant kernel, the Chebyshev SpMM filter step (CUDA events on the launching
 * stream around every filter application since the last reset): out4_host = {milliseconds,
 * launches, algorithmic bytes (12 nnz + 20 N + 24 b N per launch), 0}.  bench.py's roofline line.
 * focusr_profile_get counts the fp64 steps (k_spmm); focusr_profile_get_kind(kind, ...) the steps of one kind:
 * 0 = fp64, 1 = fp32 (k_filter_sell mode 0: 8 nnz + 12 N + 12 b N per launch), 2 = fp32 correction form (mode 3:
 * 8 nnz + 12 N + 16 b N per launch); reset clears all three.  kind 3 = the persistent filter kernels of the last
 * row-partitioned solve of this process: {nanoseconds CTA 0 spent at the in-kernel barriers, nanoseconds it spent
 * working, steps, 0}.  kind 4 = the pruned KNN: {(query, reference) distance evaluations since the last reset, 0, 0,
 * 0} (synchronises the device). */
void focusr_profile_reset(void);
void focusr_profile_get(double* out4_host);
void focusr_profile_get_kind(int kind, double* out4_host);

/* y = L x for a dense block of n_cols vectors (n_cols a multiple of 8, <= 96), used by tests and
 * residual checks: y[i][:] = dinv_i (d_i x_i - sum_j w_ij x_j). */
int focusr_laplacian_apply(const int* row_ptr, const int* cols, const double* weights,
                           const double* degree, const double* degree_inv,
                           const int* mesh_point_off, int n_meshes, int max_mesh_points,
                           const double* x, double* y, int n_cols, focusr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * B2  eigenvector normalisation (graph.py:254-257): per mesh, per column j < n_cols[m]:
 * v <- (v - min v) / ptp(v) - 0.5.   In place on vecs [n_points][ld].
 * ------------------------------------------------------------------------------------------- */
int focusr_normalize_columns(double* vecs, int n_points, int ld, const int* mesh_point_off,
                             int n_meshes, const int* n_cols, focusr_stream_t stream);

/* C5  eigsort's flip + reorder (eigsort.py:108-122), applied to every mesh m of the given offset
 * table:  new[:, dst[m][t]] = sign[m][t] * old[:, src[m][t]] for t < n_moves (sign = +1/-1), other
 * columns unchanged.  A mesh that must stay as it is gets the identity (dst = src, sign = +1). */
int focusr_flip_permute_columns(double* vecs, int n_points, int ld, const int* mesh_point_off,
                                int n_meshes, int max_mesh_points, const int* dst, const int* src,
                                const int* sign, int n_moves, focusr_stream_t stream);

/* D1  spectral coordinates (focusr.py:492-508): out[i][u] = vecs[i][u] * weights[m][u], u < ns;
 * out is [n_points][ns]. */
int focusr_spectral_coords(const double* vecs, int n_points, int ld, const int* mesh_point_off,
                           int n_meshes, int max_mesh_points, const double* weights, int ns,
                           double* out, focusr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * C1, C3, C4  eigsort cost matrices (eigsort.py:34-41, 162-233) for n_pairs (target, source)
 * pairs.  Pair p uses mesh t_mesh[p] / s_mesh[p] of the batch, sample rows idx_t[p][0..n_samp_t)
 * and idx_s[p][..] (local row ids = Graph.rand_idxs).  Outputs [n_pairs][n][n] each:
 * c_hist / c_hist_f (1-D Wasserstein distance of log(v + 0.5 + eps), source flipped for _f) and
 * c_spatial / c_spatial_f (RMS difference at xyz nearest neighbours / n_samp_t); nn_idx
 * [n_pairs][n_samp_t] is the nearest sampled source point of each sampled target point.
 * c_lambda, min/compare, the n x n assignment and the flip list: focusr_eigsort_decide (device) or the host classes.
 * ------------------------------------------------------------------------------------------- */
size_t focusr_eigsort_workspace_bytes(int n_pairs, int n_samp_t, int n_samp_s, int n_features);
int focusr_eigsort_costs(const double* vecs, int ld, const double* points,
                         const int* mesh_point_off, const int* t_mesh, const int* s_mesh,
                         int n_pairs, const long long* idx_t, const long long* idx_s, int n_samp_t,
                         int n_samp_s, int n_features, double* c_hist, double* c_hist_f,
                         double* c_spatial, double* c_spatial_f, long long* nn_idx, void* workspace,
                         size_t workspace_bytes, focusr_stream_t stream);

/* C2, C5, D1  the n x n decisions of eigsort for every pair, on the device (eigsort.py:66-122, 142-160; focusr.py:
 * 459-490): c_lambda from the eigenvalues (`eig_vals` [n_meshes][ldv], `n_found` [n_meshes] = how many each mesh
 * returned: the gap averages over all of them), Q = min(c, c_f) with c = c_spatial * c_lambda * c_hist, the assignment
 * (scipy.optimize.linear_sum_assignment's algorithm with its scan order and tie rules; of Q, or Q^T when the source is
 * the reference), the flip list and the spectral weights.  Outputs: q_out [n_pairs][n] (cost of each matched pair, in
 * the order of the reference's match list); dst / src / sign [n_meshes][n] = the column moves of
 * focusr_flip_permute_columns for BOTH meshes of every pair (identity for the reference graph); weights
 * [n_meshes][ns] for focusr_spectral_coords (ones when !weighted); *status (device int) = 1 if an assignment was
 * infeasible (non-finite costs).  One thread per pair; n <= 96.  Meshes not named by t_mesh / s_mesh are not written. */
size_t focusr_eigsort_decide_workspace_bytes(int n_pairs, int n_features);
int focusr_eigsort_decide(const double* eig_vals, int ldv, const int* n_found, const int* t_mesh,
                          const int* s_mesh, int n_pairs, const double* c_hist, const double* c_hist_f,
                          const double* c_spatial, const double* c_spatial_f, int n_features, int ns,
                          int target_as_reference, int weighted, double* q_out, int* dst, int* src,
                          int* sign, double* weights, int* status, void* workspace,
                          size_t workspace_bytes, focusr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * K4  exact k-nearest neighbours (scipy KDTree(refs).query(queries, k), p=2: focusr.py:351-353,
 * 409-413; eigsort.py:203-204).  fp64 brute force on direct differences sum_c (q_c - r_c)^2 in
 * column order without FMA; ties go to the lower index.  Segmented: segment s searches
 * refs[ref_off[s]..ref_off[s+1]) for queries[query_off[s]..query_off[s+1]); returned indices are
 * local to the segment.  idx [n_queries][k], dist [n_queries][k] (Euclidean, nullable).
 * With a workspace (focusr_knn_workspace_bytes) and segments of 512..16384 points the search visits
 * Morton-ordered reference tiles and skips those whose bounding box lies beyond the current k-th
 * best: same arithmetic, same tie rule, bit-identical output, far fewer distance evaluations.
 * workspace = NULL selects plain brute force.
 * ------------------------------------------------------------------------------------------- */
size_t focusr_knn_workspace_bytes(int n_refs_total, int n_queries_total, int n_segments, int dim);
int focusr_knn(const double* refs, int ld_refs, const int* ref_off, int n_refs_total,
               int max_refs_per_segment, const double* queries, int ld_queries, const int* query_off,
               int n_queries_total, int max_queries_per_segment, int n_segments, int dim, int k,
               long long* idx, double* dist, void* workspace, size_t workspace_bytes,
               focusr_stream_t stream);

/* The distance matrix of the 'hungarian' correspondence (focusr.py:340-349: scipy cdist(spectral_pts,
 * target_pts), euclidean): out [n_a][n_b] = |a_i - b_j|_2. */
int focusr_cdist(const double* a, int n_a, const double* b, int n_b, int dim, double* out,
                 focusr_stream_t stream);

/* The assignment of the 'hungarian' correspondence (focusr.py:347: scipy.optimize.linear_sum_assignment): scipy's own
 * algorithm (shortest augmenting paths, rectangular_lsap.cpp) with its scan order and tie rules, so the assignment is
 * the one scipy returns also where the optimum is not unique; one 8-CTA thread-block cluster, column state in
 * distributed shared memory (csrc/lsap.cu).  cost: device, row-major [n_rows][n_cols], finite, n_rows <= n_cols (pass
 * the transpose otherwise), n_cols <= 51200.  col4row: device int32 [n_rows] = scipy's col_ind.  *status_host: 0, or
 * -1 when no assignment exists (non-finite costs).  Synchronises `stream`. */
size_t focusr_lsap_workspace_bytes(int n_rows);
int focusr_lsap(const double* cost, int n_rows, int n_cols, int* col4row, int* status_host, void* workspace,
                size_t workspace_bytes, focusr_stream_t stream);

/* E3  get_weighted_final_node_locations (focusr.py:401-426) from the k=3 neighbours:
 * coincident neighbour -> its target point, else inverse-distance weighted mean of the three
 * target points.  idx3 is local to the segment of `target_points` starting at point_base[i]
 * (nullable = 0). */
int focusr_weighted_positions(const long long* idx3, const double* dist3,
                              const double* target_points, const int* point_base, int n_queries,
                              double* out, focusr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * K8  Coherent Point Drift (focusr.py:297-334: cycpd.affine_registration, then
 * cycpd.deformable_registration(num_eig, alpha, beta) on subsets X (source) / Y (target) of the
 * spectral coordinates, then reg.transform_point_cloud on ALL target coordinates).  cycpd is an
 * unpinned, absent dependency: the algorithm is Myronenko & Song, TPAMI 2010, with the conventions
 * written down in oracle/cpd_port.py (the only thing these entry points are checked against).
 * x [n_x][dim], y [n_y][dim] row-major fp64 on the device, 1 <= dim <= 16.  The EM loop runs on the
 * device; the call SYNCHRONISES the stream once per 8 iterations to read the convergence state.
 *   affine:      b_out [dim][dim], t_out [dim] (TY = Y b + t), ty_out [n_y][dim] (all nullable);
 *                result_host[4] = {iterations, sigma2, objective q, |q - q_prev|}; the loop ends when
 *                |q - q_prev| <= tolerance or at max_iterations.
 *   deformable:  low-rank kernel with the num_eig (<= 152) leading eigenpairs of
 *                G = exp(-|y_i - y_j|^2 / (2 beta^2)); w_out [n_y][dim]; result_host[6] = {iterations,
 *                sigma2, |sigma2 - sigma2_prev|, eigen-iterations, eigen-residual / |lambda_1|,
 *                smallest kept |eigenvalue|}; ends when |sigma2 - sigma2_prev| <= tolerance.
 *   *_apply:     transform_point_cloud on any point set: pts b + t, or pts + G(pts, y) w.
 * `w` is the outlier weight of the E-step (0 in the reference's calls).
 * ------------------------------------------------------------------------------------------- */
size_t focusr_cpd_workspace_bytes(int n_x, int n_y, int dim, int num_eig /* 0 = affine only */);
int focusr_cpd_affine(const double* x, int n_x, const double* y, int n_y, int dim, int max_iterations,
                      double tolerance, double w, double* b_out, double* t_out, double* ty_out,
                      double* result_host, void* workspace, size_t workspace_bytes,
                      focusr_stream_t stream);
int focusr_cpd_deformable(const double* x, int n_x, const double* y, int n_y, int dim,
                          int max_iterations, double tolerance, double w, double alpha, double beta,
                          int num_eig, double* w_out, double* ty_out, double* result_host,
                          void* workspace, size_t workspace_bytes, focusr_stream_t stream);
/* g_out [n_y][n_y] = exp(-|y_i - y_j|^2 / (2 beta^2)): the `G` of cycpd's (G, W) parameter tuple. */
int focusr_cpd_kernel_matrix(const double* y, int n_y, int dim, double beta, double* g_out,
                             focusr_stream_t stream);
int focusr_cpd_affine_apply(const double* pts, int n, int dim, const double* b, const double* t,
                            double* out, focusr_stream_t stream);
int focusr_cpd_deformable_apply(const double* pts, int n, const double* y, int n_y, int dim,
                                const double* w, double beta, double* out, focusr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * K9  vtkCurvatures (vtk_functions.py:40-74; the node features of the reference's default
 * list_features_to_calc=["curvature"], graph.py:11-15,86-87): discrete Gauss, mean, minimum and
 * maximum curvature per vertex of a triangle mesh (or of a batch of meshes with global vertex ids).
 * VTK is an unpinned, absent dependency: the algorithm is vtkCurvatures.cxx as restated in
 * oracle/curvature_port.py.  Outputs [n_points] each, nullable.  SYNCHRONISES the stream (index check).
 * ------------------------------------------------------------------------------------------- */
size_t focusr_curvature_workspace_bytes(int n_points, int n_tris);
int focusr_curvatures(const double* points, const int* tris, int n_points, int n_tris, double* gauss,
                      double* mean, double* k_min, double* k_max, void* workspace,
                      size_t workspace_bytes, focusr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * K10  ICP pre-alignment (focusr.py:106-131 -> vtk_functions.py:12-37: vtkIterativeClosestPointTransform
 * with a rigid-body (similarity = 0) or similarity landmark transform, closest points ON the target
 * surface, StartByMatchingCentroids, exactly max_iterations landmark fits; landmarks = every
 * (n_source / max_landmarks)-th source point).  VTK is an unpinned, absent dependency: the algorithm is
 * VTK 9's as restated in oracle/icp_port.py.  matrix_out: device [16], row-major 4x4 acting on column
 * vectors (vtkMatrix4x4 layout); transformed_out: device [n_source_points][3] = matrix * source (the
 * `apply_transform` of vtk_functions.py:32-37); both nullable.  Target triangle ids must be in range
 * (checked by focusr_laplacian_build on the same mesh).  Does not synchronise.
 * ------------------------------------------------------------------------------------------- */
size_t focusr_icp_workspace_bytes(int n_source_points, int n_target_tris);
int focusr_icp(const double* target_points, int n_target_points, const int* target_tris,
               int n_target_tris, const double* source_points, int n_source_points, int max_landmarks,
               int max_iterations, int similarity, int start_by_matching_centroids,
               double* matrix_out, double* transformed_out, void* workspace, size_t workspace_bytes,
               focusr_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* FOCUSR_B200_H */
