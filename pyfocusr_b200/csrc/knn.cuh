// internal interface of knn.cu / knn_pruned.cu
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace fb {
// brute force over every reference of the segment.  n_segments counts query segments; query segment s searches
// reference segment ref_seg[s] (device; NULL = s).
int launch_knn(const double* refs, int ld_refs, const int* ref_off, const double* queries, int ld_queries,
               const int* query_off, int n_segments, int max_queries, int dim, int k, long long* idx,
               double* dist, cudaStream_t stream, const int* ref_seg = nullptr);

// Morton-ordered tiles with bounding-box pruning; bit-identical results.  With ref_seg, the workspace is sized for
// n_segments = the number of reference segments, and max_refs bounds every reference segment.
size_t knn_pruned_workspace_bytes(long long n_refs, long long n_queries, int n_segments, int dim);
bool knn_pruned_applicable(int max_refs, int max_queries, int dim, int k);
int launch_knn_pruned(const double* refs, int ld_refs, const int* ref_off, const double* queries, int ld_queries,
                      const int* query_off, int n_segments, int max_refs, int max_queries, long long n_refs,
                      long long n_queries, int dim, int k, long long* idx, double* dist, void* workspace,
                      size_t workspace_bytes, cudaStream_t stream, int n_ref_segments = 0,
                      const int* ref_seg = nullptr);
}  // namespace fb
