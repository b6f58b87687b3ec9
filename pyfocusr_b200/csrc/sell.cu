// The fp32 Chebyshev filter steps of the eigensolver on a sliced-ELL (SELL-64) copy of the matrix, and the smoothing
// passes of Graph.mean_filter_graph.  Both are chains of hundreds of dependent, HBM-bound launches.
//
// (1) Filter steps (chfsi_driver.hpp: plain fp32 blocks and the fp32 correction form).  Round 1 ran them on CSR: per row
//     a dependent chain row_ptr -> (col, weight) -> gather, two 4-byte loads per entry whose addresses are 6 entries
//     apart between neighbouring rows, and ncu showed the L1TEX wavefront pipe 61% busy next to DRAM at 69%.  Here the
//     fp32 copy of the matrix is stored slice by slice: 64 rows x W entries, entry k of the 64 rows contiguous, {column,
//     weight} packed in 8 bytes.  One coalesced load per k serves 8 rows of a warp, there is no row pointer, the trip
//     count W is uniform over the CTA pass, and the single-use streams (entries, z_prev, r, the stores) bypass L1 and
//     are marked evict_first in L2 so that the gathered block, which is re-used ~7 times, survives there.
//     Measured on B200, 128 pairs per launch (tools/kernel_ab.py, gpurun_out/r2_ab1.log): correction step 0.2494 ms (CSR)
//     -> 0.2793 (SELL, default cache policy) -> 0.2277 ms (SELL + stream policy) = 5.40 TB/s = 82.7% of the measured HBM
//     peak by algorithmic bytes; plain fp32 step 0.2024 -> 0.2003 ms (75%).  evict_last on the gathered block instead:
//     0.2430 / 0.2374 ms (worse for the plain step); both (the default): 0.2298 / 0.1985.  6 or 5 resident CTAs per SM
//     (40 / 46 registers): 0.2537 / 0.2593 ms; without the L2 prefetch of the CTA's streams: 0.2696 ms.  The absolute
//     numbers move by +-8% from one B200 of the pool to the next (r2_ab1..3.log); the order of the variants does not,
//     except that stream policy alone vs both is a toss-up for the correction step and both is never worse for the
//     plain step (0.1855 vs 0.2210, 0.1864 vs 0.1886, 0.1985 vs 0.2003 ms on three boxes).  The CSR kernels are gone.
// (2) Programmatic dependent launch: every step of a chain is launched with programmaticStreamSerialization; a CTA
//     first asks L2 for the data of its rows that the previous step does not write (matrix slice, r, z_prev), then
//     executes griddepcontrol.wait, then griddepcontrol.launch_dependents.  The next step's CTAs therefore become
//     resident as the last wave of this step drains and their prefetches overlap its tail; no launch gap is left.
// (3) Graph.mean_filter_graph (graph.py:349-354): one thread per row walks the CSR row of A backwards and splices the
//     diagonal in at its sorted position -- scipy's accumulation order, bit for bit.  A sliced-ELL form of the smoothing
//     matrix (entries pre-multiplied, padded [n][4] iterates fetched with one 256-bit load) was measured at 18.6 / 17.95 ms
//     against 17.8 ms for 300 passes over 128 meshes and removed: the pass is bound by its 6.4-wave launches, not by
//     the row walk (programmatic dependent launch: 17.8 -> 17.0 ms).  Marking the matrix stream evict_first in L2, which
//     pays in the filter steps, costs here (18.3 -> 20.0 ms): the 140 MB matrix of 128 targets is partly L2-resident
//     from one pass to the next.  ncu at bench size (profiles/r2_summary.md): DRAM 49% busy, L1 61%, 65% of the warp
//     slots filled (40 registers), no pipe saturated, 0.95x of the algorithmic bytes moved.  A form that loads all
//     columns, weights and iterate rows of a row before its arithmetic (rows <= 8 entries; 80 registers, 3 CTAs per SM)
//     was measured at 21.1 ms against 17.15 ms for the serial walk (gpurun_out/r2d_kernel_ab.log) and removed: fewer
//     resident threads cost more than the longer load batches of each thread bring.
#include <climits>
#include <vector>

#include "common.cuh"
#include "rowops.h"
#include "sell.cuh"

namespace fb {

constexpr int FS_THREADS = 256;

// programmatic dependent launch (see header comment)
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <class... KArgs, class... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
constexpr int FS_ROWS = 256;  // rows per CTA = 4 slices

// ---------------------------------------------------------------------------------------------------------------
// cache-policy helpers (sm_100a PTX): 128-bit loads take the eviction priority through a createpolicy descriptor
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long policy_evict_last() {
  unsigned long long p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ unsigned long long policy_evict_first() {
  unsigned long long p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// (the loads below are of data that no thread writes during the launch: plain `asm`, not `asm volatile`, so that the
// compiler is free to batch several of them before the first use)
// gathered (re-used) data
template <int HINT>
__device__ __forceinline__ float4 ld_keep(const float4* p, unsigned long long pol) {
  if (HINT) {
    float4 v;
    asm("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p), "l"(pol));
    return v;
  }
  return __ldg(p);
}
template <int HINT>
__device__ __forceinline__ double2 ld_keep(const double2* p, unsigned long long pol) {
  if (HINT) {
    double2 v;
    asm("ld.global.nc.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol));
    return v;
  }
  return __ldg(p);
}
// single-use streams
template <int HINT>
__device__ __forceinline__ float4 ld_stream(const float4* p, unsigned long long pol) {
  if (HINT) {
    float4 v;
    asm("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p), "l"(pol));
    return v;
  }
  return __ldg(p);
}
template <int HINT>
__device__ __forceinline__ int2 ld_stream(const int2* p, unsigned long long pol) {
  if (HINT) {
    int2 v;
    asm("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.s32 {%0,%1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(p), "l"(pol));
    return v;
  }
  return __ldg(p);
}
template <int HINT>
__device__ __forceinline__ void st_stream(float4* p, float4 v, unsigned long long pol) {
  if (HINT)
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w), "l"(pol)
                 : "memory");
  else
    *p = v;
}
__device__ __forceinline__ void prefetch_l2_line(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---------------------------------------------------------------------------------------------------------------
// SELL build (fp32 filter copy)
// ---------------------------------------------------------------------------------------------------------------
long long sell_entries_cap(const int* off, const int* info, int n_meshes, int extra_per_row) {
  long long cap = 0;
  for (int m = 0; m < n_meshes; ++m) {
    const long long rows = off[m + 1] - off[m];
    const long long slices = (rows + SELL_ROWS - 1) / SELL_ROWS;
    cap += slices * SELL_ROWS * (long long)(info[FOCUSR_MESH_INFO_INTS * m + 4] + extra_per_row);
  }
  return cap;
}

int sell_slice_count(const int* off, int n_meshes) {
  long long s = 0;
  for (int m = 0; m < n_meshes; ++m) s += (off[m + 1] - off[m] + SELL_ROWS - 1) / SELL_ROWS;
  return (int)s;
}

__device__ __forceinline__ int find_slice_mesh(const int* __restrict__ mso, int n_meshes, int s) {
  int lo = 0, hi = n_meshes - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (mso[mid] <= s)
      lo = mid;
    else
      hi = mid - 1;
  }
  return lo;
}

// one warp per slice: 64 * (longest row of the slice)
__global__ void __launch_bounds__(256)
k_sell_widths(const int* __restrict__ row_ptr, const int* __restrict__ mesh_off, const int* __restrict__ mso, int n_meshes,
              int n_slices, int* __restrict__ slice_cnt) {
  const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (s >= n_slices) return;
  const int m = find_slice_mesh(mso, n_meshes, s);
  const int r0 = mesh_off[m] + (s - mso[m]) * SELL_ROWS, r1 = min(mesh_off[m + 1], r0 + SELL_ROWS);
  int w = 0;
  for (int r = r0 + lane; r < r1; r += 32) w = max(w, row_ptr[r + 1] - row_ptr[r]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) w = max(w, __shfl_xor_sync(0xffffffffu, w, o));
  if (lane == 0) slice_cnt[s] = w * SELL_ROWS;
}

// one thread per (slice, row slot)
__global__ void __launch_bounds__(256)
k_sell_fill_f32(const int* __restrict__ row_ptr, const int* __restrict__ cols, const double* __restrict__ weights,
                const int* __restrict__ mesh_off, const int* __restrict__ mso, int n_meshes, int n_slices,
                const int* __restrict__ slice_ptr, int2* __restrict__ entries) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int s = (int)(t / SELL_ROWS), rl = (int)(t % SELL_ROWS);
  if (s >= n_slices) return;
  const int m = find_slice_mesh(mso, n_meshes, s);
  const int r0 = mesh_off[m] + (s - mso[m]) * SELL_ROWS, r1 = mesh_off[m + 1];
  const int e0 = slice_ptr[s], w = (slice_ptr[s + 1] - e0) / SELL_ROWS;
  const int row = r0 + rl;
  int p0 = 0, len = 0;
  if (row < r1) {
    p0 = row_ptr[row];
    len = row_ptr[row + 1] - p0;
  }
  for (int k = 0; k < w; ++k) {
    int2 e = make_int2(r0, 0);  // padding: a valid row of the same slice, weight +0.0f
    if (k < len) e = make_int2(cols[p0 + k], __float_as_int((float)weights[p0 + k]));
    entries[(size_t)e0 + (size_t)k * SELL_ROWS + rl] = e;
  }
}

__global__ void k_ddi_f32(const double* __restrict__ degree, const double* __restrict__ degree_inv, int n_rows,
                          float2* __restrict__ ddi) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n_rows) ddi[t] = make_float2((float)degree[t], (float)degree_inv[t]);
}

int sell_build_f32(const int* row_ptr, const int* cols, const double* weights, const double* degree,
                   const double* degree_inv, const int* mesh_off, const int* off_host, int n_meshes, int n_rows,
                   int* mesh_slice_off, int* slice_ptr, int2* entries, float2* ddi, int* slice_cnt, int* scan_tmp,
                   cudaStream_t stream) {
  // first slice of every mesh: tiny, built on the host and staged by the runtime (pageable source)
  static thread_local std::vector<int> mso_host;
  mso_host.assign((size_t)n_meshes + 1, 0);
  for (int m = 0; m < n_meshes; ++m) mso_host[m + 1] = mso_host[m] + (off_host[m + 1] - off_host[m] + SELL_ROWS - 1) / SELL_ROWS;
  const int n_slices = mso_host[n_meshes];
  FB_CUDA(cudaMemcpyAsync(mesh_slice_off, mso_host.data(), sizeof(int) * ((size_t)n_meshes + 1), cudaMemcpyHostToDevice, stream));
  k_sell_widths<<<div_up((long long)n_slices * 32, 256), 256, 0, stream>>>(row_ptr, mesh_off, mesh_slice_off, n_meshes, n_slices,
                                                                           slice_cnt);
  FB_COUNT_LAUNCH(1);
  int rc = exclusive_scan_i32(slice_cnt, slice_ptr, n_slices, scan_tmp, stream);
  if (rc) return rc;
  k_sell_fill_f32<<<div_up((long long)n_slices * SELL_ROWS, 256), 256, 0, stream>>>(row_ptr, cols, weights, mesh_off, mesh_slice_off,
                                                                                    n_meshes, n_slices, slice_ptr, entries);
  k_ddi_f32<<<div_up(n_rows, 256), 256, 0, stream>>>(degree, degree_inv, n_rows, ddi);
  FB_COUNT_LAUNCH(2);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// filter step on the SELL copy.  TPR threads share a row, each owns B / (4 TPR) float4 slices of it.
// MODE 0: out = al (L y - c y) - ga x_prev                    (fp32 blocks; al, ga per mesh: double tables)
// MODE 1: the same with y read from the fp64 block, ga = 0; also writes the fp32 copy of y (next step's x_prev)
// MODE 2: the same, result written to the fp64 block
// MODE 3: z_next = al_j ((L - c) z + r_j) - ga_j z_prev       (correction form; al, ga per column: float tables)
// MODE 4: x += that (fp64 block), nothing else stored
// ---------------------------------------------------------------------------------------------------------------
// ROWS: rows per CTA -- 256 (4 slices, 256 / TPR rows per pass), or one pass (256 / TPR rows) for batches that would not
// fill the GPU otherwise (a single mesh: the drop-in Focusr call).  A compile-time constant: as a kernel argument it cost
// the correction step 11% (0.221 -> 0.245 ms per launch at 32 registers).
template <int B, int TPR, int MODE, int POL, int MINB, int ROWS>
__global__ void __launch_bounds__(FS_THREADS, MINB)
k_filter_sell(const int2* __restrict__ entries, const int* __restrict__ slice_ptr, const int* __restrict__ mso,
              const float2* __restrict__ ddi, const int* __restrict__ mesh_off, const void* __restrict__ y_,
              const float* __restrict__ x_prev, const float* __restrict__ r, void* __restrict__ out_, float* __restrict__ y_copy,
              const void* __restrict__ alpha_, const void* __restrict__ gamma_, const double* __restrict__ center, int step,
              int n_steps, int has_prev, int prefetch, int early) {
  constexpr int VPT = B / (4 * TPR);
  static_assert(VPT * 4 * TPR == B, "block size must be a multiple of 4*TPR");
  constexpr bool CORR = MODE >= 3;
  constexpr int KEEP = POL & 1, STRM = (POL >> 1) & 1;
  const int mesh = blockIdx.y;
  const int r0 = mesh_off[mesh] + blockIdx.x * ROWS;
  const int r1 = min(mesh_off[mesh + 1], r0 + ROWS);
  if (r0 >= r1) return;
  const int slice0 = mso[mesh] + blockIdx.x * (ROWS / SELL_ROWS);
  const unsigned long long pol_keep = KEEP ? policy_evict_last() : 0ull;
  const unsigned long long pol_strm = STRM ? policy_evict_first() : 0ull;
  const float* yf = static_cast<const float*>(y_);
  // Before the dependency on the previous step resolves: ask L2 for what that step does not write -- this CTA's
  // matrix slice, its r rows and its z_prev rows (written two steps back: complete, because the previous step released
  // this launch only after ITS wait returned).  After it: the rows of y this CTA owns.
  const int pr = r0 + (int)threadIdx.x;
  constexpr int LINES = (B * 4 + 127) / 128;  // 128-byte lines per fp32 row
  if (!early) {
    pdl_wait();
    pdl_launch_dependents();
  }
  if (prefetch && MODE != 1) {
    if (pr < r1) {
#pragma unroll
      for (int l = 0; l < LINES; ++l) {
        if (has_prev) prefetch_l2_line(x_prev + (size_t)pr * B + 32 * l);
        if (CORR) prefetch_l2_line(r + (size_t)pr * B + 32 * l);
      }
    }
    const int ns = min(ROWS / SELL_ROWS, (r1 - r0 + SELL_ROWS - 1) / SELL_ROWS);
    const int q0 = slice_ptr[slice0], q1 = slice_ptr[slice0 + ns];
    for (int q = q0 + 16 * (int)threadIdx.x; q < q1; q += 16 * FS_THREADS) prefetch_l2_line(entries + q);
  }
  if (early) {
    pdl_wait();
    pdl_launch_dependents();
  }
  if (prefetch && MODE != 1 && pr < r1) {
#pragma unroll
    for (int l = 0; l < LINES; ++l) prefetch_l2_line(yf + (size_t)pr * B + 32 * l);
  }
  const float cc = (float)center[mesh];
  const int g = threadIdx.x / TPR, t = threadIdx.x % TPR;
  float al_s = 0.f, ga_s = 0.f;
  const float4* al_p = nullptr;
  const float4* ga_p = nullptr;
  if (CORR) {
    al_p = reinterpret_cast<const float4*>(static_cast<const float*>(alpha_) + ((size_t)mesh * n_steps + step) * B);
    ga_p = reinterpret_cast<const float4*>(static_cast<const float*>(gamma_) + ((size_t)mesh * n_steps + step) * B);
  } else {
    al_s = (float)static_cast<const double*>(alpha_)[(size_t)mesh * n_steps + step];
    ga_s = (float)static_cast<const double*>(gamma_)[(size_t)mesh * n_steps + step];
  }
  auto load_y = [&](int rr, int slice) -> float4 {
    if (MODE == 1) {
      const double2* src = reinterpret_cast<const double2*>(static_cast<const double*>(y_) + (size_t)rr * B) + 2 * slice;
      const double2 a = ld_keep<KEEP>(src, pol_keep), b = ld_keep<KEEP>(src + 1, pol_keep);
      return make_float4((float)a.x, (float)a.y, (float)b.x, (float)b.y);
    } else {
      return ld_keep<KEEP>(reinterpret_cast<const float4*>(yf + (size_t)rr * B) + slice, pol_keep);
    }
  };
  // a CTA pass covers RP = 256 / TPR rows = RP / 64 slices; a warp never straddles slices
  constexpr int RP = FS_THREADS / TPR, SPP = RP / SELL_ROWS;
  static_assert(RP % SELL_ROWS == 0, "a CTA pass must cover whole slices");
  const int gs = g / SELL_ROWS, rl = g % SELL_ROWS;
#pragma unroll 1
  for (int pass = 0; pass < ROWS / RP; ++pass) {
    const int rb = r0 + pass * RP + gs * SELL_ROWS;  // first row of this thread's slice
    if (rb >= r1) break;
    const int row = rb + rl;
    const int e0 = slice_ptr[slice0 + pass * SPP + gs];
    const int w = (slice_ptr[slice0 + pass * SPP + gs + 1] - e0) / SELL_ROWS;
    const int2* ep = entries + (size_t)e0 + rl;
    float4 acc[VPT];
#pragma unroll
    for (int v = 0; v < VPT; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    // two entries, then their two gathers, then the arithmetic: two independent gathers in flight per thread
    int k = 0;
#pragma unroll 1
    for (; k + 1 < w; k += 2) {
      const int2 e0v = ld_stream<STRM>(ep + (size_t)k * SELL_ROWS, pol_strm);
      const int2 e1v = ld_stream<STRM>(ep + (size_t)(k + 1) * SELL_ROWS, pol_strm);
      float4 g0[VPT], g1[VPT];
#pragma unroll
      for (int v = 0; v < VPT; ++v) g0[v] = load_y(e0v.x, t + v * TPR);
#pragma unroll
      for (int v = 0; v < VPT; ++v) g1[v] = load_y(e1v.x, t + v * TPR);
      const float w0 = __int_as_float(e0v.y), w1 = __int_as_float(e1v.y);
#pragma unroll
      for (int v = 0; v < VPT; ++v) {
        acc[v].x = fmaf(w0, g0[v].x, acc[v].x);
        acc[v].y = fmaf(w0, g0[v].y, acc[v].y);
        acc[v].z = fmaf(w0, g0[v].z, acc[v].z);
        acc[v].w = fmaf(w0, g0[v].w, acc[v].w);
      }
#pragma unroll
      for (int v = 0; v < VPT; ++v) {
        acc[v].x = fmaf(w1, g1[v].x, acc[v].x);
        acc[v].y = fmaf(w1, g1[v].y, acc[v].y);
        acc[v].z = fmaf(w1, g1[v].z, acc[v].z);
        acc[v].w = fmaf(w1, g1[v].w, acc[v].w);
      }
    }
    if (k < w) {
      const int2 e = ld_stream<STRM>(ep + (size_t)k * SELL_ROWS, pol_strm);
      const float wt = __int_as_float(e.y);
#pragma unroll
      for (int v = 0; v < VPT; ++v) {
        const float4 a = load_y(e.x, t + v * TPR);
        acc[v].x = fmaf(wt, a.x, acc[v].x);
        acc[v].y = fmaf(wt, a.y, acc[v].y);
        acc[v].z = fmaf(wt, a.z, acc[v].z);
        acc[v].w = fmaf(wt, a.w, acc[v].w);
      }
    }
    if (row >= r1) continue;
    const float2 dd = ddi[row];
    const float d = dd.x, di = dd.y;
#pragma unroll
    for (int v = 0; v < VPT; ++v) {
      const int slice = t + v * TPR;
      const float4 yv = load_y(row, slice);
      float4 o;
      if (CORR) {
        const float4 rv = ld_stream<STRM>(reinterpret_cast<const float4*>(r + (size_t)row * B) + slice, pol_strm);
        const float4 al = __ldg(al_p + slice);
        o.x = al.x * ((di * (d * yv.x - acc[v].x) - cc * yv.x) + rv.x);
        o.y = al.y * ((di * (d * yv.y - acc[v].y) - cc * yv.y) + rv.y);
        o.z = al.z * ((di * (d * yv.z - acc[v].z) - cc * yv.z) + rv.z);
        o.w = al.w * ((di * (d * yv.w - acc[v].w) - cc * yv.w) + rv.w);
        if (has_prev) {
          const float4 ga = __ldg(ga_p + slice);
          const float4 pv = ld_stream<STRM>(reinterpret_cast<const float4*>(x_prev + (size_t)row * B) + slice, pol_strm);
          o.x -= ga.x * pv.x;
          o.y -= ga.y * pv.y;
          o.z -= ga.z * pv.z;
          o.w -= ga.w * pv.w;
        }
      } else {
        o.x = al_s * (di * (d * yv.x - acc[v].x) - cc * yv.x);
        o.y = al_s * (di * (d * yv.y - acc[v].y) - cc * yv.y);
        o.z = al_s * (di * (d * yv.z - acc[v].z) - cc * yv.z);
        o.w = al_s * (di * (d * yv.w - acc[v].w) - cc * yv.w);
        if (MODE != 1 && ga_s != 0.f) {
          const float4 pv = ld_stream<STRM>(reinterpret_cast<const float4*>(x_prev + (size_t)row * B) + slice, pol_strm);
          o.x -= ga_s * pv.x;
          o.y -= ga_s * pv.y;
          o.z -= ga_s * pv.z;
          o.w -= ga_s * pv.w;
        }
      }
      if (MODE == 2) {
        double2* op = reinterpret_cast<double2*>(static_cast<double*>(out_) + (size_t)row * B) + 2 * slice;
        op[0] = make_double2((double)o.x, (double)o.y);
        op[1] = make_double2((double)o.z, (double)o.w);
      } else if (MODE == 4) {
        double2* xo = reinterpret_cast<double2*>(static_cast<double*>(out_) + (size_t)row * B) + 2 * slice;
        double2 a = xo[0], b = xo[1];
        a.x += (double)o.x;
        a.y += (double)o.y;
        b.x += (double)o.z;
        b.y += (double)o.w;
        xo[0] = a;
        xo[1] = b;
      } else {
        st_stream<STRM>(reinterpret_cast<float4*>(static_cast<float*>(out_) + (size_t)row * B) + slice, o, pol_strm);
      }
      if (MODE == 1) reinterpret_cast<float4*>(y_copy + (size_t)row * B)[slice] = yv;
    }
  }
}

template <int B, int TPR, int MODE, int MINB>
static void launch_fs_pol(int pol, dim3 grid, cudaStream_t stream, const SellF32& m, const int* mesh_off, const void* y,
                          const float* x_prev, const float* r, void* out, float* y_copy, const void* alpha, const void* gamma,
                          const double* center, int step, int n_steps, int has_prev, int prefetch, int pdl, int rpc) {
#define FB_FS_GO_R(P, R)                                                                                                     \
  if (pdl)                                                                                                                   \
    launch_pdl(k_filter_sell<B, TPR, MODE, P, MINB, R>, grid, dim3(FS_THREADS), stream, m.entries, m.slice_ptr,              \
               m.mesh_slice_off, m.ddi, mesh_off, y, x_prev, r, out, y_copy, alpha, gamma, center, step, n_steps, has_prev,   \
               prefetch, pdl == 2 ? 1 : 0);                                                                                  \
  else                                                                                                                       \
    k_filter_sell<B, TPR, MODE, P, MINB, R><<<grid, FS_THREADS, 0, stream>>>(m.entries, m.slice_ptr, m.mesh_slice_off, m.ddi, \
                                                                             mesh_off, y, x_prev, r, out, y_copy, alpha,      \
                                                                             gamma, center, step, n_steps, has_prev, prefetch, 0)
#define FB_FS_GO(P) FB_FS_GO_R(P, FS_ROWS)
  if (rpc != FS_ROWS) {  // small batch: one pass per CTA, default cache policy of the streams (no A/B forms of this one)
    FB_FS_GO_R(3, FS_THREADS / TPR);
    return;
  }
  switch (pol & 3) {
    case 0: FB_FS_GO(0); break;
    case 1: FB_FS_GO(1); break;
    case 2: FB_FS_GO(2); break;
    default: FB_FS_GO(3); break;
  }
#undef FB_FS_GO
#undef FB_FS_GO_R
}

template <int B, int TPR>
static int launch_fs_b(int mode, const SellF32& m, const int* mesh_off, int n_meshes, int max_mesh_rows, const void* y,
                       const float* x_prev, const float* r, void* out, float* y_copy, const void* alpha, const void* gamma,
                       const double* center, int step, int n_steps, bool has_prev, const FilterTuning& tune,
                       cudaStream_t stream) {
  // a CTA normally covers 256 rows (4 slices) in passes of 256 / TPR; a batch with fewer than two waves of such CTAs (a
  // single mesh: the drop-in Focusr call) gets one pass per CTA so that the whole GPU works on the step
  int rpc = FS_ROWS;
  if ((long long)div_up(max_mesh_rows, FS_ROWS) * n_meshes < 2 * sm_count()) rpc = FS_THREADS / TPR;
  dim3 grid(div_up(max_mesh_rows, rpc), n_meshes);
  constexpr int VPT = B / (4 * TPR);
  constexpr int MB = VPT == 1 ? 8 : (VPT == 2 ? 6 : 3);
  const int hp = has_prev ? 1 : 0, pf = tune.prefetch ? 1 : 0;
#define FB_FS_MODE(MODE_, MINB_) \
  launch_fs_pol<B, TPR, MODE_, MINB_>(tune.policy, grid, stream, m, mesh_off, y, x_prev, r, out, y_copy, alpha, gamma, center, step, n_steps, hp, pf, tune.pdl, rpc)
  // the occupancy A/B (6 or 5 resident CTAs instead of 8) exists for the two steady-state b = 16 kernels only
  if (B == 16 && (mode == 0 || mode == 3) && (tune.min_blocks == 6 || tune.min_blocks == 5)) {
    constexpr int BB = B == 16 ? B : 16, TT = B == 16 ? TPR : 4;
    if (mode == 0 && tune.min_blocks == 6) launch_fs_pol<BB, TT, 0, 6>(tune.policy, grid, stream, m, mesh_off, y, x_prev, r, out, y_copy, alpha, gamma, center, step, n_steps, hp, pf, tune.pdl, rpc);
    else if (mode == 0) launch_fs_pol<BB, TT, 0, 5>(tune.policy, grid, stream, m, mesh_off, y, x_prev, r, out, y_copy, alpha, gamma, center, step, n_steps, hp, pf, tune.pdl, rpc);
    else if (tune.min_blocks == 6) launch_fs_pol<BB, TT, 3, 6>(tune.policy, grid, stream, m, mesh_off, y, x_prev, r, out, y_copy, alpha, gamma, center, step, n_steps, hp, pf, tune.pdl, rpc);
    else launch_fs_pol<BB, TT, 3, 5>(tune.policy, grid, stream, m, mesh_off, y, x_prev, r, out, y_copy, alpha, gamma, center, step, n_steps, hp, pf, tune.pdl, rpc);
  } else {
    switch (mode) {
      case 0: FB_FS_MODE(0, MB); break;
      case 1: FB_FS_MODE(1, MB); break;
      case 2: FB_FS_MODE(2, MB); break;
      case 3: FB_FS_MODE(3, MB); break;
      default: FB_FS_MODE(4, MB); break;
    }
  }
#undef FB_FS_MODE
  FB_COUNT_LAUNCH(1);
  return FB_OK;
}

int launch_filter_sell(int mode, int b, const SellF32& m, const int* mesh_off, int n_meshes, int max_mesh_rows,
                       const void* y, const float* x_prev, const float* r, void* out, float* y_copy, const void* alpha,
                       const void* gamma, const double* center, int step, int n_steps, bool has_prev,
                       const FilterTuning& tune, cudaStream_t stream) {
#define FB_CASE(BB, TT) \
  case BB:              \
    return launch_fs_b<BB, TT>(mode, m, mesh_off, n_meshes, max_mesh_rows, y, x_prev, r, out, y_copy, alpha, gamma, center, step, n_steps, has_prev, tune, stream);
  switch (b) {
    FB_CASE(8, 2)
    FB_CASE(16, 4)
    FB_CASE(24, 2)
    FB_CASE(32, 4)
    FB_CASE(40, 2)
    FB_CASE(48, 4)
    FB_CASE(56, 2)
    FB_CASE(64, 4)
    FB_CASE(72, 2)
    FB_CASE(80, 4)
    FB_CASE(88, 2)
    FB_CASE(96, 4)
    default:
      set_error("filter (SELL): unsupported block size %d (multiples of 8 up to 96)", b);
      return FB_ERR_UNSUPPORTED;
  }
#undef FB_CASE
}

// ===============================================================================================================
// Row-partitioned solve (one mesh over several GPUs, one process per GPU): ALL steps of a filter pass in ONE
// persistent cooperative kernel per GPU.  Round 1 launched one fp64 SpMM plus one flag-barrier kernel per step and was
// bound by that latency (49 us per step against ~21 us of memory time at 8 GPUs).  Here every rank keeps its three
// vector blocks in a region shared through CUDA IPC; the fp32 forms of the step run on fp32 views of those blocks; a
// rows of the neighbours that a rank gathers are PUSHED into its ghost rows over NVLink by their owners as soon as they
// are written (posted stores, see k_filter_persist); and the steps are separated by a barrier INSIDE the kernel
// (step_barrier below).  No launch, no host involvement, no collective per step.
// ===============================================================================================================
constexpr int PEER_ROW_BITS = 24;

// ghost column n_loc + g of the local numbering -> row ghost_base + g of the fp32 views (their ghost rows)
__global__ void k_sell_remap_ghosts(int2* __restrict__ entries, const int* __restrict__ slice_ptr, int n_slices, int n_loc,
                                    int ghost_base) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= slice_ptr[n_slices]) return;  // slots past the scanned total were never written
  const int c = entries[t].x;
  if (c >= n_loc) entries[t].x = ghost_base + (c - n_loc);
}

int sell_remap_ghosts(int2* entries, long long n_entries_cap, const int* slice_ptr, int n_slices, int n_loc, int ghost_base,
                      cudaStream_t stream) {
  // padded slots hold column r0 of their slice (< n_loc) and are left alone
  k_sell_remap_ghosts<<<div_up(n_entries_cap, 256), 256, 0, stream>>>(entries, slice_ptr, n_slices, n_loc, ghost_base);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

__global__ void k_block_to_f32(const double* __restrict__ x, float* __restrict__ out, long long n) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = (float)x[t];
}

int block_to_f32(const double* x, float* out, long long n, cudaStream_t stream) {
  k_block_to_f32<<<div_up(n, 256), 256, 0, stream>>>(x, out, n);
  FB_COUNT_LAUNCH(1);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

// The vector blocks change inside the persistent kernel: ordinary C++ loads (ld.global, coherent at the fences of
// step_barrier; never .nc), which the compiler may batch between two barriers but not move across one.
__device__ __forceinline__ float4 ld_plain(const float4* p) { return *p; }

// Barrier between two steps, across the CTAs of this GPU and across the GPUs.  System-scope operations are expensive
// (a fence.sys by each of ~1000 CTAs per step cost 30-45 us per step in the first version), so exactly ONE thread per
// GPU and step executes them: every CTA releases its rows at GPU scope and arrives on a local counter; the last one to
// arrive publishes the step number to every peer (fence.sys + st.release.sys over NVLink), waits until every peer has
// published it (ld.acquire.sys on LOCAL flag lines), and then opens a local gate at GPU scope on which all other CTAs
// wait.  Causality is transitive across the scopes (rows -> fence.gpu -> counter -> last CTA -> fence.sys -> flag ->
// peer's last CTA -> gate -> peer's CTAs), and the acquiring fence.gpu of every CTA also drops its SM's L1 lines, so
// the plain loads that follow see the rows the other SMs and the other GPUs wrote in the previous step.
// Fences are spelled out: __threadfence() / st.release compile to MEMBAR.SC.* or one MEMBAR.ALL.SYS per store, the
// patterns below ("fence.acq_rel; relaxed store" to release, "relaxed load; fence.acq_rel" to acquire) to one MEMBAR.ALL
// per side.  Measured at 2 GPUs on a problem small enough to expose the barrier (18 000 rows per rank): 14.9 us per step
// with __threadfence / st.release.sys per peer, see profiles/r2_scaling.md for the current figure.
__device__ __forceinline__ void fence_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void fence_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }

__device__ __forceinline__ void step_barrier(const PersistArgs& a, unsigned target, unsigned long long epoch, bool pushed) {
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned old;
    // release: this CTA's stores of the step, ordered before by the bar.sync -- GPU scope, or system scope when the CTA
    // has posted rows into peer memory (the fence then waits for their acknowledgement)
    if (pushed) fence_sys();
    else fence_gpu();
    asm volatile("atom.relaxed.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(a.counter) : "memory");
    unsigned long long* gate = a.my_flags + (size_t)a.rank * 16;  // this rank's own line doubles as the local gate
    const long long t0 = clock64();
    if (old + 1u == target) {  // last CTA of this GPU: every local row of the step is written
      if (a.world > 1) {
        fence_sys();           // acquires the other CTAs' arrivals, releases to the peers
        for (int p = 0; p < a.world; ++p)
          if (p != a.rank) {
            unsigned long long* dst = a.peer_flags[p] + (size_t)a.rank * 16;
            asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(epoch) : "memory");
          }
        for (int p = 0; p < a.world; ++p) {
          if (p == a.rank) continue;
          const unsigned long long* src = a.my_flags + (size_t)p * 16;
          for (;;) {   // acquire loads: no fence (which would wait for the acknowledgement of the flag stores above)
            unsigned long long v;
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(src) : "memory");
            if (v >= epoch) break;
            if (clock64() - t0 > 20000000000LL) {  // ~10 s: a lost peer becomes an error, not a hang
              atomicExch(a.err, 1);
              break;
            }
          }
        }
      }
      fence_gpu();   // (cumulative) releases what was acquired, local rows and the peers' pushed rows, to the local CTAs
      asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(gate), "l"(epoch) : "memory");
    } else {
      for (;;) {
        unsigned long long v;
        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(gate) : "memory");
        if (v >= epoch) break;
        if (clock64() - t0 > 24000000000LL) {
          atomicExch(a.err, 1);
          break;
        }
      }
    }
    fence_gpu();  // acquire side (GPU scope); a fence of scope >= cluster also drops the SM's L1 lines (CCTL.IVALL)
  }
  __syncthreads();
}

// Halo by PUSH: a remote column is never loaded over NVLink inside the step (a peer load costs 1-2 us, three of them in
// a row's dependent chain made the boundary CTAs the critical path of every step: 12.6 us per step at 18 000 rows per
// rank, 25 us at 125 000).  Instead every fp32 view carries ghost rows behind the owned rows, and a CTA that has just
// written rows its peers gather copies them into the peers' ghost slots with posted stores before it arrives at the
// barrier (its arrival fence is then system-scoped, so the stores are acknowledged before the flag can be seen).  After
// the barrier every gather is local.  Tried and dropped: caching the CTA's matrix slice in shared memory and issuing the
// epilogue operands before the gathers (shorter dependent chain, but 80-128 registers: 33.9 against 25.1 us per step).
template <int B, int TPR, bool CORR>
__global__ void __launch_bounds__(FS_THREADS, (B / (4 * TPR) == 1) ? 6 : ((B / (4 * TPR) == 2) ? 4 : 3))
k_filter_persist(const PersistArgs a) {
  constexpr int VPT = B / (4 * TPR);
  constexpr int RP = FS_THREADS / TPR, SPP = RP / SELL_ROWS;
  const int g = threadIdx.x / TPR, t = threadIdx.x % TPR;
  const int gs_ = g / SELL_ROWS, rl = g % SELL_ROWS;
  const float cc = (float)a.center[0];
  const int u0 = blockIdx.x * a.units_per_cta, u1 = min(a.n_units, u0 + a.units_per_cta);
  const int n_slices = (a.n_loc + SELL_ROWS - 1) / SELL_ROWS;
  // this CTA's share of the push list (sorted by row): items [i0, i1)
  int i0 = 0, i1 = 0;
  if (a.n_push > 0) {
    auto lower = [&](int row) {
      int lo = 0, hi = a.n_push;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a.push_row[mid] < row) lo = mid + 1;
        else hi = mid;
      }
      return lo;
    };
    i0 = lower(u0 * RP);
    i1 = lower(u1 * RP);
  }
  const bool pusher = i1 > i0;
  // Units holding rows that peers gather are processed FIRST in every step and pushed right away: the posted stores are
  // acknowledged while the CTA works on its other units, so the system-scope fence of its arrival does not wait for an
  // NVLink round trip (measured at 2 GPUs, 18 000 rows per rank: that wait alone was 2.8 us of a 9.4 us barrier).
  constexpr int ORDER_CAP = 64;
  __shared__ int s_order[ORDER_CAP];
  __shared__ int s_first;
  const int nu = max(u1 - u0, 0);
  const bool reorder = pusher && nu <= ORDER_CAP;
  if (reorder && threadIdx.x == 0) {
    int nf = 0, nl = nu;
    for (int j = 0; j < nu; ++j) {   // stable: boundary units in order, then the others in order
      bool has = false;
      for (int i = i0; i < i1 && !has; ++i) has = a.push_row[i] / RP == u0 + j;
      if (has) s_order[nf++] = u0 + j;
    }
    for (int j = nu - 1; j >= 0; --j) {
      bool has = false;
      for (int i = 0; i < nf && !has; ++i) has = s_order[i] == u0 + j;
      if (!has) s_order[--nl] = u0 + j;
    }
    s_first = nf;
  }
  __syncthreads();
  const int n_first = reorder ? s_first : nu;   // the push follows unit number n_first - 1 of the CTA's order
  // rows [i0, i1) of a view this rank owns -> the ghost slots of the peers that gather them (posted stores)
  auto push_rows = [&](int view, const float* mine) {
    constexpr int Q = B / 4;
    const float* const* dst_of = a.peer_views + (size_t)view * a.world;
    for (int i = threadIdx.x; i < (i1 - i0) * Q; i += FS_THREADS) {
      const int item = i0 + i / Q, q = i % Q;
      const int dst = a.push_dst[item];
      const float4 v = reinterpret_cast<const float4*>(mine + (size_t)a.push_row[item] * B)[q];
      float* base = const_cast<float*>(dst_of[dst >> PEER_ROW_BITS]);
      reinterpret_cast<float4*>(base + ((size_t)a.ghost_base + (size_t)(dst & ((1 << PEER_ROW_BITS) - 1))) * B)[q] = v;
    }
  };
  if (a.push_first && pusher) push_rows(a.v_cur, a.peer_views[(size_t)a.v_cur * a.world + a.rank]);
  // live profile (CTA 0, thread 0): nanoseconds spent waiting at the barriers / working, per launch
  const bool timer = a.timing != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
  unsigned long long t_wait = 0, t_work = 0, t_mark = 0;
  auto now = [] {
    unsigned long long v;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
    return v;
  };
  if (timer) t_mark = now();
  for (int s = 0; s < a.len; ++s) {
    step_barrier(a, (unsigned)(s + 1) * gridDim.x, a.epoch0 + 1ull + (unsigned long long)s, pusher);
    if (timer) {
      const unsigned long long t = now();
      t_wait += t - t_mark;
      t_mark = t;
    }
    const int gstep = a.s0 + s;
    const bool last = gstep == a.deg - 1;
    // views rotate: (prev, cur, next) <- (cur, next, prev)
    const int rot = s % 3;
    const int v_prev = rot == 0 ? a.v_prev : (rot == 1 ? a.v_cur : a.v_next);
    const int v_cur = rot == 0 ? a.v_cur : (rot == 1 ? a.v_next : a.v_prev);
    const int v_next = rot == 0 ? a.v_next : (rot == 1 ? a.v_prev : a.v_cur);
    const float* cur = a.peer_views[(size_t)v_cur * a.world + a.rank];
    const float* prev = a.peer_views[(size_t)v_prev * a.world + a.rank];
    float* next = const_cast<float*>(a.peer_views[(size_t)v_next * a.world + a.rank]);
    float al_s = 0.f, ga_s = 0.f;
    const float4* al_p = nullptr;
    const float4* ga_p = nullptr;
    if (CORR) {
      al_p = reinterpret_cast<const float4*>(static_cast<const float*>(a.alpha) + (size_t)s * B);
      ga_p = reinterpret_cast<const float4*>(static_cast<const float*>(a.gamma) + (size_t)s * B);
    } else {
      al_s = (float)static_cast<const double*>(a.alpha)[s];
      ga_s = (float)static_cast<const double*>(a.gamma)[s];
    }
    const bool has_prev = CORR ? gstep > 0 : ga_s != 0.f;
    // L2 prefetch of a unit's streams (what the batch kernel does at CTA start): entries, r, prev and own cur rows
    auto prefetch_unit = [&](int u, const float* pv, const float* cu, bool want_prev) {
      const int rb0 = u * RP;
      if (rb0 >= a.n_loc) return;
      const int rows = min(RP, a.n_loc - rb0);
      constexpr int LINES = (B * 4 + 127) / 128;
      for (int i = threadIdx.x; i < rows * LINES; i += FS_THREADS) {
        const size_t o = (size_t)(rb0 + i / LINES) * B + 32 * (i % LINES);
        if (cu) prefetch_l2_line(cu + o);
        if (want_prev) prefetch_l2_line(pv + o);
        if (CORR) prefetch_l2_line(a.r + o);
      }
      const int s_lo = u * SPP, s_hi = min(s_lo + SPP, n_slices);
      const int q0 = a.slice_ptr[s_lo], q1 = a.slice_ptr[s_hi];
      for (int q = q0 + 16 * (int)threadIdx.x; q < q1; q += 16 * FS_THREADS) prefetch_l2_line(a.entries + q);
    };
    for (int j = 0; j < nu; ++j) {
      const int u = reorder ? s_order[j] : u0 + j;
      if (j == n_first && pusher && !last && n_first < nu) {   // boundary units done: push them, then the other units
        __syncthreads();
        push_rows(v_next, next);
      }
      if (a.prefetch) {
        if (j + 1 < nu) prefetch_unit(reorder ? s_order[j + 1] : u + 1, prev, cur, has_prev);
        else if (!last) prefetch_unit(reorder ? s_order[0] : u0, cur, nullptr, true);   // first unit of the next step: its prev is this cur
      }
      const int slice = u * SPP + gs_;
      const int rb = slice * SELL_ROWS;
      if (rb >= a.n_loc) continue;
      const int row = rb + rl;
      const int e0 = a.slice_ptr[slice];
      const int w = (a.slice_ptr[slice + 1] - e0) / SELL_ROWS;
      const int2* ep = a.entries + (size_t)e0 + rl;
      float4 acc[VPT];
#pragma unroll
      for (int v = 0; v < VPT; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      int k = 0;
#pragma unroll 1
      for (; k + 1 < w; k += 2) {   // two entries, their two gathers, then the arithmetic
        const int2 e0v = __ldg(ep + (size_t)k * SELL_ROWS);   // the matrix is constant during the kernel
        const int2 e1v = __ldg(ep + (size_t)(k + 1) * SELL_ROWS);
        const float4* s0 = reinterpret_cast<const float4*>(cur + (size_t)e0v.x * B);
        const float4* s1 = reinterpret_cast<const float4*>(cur + (size_t)e1v.x * B);
        float4 g0[VPT], g1[VPT];
#pragma unroll
        for (int v = 0; v < VPT; ++v) g0[v] = ld_plain(s0 + t + v * TPR);
#pragma unroll
        for (int v = 0; v < VPT; ++v) g1[v] = ld_plain(s1 + t + v * TPR);
        const float w0 = __int_as_float(e0v.y), w1 = __int_as_float(e1v.y);
#pragma unroll
        for (int v = 0; v < VPT; ++v) {
          acc[v].x = fmaf(w0, g0[v].x, acc[v].x);
          acc[v].y = fmaf(w0, g0[v].y, acc[v].y);
          acc[v].z = fmaf(w0, g0[v].z, acc[v].z);
          acc[v].w = fmaf(w0, g0[v].w, acc[v].w);
        }
#pragma unroll
        for (int v = 0; v < VPT; ++v) {
          acc[v].x = fmaf(w1, g1[v].x, acc[v].x);
          acc[v].y = fmaf(w1, g1[v].y, acc[v].y);
          acc[v].z = fmaf(w1, g1[v].z, acc[v].z);
          acc[v].w = fmaf(w1, g1[v].w, acc[v].w);
        }
      }
      if (k < w) {
        const int2 e = __ldg(ep + (size_t)k * SELL_ROWS);
        const float wt = __int_as_float(e.y);
        const float4* s0 = reinterpret_cast<const float4*>(cur + (size_t)e.x * B);
#pragma unroll
        for (int v = 0; v < VPT; ++v) {
          const float4 x4 = ld_plain(s0 + t + v * TPR);
          acc[v].x = fmaf(wt, x4.x, acc[v].x);
          acc[v].y = fmaf(wt, x4.y, acc[v].y);
          acc[v].z = fmaf(wt, x4.z, acc[v].z);
          acc[v].w = fmaf(wt, x4.w, acc[v].w);
        }
      }
      if (row >= a.n_loc) continue;
      const float2 dd = a.ddi[row];
      const float d = dd.x, di = dd.y;
#pragma unroll
      for (int v = 0; v < VPT; ++v) {
        const int sl = t + v * TPR;
        const float4 yv = ld_plain(reinterpret_cast<const float4*>(cur + (size_t)row * B) + sl);
        float4 o;
        if (CORR) {
          const float4 rv = __ldg(reinterpret_cast<const float4*>(a.r + (size_t)row * B) + sl);  // constant during the pass
          const float4 al = __ldg(al_p + sl);
          o.x = al.x * ((di * (d * yv.x - acc[v].x) - cc * yv.x) + rv.x);
          o.y = al.y * ((di * (d * yv.y - acc[v].y) - cc * yv.y) + rv.y);
          o.z = al.z * ((di * (d * yv.z - acc[v].z) - cc * yv.z) + rv.z);
          o.w = al.w * ((di * (d * yv.w - acc[v].w) - cc * yv.w) + rv.w);
          if (has_prev) {
            const float4 ga = __ldg(ga_p + sl);
            const float4 pv = ld_plain(reinterpret_cast<const float4*>(prev + (size_t)row * B) + sl);
            o.x -= ga.x * pv.x;
            o.y -= ga.y * pv.y;
            o.z -= ga.z * pv.z;
            o.w -= ga.w * pv.w;
          }
        } else {
          o.x = al_s * (di * (d * yv.x - acc[v].x) - cc * yv.x);
          o.y = al_s * (di * (d * yv.y - acc[v].y) - cc * yv.y);
          o.z = al_s * (di * (d * yv.z - acc[v].z) - cc * yv.z);
          o.w = al_s * (di * (d * yv.w - acc[v].w) - cc * yv.w);
          if (has_prev) {
            const float4 pv = ld_plain(reinterpret_cast<const float4*>(prev + (size_t)row * B) + sl);
            o.x -= ga_s * pv.x;
            o.y -= ga_s * pv.y;
            o.z -= ga_s * pv.z;
            o.w -= ga_s * pv.w;
          }
        }
        if (last) {
          double2* xo = reinterpret_cast<double2*>(a.x + (size_t)row * B) + 2 * sl;
          if (CORR) {
            double2 p0 = xo[0], p1 = xo[1];
            p0.x += (double)o.x;
            p0.y += (double)o.y;
            p1.x += (double)o.z;
            p1.y += (double)o.w;
            xo[0] = p0;
            xo[1] = p1;
          } else {
            xo[0] = make_double2((double)o.x, (double)o.y);
            xo[1] = make_double2((double)o.z, (double)o.w);
          }
        } else {
          reinterpret_cast<float4*>(next + (size_t)row * B)[sl] = o;
        }
      }
    }
    if (pusher && !last && n_first >= nu) {   // every unit of the CTA is a boundary unit: push at the end
      __syncthreads();
      push_rows(v_next, next);
    }
    if (timer) {
      const unsigned long long t = now();
      t_work += t - t_mark;
      t_mark = t;
    }
  }
  if (timer) {
    atomicAdd(a.timing, t_wait);
    atomicAdd(a.timing + 1, t_work);
    atomicAdd(a.timing + 2, (unsigned long long)a.len);
  }
}

template <int B, int TPR>
static int launch_persist_b(bool corr, PersistArgs a, cudaStream_t stream) {
  constexpr int RP = FS_THREADS / TPR;
  a.n_units = div_up(a.n_loc, RP);
  int dev = 0, sms = 0, per_sm = 0;
  FB_CUDA(cudaGetDevice(&dev));
  FB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const void* fn = corr ? (const void*)k_filter_persist<B, TPR, true> : (const void*)k_filter_persist<B, TPR, false>;
  if (corr)
    FB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_filter_persist<B, TPR, true>, FS_THREADS, 0));
  else
    FB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_filter_persist<B, TPR, false>, FS_THREADS, 0));
  const int g_max = std::max(1, sms * per_sm);
  // balanced: every CTA gets the same number of row units (the grid shrinks rather than leaving a ragged last pass)
  a.units_per_cta = div_up(a.n_units, g_max);
  const int grid = div_up(a.n_units, a.units_per_cta);
  void* args[] = {&a};
  FB_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(FS_THREADS), args, 0, stream));
  FB_COUNT_LAUNCH(1);
  return FB_OK;
}

int launch_filter_persist(bool corr, int b, const PersistArgs& a, cudaStream_t stream) {
#define FB_CASE(BB, TT) \
  case BB:              \
    return launch_persist_b<BB, TT>(corr, a, stream);
  switch (b) {
    FB_CASE(8, 2)
    FB_CASE(16, 4)
    FB_CASE(24, 2)
    FB_CASE(32, 4)
    FB_CASE(40, 2)
    FB_CASE(48, 4)
    FB_CASE(56, 2)
    FB_CASE(64, 4)
    FB_CASE(72, 2)
    FB_CASE(80, 4)
    FB_CASE(88, 2)
    FB_CASE(96, 4)
    default:
      set_error("filter (persistent): unsupported block size %d (multiples of 8 up to 96)", b);
      return FB_ERR_UNSUPPORTED;
  }
#undef FB_CASE
}

// ===============================================================================================================
// smoothing passes (Graph.mean_filter_graph)
// ===============================================================================================================
// scipy stores each row of average_mat = diag(1/(1+d)) @ (A + I) in DESCENDING column order and `average_mat @ x`
// accumulates y += a * x in stored order (multiply, then add); one thread per row (any column count up to 8) walks the
// row of A backwards and splices the diagonal in at its sorted position, which reproduces that bit for bit.  Passes are
// chained by programmatic dependent launch: the CTA prefetches its slice of the matrix, which no pass writes, into L2
// before it waits for the previous pass.
// Occupancy of the smoothing pass (A/B: tools/smooth_ab.sh, gpurun_out/r2s_smooth_ab.log; 300 passes over 128 meshes):
// compiled for 4 / 6 / 8 resident CTAs of 256 threads per SM (64 / 40 / 32 registers): 20.50 / 17.47 / 16.67 ms; at full
// occupancy (32 registers) with 512 / 256 / 128 / 96 / 64 threads per CTA: 17.49 / 16.66 / 16.01 / 16.00 / 16.07 ms (the
// round started at 17.15 ms: 40 registers, 256 threads).  The pass is latency-bound (header comment), so every resident
// warp counts, and small CTAs leave fewer warp slots idle while a CTA drains.
#ifndef FB_SMOOTH_THREADS
#define FB_SMOOTH_THREADS 128
#endif
#ifndef FB_SMOOTH_MINB
#define FB_SMOOTH_MINB (2048 / FB_SMOOTH_THREADS)
#endif
// MAP = false: value row = graph row, rows [row_begin, row_end) (focusr_mean_filter).  MAP = true: CTA b smooths graph
// rows [t.x, t.x + t.y) with t = cta_rows[b], and graph row i is value row i + t.z (focusr_mean_filter_mapped).  The
// host builds the table so that no CTA spans two segments: one table load per thread, no search, and the CTA's graph
// rows stay contiguous, so the L2 prefetch of its matrix slice is that of the identity form.
template <int C, bool MAP>
__global__ void __launch_bounds__(FB_SMOOTH_THREADS, FB_SMOOTH_MINB)
k_mean_filter(const int* __restrict__ row_ptr, const int* __restrict__ cols, const double* __restrict__ weights,
              const double* __restrict__ degree, int row_begin, int row_end, const int4* __restrict__ cta_rows,
              const double* __restrict__ x, double* __restrict__ out, int n_cols_rt) {
  int c0, c1, shift = 0;
  if (MAP) {
    const int4 t = cta_rows[blockIdx.x];
    c0 = t.x;
    c1 = t.x + t.y;
    shift = t.z;
  } else {
    c0 = row_begin + blockIdx.x * blockDim.x;
    c1 = min(row_end, c0 + (int)blockDim.x);
  }
  const int i = c0 + threadIdx.x;
  {
    const int q0 = row_ptr[c0], q1 = row_ptr[c1];
    for (int q = q0 + 32 * (int)threadIdx.x; q < q1; q += 32 * (int)blockDim.x) prefetch_l2_line(cols + q);
    for (int q = q0 + 16 * (int)threadIdx.x; q < q1; q += 16 * (int)blockDim.x) prefetch_l2_line(weights + q);
  }
  pdl_wait();
  pdl_launch_dependents();
  if (i >= (MAP ? c1 : row_end)) return;
  const int nc = C > 0 ? C : n_cols_rt;
  const double dsm = FB_DIV(1.0, FB_ADD(1.0, degree[i]));
  const int p0 = row_ptr[i], p1 = row_ptr[i + 1];
  constexpr int CMAX = C > 0 ? C : 8;
  double acc[CMAX];
#pragma unroll
  for (int k = 0; k < CMAX; ++k) acc[k] = 0.0;
  bool diag_done = false;
  for (int p = p1 - 1; p >= p0; --p) {
    const int j = cols[p];
    const double wp = weights[p];
    if (!diag_done && j < i) {
      const double* xi = x + (size_t)(i + shift) * nc;
#pragma unroll
      for (int k = 0; k < CMAX; ++k)
        if (k < nc) acc[k] = FB_ADD(acc[k], FB_MUL(dsm, xi[k]));
      diag_done = true;
    }
    double val;
    if (j == i) {
      val = FB_MUL(dsm, FB_ADD(wp, 1.0));
      diag_done = true;
    } else {
      val = FB_MUL(dsm, wp);
    }
    const double* xj = x + (size_t)(j + shift) * nc;
#pragma unroll
    for (int k = 0; k < CMAX; ++k)
      if (k < nc) acc[k] = FB_ADD(acc[k], FB_MUL(val, xj[k]));
  }
  if (!diag_done) {
    const double* xi = x + (size_t)(i + shift) * nc;
#pragma unroll
    for (int k = 0; k < CMAX; ++k)
      if (k < nc) acc[k] = FB_ADD(acc[k], FB_MUL(dsm, xi[k]));
  }
  double* o = out + (size_t)(i + shift) * nc;
#pragma unroll
  for (int k = 0; k < CMAX; ++k)
    if (k < nc) o[k] = acc[k];
}

__global__ void k_copy_rows(const double* __restrict__ in, double* __restrict__ out, long long begin, long long end) {
  const long long t = begin + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < end) out[t] = in[t];
}

struct SmoothLayout {
  double *buf_a, *buf_b;
  size_t bytes;
};

static SmoothLayout smooth_layout(int n_rows, int n_cols, void* ws) {
  Carver cv(ws, (size_t)-1);
  SmoothLayout l;
  l.buf_a = cv.take<double>((size_t)n_rows * n_cols);
  l.buf_b = cv.take<double>((size_t)n_rows * n_cols);
  l.bytes = cv.used + 256;
  return l;
}

// the mapped form adds its CTA table: segment s of n_s rows takes ceil(n_s / threads) CTAs, so n_rows / threads +
// n_segments entries bound it
static SmoothLayout smooth_mapped_layout(int n_rows, int n_cols, int n_segments, void* ws, int4** table) {
  Carver cv(ws, (size_t)-1);
  SmoothLayout l;
  l.buf_a = cv.take<double>((size_t)n_rows * n_cols);
  l.buf_b = cv.take<double>((size_t)n_rows * n_cols);
  *table = cv.take<int4>((size_t)n_rows / FB_SMOOTH_THREADS + n_segments + 1);
  l.bytes = cv.used + 256;
  return l;
}

// the chain of passes of both entry points: ping-pong between pa and pb, the last pass into out
template <bool MAP>
static int smooth_chain(const int* row_ptr, const int* cols, const double* weights, const double* degree, int row_begin,
                        int row_end, const int4* cta_rows, int n_ctas, const double* src, double* pa, double* pb,
                        double* out, int n_cols, int iterations, cudaStream_t stream) {
  const dim3 grid(n_ctas), block(FB_SMOOTH_THREADS);
  for (int it = 0; it < iterations; ++it) {
    double* dst = it == iterations - 1 ? out : ((it & 1) ? pb : pa);
    cudaError_t e;
#define FB_SMOOTH(CC, NC)                                                                                             \
  launch_pdl(k_mean_filter<CC, MAP>, grid, block, stream, row_ptr, cols, weights, degree, row_begin, row_end, cta_rows, \
             src, dst, NC)
    if (n_cols == 3)
      e = FB_SMOOTH(3, 3);
    else if (n_cols == 1)
      e = FB_SMOOTH(1, 1);
    else if (n_cols == 2)  // the two curvature columns of node features (SpectralBatch)
      e = FB_SMOOTH(2, 2);
    else
      e = FB_SMOOTH(0, n_cols);
#undef FB_SMOOTH
    FB_CUDA(e);
    src = dst;
  }
  FB_COUNT_LAUNCH(iterations);
  FB_LAUNCH_CHECK();
  return FB_OK;
}

}  // namespace fb

using namespace fb;

extern "C" {

long long focusr_sell_entries_cap(const int* mesh_point_off_host, const int* mesh_info_host, int n_meshes) {
  return sell_entries_cap(mesh_point_off_host, mesh_info_host, n_meshes, 0);
}

size_t focusr_mean_filter_workspace_bytes(int n_rows, int n_cols) { return smooth_layout(n_rows, n_cols, nullptr).bytes; }

int focusr_mean_filter(const int* row_ptr, const int* cols, const double* weights, const double* degree,
                       int row_begin, int row_end, const double* values_in, double* values_out, int n_cols,
                       int iterations, void* workspace, size_t workspace_bytes, focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FB_REQUIRE(row_end > row_begin && n_cols >= 1 && n_cols <= 8 && iterations >= 0,
             "mean_filter: need rows, 1 <= n_cols <= 8, iterations >= 0");
  const int n = row_end - row_begin;
  const int T = FB_SMOOTH_THREADS;
  if (iterations == 0) {
    const long long b = (long long)row_begin * n_cols, e = (long long)row_end * n_cols;
    k_copy_rows<<<div_up(e - b, T), T, 0, stream>>>(values_in, values_out, b, e);
    FB_COUNT_LAUNCH(1);
    FB_LAUNCH_CHECK();
    return FB_OK;
  }
  const SmoothLayout l = smooth_layout(n, n_cols, workspace);
  FB_REQUIRE(iterations == 1 || (workspace != nullptr && workspace_bytes >= l.bytes),
             "mean_filter: workspace too small (%zu < %zu)", workspace_bytes, l.bytes);
  // ping-pong between two buffers indexed by global row (shifted so that row_begin lands on their start)
  const size_t rb = (size_t)row_begin;
  return smooth_chain<false>(row_ptr, cols, weights, degree, row_begin, row_end, nullptr, div_up(n, T), values_in,
                             l.buf_a - rb * n_cols, l.buf_b - rb * n_cols, values_out, n_cols, iterations, stream);
}

size_t focusr_mean_filter_mapped_workspace_bytes(int n_rows, int n_cols, int n_segments) {
  int4* table;
  return smooth_mapped_layout(n_rows, n_cols, n_segments, nullptr, &table).bytes;
}

int focusr_mean_filter_mapped(const int* row_ptr, const int* cols, const double* weights, const double* degree,
                              const int* mesh_off, const int* mesh_off_host, int n_meshes, const int* seg_mesh,
                              const int* seg_mesh_host, int n_segments, const double* values_in, double* values_out,
                              int n_cols, int iterations, void* workspace, size_t workspace_bytes,
                              focusr_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  (void)mesh_off;
  (void)seg_mesh;
  FB_REQUIRE(n_meshes > 0 && n_segments > 0 && n_cols >= 1 && n_cols <= 8 && iterations >= 0,
             "mean_filter_mapped: need meshes and segments, 1 <= n_cols <= 8, iterations >= 0");
  FB_REQUIRE(mesh_off_host != nullptr && seg_mesh_host != nullptr,
             "mean_filter_mapped: the host copies of mesh_off and seg_mesh are required");
  long long n_rows = 0;
  for (int s = 0; s < n_segments; ++s) {
    const int m = seg_mesh_host[s];
    FB_REQUIRE(m >= 0 && m < n_meshes, "mean_filter_mapped: segment %d maps to mesh %d, outside [0, %d)", s, m, n_meshes);
    n_rows += mesh_off_host[m + 1] - mesh_off_host[m];
  }
  FB_REQUIRE(n_rows > 0 && n_rows <= INT_MAX, "mean_filter_mapped: the segments hold %lld rows", n_rows);
  const int T = FB_SMOOTH_THREADS;
  if (iterations == 0) {
    k_copy_rows<<<div_up(n_rows * n_cols, T), T, 0, stream>>>(values_in, values_out, 0, n_rows * n_cols);
    FB_COUNT_LAUNCH(1);
    FB_LAUNCH_CHECK();
    return FB_OK;
  }
  int4* table;
  const SmoothLayout l = smooth_mapped_layout((int)n_rows, n_cols, n_segments, workspace, &table);
  FB_REQUIRE(workspace != nullptr && workspace_bytes >= l.bytes, "mean_filter_mapped: workspace too small (%zu < %zu)",
             workspace_bytes, l.bytes);
  // Segments that are consecutive graph meshes in ascending order are the graph rows [rb, re) shifted by rb: the
  // identity form on pointers shifted by rb rows, as focusr_mean_filter shifts its ping-pong buffers.  The table form
  // costs a dependent table load in every CTA's prologue (B200 at 1000 W, 128 meshes of 15 212 vertices: 18.1 against
  // 17.2 ms for 300 passes, tools/batch_mesh_pairs_bench.py), so the identity form is used wherever the map allows it.
  bool run = true;
  for (int s = 1; s < n_segments && run; ++s) run = seg_mesh_host[s] == seg_mesh_host[s - 1] + 1;
  if (run) {
    const int rb = mesh_off_host[seg_mesh_host[0]], re = mesh_off_host[seg_mesh_host[n_segments - 1] + 1];
    const size_t sh = (size_t)rb * n_cols;
    return smooth_chain<false>(row_ptr, cols, weights, degree, rb, re, nullptr, div_up(re - rb, T), values_in - sh,
                               l.buf_a - sh, l.buf_b - sh, values_out - sh, n_cols, iterations, stream);
  }
  // one entry per CTA {first graph row, rows, value row - graph row}; tiny, built here and staged by the runtime
  // (pageable source)
  std::vector<int4> cta;
  int seg0 = 0;
  for (int s = 0; s < n_segments; ++s) {
    const int m = seg_mesh_host[s], g0 = mesh_off_host[m], n = mesh_off_host[m + 1] - g0;
    for (int r = 0; r < n; r += T) cta.push_back(make_int4(g0 + r, n - r < T ? n - r : T, seg0 - g0, 0));
    seg0 += n;
  }
  FB_CUDA(cudaMemcpyAsync(table, cta.data(), sizeof(int4) * cta.size(), cudaMemcpyHostToDevice, stream));
  return smooth_chain<true>(row_ptr, cols, weights, degree, 0, 0, table, (int)cta.size(), values_in, l.buf_a, l.buf_b,
                            values_out, n_cols, iterations, stream);
}
}
