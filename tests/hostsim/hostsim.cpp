// TEST DOUBLE -- never shipped, never loaded by pyfocusr_b200.
//
// Plain-loop implementation of the `Backend` concept of pyfocusr_b200/csrc/chfsi_driver.hpp so the
// solver's host logic (filter bounds, degree schedule, retry contract, symmetric warp-Jacobi code
// path in its sequential instantiation, non-symmetric complex-Schur path) can be exercised by
// `pytest -m "not gpu"` on a machine without a GPU.  The product backend is CudaBackend in
// pyfocusr_b200/csrc/eigs.cu; nothing in the product links or calls this file.
//
// Build: tests/hostsim/build.sh  (g++ -O2 -ffp-contract=off -shared -fPIC)
#include <cstring>
#include <vector>

#include "../../pyfocusr_b200/csrc/cpd_host.hpp"
#include "../../pyfocusr_b200/csrc/chfsi_driver.hpp"
#include "../../pyfocusr_b200/csrc/eigsort_decide.h"
#include "../../pyfocusr_b200/csrc/nonsym_small.h"
#include "../../pyfocusr_b200/csrc/rowops.h"

namespace {

double g_lowp_floor = 0.0;   // hostsim_set_lowp: SolveParams::lowp_floor of the next solves
int g_last_lowp_degree = 0;  // lowp_degree of mesh 0 of the last solve
int g_nonsym_small = 1;      // hostsim_set_nonsym_small: 1 = the device algorithm (nonsym_small.h, sequential Par), 0 = nonsym_host.hpp

// A second sequential `Par`: the indices of every parallel loop in DESCENDING order.  A loop body that reads what another
// index of the same loop writes (a race on the GPU) gives different results under the two orders.
struct RevPar {
  template <class F>
  void for_n(int n, F f) const {
    for (int i = n - 1; i >= 0; --i) f(i);
  }
  void sync() const {}
  double sum(double v) const { return v; }
  int lane() const { return 0; }
};

template <class Par>
int rr_nonsym_small_par(const double* g, const double* h, int b, double cut, double* w, double* theta, int* n_low) {
  std::vector<double> gh((size_t)2 * b * b), rs((size_t)b * b);
  std::memcpy(gh.data(), g, sizeof(double) * b * b);
  std::memcpy(gh.data() + (size_t)b * b, h, sizeof(double) * b * b);
  std::vector<fb::Cd> hc((size_t)b * b), qc((size_t)b * b);
  std::vector<unsigned char> scratch(fb::nonsym_small_scratch_bytes(b) + 16);
  Par par;
  return fb::rr_nonsym_small(gh.data(), gh.data() + (size_t)b * b, hc.data(), qc.data(), rs.data(), b, cut, w, theta, n_low,
                             scratch.data(), par);
}

int rr_nonsym_small_host(const double* g, const double* h, int b, double cut, double* w, double* theta, int* n_low) {
  std::vector<double> gh((size_t)2 * b * b), rs((size_t)b * b);
  std::memcpy(gh.data(), g, sizeof(double) * b * b);
  std::memcpy(gh.data() + (size_t)b * b, h, sizeof(double) * b * b);
  std::vector<fb::Cd> hc((size_t)b * b), qc((size_t)b * b);
  std::vector<unsigned char> scratch(fb::nonsym_small_scratch_bytes(b) + 16);
  fb::SeqPar par;
  return fb::rr_nonsym_small(gh.data(), gh.data() + (size_t)b * b, hc.data(), qc.data(), rs.data(), b, cut, w, theta, n_low,
                             scratch.data(), par);
}

struct HostBackend {
  const int* rp;
  const int* cols;
  const double* w;
  const double* deg;
  const double* dinv;
  const double* pts;
  const int* off;
  const int* zr;
  int N, M, B;
  bool sym;
  double* out_vals;
  double* out_vecs;
  int ldv;
  std::vector<double> X, Y, Xn, Z, G, H, W, theta, res, R;

  int n_meshes() const { return M; }
  int block() const { return B; }
  bool symmetric() const { return sym; }
  int zero_rows(int m) const { return zr[m]; }
  bool lowp_available() const { return true; }

  void init_block() {
    X.assign((size_t)N * B, 0.0);
    Y = X;
    Xn = X;
    Z = X;
    G.assign((size_t)M * B * B, 0.0);
    H = G;
    W = G;
    theta.assign((size_t)M * B, 0.0);
    res = theta;
    for (int m = 0; m < M; ++m) {
      double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
      for (int i = off[m]; i < off[m + 1]; ++i)
        for (int a = 0; a < 3; ++a) {
          lo[a] = std::min(lo[a], pts[3 * i + a]);
          hi[a] = std::max(hi[a], pts[3 * i + a]);
        }
      double scale = 0.0;
      for (int a = 0; a < 3; ++a) scale = std::max(scale, 0.5 * (hi[a] - lo[a]));
      if (!(scale > 0.0)) scale = 1.0;
      for (int i = off[m]; i < off[m + 1]; ++i) {
        if (deg[i] == 0.0) continue;
        const double x = (pts[3 * i] - 0.5 * (lo[0] + hi[0])) / scale;
        const double y = (pts[3 * i + 1] - 0.5 * (lo[1] + hi[1])) / scale;
        const double z = (pts[3 * i + 2] - 0.5 * (lo[2] + hi[2])) / scale;
        for (int c = 0; c < B; ++c)
          X[(size_t)i * B + c] = fb::start_block_value(c, x, y, z, (uint32_t)(i - off[m]), 1u);
      }
    }
  }
  void spmm(const std::vector<double>& in, int i, double* acc) const {
    for (int c = 0; c < B; ++c) acc[c] = 0.0;
    for (int p = rp[i]; p < rp[i + 1]; ++p) {
      const double* row = &in[(size_t)cols[p] * B];
      for (int c = 0; c < B; ++c) acc[c] += w[p] * row[c];
    }
  }
  void apply_DmA() {
    std::vector<double> acc(B);
    for (int i = 0; i < N; ++i) {
      spmm(X, i, acc.data());
      for (int c = 0; c < B; ++c) Z[(size_t)i * B + c] = deg[i] * X[(size_t)i * B + c] - acc[c];
    }
  }
  void gram() {
    std::fill(G.begin(), G.end(), 0.0);
    std::fill(H.begin(), H.end(), 0.0);
    for (int m = 0; m < M; ++m)
      for (int i = off[m]; i < off[m + 1]; ++i) {
        const double gw = sym ? deg[i] + 1e-8 : 1.0;
        const double hw = sym ? 1.0 : dinv[i];
        const double* x = &X[(size_t)i * B];
        const double* z = &Z[(size_t)i * B];
        for (int p = 0; p < B; ++p)
          for (int q = 0; q < B; ++q) {
            G[((size_t)m * B + p) * B + q] += x[p] * gw * x[q];
            H[((size_t)m * B + p) * B + q] += x[p] * hw * z[q];
          }
      }
  }
  int rr_sym() {
    fb::SeqPar par;
    std::vector<double> y((size_t)B * B), rot(B + 2);
    std::vector<int> rank(B), pq(B + 2);
    int worst = 0;
    for (int m = 0; m < M; ++m) {
      double* g = &G[(size_t)m * B * B];
      double* h = &H[(size_t)m * B * B];
      worst |= fb::rayleigh_ritz_sym(g, h, y.data(), &W[(size_t)m * B * B], &theta[(size_t)m * B],
                                     rank.data(), rot.data(), pq.data(), B, par);
    }
    return worst;
  }
  // the device form of the non-symmetric Rayleigh-Ritz step (what CudaBackend runs in one CTA per mesh)
  std::vector<int> ns_rc, ns_low;
  bool rr_nonsym_device(const double* cut) {
    if (!g_nonsym_small || B > 64) return false;
    ns_rc.assign(M, 0);
    ns_low.assign(M, 0);
    for (int m = 0; m < M; ++m)
      ns_rc[m] = rr_nonsym_small_host(&G[(size_t)m * B * B], &H[(size_t)m * B * B], B, cut[m], &W[(size_t)m * B * B],
                                      &theta[(size_t)m * B], &ns_low[m]);
    return true;
  }
  void get_nonsym_info(int* rc, int* n_low) {
    for (int m = 0; m < M; ++m) {
      rc[m] = ns_rc[m];
      n_low[m] = ns_low[m];
    }
  }
  void get_GH(double* g, double* h) {
    std::memcpy(g, G.data(), G.size() * sizeof(double));
    std::memcpy(h, H.data(), H.size() * sizeof(double));
  }
  void set_W_theta(const double* wv, const double* th) {
    std::memcpy(W.data(), wv, W.size() * sizeof(double));
    std::memcpy(theta.data(), th, theta.size() * sizeof(double));
  }
  void rotate_and_residual() {
    std::vector<double> xr(B), zr_(B), num((size_t)M * B, 0.0), den((size_t)M * B, 0.0);
    for (int m = 0; m < M; ++m) {
      const double* wm = &W[(size_t)m * B * B];
      for (int i = off[m]; i < off[m + 1]; ++i) {
        double* x = &X[(size_t)i * B];
        const double* z = &Z[(size_t)i * B];
        for (int j = 0; j < B; ++j) {
          double a = 0.0, b2 = 0.0;
          for (int k = 0; k < B; ++k) {
            a += x[k] * wm[k * B + j];
            b2 += z[k] * wm[k * B + j];
          }
          xr[j] = a;
          zr_[j] = b2;
        }
        if (R.size() != X.size()) R.assign(X.size(), 0.0);
        for (int j = 0; j < B; ++j) {
          x[j] = xr[j];
          const double r = dinv[i] * zr_[j] - theta[(size_t)m * B + j] * xr[j];
          R[(size_t)i * B + j] = r;  // residual block, consumed by filter_correction
          num[(size_t)m * B + j] += r * r;
          den[(size_t)m * B + j] += xr[j] * xr[j];
        }
      }
      for (int j = 0; j < B; ++j)
        res[(size_t)m * B + j] = std::sqrt(num[(size_t)m * B + j] / den[(size_t)m * B + j]);
    }
  }
  void get_theta_res(double* th, double* rs) {
    std::memcpy(th, theta.data(), theta.size() * sizeof(double));
    std::memcpy(rs, res.data(), res.size() * sizeof(double));
  }
  // fp32 pass as k_filter_sell (modes 0-2) runs it: blocks, matrix entries and table values rounded to float, float arithmetic
  void filter_lowp(int deg_m, const double* alpha, const double* gamma, const double* center) {
    std::vector<float> p(X.size()), y(X.size()), n(X.size()), acc(B);
    for (size_t t = 0; t < X.size(); ++t) y[t] = (float)X[t];
    for (int s = 0; s < deg_m; ++s) {
      for (int m = 0; m < M; ++m) {
        const float al = (float)alpha[(size_t)m * deg_m + s], ga = (float)gamma[(size_t)m * deg_m + s], c = (float)center[m];
        for (int i = off[m]; i < off[m + 1]; ++i) {
          for (int k = 0; k < B; ++k) acc[k] = 0.0f;
          for (int q = rp[i]; q < rp[i + 1]; ++q) {
            const float wq = (float)w[q];
            const float* row = &y[(size_t)cols[q] * B];
            for (int k = 0; k < B; ++k) acc[k] += wq * row[k];
          }
          const float d = (float)deg[i], di = (float)dinv[i];
          for (int k = 0; k < B; ++k) {
            const float yv = y[(size_t)i * B + k];
            const float ly = di * (d * yv - acc[k]);
            float r = al * (ly - c * yv);
            if (ga != 0.0f) r -= ga * p[(size_t)i * B + k];
            n[(size_t)i * B + k] = r;
          }
        }
      }
      p.swap(y);
      y.swap(n);
    }
    for (size_t t = 0; t < X.size(); ++t) X[t] = (double)y[t];
  }
  // fp32 correction pass as k_filter_sell (modes 3-4) runs it: X += z_deg, z_{k+1} = alpha_kj ((L - c) z_k + r_j) - gamma_kj z_{k-1}, z_0 = 0;
  // z, r, matrix entries and tables rounded to float, float arithmetic; tables are [mesh][step][column]
  void filter_correction(int deg_m, const double* a_m, const double* beta_m) {
    // the per-column tables, as k_corr_tables builds them on the GPU
    std::vector<double> alpha((size_t)M * deg_m * B), gamma((size_t)M * deg_m * B), center(M);
    for (int m = 0; m < M; ++m) {
      center[m] = 0.5 * (beta_m[m] + a_m[m]);
      for (int j = 0; j < B; ++j)
        fb::corr_table_column(a_m[m], theta[(size_t)m * B + j], beta_m[m], deg_m, [&](int s, double al, double ga) {
          alpha[((size_t)m * deg_m + s) * B + j] = al;
          gamma[((size_t)m * deg_m + s) * B + j] = ga;
        });
    }
    std::vector<float> p(X.size(), 0.f), z(X.size(), 0.f), n(X.size()), acc(B), r(X.size());
    for (size_t t = 0; t < X.size(); ++t) r[t] = (float)R[t];
    for (int s = 0; s < deg_m; ++s) {
      for (int m = 0; m < M; ++m) {
        const float c = (float)center[m];
        const double* al = &alpha[((size_t)m * deg_m + s) * B];
        const double* ga = &gamma[((size_t)m * deg_m + s) * B];
        for (int i = off[m]; i < off[m + 1]; ++i) {
          for (int k = 0; k < B; ++k) acc[k] = 0.0f;
          for (int q = rp[i]; q < rp[i + 1]; ++q) {
            const float wq = (float)w[q];
            const float* row = &z[(size_t)cols[q] * B];
            for (int k = 0; k < B; ++k) acc[k] += wq * row[k];
          }
          const float d = (float)deg[i], di = (float)dinv[i];
          for (int k = 0; k < B; ++k) {
            const float zv = z[(size_t)i * B + k];
            const float lz = di * (d * zv - acc[k]);
            float o = (float)al[k] * ((lz - c * zv) + r[(size_t)i * B + k]);
            if (s > 0) o -= (float)ga[k] * p[(size_t)i * B + k];
            n[(size_t)i * B + k] = o;
          }
        }
      }
      p.swap(z);
      z.swap(n);
    }
    for (size_t t = 0; t < X.size(); ++t) X[t] += (double)z[t];
  }
  void filter(int deg_m, const double* alpha, const double* gamma, const double* center, bool lowp) {
    if (lowp) {
      filter_lowp(deg_m, alpha, gamma, center);
      return;
    }
    std::vector<double> acc(B);
    Y = X;  // Y = current, X = previous
    for (int s = 0; s < deg_m; ++s) {
      for (int m = 0; m < M; ++m) {
        const double al = alpha[(size_t)m * deg_m + s], ga = gamma[(size_t)m * deg_m + s], c = center[m];
        for (int i = off[m]; i < off[m + 1]; ++i) {
          spmm(Y, i, acc.data());
          for (int k = 0; k < B; ++k) {
            const double y = Y[(size_t)i * B + k];
            const double ly = dinv[i] * (deg[i] * y - acc[k]);
            Xn[(size_t)i * B + k] = al * (ly - c * y) - ga * X[(size_t)i * B + k];
          }
        }
      }
      X.swap(Y);   // X <- old Y
      Y.swap(Xn);  // Y <- new
    }
    X = Y;
  }
  void finalize(const int* flags, const int* sel, const int* n_out) {
    for (int m = 0; m < M; ++m) {
      if (!flags[m]) continue;
      for (int j = 0; j < n_out[m]; ++j) {
        const int c = sel[(size_t)m * B + j];
        double ss = 0.0, best = -1.0, bestv = 0.0;
        for (int i = off[m]; i < off[m + 1]; ++i) {
          const double v = X[(size_t)i * B + c];
          ss += v * v;
          if (std::fabs(v) > best) {
            best = std::fabs(v);
            bestv = v;
          }
        }
        const double sc = (bestv < 0.0 ? -1.0 : 1.0) / std::sqrt(ss);
        for (int i = off[m]; i < off[m + 1]; ++i) out_vecs[(size_t)i * ldv + j] = X[(size_t)i * B + c] * sc;
        out_vals[(size_t)m * ldv + j] = theta[(size_t)m * B + c];
      }
    }
  }
};

}  // namespace

extern "C" {

// result_i: per mesh [status, n_out, k_final, outer_iters, total_degree, block]; result_d: per mesh [max_residual, filter upper edge]
int hostsim_eigs(const int* rp, const int* cols, const double* w, const double* deg, const double* dinv,
                 const double* pts, int n_rows, const int* off, int n_meshes, int symmetric,
                 const int* zero_rows, int block, int k0, int n_needed, int k_buffer, double min_eig,
                 double tol, int max_outer, double amp_target, int max_degree, double beta, int ldv,
                 double* eig_vals, double* eig_vecs, int* result_i, double* result_d) {
  HostBackend be;
  be.rp = rp; be.cols = cols; be.w = w; be.deg = deg; be.dinv = dinv; be.pts = pts; be.off = off;
  be.zr = zero_rows; be.N = n_rows; be.M = n_meshes; be.B = block; be.sym = symmetric != 0;
  be.out_vals = eig_vals; be.out_vecs = eig_vecs; be.ldv = ldv;
  fb::SolveParams p;
  p.k0 = k0; p.n_needed = n_needed; p.k_buffer = k_buffer; p.min_eig = min_eig; p.tol = tol;
  p.max_outer = max_outer; p.amp_target = amp_target; p.max_degree = max_degree; p.beta = beta > 0.0 ? beta : 2.0; p.ldv = ldv;
  p.probe_degree = beta == 0.0 ? 10 : 0; p.land = 0.4; p.lowp_floor = g_lowp_floor; p.lowp_aim = 1.5e-6;
  std::vector<fb::MeshResult> r(n_meshes);
  const int rc = fb::chfsi_solve(be, p, r.data());
  g_last_lowp_degree = r[0].lowp_degree;
  for (int m = 0; m < n_meshes; ++m) {
    int* ri = result_i + 6 * m;
    ri[0] = r[m].status; ri[1] = r[m].n_out; ri[2] = r[m].k_final; ri[3] = r[m].outer_iters;
    ri[4] = r[m].total_degree; ri[5] = r[m].block;
    result_d[2 * m] = r[m].max_residual;
    result_d[2 * m + 1] = r[m].beta;
  }
  return rc;
}

void hostsim_set_lowp(double floor) { g_lowp_floor = floor; }
void hostsim_set_nonsym_small(int on) { g_nonsym_small = on; }

// the non-symmetric Rayleigh-Ritz step in its device form (nonsym_small.h) and in its host form (chfsi_driver.hpp)
int hostsim_rr_nonsym(int device_form, const double* g, const double* h, int b, double cut, double* w, double* theta, int* n_low) {
  if (device_form == 2) return rr_nonsym_small_par<RevPar>(g, h, b, cut, w, theta, n_low);   // loops in reverse order
  if (device_form) return rr_nonsym_small_host(g, h, b, cut, w, theta, n_low);
  std::vector<double> gg(g, g + (size_t)b * b), hh(h, h + (size_t)b * b);
  return fb::rr_nonsym_host(gg.data(), hh.data(), b, cut, w, theta, n_low);
}
int hostsim_last_lowp_degree(void) { return g_last_lowp_degree; }

int hostsim_rr_sym(double* g, double* h, double* w, double* theta, int b) {
  std::vector<double> y((size_t)b * b), rot(b + 2);
  std::vector<int> rank(b), pq(b + 2);
  fb::SeqPar par;
  return fb::rayleigh_ritz_sym(g, h, y.data(), w, theta, rank.data(), rot.data(), pq.data(), b, par);
}

// the same with every parallel loop in descending index order (race check, see RevPar)
int hostsim_rr_sym_rev(double* g, double* h, double* w, double* theta, int b) {
  std::vector<double> y((size_t)b * b), rot(b + 2);
  std::vector<int> rank(b), pq(b + 2);
  RevPar par;
  return fb::rayleigh_ritz_sym(g, h, y.data(), w, theta, rank.data(), rot.data(), pq.data(), b, par);
}

// a (n x n, symmetric) is overwritten by the eigenvectors (columns); evals unsorted
int hostsim_eig_sym(double* a, double* evals, int n) { return fb::eig_sym_host(a, evals, n); }

int hostsim_rr_leading(double* g, double* h, int b, double* w, double* theta) {
  return fb::rr_leading_host(g, h, b, w, theta);
}

int hostsim_eig_general(const double* a, int n, double* evals_ri, double* evecs_ri) {
  std::vector<fb::cplx> ev(n), vec((size_t)n * n);
  const int rc = fb::eig_general(a, n, ev.data(), vec.data());
  for (int i = 0; i < n; ++i) {
    evals_ri[2 * i] = ev[i].real();
    evals_ri[2 * i + 1] = ev[i].imag();
  }
  for (int i = 0; i < n * n; ++i) {
    evecs_ri[2 * i] = vec[i].real();
    evecs_ri[2 * i + 1] = vec[i].imag();
  }
  return rc;
}

double hostsim_edge_weight(const double* p1, const double* p2, int dim) { return fb::edge_weight(p1, p2, dim); }

// the device-side decisions of eigsort (csrc/eigsort_decide.h), compiled for the host
int hostsim_lsap(const double* cost, int n, int* col4row) { return fb::lsap_square(cost, n, col4row); }

int hostsim_eigsort_decide(const double* vals_t, int nf_t, const double* vals_s, int nf_s, const double* c_hist,
                           const double* c_hist_f, const double* c_spatial, const double* c_spatial_f, int n, int ns,
                           int target_as_reference, int weighted, double* q, int* dst, int* src, int* sign, double* w) {
  std::vector<double> scratch((size_t)2 * n * n);
  return fb::eigsort_decide_pair(vals_t, nf_t, vals_s, nf_s, c_hist, c_hist_f, c_spatial, c_spatial_f, n, ns,
                                 target_as_reference != 0, weighted != 0, q, dst, src, sign, w, scratch.data());
}
}
