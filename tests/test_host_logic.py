"""Host-side logic without a GPU: the solver driver (through the plain-loop test double in
tests/hostsim), mesh IO / generators, eigsort's n x n decisions, and the C ABI surface."""
import os
import re

import numpy as np
import pytest
import scipy.linalg as sla

from oracle import port
from pyfocusr_b200 import mesh as fmesh

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ dense kernels
@pytest.mark.parametrize("b", [8, 16, 24, 40, 96])
def test_rayleigh_ritz_sym_matches_lapack(hostsim, b):
    rng = np.random.RandomState(b)
    x = rng.standard_normal((300, b)) * np.logspace(0, 3, b)[None, :]  # graded columns, as after a filter
    d = rng.uniform(1, 3, 300)
    s = rng.standard_normal((300, 300))
    g = x.T @ (d[:, None] * x)
    h = x.T @ (s + s.T) @ x
    h = 0.5 * (h + h.T)
    ref = sla.eigh(h, g, eigvals_only=True)
    gg, hh, w, th = g.copy(), h.copy(), np.zeros((b, b)), np.zeros(b)
    rc = hostsim.hostsim_rr_sym(gg, hh, w, th, b)
    assert rc >> 8 == 0 and (rc & 0xFF) < 30
    assert np.max(np.abs(th - ref)) <= 1e-11 * np.max(np.abs(ref))
    assert np.max(np.abs(w.T @ g @ w - np.eye(b))) <= 1e-10
    assert np.all(np.diff(th) >= 0)


@pytest.mark.parametrize("b", [8, 16, 32, 48, 96])
def test_rayleigh_ritz_sym_has_no_loop_order_dependence(hostsim, b):
    """The same race check for the symmetric step (csrc/dense_small.h: Cholesky, congruence, round-robin Jacobi)."""
    rng = np.random.RandomState(7 * b)
    x = rng.randn(6 * b, b)
    d = np.sort(rng.rand(6 * b)) * 2.0
    g, h = x.T @ x, x.T @ (d[:, None] * x)
    out = []
    for fn in (hostsim.hostsim_rr_sym, hostsim.hostsim_rr_sym_rev):
        gg, hh, w, th = g.copy(), h.copy(), np.zeros((b, b)), np.zeros(b)   # both are overwritten
        rc = fn(gg, hh, w, th, b)
        assert rc >> 8 == 0 and (rc & 0xFF) < 30          # no clamped pivot, Jacobi converged
        out.append((w, th))
    (w1, t1), (w2, t2) = out
    assert np.allclose(t1, t2, rtol=1e-11, atol=1e-13)
    for j in range(b):
        c = abs(w1[:, j] @ g @ w2[:, j]) / np.sqrt((w1[:, j] @ g @ w1[:, j]) * (w2[:, j] @ g @ w2[:, j]))
        assert abs(c - 1.0) <= 1e-8, j


@pytest.mark.parametrize("n", [2, 7, 32, 64])
def test_eig_general_matches_numpy(hostsim, n):
    rng = np.random.RandomState(n)
    a = np.ascontiguousarray(rng.standard_normal((n, n)))
    ev, vec = np.zeros(2 * n), np.zeros(2 * n * n)
    assert hostsim.hostsim_eig_general(a, n, ev, vec) == 0
    e = ev[0::2] + 1j * ev[1::2]
    v = (vec[0::2] + 1j * vec[1::2]).reshape(n, n)
    ref = np.linalg.eigvals(a)
    assert max(np.min(np.abs(ref - x)) for x in e) <= 1e-11 * np.max(np.abs(ref))
    assert np.max(np.abs(a @ v - v * e[None, :])) <= 1e-11 * np.max(np.abs(ref))


@pytest.mark.parametrize("b", [8, 16, 24, 48, 64])
def test_rr_nonsym_device_form_matches_numpy_and_the_host_form(hostsim, b):
    """csrc/nonsym_small.h (the algorithm one CTA per mesh runs on the B200, here with the sequential Par) against
    numpy's eig of the same pencil and against csrc/nonsym_host.hpp: same low real Ritz values in the same order, Ritz
    vectors that satisfy the projected problem, a full-rank basis."""
    rng = np.random.RandomState(b)
    n = 6 * b
    x = rng.randn(n, b)
    # a nearly diagonalisable operator with a few complex pairs, like the one-way entries of an open mesh produce
    d = np.sort(rng.rand(n)) * 2.0
    lop = np.diag(d)
    for i in range(0, 6, 2):
        lop[n - 2 - i, n - 1 - i], lop[n - 1 - i, n - 2 - i] = 0.3, -0.3
    lop += 1e-3 * rng.randn(n, n)
    g, h = x.T @ x, x.T @ (lop @ x)
    outs = []
    for form in (1, 0):
        w, th, nl = np.zeros((b, b)), np.zeros(b), np.zeros(1, np.int32)
        rc = hostsim.hostsim_rr_nonsym(form, np.ascontiguousarray(g), np.ascontiguousarray(h), b, 1.2, w, th, nl)
        assert rc == 0
        outs.append((w, th, int(nl[0])))
    (w, th, nl), (w0, th0, nl0) = outs
    ev = np.linalg.eigvals(np.linalg.solve(g, h))
    real_low = np.sort(ev[(np.abs(ev.imag) <= 1e-8 * np.abs(ev)) & (ev.real <= 1.2)].real)
    assert nl == nl0 == real_low.size and nl > 0
    assert np.allclose(th[:nl], real_low, rtol=1e-9, atol=1e-12) and np.allclose(th[:nl], th0[:nl], rtol=1e-9, atol=1e-12)
    for j in range(nl):   # H w = theta G w
        r = h @ w[:, j] - th[j] * (g @ w[:, j])
        assert np.linalg.norm(r) <= 1e-8 * np.linalg.norm(h @ w[:, j])
        c = abs(w[:, j] @ g @ w0[:, j]) / np.sqrt((w[:, j] @ g @ w[:, j]) * (w0[:, j] @ g @ w0[:, j]))
        assert abs(c - 1.0) <= 1e-8   # same Ritz vector as the host form, up to sign
    assert np.linalg.matrix_rank(w) == b and np.linalg.cond(w) < 1e10
    # the two forms span the same invariant subspaces pair by pair: compare the sorted real parts of all Ritz values
    assert np.allclose(np.sort(th), np.sort(th0), rtol=1e-8, atol=1e-10)


@pytest.mark.parametrize("b", [8, 24, 40, 64])
def test_rr_nonsym_device_form_has_no_loop_order_dependence(hostsim, b):
    """Race check of csrc/nonsym_small.h without a GPU: every `par.for_n` of the device algorithm run once in ascending
    and once in descending index order.  A body that read what another index of the same loop writes -- a data race in
    the CUDA kernel, where the indices are threads -- would change the result; only the accumulation order of the few
    reductions may differ (rounding)."""
    rng = np.random.RandomState(100 + b)
    n = 5 * b
    x = rng.randn(n, b)
    lop = np.diag(np.sort(rng.rand(n)) * 2.0) + 1e-3 * rng.randn(n, n)
    for i in range(0, 4, 2):
        lop[n - 2 - i, n - 1 - i], lop[n - 1 - i, n - 2 - i] = 0.25, -0.25
    g, h = np.ascontiguousarray(x.T @ x), np.ascontiguousarray(x.T @ (lop @ x))
    res = []
    for form in (1, 2):
        w, th, nl = np.zeros((b, b)), np.zeros(b), np.zeros(1, np.int32)
        assert hostsim.hostsim_rr_nonsym(form, g, h, b, 1.2, w, th, nl) == 0
        res.append((w, th, int(nl[0])))
    (w1, t1, n1), (w2, t2, n2) = res
    assert n1 == n2 and np.allclose(t1, t2, rtol=1e-10, atol=1e-12)
    for j in range(b):   # same columns up to sign and rounding; the (Re, Im) columns of a complex pair up to the phase of
        # its eigenvector, i.e. as the plane they span
        same = np.nonzero(np.abs(t2 - t1[j]) <= 1e-9 * max(1.0, abs(t1[j])))[0]
        basis = w2[:, same]
        coef = np.linalg.lstsq(basis, w1[:, j], rcond=None)[0]
        assert np.linalg.norm(basis @ coef - w1[:, j]) <= 1e-7 * np.linalg.norm(w1[:, j]), (j, same.tolist())
        if j < n1:
            assert same.size == 1


def test_edge_weight_matches_numpy(hostsim):
    rng = np.random.RandomState(0)
    for _ in range(200):
        for dim in (3, 4, 5):
            p1, p2 = rng.standard_normal(dim) * 50, rng.standard_normal(dim) * 50
            assert hostsim.hostsim_edge_weight(p1, p2, dim) == 1.0 / np.sqrt(np.sum(np.square(p1 - p2)))


# ------------------------------------------------------------------------------------------------ solver driver
def _solve(hostsim, meshes, k0, n_needed, block, ldv=32, tol=1e-10, beta=0.0, full=False):
    rps, cols, ws, degs, pts, offs, zrs = [], [], [], [], [], [0], []
    nnz = 0
    sym = True
    for m in meshes:
        a = port.adjacency(m.points, m.tris)
        deg = port.row_sums_sequential(a)
        rps.append(a.indptr[:-1].astype(np.int64) + nnz)
        cols.append(a.indices.astype(np.int64) + offs[-1])
        ws.append(a.data)
        degs.append(deg)
        pts.append(m.points)
        nnz += a.nnz
        offs.append(offs[-1] + m.points.shape[0])
        zrs.append(int(np.sum(deg == 0)))
        pat = (a != 0).astype(np.int8)
        sym &= (pat - pat.multiply(pat.T)).nnz == 0
    rp = np.concatenate(rps + [np.array([nnz])]).astype(np.int32)
    deg = np.concatenate(degs)
    M, N = len(meshes), offs[-1]
    vals, vecs = np.zeros((M, ldv)), np.zeros((N, ldv))
    ri, rd = np.zeros(6 * M, np.int32), np.zeros(2 * M)
    rc = hostsim.hostsim_eigs(rp, np.concatenate(cols).astype(np.int32), np.concatenate(ws), deg, port.degree_inv(deg),
                              np.ascontiguousarray(np.concatenate(pts)), N, np.array(offs, np.int32), M, int(sym),
                              np.array(zrs, np.int32), block, k0, n_needed, 1, 1e-10, tol, 60, 1e3, 4096, beta, ldv,
                              vals, vecs, ri, rd)
    if full:
        return rc, vals, vecs, ri.reshape(M, 6), offs, sym, rd.reshape(M, 2)
    return rc, vals, vecs, ri.reshape(M, 6), offs, sym


def _check(mesh, vals, vecs, n):
    lap = port.laplacian(port.adjacency(mesh.points, mesh.tris))
    rv, rvec = port.recursive_eig(lap, n + 1, n, 1)
    o = np.argsort(rv)
    rv, rvec = rv[o], rvec[:, o]
    assert vals.size == rv.size
    assert np.max(np.abs(vals - rv) / rv) <= 1e-6           # BASELINE.json tolerance
    for i in range(rv.size):
        r = rvec[:, i] / np.linalg.norm(rvec[:, i])
        assert min(np.linalg.norm(vecs[:, i] - r), np.linalg.norm(vecs[:, i] + r)) <= 1e-5


def test_driver_symmetric_batch(hostsim, shipped_meshes):
    ms = [shipped_meshes["target_mesh"], shipped_meshes["source_mesh"]]
    rc, vals, vecs, ri, offs, sym = _solve(hostsim, ms, 7, 6, 16)
    assert rc == 0 and sym and ri[:, 0].tolist() == [0, 0] and ri[:, 1].tolist() == [6, 6] and ri[:, 2].tolist() == [7, 7]
    for k, m in enumerate(ms):
        _check(m, vals[k, :6], vecs[offs[k]:offs[k + 1], :6], 6)


def test_driver_mixed_precision_passes(hostsim, shipped_meshes):
    """Filter passes in fp32 (the test double rounds as the k_filter_sell steps do): a pass that lands above the fp32
    floor runs on fp32 blocks, the pass that reaches the tolerance runs in fp32 correction form (z = p(L)x - x driven by
    the fp64 residual).  Rayleigh-Ritz and residuals stay fp64, so tolerance and parity hold, at no extra degree."""
    ms = [shipped_meshes["target_mesh"], fmesh.perturbed_ellipsoid(20, 3)]
    rc0, vals0, vecs0, ri0, offs, sym = _solve(hostsim, ms, 7, 6, 16)
    assert hostsim.hostsim_last_lowp_degree() == 0
    hostsim.hostsim_set_lowp(1.4e-6)
    try:
        rc, vals, vecs, ri, offs, sym, rd = _solve(hostsim, ms, 7, 6, 16, full=True)
        lowp = hostsim.hostsim_last_lowp_degree()
    finally:
        hostsim.hostsim_set_lowp(0.0)
    assert rc == 0 and rc0 == 0 and sym and ri[:, 1].tolist() == [6, 6]
    assert lowp == 10 + ri[0, 4]                               # probe and every pass ran in an fp32 form
    assert ri[:, 4].max() <= ri0[:, 4].max() * 1.15            # fp32 rounding does not cost filter degree
    assert ri[:, 3].max() <= ri0[:, 3].max() + 1
    assert rd[:, 0].max() <= 1e-10
    assert np.max(np.abs(vals[:, :6] - vals0[:, :6]) / vals0[:, :6]) <= 1e-9
    for k, m in enumerate(ms):
        _check(m, vals[k, :6], vecs[offs[k]:offs[k + 1], :6], 6)
    # a tighter tolerance than the correction form's noise allows in one go: more passes, still converges
    hostsim.hostsim_set_lowp(1.4e-6)
    try:
        rc, vals, vecs, ri, offs, sym, rd = _solve(hostsim, ms[:1], 7, 6, 16, tol=1e-12, full=True)
        assert rc == 0 and rd[0, 0] <= 1e-12
        # the non-symmetric path takes the fp32 forms too (test_driver_nonsymmetric_fp32_passes)
        _solve(hostsim, [shipped_meshes["target_mesh_15k"]], 7, 6, 48)
        assert hostsim.hostsim_last_lowp_degree() > 0
    finally:
        hostsim.hostsim_set_lowp(0.0)


def test_driver_mixed_precision_on_rough_anisotropic_and_shuffled_meshes(hostsim):
    """The fp32 pass logic away from the smooth bench meshes: vertex noise of a quarter edge length, an 8 : 1 : 0.3
    ellipsoid (poor start block: several short unsettled passes first), a random vertex order, all in one batch and
    alone with k = 14.  Same answers as fp64, no more than one extra Rayleigh-Ritz step, no extra filter degree to speak of."""
    rng = np.random.RandomState(0)
    base = fmesh.perturbed_ellipsoid(14, 7)
    e = np.linalg.norm(base.points[base.tris[:, 0]] - base.points[base.tris[:, 1]], axis=1).mean()
    rough = fmesh.PolyData(base.points + rng.standard_normal(base.points.shape) * 0.25 * e, base.tris)
    thin = fmesh.PolyData(base.points * np.array([8.0, 1.0, 0.3]), base.tris)
    perm = rng.permutation(base.points.shape[0])
    shuf = fmesh.PolyData(base.points[perm], np.argsort(perm)[base.tris].astype(base.tris.dtype))
    for ms, k, b in (([rough, thin, shuf], 7, 16), ([rough], 14, 24)):
        rc0, vals0, vecs0, ri0, offs, sym = _solve(hostsim, ms, k, k - 1, b)
        hostsim.hostsim_set_lowp(1.4e-6)
        try:
            rc, vals, vecs, ri, offs, sym, rd = _solve(hostsim, ms, k, k - 1, b, full=True)
            lowp = hostsim.hostsim_last_lowp_degree()
        finally:
            hostsim.hostsim_set_lowp(0.0)
        assert rc == 0 and rc0 == 0 and sym and lowp == 10 + ri[0, 4]
        assert rd[:, 0].max() <= 1e-10
        assert ri[:, 3].max() <= ri0[:, 3].max() + 1 and ri[:, 4].max() <= 1.2 * ri0[:, 4].max()
        assert np.max(np.abs(vals[:, :k - 1] - vals0[:, :k - 1]) / vals0[:, :k - 1]) <= 1e-9
        for i, m in enumerate(ms):
            _check(m, vals[i, :k - 1], vecs[offs[i]:offs[i + 1], :k - 1], k - 1)


def test_driver_pass_plan_on_a_bench_mesh(hostsim):
    """The filter degree IS the cost of the eigensolve on the GPU (one launch per degree over the whole batch), so the pass
    plan on a bench mesh (BASELINE.json configs[2]: nu = 39, 15 212 vertices) is pinned here, where no GPU is needed: probe
    + 3 Rayleigh-Ritz steps, every filter step in an fp32 form, ~275 steps in all (292 with the first fp64-only driver)."""
    m = fmesh.perturbed_ellipsoid(39, 0)
    hostsim.hostsim_set_lowp(1.4e-6)
    try:
        rc, vals, vecs, ri, offs, sym, rd = _solve(hostsim, [m], 7, 6, 16, full=True)
        lowp = hostsim.hostsim_last_lowp_degree()
    finally:
        hostsim.hostsim_set_lowp(0.0)
    assert rc == 0 and sym and ri[0, 1] == 6 and ri[0, 3] == 3
    assert 240 <= ri[0, 4] <= 285 and lowp == 10 + ri[0, 4]
    assert rd[0, 0] <= 6e-11 and 1.5 < rd[0, 1] < 1.56        # lands well inside the tolerance; probed spectrum bound
    _check(m, vals[0, :6], vecs[:, :6], 6)


def test_driver_nonsymmetric_with_retry(hostsim, shipped_meshes):
    """15k source: 8 one-way entries (complex eigenvalue pairs), 2 unreferenced vertices -> k=14, 11 pairs."""
    m = shipped_meshes["source_mesh_15k"]
    rc, vals, vecs, ri, offs, sym = _solve(hostsim, [m], 7, 6, 48)
    assert rc == 0 and not sym and ri[0, 0] == 0 and ri[0, 1] == 11 and ri[0, 2] == 14
    _check(m, vals[0, :11], vecs[:, :11], 6)


def test_driver_nonsymmetric_fp32_passes(hostsim, shipped_meshes):
    """The fp32 filter forms on the reference's own open meshes (non-symmetric adjacency, complex pairs carried in the
    block): every pass iterates in fp32 (plain blocks, then the correction form), no more steps than in fp64, same parity."""
    for name in ("source_mesh_15k", "target_mesh_15k"):
        m = shipped_meshes[name]
        rc0, _, _, ri0, _, sym = _solve(hostsim, [m], 7, 6, 40)
        hostsim.hostsim_set_lowp(1.4e-6)
        try:
            rc, vals, vecs, ri, offs, sym, rd = _solve(hostsim, [m], 7, 6, 40, full=True)
            lowp = hostsim.hostsim_last_lowp_degree()
        finally:
            hostsim.hostsim_set_lowp(0.0)
        assert rc0 == 0 and rc == 0 and not sym
        assert lowp == ri[0, 4] > 0                        # every filter step of the solve ran in fp32
        assert ri[0, 4] <= 1.05 * ri0[0, 4] and ri[0, 1] == ri0[0, 1] and ri[0, 2] == ri0[0, 2]
        assert rd[0, 0] <= 1e-10
        _check(m, vals[0, :ri[0, 1]], vecs[:, :ri[0, 1]], 6)


def test_driver_isolated_vertices_symmetric(hostsim):
    """Zero-degree rows are pinned and counted analytically (SURVEY.md section 7.3-2)."""
    base = fmesh.perturbed_ellipsoid(8, 4)
    pts = np.concatenate([base.points, [[0.0, 0.0, 0.0], [1.0, 2.0, 3.0]]])
    m = fmesh.PolyData(pts, base.tris)
    rc, vals, vecs, ri, offs, sym = _solve(hostsim, [m], 7, 6, 24)
    assert rc == 0 and sym and ri[0, 2] == 14 and ri[0, 1] == 11  # 3 null eigenvalues: 14 - 3
    _check(m, vals[0, :11], vecs[:, :11], 6)
    assert np.all(vecs[-2:, :11] == 0.0)


def test_driver_reports_small_block(hostsim):
    m = fmesh.icosphere(8)  # exact 3/5/7-fold multiplets; block 16 = 1+3+5+7 cuts right at a multiplet edge
    rc, vals, vecs, ri, offs, sym = _solve(hostsim, [m], 11, 10, 16)
    assert ri[0, 0] in (2, 0)
    rc, vals, vecs, ri, offs, sym = _solve(hostsim, [m], 11, 10, 32)
    assert rc == 0 and ri[0, 1] == 10


# ------------------------------------------------------------------------------------------------ meshes
def test_icosphere_and_vtk_roundtrip(tmp_path):
    for nu in (1, 2, 7):
        s = fmesh.icosphere(nu)
        assert s.points.shape == (10 * nu * nu + 2, 3) and s.tris.shape == (20 * nu * nu, 3)
        assert np.allclose(np.linalg.norm(s.points, axis=1), 1.0)
        a = port.adjacency(s.points, s.tris)
        assert (abs(a - a.T)).nnz == 0 and a.nnz == 3 * s.tris.shape[0]  # closed, consistently oriented
    m = fmesh.perturbed_ellipsoid(5, 1)
    path = tmp_path / "m.vtk"
    with open(path, "w") as f:
        f.write("# vtk DataFile Version 4.2\nvtk output\nASCII\nDATASET POLYDATA\nPOINTS %d double\n" % m.points.shape[0])
        f.write("\n".join(" ".join(repr(float(v)) for v in p) for p in m.points))
        f.write("\nPOLYGONS %d %d\n" % (m.tris.shape[0], 4 * m.tris.shape[0]))
        f.write("\n".join("3 %d %d %d" % tuple(t) for t in m.tris))
        f.write("\nPOINT_DATA %d\nSCALARS thickness double\nLOOKUP_TABLE default\n" % m.points.shape[0])
        f.write(" ".join("%d.5" % i for i in range(m.points.shape[0])) + "\n")
    r = fmesh.read_vtk_mesh(str(path))
    assert np.array_equal(r.points, m.points) and np.array_equal(r.tris, m.tris)
    assert r.point_scalars["thickness"][3] == 3.5
    # generic accessor path (what a foreign vtkPolyData-like object goes through)

    class Foreign:
        def __init__(self, m):
            self._m = m

        def __getattr__(self, name):
            if name in ("points", "tris"):
                raise AttributeError(name)
            return getattr(self._m, name)

    p, t = fmesh.mesh_arrays(Foreign(m))
    assert np.array_equal(p, m.points) and np.array_equal(t, m.tris)
    assert m.GetCell(0).GetEdge(2).GetPointId(1) == m.tris[0, 0]


# ------------------------------------------------------------------------------------------------ eigsort decisions
def test_decide_matches_and_moves(golden):
    from pyfocusr_b200.eigsort import c_lambda_matrix, decide_matches, moves_from_matches

    for tag, n in (("5k", 6), ("15k", 6), ("5k_n13", 13)):
        cl = c_lambda_matrix(golden[tag + "_t_eig_vals"], golden[tag + "_s_eig_vals"], n)
        assert np.array_equal(cl, golden[tag + "_c_lambda"])
        for ref_is_target in (True, False):
            q, tm, sm, fl = decide_matches(cl, golden[tag + "_c_hist"], golden[tag + "_c_hist_f"], golden[tag + "_c_spatial"],
                                           golden[tag + "_c_spatial_f"], ref_is_target)
            q2, tm2, sm2, fl2 = port.eigen_sort_decide(cl, golden[tag + "_c_hist"], golden[tag + "_c_hist_f"],
                                                       golden[tag + "_c_spatial"], golden[tag + "_c_spatial_f"], ref_is_target)
            assert np.array_equal(q, q2) and np.array_equal(tm, tm2) and np.array_equal(sm, sm2) and fl == fl2
            # the (dst, src, sign) move list applied to random columns == the reference's flip + fancy-index copy
            rng = np.random.RandomState(0)
            vt, vs = rng.standard_normal((50, n + 2)), rng.standard_normal((40, n + 3))
            et, es = vt.copy(), vs.copy()
            port.eigen_sort_apply(et, es, tm, sm, fl, ref_is_target)
            d, s, sg = moves_from_matches(tm, sm, fl, ref_is_target)
            mine = (vs if ref_is_target else vt).copy()
            old = mine.copy()
            mine[:, d] = old[:, s] * sg[None, :]
            assert np.array_equal(mine, es if ref_is_target else et)
        if tag == "5k":
            assert np.array_equal(q2 if not ref_is_target else q2, q2)


# ------------------------------------------------------------------------------------------------ C ABI surface
def test_library_exports_every_declared_symbol():
    import ctypes

    from pyfocusr_b200 import _lib

    header = open(os.path.join(ROOT, "include", "focusr_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(focusr_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name + " is declared in include/focusr_b200.h but not exported"
        assert name in _lib.SIGNATURES, name + " has no ctypes signature in pyfocusr_b200/_lib.py"
    assert sorted(_lib.SIGNATURES) == declared
    loaded = _lib.load()
    assert loaded.focusr_version() >= 100 and loaded.focusr_last_error() is not None
    assert loaded.focusr_eigs_block_size(7, 6, 1, 0, 0) == 16 and loaded.focusr_eigs_block_size(7, 6, 1, 4, 2) == 40


def test_product_never_imports_the_oracle_and_has_no_cpu_fallback():
    pkg = os.path.join(ROOT, "pyfocusr_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h", ".hpp")):
                src = open(os.path.join(dirpath, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), fn
                assert "hostsim" not in src or fn in ("dense_small.h", "chfsi_driver.hpp", "rowops.h", "cpd_host.hpp", "eigsort_decide.h", "nonsym_small.h"), fn
    import torch

    if not torch.cuda.is_available():
        from pyfocusr_b200 import Graph, _lib

        with pytest.raises(RuntimeError):
            _lib.require_cuda()
        g = Graph(fmesh.icosphere(2), n_rand_samples=5)
        with pytest.raises(RuntimeError):
            g.get_graph_spectrum()  # fails loudly: no CPU path


def test_decide_batch_equals_per_pair_scipy():
    """The vectorised all-permutations assignment == scipy LSAP + the reference's flip logic, pair by pair."""
    from pyfocusr_b200.eigsort import decide_batch, decide_matches, moves_from_matches

    rng = np.random.RandomState(5)
    for n in (3, 6, 8, 10):
        P = 40
        mats = [np.exp(rng.standard_normal((P, n, n))) for _ in range(5)]
        for ref_is_target in (True, False):
            q, d, s, sg = decide_batch(*mats, ref_is_target)
            for p in range(P):
                q1, tm, sm, fl = decide_matches(*[m[p] for m in mats], ref_is_target)
                d1, s1, sg1 = moves_from_matches(tm, sm, fl, ref_is_target)
                assert np.array_equal(q[p], q1) and np.array_equal(d[p], d1) and np.array_equal(s[p], s1)
                assert np.array_equal(sg[p], sg1)


def test_device_lsap_is_scipys_algorithm_including_ties(hostsim):
    """csrc/eigsort_decide.h lsap_square (what the GPU runs, one thread per pair) against scipy's
    linear_sum_assignment: identical assignments, not just identical optima -- on generic matrices, on integer matrices
    with few distinct values (many tied optima), on constant matrices and on matrices with repeated rows."""
    from scipy.optimize import linear_sum_assignment

    rng = np.random.RandomState(11)
    cases = []
    for n in (1, 2, 3, 6, 7, 13, 40, 96):
        for _ in range(12):
            cases.append(np.exp(rng.standard_normal((n, n))))
            cases.append(rng.randint(0, 3, size=(n, n)).astype(np.float64))       # heavy ties
            cases.append(rng.randint(0, 2, size=(n, n)).astype(np.float64))
        cases.append(np.ones((n, n)))
        cases.append(np.zeros((n, n)))
        rep = np.exp(rng.standard_normal((n, n)))
        rep[n // 2:] = rep[: n - n // 2]                                            # duplicated eigenvector-like rows
        cases.append(rep)
    for c in cases:
        n = c.shape[0]
        out = np.zeros(n, dtype=np.int32)
        assert hostsim.hostsim_lsap(np.ascontiguousarray(c), n, out) == 0
        assert np.array_equal(out, linear_sum_assignment(c)[1]), (n, c)
    bad = np.full((3, 3), np.inf)
    assert hostsim.hostsim_lsap(bad, 3, np.zeros(3, dtype=np.int32)) == -1


def test_lsap_cluster_scheme_is_scipys_scan():
    """The bookkeeping csrc/lsap.cu uses in place of scipy's `remaining` array and serial scan, restated in numpy: every
    column keeps its POSITION in scipy's scan order (removing position p moves the last position to p), the minimum is
    taken by (value, tie key) with key = 2^30 + position for unassigned columns (the last one in scan order wins) and
    2^30 - 1 - position for assigned ones (the first one wins), and the duals are updated per visited column.  Must give
    scipy's assignment on matrices full of ties, square and rectangular."""
    from scipy.optimize import linear_sum_assignment

    def scheme(cost):
        nr, nc = cost.shape
        u, v = np.zeros(nr), np.zeros(nc)
        col4row, r4c, path = -np.ones(nr, int), -np.ones(nc, int), -np.ones(nc, int)
        for cur in range(nr):
            spc, sc, pos = np.full(nc, np.inf), np.zeros(nc, bool), nc - 1 - np.arange(nc)
            min_val, i, nrem, sink, prev_last, prev_index = 0.0, cur, nc, -1, -1, -1
            while sink < 0:
                best = None
                for j in range(nc):            # "every thread updates its columns"
                    if sc[j]:
                        continue
                    if pos[j] == prev_last:
                        pos[j] = prev_index
                    r = ((min_val + cost[i, j]) - u[i]) - v[j]
                    if r < spc[j]:
                        spc[j], path[j] = r, i
                    key = (0x40000000 + pos[j]) if r4c[j] < 0 else (0x3FFFFFFF - pos[j])
                    if best is None or spc[j] < best[0] or (spc[j] == best[0] and key > best[1]):
                        best = (spc[j], key, j)
                min_val, key, js = best
                index = key - 0x40000000 if key >= 0x40000000 else 0x3FFFFFFF - key
                sc[js] = True
                prev_last, prev_index, nrem = nrem - 1, index, nrem - 1
                if r4c[js] < 0:
                    sink = js
                else:
                    i = r4c[js]
            u[cur] += min_val
            for j in np.nonzero(sc)[0]:
                d = min_val - spc[j]
                if r4c[j] >= 0:
                    u[r4c[j]] += d
                v[j] -= d
            j = sink
            while True:
                ii = path[j]
                r4c[j] = ii
                col4row[ii], j = j, col4row[ii]
                if ii == cur:
                    break
        return col4row

    rng = np.random.RandomState(5)
    for t in range(60):
        n = rng.randint(2, 24)
        m = n + rng.randint(0, 4)
        if t % 3 == 0:
            c = rng.rand(n, m)
        elif t % 3 == 1:
            c = rng.randint(0, 3, (n, m)).astype(float)
        else:
            p = rng.randint(0, 3, (m, 2)).astype(float)
            c = np.sqrt(((p[:n, None] - p[None]) ** 2).sum(-1))
        assert np.array_equal(scheme(c), linear_sum_assignment(c)[1]), (t, n, m)


def test_device_eigsort_decisions_equal_the_host_classes(hostsim):
    """eigsort_decide_pair (the kernel body of focusr_eigsort_decide) against the drop-in classes' host code
    (c_lambda_matrix + decide_matches + moves_from_matches, i.e. the reference's eigsort.py:66-122, 142-160) and the
    spectral weights of focusr.py:481-490: same matches, flips and moves; Q and weights to rounding."""
    from pyfocusr_b200.eigsort import c_lambda_matrix, decide_matches, moves_from_matches

    rng = np.random.RandomState(3)
    for n, ns, nf_t, nf_s in ((6, 3, 6, 11), (6, 3, 6, 6), (13, 10, 13, 13), (4, 4, 9, 5)):
        for ref_is_target in (True, False):
            for weighted in (True, False):
                vt = np.sort(rng.rand(nf_t)) * 1e-3 + 1e-4
                vs = np.sort(rng.rand(nf_s)) * 1e-3 + 1e-4
                ch, chf, cs, csf = (np.exp(rng.standard_normal((n, n))) for _ in range(4))
                cl = c_lambda_matrix(vt, vs, n)
                q1, tm, sm, fl = decide_matches(cl, ch, chf, cs, csf, ref_is_target)
                d1, s1, g1 = moves_from_matches(tm, sm, fl, ref_is_target)
                w1 = q1[:ns] * np.maximum(vs[:ns], vt[:ns])
                w1 = np.exp(-(w1 ** 2) / (2 * np.mean(w1) ** 2)) if weighted else np.ones(ns)
                q, w = np.zeros(n), np.zeros(ns)
                d, s_, g = (np.zeros(n, dtype=np.int32) for _ in range(3))
                rc = hostsim.hostsim_eigsort_decide(vt, nf_t, vs, nf_s, ch, chf, cs, csf, n, ns, int(ref_is_target),
                                                    int(weighted), q, d, s_, g, w)
                assert rc == 0
                assert np.array_equal(d, d1) and np.array_equal(s_, s1) and np.array_equal(g, g1)
                assert np.allclose(q, q1, rtol=1e-13, atol=0) and np.allclose(w, w1, rtol=1e-12, atol=0)


def test_polydata_scalar_setters():
    """focusr.py:576-599 sets point scalars on the meshes for visualisation; the PolyData stand-in takes them."""
    m = fmesh.icosphere(2)
    vals = np.arange(m.points.shape[0])
    m.GetPointData().SetScalars(vals)
    assert np.array_equal(m.GetPointData().GetScalars().values if hasattr(m.GetPointData().GetScalars(), "values")
                          else m.point_scalars["scalars"], vals)
    with pytest.raises(ValueError):
        m.GetPointData().SetScalars(vals[:-1])


def test_non_triangle_cells_are_rejected():
    class Quad:
        def GetNumberOfPoints(self): return 4
        def GetPoint(self, i): return (float(i), 0.0, 0.0)
        def GetNumberOfCells(self): return 1
        def GetCell(self, i):
            class C:
                def GetNumberOfEdges(self): return 4
            return C()

    with pytest.raises(ValueError, match="triangle"):
        fmesh.mesh_arrays(Quad())


def test_driver_nonsymmetric_on_damaged_meshes(hostsim):
    """Open / badly oriented meshes: removed triangles and flipped triangles give one-way adjacency entries, hence
    complex eigenvalue pairs that the Chebyshev filter amplifies; the Euclidean Rayleigh-Ritz path must still
    return the reference's eigenpairs (SURVEY.md section 7.3-1)."""
    import ctypes

    from pyfocusr_b200 import _lib

    rng = np.random.RandomState(0)
    lib = ctypes.CDLL(_lib.LIB_PATH)
    lib.focusr_eigs_block_size.argtypes = [ctypes.c_int] * 5
    for nu, holes, flips in ((12, 5, 0), (16, 20, 10), (20, 3, 30)):
        base = fmesh.perturbed_ellipsoid(nu, 3)
        t = base.tris.copy()
        keep = np.ones(len(t), bool)
        keep[rng.choice(len(t), holes, replace=False)] = False
        t = t[keep]
        fl = rng.choice(len(t), flips, replace=False)
        t[fl] = t[fl][:, [0, 2, 1]]
        m = fmesh.PolyData(base.points, t)
        a = port.adjacency(m.points, m.tris)
        pat = (a != 0).astype(np.int8)
        oneway = int((pat - pat.multiply(pat.T)).nnz)
        assert oneway > 0
        b = lib.focusr_eigs_block_size(7, 6, 1, oneway, 0)
        rc, vals, vecs, ri, offs, sym = _solve(hostsim, [m], 7, 6, b, ldv=64)
        assert rc == 0 and not sym and ri[0, 1] == 6
        _check(m, vals[0, :6], vecs[:, :6], 6)


def test_legacy_vtk_reader_ascii_binary_and_v5_layout(tmp_path, shipped_meshes):
    """SURVEY.md section 8f-2: mesh ingest without VTK.  ASCII and BINARY round trips are bit-exact, the
    version 5.x OFFSETS/CONNECTIVITY layout is understood, other sections are skipped."""
    m = shipped_meshes["source_mesh_15k"]
    scal = dict(m.point_scalars)
    assert scal                                                  # the shipped files carry thickness_change_(mm)
    for binary in (False, True):
        p = str(tmp_path / ("m%d.vtk" % binary))
        fmesh.write_vtk_mesh(m, p, binary=binary)
        r = fmesh.read_vtk_mesh(p)
        assert np.array_equal(r.points, m.points) and np.array_equal(r.tris, m.tris)
        for k, v in scal.items():
            assert np.array_equal(r.point_scalars[k.replace(" ", "_")], v)
    # version 5.1 layout written by hand, with a LINES section and CELL_DATA to skip, ASCII and BINARY
    small = fmesh.icosphere(2)
    n, f = small.points.shape[0], small.tris.shape[0]
    offs, conn = np.arange(0, 3 * f + 1, 3), small.tris.reshape(-1)
    for binary in (False, True):
        p = str(tmp_path / ("v5_%d.vtk" % binary))
        with open(p, "wb") as out:
            out.write(b"# vtk DataFile Version 5.1\nv5\n" + (b"BINARY\n" if binary else b"ASCII\n") + b"DATASET POLYDATA\n")
            out.write(b"POINTS %d float\n" % n)
            p32 = small.points.astype(np.float32)
            out.write(p32.astype(">f4").tobytes() + b"\n" if binary else (" ".join("%.9g" % v for v in p32.reshape(-1)) + "\n").encode())
            out.write(b"LINES 2 2\nOFFSETS vtktypeint64\n")
            out.write(np.array([0, 2], ">i8").tobytes() + b"\n" if binary else b"0 2\n")
            out.write(b"CONNECTIVITY vtktypeint64\n")
            out.write(np.array([0, 1], ">i8").tobytes() + b"\n" if binary else b"0 1\n")
            out.write(b"POLYGONS %d %d\nOFFSETS vtktypeint64\n" % (f + 1, 3 * f))
            out.write(offs.astype(">i8").tobytes() + b"\n" if binary else (" ".join(map(str, offs)) + "\n").encode())
            out.write(b"CONNECTIVITY vtktypeint64\n")
            out.write(conn.astype(">i8").tobytes() + b"\n" if binary else (" ".join(map(str, conn)) + "\n").encode())
            out.write(b"CELL_DATA %d\nSCALARS cid int 1\nLOOKUP_TABLE default\n" % (f + 1))
            cid = np.arange(f + 1)
            out.write(cid.astype(">i4").tobytes() + b"\n" if binary else (" ".join(map(str, cid)) + "\n").encode())
            out.write(b"POINT_DATA %d\nSCALARS height float\nLOOKUP_TABLE default\n" % n)
            out.write(p32[:, 2].astype(">f4").tobytes() + b"\n" if binary else (" ".join("%.9g" % v for v in p32[:, 2]) + "\n").encode())
        r = fmesh.read_vtk_mesh(p)
        assert np.array_equal(r.points, p32.astype(np.float64)) and np.array_equal(r.tris, small.tris)
        assert list(r.point_scalars) == ["height"] and np.array_equal(r.point_scalars["height"], p32[:, 2].astype(np.float64))
    # error behaviour
    bad = str(tmp_path / "bad.vtk")
    open(bad, "wb").write(b"# vtk DataFile Version 3.0\nx\nASCII\nDATASET POLYDATA\nPOINTS 3 double\n0 0 0 1 0 0 0 1 0\nPOLYGONS 1 5\n4 0 1 2 0\n")
    with pytest.raises(ValueError):
        fmesh.read_vtk_mesh(bad)                                  # a quad
    open(bad, "wb").write(b"# vtk DataFile Version 3.0\nx\nASCII\nDATASET POLYDATA\nPOINTS 3 double\n0 0 0 1 0 0 0 1 0\nPOLYGONS 1 4\n3 0 1 7\n")
    with pytest.raises(ValueError):
        fmesh.read_vtk_mesh(bad)                                  # index out of range
    open(bad, "wb").write(b"not a vtk file\n\n\n\n")
    with pytest.raises(ValueError):
        fmesh.read_vtk_mesh(bad)


def test_pack_meshes_offsets_and_global_ids():
    """SpectralBatch.pack_meshes: targets then sources, triangle ids shifted by each mesh's row offset."""
    from pyfocusr_b200 import SpectralBatch

    a, b, c = fmesh.icosphere(2), fmesh.icosphere(3), fmesh.perturbed_ellipsoid(2, 1)
    pts, tris, off, n_pairs = SpectralBatch.pack_meshes([a, b], [c, a])
    sizes = [m.points.shape[0] for m in (a, b, c, a)]
    assert n_pairs == 2 and off.dtype == np.int32 and off.tolist() == np.concatenate([[0], np.cumsum(sizes)]).tolist()
    assert tuple(pts.shape) == (sum(sizes), 3) and str(pts.dtype) == "torch.float64" and str(tris.dtype) == "torch.int32"
    t = tris.numpy()
    f0 = 0
    for m, o in zip((a, b, c, a), off[:-1]):
        f1 = f0 + m.tris.shape[0]
        assert np.array_equal(t[f0:f1], m.tris + o)
        assert np.array_equal(pts.numpy()[o:o + m.points.shape[0]], m.points)
        f0 = f1
    with pytest.raises(ValueError):
        SpectralBatch.pack_meshes([a], [])
