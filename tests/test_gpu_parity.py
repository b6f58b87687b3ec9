"""Parity of the CUDA path (through the C ABI / the drop-in Python API) against the CPU oracle
(oracle/port.py, pinned bitwise to the unmodified reference) and the committed golden fixtures.

Tolerances are BASELINE.json's: Laplacian CSR structure bit-exact and values <= 1e-12 relative
(we assert bit-exact), eigenvalues <= 1e-6 relative, eigenvectors <= 1e-5 up to sign (rotation
inside degenerate subspaces), KNN indices bit-exact on the reference's features.
"""
import hashlib

import numpy as np
import pytest
from scipy import sparse

pytestmark = pytest.mark.gpu


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def torch():
    import torch

    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module")
def synth():
    from pyfocusr_b200.mesh import icosphere, perturbed_ellipsoid

    base = icosphere(20)
    return dict(ico20=base, ell20a=perturbed_ellipsoid(20, 0, base=base), ell20b=perturbed_ellipsoid(20, 1, base=base),
                ell39=perturbed_ellipsoid(39, 3))


def all_meshes(shipped_meshes, synth):
    d = dict(shipped_meshes)
    d.update(synth)
    return d


# ------------------------------------------------------------------------------------------- K1
def test_laplacian_bit_exact(torch, shipped_meshes, synth, golden):
    from oracle import port
    from pyfocusr_b200._device import DeviceGraph

    for name, m in all_meshes(shipped_meshes, synth).items():
        g = DeviceGraph([m.points], [m.tris])
        a = port.adjacency(m.points, m.tris)
        deg = port.row_sums_sequential(a)
        rp, ci, w = g.adjacency_host()
        assert np.array_equal(rp, a.indptr) and np.array_equal(ci, a.indices), name
        assert np.array_equal(w, a.data), name + ": adjacency weights not bit-exact"
        assert np.array_equal(g.degree.cpu().numpy(), deg), name + ": degree"
        assert np.array_equal(g.degree_inv.cpu().numpy(), port.degree_inv(deg)), name
        lap = port.laplacian(a, deg)
        lrp, lci, lv = g.laplacian_host()
        assert np.array_equal(lrp, lap.indptr) and np.array_equal(lci, lap.indices), name
        assert np.array_equal(lv, lap.data), name + ": Laplacian values not bit-exact"
        pat = (a != 0).astype(np.int8)
        oneway = int((pat - pat.multiply(pat.T)).nnz)  # stored (i,j) whose mirror (j,i) is not stored
        longest = int(np.max(np.diff(a.indptr)))
        assert g.mesh_info_host[0].tolist() == [a.nnz, oneway, int(np.sum(deg == 0)), 0, longest, 0, 0, 0], name
    # golden counts of the shipped 15k meshes (SURVEY.md section 8 table)
    for tag, nm in (("15k_t", "target_mesh_15k"), ("15k_s", "source_mesh_15k")):
        m = shipped_meshes[nm]
        g = DeviceGraph([m.points], [m.tris])
        cnt = golden[tag + "_counts"]
        assert g.mesh_info_host[0, 0] == cnt[0] and 2 * g.mesh_info_host[0, 1] == cnt[2] and g.mesh_info_host[0, 2] == cnt[4]
        lrp, lci, lv = g.laplacian_host()
        assert sha(lv) + sha(lci) + sha(lrp) == str(golden[tag + "_L_sha"])


def test_laplacian_batched_equals_single(torch, shipped_meshes, synth):
    from pyfocusr_b200._device import DeviceGraph

    ms = [shipped_meshes["target_mesh"], synth["ell20a"], shipped_meshes["source_mesh_15k"]]
    g = DeviceGraph([m.points for m in ms], [m.tris for m in ms])
    rp, ci, w = g.adjacency_host()
    deg = g.degree.cpu().numpy()
    for k, m in enumerate(ms):
        s = DeviceGraph([m.points], [m.tris])
        srp, sci, sw = s.adjacency_host()
        o0, o1 = g.mesh_off_host[k], g.mesh_off_host[k + 1]
        assert np.array_equal(rp[o0:o1 + 1] - rp[o0], srp)
        assert np.array_equal(ci[rp[o0]:rp[o1]] - o0, sci)
        assert np.array_equal(w[rp[o0]:rp[o1]], sw)
        assert np.array_equal(deg[o0:o1], s.degree.cpu().numpy())
        assert np.array_equal(g.mesh_info_host[k], s.mesh_info_host[0])


def test_bad_triangle_index_raises(torch):
    from pyfocusr_b200._device import DeviceGraph
    from pyfocusr_b200._lib import FocusrB200Error

    pts = np.random.RandomState(0).rand(10, 3)
    with pytest.raises(FocusrB200Error):
        DeviceGraph([pts], [np.array([[0, 1, 12]], dtype=np.int32)])


# ------------------------------------------------------------------------------------------- K5
def test_mean_filter_bit_exact(torch, shipped_meshes, synth, golden):
    from oracle import port
    from pyfocusr_b200 import Graph

    for name in ("target_mesh", "source_mesh_15k", "ell20a"):
        m = all_meshes(shipped_meshes, synth)[name]
        g = Graph(m, n_rand_samples=100)
        a = port.adjacency(m.points, m.tris)
        for it in (1, 7, 40):
            assert np.array_equal(g.mean_filter_graph(m.points, it), port.mean_filter(a, m.points, it)), (name, it)
        assert np.array_equal(g.mean_filter_graph(m.points[:, 0], 5), port.mean_filter(a, m.points[:, 0], 5))
        assert np.array_equal(g.mean_filter_graph(m.points, 0), m.points)
    # 300 iterations on the 15k target = the golden smoothed target coordinates
    m = shipped_meshes["target_mesh_15k"]
    out = Graph(m, n_rand_samples=100).mean_filter_graph(m.points, 300)
    assert sha(out) == str(golden["15k_smoothed_target_sha"])


def test_laplacian_apply(torch, shipped_meshes):
    from oracle import port
    from pyfocusr_b200._device import DeviceGraph

    m = shipped_meshes["source_mesh_15k"]
    g = DeviceGraph([m.points], [m.tris])
    lap = port.laplacian(port.adjacency(m.points, m.tris))
    for b in (8, 16, 24, 48, 96):
        x = np.random.RandomState(b).standard_normal((m.points.shape[0], b))
        y = g.laplacian_apply(torch.from_numpy(x).cuda()).cpu().numpy()
        ref = lap @ x
        assert np.max(np.abs(y - ref)) <= 1e-13 * np.max(np.abs(ref)) * 8, b


# ------------------------------------------------------------------------------------------- K2
def check_eigs(vals, vecs, mesh, n, tol_val=1e-6, tol_vec=1e-5):
    from oracle import port

    lap = port.laplacian(port.adjacency(mesh.points, mesh.tris))
    rv, rvec = port.recursive_eig(lap, n + 1, n, 1)
    o = np.argsort(rv)
    rv, rvec = rv[o], rvec[:, o]
    assert vals.shape == rv.shape, (vals.shape, rv.shape)
    assert np.all(np.diff(vals) >= 0)
    assert np.max(np.abs(vals - rv) / rv) <= tol_val
    assert np.allclose(np.linalg.norm(vecs, axis=0), 1.0, atol=1e-12)
    # residual of every returned pair against the oracle's own Laplacian
    r = lap @ vecs - vecs * vals[None, :]
    assert np.max(np.linalg.norm(r, axis=0)) <= 1e-9
    # eigenvectors up to sign; near-degenerate neighbours (relative gap < 1e-6) compared as a subspace
    i = 0
    while i < rv.size:
        j = i + 1
        while j < rv.size and (rv[j] - rv[j - 1]) <= 1e-6 * rv[j]:
            j += 1
        q = rvec[:, i:j] / np.linalg.norm(rvec[:, i:j], axis=0)
        if j - i == 1:
            s = np.sign(q[:, 0] @ vecs[:, i])
            assert np.linalg.norm(vecs[:, i] * s - q[:, 0]) <= tol_vec, (i, np.linalg.norm(vecs[:, i] * s - q[:, 0]))
        else:
            qq, _ = np.linalg.qr(q)
            proj = vecs[:, i:j] - qq @ (qq.T @ vecs[:, i:j])
            assert np.max(np.linalg.norm(proj, axis=0)) <= tol_vec, (i, j)
        i = j
    return rv


def test_eigs_shipped_pairs(torch, shipped_meshes, golden):
    """configs[0] (15k pair: non-symmetric adjacency, source retries to k=14 -> 11 pairs) and the 5k pair."""
    from pyfocusr_b200._device import DeviceGraph

    for tag, names in (("5k", ("target_mesh", "source_mesh")), ("15k", ("target_mesh_15k", "source_mesh_15k"))):
        ms = [shipped_meshes[n] for n in names]
        g = DeviceGraph([m.points for m in ms], [m.tris for m in ms])
        vals, vecs, info = g.eigs_smallest(k=7, n_k_needed=6, k_buffer=1)
        vals, vecs = vals.cpu().numpy(), vecs.cpu().numpy()
        assert info["status"].tolist() == [0, 0]
        for k, (m, side) in enumerate(zip(ms, "ts")):
            gold = np.sort(golden["%s_%s_eig_vals" % (tag, side)])
            nf = int(info["n_found"][k])
            assert nf == gold.size, (tag, side, nf, gold.size)
            o0, o1 = g.mesh_off_host[k], g.mesh_off_host[k + 1]
            assert np.max(np.abs(vals[k, :nf] - gold) / gold) <= 1e-6
            check_eigs(vals[k, :nf], vecs[o0:o1, :nf], m, 6)
        if tag == "15k":
            assert info["k_final"].tolist() == [7, 14] and info["symmetric"].tolist() == [0, 0]
        else:
            assert info["symmetric"].tolist() == [1, 1]


def test_eigs_config2_n13(torch, shipped_meshes, golden):
    from pyfocusr_b200._device import DeviceGraph

    m = shipped_meshes["target_mesh"]
    g = DeviceGraph([m.points], [m.tris])
    vals, vecs, info = g.eigs_smallest(k=14, n_k_needed=13)
    nf = int(info["n_found"][0])
    assert nf == 13
    gold = np.sort(golden["5k_n13_t_eig_vals"])
    assert np.max(np.abs(vals[0, :nf].cpu().numpy() - gold) / gold) <= 1e-6
    check_eigs(vals[0, :nf].cpu().numpy(), vecs[:, :nf].cpu().numpy(), m, 13)


def test_eigs_synthetic_and_batch_consistency(torch, synth):
    from pyfocusr_b200._device import DeviceGraph

    ms = [synth["ell20a"], synth["ell20b"], synth["ell39"]]
    g = DeviceGraph([m.points for m in ms], [m.tris for m in ms])
    vals, vecs, info = g.eigs_smallest(k=7, n_k_needed=6)
    assert info["status"].tolist() == [0, 0, 0] and info["n_found"].tolist() == [6, 6, 6]
    vals, vecs = vals.cpu().numpy(), vecs.cpu().numpy()
    for k, m in enumerate(ms):
        o0, o1 = g.mesh_off_host[k], g.mesh_off_host[k + 1]
        check_eigs(vals[k, :6], vecs[o0:o1, :6], m, 6)
    # a mesh solved alone gives the same answer as inside a batch (deterministic kernels)
    s = DeviceGraph([ms[1].points], [ms[1].tris])
    sv, svec, _ = s.eigs_smallest(k=7, n_k_needed=6)
    assert np.allclose(sv[0, :6].cpu().numpy(), vals[1, :6], rtol=1e-9, atol=0)


@pytest.mark.parametrize("block", [16, 24, 32, 48])
def test_eigs_mixed_precision_passes(torch, shipped_meshes, synth, block):
    """By default the filter passes iterate in fp32 (k_filter_sell on the sliced-ELL fp32 copy of the matrix: plain fp32
    blocks, then the correction form driven by the fp64 residual; float4 slices, 2 or 4 threads per row);
    options.mixed_precision = 0 keeps fp64 throughout.  Both meet the fp64 tolerance and the oracle; the fp32 passes cost
    no extra filter degree.  The eigenvectors do not change with the filter options.  This batch is small enough that
    the filter steps run one pass per CTA, a form that ignores filter_policy, so the loop below varies only the prefetch
    and the resident-CTA build; test_gpu_kernels.py checks every cache policy on the 256-row form step by step."""
    from pyfocusr_b200._device import DeviceGraph

    ms = [shipped_meshes["target_mesh"], synth["ell20a"], synth["ell39"]]
    g = DeviceGraph([m.points for m in ms], [m.tris for m in ms])
    out = {}
    for mixed in (1, 0):
        vals, vecs, info = g.eigs_smallest(k=7, n_k_needed=6, block_size=block, options=dict(mixed_precision=mixed))
        out[mixed] = (vals.cpu().numpy(), vecs.cpu().numpy(), info)
    (v1, x1, i1), (v0, x0, i0) = out[1], out[0]
    for opt in (dict(filter_policy=0, filter_prefetch=0), dict(filter_policy=3), dict(filter_min_blocks=6)):
        _, xv, iv = g.eigs_smallest(k=7, n_k_needed=6, block_size=block, options=opt)
        assert np.array_equal(xv.cpu().numpy(), x1), opt
        assert np.array_equal(iv["filter_degree"], i1["filter_degree"])
    assert i1["status"].tolist() == [0, 0, 0] and i0["status"].tolist() == [0, 0, 0]
    assert np.all(i0["fp32_filter_degree"] == 0)
    assert np.all(i1["fp32_filter_degree"] > 10) and np.all(i1["fp32_filter_degree"] <= 10 + i1["filter_degree"])
    assert i1["filter_degree"].max() <= 1.15 * i0["filter_degree"].max()
    assert i1["outer_iterations"].max() <= i0["outer_iterations"].max() + 1
    assert i1["max_residual"].max() <= 1e-10 and i0["max_residual"].max() <= 1e-10
    assert np.max(np.abs(v1[:, :6] - v0[:, :6]) / v0[:, :6]) <= 1e-9
    for k, m in enumerate(ms):
        o0, o1 = g.mesh_off_host[k], g.mesh_off_host[k + 1]
        check_eigs(v1[k, :6], x1[o0:o1, :6], m, 6)
    # bit-reproducible
    _, x1b, _ = g.eigs_smallest(k=7, n_k_needed=6, block_size=block)
    assert sha(x1b.cpu().numpy()) == sha(x1)


def test_eigs_nonsymmetric_fp32_passes_and_device_rayleigh_ritz(torch, shipped_meshes):
    """The reference's own open meshes (structurally non-symmetric adjacency) as one batch: the fp32 filter forms against
    options.mixed_precision = 0, and the device form of the general b x b Rayleigh-Ritz step (k_rr_nonsym) against the
    host form (options.nonsym_device = 0): same retry contract, same eigenvalues, same parity with scipy."""
    from pyfocusr_b200._device import DeviceGraph

    ms = [shipped_meshes["target_mesh_15k"], shipped_meshes["source_mesh_15k"]]
    g = DeviceGraph([m.points for m in ms], [m.tris for m in ms])
    assert np.all(g.mesh_info_host[:, 1] > 0)                       # one-way entries: the non-symmetric path
    runs = {}
    for tag, opt in (("default", None), ("fp64", dict(mixed_precision=0)), ("host_rr", dict(nonsym_device=0))):
        vals, vecs, info = g.eigs_smallest(k=7, n_k_needed=6, options=opt)
        runs[tag] = (vals.cpu().numpy(), vecs.cpu().numpy(), info)
        assert info["status"].tolist() == [0, 0] and info["max_residual"].max() <= 1e-10
        assert info["k_final"].tolist() == [7, 14] and info["n_found"].tolist() == [6, 11]
    v, x, i = runs["default"]
    assert np.all(i["fp32_filter_degree"] == i["filter_degree"]) and np.all(runs["fp64"][2]["fp32_filter_degree"] == 0)
    assert i["filter_degree"].max() <= 1.1 * runs["fp64"][2]["filter_degree"].max()
    for tag in ("fp64", "host_rr"):
        for k, n in enumerate((6, 11)):
            assert np.max(np.abs(v[k, :n] - runs[tag][0][k, :n]) / runs[tag][0][k, :n]) <= 1e-8, tag
    for k, (m, n) in enumerate(zip(ms, (6, 11))):
        o0, o1 = g.mesh_off_host[k], g.mesh_off_host[k + 1]
        check_eigs(v[k, :n], x[o0:o1, :n], m, 6)


def test_eigs_icosphere_multiplets(torch, synth):
    """Exact 3/5/7-fold multiplets (SURVEY.md section 7.3-3): k=11 cuts the l=3 multiplet."""
    from oracle import port
    from pyfocusr_b200._device import DeviceGraph

    m = synth["ico20"]
    g = DeviceGraph([m.points], [m.tris])
    vals, vecs, info = g.eigs_smallest(k=11, n_k_needed=10)
    assert info["status"][0] == 0 and info["n_found"][0] == 10
    vals, vecs = vals[0, :10].cpu().numpy(), vecs[:, :10].cpu().numpy()
    lap = port.laplacian(port.adjacency(m.points, m.tris))
    rv, _ = port.recursive_eig(lap, 11, 10, 1)
    assert np.max(np.abs(vals - np.sort(rv)) / np.sort(rv)) <= 1e-6
    assert np.max(np.linalg.norm(lap @ vecs - vecs * vals[None], axis=0)) <= 1e-9


def test_eigs_damaged_meshes_nonsymmetric_batch(torch, synth):
    """Holes and flipped triangles (one-way adjacency entries -> complex eigenvalue pairs of L) in a batch that
    also holds a clean mesh: every mesh must still return the reference's pairs (SURVEY.md section 7.3-1)."""
    import pyfocusr_b200.mesh as fmesh
    from pyfocusr_b200._device import DeviceGraph

    rng = np.random.RandomState(1)
    ms = [synth["ell20a"]]
    for nu, holes, flips in ((16, 12, 0), (20, 4, 25), (24, 30, 30)):
        base = fmesh.perturbed_ellipsoid(nu, 5)
        t = base.tris.copy()
        keep = np.ones(len(t), bool)
        keep[rng.choice(len(t), holes, replace=False)] = False
        t = t[keep]
        fl = rng.choice(len(t), flips, replace=False)
        t[fl] = t[fl][:, [0, 2, 1]]
        ms.append(fmesh.PolyData(base.points, t))
    g = DeviceGraph([m.points for m in ms], [m.tris for m in ms])
    vals, vecs, info = g.eigs_smallest(k=7, n_k_needed=6)
    assert info["status"].tolist() == [0] * 4
    assert info["symmetric"].tolist() == [1, 0, 0, 0]
    vals, vecs = vals.cpu().numpy(), vecs.cpu().numpy()
    for k, m in enumerate(ms):
        nf = int(info["n_found"][k])
        o0, o1 = g.mesh_off_host[k], g.mesh_off_host[k + 1]
        check_eigs(vals[k, :nf], vecs[o0:o1, :nf], m, 6)


def test_recursive_eig_function(torch, shipped_meshes, golden):
    from oracle import port
    from pyfocusr_b200 import recursive_eig

    m = shipped_meshes["target_mesh"]
    lap = port.laplacian(port.adjacency(m.points, m.tris))
    vals, vecs = recursive_eig(lap, k=7, n_k_needed=6, k_buffer=1)
    gold = np.sort(golden["5k_t_eig_vals"])
    assert vals.shape == gold.shape and np.max(np.abs(vals - gold) / gold) <= 1e-6
    assert np.max(np.linalg.norm(lap @ vecs - vecs * vals[None], axis=0)) <= 1e-9


# ------------------------------------------------------------------------------------------- B2, C1-C5, D1
def test_graph_dropin_attributes(torch, shipped_meshes, golden):
    from oracle import port
    from pyfocusr_b200 import Graph

    m = shipped_meshes["target_mesh"]
    np.random.seed(0)
    g = Graph(m, n_spectral_features=6, n_rand_samples=5000, list_features_to_calc=[], feature_weights=np.eye(2))
    assert np.array_equal(g.rand_idxs, golden["5k_t_rand_idxs"])  # same RNG consumption as the reference
    g.get_graph_spectrum()
    assert sparse.issparse(g.adjacency_matrix) and g.laplacian_matrix.shape == (5000, 5000)
    assert np.array_equal(g.normed_points, port.normed_points(m.points))
    assert g.eig_vecs.shape == (5000, 6) and g.eig_vecs.flags.writeable
    assert np.allclose(np.ptp(g.eig_vecs, axis=0), 1.0, atol=1e-15)       # notebook cell 15
    assert np.allclose(np.min(g.eig_vecs, axis=0), -0.5, atol=1e-15)
    gold = np.sort(golden["5k_t_eig_vals"])
    assert np.max(np.abs(g.eig_vals - gold) / gold) <= 1e-6
    # normalised eigenvectors == reference's up to sign (flip <-> v -> -v exactly)
    ref = golden["5k_t_eig_vecs_raw_normed"]
    ro = np.argsort(golden["5k_t_eig_vals"])
    for j in range(6):
        a, b = g.eig_vecs[:, j], ref[:, ro[j]]
        assert min(np.max(np.abs(a - b)), np.max(np.abs(a + b))) <= 1e-5
    g.get_eig_val_gap()
    assert g.eig_val_gap == np.mean(np.diff(g.eig_vals))


def _reference_pair_vectors(golden, tag):
    vt = golden[tag + "_t_eig_vecs_raw_normed"].copy()
    vs = golden[tag + "_s_eig_vecs_raw_normed"].copy()
    return vt, vs


def test_eigsort_costs_and_moves_on_reference_vectors(torch, shipped_meshes, golden):
    """Feed the reference's own (pre-sort) eigenvectors: cost matrices, decisions and the permuted
    source eigenvectors must equal what the unmodified reference produced."""
    from pyfocusr_b200._device import DeviceGraph, eigsort_costs
    from pyfocusr_b200.eigsort import c_lambda_matrix, decide_matches, moves_from_matches

    for tag, names, n in (("5k", ("target_mesh", "source_mesh"), 6), ("15k", ("target_mesh_15k", "source_mesh_15k"), 6),
                          ("5k_n13", ("target_mesh", "source_mesh"), 13)):
        mt, ms = shipped_meshes[names[0]], shipped_meshes[names[1]]
        vt, vs = _reference_pair_vectors(golden, tag)
        g = DeviceGraph([mt.points, ms.points], [mt.tris, ms.tris])
        ld = max(vt.shape[1], vs.shape[1])
        host = np.zeros((g.n_points, ld))
        host[: mt.points.shape[0], : vt.shape[1]] = vt
        host[mt.points.shape[0]:, : vs.shape[1]] = vs
        vecs = torch.from_numpy(host).cuda()
        it, is_ = golden[tag + "_t_rand_idxs"][None], golden[tag + "_s_rand_idxs"][None]
        ch, chf, cs, csf, nn = eigsort_costs(g, vecs, [0], [1], it, is_, n)
        for got, name in ((ch, "c_hist"), (chf, "c_hist_f"), (cs, "c_spatial"), (csf, "c_spatial_f")):
            ref = golden["%s_%s" % (tag, name)]
            assert np.max(np.abs(got[0].cpu().numpy() - ref) / np.abs(ref)) <= 1e-10, (tag, name)
        cl = c_lambda_matrix(golden[tag + "_t_eig_vals"], golden[tag + "_s_eig_vals"], n)
        assert np.array_equal(cl, golden[tag + "_c_lambda"])
        q, tm, sm, flipped = decide_matches(cl, ch[0].cpu().numpy(), chf[0].cpu().numpy(), cs[0].cpu().numpy(),
                                            csf[0].cpu().numpy(), True)
        assert np.array_equal(tm, golden[tag + "_target_matches"]) and np.array_equal(sm, golden[tag + "_source_matches"])
        assert np.array_equal(np.asarray(flipped, dtype=np.int64).reshape(-1, 2), golden[tag + "_flipped_pairs"])
        assert np.max(np.abs(q - golden[tag + "_Q"]) / golden[tag + "_Q"]) <= 1e-10
        d, s, sg = moves_from_matches(tm, sm, flipped, True)
        ident = np.arange(n, dtype=np.int32)
        g.flip_permute(vecs, np.stack([ident, d]), np.stack([ident, s]), np.stack([np.ones(n, np.int32), sg]))
        out = vecs.cpu().numpy()
        assert np.array_equal(out[: mt.points.shape[0], : vt.shape[1]], vt)            # target untouched
        assert sha(np.ascontiguousarray(out[mt.points.shape[0]:, : vs.shape[1]])) == str(golden[tag + "_sorted_vecs_s_sha"])


def _reference_coords(golden, tag, n_spec):
    """Spectral coordinates exactly as the reference computed them (from golden vectors/decisions)."""
    from oracle import port

    vt, vs = _reference_pair_vectors(golden, tag)
    flipped = [tuple(r) for r in golden[tag + "_flipped_pairs"].tolist()]
    port.eigen_sort_apply(vt, vs, golden[tag + "_target_matches"], golden[tag + "_source_matches"], flipped, True)
    w = golden[tag + "_spectral_weights"]
    return port.spectral_coords(vt, w, n_spec), port.spectral_coords(vs, w, n_spec), vt, vs, w


# ------------------------------------------------------------------------------------------- K4, E1-E4
def test_knn_on_reference_features_bit_exact(torch, shipped_meshes, golden):
    from oracle import port
    from pyfocusr_b200 import _device

    for tag, names, n_spec in (("5k", ("target_mesh", "source_mesh"), 3), ("15k", ("target_mesh_15k", "source_mesh_15k"), 3),
                               ("5k_n13", ("target_mesh", "source_mesh"), 10)):
        tc, sc, vt, vs, w = _reference_coords(golden, tag, n_spec)
        idx, dist = _device.knn(torch.from_numpy(tc).cuda(), torch.from_numpy(sc).cuda(), k=1)
        assert np.array_equal(idx[:, 0].cpu().numpy(), golden[tag + "_initial_idx"].astype(np.int64)), tag
        # device spectral-coordinate kernel == numpy broadcast multiply (bitwise)
        mt, ms = shipped_meshes[names[0]], shipped_meshes[names[1]]
        g = _device.DeviceGraph([mt.points, ms.points], [mt.tris, ms.tris])
        ld = max(vt.shape[1], vs.shape[1])
        host = np.zeros((g.n_points, ld))
        host[: vt.shape[0], : vt.shape[1]] = vt
        host[vt.shape[0]:, : vs.shape[1]] = vs
        coords = g.spectral_coords(torch.from_numpy(host).cuda(), np.stack([w, w]), n_spec).cpu().numpy()
        assert np.array_equal(coords[: vt.shape[0]], tc) and np.array_equal(coords[vt.shape[0]:], sc)
        # smoothing + second KNN + k=3 + weighted positions, all against golden / oracle
        a_t, a_s = port.adjacency(mt.points, mt.tris), port.adjacency(ms.points, ms.tris)
        sm_t = port.mean_filter(a_t, mt.points, 300)
        proj = port.mean_filter(a_s, sm_t[golden[tag + "_initial_idx"]], 40)
        assert sha(proj) == str(golden[tag + "_source_projected_sha"])
        refs, qs = torch.from_numpy(sm_t).cuda(), torch.from_numpy(proj).cuda()
        idx1, _ = _device.knn(refs, qs, k=1)
        assert np.array_equal(idx1[:, 0].cpu().numpy(), golden[tag + "_final_idx"].astype(np.int64)), tag
        idx3, dist3 = _device.knn(refs, qs, k=3)
        assert np.array_equal(idx3.cpu().numpy(), golden[tag + "_knn3_idx"].astype(np.int64)), tag
        wavg_ref, d3_ref, _ = port.weighted_final_positions(sm_t, proj, mt.points)
        assert np.array_equal(dist3.cpu().numpy(), d3_ref), tag
        wavg = _device.weighted_positions(idx3, dist3, torch.from_numpy(mt.points).cuda()).cpu().numpy()
        assert np.array_equal(wavg, wavg_ref) and sha(wavg) == str(golden[tag + "_weighted_avg_sha"]), tag


def test_knn_generic_dims_ties_and_segments(torch):
    from oracle import port
    from pyfocusr_b200 import _device

    rng = np.random.RandomState(1)
    for dim, k in ((1, 1), (2, 3), (3, 3), (5, 2), (10, 1), (13, 3), (16, 8), (32, 1)):
        refs, qs = rng.standard_normal((1500, dim)), rng.standard_normal((700, dim))
        d_ref, i_ref = port.knn_bruteforce(refs, qs, k)
        idx, dist = _device.knn(torch.from_numpy(refs).cuda(), torch.from_numpy(qs).cuda(), k=k)
        assert np.array_equal(idx.cpu().numpy(), i_ref), (dim, k)
        assert np.array_equal(dist.cpu().numpy(), d_ref), (dim, k)
    # exact ties: duplicated reference rows -> the lower index wins; coincident query -> distance 0
    refs = rng.standard_normal((300, 3))
    refs[200:] = refs[:100]
    qs = np.concatenate([refs[:50], rng.standard_normal((50, 3))])
    idx, dist = _device.knn(torch.from_numpy(refs).cuda(), torch.from_numpy(qs).cuda(), k=3)
    idx, dist = idx.cpu().numpy(), dist.cpu().numpy()
    assert np.array_equal(idx[:50, 0], np.arange(50)) and np.array_equal(idx[:50, 1], np.arange(200, 250))
    assert np.all(dist[:50, :2] == 0)
    d_ref, i_ref = port.knn_bruteforce(refs, qs, 3)
    assert np.array_equal(idx, i_ref)
    tp = rng.standard_normal((300, 3))
    wavg = _device.weighted_positions(torch.from_numpy(idx).cuda(), torch.from_numpy(dist).cuda(),
                                      torch.from_numpy(tp).cuda()).cpu().numpy()
    assert np.array_equal(wavg[:50], tp[:50])  # focusr.py:415-419: coincident -> copy that target point
    # ragged segments (one of them a single reference)
    r_sizes, q_sizes = [1, 517, 40], [33, 1, 300]
    refs, qs = rng.standard_normal((sum(r_sizes), 4)), rng.standard_normal((sum(q_sizes), 4))
    ro = torch.tensor(np.concatenate([[0], np.cumsum(r_sizes)]), dtype=torch.int32).cuda()
    qo = torch.tensor(np.concatenate([[0], np.cumsum(q_sizes)]), dtype=torch.int32).cuda()
    idx, dist = _device.knn(torch.from_numpy(refs).cuda(), torch.from_numpy(qs).cuda(), k=1, ref_off=ro, query_off=qo,
                            max_queries=max(q_sizes))
    r0 = q0 = 0
    for rs, qsz in zip(r_sizes, q_sizes):
        d_ref, i_ref = port.knn_bruteforce(refs[r0:r0 + rs], qs[q0:q0 + qsz], 1)
        assert np.array_equal(idx[q0:q0 + qsz].cpu().numpy(), i_ref)
        r0 += rs
        q0 += qsz


# ------------------------------------------------------------------------------------------- whole path
def test_focusr_dropin_15k_pair(torch, shipped_meshes, golden):
    """configs[0] through the reference-facing API (ICP/CPD are outside the path: off / identity)."""
    import pyfocusr_b200 as pyfocusr

    np.random.seed(0)
    mt, ms = shipped_meshes["target_mesh_15k"], shipped_meshes["source_mesh_15k"]

    class Seeded(pyfocusr.Focusr):
        pass

    # the reference draws rand_idxs from the global RNG inside each Graph(); reproduce the golden seeds
    orig = pyfocusr.graph.Graph.get_list_rand_idxs
    seeds = iter([0, 1])

    def seeded(self, n, replace=False, force_randomization=False):
        np.random.seed(next(seeds))
        return orig(self, n, replace, force_randomization)

    pyfocusr.graph.Graph.get_list_rand_idxs = seeded
    try:
        f = pyfocusr.Focusr(mt, ms, icp_register_first=False, list_features_to_calc=[], feature_weights=np.eye(2),
                            registration="identity")
    finally:
        pyfocusr.graph.Graph.get_list_rand_idxs = orig
    assert np.array_equal(f.graph_target.rand_idxs, golden["15k_t_rand_idxs"])
    assert f.graph_target.eig_vals.size == 6 and f.graph_source.eig_vals.size == 11
    # eigsort's costs depend on the (arbitrary) sign of the target eigenvectors, so the stages after
    # the solver are checked against the oracle run on OUR pre-sort eigenvectors
    from oracle import port
    vt0, vs0 = f.graph_target.eig_vecs.copy(), f.graph_source.eig_vecs.copy()
    f.align_maps()
    srt = port.sort_eigenmaps(mt.points, ms.points, f.graph_target.rand_idxs, f.graph_source.rand_idxs,
                              f.graph_target.eig_vals, f.graph_source.eig_vals, vt0, vs0, 6, True)
    assert np.max(np.abs(f.Q - srt["Q"]) / srt["Q"]) <= 1e-9
    assert np.array_equal(f.graph_source.eig_vecs, vs0) and np.array_equal(f.graph_target.eig_vecs, vt0)
    w = port.spectral_weights(srt["Q"], f.graph_source.eig_vals, f.graph_target.eig_vals, 3)
    assert np.max(np.abs(f.spectral_weights - w)) <= 1e-9
    cs = port.correspondence_stage(dict(A=port.adjacency(mt.points, mt.tris)), dict(A=port.adjacency(ms.points, ms.tris)),
                                   mt.points, ms.points, f.target_spectral_coords, f.source_spectral_coords)
    assert np.array_equal(f.corresponding_target_idx_for_each_source_pt, cs["final_idx"])
    assert np.array_equal(f.smoothed_target_coords, cs["smoothed_target_coords"])
    assert np.array_equal(f.source_projected_on_target, cs["source_projected_on_target"])
    assert np.array_equal(f.weighted_avg_transformed_points, cs["weighted_avg_transformed_points"])
    idx = f.corresponding_target_idx_for_each_source_pt
    assert idx.dtype == np.int64 and idx.shape == (ms.points.shape[0],)
    # (no comparison with the golden run's indices: eigsort's costs -- hence the spectral weights and the
    # correspondences -- depend on the sign ARPACK happens to give the target eigenvectors, so two runs of
    # the reference itself agree on only about half of the points)
    assert f.weighted_avg_transformed_points.shape == ms.points.shape
    assert np.array_equal(f.nearest_neighbor_transformed_points, mt.points[idx])
    assert f.weighted_avg_transformed_mesh.points.shape == ms.points.shape


def test_batch_equals_oracle_and_single(torch, synth):
    from oracle import port
    from pyfocusr_b200 import SpectralBatch

    t = [synth["ell20a"], synth["ico20"]]
    s = [synth["ell20b"], synth["ell20a"]]
    sb = SpectralBatch(n_coords_spectral_ordering=2000, graph_smoothing_iterations=30, projection_smooth_iterations=10)
    out = sb.run_meshes(t, s, record_events=True, keep_presort=True)
    assert set(sb.timings) >= {"laplacian", "eigensolve", "eigsort", "smoothing", "knn_final"}
    pre, post = out["eig_vecs_presort"].cpu().numpy(), out["eig_vecs"].cpu().numpy()
    vals, nf, off = out["eig_vals"].cpu().numpy(), out["eigs_info"]["n_found"], out["graph"].mesh_off_host
    n_s = [m.points.shape[0] for m in s]
    fin = out["final_idx"].cpu().numpy()
    wavg = out["weighted_avg_transformed_points"].cpu().numpy()
    from parity_checks import check_pair_against_oracle

    for p in range(2):
        # stages after the solver against the oracle: indices EQUAL (tests/parity_checks.py has the chain of custody)
        check_pair_against_oracle(port, out, p, 2, t[p].points, t[p].tris, s[p].points, s[p].tris, 6, 3, 30, 10)
    single = SpectralBatch(n_coords_spectral_ordering=2000, graph_smoothing_iterations=30, projection_smooth_iterations=10)
    o1 = single.run_meshes(t[:1], s[:1], idx_t=out["idx_t"][:1], idx_s=out["idx_s"][:1])
    assert np.array_equal(o1["final_idx"].cpu().numpy(), fin[: n_s[0]])
    assert np.array_equal(o1["weighted_avg_transformed_points"].cpu().numpy(), wavg[: n_s[0]])


def test_concurrent_sub_batches_equal_separate_runs(torch, synth, shipped_meshes):
    """SpectralBatch.run_concurrent (one host thread + CUDA stream per sub-batch, target smoothing on a side stream
    each) returns exactly what `run` returns for every sub-batch on its own."""
    from pyfocusr_b200 import SpectralBatch

    kw = dict(n_coords_spectral_ordering=2000, graph_smoothing_iterations=30, projection_smooth_iterations=10)
    subs = [([synth["ell20a"], synth["ico20"]], [synth["ell20b"], synth["ell20a"]]),
            ([synth["ell39"]], [synth["ell39"]]),
            ([shipped_meshes["target_mesh"]], [shipped_meshes["source_mesh"]])]
    sb = SpectralBatch(**kw)
    packed = [sb.pack_meshes(t, s) for t, s in subs]
    rng = np.random.RandomState(5)
    jobs = []
    for pts, tris, off, P in packed:
        sizes = np.diff(off)
        jobs.append(dict(points=pts, tris=tris, mesh_off_host=off, n_pairs=P, idx_t=sb.sample_indices(sizes[:P], rng),
                         idx_s=sb.sample_indices(sizes[P:], rng)))
    keys = ("final_idx", "weighted_avg_transformed_points", "eig_vecs", "smoothed_target_coords", "knn3_dist")
    for rep in range(2):  # second round: worker threads, streams and pinned pools are reused
        outs = sb.run_concurrent(jobs)
        torch.cuda.synchronize()
        assert len(outs) == 3
        for job, out in zip(jobs, outs):
            ref = SpectralBatch(**kw)
            ref.overlap_smoothing = False
            alone = ref.run(**job)
            for k in keys:
                assert torch.equal(out[k], alone[k]), (rep, k)


def test_knn_pruned_is_bit_identical_to_brute_force(torch, shipped_meshes, synth):
    """Morton-tile pruning must change nothing: indices AND distances equal the brute-force kernel's
    (and the oracle's) on surfaces, clustered points with duplicates, and higher dimensions."""
    from oracle import port
    from pyfocusr_b200 import _device

    rng = np.random.RandomState(7)
    mt, ms = shipped_meshes["target_mesh_15k"], shipped_meshes["source_mesh_15k"]
    cases = [(mt.points, ms.points, 3), (synth["ell39"].points, synth["ell39"].points + 0.01, 1)]
    cl = rng.standard_normal((40, 3))[rng.randint(0, 40, 6000)] + 0.01 * rng.standard_normal((6000, 3))
    cl[3000:3100] = cl[:100]                                   # exact duplicates -> ties
    cases.append((cl, np.concatenate([cl[:2000], rng.standard_normal((1500, 3))]), 3))
    cases.append((rng.standard_normal((5000, 10)) * np.logspace(0, -2, 10), rng.standard_normal((4000, 10)) * np.logspace(0, -2, 10), 3))
    cases.append((rng.standard_normal((3000, 13)), rng.standard_normal((900, 13)), 8))
    for refs, qs, k in cases:
        r, q = torch.from_numpy(np.ascontiguousarray(refs)).cuda(), torch.from_numpy(np.ascontiguousarray(qs)).cuda()
        i_p, d_p = _device.knn(r, q, k=k)
        i_b, d_b = _device.knn(r, q, k=k, brute_force=True)
        assert torch.equal(i_p, i_b) and torch.equal(d_p, d_b), (refs.shape, k)
    d_ref, i_ref = port.knn_bruteforce(cases[2][0], cases[2][1], 3)
    i_p, d_p = _device.knn(torch.from_numpy(cases[2][0]).cuda(), torch.from_numpy(cases[2][1]).cuda(), k=3)
    assert np.array_equal(i_p.cpu().numpy(), i_ref) and np.array_equal(d_p.cpu().numpy(), d_ref)
    # ragged batched segments through the pruned path
    sizes_r, sizes_q = [700, 5000, 1200], [900, 600, 5000]
    refs, qs = rng.standard_normal((sum(sizes_r), 3)), rng.standard_normal((sum(sizes_q), 3))
    ro = torch.tensor(np.concatenate([[0], np.cumsum(sizes_r)]), dtype=torch.int32).cuda()
    qo = torch.tensor(np.concatenate([[0], np.cumsum(sizes_q)]), dtype=torch.int32).cuda()
    a = _device.knn(torch.from_numpy(refs).cuda(), torch.from_numpy(qs).cuda(), k=3, ref_off=ro, query_off=qo, max_queries=5000, max_refs=5000)
    b = _device.knn(torch.from_numpy(refs).cuda(), torch.from_numpy(qs).cuda(), k=3, ref_off=ro, query_off=qo, max_queries=5000, max_refs=5000, brute_force=True)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_focusr_dropin_variants_5k(torch, shipped_meshes):
    """API variants of the drop-in on the 5k pair, each checked against the oracle fed our pre-sort eigenvectors:
    source as the reference eigenmap, unweighted coordinates, xyz appended as features (d = 6), n_spectral_features=10,
    more ordering samples than vertices (arange path of graph.py:284-288)."""
    from oracle import port
    import pyfocusr_b200 as pyfocusr

    mt, ms = shipped_meshes["target_mesh"], shipped_meshes["source_mesh"]
    at, as_ = port.adjacency(mt.points, mt.tris), port.adjacency(ms.points, ms.tris)
    variants = [dict(target_eigenmap_as_reference=False), dict(get_weighted_spectral_coords=False),
                dict(include_points_as_features=True), dict(include_points_as_features=True, norm_physical_and_spectral=False),
                dict(n_spectral_features=10, n_extra_spectral=3), dict(n_coords_spectral_ordering=20000),
                dict(graph_smoothing_iterations=7, projection_smooth_iterations=0, smooth_correspondences=True)]
    for kw in variants:
        np.random.seed(3)
        f = pyfocusr.Focusr(mt, ms, icp_register_first=False, list_features_to_calc=[], registration="identity", **kw)
        n_spec = kw.get("n_spectral_features", 3)
        n = n_spec + 3
        tref = kw.get("target_eigenmap_as_reference", True)
        vt0, vs0 = f.graph_target.eig_vecs.copy(), f.graph_source.eig_vecs.copy()
        f.align_maps()
        srt = port.sort_eigenmaps(mt.points, ms.points, f.graph_target.rand_idxs, f.graph_source.rand_idxs,
                                  f.graph_target.eig_vals, f.graph_source.eig_vals, vt0, vs0, n, tref)
        assert np.max(np.abs(f.Q - srt["Q"]) / srt["Q"]) <= 1e-9, kw
        assert np.array_equal(f.graph_source.eig_vecs, vs0) and np.array_equal(f.graph_target.eig_vecs, vt0), kw
        assert f.target_spectral_coords.shape[1] == n_spec + (3 if kw.get("include_points_as_features") else 0)
        cs = port.correspondence_stage(dict(A=at), dict(A=as_), mt.points, ms.points, f.target_spectral_coords,
                                       f.source_spectral_coords, f.graph_smoothing_iterations, f.projection_smooth_iterations)
        assert np.array_equal(f.corresponding_target_idx_for_each_source_pt, cs["final_idx"]), kw
        assert np.array_equal(f.weighted_avg_transformed_points, cs["weighted_avg_transformed_points"]), kw
        if "n_coords_spectral_ordering" in kw:
            assert np.array_equal(f.graph_target.rand_idxs, np.arange(5000))


def test_mesh_scalar_features_in_adjacency_and_as_coordinates(torch, shipped_meshes, golden):
    """SURVEY.md section 8f-3: a mesh point scalar as extra node feature -- inside the edge weights
    (graph.py:166-175; K1 with point_dim = 4) and smoothed + appended to the spectral coordinates
    (focusr.py:218-269; K5 with one column)."""
    from oracle import port
    import pyfocusr_b200 as pyfocusr

    name = "thickness_change_(mm)"
    mt, ms = shipped_meshes["target_mesh"], shipped_meshes["source_mesh"]
    for side, m in (("t", mt), ("s", ms)):
        g = pyfocusr.Graph(m, n_spectral_features=6, n_rand_samples=100, list_features_to_get_from_mesh=[name],
                           include_features_in_adj_matrix=True)
        g.get_graph_spectrum()
        a = g.adjacency_matrix
        assert sha(a.data) + sha(a.indices) + sha(a.indptr) == str(golden["5k_feat_%s_A_sha" % side])
        gold = np.sort(golden["5k_feat_%s_eig_vals" % side])
        assert g.eig_vals.shape == gold.shape and np.max(np.abs(g.eig_vals - gold) / gold) <= 1e-6
    np.random.seed(11)
    f = pyfocusr.Focusr(mt, ms, icp_register_first=False, list_features_to_calc=[], list_features_to_get_from_mesh=[name],
                        include_features_in_adj_matrix=True, use_features_as_coords=True, registration="identity")
    vt0, vs0 = f.graph_target.eig_vecs.copy(), f.graph_source.eig_vecs.copy()
    f.align_maps()
    feats = [port.normalized_node_feature(m.point_scalars[name]) for m in (mt, ms)]
    at = port.adjacency(port.feature_augmented_points(mt.points, [feats[0]]), mt.tris)
    as_ = port.adjacency(port.feature_augmented_points(ms.points, [feats[1]]), ms.tris)
    srt = port.sort_eigenmaps(mt.points, ms.points, f.graph_target.rand_idxs, f.graph_source.rand_idxs,
                              f.graph_target.eig_vals, f.graph_source.eig_vals, vt0, vs0, 6, True)
    assert np.max(np.abs(f.Q - srt["Q"]) / srt["Q"]) <= 1e-9
    w = f.spectral_weights
    tc = port.features_as_coords(at, [feats[0]], port.spectral_coords(vt0, w, 3), 40)
    sc = port.features_as_coords(as_, [feats[1]], port.spectral_coords(vs0, w, 3), 40)
    assert f.target_spectral_coords.shape == (5000, 4)
    assert np.array_equal(f.target_spectral_coords, tc) and np.array_equal(f.source_spectral_coords, sc)
    cs = port.correspondence_stage(dict(A=at), dict(A=as_), mt.points, ms.points, tc, sc)
    assert np.array_equal(f.corresponding_target_idx_for_each_source_pt, cs["final_idx"])
    with pytest.raises(NotImplementedError):
        pyfocusr.Graph(mt, list_features_to_get_from_mesh=[name], include_features_in_G_matrix=True)


def test_error_behaviour_and_degenerate_inputs(torch):
    """Degenerate geometry the reference does not check (SURVEY.md section 9) is reported, not propagated."""
    from pyfocusr_b200 import _device
    from pyfocusr_b200._device import DeviceGraph
    from pyfocusr_b200._lib import FocusrB200Error
    from pyfocusr_b200.mesh import icosphere

    m = icosphere(6)
    pts = m.points.copy()
    pts[m.tris[0, 1]] = pts[m.tris[0, 0]]                      # zero-length edge -> 1/0 weight (graph.py:177-178)
    g = DeviceGraph([pts], [m.tris])
    assert g.mesh_info_host[0, 3] > 0
    with pytest.raises(FocusrB200Error, match="non-finite"):
        g.eigs_smallest(k=7, n_k_needed=6)
    tiny = icosphere(1)                                         # 12 vertices < block size
    with pytest.raises(FocusrB200Error, match="fewer vertices"):
        DeviceGraph([tiny.points], [tiny.tris]).eigs_smallest(k=7, n_k_needed=6)
    # a mesh without any triangle: every row has zero degree, the Laplacian is empty
    g0 = DeviceGraph([m.points], [np.zeros((0, 3), dtype=np.int32)])
    assert g0.nnz == 0 and g0.mesh_info_host[0].tolist() == [0, 0, m.points.shape[0], 0, 0, 0, 0, 0]
    assert g0.laplacian_host()[0][-1] == 0
    # more neighbours requested than references exist: missing slots are -1 / inf
    refs = torch.from_numpy(np.random.RandomState(0).rand(2, 3)).cuda()
    qs = torch.from_numpy(np.random.RandomState(1).rand(5, 3)).cuda()
    idx, dist = _device.knn(refs, qs, k=3)
    assert torch.all(idx[:, 2] == -1) and torch.all(torch.isinf(dist[:, 2])) and torch.all(idx[:, :2] >= 0)
    with pytest.raises(FocusrB200Error):
        _device.knn(refs, qs, k=9)


def test_device_lsap_equals_scipy(torch):
    """focusr_lsap (csrc/lsap.cu: scipy's shortest-augmenting-path algorithm in one thread-block cluster) against
    scipy.optimize.linear_sum_assignment: the same assignment, also on matrices full of ties (integer costs, duplicated
    points), rectangular both ways, tiny, and a 2500-point geometric instance with long augmenting paths."""
    from scipy.optimize import linear_sum_assignment
    from scipy.spatial.distance import cdist

    from pyfocusr_b200 import _device

    rng = np.random.RandomState(3)
    cases = []
    for n, m in ((1, 1), (2, 2), (9, 9), (40, 47), (47, 40), (300, 300), (257, 400), (1030, 1030)):
        cases.append(rng.rand(n, m))
        cases.append(rng.randint(0, 4, (n, m)).astype(np.float64))
    pts = rng.randint(0, 6, (600, 2)).astype(np.float64)              # duplicated points: many equal distances
    cases.append(cdist(pts[:500], pts))
    p = rng.randn(2500, 3)
    p /= np.linalg.norm(p, axis=1)[:, None]
    cases.append(cdist(p[rng.permutation(2500)] + 0.3 * rng.randn(2500, 3), p))
    for c in cases:
        row, col = _device.linear_sum_assignment(torch.from_numpy(np.ascontiguousarray(c)).cuda())
        r_ref, c_ref = linear_sum_assignment(c)
        assert np.array_equal(row, r_ref) and np.array_equal(col, c_ref), c.shape
    bad = np.ones((3, 3))
    bad[0, :] = np.inf
    with pytest.raises(ValueError):
        _device.linear_sum_assignment(torch.from_numpy(bad).cuda())


def test_hungarian_correspondence(torch, synth):
    """focusr.py:340-349: cdist on the GPU bit-equal to scipy's; the assignment (focusr_lsap on the GPU) equal to the scipy
    call the reference makes."""
    import pyfocusr_b200 as pyfocusr
    from scipy.optimize import linear_sum_assignment
    from scipy.spatial.distance import cdist

    from pyfocusr_b200 import _lib

    rng = np.random.RandomState(0)
    for na, nb, d in ((300, 300, 3), (257, 400, 6), (50, 31, 13)):
        a, b = rng.rand(na, d), rng.rand(nb, d)
        ad, bd = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        out = torch.empty((na, nb), dtype=torch.float64, device="cuda")
        _lib.call("focusr_cdist", _lib.ptr(ad), na, _lib.ptr(bd), nb, d, _lib.ptr(out), _lib.stream_ptr())
        ref = cdist(a, b)
        got = out.cpu().numpy()
        assert np.max(np.abs(got - ref)) <= 4e-16 * np.max(ref)          # same formula; scipy's build may contract an FMA
        assert np.array_equal(linear_sum_assignment(got)[1], linear_sum_assignment(ref)[1])
    t, s = synth["ell20a"], synth["ell20b"]
    np.random.seed(0)
    f = pyfocusr.Focusr(t, s, icp_register_first=False, list_features_to_calc=[], registration="identity",
                        initial_correspondence_type="hungarian", final_correspondence_type="hungarian",
                        n_coords_spectral_ordering=1000, graph_smoothing_iterations=20, projection_smooth_iterations=5)
    f.align_maps()
    idx = f.corresponding_target_idx_for_each_source_pt
    assert idx.shape == (s.points.shape[0],) and len(np.unique(idx)) == idx.size      # a one-to-one assignment
    _, ref_idx = linear_sum_assignment(cdist(f.source_projected_on_target, f.smoothed_target_coords))
    assert np.array_equal(idx, ref_idx)
    with pytest.raises(ValueError):
        pyfocusr.Focusr(t, s, icp_register_first=False, initial_correspondence_type="nearest")


def test_smoothing_sub_ranges_and_columns(torch, shipped_meshes, synth):
    """focusr_mean_filter on sub-ranges of a batch (mixed mesh sizes, an isolated vertex), 1 and 3 columns, odd / even /
    single iteration counts: equal to the oracle's scipy product, bit for bit, mesh by mesh."""
    from oracle import port
    from pyfocusr_b200._device import DeviceGraph
    from pyfocusr_b200.mesh import icosphere

    small = icosphere(3)
    pts = np.concatenate([small.points, [[9.0, 9.0, 9.0]]])                    # unreferenced vertex: empty row
    ms = [shipped_meshes["source_mesh_15k"], synth["ell20a"], shipped_meshes["target_mesh"], synth["ell39"]]
    all_pts, all_tris = [m.points for m in ms] + [pts], [m.tris for m in ms] + [small.tris]
    g = DeviceGraph(all_pts, all_tris)
    off = g.mesh_off_host
    adj = [port.adjacency(p, t) for p, t in zip(all_pts, all_tris)]
    rng = np.random.RandomState(0)
    for c in (3, 1):
        x_h = rng.standard_normal((g.n_points, c))
        x = torch.from_numpy(x_h).cuda()
        for iters, (mb, me) in ((1, (0, 5)), (2, (1, 3)), (7, (0, 5)), (40, (2, 5)), (301, (3, 4))):
            r0, r1 = int(off[mb]), int(off[me])
            got = g.mean_filter(x, iters, r0, r1).cpu().numpy()
            for m in range(mb, me):
                ref = port.mean_filter(adj[m], x_h[off[m]:off[m + 1]], iters)
                assert np.array_equal(got[off[m]:off[m + 1]], ref), (c, iters, m)
    with pytest.raises(ValueError):
        g.mean_filter(x, 3, 10, 5000)   # not whole meshes
