"""Meshes of any size in one SpectralBatch: a sample count per pair in eigsort's cost stage
(``focusr_eigsort_costs_ragged``), and more than 16 384 ordering samples per mesh (a global segmented sort of the
columns).  The uniform entry point is the ragged one with linear offsets, bit for bit; the costs of a pair do not
depend on which sort ran; every cost matches the oracle on the same eigenvectors and samples."""
import os
import sys

import numpy as np
import pytest

import pyfocusr_b200.mesh as fmesh
from pyfocusr_b200 import _device
from pyfocusr_b200.batch import SpectralBatch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

AXES = (43.0, 25.0, 33.0)
SMOOTH = dict(graph_smoothing_iterations=30, projection_smooth_iterations=10)
NU_MIXED = (20, 22, 23, 39)  # 4 002, 4 842, 5 292 and 15 212 vertices: below, around and above 5 000 samples


# --------------------------------------------------------------------------------------------- CPU
def test_ragged_draws_equal_reference():
    """One Graph.rand_idxs draw per mesh, targets then sources, from one generator: the list the reference draws."""
    from oracle import port

    sb = SpectralBatch(n_coords_spectral_ordering=500)
    sizes = [300, 500, 501, 2000, 499, 500, 12]  # below, equal (a permutation), above
    got = sb.sample_indices(sizes, np.random.RandomState(11))
    np.random.seed(11)
    want = [port.rand_idxs(n, 500) for n in sizes]
    assert isinstance(got, list) and len(got) == len(sizes)
    for g, w in zip(got, want):
        assert g.dtype == np.int64 and np.array_equal(g, w)
    assert np.array_equal(np.sort(got[1]), np.arange(500)) and not np.array_equal(got[1], np.arange(500))
    # equal counts keep the 2-D form
    same = sb.sample_indices([500, 800, 600], np.random.RandomState(11))
    np.random.seed(11)
    assert isinstance(same, np.ndarray) and same.shape == (3, 500)
    assert np.array_equal(same, np.stack([port.rand_idxs(n, 500) for n in (500, 800, 600)]))


def test_argument_rules():
    meshes = [fmesh.icosphere(k) for k in (2, 3, 4, 1)]  # 42, 92, 162 and 12 vertices
    pts, tris, off = SpectralBatch._pack(meshes)
    sb = SpectralBatch(n_coords_spectral_ordering=50)
    good_t, good_s = [np.arange(42), np.arange(50)], [np.arange(50), np.arange(12)]
    cases = [
        ([np.arange(42)], good_s, "idx_t needs one sample array per pair \\(2\\), got 1"),
        (good_t, good_s + [np.arange(3)], "idx_s needs one sample array per pair \\(2\\), got 3"),
        ([np.arange(42), np.arange(0)], good_s, "idx_t\\[1\\] is empty"),
        (good_t, [np.arange(50), np.array([0, 12])], "idx_s\\[1\\] holds index 12 outside \\[0, 12\\)"),
        ([np.array([3, -1]), np.arange(50)], good_s, "idx_t\\[0\\] holds index -1 outside \\[0, 42\\)"),
        (np.zeros((2, 50), dtype=np.int64) + 42, good_s, "idx_t\\[0\\] holds index 42 outside"),
        (good_t, None, "together"),
    ]
    # every rule is checked before the batch needs a device
    for it, is_, msg in cases:
        with pytest.raises(ValueError, match=msg):
            sb.run(pts, tris, off, 2, idx_t=it, idx_s=is_)
    # with a pair list, the sizes are those of each pair's meshes
    with pytest.raises(ValueError, match="idx_s\\[0\\] holds index 42 outside \\[0, 42\\)"):
        sb.run_mesh_pairs(meshes, [(1, 0), (2, 3)], idx_t=[np.arange(50), np.arange(50)],
                          idx_s=[np.arange(43), np.arange(12)])


# --------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch():
    import torch as t

    if not t.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return t


def _mixed_pairs():
    """Four pairs over meshes of 4 002, 4 842, 5 292 and 15 212 vertices, n_t != n_s within every pair."""
    meshes = [fmesh.perturbed_ellipsoid(nu, k, semi_axes=AXES) for k, nu in enumerate(NU_MIXED)]
    return meshes, [(0, 3), (3, 1), (2, 0), (1, 2)]


@pytest.fixture(scope="module")
def mixed_run(torch):
    meshes, mp = _mixed_pairs()
    sb = SpectralBatch(**SMOOTH)
    out = sb.run_meshes([meshes[t] for t, _ in mp], [meshes[s] for _, s in mp], keep_presort=True)
    torch.cuda.synchronize()
    return meshes, mp, out


def _pair_vectors(out, p, P):
    off, nf = out["graph"].mesh_off_host, out["eigs_info"]["n_found"]
    pre = out["eig_vecs_presort"].cpu().numpy()
    vt = pre[off[p]:off[p + 1], :nf[p]].copy()
    vs = pre[off[P + p]:off[P + p + 1], :nf[P + p]].copy()
    return vt, vs


def _assert_costs_match_oracle(costs, p, pts_t, pts_s, it, is_, vt, vs, n, nn=None):
    from scipy.spatial import cKDTree

    from oracle import port

    rt, rs = vt[it], vs[is_]
    ch, chf = port.c_hist(rt, rs, n)
    pt, ps = port.rand_normalized_points(pts_t, it), port.rand_normalized_points(pts_s, is_)
    cs, csf, _ = port.c_spatial(pt, ps, rt, rs, n)
    for got, ref, name in zip(costs, (ch, chf, cs, csf), ("c_hist", "c_hist_f", "c_spatial", "c_spatial_f")):
        assert np.max(np.abs(got[p].cpu().numpy() - ref) / np.abs(ref)) <= 1e-10, (p, name)
    if nn is not None:  # equal to cKDTree's except at exact distance ties
        _, i_ref = cKDTree(ps).query(pt)
        ours = nn.cpu().numpy()
        diff = np.nonzero(ours != i_ref)[0]
        assert np.array_equal(np.linalg.norm(ps[ours[diff]] - pt[diff], axis=1),
                              np.linalg.norm(ps[i_ref[diff]] - pt[diff], axis=1)), p


@pytest.mark.gpu
def test_mixed_costs_against_oracle(torch, mixed_run):
    meshes, mp, out = mixed_run
    P, n = len(mp), 6
    assert isinstance(out["idx_t"], list) and isinstance(out["idx_s"], list)
    assert [len(i) for i in out["idx_t"]] == [4002, 5000, 5000, 4842]
    assert [len(i) for i in out["idx_s"]] == [5000, 4842, 4002, 5000]
    # the stage alone, on the run's pre-sort vectors and samples, gives the run's costs and the nearest neighbours
    g = out["graph"]
    vecs = out["eig_vecs_presort"]
    costs = _device.eigsort_costs(g, vecs, np.arange(P), np.arange(P, 2 * P), out["idx_t"], out["idx_s"], n)
    for a, b in zip(costs[:4], out["costs"]):
        assert torch.equal(a, b)
    nn = costs[4]
    assert isinstance(nn, list) and [int(x.numel()) for x in nn] == [len(i) for i in out["idx_t"]]
    for p, (t, s) in enumerate(mp):
        vt, vs = _pair_vectors(out, p, P)
        _assert_costs_match_oracle(out["costs"], p, meshes[t].points, meshes[s].points, out["idx_t"][p], out["idx_s"][p],
                                   vt, vs, n, nn[p])


@pytest.mark.gpu
def test_uniform_equals_ragged(torch, mixed_run):
    """focusr_eigsort_costs is focusr_eigsort_costs_ragged with linear offsets, bit for bit (n_t == n_s and n_t != n_s)."""
    _, _, out = mixed_run
    g, vecs = out["graph"], out["eig_vecs_presort"]
    sizes = np.diff(g.mesh_off_host)
    rng = np.random.RandomState(5)
    for t_mesh, s_mesh, n_t, n_s in (([1, 2, 7], [4, 7, 1], 5000, 5000), ([4, 5, 7], [3, 1, 2], 4000, 4842)):
        it = np.stack([rng.choice(sizes[m], n_t, replace=False) for m in t_mesh])
        is_ = np.stack([rng.choice(sizes[m], n_s, replace=False) for m in s_mesh])
        uni = _device.eigsort_costs(g, vecs, t_mesh, s_mesh, it, is_, 6)
        rag = _device.eigsort_costs(g, vecs, t_mesh, s_mesh, list(it), list(is_), 6)
        for a, b in zip(uni[:4], rag[:4]):
            assert torch.equal(a, b)
        assert torch.equal(uni[4], torch.stack(rag[4]))


@pytest.mark.gpu
def test_run_meshes_mixed_against_oracle(torch, mixed_run):
    from oracle import port
    from parity_checks import check_pair_against_oracle

    meshes, mp, out = mixed_run
    P = len(mp)
    for p, (t, s) in enumerate(mp):
        mt, ms = meshes[t], meshes[s]
        check_pair_against_oracle(port, out, p, P, mt.points, mt.tris, ms.points, ms.tris, 6, 3,
                                  SMOOTH["graph_smoothing_iterations"], SMOOTH["projection_smooth_iterations"])
    # a pair's samples sliced out of the result and passed back give that pair alone its costs
    sub = SpectralBatch(**SMOOTH).run_meshes([meshes[mp[1][0]]], [meshes[mp[1][1]]], idx_t=out["idx_t"][1:2],
                                             idx_s=out["idx_s"][1:2])
    assert isinstance(sub["idx_t"], list) and np.array_equal(sub["idx_t"][0], out["idx_t"][1])


@pytest.mark.gpu
def test_mesh_pairs_mixed_all_vs_all(torch):
    from test_batch_mesh_pairs import assert_matches_pair_layout

    meshes = [fmesh.perturbed_ellipsoid(nu, 30 + k, semi_axes=AXES) for k, nu in enumerate((20, 22, 23, 39, 22))]
    mp = [(a, b) for a in range(5) for b in range(5) if a != b]
    sb = SpectralBatch(**SMOOTH)
    out = sb.run_mesh_pairs(meshes, mp)
    ref = SpectralBatch(**SMOOTH).run_meshes([meshes[t] for t, _ in mp], [meshes[s] for _, s in mp])
    torch.cuda.synchronize()
    assert isinstance(out["idx_t"], list)
    assert_matches_pair_layout(torch, out, ref, mp)
    pts, tris, off = sb._pack(meshes)
    (conc,) = sb.run_concurrent([dict(points=pts, tris=tris, mesh_off_host=off, n_pairs=len(mp), mesh_pairs=mp)])
    conc2 = sb.run_concurrent([dict(points=pts, tris=tris, mesh_off_host=off, n_pairs=len(mp), mesh_pairs=mp)] * 2)
    torch.cuda.synchronize()
    for o in [conc] + conc2:
        assert_matches_pair_layout(torch, o, ref, mp)


@pytest.fixture(scope="module")
def large_run(torch):
    """Three pairs of 25 002-vertex meshes with 16 384, 16 385 and 20 000 samples per mesh."""
    meshes = [fmesh.perturbed_ellipsoid(50, k, semi_axes=AXES) for k in range(6)]
    counts = (16384, 16385, 20000)
    rng = np.random.RandomState(2)
    n = meshes[0].points.shape[0]
    it = [rng.choice(n, c, replace=False) for c in counts]
    is_ = [rng.choice(n, c, replace=False) for c in counts]
    out = SpectralBatch(**SMOOTH).run_meshes(meshes[:3], meshes[3:], idx_t=it, idx_s=is_, keep_presort=True)
    torch.cuda.synchronize()
    return meshes, out


@pytest.mark.gpu
def test_beyond_16384_against_oracle(torch, large_run):
    meshes, out = large_run
    P, n = 3, 6
    for p in range(P):
        vt, vs = _pair_vectors(out, p, P)
        _assert_costs_match_oracle(out["costs"], p, meshes[p].points, meshes[P + p].points, out["idx_t"][p],
                                   out["idx_s"][p], vt, vs, n)


@pytest.mark.gpu
def test_sort_choice_changes_no_cost(torch, large_run):
    """The 16 384-sample pair alone takes the shared-memory sort, next to a 20 000-sample pair the global one."""
    _, out = large_run
    g, vecs = out["graph"], out["eig_vecs_presort"]
    it, is_ = out["idx_t"], out["idx_s"]
    alone = _device.eigsort_costs(g, vecs, [0], [3], it[:1], is_[:1], 6)
    with_large = _device.eigsort_costs(g, vecs, [0, 2], [3, 5], [it[0], it[2]], [is_[0], is_[2]], 6)
    for a, b in zip(alone[:4], with_large[:4]):
        assert torch.equal(a[0], b[0])
    assert torch.equal(alone[4][0], with_large[4][0])
    for a, b in zip(with_large[:4], out["costs"]):  # and the 20 000-sample pair's costs are those of the batch
        assert torch.equal(a[1], b[2])


@pytest.mark.gpu
def test_dropin_beyond_16384(torch, large_run):
    from oracle import port
    import pyfocusr_b200 as pyfocusr

    meshes, _ = large_run
    mt, ms = meshes[0], meshes[3]
    np.random.seed(4)
    f = pyfocusr.Focusr(mt, ms, n_coords_spectral_ordering=20000, icp_register_first=False, registration="identity",
                        list_features_to_calc=[], **SMOOTH)
    vt0, vs0 = f.graph_target.eig_vecs.copy(), f.graph_source.eig_vecs.copy()
    assert len(f.graph_target.rand_idxs) == 20000 and len(f.graph_source.rand_idxs) == 20000
    f.align_maps()
    srt = port.sort_eigenmaps(mt.points, ms.points, f.graph_target.rand_idxs, f.graph_source.rand_idxs,
                              f.graph_target.eig_vals, f.graph_source.eig_vals, vt0, vs0, 6, True)
    assert np.max(np.abs(f.Q - srt["Q"]) / srt["Q"]) <= 1e-9
    assert np.array_equal(f.graph_source.eig_vecs, vs0) and np.array_equal(f.graph_target.eig_vecs, vt0)
    assert f.corresponding_target_idx_for_each_source_pt.shape == (ms.points.shape[0],)
