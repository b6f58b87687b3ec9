"""Pair lists in SpectralBatch (``run(..., mesh_pairs=...)``, ``run_mesh_pairs``) and the smoothing of mapped segments
(``focusr_mean_filter_mapped``).  M meshes in any order and any (target, source) pairs over them give, in every key but
``graph`` and ``eigs_info``, exactly what the pair layout (every pair's target, then every pair's source, packed once
per pair) gives, bit for bit; the mapped smoothing equals ``focusr_mean_filter`` on materialised copies of the meshes."""
import numpy as np
import pytest

import pyfocusr_b200.mesh as fmesh
from pyfocusr_b200.batch import SpectralBatch, check_icp_moving, mesh_pairs_checked

SPECTRAL_KW = dict(n_coords_spectral_ordering=1000, graph_smoothing_iterations=30, projection_smooth_iterations=10)
AXES = (43.0, 25.0, 33.0)
ALL_VS_ALL_4 = [(a, b) for a in range(4) for b in range(4) if a != b]


# --------------------------------------------------------------------------------------------- CPU
def test_argument_rules():
    a, b, c = fmesh.icosphere(2), fmesh.icosphere(3), fmesh.icosphere(4)
    pts, tris, off = SpectralBatch._pack([a, b, c])
    sb = SpectralBatch(**SPECTRAL_KW)
    cases = [
        ([0, 1, 2], 3, "must be \\[P\\]\\[2\\]"),
        ([[0, 1, 2]], 1, "must be \\[P\\]\\[2\\]"),
        (np.zeros((0, 2), dtype=np.int64), 0, "at least one pair"),
        ([[0, 1], [2, 0.5]], 2, "integers"),
        ([[0, 1], [2, np.nan]], 2, "integers"),
        ([[0, 1], [2, 3]], 2, "outside \\[0, 3\\)"),
        ([[0, 1], [-1, 2]], 2, "outside \\[0, 3\\)"),
        ([[0, 1], [1, 0]], 2, "used by no pair"),
        ([[0, 1], [2, 0]], 3, "n_pairs \\(3\\) must equal"),
    ]
    # run checks every rule before it needs a device
    for mp, n_pairs, msg in cases:
        with pytest.raises(ValueError, match=msg):
            sb.run(pts, tris, off, n_pairs, mesh_pairs=mp)
    with pytest.raises(ValueError, match="not both"):
        sb.run(pts, tris, off, 2, mesh_pairs=[[0, 1], [2, 0]], target_of_pair=[0, 0])
    with pytest.raises(ValueError, match="used by no pair"):
        sb.run_mesh_pairs([a, b, c], [[0, 1]])
    with pytest.raises(ValueError, match="outside"):
        sb.run_mesh_pairs([a, b], [[0, 2]])
    mp = mesh_pairs_checked(np.array([[2.0, 0.0], [1.0, 1.0]]), 3, 2)
    assert mp.dtype == np.int32 and mp.tolist() == [[2, 0], [1, 1]]


def test_icp_rule():
    a, b, c, d = (fmesh.icosphere(k) for k in (1, 2, 3, 4))
    pts, tris, off = SpectralBatch._pack([a, b, c, d])
    icp = SpectralBatch(icp_register_first=True, **SPECTRAL_KW)
    # a moving source in two pairs, a moving source that is fixed in another pair, a self pair
    for mp, msg in (([[0, 2], [1, 2], [0, 3]], "mesh 2 .*pairs \\[0, 1\\]"),
                    ([[0, 1], [1, 2], [0, 3]], "mesh 1 .*pairs \\[0, 1\\]"),
                    ([[0, 1], [2, 2], [0, 3]], "mesh 2 .*pairs \\[1\\]")):
        with pytest.raises(ValueError, match=msg):
            icp.run(pts, tris, off, 3, mesh_pairs=mp)
    # moving the target: the targets must be unique instead
    icp_t = SpectralBatch(icp_register_first=True, icp_reg_target_to_source=True, **SPECTRAL_KW)
    with pytest.raises(ValueError, match="mesh 0 .*pairs \\[0, 2\\]"):
        icp_t.run(pts, tris, off, 3, mesh_pairs=[[0, 1], [2, 1], [0, 3]])
    # fixed meshes may be shared: sources 1, 2, 3 move onto shared target 0
    check_icp_moving(np.array([[0, 1], [0, 2], [0, 3]]), False)
    check_icp_moving(np.array([[1, 0], [2, 0], [3, 0]]), True)
    # the error of target_of_pair keeps its wording
    with pytest.raises(ValueError, match="icp_reg_target_to_source moves each pair's target"):
        icp_t.run(pts, tris, off, 3, target_of_pair=[0, 0, 0])


def _with_scalar(m, k):
    return fmesh.PolyData(m.points, m.tris, {"scal": np.sin(m.points[:, 0] * (0.3 + 0.1 * k)) + m.points[:, 1] ** 2 * 1e-3})


def test_run_mesh_pairs_packs_each_mesh_once():
    meshes = [_with_scalar(fmesh.icosphere(k), k) for k in (2, 1, 3)]  # 42, 12 and 92 vertices
    sb = SpectralBatch(list_features_to_get_from_mesh=["scal"], **SPECTRAL_KW)
    seen = {}
    sb.run = lambda *args, **kw: seen.update(args=args, kw=kw)  # the packed arguments, without a device
    sb.run_mesh_pairs(meshes, [[1, 0], [0, 1], [2, 0], [2, 2]])
    pts, tris, off, n_pairs = seen["args"]
    kw = seen["kw"]
    assert n_pairs == 4 and off.dtype == np.int32 and off.tolist() == [0, 42, 54, 146]
    assert np.array_equal(pts.numpy(), np.concatenate([m.points for m in meshes]))
    assert np.array_equal(tris.numpy(), np.concatenate([m.tris + o for m, o in zip(meshes, off[:-1])]).astype(np.int32))
    assert kw["mesh_pairs"].dtype == np.int32 and kw["mesh_pairs"].tolist() == [[1, 0], [0, 1], [2, 0], [2, 2]]
    assert kw["tri_off_host"].tolist() == np.concatenate([[0], np.cumsum([m.tris.shape[0] for m in meshes])]).tolist()
    assert np.array_equal(kw["node_features"].numpy()[:, 0], np.concatenate([m.point_scalars["scal"] for m in meshes]))
    assert "target_of_pair" not in kw


# --------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch():
    import torch as t

    if not t.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return t


def _same(torch, a, b):
    if a is None or b is None:
        return a is None and b is None
    if isinstance(a, torch.Tensor):
        return isinstance(b, torch.Tensor) and a.dtype == b.dtype and torch.equal(a, b)
    if isinstance(a, np.ndarray):
        return isinstance(b, np.ndarray) and a.dtype == b.dtype and np.array_equal(a, b)
    if isinstance(a, (tuple, list)):
        return type(a) is type(b) and len(a) == len(b) and all(_same(torch, x, y) for x, y in zip(a, b))
    return a == b


def assert_matches_pair_layout(torch, out, ref, mesh_pairs):
    """``out`` (M meshes, pairs ``mesh_pairs``) against ``ref`` (the pair layout: every pair's target, then every pair's
    source): the solver took the same passes for every copy of a mesh, and every key but graph / eigs_info is
    bit-identical."""
    mp = np.asarray(mesh_pairs)
    P = mp.shape[0]
    M = out["graph"].n_meshes
    assert M == int(mp.max()) + 1 and ref["graph"].n_meshes == 2 * P
    ia, ib = out["eigs_info"], ref["eigs_info"]
    assert ia["block_size"] == ib["block_size"]
    for m in range(M):
        copies = np.concatenate([np.nonzero(mp[:, 0] == m)[0], P + np.nonzero(mp[:, 1] == m)[0]])
        assert copies.size
        for r in copies:
            for key in ("filter_degree", "outer_iterations", "n_found", "k_final", "status", "symmetric"):
                assert ia[key][m] == ib[key][r], (key, m, r)
    assert set(out) == set(ref)
    assert np.array_equal(out["pair_mesh_off"], ref["graph"].mesh_off_host)
    for key in ref:
        if key in ("graph", "eigs_info"):
            continue
        assert _same(torch, out[key], ref[key]), key


def _run_both(torch, sb_kw, meshes, mesh_pairs, **kw):
    out = SpectralBatch(**sb_kw).run_mesh_pairs(meshes, mesh_pairs, **kw)
    ref = SpectralBatch(**sb_kw).run_meshes([meshes[t] for t, _ in mesh_pairs], [meshes[s] for _, s in mesh_pairs], **kw)
    torch.cuda.synchronize()
    assert_matches_pair_layout(torch, out, ref, mesh_pairs)
    return out, ref


def _cohort(n, first_seed=0):
    """Meshes of 1002, 1212, 1442 and 1692 vertices (none a multiple of 128)."""
    return [fmesh.perturbed_ellipsoid(10 + k % 4, first_seed + k, semi_axes=AXES) for k in range(n)]


# ------------------------------------------------------------------------ focusr_mean_filter_mapped
@pytest.mark.gpu
@pytest.mark.parametrize("n_cols", [1, 2, 3, 5])
def test_mean_filter_mapped_equals_copies(torch, n_cols):
    from pyfocusr_b200._device import DeviceGraph

    meshes = [fmesh.icosphere(1), fmesh.perturbed_ellipsoid(10, 3, semi_axes=AXES), fmesh.icosphere(3),
              fmesh.icosphere(4)]  # 12 (less than a CTA), 1002, 92 and 162 vertices
    g = DeviceGraph([m.points for m in meshes], [m.tris for m in meshes])
    rng = np.random.RandomState(n_cols)
    # mesh 1 in three segments, the segments out of graph order, mesh 3 in none (the table form); consecutive meshes in
    # ascending order (the identity form on shifted rows)
    for seg in ([1, 0, 1, 2, 1], [1, 2, 3]):
        copies = DeviceGraph([meshes[m].points for m in seg], [meshes[m].tris for m in seg])
        vals = torch.from_numpy(rng.normal(size=(copies.n_points, n_cols))).cuda()
        for it in (0, 1, 2, 7):
            got = g.mean_filter_mapped(vals, it, seg)
            want = copies.mean_filter(vals, it)
            torch.cuda.synchronize()
            assert torch.equal(got, want), (seg, it)
    copies = DeviceGraph([meshes[m].points for m in (1, 0)], [meshes[m].tris for m in (1, 0)])
    vals = torch.from_numpy(rng.normal(size=(copies.n_points, n_cols))).cuda()
    # one mesh as the only segment
    one = vals[:1002].contiguous()
    assert torch.equal(g.mean_filter_mapped(one, 7, [1]), copies.mean_filter(vals, 7)[:1002])


@pytest.mark.gpu
def test_mean_filter_mapped_rejects_bad_map(torch):
    from pyfocusr_b200 import _lib
    from pyfocusr_b200._device import DeviceGraph

    meshes = [fmesh.icosphere(1), fmesh.icosphere(2)]
    g = DeviceGraph([m.points for m in meshes], [m.tris for m in meshes])
    vals = torch.zeros((24, 3), dtype=torch.float64, device="cuda")
    with pytest.raises(_lib.FocusrB200Error, match="outside"):
        g.mean_filter_mapped(vals, 3, [0, 2])
    with pytest.raises(_lib.FocusrB200Error, match="outside"):
        g.mean_filter_mapped(vals, 3, [-1, 0])
    with pytest.raises(ValueError, match="hold 54 rows"):
        g.mean_filter_mapped(vals, 3, [0, 1])


# ------------------------------------------------------------------------------------ SpectralBatch
@pytest.mark.gpu
def test_all_vs_all(torch):
    meshes = _cohort(4)
    sb = SpectralBatch(**SPECTRAL_KW)
    out = sb.run_mesh_pairs(meshes, ALL_VS_ALL_4, record_events=True, keep_presort=True)
    assert "pair_layout" in sb.timings and "smoothing" in sb.timings
    ref = SpectralBatch(**SPECTRAL_KW).run_meshes([meshes[t] for t, _ in ALL_VS_ALL_4], [meshes[s] for _, s in ALL_VS_ALL_4],
                                                  keep_presort=True)
    torch.cuda.synchronize()
    assert out["graph"].n_meshes == 4 and out["eig_vecs"].shape[0] == int(out["pair_mesh_off"][-1])
    assert_matches_pair_layout(torch, out, ref, ALL_VS_ALL_4)


@pytest.mark.gpu
@pytest.mark.parametrize("target_as_reference", [True, False])
def test_mixed_pair_list(torch, target_as_reference):
    # mesh 0 is the source of three pairs, mesh 1 a target (pair 0) and a source (pair 3), (4, 4) a self pair
    meshes = _cohort(5, first_seed=7)
    mp = [(1, 0), (2, 0), (3, 0), (2, 1), (4, 4)]
    _run_both(torch, dict(target_eigenmap_as_reference=target_as_reference, **SPECTRAL_KW), meshes, mp)


@pytest.mark.gpu
def test_node_features(torch):
    meshes = [_with_scalar(m, k) for k, m in enumerate(_cohort(3, first_seed=3))]
    kw = dict(list_features_to_calc=["curvature"], list_features_to_get_from_mesh=["scal"], include_features_in_adj_matrix=True,
              use_features_as_coords=True, include_points_as_features=True, **SPECTRAL_KW)
    out, _ = _run_both(torch, kw, meshes, [(0, 1), (1, 0), (2, 0), (2, 1)])
    assert out["node_features"].shape == (int(out["pair_mesh_off"][-1]), 3)
    assert out["coords"].shape[1] == 3 + 3 + 3


def _misalign(points, deg, axis, shift):
    from scipy.spatial.transform import Rotation

    axis = np.asarray(axis, dtype=np.float64)
    r = Rotation.from_rotvec(np.deg2rad(deg) * axis / np.linalg.norm(axis)).as_matrix()
    return points @ r.T + np.asarray(shift, dtype=np.float64)


@pytest.mark.gpu
def test_icp(torch):
    base = _cohort(5, first_seed=11)
    meshes = base[:2] + [fmesh.PolyData(_misalign(m.points, 10 + 4 * k, [1, 0.5, -0.3], [3, -2, 1]), m.tris)
                         for k, m in enumerate(base[2:])]
    # moving sources 2, 3, 4 each in one pair; fixed meshes 0 and 1 shared
    mp = [(0, 2), (1, 3), (0, 4)]
    out, _ = _run_both(torch, dict(icp_register_first=True, **SPECTRAL_KW), meshes, mp)
    assert out["icp_matrices"].shape == (3, 4, 4)
    # moving targets: each target in one pair, the fixed sources shared
    _run_both(torch, dict(icp_register_first=True, icp_reg_target_to_source=True, **SPECTRAL_KW), meshes,
              [(2, 0), (3, 0), (4, 1)])
    with pytest.raises(ValueError, match="moving mesh"):
        SpectralBatch(icp_register_first=True, **SPECTRAL_KW).run_mesh_pairs(meshes, [(0, 2), (1, 2), (0, 3), (1, 4)])


@pytest.mark.gpu
def test_cpd_registration(torch):
    meshes = [fmesh.perturbed_ellipsoid(8, k, semi_axes=AXES) for k in range(3)]
    kw = dict(registration="b200", non_rigid_max_iterations=50, cpd_streams=2, n_coords_spectral_ordering=500,
              graph_smoothing_iterations=30, projection_smooth_iterations=10)
    out, _ = _run_both(torch, kw, meshes, [(0, 1), (1, 0), (2, 0)])
    assert not torch.equal(out["coords"], out["coords_b4_reg"])


@pytest.mark.gpu
def test_run_concurrent_and_pipelined(torch):
    meshes = _cohort(4, first_seed=20)
    lists = ([(0, 1), (1, 0), (2, 1)], [(3, 0), (0, 3), (3, 3), (1, 2)])
    sb = SpectralBatch(**SPECTRAL_KW)
    jobs, refs = [], []
    for mp in lists:
        used = sorted({m for pair in mp for m in pair})
        sub = [meshes[m] for m in used]
        local = [(used.index(t), used.index(s)) for t, s in mp]
        pts, tris, off = sb._pack(sub)
        ref = SpectralBatch(**SPECTRAL_KW).run_meshes([sub[t] for t, _ in local], [sub[s] for _, s in local])
        refs.append((ref, local))
        jobs.append(dict(points=pts, tris=tris, mesh_off_host=off, n_pairs=len(local), mesh_pairs=local))
    for outs in (sb.run_concurrent(jobs), sb.run_pipelined(jobs, depth=2)):
        torch.cuda.synchronize()
        for o, (r, local) in zip(outs, refs):
            assert_matches_pair_layout(torch, o, r, local)
    # the keyword passed once for every sub-batch
    same = [{k: v for k, v in jobs[0].items() if k != "mesh_pairs"}] * 2
    for o in sb.run_concurrent(same, mesh_pairs=lists[0]):
        torch.cuda.synchronize()
        assert_matches_pair_layout(torch, o, refs[0][0], lists[0])


@pytest.mark.gpu
def test_equals_target_of_pair(torch):
    targets = [fmesh.perturbed_ellipsoid(12, 0, semi_axes=AXES), fmesh.perturbed_ellipsoid(11, 2, semi_axes=AXES)]
    sources = [fmesh.perturbed_ellipsoid(10 + k % 4, 1 + 2 * k, semi_axes=AXES) for k in range(5)]
    top = [1, 0, 0, 1, 0]
    a = SpectralBatch(**SPECTRAL_KW).run_meshes(targets, sources, target_of_pair=top, keep_presort=True)
    b = SpectralBatch(**SPECTRAL_KW).run_mesh_pairs(targets + sources, [(t, 2 + p) for p, t in enumerate(top)],
                                                    keep_presort=True)
    torch.cuda.synchronize()
    assert set(a) == set(b)
    for key in a:
        if key == "graph":
            ga, gb = a[key], b[key]
            assert ga.n_meshes == gb.n_meshes == 7 and np.array_equal(ga.mesh_off_host, gb.mesh_off_host)
            assert torch.equal(ga.points, gb.points)
        elif key == "eigs_info":
            assert set(a[key]) == set(b[key]) and all(_same(torch, a[key][k], b[key][k]) for k in a[key])
        else:
            assert _same(torch, a[key], b[key]), key
