"""Shared targets in SpectralBatch (``run(..., target_of_pair=...)``) and the closest-point search against shared
reference segments (``focusr_knn_mapped``).  A batch of T targets and P sources gives, in every key but ``graph`` and
``eigs_info``, exactly what the batch with every target repeated once per pair gives, bit for bit; the mapped search
equals ``focusr_knn`` on materialised copies of the references."""
import numpy as np
import pytest

import pyfocusr_b200.mesh as fmesh
from pyfocusr_b200.batch import SpectralBatch, shared_targets

SPECTRAL_KW = dict(n_coords_spectral_ordering=1000, graph_smoothing_iterations=30, projection_smooth_iterations=10)
AXES = (43.0, 25.0, 33.0)


# --------------------------------------------------------------------------------------------- CPU
def _old_pack(targets, sources):
    """pack_meshes before target_of_pair, restated."""
    meshes = list(targets) + list(sources)
    off = np.zeros(len(meshes) + 1, dtype=np.int32)
    off[1:] = np.cumsum([m.points.shape[0] for m in meshes])
    pts = np.concatenate([m.points for m in meshes])
    tris = np.concatenate([m.tris.astype(np.int64) + int(o) for m, o in zip(meshes, off[:-1])]).astype(np.int32)
    return pts, tris, off, len(targets)


def test_pack_meshes_without_target_of_pair_unchanged():
    t = [fmesh.icosphere(2), fmesh.icosphere(3)]
    s = [fmesh.icosphere(4), fmesh.perturbed_ellipsoid(3, 1)]
    pts, tris, off, P = SpectralBatch.pack_meshes(t, s)
    rp, rt, ro, rP = _old_pack(t, s)
    assert P == rP == 2
    assert off.dtype == ro.dtype and np.array_equal(off, ro)
    assert pts.numpy().dtype == rp.dtype and np.array_equal(pts.numpy(), rp)
    assert tris.numpy().dtype == rt.dtype and np.array_equal(tris.numpy(), rt)
    with pytest.raises(ValueError, match="as many source meshes"):
        SpectralBatch.pack_meshes([t[0]], [])
    with pytest.raises(ValueError, match="as many source meshes"):
        SpectralBatch.pack_meshes([t[0]], s)
    with pytest.raises(ValueError, match="as many source meshes"):
        SpectralBatch.pack_meshes([], [])


def test_pack_meshes_shared_layout():
    t = [fmesh.icosphere(2), fmesh.icosphere(3)]                                  # 42 and 92 vertices
    s = [fmesh.icosphere(4), fmesh.perturbed_ellipsoid(3, 1), fmesh.icosphere(1)]  # 162, 92, 12
    pts, tris, off, P = SpectralBatch.pack_meshes(t, s, target_of_pair=[1, 0, 1])
    assert P == 3
    assert off.tolist() == [0, 42, 134, 296, 388, 400]
    rp, rt, ro, _ = _old_pack(t, s)  # T targets, then the P sources, in the order given
    assert np.array_equal(off, ro) and np.array_equal(pts.numpy(), rp) and np.array_equal(tris.numpy(), rt)
    # one template for every source
    pts, tris, off, P = SpectralBatch.pack_meshes(t[:1], s, target_of_pair=np.zeros(3, dtype=np.int64))
    assert P == 3 and off.tolist() == [0, 42, 204, 296, 308]


def test_argument_rules():
    a, b, c = fmesh.icosphere(2), fmesh.icosphere(3), fmesh.icosphere(4)
    with pytest.raises(ValueError, match="outside"):
        SpectralBatch.pack_meshes([a], [b, c], target_of_pair=[0, 1])
    with pytest.raises(ValueError, match="outside"):
        SpectralBatch.pack_meshes([a], [b, c], target_of_pair=[0, -1])
    with pytest.raises(ValueError, match="used by no pair"):
        SpectralBatch.pack_meshes([a, b], [c, c], target_of_pair=[0, 0])
    with pytest.raises(ValueError, match="one entry per pair"):
        SpectralBatch.pack_meshes([a], [b, c], target_of_pair=[0])
    with pytest.raises(ValueError, match="one entry per pair"):
        SpectralBatch.pack_meshes([a], [b, c], target_of_pair=[[0, 0]])
    with pytest.raises(ValueError, match="integers"):
        SpectralBatch.pack_meshes([a], [b, c], target_of_pair=[0, 0.5])
    with pytest.raises(ValueError, match="at least one pair and one target"):
        SpectralBatch.pack_meshes([a], [], target_of_pair=[])
    with pytest.raises(ValueError, match="at least one pair and one target"):
        SpectralBatch.pack_meshes([], [b, c], target_of_pair=[0, 0])
    top, T = shared_targets(np.array([1, 0, 0, 1, 0]), 7, 5)
    assert T == 2 and top.dtype == np.int32 and top.tolist() == [1, 0, 0, 1, 0]
    # run checks the same rules before it needs a device
    pts, tris, off, P = SpectralBatch.pack_meshes([a, b], [c, c, c], target_of_pair=[0, 1, 1])
    sb = SpectralBatch(**SPECTRAL_KW)
    with pytest.raises(ValueError, match="outside"):
        sb.run(pts, tris, off, P, target_of_pair=[0, 2, 1])
    with pytest.raises(ValueError, match="used by no pair"):
        sb.run(pts, tris, off, P, target_of_pair=[1, 1, 1])
    with pytest.raises(ValueError, match="at least one pair and one target"):
        sb.run(pts, tris, off[:4], P, target_of_pair=[0, 0, 0])
    # moving a shared target onto each of its sources cannot be one move
    icp = SpectralBatch(icp_register_first=True, icp_reg_target_to_source=True, **SPECTRAL_KW)
    with pytest.raises(ValueError, match="icp_reg_target_to_source"):
        icp.run(pts, tris, off, P, target_of_pair=[0, 1, 1])


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


def assert_matches_repeated(torch, out, ref, top):
    """``out`` (T targets + P sources) against ``ref`` (every target repeated once per pair): the solver took the same
    passes for every distinct mesh, and every key but graph / eigs_info is bit-identical."""
    top = np.asarray(top)
    P = top.size
    T = out["graph"].n_meshes - P
    assert ref["graph"].n_meshes == 2 * P
    ia, ib = out["eigs_info"], ref["eigs_info"]
    assert ia["block_size"] == ib["block_size"]
    for m in range(T + P):
        ref_meshes = np.nonzero(top == m)[0] if m < T else [P + m - T]
        for r in ref_meshes:
            for key in ("filter_degree", "outer_iterations", "n_found", "k_final", "status"):
                assert ia[key][m] == ib[key][r], (key, m, r)
    assert set(out) == set(ref)
    assert np.array_equal(out["pair_mesh_off"], ref["graph"].mesh_off_host)
    assert np.array_equal(ref["pair_mesh_off"], ref["graph"].mesh_off_host)
    for key in ref:
        if key in ("graph", "eigs_info"):
            continue
        assert _same(torch, out[key], ref[key]), key


def _run_both(torch, sb_kw, targets, sources, top, **kw):
    out = SpectralBatch(**sb_kw).run_meshes(targets, sources, target_of_pair=top, **kw)
    ref = SpectralBatch(**sb_kw).run_meshes([targets[t] for t in top], sources, **kw)  # its own draws: the same
    torch.cuda.synchronize()
    assert_matches_repeated(torch, out, ref, top)
    return out, ref


def _sources(n, first_seed=1):
    return [fmesh.perturbed_ellipsoid(10 + k % 4, first_seed + 2 * k, semi_axes=AXES) for k in range(n)]


@pytest.mark.gpu
def test_one_template_six_sources(torch):
    template = fmesh.perturbed_ellipsoid(12, 0, semi_axes=AXES)
    out, _ = _run_both(torch, dict(SPECTRAL_KW), [template], _sources(6), [0] * 6, keep_presort=True)
    assert out["graph"].n_meshes == 7 and out["eig_vecs"].shape[0] == int(out["pair_mesh_off"][-1])


@pytest.mark.gpu
def test_two_targets_interleaved(torch):
    targets = [fmesh.perturbed_ellipsoid(12, 0, semi_axes=AXES), fmesh.perturbed_ellipsoid(11, 2, semi_axes=AXES)]
    sb = SpectralBatch(**SPECTRAL_KW)
    top = [1, 0, 0, 1, 0]
    sources = _sources(5)
    out = sb.run_meshes(targets, sources, target_of_pair=np.array(top), record_events=True)
    assert "pair_layout" in sb.timings
    ref = SpectralBatch(**SPECTRAL_KW).run_meshes([targets[t] for t in top], sources)
    assert_matches_repeated(torch, out, ref, top)
    # target_of_pair=None adds no stage
    sb2 = SpectralBatch(**SPECTRAL_KW)
    sb2.run_meshes([targets[t] for t in top], sources, record_events=True)
    assert "pair_layout" not in sb2.timings


@pytest.mark.gpu
def test_source_as_reference(torch):
    targets = [fmesh.perturbed_ellipsoid(12, 0, semi_axes=AXES), fmesh.perturbed_ellipsoid(11, 2, semi_axes=AXES)]
    _run_both(torch, dict(target_eigenmap_as_reference=False, **SPECTRAL_KW), targets, _sources(4), [0, 1, 1, 0])


def _with_scalar(m, k):
    return fmesh.PolyData(m.points, m.tris, {"scal": np.sin(m.points[:, 0] * (0.3 + 0.1 * k)) + m.points[:, 1] ** 2 * 1e-3})


@pytest.mark.gpu
def test_node_features(torch):
    targets = [_with_scalar(fmesh.perturbed_ellipsoid(12, 0, semi_axes=AXES), 0)]
    sources = [_with_scalar(m, k + 1) for k, m in enumerate(_sources(4))]
    kw = dict(list_features_to_calc=["curvature"], list_features_to_get_from_mesh=["scal"], include_features_in_adj_matrix=True,
              use_features_as_coords=True, include_points_as_features=True, **SPECTRAL_KW)
    out, _ = _run_both(torch, kw, targets, sources, [0] * 4)
    assert out["node_features"].shape == (int(out["pair_mesh_off"][-1]), 3)
    assert out["coords"].shape[1] == 3 + 3 + 3


def _misalign(points, deg, axis, shift):
    from scipy.spatial.transform import Rotation

    axis = np.asarray(axis, dtype=np.float64)
    r = Rotation.from_rotvec(np.deg2rad(deg) * axis / np.linalg.norm(axis)).as_matrix()
    return points @ r.T + np.asarray(shift, dtype=np.float64)


@pytest.mark.gpu
def test_icp_onto_shared_template(torch):
    targets = [fmesh.perturbed_ellipsoid(12, 0, semi_axes=AXES)]
    sources = [fmesh.PolyData(_misalign(s.points, 10 + 4 * k, [1, 0.5, -0.3], [3, -2, 1]), s.tris)
               for k, s in enumerate(_sources(4))]
    out, _ = _run_both(torch, dict(icp_register_first=True, **SPECTRAL_KW), targets, sources, [0] * 4)
    assert out["icp_matrices"].shape == (4, 4, 4)
    # unshared targets may still move onto their sources
    targets = [fmesh.perturbed_ellipsoid(12, 0, semi_axes=AXES), fmesh.perturbed_ellipsoid(11, 2, semi_axes=AXES)]
    _run_both(torch, dict(icp_register_first=True, icp_reg_target_to_source=True, **SPECTRAL_KW), targets, sources[:2], [1, 0])


@pytest.mark.gpu
def test_cpd_registration(torch):
    targets = [fmesh.perturbed_ellipsoid(8, 0, semi_axes=AXES)]
    sources = [fmesh.perturbed_ellipsoid(8, 1 + 2 * k, semi_axes=AXES) for k in range(3)]
    kw = dict(registration="b200", non_rigid_max_iterations=50, cpd_streams=2, n_coords_spectral_ordering=500,
              graph_smoothing_iterations=30, projection_smooth_iterations=10)
    out, _ = _run_both(torch, kw, targets, sources, [0] * 3)
    assert not torch.equal(out["coords"], out["coords_b4_reg"])


@pytest.mark.gpu
def test_run_concurrent_and_pipelined(torch):
    template = fmesh.perturbed_ellipsoid(12, 0, semi_axes=AXES)
    sources = _sources(5)
    sb = SpectralBatch(**SPECTRAL_KW)
    parts = ((0, 2), (2, 5))
    jobs, refs = [], []
    for a, b in parts:
        pts, tris, off, n = sb.pack_meshes([template], sources[a:b], target_of_pair=[0] * (b - a))
        ref = SpectralBatch(**SPECTRAL_KW).run_meshes([template] * (b - a), sources[a:b])
        refs.append(ref)
        jobs.append(dict(points=pts, tris=tris, mesh_off_host=off, n_pairs=n, idx_t=ref["idx_t"], idx_s=ref["idx_s"]))
    outs = sb.run_concurrent([dict(j, target_of_pair=[0] * j["n_pairs"]) for j in jobs])
    torch.cuda.synchronize()
    for o, r, (a, b) in zip(outs, refs, parts):
        assert_matches_repeated(torch, o, r, [0] * (b - a))
    outs = sb.run_pipelined([dict(j, target_of_pair=[0] * j["n_pairs"]) for j in jobs], depth=2)
    torch.cuda.synchronize()
    for o, r, (a, b) in zip(outs, refs, parts):
        assert_matches_repeated(torch, o, r, [0] * (b - a))
    # the keyword passed once for every sub-batch of equal size
    same = [jobs[0], dict(jobs[0])]
    outs = sb.run_concurrent(same, target_of_pair=[0, 0])
    torch.cuda.synchronize()
    for o in outs:
        assert_matches_repeated(torch, o, refs[0], [0, 0])


@pytest.mark.gpu
def test_shipped_5k_template(torch, shipped_meshes):
    """The reference's shipped 5k target as template for 3 jittered copies of the 5k source (open meshes; their
    adjacencies are symmetric, as test_gpu_parity.py records)."""
    template, src = shipped_meshes["target_mesh"], shipped_meshes["source_mesh"]
    rng = np.random.RandomState(5)
    sources = [fmesh.PolyData(src.points + rng.normal(scale=0.05, size=src.points.shape), src.tris) for _ in range(3)]
    out, _ = _run_both(torch, dict(SPECTRAL_KW), [template], sources, [0] * 3)
    assert out["eigs_info"]["symmetric"].tolist() == [1] * 4


@pytest.mark.gpu
def test_shipped_15k_template_nonsymmetric(torch, shipped_meshes):
    """The reference's shipped 15k target as template for 3 jittered copies of the 15k source: non-symmetric adjacencies
    (the solver's general path, complex Rayleigh-Ritz), and every source retries from k = 7 to k = 14 while the template
    does not (test_gpu_parity.py records both for the pair), so the batch merges meshes that differ in k."""
    template, src = shipped_meshes["target_mesh_15k"], shipped_meshes["source_mesh_15k"]
    rng = np.random.RandomState(15)
    sources = [fmesh.PolyData(src.points + rng.normal(scale=0.05, size=src.points.shape), src.tris) for _ in range(3)]
    out, ref = _run_both(torch, dict(SPECTRAL_KW), [template], sources, [0] * 3)
    info = out["eigs_info"]
    assert info["symmetric"].tolist() == [0] * 4 and ref["eigs_info"]["symmetric"].tolist() == [0] * 6
    assert info["k_final"].tolist() == [7, 14, 14, 14]


# ------------------------------------------------------------------------------ focusr_knn_mapped
REF_LAYOUTS = {
    "brute_force": [100, 37, 255],      # every reference segment below the pruning threshold
    "threshold": [256, 256, 300],       # at it
    "large": [16384, 1000, 256],
}


def _grid_points(rng, n, dim, dup_from=None):
    """Points on a coarse integer grid (many equal distances), with every fifth row a duplicate of an earlier one."""
    x = np.round(rng.normal(scale=6.0, size=(n, dim)))
    if n > 5:
        x[5::5] = x[rng.randint(0, 5, size=x[5::5].shape[0])]
    if dup_from is not None and n > 1:
        x[::3] = dup_from[rng.randint(0, dup_from.shape[0], size=x[::3].shape[0])]
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("layout", sorted(REF_LAYOUTS))
@pytest.mark.parametrize("dim", [3, 6, 32])
@pytest.mark.parametrize("k", [1, 3])
def test_knn_mapped_equals_knn_on_copies(torch, layout, dim, k):
    from pyfocusr_b200 import _device

    rng = np.random.RandomState(dim * 10 + k)
    ref_sizes = REF_LAYOUTS[layout]
    refs = [_grid_points(rng, n, dim) for n in ref_sizes]
    # query segments of 1 and 16 384 points; several on reference 0, none on reference 1 (unused)
    ref_seg = np.array([0, 2, 0, 0, 2], dtype=np.int32)
    q_sizes = [1, 16384, 700, 16384, 33]
    queries = [_grid_points(rng, n, dim, dup_from=refs[r]) for n, r in zip(q_sizes, ref_seg)]
    dev = torch.device("cuda")

    def offs(sizes):
        return torch.from_numpy(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)).to(dev)

    R = torch.from_numpy(np.concatenate(refs)).to(dev)
    Q = torch.from_numpy(np.concatenate(queries)).to(dev)
    copies = torch.from_numpy(np.concatenate([refs[r] for r in ref_seg])).to(dev)
    copy_sizes = [ref_sizes[r] for r in ref_seg]
    for brute in (False, True):
        idx, dist = _device.knn_mapped(R, Q, offs(ref_sizes), offs(q_sizes), ref_seg, k=k, max_queries=max(q_sizes),
                                       max_refs=max(ref_sizes), brute_force=brute)
        ri, rd = _device.knn(copies, Q, k=k, ref_off=offs(copy_sizes), query_off=offs(q_sizes), max_queries=max(q_sizes),
                             max_refs=max(copy_sizes), brute_force=brute)
        assert torch.equal(idx, ri), (layout, brute)
        assert torch.equal(dist, rd), (layout, brute)
    # the pruned and brute-force searches agree (the mapped form of knn_pruned_applicable picks one of them)
    bi, bd = _device.knn(copies, Q, k=k, ref_off=offs(copy_sizes), query_off=offs(q_sizes), max_queries=max(q_sizes),
                         max_refs=max(copy_sizes), brute_force=True)
    assert torch.equal(idx, bi) and torch.equal(dist, bd)


@pytest.mark.gpu
def test_knn_mapped_rejects_bad_map(torch):
    from pyfocusr_b200 import _device, _lib

    R = torch.zeros((600, 3), dtype=torch.float64, device="cuda")
    Q = torch.zeros((10, 3), dtype=torch.float64, device="cuda")
    ro = torch.tensor([0, 300, 600], dtype=torch.int32, device="cuda")
    qo = torch.tensor([0, 5, 10], dtype=torch.int32, device="cuda")
    with pytest.raises(_lib.FocusrB200Error, match="outside"):
        _device.knn_mapped(R, Q, ro, qo, [0, 2])
    with pytest.raises(ValueError, match="one entry per query segment"):
        _device.knn_mapped(R, Q, ro, qo, [0])
