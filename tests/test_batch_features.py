"""Node features in SpectralBatch (``focusr_node_features``, ``focusr_feature_coords``): curvature and mesh scalars,
normalised per mesh, in the edge weights and as extra correspondence coordinates, with xyz appended.  Every per-mesh
result equals the numpy restatement of the reference (graph.py:121-142,166-175; focusr.py:218-295) bit for bit, and a
pair's results do not depend on the batch it is in."""
import numpy as np
import pytest

import pyfocusr_b200.mesh as fmesh


def pairwise_sum(a):
    """numpy's pairwise summation of a contiguous float64 array (the rule csrc/features.cu restates)."""
    n = a.size
    if n < 8:
        res = -0.0
        for x in a:
            res = res + x
        return np.float64(res)
    if n <= 128:
        r = list(a[:8])
        i = 8
        while i < n - n % 8:
            for j in range(8):
                r[j] = r[j] + a[i + j]
            i += 8
        res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
        for k in range(i, n):
            res = res + a[k]
        return np.float64(res)
    n2 = n // 2
    n2 -= n2 % 8
    return pairwise_sum(a[:n2]) + pairwise_sum(a[n2:])


# --------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 6, 7, 8, 9, 127, 128, 129, 5000, 8193, 15212, 100003])
def test_pairwise_rule_equals_numpy_mean_and_std(n):
    rng = np.random.default_rng(n)
    a = rng.standard_normal(n) * rng.uniform(0.1, 100.0) + rng.uniform(-50.0, 50.0)
    mean = pairwise_sum(a) / n
    d = a - mean
    std = np.sqrt(pairwise_sum(d * d) / n)
    assert mean.tobytes() == np.mean(a).tobytes()
    assert std.tobytes() == np.std(a).tobytes()


def test_argument_rules():
    import torch

    from pyfocusr_b200 import SpectralBatch

    with pytest.raises(ValueError, match="unknown feature"):
        SpectralBatch(list_features_to_calc=["gauss_curvature"])
    a, b = fmesh.icosphere(2), fmesh.icosphere(3)
    pts, tris, off, P = SpectralBatch.pack_meshes([a], [b])
    sb = SpectralBatch(list_features_to_get_from_mesh=["thickness"], include_features_in_adj_matrix=True)
    with pytest.raises(ValueError, match="node_features"):
        sb.run(pts, tris, off, P)
    with pytest.raises(ValueError, match="node_features must be"):
        sb.run(pts, tris, off, P, node_features=torch.zeros((int(off[-1]), 2), dtype=torch.float64))
    with pytest.raises(ValueError, match="node_features must be"):
        sb.run(pts, tris, off, P, node_features=np.zeros(int(off[-1])))
    with pytest.raises(Exception, match="NO SCALARS WITH SPECIFIED NAME: thickness"):
        sb.run_meshes([a], [b])
    # coordinates too wide: KNN takes 32 columns, CPD 16
    many = ["curvature"] * 14  # 28 feature columns
    SpectralBatch(list_features_to_calc=many, use_features_as_coords=True)  # 3 + 28 = 31
    with pytest.raises(ValueError, match="KNN"):
        SpectralBatch(list_features_to_calc=many, use_features_as_coords=True, include_points_as_features=True)  # 31 + 3
    with pytest.raises(ValueError, match="CPD"):
        SpectralBatch(list_features_to_calc=["curvature"] * 7, use_features_as_coords=True, registration="b200")  # 3 + 14
    SpectralBatch(list_features_to_calc=["curvature"] * 5, use_features_as_coords=True, include_points_as_features=True,
                  registration="b200")  # 3 + 10 + 3 = 16
    # features that nothing consumes widen nothing
    SpectralBatch(list_features_to_calc=many, registration="b200")
    # bench.py passes the first five positionally
    sb = SpectralBatch(3, 3, 5000, 300, 40, seed=0)
    assert (sb.ns, sb.n, sb.n_samples, sb.graph_smoothing_iterations, sb.projection_smooth_iterations) == (3, 6, 5000, 300, 40)
    assert not sb.features_on and sb.n_coords == 3


# --------------------------------------------------------------------------------------------- GPU
SPECTRAL_KW = dict(n_coords_spectral_ordering=1000, graph_smoothing_iterations=30, projection_smooth_iterations=10)


@pytest.fixture(scope="module")
def torch():
    import torch as t

    if not t.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return t


@pytest.fixture(scope="module")
def feature_meshes(shipped_meshes):
    """Icospheres of 42 to 10 242 vertices, a 15k bench mesh and the shipped 5k pair, each with a scalar column."""
    ms = [fmesh.icosphere(2), fmesh.perturbed_ellipsoid(7, 3, semi_axes=(40.0, 30.0, 20.0)), fmesh.icosphere(12, 25.0),
          fmesh.icosphere(32, 30.0), fmesh.ellipsoid_pair(0, 39)[0], shipped_meshes["target_mesh"], shipped_meshes["source_mesh"]]
    out = []
    for k, m in enumerate(ms):
        s = m.point_scalars.get("thickness_change_(mm)")
        if s is None:
            s = np.sin(m.points[:, 0] * (0.3 + 0.1 * k)) + m.points[:, 1] ** 2 * 1e-3
        out.append((m, np.asarray(s, dtype=np.float64)))
    return out


def _pack(meshes):
    off = np.zeros(len(meshes) + 1, dtype=np.int32)
    off[1:] = np.cumsum([m.points.shape[0] for m in meshes])
    pts = np.concatenate([m.points for m in meshes])
    tris = np.concatenate([m.tris.astype(np.int64) + o for m, o in zip(meshes, off[:-1])]).astype(np.int32)
    return pts, tris, off


def _csr_rows(graph, m):
    """Mesh m's rows of a batch graph as (data, local column ids, indptr from 0)."""
    rp, ci, w = graph.adjacency_host()
    o = graph.mesh_off_host
    b, e = int(rp[o[m]]), int(rp[o[m + 1]])
    return w[b:e], ci[b:e] - o[m], rp[o[m]:o[m + 1] + 1] - rp[o[m]]


def _same(a, b):
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


@pytest.mark.gpu
def test_curvature_of_a_batch_equals_per_mesh(torch, feature_meshes):
    from pyfocusr_b200 import _device

    meshes = [m for m, _ in feature_meshes]
    pts, tris, off = _pack(meshes)
    batch = _device.curvatures(pts, tris)
    for k, m in enumerate(meshes):
        one = _device.curvatures(m.points, m.tris)
        for name in ("minimum", "maximum"):
            assert np.array_equal(batch[name][off[k]:off[k + 1]].cpu().numpy(), one[name].cpu().numpy()), (k, name)


@pytest.mark.gpu
def test_normalised_features_equal_numpy(torch, feature_meshes):
    """Every (mesh, column) of a batch against port.normalized_node_feature for every std / cap / 0-1 setting; edge points
    against port.feature_augmented_points.  Two extra point sets without triangles take the n < 8 and n <= 128 branches
    of numpy's summation, and a constant column gives NaN as numpy does."""
    from oracle import port
    from pyfocusr_b200 import _device

    rng = np.random.RandomState(0)
    pts_l, raw_l = [], []
    for m, s in feature_meshes:
        c = _device.curvatures(m.points, m.tris)
        pts_l.append(m.points)
        raw_l.append(np.stack([c["minimum"].cpu().numpy(), c["maximum"].cpu().numpy(), s], axis=1))
    for n in (5, 100):
        pts_l.append(rng.standard_normal((n, 3)) * 10.0)
        raw_l.append(rng.standard_normal((n, 3)) * 3.0 + 1.0)
    raw_l[1][:, 2] = 0.7  # zero spread
    off = np.zeros(len(pts_l) + 1, dtype=np.int32)
    off[1:] = np.cumsum([p.shape[0] for p in pts_l])
    pts, raw = torch.from_numpy(np.concatenate(pts_l)).cuda(), torch.from_numpy(np.concatenate(raw_l)).cuda()
    off_d = torch.from_numpy(off).cuda()
    for std in (True, False):
        for cap in (3, 1.5, False):
            for zero_one in (True, False):
                feats, ep = _device.node_features(raw, pts, off_d, std, cap, zero_one, want_edge_points=True)
                feats, ep = feats.cpu().numpy(), ep.cpu().numpy()
                for k in range(len(pts_l)):
                    mine = feats[off[k]:off[k + 1]]
                    ref = [port.normalized_node_feature(raw_l[k][:, c], std, cap, zero_one) for c in range(3)]
                    for c in range(3):
                        assert _same(mine[:, c], ref[c]), (std, cap, zero_one, k, c)
                    assert _same(ep[off[k]:off[k + 1]], port.feature_augmented_points(pts_l[k], ref)), (std, cap, zero_one, k)
    # the drop-in Graph (numpy normalisation) on the shipped 5k target, curvature + thickness
    import pyfocusr_b200 as pyfocusr

    m = feature_meshes[5][0]
    g = pyfocusr.Graph(m, list_features_to_calc=["curvature"], list_features_to_get_from_mesh=["thickness_change_(mm)"])
    feats, _ = _device.node_features(raw, pts, off_d)
    mine = feats[off[5]:off[6]].cpu().numpy()
    for c in range(3):
        assert np.array_equal(mine[:, c], g.node_features[c]), c


def _feature_pairs():
    axes = (43.0, 25.0, 33.0)
    t = [fmesh.perturbed_ellipsoid(12, 0, semi_axes=axes), fmesh.perturbed_ellipsoid(10, 2, semi_axes=axes)]
    s = [fmesh.perturbed_ellipsoid(12, 1, semi_axes=axes), fmesh.perturbed_ellipsoid(11, 3, semi_axes=axes)]
    return t, s


def _oracle_feature_block(torch, out, m, mesh, curvature_columns=("minimum", "maximum")):
    """The batch's own normalised features of mesh m, checked against numpy's normalisation of per-mesh curvature."""
    from oracle import port
    from pyfocusr_b200 import _device

    off = out["graph"].mesh_off_host
    mine = out["node_features"][off[m]:off[m + 1]].cpu().numpy()
    c = _device.curvatures(mesh.points, mesh.tris)
    ref = [port.normalized_node_feature(c[name].cpu().numpy()) for name in curvature_columns]
    for k in range(len(ref)):
        assert np.array_equal(mine[:, k], ref[k]), (m, k)
    return ref


def _expected_coords(out, m, p, mesh, a, feats, ns, use_features, include_points, norm_physical, iterations=40):
    """focusr.py:218-295 in numpy, fed the batch's own sorted eigenvectors and spectral weights."""
    from oracle import port

    off = out["graph"].mesh_off_host
    vecs = out["eig_vecs"][off[m]:off[m + 1]].cpu().numpy()
    coords = port.spectral_coords(vecs, out["spectral_weights"][p].cpu().numpy(), ns)
    if use_features:
        coords = port.features_as_coords(a, feats, coords, iterations)
    if include_points:
        if norm_physical:
            coords = np.concatenate((coords, port.normed_points(mesh.points)), axis=1)
        else:
            coords = np.concatenate((coords * np.mean(np.ptp(mesh.points, axis=0)), mesh.points), axis=1)
    return coords


@pytest.mark.gpu
@pytest.mark.parametrize("in_adj,use_feats,incl_pts,norm_phys,calc", [
    (True, True, True, True, ["curvature"]), (True, True, True, False, ["curvature"]),
    (False, True, False, True, ["curvature"]), (False, False, True, False, ["curvature"]),
    (False, True, False, True, ["curvature", "min_curvature", "max_curvature"] * 3)])  # 12 columns: smoothed 8 + 4
def test_adjacency_coordinates_and_correspondences_equal_oracle(torch, in_adj, use_feats, incl_pts, norm_phys, calc):
    from oracle import port
    from pyfocusr_b200 import SpectralBatch
    from pyfocusr_b200.batch import CURVATURE_FEATURES

    targets, sources = _feature_pairs()
    sb = SpectralBatch(list_features_to_calc=calc, include_features_in_adj_matrix=in_adj, use_features_as_coords=use_feats,
                       include_points_as_features=incl_pts, norm_physical_and_spectral=norm_phys, **SPECTRAL_KW)
    columns = [c for name in calc for c in CURVATURE_FEATURES[name]]
    out = sb.run_meshes(targets, sources, record_events=True)
    assert ("features" in sb.timings) == (in_adj or use_feats)
    assert ("feature_coords" in sb.timings) == (use_feats or incl_pts)
    P, g = len(targets), out["graph"]
    off = g.mesh_off_host
    coords = out["coords"].cpu().numpy()
    assert coords.shape[1] == 3 + len(columns) * use_feats + 3 * incl_pts
    adj = {}
    for m, mesh in enumerate(targets + sources):
        feats = _oracle_feature_block(torch, out, m, mesh, columns) if (in_adj or use_feats) else None
        if not (in_adj or use_feats):
            assert out["node_features"] is None
        a = port.adjacency(port.feature_augmented_points(mesh.points, feats) if in_adj else mesh.points, mesh.tris)
        data, cols, indptr = _csr_rows(g, m)
        assert np.array_equal(data, a.data) and np.array_equal(cols, a.indices) and np.array_equal(indptr, a.indptr), m
        adj[m] = a
        exp = _expected_coords(out, m, m % P, mesh, a, feats, 3, use_feats, incl_pts, norm_phys)
        assert np.array_equal(coords[off[m]:off[m + 1]], exp), m
    for p in range(P):
        t, s = targets[p], sources[p]
        cs = port.correspondence_stage(dict(A=adj[p]), dict(A=adj[P + p]), t.points, s.points,
                                       coords[off[p]:off[p + 1]], coords[off[P + p]:off[P + p + 1]], 30, 10)
        nt = int(off[P])
        q0, q1 = off[P + p] - nt, off[P + p + 1] - nt
        for key in ("initial_idx", "final_idx", "knn3_idx", "source_projected_on_target", "weighted_avg_transformed_points"):
            mine = out[key][q0:q1].cpu().numpy()
            assert np.array_equal(mine, cs[key]), (p, key)
        assert np.array_equal(out["smoothed_target_coords"][off[p]:off[p + 1]].cpu().numpy(), cs["smoothed_target_coords"]), p


KEYS = ("eig_vals", "eig_vecs", "coords", "node_features", "initial_idx", "final_idx", "knn3_idx", "knn3_dist",
        "smoothed_target_coords", "source_projected_on_target", "weighted_avg_transformed_points",
        "nearest_neighbor_transformed_points", "Q", "spectral_weights")


def _pair_rows(out, key, p, P):
    """Pair p's part of a result: its two meshes' rows (per-vertex / per-mesh keys), its source rows, or its row."""
    off = out["graph"].mesh_off_host
    v = out[key]
    nt = int(off[P])
    if key in ("initial_idx", "final_idx", "knn3_idx", "knn3_dist", "source_projected_on_target",
               "weighted_avg_transformed_points", "nearest_neighbor_transformed_points"):
        return v[off[P + p] - nt:off[P + p + 1] - nt]
    if key == "smoothed_target_coords":
        return v[off[p]:off[p + 1]]
    if key in ("Q", "spectral_weights"):
        return v[p]
    if key == "eig_vals":
        return v[[p, P + p]]
    return torch_module().cat([v[off[p]:off[p + 1]], v[off[P + p]:off[P + p + 1]]])


def torch_module():
    import torch

    return torch


def _six_pairs():
    axes = (43.0, 25.0, 33.0)
    t = [fmesh.perturbed_ellipsoid(10 + k, 2 * k, semi_axes=axes) for k in range(6)]
    s = [fmesh.perturbed_ellipsoid(11 + k, 2 * k + 1, semi_axes=axes) for k in range(6)]
    return t, s


@pytest.mark.gpu
def test_pairs_equal_batches_of_one(torch):
    """A pair's results do not depend on the batch it is in.  The eigensolver runs one Chebyshev degree for a whole batch
    (the largest any of its meshes needs), so a mesh's eigenpairs, and everything computed from them, are bit-identical to
    those of a batch of one where that degree is the same: six copies of one pair are compared in every output, also
    through run_concurrent.  For six different pairs everything before the solver (the normalised features and the edge
    weights) is compared bit for bit, and the eigenvalues to 1e-9."""
    from pyfocusr_b200 import SpectralBatch

    kw = dict(list_features_to_calc=["curvature", "max_curvature"], include_features_in_adj_matrix=True,
              use_features_as_coords=True, include_points_as_features=True, **SPECTRAL_KW)
    targets, sources = _six_pairs()
    out = SpectralBatch(**kw).run_meshes(targets, sources)
    P = len(targets)
    assert out["coords"].shape[1] == 3 + 3 + 3
    for p in range(P):
        one = SpectralBatch(**kw).run_meshes(targets[p:p + 1], sources[p:p + 1], idx_t=out["idx_t"][p:p + 1],
                                             idx_s=out["idx_s"][p:p + 1])
        assert torch.equal(_pair_rows(out, "node_features", p, P), _pair_rows(one, "node_features", 0, 1)), p
        for m, m1 in ((p, 0), (P + p, 1)):
            for a, b in zip(_csr_rows(out["graph"], m), _csr_rows(one["graph"], m1)):
                assert np.array_equal(a, b), (p, m)
        v, v1 = _pair_rows(out, "eig_vals", p, P)[:, :6].cpu().numpy(), _pair_rows(one, "eig_vals", 0, 1)[:, :6].cpu().numpy()
        assert np.max(np.abs(v - v1) / v1) <= 1e-9, p

    t, s = targets[2], sources[2]
    sb = SpectralBatch(**kw)
    out = sb.run_meshes([t] * P, [s] * P)
    for p in range(P):
        one = SpectralBatch(**kw).run_meshes([t], [s], idx_t=out["idx_t"][p:p + 1], idx_s=out["idx_s"][p:p + 1])
        for key in KEYS:
            assert torch.equal(_pair_rows(out, key, p, P), _pair_rows(one, key, 0, 1)), (p, key)
    # through run_concurrent: sub-batches of 2 and 4 pairs
    jobs = []
    for a, b in ((0, 2), (2, 6)):
        pts, tris, off, n = sb.pack_meshes([t] * (b - a), [s] * (b - a))
        jobs.append(dict(points=pts, tris=tris, mesh_off_host=off, n_pairs=n, idx_t=out["idx_t"][a:b], idx_s=out["idx_s"][a:b]))
    outs = sb.run_concurrent(jobs)
    torch.cuda.synchronize()
    for (a, b), o in zip(((0, 2), (2, 6)), outs):
        for p in range(a, b):
            for key in KEYS:
                assert torch.equal(_pair_rows(o, key, p - a, b - a), _pair_rows(out, key, p, P)), (p, key)


@pytest.mark.gpu
def test_defaults_unchanged(torch):
    from pyfocusr_b200 import SpectralBatch

    targets, sources = _feature_pairs()
    ref = SpectralBatch(**SPECTRAL_KW).run_meshes(targets, sources)
    assert ref["node_features"] is None and ref["coords"].shape[1] == 3
    for kw in (dict(list_features_to_calc=[], include_features_in_adj_matrix=True, use_features_as_coords=True),
               dict(list_features_to_calc=["curvature"], include_features_in_adj_matrix=False, use_features_as_coords=False)):
        sb = SpectralBatch(**kw, **SPECTRAL_KW)
        out = sb.run_meshes(targets, sources, record_events=True)
        assert "features" not in sb.timings and "feature_coords" not in sb.timings
        assert out["node_features"] is None
        for key in KEYS:
            if key != "node_features":
                assert torch.equal(out[key], ref[key]), (kw, key)


def _misalign(points, deg, axis, shift):
    from scipy.spatial.transform import Rotation

    axis = np.asarray(axis, dtype=np.float64)
    r = Rotation.from_rotvec(np.deg2rad(deg) * axis / np.linalg.norm(axis)).as_matrix()
    return points @ r.T + np.asarray(shift, dtype=np.float64)


@pytest.mark.gpu
def test_features_after_icp_equal_premoved(torch):
    from pyfocusr_b200 import SpectralBatch, _device

    targets, sources = _feature_pairs()
    sources = [fmesh.PolyData(_misalign(s.points, 20 + 5 * k, [1, 0.5, -0.3], [4, -2, 3]), s.tris) for k, s in enumerate(sources)]
    kw = dict(include_features_in_adj_matrix=True, **SPECTRAL_KW)
    out = SpectralBatch(icp_register_first=True, **kw).run_meshes(targets, sources)
    moved = [fmesh.PolyData(_device.icp(t.points, t.tris, s.points, max_iterations=100, max_landmarks=1000)[1].cpu().numpy(), s.tris)
             for t, s in zip(targets, sources)]
    ref = SpectralBatch(**kw).run_meshes(targets, moved, idx_t=out["idx_t"], idx_s=out["idx_s"])
    for key in KEYS:
        assert torch.equal(out[key], ref[key]), key


@pytest.mark.gpu
def test_cpd_with_feature_coordinates_equals_batches_of_one(torch):
    from pyfocusr_b200 import SpectralBatch

    # two copies of one pair: the solver's degree is common to a batch (test_pairs_equal_batches_of_one); 642 vertices
    # < n_coords_spectral_registration, so CPD draws no random subsets and pair 1 sees what a batch of one sees
    axes = (43.0, 25.0, 33.0)
    targets = [fmesh.perturbed_ellipsoid(8, 0, semi_axes=axes)] * 2
    sources = [fmesh.perturbed_ellipsoid(8, 1, semi_axes=axes)] * 2
    kw = dict(registration="b200", use_features_as_coords=True, include_points_as_features=True,
              non_rigid_max_iterations=50, cpd_streams=2, **SPECTRAL_KW)
    out = SpectralBatch(**kw).run_meshes(targets, sources)
    assert out["coords"].shape[1] == 8 and out["coords_b4_reg"].shape[1] == 8
    assert not torch.equal(out["coords"], out["coords_b4_reg"])
    P = len(targets)
    for p in range(P):
        one = SpectralBatch(**kw).run_meshes(targets[p:p + 1], sources[p:p + 1], idx_t=out["idx_t"][p:p + 1],
                                             idx_s=out["idx_s"][p:p + 1])
        for key in KEYS:
            assert torch.equal(_pair_rows(out, key, p, P), _pair_rows(one, key, 0, 1)), (p, key)


@pytest.mark.gpu
def test_shipped_5k_pair_with_mesh_scalar(torch, shipped_meshes, golden):
    """test_gpu_parity.py::test_mesh_scalar_features_in_adjacency_and_as_coordinates through the batch path: the open 5k
    pair (non-symmetric solver path), thickness in the edge weights and as a coordinate."""
    from oracle import port
    from pyfocusr_b200 import SpectralBatch

    name = "thickness_change_(mm)"
    mt, ms = shipped_meshes["target_mesh"], shipped_meshes["source_mesh"]
    sb = SpectralBatch(list_features_to_calc=[], list_features_to_get_from_mesh=[name], include_features_in_adj_matrix=True,
                       use_features_as_coords=True, **SPECTRAL_KW)
    out = sb.run_meshes([mt], [ms])
    g = out["graph"]
    vals = out["eig_vals"].cpu().numpy()
    coords = out["coords"].cpu().numpy()
    assert coords.shape == (g.n_points, 4)
    off = g.mesh_off_host
    for m, (side, mesh) in enumerate((("t", mt), ("s", ms))):
        feat = port.normalized_node_feature(mesh.point_scalars[name])
        assert np.array_equal(out["node_features"][off[m]:off[m + 1], 0].cpu().numpy(), feat)
        a = port.adjacency(port.feature_augmented_points(mesh.points, [feat]), mesh.tris)
        data, cols, indptr = _csr_rows(g, m)
        assert np.array_equal(data, a.data) and np.array_equal(cols, a.indices) and np.array_equal(indptr, a.indptr)
        gold = np.sort(golden["5k_feat_%s_eig_vals" % side])
        assert np.max(np.abs(vals[m, :6] - gold) / gold) <= 1e-6
        exp = _expected_coords(out, m, 0, mesh, a, [feat], 3, True, False, True)
        assert np.array_equal(coords[off[m]:off[m + 1]], exp)
