"""Batched ICP pre-alignment (``focusr_icp_batch``, ``SpectralBatch(icp_register_first=True)``): every pair's result is
bit-for-bit that of the one-pair call, the tile-pruned closest-point search agrees with the oracle's brute force where
pruning is hardest, and the spectral stage run after ICP equals the one run on pre-moved points."""
import numpy as np
import pytest

import pyfocusr_b200.mesh as fmesh
from oracle import icp_port as ip


def _rot(rv):
    from scipy.spatial.transform import Rotation

    return Rotation.from_rotvec(rv).as_matrix()


def _misalign(points, deg, axis, shift):
    axis = np.asarray(axis, dtype=np.float64)
    return points @ _rot(np.deg2rad(deg) * axis / np.linalg.norm(axis)).T + np.asarray(shift, dtype=np.float64)


def _pack(pairs):
    """[(fixed points, fixed tris, moving points, moving tris)] -> batch layout: meshes fixed_0, moving_0, fixed_1, ..."""
    pts, tris, off, toff = [], [], [0], [0]
    for fp, ft, mp, mt in pairs:
        for p, t in ((fp, ft), (mp, mt)):
            tris.append(np.asarray(t, dtype=np.int64) + off[-1])
            pts.append(np.asarray(p, dtype=np.float64))
            off.append(off[-1] + len(p))
            toff.append(toff[-1] + len(t))
    P = len(pairs)
    return (np.concatenate(pts), np.concatenate(tris).astype(np.int32), np.array(off, dtype=np.int32),
            np.array(toff, dtype=np.int32), np.arange(0, 2 * P, 2, dtype=np.int32), np.arange(1, 2 * P, 2, dtype=np.int32))


# --------------------------------------------------------------------------------------------- CPU
def test_bad_icp_mode_raises_type_error():
    from pyfocusr_b200 import SpectralBatch

    with pytest.raises(TypeError):
        SpectralBatch(icp_register_first=True, icp_registration_mode="affine")
    SpectralBatch(icp_registration_mode="similarity")


def test_triangle_ranges_from_grouped_tris():
    import torch

    from pyfocusr_b200 import SpectralBatch

    a, b = fmesh.icosphere(2), fmesh.icosphere(3)
    pts, tris, off, P = SpectralBatch.pack_meshes([a, b], [b, a])
    toff = SpectralBatch.tri_offsets(tris, off)
    assert toff.tolist() == np.cumsum([0, 80, 180, 180, 80]).tolist()
    shuffled = tris[torch.from_numpy(np.random.RandomState(0).permutation(tris.shape[0]))]
    with pytest.raises(ValueError):
        SpectralBatch.tri_offsets(shuffled, off)
    straddling = tris.clone()
    straddling[0, 0] = int(off[1])  # a triangle with vertices in two meshes
    with pytest.raises(ValueError):
        SpectralBatch.tri_offsets(straddling, off)
    swapped = torch.cat([tris[80:260], tris[:80], tris[260:]])  # every triangle whole, meshes out of order
    with pytest.raises(ValueError):
        SpectralBatch.tri_offsets(swapped, off)


def test_landmark_rule_matches_oracle(monkeypatch):
    from pyfocusr_b200 import _device

    seen = []
    real = ip.closest_points_on_mesh

    def spy(points, *a, **k):
        seen.append(np.array(points))
        return real(points, *a, **k)

    monkeypatch.setattr(ip, "closest_points_on_mesh", spy)
    tm = fmesh.icosphere(2)
    for n, ml in ((40, 57), (57, 57), (58, 57), (1999, 1000), (4002, 1000), (15212, 1000), (3000, 1000)):
        src = np.random.RandomState(n).randn(n, 3)
        seen.clear()
        ip.icp_transform(tm.points, tm.tris, src, max_iterations=1, max_landmarks=ml, start_by_matching_centroids=False)
        step, count = _device.icp_landmarks(n, ml)
        assert np.array_equal(seen[0], src[np.arange(count) * step]), (n, ml)


# --------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch():
    import torch as t

    if not t.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return t


@pytest.fixture(scope="module")
def meshes():
    axes = (43.0, 25.0, 33.0)
    return dict(ell8a=fmesh.perturbed_ellipsoid(8, 0, semi_axes=axes), ell8b=fmesh.perturbed_ellipsoid(8, 1, semi_axes=axes),
                ell20a=fmesh.perturbed_ellipsoid(20, 2, semi_axes=axes), ell20b=fmesh.perturbed_ellipsoid(20, 3, semi_axes=axes),
                ico=fmesh.icosphere(12, radius=30.0), ell12a=fmesh.perturbed_ellipsoid(12, 4, semi_axes=axes),
                ell12b=fmesh.perturbed_ellipsoid(12, 5, semi_axes=axes), ell12c=fmesh.perturbed_ellipsoid(12, 6, semi_axes=axes),
                ell12d=fmesh.perturbed_ellipsoid(12, 7, semi_axes=axes))


def _four_pairs(meshes, shipped):
    """642 / 4002 / 1442 / 15k moving points: step 1, n not divisible by the landmark count, the open 15k pair."""
    m, t15, s15 = meshes, shipped["target_mesh_15k"], shipped["source_mesh_15k"]
    return [(m["ell8a"].points, m["ell8a"].tris, _misalign(m["ell8b"].points, 60, [1, 2, 0.5], [5, -3, 2]), m["ell8b"].tris),
            (m["ell20a"].points, m["ell20a"].tris, _misalign(m["ell20b"].points, 35, [-1, 0.3, 1], [-2, 4, 1]), m["ell20b"].tris),
            (m["ico"].points, m["ico"].tris, _misalign(1.05 * m["ico"].points, 45, [0, 1, 1], [1, 1, -6]), m["ico"].tris),
            (t15.points, t15.tris, _misalign(s15.points, 20, [0.2, -1, 0.4], [3, 2, -4]), s15.tris)]


@pytest.mark.gpu
@pytest.mark.parametrize("similarity", [False, True])
@pytest.mark.parametrize("match", [True, False])
@pytest.mark.parametrize("max_landmarks", [57, 1000])
def test_batch_equals_single_pair_bitwise(torch, meshes, shipped_meshes, similarity, match, max_landmarks):
    from pyfocusr_b200 import _device

    pairs = _four_pairs(meshes, shipped_meshes)
    pts, tris, off, toff, fixed, moving = _pack(pairs)
    kw = dict(max_iterations=25, max_landmarks=max_landmarks, similarity=similarity, start_by_matching_centroids=match)
    mats, moved = _device.icp_batch(pts, tris, off, toff, fixed, moving, **kw)
    moved = moved.cpu().numpy()
    assert mats.shape == (4, 4, 4)
    for p, (fp, ft, mp, mt) in enumerate(pairs):
        mat1, moved1 = _device.icp(fp, ft, mp, **kw)
        assert np.array_equal(mats[p], mat1), p
        assert np.array_equal(moved[off[2 * p + 1]:off[2 * p + 2]], moved1.cpu().numpy()), p
        assert np.array_equal(moved[off[2 * p]:off[2 * p + 1]], fp), p  # fixed meshes are copied unchanged


@pytest.mark.gpu
@pytest.mark.parametrize("similarity", [False, True])
def test_batch_matches_oracle(torch, meshes, similarity):
    """test_icp.py's misalignment size (about 0.2 rad), horizons and tolerances, for the nu <= 20 pairs of a batch."""
    from pyfocusr_b200 import _device

    m = meshes
    sc = 1.08 if similarity else 1.0
    pairs = [(m["ell8a"].points, m["ell8a"].tris, sc * (m["ell8b"].points @ _rot([0.12, -0.1, 0.2]).T) + [4.0, -3.0, 2.0], m["ell8b"].tris),
             (m["ell20a"].points, m["ell20a"].tris, sc * (m["ell20b"].points @ _rot([-0.1, 0.15, 0.1]).T) + [-3.0, 2.0, 1.0], m["ell20b"].tris)]
    pts, tris, off, toff, fixed, moving = _pack(pairs)
    for iters, lm, tol in ((1, 1000, 1e-11), (12, 100, 1e-9), (40, 57, 1e-7)):
        mats, moved = _device.icp_batch(pts, tris, off, toff, fixed, moving, max_iterations=iters, max_landmarks=lm,
                                        similarity=similarity)
        moved = moved.cpu().numpy()
        for p, (fp, ft, mp, mt) in enumerate(pairs):
            ref = ip.icp_transform(fp, ft, mp, max_iterations=iters, max_landmarks=lm, similarity=similarity)
            assert np.max(np.abs(mats[p] - ref)) <= tol * 50.0, (iters, p, np.max(np.abs(mats[p] - ref)))
            assert np.max(np.abs(moved[off[2 * p + 1]:off[2 * p + 2]] - ip.apply_transform(mp, ref))) <= tol * 50.0
            assert np.array_equal(mats[p][3], [0.0, 0.0, 0.0, 1.0])


@pytest.mark.gpu
def test_pruning_exact_where_hardest(torch, meshes, shipped_meshes):
    """Distance ties at 0 across whole fans (source = target), a 60 degree misalignment (almost nothing prunable at
    first), and the open 15k target, against the oracle's brute force after one iteration; plus the 60 degree cases of
    the bit-identity batch after one iteration.  Where whole fans tie at distance 0, every tying triangle gives the same
    closest point (the shared vertex), so this cannot tell which triangle won: the tie rule itself is checked by
    test_ties_go_to_the_lowest_triangle_index."""
    from pyfocusr_b200 import _device

    m, t15, s15 = meshes, shipped_meshes["target_mesh_15k"], shipped_meshes["source_mesh_15k"]
    pairs = [(m["ell20a"].points, m["ell20a"].tris, m["ell20a"].points.copy(), m["ell20a"].tris),
             (m["ell20a"].points, m["ell20a"].tris, _misalign(m["ell20b"].points, 60, [1, -1, 0.5], [2, 3, -1]), m["ell20b"].tris),
             (t15.points, t15.tris, _misalign(s15.points, 8, [0.3, 1, -0.2], [1, -2, 2]), s15.tris)]
    pairs += _four_pairs(meshes, shipped_meshes)[:1]
    pts, tris, off, toff, fixed, moving = _pack(pairs)
    mats, _ = _device.icp_batch(pts, tris, off, toff, fixed, moving, max_iterations=1, max_landmarks=1000)
    for p, (fp, ft, mp, mt) in enumerate(pairs):
        ref = ip.icp_transform(fp, ft, mp, max_iterations=1, max_landmarks=1000)
        assert np.max(np.abs(mats[p] - ref)) <= 1e-11 * 50.0, (p, np.max(np.abs(mats[p] - ref)))


def _spectral_kw():
    return dict(n_coords_spectral_ordering=1000, graph_smoothing_iterations=30, projection_smooth_iterations=10)


def _misaligned_pairs(meshes):
    m = meshes
    targets = [m["ell12a"], m["ell12c"]]
    sources = [fmesh.PolyData(_misalign(m["ell12b"].points, 25, [1, 0.5, -0.3], [4, -2, 3]), m["ell12b"].tris),
               fmesh.PolyData(_misalign(m["ell12d"].points, 15, [-0.2, 1, 0.6], [-3, 1, 2]), m["ell12d"].tris)]
    return targets, sources


@pytest.mark.gpu
@pytest.mark.parametrize("target_to_source,mode", [(False, "rigid"), (True, "rigid"), (False, "similarity")])
def test_spectral_batch_with_icp_equals_premoved(torch, meshes, target_to_source, mode):
    from pyfocusr_b200 import SpectralBatch, _device

    targets, sources = _misaligned_pairs(meshes)
    sb = SpectralBatch(icp_register_first=True, icp_registration_mode=mode, icp_reg_target_to_source=target_to_source,
                       **_spectral_kw())
    pts, tris, off, P = sb.pack_meshes(targets, sources)
    sizes = np.diff(off)
    rng = np.random.RandomState(3)
    idx_t, idx_s = sb.sample_indices(sizes[:P], rng), sb.sample_indices(sizes[P:], rng)
    dpts = pts.cuda()
    before = dpts.clone()
    out = sb.run(dpts, tris, off, P, idx_t=idx_t, idx_s=idx_s)   # triangle ranges derived from the grouped tris
    torch.cuda.synchronize()
    assert torch.equal(dpts, before)

    premoved = pts.clone().numpy()
    mats = []
    for p in range(P):
        fixed, moving = (sources[p], targets[p]) if target_to_source else (targets[p], sources[p])
        mrow = p if target_to_source else P + p
        mat, moved = _device.icp(fixed.points, fixed.tris, moving.points, max_iterations=100, max_landmarks=1000,
                                 similarity=mode == "similarity")
        premoved[off[mrow]:off[mrow + 1]] = moved.cpu().numpy()
        mats.append(mat)
    ref = SpectralBatch(**_spectral_kw()).run(torch.from_numpy(premoved).cuda(), tris, off, P, idx_t=idx_t, idx_s=idx_s)
    assert ref["icp_matrices"] is None
    assert out["icp_matrices"].dtype == torch.float64 and out["icp_matrices"].shape == (P, 4, 4)
    assert np.array_equal(out["icp_matrices"].cpu().numpy(), np.stack(mats))
    for k in ("final_idx", "weighted_avg_transformed_points", "eig_vecs", "smoothed_target_coords"):
        assert torch.equal(out[k], ref[k]), k


@pytest.mark.gpu
def test_concurrent_sub_batches_with_icp_equal_separate_runs(torch, meshes):
    from pyfocusr_b200 import SpectralBatch

    targets, sources = _misaligned_pairs(meshes)
    kw = dict(icp_register_first=True, **_spectral_kw())
    sb = SpectralBatch(**kw)
    packed = [sb.pack_meshes(targets[:1], sources[:1]), sb.pack_meshes(targets[1:] + targets[:1], sources[1:] + sources[:1])]
    rng = np.random.RandomState(5)
    jobs = []
    for pts, tris, off, P in packed:
        sizes = np.diff(off)
        jobs.append(dict(points=pts, tris=tris, mesh_off_host=off, n_pairs=P, idx_t=sb.sample_indices(sizes[:P], rng),
                         idx_s=sb.sample_indices(sizes[P:], rng)))
    keys = ("final_idx", "weighted_avg_transformed_points", "eig_vecs", "smoothed_target_coords", "icp_matrices")
    for rep in range(2):
        outs = sb.run_concurrent(jobs)
        torch.cuda.synchronize()
        for job, out in zip(jobs, outs):
            ref = SpectralBatch(**kw)
            ref.overlap_smoothing = False
            alone = ref.run(**job)
            for k in keys:
                assert torch.equal(out[k], alone[k]), (rep, k)


@pytest.mark.gpu
def test_groups_of_32_equal_single_pairs(torch, meshes):
    """A batch large enough for 32 landmarks per warp (the one-pair calls use 4) gives every pair its one-pair result."""
    from pyfocusr_b200 import _device

    m = meshes
    rng = np.random.RandomState(11)
    pairs = [(m["ell12a"].points, m["ell12a"].tris,
              _misalign(m["ell12b"].points, rng.uniform(0, 40), rng.normal(size=3), rng.uniform(-5, 5, 3)), m["ell12b"].tris)
             for _ in range(40)]
    n_warps_of_32 = sum(-(-_device.icp_landmarks(len(p[2]), 1000)[1] // 32) for p in pairs)
    assert n_warps_of_32 >= 8 * torch.cuda.get_device_properties(0).multi_processor_count  # the premise of this test
    pts, tris, off, toff, fixed, moving = _pack(pairs)
    mats, _ = _device.icp_batch(pts, tris, off, toff, fixed, moving, max_iterations=20)
    for p, (fp, ft, mp, mt) in enumerate(pairs):
        assert np.array_equal(mats[p], _device.icp(fp, ft, mp, max_iterations=20)[0]), p


@pytest.mark.gpu
def test_ties_go_to_the_lowest_triangle_index(torch):
    """Landmarks exactly half-way between two parallel triangles: both give d^2 = 1 bit for bit, with different closest
    points, so the fitted translation (+1 or -1 in z) shows which triangle won.  The lower original index must win,
    whichever of the two comes first in the mesh."""
    from pyfocusr_b200 import _device

    tri = np.array([[0.0, 0.0], [4.0, 0.0], [0.0, 4.0]])
    up, down = np.c_[tri, np.ones(3)], np.c_[tri, -np.ones(3)]
    moving = np.array([[0.5, 0.5, 0.0], [2.0, 0.5, 0.0], [0.5, 2.0, 0.0], [1.0, 1.0, 0.0]])
    mt = np.array([[0, 1, 2], [0, 1, 3]], dtype=np.int32)
    for first, z in ((up, 1.0), (down, -1.0)):
        second = down if first is up else up
        fp = np.vstack([first, second])
        ft = np.array([[0, 1, 2], [3, 4, 5]], dtype=np.int32)
        pts, tris, off, toff, fixed, mov = _pack([(fp, ft, moving, mt)] * 3)
        mats, _ = _device.icp_batch(pts, tris, off, toff, fixed, mov, max_iterations=1, start_by_matching_centroids=False)
        ref = ip.icp_transform(fp, ft, moving, max_iterations=1, start_by_matching_centroids=False)
        assert abs(ref[2, 3] - z) < 1e-12
        for p in range(3):
            assert abs(mats[p][2, 3] - z) < 1e-12, (z, mats[p])


@pytest.mark.gpu
def test_large_batch_call_does_not_wait_for_the_device(torch):
    """focusr_icp_batch only enqueues work, also for batches of more than 250 pairs (500 sort segments): while the
    stream is still busy with earlier work, the call returns."""
    import time

    from pyfocusr_b200 import _device, _lib

    ico = fmesh.icosphere(2)
    P = 300
    pairs = [(ico.points, ico.tris, _misalign(ico.points, 10 + p % 7, [1, 0, 0], [0, 0, 0.1]), ico.tris) for p in range(P)]
    pts, tris, off, toff, fixed, moving = _pack(pairs)
    lib = _lib.load()
    nbytes = int(lib.focusr_icp_batch_workspace_bytes(_lib.ptr(off), _lib.ptr(toff), 2 * P, _lib.ptr(fixed), _lib.ptr(moving),
                                                      P, 1000))
    d = [torch.from_numpy(a).cuda() for a in (pts, tris, off, toff, fixed, moving)]
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    mats = torch.empty((P, 4, 4), dtype=torch.float64, device="cuda")
    moved = torch.empty_like(d[0])
    torch.cuda.synchronize()
    torch.cuda._sleep(int(3e9))  # about a second of device time ahead of the call on this stream
    t0 = time.perf_counter()
    _lib.call("focusr_icp_batch", _lib.ptr(d[0]), 2 * P * 42, _lib.ptr(d[1]), _lib.ptr(d[2]), _lib.ptr(off), _lib.ptr(d[3]),
              _lib.ptr(toff), 2 * P, _lib.ptr(d[4]), _lib.ptr(d[5]), _lib.ptr(fixed), _lib.ptr(moving), P, 1000, 5, 0, 1,
              _lib.ptr(mats), _lib.ptr(moved), _lib.ptr(ws), nbytes, _lib.stream_ptr())
    returned_after = time.perf_counter() - t0
    still_busy = not torch.cuda.current_stream().query()
    torch.cuda.synchronize()
    assert still_busy and returned_after < 0.3, returned_after
    fp, ft, mp, _ = pairs[P - 1]
    assert np.array_equal(mats[P - 1].cpu().numpy(), _device.icp(fp, ft, mp, max_iterations=5)[0])
