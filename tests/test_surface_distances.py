"""Surface distances (``focusr_closest_points`` / ``focusr_surface_distance_stats``, K14 in csrc/surface.cu;
``pyfocusr_b200.surface``; ``SpectralBatch(surface_distances=...)``): the tile-pruned search equals the brute force bit
for bit and agrees with ``oracle/surface_port.py``, mapped surfaces equal copies, and the batch keys are those of the
search on the run's own positions and triangles, with every pre-existing key unchanged."""
import numpy as np
import pytest

import pyfocusr_b200.mesh as fmesh
from oracle import surface_port as sp
from pyfocusr_b200 import SpectralBatch, surface_distances
from pyfocusr_b200.batch import SURFACE_POSITIONS

SPECTRAL_KW = dict(n_coords_spectral_ordering=1000, graph_smoothing_iterations=30, projection_smooth_iterations=10)
AXES = (43.0, 25.0, 33.0)
NEW_KEYS = ("source_to_target_surface_dist", "source_to_target_closest_points", "source_to_target_closest_tri",
            "target_to_source_surface_dist", "target_to_source_closest_tri", "surface_distance_stats")


# --------------------------------------------------------------------------------------------- CPU
def test_oracle_hand_cases():
    a, b, c = np.array([0.0, 0, 0]), np.array([2.0, 0, 0]), np.array([0.0, 2, 0])
    pts, tri = np.stack([a, b, c]), np.array([[0, 1, 2]])
    # over the face, beyond an edge, beyond a vertex
    for q, want in (([0.5, 0.5, 3.0], [0.5, 0.5, 0.0]), ([1.5, 1.5, 0.0], [1.0, 1.0, 0.0]), ([-1.0, -2.0, 1.0], [0.0, 0.0, 0.0])):
        cl, d2, win, _ = sp.closest_points([q], pts, tri)
        assert np.allclose(cl[0], want, atol=1e-15) and np.isclose(d2[0], np.sum((np.array(q) - want) ** 2)) and win[0] == 0
    # a triangle collapsed to a segment (a, a, b) and to a point (a, a, a): scored by its edges
    seg = np.array([[0, 0, 1]])
    cl, d2, _, _ = sp.closest_points([[1.0, 3.0, 0.0]], pts, seg)
    assert np.array_equal(cl[0], [1.0, 0.0, 0.0]) and d2[0] == 9.0
    cl, d2, _, _ = sp.closest_points([[1.0, 3.0, 0.0]], pts, np.array([[1, 1, 1]]))
    assert np.array_equal(cl[0], b) and d2[0] == 10.0
    # collinear: c on the segment a-b
    line = np.array([a, b, [1.0, 0.0, 0.0]])
    cl, d2, _, _ = sp.closest_points([[0.5, 1.0, 0.0]], line, np.array([[0, 1, 2]]))
    assert np.array_equal(cl[0], [0.5, 0.0, 0.0]) and d2[0] == 1.0
    # two triangles at equal distance: the lower index wins
    pts2 = np.array([[0.0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 2], [1, 0, 2], [0, 1, 2]])
    for tris, want in ((np.array([[0, 1, 2], [3, 4, 5]]), 0), (np.array([[3, 4, 5], [0, 1, 2]]), 0)):
        _, d2, win, second = sp.closest_points([[0.2, 0.2, 1.0]], pts2, tris)
        assert win[0] == want and d2[0] == second[0] == 1.0


def _lib():
    from pyfocusr_b200 import _lib

    return _lib.load(), _lib.ptr


def test_workspace_bytes_is_zero_for_invalid_descriptions():
    lib, ptr = _lib()
    i32 = lambda *v: np.array(v, dtype=np.int32)  # noqa: E731

    def size(poff, toff, qoff, seg):
        return int(lib.focusr_closest_points_workspace_bytes(ptr(poff), ptr(toff), poff.size - 1, ptr(qoff), qoff.size - 1,
                                                             ptr(seg)))

    poff, toff, qoff = i32(0, 3, 6, 9), i32(0, 1, 1, 2), i32(0, 5, 5, 9)
    assert size(poff, toff, qoff, i32(0, 2, 0)) > 0  # surface 1 has no triangles and no segment: fine; segment 1 empty
    assert size(poff, toff, qoff, i32(0, 1, 0)) == 0  # a mapped surface without triangles
    assert size(poff, toff, qoff, i32(0, 3, 0)) == 0  # surface index out of range
    assert size(poff, toff, qoff, i32(0, -1, 0)) == 0
    assert size(i32(0, 3, 2, 9), toff, qoff, i32(0, 2, 0)) == 0  # point offsets not monotone
    assert size(poff, i32(0, 2, 1, 2), qoff, i32(0, 2, 0)) == 0  # triangle offsets not monotone
    assert size(poff, toff, i32(0, 5, 4, 9), i32(0, 2, 0)) == 0  # query offsets not monotone
    assert size(poff, toff, i32(-1, 5, 5, 9), i32(0, 2, 0)) == 0
    assert int(lib.focusr_closest_points_workspace_bytes(ptr(poff), ptr(toff), 3, ptr(qoff), 0, ptr(i32(0)))) == 0
    assert int(lib.focusr_closest_points_workspace_bytes(None, ptr(toff), 3, ptr(qoff), 3, ptr(i32(0, 2, 0)))) == 0


def test_value_errors():
    for bad in ("weight", "", 1, True, ("weighted",)):
        with pytest.raises(ValueError, match="surface_distances must be"):
            SpectralBatch(surface_distances=bad)
    for ok in (None, "weighted", "nearest"):
        assert SpectralBatch(surface_distances=ok).surface_distances == ok
    assert set(SURFACE_POSITIONS) == {"weighted", "nearest"}
    m = fmesh.icosphere(2)
    with pytest.raises(ValueError, match="as many targets"):
        surface_distances([m, m], [m])
    with pytest.raises(ValueError, match="as many targets"):
        surface_distances([], [])
    for tris, msg in ((np.where(m.tris == 5, m.points.shape[0], m.tris), "outside"), (m.tris - 1, "outside"),
                      (np.zeros((0, 3), dtype=np.int64), "F >= 1")):
        with pytest.raises(ValueError, match=msg):
            surface_distances([m], [fmesh.PolyData(m.points, tris)])
        with pytest.raises(ValueError, match=msg):
            surface_distances([fmesh.PolyData(m.points, tris)], [m])


# --------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch():
    import torch as t

    if not t.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return t


def _queries(points, tris, seed, n_random=300):
    """far outside, well inside, exactly on vertices, on edge midpoints and near the surface"""
    rng = np.random.RandomState(seed)
    c = points.mean(0)
    ext = float(np.ptp(points, axis=0).max()) or 1.0
    far = c + rng.normal(size=(n_random // 3, 3)) * 5 * ext
    inside = c + (points[rng.randint(0, len(points), n_random // 3)] - c) * 0.3
    verts = points[rng.randint(0, len(points), n_random // 3)]
    t = tris[rng.randint(0, len(tris), n_random // 3)]
    edges = 0.5 * (points[t[:, 0]] + points[t[:, 1]])
    near = points[rng.randint(0, len(points), n_random // 3)] + rng.normal(size=(n_random // 3, 3)) * 0.05 * ext
    return np.concatenate([far, inside, verts, edges, near])


def _surfaces(shipped):
    """(points, tris) of surfaces of every kind the search must handle"""
    base = fmesh.icosphere(12)
    ell_t, _ = fmesh.ellipsoid_pair(0, 12, base=base)
    open15 = shipped["target_mesh_15k"]
    ico = fmesh.icosphere(3)
    ico_tris = ico.tris.copy()
    ico_tris[5] = [ico_tris[5][0]] * 2 + [ico_tris[5][1]]  # collapsed to a segment
    ico_tris[17] = [ico_tris[17][2]] * 3  # collapsed to a point
    ico_tris = np.concatenate([ico_tris, [[0, 1, 1], [3, 3, 3]]])
    small_p = np.array([[0.0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0.5], [2, 0, 0.2], [0, 2, -0.3]])
    small_t = np.array([[0, 1, 2], [1, 3, 2], [1, 4, 3], [2, 3, 5], [0, 0, 4]])
    one_p, one_t = np.array([[0.0, 0, 0], [3, 0.5, 0], [1, 2, 1]]), np.array([[0, 1, 2]])
    return [(ell_t.points, ell_t.tris), (open15.points, open15.tris), (ico.points, ico_tris), (small_p, small_t),
            (one_p, one_t)]


def _pack(surfs):
    pts = np.concatenate([p for p, _ in surfs])
    poff = np.cumsum([0] + [len(p) for p, _ in surfs]).astype(np.int32)
    toff = np.cumsum([0] + [len(t) for _, t in surfs]).astype(np.int32)
    tris = np.concatenate([np.asarray(t, dtype=np.int64) + o for (_, t), o in zip(surfs, poff[:-1])]).astype(np.int32)
    return pts, tris, poff, toff


def _search(torch, surfs, qlist, seg, brute=False):
    from pyfocusr_b200 import surface

    pts, tris, poff, toff = _pack(surfs)
    q = np.concatenate(qlist) if qlist else np.zeros((0, 3))
    qoff = np.cumsum([0] + [len(x) for x in qlist]).astype(np.int32)
    d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to("cuda", dt)  # noqa: E731
    cl, tri, dist = surface.closest_points(d(pts, torch.float64), d(tris, torch.int32), poff, toff, d(q, torch.float64), qoff,
                                           seg, brute_force=brute)
    return cl.cpu().numpy(), tri.cpu().numpy(), dist.cpu().numpy(), qoff


@pytest.mark.gpu
def test_pruned_equals_brute_force_oracle_and_copies(torch, shipped_meshes):
    surfs = _surfaces(shipped_meshes)
    qs = [_queries(p, t, k) for k, (p, t) in enumerate(surfs)]
    qs.append(np.concatenate([_queries(surfs[1][0], surfs[1][1], 99), surfs[0][0][:50]]))  # surface 1 again, other queries
    qs.append(np.zeros((0, 3)))  # an empty segment
    # every surface mapped, surface 1 by two segments; an unmapped surface with triangles in front (index 0)
    extra = (surfs[3][0] + 100.0, surfs[3][1])
    all_surfs = [extra] + surfs
    seg = np.array([1, 2, 3, 4, 5, 2, 4], dtype=np.int32)
    pruned = _search(torch, all_surfs, qs, seg)
    brute = _search(torch, all_surfs, qs, seg, brute=True)
    again = _search(torch, all_surfs, qs, seg)
    for x, y, z in zip(pruned[:3], brute[:3], again[:3]):
        assert np.array_equal(x, y) and np.array_equal(x, z)
    cl, tri, dist, qoff = pruned
    for s, m in enumerate(seg):
        r = slice(qoff[s], qoff[s + 1])
        if qoff[s] == qoff[s + 1]:
            continue
        # one segment alone, on its own copy of the surface, equals the segment inside the batch
        alone = _search(torch, [all_surfs[m]], [qs[s]], np.array([0], dtype=np.int32))
        for x, y in zip(alone[:3], (cl[r], tri[r], dist[r])):
            assert np.array_equal(x, y), (s, m)
        p, t = all_surfs[m]
        o_cl, o_d2, o_win, o_second = sp.closest_points(qs[s], p, t)
        tol = 1e-12 * float(np.ptp(p, axis=0).max())
        assert np.max(np.abs(dist[r] - np.sqrt(o_d2))) <= tol, (s, m)
        clear = np.sqrt(o_second) - np.sqrt(o_d2) > tol
        assert np.array_equal(tri[r][clear], o_win[clear]), (s, m)
        assert np.max(np.abs(cl[r][clear] - o_cl[clear])) <= 1e-9 * max(1.0, float(np.abs(p).max()))


@pytest.mark.gpu
def test_coincident_triangles_lowest_index_wins(torch):
    ico = fmesh.icosphere(2)
    t = ico.tris.copy()
    dup = t[7].copy()
    t[30], t[55] = dup, dup  # triangles 7, 30 and 55 coincide
    c = ico.points[dup].mean(0)
    q = np.concatenate([c[None] * s for s in (0.5, 1.0, 1.5, 3.0)])
    q = np.concatenate([q, ico.points[dup]])  # and the three vertices (fans of ties at d = 0)
    for brute in (False, True):
        _, tri, dist, _ = _search(torch, [(ico.points, t)], [q], np.array([0], dtype=np.int32), brute)
        assert np.all(tri[:4] == 7)
        for k, v in enumerate(dup):
            assert dist[4 + k] == 0.0 and tri[4 + k] == np.nonzero((t == v).any(1))[0].min()


@pytest.mark.gpu
def test_large_call_does_not_wait_for_the_device(torch):
    import time

    from pyfocusr_b200 import _lib, surface

    ico = fmesh.icosphere(4)
    P = 300
    pts = torch.from_numpy(np.concatenate([ico.points * (1 + 0.01 * p) for p in range(P)])).cuda()
    n, f = ico.points.shape[0], ico.tris.shape[0]
    tris = torch.from_numpy(np.concatenate([ico.tris + p * n for p in range(P)]).astype(np.int32)).cuda()
    poff, toff = np.arange(P + 1, dtype=np.int32) * n, np.arange(P + 1, dtype=np.int32) * f
    seg = np.arange(P)[::-1].copy()
    surface.closest_points(pts, tris, poff, toff, pts, poff, seg)  # warm
    torch.cuda.synchronize()
    torch.cuda._sleep(int(3e9))
    t0 = time.perf_counter()
    _, tri, dist = surface.closest_points(pts, tris, poff, toff, pts, poff, seg)
    returned_after = time.perf_counter() - t0
    still_busy = not torch.cuda.current_stream().query()
    torch.cuda.synchronize()
    assert still_busy and returned_after < 0.3, returned_after
    assert _lib.launch_count() > 0 and bool(torch.isfinite(dist).all())


@pytest.mark.gpu
def test_known_answers(torch):
    m = fmesh.perturbed_ellipsoid(8, 3, semi_axes=AXES)
    out = surface_distances([m], [m])
    assert float(out["source_to_target_surface_dist"].abs().max()) == 0.0
    assert float(out["target_to_source_surface_dist"].abs().max()) == 0.0
    assert np.array_equal(out["surface_distance_stats"].cpu().numpy(), np.zeros((1, 6)))
    # a flat grid and a copy of it shifted by delta along its normal
    g = np.stack(np.meshgrid(np.arange(12.0), np.arange(9.0), indexing="ij"), -1).reshape(-1, 2)
    pts = np.concatenate([g, np.zeros((len(g), 1))], 1)
    idx = np.arange(12 * 9).reshape(12, 9)
    quads = np.stack([idx[:-1, :-1], idx[1:, :-1], idx[1:, 1:], idx[:-1, 1:]], -1).reshape(-1, 4)
    tris = np.concatenate([quads[:, [0, 1, 2]], quads[:, [0, 2, 3]]])
    delta = 0.37
    out = surface_distances([fmesh.PolyData(pts + [0, 0, delta], tris)], [fmesh.PolyData(pts, tris)])
    for k in ("source_to_target_surface_dist", "target_to_source_surface_dist"):
        assert np.max(np.abs(out[k].cpu().numpy() - delta)) <= 1e-12
    assert np.allclose(out["surface_distance_stats"].cpu().numpy(), delta, rtol=0, atol=1e-12)


def _pairs(n, seed0=0, nu=8):
    base = fmesh.icosphere(nu)
    return [fmesh.perturbed_ellipsoid(nu, seed0 + k, semi_axes=AXES, base=base) for k in range(n)]


@pytest.mark.gpu
def test_batch_keys_and_unchanged_outputs(torch):
    from pyfocusr_b200 import surface

    t, s = _pairs(2, 0), _pairs(2, 10)
    ref = SpectralBatch(**SPECTRAL_KW).run_meshes(t, s)
    sb = SpectralBatch(**SPECTRAL_KW, surface_distances="weighted")
    out = sb.run_meshes(t, s, record_events=True)
    assert "surface" in sb.timings
    assert set(out) == set(ref) | set(NEW_KEYS)
    for k, v in ref.items():
        if isinstance(v, torch.Tensor):
            assert torch.equal(v, out[k]), k
    P, off = 2, out["pair_mesh_off"]
    X = out["weighted_avg_transformed_points"]
    src_off = (off[P:] - off[P]).astype(np.int32)
    g = out["graph"]
    toff = np.cumsum([0] + [m.tris.shape[0] for m in t + s]).astype(np.int32)
    cl, tri, dist = surface.closest_points(g.points, g.tris, g.mesh_off_host, toff, X, src_off, np.arange(P))
    assert torch.equal(cl, out["source_to_target_closest_points"]) and torch.equal(tri, out["source_to_target_closest_tri"])
    assert torch.equal(dist, out["source_to_target_surface_dist"])
    s_tris = torch.from_numpy(np.concatenate([m.tris + o for m, o in zip(s, src_off[:-1])]).astype(np.int32)).cuda()
    s_toff = np.cumsum([0] + [m.tris.shape[0] for m in s]).astype(np.int32)
    _, tri2, dist2 = surface.closest_points(X, s_tris, src_off, s_toff, g.points[:off[P]], off[:P + 1], np.arange(P))
    assert torch.equal(tri2, out["target_to_source_closest_tri"]) and torch.equal(dist2, out["target_to_source_surface_dist"])
    a, b = dist.cpu().numpy(), dist2.cpu().numpy()
    stats = out["surface_distance_stats"].cpu().numpy()
    for p in range(P):
        x, y = a[src_off[p]:src_off[p + 1]], b[off[p]:off[p + 1]]
        want = [x.mean(), x.max(), y.mean(), y.max(), (x.sum() + y.sum()) / (x.size + y.size), max(x.max(), y.max())]
        assert np.allclose(stats[p], want, rtol=1e-12, atol=0)
    # the default option adds nothing
    assert not set(NEW_KEYS) & set(ref)


@pytest.mark.gpu
def test_nearest_positions_lie_on_the_target(torch):
    t, s = _pairs(2, 0), _pairs(2, 10)
    out = SpectralBatch(**SPECTRAL_KW, surface_distances="nearest").run_meshes(t, s)
    assert float(out["source_to_target_surface_dist"].abs().max()) == 0.0
    off = out["pair_mesh_off"]
    P = 2
    tri = out["source_to_target_closest_tri"].cpu().numpy()
    idx = out["final_idx"].cpu().numpy()
    for p in range(P):
        r = slice(off[P + p] - off[P], off[P + p + 1] - off[P])
        first = np.full(t[p].points.shape[0], np.iinfo(np.int64).max)
        np.minimum.at(first, t[p].tris.reshape(-1), np.repeat(np.arange(t[p].tris.shape[0]), 3))
        assert np.array_equal(tri[r], first[idx[r]])


@pytest.mark.gpu
def test_shared_meshes_equal_repeated_meshes(torch):
    a, b, c = _pairs(3, 30)
    sb = SpectralBatch(**SPECTRAL_KW, surface_distances="weighted")
    got = sb.run_mesh_pairs([a, b, c], [(0, 1), (0, 2), (2, 1)])
    want = sb.run_meshes([a, a, c], [b, c, b])
    for k in NEW_KEYS:
        assert torch.equal(got[k], want[k]), k
    got = sb.run_meshes([a], [b, c], target_of_pair=[0, 0])
    want = sb.run_meshes([a, a], [b, c])
    for k in NEW_KEYS:
        assert torch.equal(got[k], want[k]), k


@pytest.mark.gpu
def test_icp_concurrent_and_mixed_sizes(torch):
    small, large = _pairs(2, 40, nu=6), _pairs(2, 50, nu=8)
    t, s = [small[0], large[0]], [large[1], small[1]]  # every pair mixes sizes
    sb = SpectralBatch(**SPECTRAL_KW, surface_distances="nearest", icp_register_first=True)
    one = sb.run_meshes(t, s)
    assert float(one["source_to_target_surface_dist"].abs().max()) == 0.0  # on the ICP-moved target: nearest vertices
    both = sb.run_concurrent([dict(zip(("points", "tris", "mesh_off_host", "n_pairs"), SpectralBatch.pack_meshes(t, s)),
                                   tri_off_host=np.cumsum([0] + [m.tris.shape[0] for m in t + s]).astype(np.int32))] * 2)
    for out in both:
        for k in NEW_KEYS:
            assert torch.equal(out[k], one[k]), k
    tt = one["target_to_source_surface_dist"]
    assert bool(torch.isfinite(tt).all()) and tt.shape[0] == one["pair_mesh_off"][2]


@pytest.mark.gpu
def test_shape_model_reports_stats(torch):
    base = fmesh.icosphere(8)
    subjects = [fmesh.perturbed_ellipsoid(8, 20 + i, semi_axes=AXES, base=base) for i in range(4)]
    template = fmesh.perturbed_ellipsoid(7, 99, semi_axes=AXES)
    off = SpectralBatch(**SPECTRAL_KW).build_shape_model(subjects, template, rounds=2, template_tolerance=0.0, n_modes=2)
    on = SpectralBatch(**SPECTRAL_KW, surface_distances="weighted").build_shape_model(subjects, template, rounds=2,
                                                                                       template_tolerance=0.0, n_modes=2)
    for k in ("mean_points", "aligned", "procrustes_matrices", "modes"):
        assert torch.equal(on[k], off[k]), k
    for k in ("variances", "scores"):
        assert np.array_equal(on[k], off[k]), k
    assert len(on["rounds"]) == len(off["rounds"]) == 2
    for r_on, r_off in zip(on["rounds"], off["rounds"]):
        assert "surface_distance_stats" not in r_off
        st = r_on["surface_distance_stats"]
        assert isinstance(st, np.ndarray) and st.shape == (4, 6) and np.all(np.isfinite(st)) and np.all(st >= 0)
        assert np.all(st[:, 4] <= st[:, 5])
