"""Shape models (``pyfocusr_b200.shape``, ``SpectralBatch.build_shape_model``, K13 in csrc/shape.cu): the Procrustes fit
against vtkLandmarkTransform's numpy restatement, GPA and PCA against ``oracle/shape_port.py``, and the cohort workflow
end to end against the registration it is built on."""
import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import pyfocusr_b200.mesh as fmesh
from oracle import shape_port
from oracle.icp_port import landmark_transform
from pyfocusr_b200 import shape
from pyfocusr_b200.batch import SpectralBatch

SPECTRAL_KW = dict(n_coords_spectral_ordering=1000, graph_smoothing_iterations=30, projection_smooth_iterations=10)


def similarity_copies(x, n, seed, noise=0.0, scale_range=(0.8, 1.25)):
    """n copies of the shape x (N, 3), each rotated, scaled, translated and optionally jittered"""
    rng = np.random.RandomState(seed)
    out = []
    for _ in range(n):
        r = Rotation.from_rotvec(rng.normal(size=3) * 0.6).as_matrix()
        s, t = rng.uniform(*scale_range), rng.normal(size=3) * 5.0
        out.append(s * x @ r.T + t + noise * rng.normal(size=x.shape))
    return np.stack(out)


# --------------------------------------------------------------------------------------------- CPU
def test_argument_rules():
    a, b, t = fmesh.icosphere(2), fmesh.icosphere(3), fmesh.icosphere(4)
    sb = SpectralBatch(**SPECTRAL_KW)
    for kw, msg in ((dict(subjects=[]), "at least one subject"),
                    (dict(procrustes="affine"), "'rigid' or 'similarity'"),
                    (dict(align_type="closest"), "'weighted' or 'nearest'"),
                    (dict(n_modes=0), "n_modes"),
                    (dict(n_modes=2.5), "n_modes"),
                    (dict(rounds=0), "rounds")):
        args = dict(subjects=[a, b], template=t)
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            sb.build_shape_model(**args)
    icp = SpectralBatch(icp_register_first=True, **SPECTRAL_KW)
    with pytest.raises(ValueError, match="icp_reg_target_to_source=True"):
        icp.build_shape_model([a, b], t)
    with pytest.raises(ValueError, match="'rigid' or 'similarity'"):
        shape.procrustes(np.zeros((2, 4, 3)), np.zeros((4, 3)), mode="affine")
    with pytest.raises(ValueError, match="n_modes"):
        shape.pca(np.zeros((2, 4, 3)), np.zeros((4, 3)), 0)


@pytest.mark.parametrize("similarity", [False, True])
def test_oracle_gpa_recovers_known_mean(similarity):
    rng = np.random.RandomState(3)
    x = rng.normal(size=(60, 3)) * np.array([4.0, 2.0, 1.0])
    scale_range = (0.8, 1.25) if similarity else (1.0, 1.0)
    configs = similarity_copies(x, 9, 1, scale_range=scale_range)
    reference = similarity_copies(x, 1, 2, scale_range=scale_range)[0]  # the mean that fits the reference best
    g = shape_port.procrustes(configs, reference, similarity)
    assert g["iterations"] <= 2
    scale = shape_port.rms(reference, reference.mean(0)[None])
    assert np.max(np.abs(g["mean"] - reference)) <= 1e-12 * scale
    assert np.max(np.abs(g["aligned"] - reference[None])) <= 1e-12 * scale


# --------------------------------------------------------------------------------------------- GPU
def _dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))


@pytest.mark.gpu
@pytest.mark.parametrize("similarity", [False, True])
def test_fit_matches_landmark_transform(similarity):
    from pyfocusr_b200 import _device

    rng = np.random.RandomState(5)
    ref = rng.normal(size=(300, 3)) * 10.0
    configs = similarity_copies(ref, 6, 7, noise=0.3)
    mats, aligned = _device.procrustes_fit(_dev(configs), _dev(ref), similarity)
    mats, aligned = mats.cpu().numpy(), aligned.cpu().numpy()
    for p in range(configs.shape[0]):
        want = landmark_transform(configs[p], ref, similarity)
        assert _rel(mats[p], want) <= 1e-12, p
        assert _rel(aligned[p], shape_port.apply(want, configs[p])) <= 1e-12, p
    # degenerate sets: one point; coincident points (dyadic coordinates, so every centroid is exact) on either side
    one_cfg, one_ref = rng.normal(size=(3, 1, 3)), rng.normal(size=(1, 3))
    same = np.tile(np.array([[1.5, -2.25, 0.75]]), (64, 1))
    cases = [(one_cfg, one_ref), (same[None], rng.normal(size=(64, 3))), (rng.normal(size=(1, 64, 3)), same)]
    for cfg, r in cases:
        mats, aligned = _device.procrustes_fit(_dev(cfg), _dev(r), similarity)
        mats = mats.cpu().numpy()
        for p in range(cfg.shape[0]):
            want = landmark_transform(cfg[p], r, similarity)
            assert np.array_equal(want[:3, :3], np.eye(3))
            assert np.array_equal(mats[p][:3, :3], np.eye(3)) and np.array_equal(mats[p][3], [0, 0, 0, 1])
            assert _rel(mats[p], want) <= 1e-12


@pytest.mark.gpu
def test_fit_does_not_depend_on_batch():
    import torch

    from pyfocusr_b200 import _device

    rng = np.random.RandomState(8)
    ref = rng.normal(size=(1000, 3)) * 20.0
    configs = _dev(similarity_copies(ref, 7, 9, noise=0.5))
    mats, aligned = _device.procrustes_fit(configs, _dev(ref), True)
    for p in range(7):
        m1, a1 = _device.procrustes_fit(configs[p:p + 1].contiguous(), _dev(ref), True)
        assert torch.equal(m1[0], mats[p]) and torch.equal(a1[0], aligned[p]), p


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["rigid", "similarity"])
def test_gpa_matches_oracle(mode):
    import torch

    rng = np.random.RandomState(11)
    x = rng.normal(size=(400, 3)) * np.array([30.0, 20.0, 10.0])
    configs = similarity_copies(x, 10, 12, noise=0.8, scale_range=(0.8, 1.25) if mode == "similarity" else (1.0, 1.0))
    reference = x + rng.normal(size=x.shape)
    got = shape.procrustes(_dev(configs), _dev(reference), mode)
    want = shape_port.procrustes(configs, reference, mode == "similarity")
    assert got["iterations"] == want["iterations"] > 1
    for k in ("mean", "aligned", "matrices"):
        assert np.max(np.abs(got[k].cpu().numpy() - want[k])) <= 1e-10, k
    again = shape.procrustes(_dev(configs), _dev(reference), mode)
    for k in ("mean", "aligned", "matrices"):
        assert torch.equal(got[k], again[k]), k
    assert np.array_equal(got["changes"], again["changes"])


@pytest.mark.gpu
def test_pca_matches_oracle():
    import torch

    rng = np.random.RandomState(13)
    P, N = 12, 500
    base = rng.normal(size=(N, 3)) * 10.0
    # a few strong directions and a little noise, so the eigenvalues are well separated
    dirs = rng.normal(size=(4, N, 3))
    aligned = base[None] + np.einsum("pk,knd->pnd", rng.normal(size=(P, 4)) * np.array([8.0, 4.0, 2.0, 1.0]), dirs)
    aligned += 0.05 * rng.normal(size=aligned.shape)
    mean = aligned.mean(0)
    got = shape.pca(_dev(aligned), _dev(mean), P)
    want = shape_port.pca(aligned, mean, P)
    K = P - 1
    assert got["modes"].shape == (K, N, 3) and got["variances"].shape == (K,) and got["scores"].shape == (P, K)
    assert np.all(np.abs(got["variances"] / want["variances"] - 1.0) <= 1e-10)
    modes = got["modes"].cpu().numpy()
    assert np.max(np.abs(modes - want["modes"])) <= 1e-9
    assert np.max(np.abs(got["scores"] - want["scores"])) <= 1e-9
    # unit norm up to the accuracy of the Gram eigenvalues (eps * lambda_max / lambda_k)
    assert np.allclose(np.linalg.norm(modes.reshape(K, -1), axis=1), 1.0, rtol=0, atol=1e-10)
    recon = mean[None] + np.einsum("pk,knd->pnd", got["scores"], modes)
    assert np.max(np.abs(recon - aligned)) <= 1e-9
    few = shape.pca(_dev(aligned), _dev(mean), 3)
    assert torch.equal(few["modes"], got["modes"][:3]) and np.array_equal(few["variances"], got["variances"][:3])


def _cohort():
    base = fmesh.icosphere(8)
    subjects = [fmesh.perturbed_ellipsoid(8, 20 + i, semi_axes=(43.0, 25.0, 33.0), base=base) for i in range(6)]
    template = fmesh.perturbed_ellipsoid(7, 99, semi_axes=(43.0, 25.0, 33.0))  # another frequency: another topology
    return subjects, template


def _rounds_by_hand(sb, subjects, template, n_rounds, key, mode="similarity"):
    """the rounds of build_shape_model, one call at a time, each round's GPA also run by the oracle"""
    P = len(subjects)
    tmpl, rounds = template, []
    for _ in range(n_rounds):
        out = sb.run_mesh_pairs(subjects + [tmpl], [(m, P) for m in range(P)])
        configs = out[key].view(P, -1, 3)
        got = shape.procrustes(configs, _dev(tmpl.points), mode)
        want = shape_port.procrustes(configs.cpu().numpy(), tmpl.points, mode == "similarity")
        mean = got["mean"].cpu().numpy()
        rounds.append(dict(gpa=got, oracle=want, change=float(np.sqrt(np.mean(np.sum((mean - tmpl.points) ** 2, 1)))),
                           icp=out["icp_matrices"]))
        tmpl = fmesh.PolyData(mean, template.tris)
    return rounds


@pytest.mark.gpu
@pytest.mark.parametrize("icp", [False, True])
def test_build_shape_model_end_to_end(icp):
    import torch

    subjects, template = _cohort()
    kw = dict(icp_register_first=True, icp_reg_target_to_source=True) if icp else {}
    sb = SpectralBatch(**SPECTRAL_KW, **kw)
    by_hand = _rounds_by_hand(sb, subjects, template, 3, "weighted_avg_transformed_points")
    for r in by_hand:  # each round's GPU mean against the oracle's GPA on the same configurations
        assert r["gpa"]["iterations"] == r["oracle"]["iterations"]
        assert np.max(np.abs(r["gpa"]["mean"].cpu().numpy() - r["oracle"]["mean"])) <= 1e-10
    changes = [r["change"] for r in by_hand]
    tol = changes[1]
    stop = next(k for k, c in enumerate(changes) if c <= tol) + 1
    model = sb.build_shape_model(subjects, template, rounds=5, template_tolerance=tol, n_modes=3)
    assert len(model["rounds"]) == stop
    last = by_hand[stop - 1]["gpa"]
    # template k+1 is mean k on the template's triangles, and every round is the one run by hand
    assert torch.equal(model["mean_points"], last["mean"]) and torch.equal(model["aligned"], last["aligned"])
    assert torch.equal(model["procrustes_matrices"], last["matrices"])
    assert np.array_equal(model["mean_mesh"].points, last["mean"].cpu().numpy())
    assert np.array_equal(model["mean_mesh"].tris, template.tris)
    for got, want in zip(model["rounds"], by_hand):
        assert got["template_change"] == want["change"] and got["gpa_iterations"] == want["gpa"]["iterations"]
        assert np.array_equal(got["gpa_changes"], want["gpa"]["changes"])
        assert ("icp_matrices" in got) == icp
        if icp:
            assert torch.equal(got["icp_matrices"], want["icp"])
    want_pca = shape.pca(last["aligned"], last["mean"], 3)
    assert torch.equal(model["modes"], want_pca["modes"]) and np.array_equal(model["scores"], want_pca["scores"])
    assert model["modes"].shape == (3, template.points.shape[0], 3)


@pytest.mark.gpu
@pytest.mark.parametrize("align_type,key", [("weighted", "weighted_avg_transformed_points"),
                                            ("nearest", "nearest_neighbor_transformed_points")])
def test_round_one_uses_the_registration(align_type, key):
    import torch

    subjects, template = _cohort()
    sb = SpectralBatch(**SPECTRAL_KW)
    P = len(subjects)
    out = sb.run_mesh_pairs(subjects + [template], [(m, P) for m in range(P)])
    gpa = shape.procrustes(out[key].view(P, -1, 3), _dev(template.points), "rigid")
    model = sb.build_shape_model(subjects, template, rounds=1, procrustes="rigid", align_type=align_type, n_modes=2)
    assert len(model["rounds"]) == 1
    assert torch.equal(model["mean_points"], gpa["mean"]) and torch.equal(model["aligned"], gpa["aligned"])


@pytest.mark.gpu
def test_eigensolve_failure_names_round_and_mesh():
    subjects, template = _cohort()
    pts = template.points.copy()
    pts[template.tris[0, 1]] = pts[template.tris[0, 0]]  # a zero-length edge in the template
    with pytest.raises(RuntimeError, match="round 1 failed for the round-1 template"):
        SpectralBatch(**SPECTRAL_KW).build_shape_model(subjects, fmesh.PolyData(pts, template.tris))
