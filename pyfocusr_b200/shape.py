"""Statistical shape models on the device: generalized Procrustes analysis (GPA) and PCA of a cohort's configurations.

A configuration is the N vertices of one template located on one subject (``SpectralBatch.run_mesh_pairs`` with the
subjects as targets and the template as the shared source gives them in ``weighted_avg_transformed_points``).  The
fits, means, Gram matrix and modes run in ``csrc/shape.cu`` (K13); the fit is the landmark transform of the ICP
iterations (vtkLandmarkTransform, Horn's quaternion solution).  The P x P eigendecomposition of the PCA runs on the
host in fp64, one host visit per model.  ``SpectralBatch.build_shape_model`` runs the whole workflow: registration,
GPA, the GPA mean as the next template, repeated until the template stops moving, then PCA.
"""
from __future__ import annotations

import re

import numpy as np

from . import _device, _lib

__all__ = ["procrustes", "pca", "build_shape_model"]

PROCRUSTES_MODES = ("rigid", "similarity")
ALIGN_TYPES = {"weighted": "weighted_avg_transformed_points", "nearest": "nearest_neighbor_transformed_points"}


def _check_mode(mode):
    if mode not in PROCRUSTES_MODES:
        raise ValueError("procrustes mode must be 'rigid' or 'similarity', got %r" % (mode,))


def _check_n_modes(n_modes):
    if int(n_modes) != n_modes or int(n_modes) < 1:
        raise ValueError("n_modes must be an integer >= 1, got %r" % (n_modes,))


def rms_radius(points):
    """RMS distance of the points (N, 3) from their centroid: the scale GPA's tolerance is relative to."""
    p = np.asarray(points, dtype=np.float64)
    return float(np.sqrt(np.mean(np.sum((p - p.mean(0)) ** 2, axis=1))))


def _as_device(x, dev=None):
    torch = _lib.require_cuda()
    t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
    return t.to(device=dev or "cuda", dtype=torch.float64).contiguous()


def procrustes(configs, reference, mode="similarity", max_iterations=100, tolerance=1e-10):
    """Generalized Procrustes analysis of ``configs`` (P, N, 3) with the mean's frame fixed by ``reference`` (N, 3).

    M_0 = reference.  Iteration k fits every original configuration onto M_k (``mode``: rigid or similarity), averages
    the fitted sets in configuration order, fits that average back onto the reference (which fixes the frame and, for a
    similarity, the scale) and takes the result as M_{k+1}; d_k = RMS(M_{k+1} - M_k) over the N points.  It stops when
    d_k <= ``tolerance`` * the reference's RMS distance from its centroid, or after ``max_iterations``.

    Returns a dict: ``mean`` (N, 3), the last M_{k+1}; ``aligned`` (P, N, 3), the configurations fitted onto the last
    M_k; ``matrices`` (P, 4, 4) those fits (row-major, column vectors) -- all device tensors; ``iterations``; ``changes``
    (numpy, d_k per iteration)."""
    _check_mode(mode)
    if int(max_iterations) < 1:
        raise ValueError("max_iterations must be >= 1, got %r" % (max_iterations,))
    if not tolerance >= 0.0:
        raise ValueError("tolerance must be >= 0, got %r" % (tolerance,))
    torch = _lib.require_cuda()
    configs = _as_device(configs)
    if configs.dim() != 3 or configs.shape[2] != 3 or configs.shape[0] < 1 or configs.shape[1] < 1:
        raise ValueError("configs must be (P, N, 3) with P, N >= 1, got %s" % (tuple(configs.shape),))
    ref_host = reference.detach().cpu().numpy() if isinstance(reference, torch.Tensor) else np.asarray(reference, np.float64)
    if ref_host.shape != tuple(configs.shape[1:]):
        raise ValueError("reference must be (%d, 3), got %s" % (configs.shape[1], ref_host.shape))
    reference = _as_device(reference, configs.device)
    threshold = float(tolerance) * rms_radius(ref_host)
    sim = mode == "similarity"
    mean, nxt = reference.clone(), torch.empty_like(reference)
    change = torch.empty(int(max_iterations), dtype=torch.float64, device=configs.device)
    changes, ws = [], None
    for k in range(int(max_iterations)):
        mats, aligned = _device.procrustes_fit(configs, mean, sim)
        ws = _device.procrustes_mean(aligned, reference, sim, mean, nxt, change[k:k + 1], ws)
        mean, nxt = nxt, mean
        changes.append(float(change[k].item()))
        if changes[-1] <= threshold:
            break
    return dict(mean=mean, aligned=aligned, matrices=mats, iterations=len(changes), changes=np.array(changes))


def pca(aligned, mean, n_modes):
    """PCA of the configurations ``aligned`` (P, N, 3) about ``mean`` (N, 3): D = aligned - mean as [P][3N], its Gram
    matrix D D^T on the device, the eigendecomposition on the host (fp64), the modes D^T u / sqrt(lambda) on the device.

    K = min(``n_modes``, P - 1, the number of eigenvalues above rounding, lambda > P * eps * lambda_max).  Returns a
    dict: ``modes`` (K, N, 3) device tensor, each of unit norm over its 3N entries with its entry of largest magnitude
    positive (the lowest index on ties); ``variances`` (K,) lambda / (P - 1), descending, and ``scores`` (P, K), the
    coordinates D modes^T of every configuration -- both host numpy."""
    _check_n_modes(n_modes)
    torch = _lib.require_cuda()
    aligned = _as_device(aligned)
    mean = _as_device(mean, aligned.device)
    P, N = int(aligned.shape[0]), int(aligned.shape[1])
    lam, U = np.linalg.eigh(_device.shape_gram(aligned, mean).cpu().numpy())
    lam, U = lam[::-1], U[:, ::-1]
    n_pos = int(np.count_nonzero(lam > P * np.finfo(np.float64).eps * max(lam[0], 0.0)))
    K = min(int(n_modes), P - 1, n_pos)
    if K == 0:
        return dict(modes=torch.zeros((0, N, 3), dtype=torch.float64, device=aligned.device), variances=np.zeros(0),
                    scores=np.zeros((P, 0)))
    root = np.sqrt(lam[:K])
    modes = _device.shape_modes(aligned, mean, torch.from_numpy(np.ascontiguousarray(U[:, :K] / root)))
    flat = modes.view(K, -1)
    sign = torch.sign(flat.gather(1, flat.abs().argmax(1, keepdim=True)))
    flat.mul_(sign)
    return dict(modes=modes, variances=lam[:K] / (P - 1), scores=U[:, :K] * root * sign.view(1, K).cpu().numpy())


def _round_error(exc, rnd, P):
    """A failure of round ``rnd``'s registration, the meshes its message names said as subjects / the template."""
    named = []
    for m in (int(x) for x in re.findall(r"\bmesh (\d+)", str(exc))):
        name = "subject %d" % m if m < P else "the round-%d template" % rnd
        if name not in named:
            named.append(name)
    who = " for " + ", ".join(named) if named else ""
    return RuntimeError("shape model round %d failed%s (mesh m < %d is subject m, mesh %d the template): %s" % (
        rnd, who, P, P, exc))


def build_shape_model(sb, subjects, template, rounds=5, template_tolerance=1e-3, procrustes_mode="similarity",
                      align_type="weighted", n_modes=10, **run_kw):
    """``SpectralBatch.build_shape_model`` (see there) for the batch object ``sb``."""
    P = len(subjects)
    if P == 0:
        raise ValueError("build_shape_model needs at least one subject")
    _check_mode(procrustes_mode)
    if align_type not in ALIGN_TYPES:
        raise ValueError("align_type must be 'weighted' or 'nearest', got %r" % (align_type,))
    _check_n_modes(n_modes)
    if int(rounds) < 1:
        raise ValueError("rounds must be >= 1, got %r" % (rounds,))
    if sb.icp_register_first and not sb.icp_reg_target_to_source:
        raise ValueError("icp_register_first without icp_reg_target_to_source would move the template, the source of "
                         "every pair, once per subject; set icp_reg_target_to_source=True to move each subject onto "
                         "the template instead")
    from .mesh import PolyData

    torch = _lib.require_cuda()
    subjects = list(subjects)
    pairs = [(m, P) for m in range(P)]
    key = ALIGN_TYPES[align_type]
    tmpl = template
    per_round = []
    for rnd in range(1, int(rounds) + 1):
        try:
            out = sb.run_mesh_pairs(subjects + [tmpl], pairs, **run_kw)
        except RuntimeError as exc:
            raise _round_error(exc, rnd, P) from exc
        n_t = int(tmpl.points.shape[0])
        configs = out[key].view(P, n_t, 3)
        gpa = procrustes(configs, torch.from_numpy(np.ascontiguousarray(tmpl.points, dtype=np.float64)).to(configs.device),
                         procrustes_mode)
        new_points = gpa["mean"].cpu().numpy()
        change = float(np.sqrt(np.mean(np.sum((new_points - tmpl.points) ** 2, axis=1))))
        info = dict(template_change=change, gpa_iterations=gpa["iterations"], gpa_changes=gpa["changes"])
        if sb.icp_register_first:
            info["icp_matrices"] = out["icp_matrices"]
        if sb.surface_distances is not None:  # the template is every pair's source: one row per subject
            info["surface_distance_stats"] = out["surface_distance_stats"].cpu().numpy()
        per_round.append(info)
        del out, configs
        tmpl = PolyData(new_points, template.tris, getattr(template, "point_scalars", None))
        if change <= template_tolerance:
            break
    model = pca(gpa["aligned"], gpa["mean"], n_modes)
    return dict(mean_points=gpa["mean"], mean_mesh=tmpl, aligned=gpa["aligned"], procrustes_matrices=gpa["matrices"],
                modes=model["modes"], variances=model["variances"], scores=model["scores"], rounds=per_round)
