"""CPU oracle for the shape-model stage (generalized Procrustes analysis and PCA)  --  TEST INFRASTRUCTURE ONLY.

The reference has one piece of this, ``Focusr.get_average_shape`` (focusr.py:433-453), the average of one pair; the
cohort workflow built on FOCUSR (every subject on the template's vertices, GPA, the mean as the next template, PCA modes)
is restated here in numpy as ``pyfocusr_b200.shape`` defines it:

  * GPA: M_0 = the reference; iteration k fits every original configuration onto M_k with
    ``icp_port.landmark_transform`` (vtkLandmarkTransform, rigid or similarity), averages the fitted sets, fits the
    average back onto the reference and takes the result as M_{k+1}; d_k = RMS(M_{k+1} - M_k); stop when
    d_k <= tolerance * the reference's RMS distance from its centroid, or after max_iterations.
  * PCA: the SVD of D = aligned - mean as [P][3N]; modes = rows of V^T with the entry of largest magnitude positive,
    variances = s^2 / (P - 1), scores = U s (with the same signs).
Only tests/ and tools/ may import this module.
"""
from __future__ import annotations

import numpy as np

from oracle.icp_port import landmark_transform


def apply(mat, pts):
    return pts @ mat[:3, :3].T + mat[:3, 3]


def rms(a, b):
    return float(np.sqrt(np.mean(np.sum((a - b) ** 2, axis=1))))


def procrustes(configs, reference, similarity=True, max_iterations=100, tolerance=1e-10):
    """Returns dict(mean, aligned, matrices, iterations, changes) as ``pyfocusr_b200.shape.procrustes``."""
    configs = np.asarray(configs, dtype=np.float64)
    reference = np.asarray(reference, dtype=np.float64)
    threshold = tolerance * rms(reference, reference.mean(0)[None])
    mean = reference.copy()
    changes = []
    for _ in range(max_iterations):
        mats = np.stack([landmark_transform(c, mean, similarity) for c in configs])
        aligned = np.stack([apply(m, c) for m, c in zip(mats, configs)])
        raw = aligned.mean(0)
        new = apply(landmark_transform(raw, reference, similarity), raw)
        changes.append(rms(new, mean))
        mean = new
        if changes[-1] <= threshold:
            break
    return dict(mean=mean, aligned=aligned, matrices=mats, iterations=len(changes), changes=np.array(changes))


def pca(aligned, mean, n_modes):
    """Returns dict(modes (K, N, 3), variances (K,), scores (P, K)) with K = min(n_modes, P - 1, rank of D)."""
    aligned = np.asarray(aligned, dtype=np.float64)
    P, N = aligned.shape[:2]
    D = (aligned - np.asarray(mean)[None]).reshape(P, 3 * N)
    U, s, Vt = np.linalg.svd(D, full_matrices=False)
    lam = s * s
    K = min(int(n_modes), P - 1, int(np.count_nonzero(lam > P * np.finfo(np.float64).eps * max(lam[0], 0.0))))
    modes, scores = Vt[:K].copy(), U[:, :K] * s[:K]
    sign = np.sign(modes[np.arange(K), np.argmax(np.abs(modes), axis=1)])
    return dict(modes=(modes * sign[:, None]).reshape(K, N, 3), variances=lam[:K] / (P - 1), scores=scores * sign[None])
