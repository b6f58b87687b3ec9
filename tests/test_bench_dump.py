"""bench.py --dump-outputs: the files do not depend on how a step's pairs were split into sub-batches, hold the
sampled rows of the step's results in pair order, and stay under 64 MB at the bench's shape."""
import os

import numpy as np

import bench
from pyfocusr_b200 import dist as fdist


def _step_outputs(pairs, P, n_vert, arrays):
    """The DUMP_KEYS of SpectralBatch.run for a sub-batch of `pairs` (targets, then sources)."""
    import torch

    vals, vecs, q, w, fin, wavg, near = arrays
    rows = lambda a, ids: np.concatenate([a[i * n_vert:(i + 1) * n_vert] for i in ids])
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    return {"eig_vals": t(np.concatenate([vals[pairs], vals[[P + i for i in pairs]]])),
            "eig_vecs": t(np.concatenate([rows(vecs, pairs), rows(vecs, [P + i for i in pairs])])),
            "Q": t(q[pairs]), "spectral_weights": t(w[pairs]), "final_idx": t(rows(fin, pairs)),
            "weighted_avg_transformed_points": t(rows(wavg, pairs)), "nearest_neighbor_transformed_points": t(rows(near, pairs))}


def test_dump_outputs_layout(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_ROWS", 64)
    P, n_vert, ldv, n = 5, 40, 8, 6
    rng = np.random.RandomState(0)
    arrays = (rng.rand(2 * P, ldv), rng.rand(2 * P * n_vert, ldv), rng.rand(P, n), rng.rand(P, 3),
              rng.randint(0, n_vert, P * n_vert).astype(np.int32), rng.rand(P * n_vert, 3), rng.rand(P * n_vert, 3))
    whole, split = str(tmp_path / "whole"), str(tmp_path / "split")
    bench.dump_outputs([_step_outputs(list(range(P)), P, n_vert, arrays)], n, whole)
    bench.dump_outputs([_step_outputs(ids, P, n_vert, arrays) for ids in fdist.sub_batches(range(P), 2)], n, split)
    names = sorted(os.listdir(whole))
    assert names == sorted(os.listdir(split)) and len(names) == 10
    for name in names:
        a = np.load(os.path.join(whole, name))
        assert a.dtype == np.float64 and np.array_equal(a, np.load(os.path.join(split, name))), name
    load = lambda name: np.load(os.path.join(whole, name + ".npy"))
    vals, vecs, q, w, fin, wavg, near = arrays
    r = load("sample_vertex_rows").astype(np.int64)
    assert r.size == 64 and np.all(np.diff(r) > 0) and r.max() < P * n_vert
    assert np.array_equal(load("eig_vals_target"), vals[:P, :n]) and np.array_equal(load("eig_vals_source"), vals[P:, :n])
    assert np.array_equal(load("Q"), q) and np.array_equal(load("spectral_weights"), w)
    assert np.array_equal(load("eig_vecs_target"), vecs[:P * n_vert][r, :n])
    assert np.array_equal(load("eig_vecs_source"), vecs[P * n_vert:][r, :n])
    assert np.array_equal(load("final_idx"), fin[r]) and np.array_equal(load("weighted_avg_transformed_points"), wavg[r])
    assert np.array_equal(load("nearest_neighbor_transformed_points"), near[r])


def test_dump_outputs_size_at_bench_shape():
    """128 pairs: per-vertex results (2 x 6 eigenvector columns, index, 2 x 3 coordinates, row id) for the sample, plus
    the per-pair arrays, must stay under 64 MB."""
    per_row = 2 * (bench.N_SPECTRAL + bench.N_EXTRA) + 1 + 3 + 3 + 1
    per_pair = 3 * (bench.N_SPECTRAL + bench.N_EXTRA) + bench.N_SPECTRAL
    assert 8 * (bench.DUMP_ROWS * per_row + 128 * per_pair) < 64 * 2 ** 20
