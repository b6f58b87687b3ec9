"""Node features in SpectralBatch at bench shape: 128 pairs of ``mesh.ellipsoid_pair(i, 39)`` (15 212 vertices each) in
one batch, the bench configuration (``SpectralBatch(3, 3, 5000, 300, 40)``, registration = identity).  Prints one JSON
line with the GPU's name and power limit (``--out FILE`` also writes it there).

    python tools/batch_features_bench.py --out profiles/r4_batch_features_bench.json

  * ``SpectralBatch.run`` pairs/s (CUDA events around ``--steps`` warm steps, after a warm-up step) in four
    configurations: defaults; curvature in the edge weights; curvature as coordinates; both plus xyz as coordinates.
    Per configuration: the per-stage times of one more step with ``record_events`` and the eigensolver's
    ``outer_iterations`` / ``filter_degree`` (largest and mean over the 256 meshes);
  * each new stage alone on the whole batch (device time, warm, mean of ``--reps``): the batch curvature
    (``focusr_curvatures``, which synchronises once for its index check), the normalisation with edge points
    (``focusr_node_features``), the feature smoothing (40 passes x 2 columns x 256 meshes, ``focusr_mean_filter``) and
    the coordinate assembly (``focusr_feature_coords``, 3 + 2 + 3 columns).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {
    "defaults": dict(),
    "curvature_in_adjacency": dict(include_features_in_adj_matrix=True),
    "curvature_as_coords": dict(use_features_as_coords=True),
    "both_and_points": dict(include_features_in_adj_matrix=True, use_features_as_coords=True, include_points_as_features=True),
}


def timed(fn, reps):
    import torch

    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=128)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    from pyfocusr_b200 import _device, _lib
    from pyfocusr_b200 import mesh as fmesh
    from pyfocusr_b200._device import DeviceGraph
    from pyfocusr_b200.batch import SpectralBatch

    assert torch.cuda.is_available(), "batch_features_bench needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    P = args.pairs
    base = fmesh.icosphere(39)
    pairs = [fmesh.ellipsoid_pair(i, 39, base=base) for i in range(P)]
    pts, tris, off, _ = SpectralBatch.pack_meshes([t for t, _ in pairs], [s for _, s in pairs])
    dp, dt = pts.cuda(), tris.cuda()
    n = int(off[-1])
    res = dict(gpu=smi, pairs=P, vertices_per_mesh=int(pairs[0][0].points.shape[0]), steps=args.steps, configs={})

    for name, kw in CONFIGS.items():
        sb = SpectralBatch(3, 3, 5000, 300, 40, seed=0, **kw)
        run = lambda: sb.run(dp, dt, off, P)  # noqa: E731
        ms = timed(run, args.steps)
        out = sb.run(dp, dt, off, P, record_events=True)
        info = out["eigs_info"]
        res["configs"][name] = dict(
            kwargs=kw, step_ms=ms, pairs_per_s=1e3 * P / ms, coords_columns=int(out["coords"].shape[1]),
            stages_ms={k: round(v, 3) for k, v in sb.timings.items()},
            outer_iterations_max=int(info["outer_iterations"].max()), outer_iterations_mean=float(info["outer_iterations"].mean()),
            filter_degree_max=int(info["filter_degree"].max()), filter_degree_mean=float(info["filter_degree"].mean()),
            block_size=int(info["block_size"]))
        del out

    # each new stage alone on the whole batch
    lib = _lib.load()
    nf = int(dt.shape[0])
    curv = torch.empty((2, n), dtype=torch.float64, device="cuda")
    ws_c = torch.empty(int(lib.focusr_curvature_workspace_bytes(n, nf)), dtype=torch.uint8, device="cuda")

    def curvature():
        _lib.call("focusr_curvatures", _lib.ptr(dp), _lib.ptr(dt), n, nf, None, None, _lib.ptr(curv[0]), _lib.ptr(curv[1]),
                  _lib.ptr(ws_c), ws_c.numel(), _lib.stream_ptr())

    stages = dict(curvature_ms=timed(curvature, args.reps))
    raw = curv.t().contiguous()
    off_d = torch.from_numpy(off).cuda()
    stages["normalisation_ms"] = timed(lambda: _device.node_features(raw, dp, off_d, want_edge_points=True), args.reps)
    feats, ep = _device.node_features(raw, dp, off_d, want_edge_points=True)
    g = DeviceGraph.from_device(dp, dt, off, ep)
    stages["feature_smoothing_ms"] = timed(lambda: g.mean_filter(feats, 40), args.reps)
    smoothed = g.mean_filter(feats, 40)
    spectral = torch.rand((n, 3), dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    stages["coordinate_assembly_ms"] = timed(lambda: _device.feature_coords(spectral, smoothed, dp, off_d, True, True), args.reps)
    res["stages_alone"] = stages
    res["feature_stages_total_ms"] = sum(stages.values())

    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
