"""Shape models at bench shape: a cohort of 128 subjects (the sources of ``mesh.ellipsoid_pair(i, 39)``, 15 212 vertices
each) on the vertices of a template (``perturbed_ellipsoid(39, seed=1000)``, a seed no subject uses), the bench
configuration ``SpectralBatch(3, 3, 5000, 300, 40)`` with identity registration.  Prints one JSON line with the GPU's
name and power limit, read in the same call (``--out FILE`` also writes it there).

    python tools/shape_model_bench.py --out profiles/r7_shape_model_bench.json

  * every round of ``build_shape_model`` run one call at a time, each part timed by the host clock between device
    synchronisations: registration (``run_mesh_pairs``), GPA (``shape.procrustes``, which reads each iteration's change
    back), and PCA of the last round (``shape.pca``, first call and warm); the GPA iterations and the template change
    per round;
  * GPA alone on the last round's 128 configurations, and its parts: one ``focusr_procrustes_fit`` (128 fits plus the
    aligned sets), one ``focusr_procrustes_mean``, and PCA's ``focusr_shape_gram`` and ``focusr_shape_modes``, CUDA
    events over ``--reps`` warm calls; the configurations are 128 x 15 212 x 24 B = 46.7 MB, which the 126 MB L2 holds,
    so these are times, not HBM fractions;
  * ``build_shape_model`` end to end with the same settings (wall clock), and whether its mean equals the one of the
    rounds run by hand bit for bit.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def events_ms(torch, fn, reps):
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
    ap.add_argument("--subjects", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--template-tolerance", type=float, default=1e-3)
    ap.add_argument("--n-modes", type=int, default=10)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    from pyfocusr_b200 import _device, mesh as fmesh, shape
    from pyfocusr_b200.batch import SpectralBatch

    assert torch.cuda.is_available(), "shape_model_bench needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    P = args.subjects
    base = fmesh.icosphere(39)
    subjects = [fmesh.ellipsoid_pair(i, 39, base=base)[1] for i in range(P)]
    template = fmesh.perturbed_ellipsoid(39, 1000, base=base)
    sb = SpectralBatch(3, 3, 5000, 300, 40, seed=0)
    pairs = [(m, P) for m in range(P)]
    res = dict(gpu=smi, subjects=P, vertices_per_mesh=int(template.points.shape[0]), rounds_max=args.rounds,
               template_tolerance=args.template_tolerance, procrustes="similarity", align_type="weighted",
               n_modes=args.n_modes)
    sb.run_mesh_pairs(subjects + [template], pairs)  # warm-up: module loads, allocator pools
    torch.cuda.synchronize()

    def clock(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return r, 1e3 * (time.perf_counter() - t0)

    tmpl, rounds, configs = template, [], None
    for _ in range(args.rounds):
        out, reg_ms = clock(lambda: sb.run_mesh_pairs(subjects + [tmpl], pairs))
        configs = out["weighted_avg_transformed_points"].view(P, -1, 3)
        ref = torch.from_numpy(tmpl.points).cuda()
        gpa, gpa_ms = clock(lambda: shape.procrustes(configs, ref, "similarity"))
        mean = gpa["mean"].cpu().numpy()
        change = float(np.sqrt(np.mean(np.sum((mean - tmpl.points) ** 2, 1))))
        rounds.append(dict(registration_ms=round(reg_ms, 3), gpa_ms=round(gpa_ms, 3), gpa_iterations=gpa["iterations"],
                           template_change=change))
        del out
        tmpl = fmesh.PolyData(mean, template.tris)
        if change <= args.template_tolerance:
            break
    model, pca_ms = clock(lambda: shape.pca(gpa["aligned"], gpa["mean"], args.n_modes))
    res["rounds"] = rounds
    res["pca_first_call_ms"] = round(pca_ms, 3)
    times = [clock(lambda: shape.pca(gpa["aligned"], gpa["mean"], args.n_modes))[1] for _ in range(5)]
    res["pca_ms"] = dict(median=float(np.median(times)), all=[round(t, 3) for t in times])
    res["variances"] = [float(v) for v in model["variances"]]

    # GPA alone on the last round's configurations, and its kernels
    ref = torch.from_numpy(np.ascontiguousarray(template.points)).cuda()
    times = [clock(lambda: shape.procrustes(configs, ref, "similarity"))[1] for _ in range(5)]
    res["gpa_alone_ms"] = dict(median=float(np.median(times)), all=[round(t, 3) for t in times])
    mats, aligned = _device.procrustes_fit(configs, ref, True)
    nxt, change = torch.empty_like(ref), torch.empty(1, dtype=torch.float64, device="cuda")
    ws = _device.procrustes_mean(aligned, ref, True, ref, nxt, change)
    res["procrustes_fit_ms"] = events_ms(torch, lambda: _device.procrustes_fit(configs, ref, True), args.reps)
    res["procrustes_mean_ms"] = events_ms(torch, lambda: _device.procrustes_mean(aligned, ref, True, ref, nxt, change, ws),
                                          args.reps)
    res["shape_gram_ms"] = events_ms(torch, lambda: _device.shape_gram(aligned, ref), args.reps)
    w = torch.ones((P, args.n_modes), dtype=torch.float64, device="cuda")
    res["shape_modes_ms"] = events_ms(torch, lambda: _device.shape_modes(aligned, ref, w), args.reps)
    res["config_bytes"] = int(configs.numel() * 8)

    model2, e2e_ms = clock(lambda: sb.build_shape_model(subjects, template, rounds=args.rounds,
                                                        template_tolerance=args.template_tolerance, n_modes=args.n_modes))
    res["build_shape_model_ms"] = round(e2e_ms, 3)
    res["build_shape_model_rounds"] = len(model2["rounds"])
    res["build_shape_model_mean_equals_by_hand"] = bool(np.array_equal(model2["mean_mesh"].points, tmpl.points))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
