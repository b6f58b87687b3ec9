"""Meshes of mixed sizes in one SpectralBatch, and eigsort's cost stage beyond 16 384 ordering samples.  Prints one JSON
line with the GPU's name and power limit (``--out FILE`` also writes it there).

    python tools/batch_mixed_sizes_bench.py --out profiles/r7_batch_mixed_sizes_bench.json

  * (a) 64 pairs whose meshes have 4 842, 5 292, 9 002 or 15 212 vertices (``mesh.ellipsoid_pair`` at icosphere
    frequencies 22, 23, 30, 39; pair i: target frequency i % 4, source frequency (i // 4) % 4, so every combination
    occurs), the bench configuration ``SpectralBatch(3, 3, 5000, 300, 40)``.  A 4 842-vertex mesh yields all of its rows
    as ordering samples, the others 5 000, so without per-pair counts the cohort must run as four batches, one per
    (target count, source count).  Timed both ways, alternating for ``--rounds`` rounds, CUDA events around ``--steps``
    warm steps: one batch of 64 pairs, and the four same-count batches one after the other on one stream.  Both take
    the same ordering samples (those the one batch draws).  Also the per-stage times of one more step of each.
  * (b) ``focusr_eigsort_costs`` alone on ``--cost-pairs`` pairs of 49 002-vertex meshes (frequency 70) at 5 000,
    16 384, 16 385 and 40 000 samples per mesh (up to 16 384 the shared-memory sort, above it the global segmented sort),
    n = 6 columns of smooth functions of the vertices scaled to [-0.5, 0.5]; mean of ``--reps`` warm calls, each with its
    host-to-device index copies and workspace allocation, as ``SpectralBatch.run`` makes them.
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

from tools.batch_shared_target_bench import events_ms  # noqa: E402

NUS = (22, 23, 30, 39)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=64)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cost-pairs", type=int, default=8)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    from pyfocusr_b200 import _device
    from pyfocusr_b200 import mesh as fmesh
    from pyfocusr_b200._device import DeviceGraph
    from pyfocusr_b200.batch import SpectralBatch

    assert torch.cuda.is_available(), "batch_mixed_sizes_bench needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    res = dict(gpu=smi)

    # (a) one ragged batch against the same-count batches a user needs without per-pair counts
    P = args.pairs
    bases = {nu: fmesh.icosphere(nu) for nu in NUS}
    nu_t = [NUS[i % 4] for i in range(P)]
    nu_s = [NUS[(i // 4) % 4] for i in range(P)]
    targets = [fmesh.ellipsoid_pair(i, nu_t[i], base=bases[nu_t[i]])[0] for i in range(P)]
    sources = [fmesh.ellipsoid_pair(i, nu_s[i], base=bases[nu_s[i]])[1] for i in range(P)]
    sb = SpectralBatch(3, 3, 5000, 300, 40, seed=0)
    rng = np.random.RandomState(0)
    idx_t = sb.sample_indices([m.points.shape[0] for m in targets], rng)
    idx_s = sb.sample_indices([m.points.shape[0] for m in sources], rng)
    groups = {}
    for p in range(P):
        groups.setdefault((len(idx_t[p]), len(idx_s[p])), []).append(p)
    jobs = {}

    def packed(pairs):
        pts, tris, off, n = SpectralBatch.pack_meshes([targets[p] for p in pairs], [sources[p] for p in pairs])
        it, is_ = [idx_t[p] for p in pairs], [idx_s[p] for p in pairs]
        if len({len(i) for i in it}) == 1 and len({len(i) for i in is_}) == 1:
            it, is_ = np.stack(it), np.stack(is_)
        return dict(points=pts.cuda(), tris=tris.cuda(), mesh_off_host=off, n_pairs=n, idx_t=it, idx_s=is_)

    jobs["one_batch"] = [packed(list(range(P)))]
    jobs["same_count_batches"] = [packed(g) for _, g in sorted(groups.items())]

    def step(name):
        return [sb.run(**j) for j in jobs[name]]

    for name in jobs:  # warm-up
        step(name)
    torch.cuda.synchronize()
    ms = {name: [] for name in jobs}
    for _ in range(args.rounds):
        for name in jobs:
            ms[name].append(events_ms(lambda: step(name), args.steps))
    a = dict(pairs=P, steps=args.steps, rounds=args.rounds,
             vertices={str(nu): int(bases[nu].points.shape[0]) for nu in NUS},
             same_count_batches={"%d x %d samples" % k: len(v) for k, v in sorted(groups.items())})
    for name in jobs:
        stages = {}
        for j in jobs[name]:
            sb.run(record_events=True, **j)
            for k, v in sb.timings.items():
                stages[k] = stages.get(k, 0.0) + v
        med = float(np.median(ms[name]))
        a[name] = dict(batches=len(jobs[name]), step_ms=med, step_ms_rounds=[round(v, 3) for v in ms[name]],
                       pairs_per_s=1e3 * P / med, stages_ms={k: round(v, 3) for k, v in stages.items()})
    a["one_batch_over_split_time"] = a["one_batch"]["step_ms"] / a["same_count_batches"]["step_ms"]
    res["a_mixed_cohort"] = a
    del jobs
    torch.cuda.empty_cache()

    # (b) the cost stage alone at and beyond the shared-memory sort's 16 384 samples
    C = args.cost_pairs
    base = fmesh.icosphere(70)
    meshes = [m for i in range(C) for m in fmesh.ellipsoid_pair(i, 70, base=base)]
    meshes = meshes[0::2] + meshes[1::2]  # targets, then sources
    g = DeviceGraph([m.points for m in meshes], [m.tris for m in meshes])
    n, nv = 6, int(meshes[0].points.shape[0])
    cols = []
    for m in meshes:
        x = m.points / np.ptp(m.points, axis=0)
        f = np.stack([np.sin(3 * x[:, 0] + k) * np.cos(2 * x[:, 1] - k) + x[:, 2] * k for k in range(n)], axis=1)
        cols.append((f - f.min(axis=0)) / np.ptp(f, axis=0) - 0.5)
    vecs = torch.from_numpy(np.concatenate(cols)).cuda()
    t_mesh, s_mesh = np.arange(C), np.arange(C, 2 * C)
    b = dict(pairs=C, vertices=nv, n_features=n, reps=args.reps)
    for count in (5000, 16384, 16385, 40000):
        r = np.random.RandomState(count)
        it = np.stack([r.choice(nv, count, replace=False) for _ in range(C)])
        is_ = np.stack([r.choice(nv, count, replace=False) for _ in range(C)])

        def costs():
            return _device.eigsort_costs(g, vecs, t_mesh, s_mesh, it, is_, n)

        costs()
        torch.cuda.synchronize()
        t = [events_ms(costs, args.reps) for _ in range(args.rounds)]
        b["samples_%d" % count] = dict(sort="shared memory" if count <= 16384 else "global segmented radix",
                                       ms=float(np.median(t)), ms_rounds=[round(v, 3) for v in t],
                                       ms_per_pair=float(np.median(t)) / C)
    res["b_cost_stage"] = b

    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
