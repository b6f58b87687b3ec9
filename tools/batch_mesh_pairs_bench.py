"""Pair lists in SpectralBatch at bench shape: a cohort of 12 meshes of 15 212 vertices (the sources of
``mesh.ellipsoid_pair(i, 39)``, i < 12) with all 132 ordered pairs, the bench configuration
(``SpectralBatch(3, 3, 5000, 300, 40)``, registration = identity, one stream).  Prints one JSON line with the GPU's name
and power limit (``--out FILE`` also writes it there).

    python tools/batch_mesh_pairs_bench.py --out profiles/r6_batch_mesh_pairs_bench.json

  * pairs/s of ``run(..., mesh_pairs=...)`` (12 meshes built and solved) against ``run`` on the pair layout (264 meshes,
    every pair's target and source packed once per pair): CUDA events around ``--steps`` warm steps, after a warm-up
    step of each, the two alternating for ``--rounds`` rounds;
  * the per-stage times of one more step of each with ``record_events``, and the eigensolver's ``filter_degree`` and
    ``outer_iterations`` (largest over the meshes);
  * whether every key of the output contract is equal between the two runs;
  * kernel A/B on 128 meshes, 300 passes (the target smoothing) and 40 passes (the projection smoothing), warm,
    alternating, mean of ``--reps``: ``focusr_mean_filter`` against ``focusr_mean_filter_mapped`` with identity segments
    (which it runs with the identity kernel form) and with the segments in reverse mesh order (the table form), and
    whether the results are equal;
  * ``tools/batch_shared_target_bench.py`` run again in the same process tree, beside r5's recorded step time and card
    (``profiles/r5_batch_shared_target_bench.json``).
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

from tools.batch_shared_target_bench import events_ms, same  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--meshes", type=int, default=12)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ab-meshes", type=int, default=128)
    ap.add_argument("--skip-shared-target-rerun", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    from pyfocusr_b200 import mesh as fmesh
    from pyfocusr_b200._device import DeviceGraph
    from pyfocusr_b200.batch import SpectralBatch

    assert torch.cuda.is_available(), "batch_mesh_pairs_bench needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    M = args.meshes
    base = fmesh.icosphere(39)
    meshes = [fmesh.ellipsoid_pair(i, 39, base=base)[1] for i in range(M)]
    mp = np.array([(a, b) for a in range(M) for b in range(M) if a != b], dtype=np.int32)
    P = mp.shape[0]
    batches = {}
    pts, tris, off = SpectralBatch._pack(meshes)
    batches["mesh_pairs"] = (pts.cuda(), tris.cuda(), off, dict(mesh_pairs=mp))
    pts, tris, off, _ = SpectralBatch.pack_meshes([meshes[t] for t in mp[:, 0]], [meshes[s] for s in mp[:, 1]])
    batches["pair_layout"] = (pts.cuda(), tris.cuda(), off, {})
    sb = SpectralBatch(3, 3, 5000, 300, 40, seed=0)

    def step(name):
        dp, dt, off, kw = batches[name]
        return sb.run(dp, dt, off, P, **kw)

    res = dict(gpu=smi, meshes=M, pairs=P, vertices_per_mesh=int(meshes[0].points.shape[0]), steps=args.steps,
               rounds=args.rounds)
    for name in batches:  # warm-up
        step(name)
    torch.cuda.synchronize()
    ms = {name: [] for name in batches}
    for _ in range(args.rounds):
        for name in batches:
            ms[name].append(events_ms(lambda: step(name), args.steps))
    outs = {}
    for name in batches:
        dp, dt, off, kw = batches[name]
        outs[name] = sb.run(dp, dt, off, P, record_events=True, **kw)
        info = outs[name]["eigs_info"]
        res[name] = dict(
            meshes_solved=int(outs[name]["graph"].n_meshes), step_ms=float(np.median(ms[name])),
            step_ms_rounds=[round(v, 3) for v in ms[name]], pairs_per_s=1e3 * P / float(np.median(ms[name])),
            stages_ms={k: round(v, 3) for k, v in sb.timings.items()},
            filter_degree_max=int(info["filter_degree"].max()), outer_iterations_max=int(info["outer_iterations"].max()),
            block_size=int(info["block_size"]))
    res["speedup"] = res["mesh_pairs"]["pairs_per_s"] / res["pair_layout"]["pairs_per_s"]
    a, b = outs["mesh_pairs"], outs["pair_layout"]
    res["keys_differing"] = sorted(k for k in b if k not in ("graph", "eigs_info") and not same(torch, a[k], b[k]))
    res["all_contract_keys_equal"] = not res["keys_differing"] and set(a) == set(b)
    del outs, a, b, batches
    torch.cuda.empty_cache()

    # kernel A/B on 128 meshes: focusr_mean_filter against focusr_mean_filter_mapped in both of its forms
    nm = args.ab_meshes
    ab_meshes = [fmesh.ellipsoid_pair(i, 39, base=base)[0] for i in range(nm)]
    g = DeviceGraph([m.points for m in ab_meshes], [m.tris for m in ab_meshes])
    seg = np.arange(nm, dtype=np.int32)
    rev = seg[::-1].copy()  # the same work through the table form: no two consecutive segments are ascending meshes
    off = g.mesh_off_host

    def reorder(x, order):
        return torch.cat([x[off[m]:off[m + 1]] for m in order]).contiguous()

    pts_rev = reorder(g.points, rev)
    ab = {}
    for passes in (300, 40):
        def plain():
            return g.mean_filter(g.points, passes)

        def identity_segments():
            return g.mean_filter_mapped(g.points, passes, seg)

        def reversed_segments():
            return g.mean_filter_mapped(pts_rev, passes, rev)

        ref = plain()
        eq = dict(identity_segments=bool(torch.equal(ref, identity_segments())),
                  reversed_segments=bool(torch.equal(reorder(ref, rev), reversed_segments())))
        fns = dict(plain=plain, identity_segments=identity_segments, reversed_segments=reversed_segments)
        t = {k: [] for k in fns}
        for _ in range(args.rounds):
            for k, fn in fns.items():
                t[k].append(events_ms(fn, args.reps))
        ab["passes_%d" % passes] = dict(equal=eq, ms={k: float(np.median(v)) for k, v in t.items()},
                                        ms_rounds={k: [round(x, 4) for x in v] for k, v in t.items()})
    res["smoothing_ab"] = dict(meshes=nm, vertices=int(g.n_points), **ab)
    del g
    torch.cuda.empty_cache()

    if not args.skip_shared_target_rerun:  # target_of_pair now runs through the mesh_pairs path: against r5's step
        line = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "batch_shared_target_bench.py")],
                              capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1]
        rerun = json.loads(line)
        with open(os.path.join(ROOT, "profiles", "r5_batch_shared_target_bench.json")) as f:
            r5 = json.loads(f.readline())
        res["shared_target_rerun"] = dict(
            gpu=rerun["gpu"], step_ms=rerun["shared"]["step_ms"], stages_ms=rerun["shared"]["stages_ms"],
            repeated_step_ms=rerun["repeated"]["step_ms"], keys_differing=rerun["keys_differing"],
            r5_gpu=r5["gpu"], r5_step_ms=r5["shared"]["step_ms"], r5_repeated_step_ms=r5["repeated"]["step_ms"],
            same_card_and_power_limit=rerun["gpu"] == r5["gpu"])

    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
