"""Shared targets in SpectralBatch at bench shape: one template and 128 sources, all ``mesh.ellipsoid_pair(i, 39)`` meshes
of 15 212 vertices (template = target of pair 0, source i = source of pair i), the bench configuration
(``SpectralBatch(3, 3, 5000, 300, 40)``, registration = identity).  Prints one JSON line with the GPU's name and power
limit (``--out FILE`` also writes it there).

    python tools/batch_shared_target_bench.py --out profiles/r5_batch_shared_target_bench.json

  * pairs/s of ``run(..., target_of_pair=zeros(128))`` (129 meshes built and solved) against ``run`` on the batch with
    the template repeated once per pair (256 meshes): CUDA events around ``--steps`` warm steps, after a warm-up step of
    each, the two alternating for ``--rounds`` rounds;
  * the per-stage times of one more step of each with ``record_events``, and the eigensolver's ``filter_degree`` and
    ``outer_iterations`` (largest over the meshes);
  * the final k = 3 search alone (device time, warm, alternating, mean of ``--reps``): ``focusr_knn_mapped`` with the
    smoothed template as the one reference segment, against ``focusr_knn`` on 128 copies of it;
  * whether ``final_idx`` and ``weighted_avg_transformed_points`` of the two runs are equal (and every other key of the
    output contract).
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


def events_ms(fn, reps):
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def same(torch, a, b):
    if a is None or b is None:
        return a is None and b is None
    if isinstance(a, torch.Tensor):
        return isinstance(b, torch.Tensor) and torch.equal(a, b)
    if isinstance(a, np.ndarray):
        return np.array_equal(a, b)
    if isinstance(a, (tuple, list)):
        return len(a) == len(b) and all(same(torch, x, y) for x, y in zip(a, b))
    return a == b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=128)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    from pyfocusr_b200 import _device
    from pyfocusr_b200 import mesh as fmesh
    from pyfocusr_b200.batch import SpectralBatch

    assert torch.cuda.is_available(), "batch_shared_target_bench needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    P = args.pairs
    base = fmesh.icosphere(39)
    pairs = [fmesh.ellipsoid_pair(i, 39, base=base) for i in range(P)]
    template, sources = pairs[0][0], [s for _, s in pairs]
    top = np.zeros(P, dtype=np.int32)
    batches = {}
    for name, (targets, kw) in dict(shared=([template], dict(target_of_pair=top)), repeated=([template] * P, {})).items():
        pts, tris, off, _ = SpectralBatch.pack_meshes(targets, sources, **kw)
        batches[name] = (pts.cuda(), tris.cuda(), off, kw)
    sb = SpectralBatch(3, 3, 5000, 300, 40, seed=0)

    def step(name):
        dp, dt, off, kw = batches[name]
        return sb.run(dp, dt, off, P, **kw)

    res = dict(gpu=smi, pairs=P, vertices_per_mesh=int(template.points.shape[0]), steps=args.steps, rounds=args.rounds)
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
    res["speedup"] = res["shared"]["pairs_per_s"] / res["repeated"]["pairs_per_s"]

    a, b = outs["shared"], outs["repeated"]
    res["final_idx_equal"] = bool(torch.equal(a["final_idx"], b["final_idx"]))
    res["weighted_positions_equal"] = bool(torch.equal(a["weighted_avg_transformed_points"], b["weighted_avg_transformed_points"]))
    res["keys_differing"] = sorted(k for k in b if k not in ("graph", "eigs_info") and not same(torch, a[k], b[k]))

    # the final k = 3 search alone: the smoothed template against the 128 projected sources
    nt = int(template.points.shape[0])
    copies = b["smoothed_target_coords"].contiguous()           # 128 copies of the smoothed template
    ref1 = copies[:nt].contiguous()
    queries = a["source_projected_on_target"].contiguous()
    off_pair = b["graph"].mesh_off_host
    q_off = torch.from_numpy((off_pair[P:] - off_pair[P]).astype(np.int32)).cuda()
    r_off_copies = torch.from_numpy(off_pair[:P + 1].astype(np.int32)).cuda()
    r_off_one = torch.tensor([0, nt], dtype=torch.int32, device="cuda")
    max_q = int(np.diff(off_pair[P:]).max())

    def mapped():
        return _device.knn_mapped(ref1, queries, r_off_one, q_off, top, k=3, max_queries=max_q, max_refs=nt)

    def on_copies():
        return _device.knn(copies, queries, k=3, ref_off=r_off_copies, query_off=q_off, max_queries=max_q, max_refs=nt)

    mi, md = mapped()
    ci, cd = on_copies()
    res["final_search_equal"] = bool(torch.equal(mi, ci) and torch.equal(md, cd))
    t = {"mapped": [], "copies": []}
    for _ in range(args.rounds):
        t["mapped"].append(events_ms(mapped, args.reps))
        t["copies"].append(events_ms(on_copies, args.reps))
    res["final_search_ms"] = {k: float(np.median(v)) for k, v in t.items()}
    res["final_search_ms_rounds"] = {k: [round(x, 4) for x in v] for k, v in t.items()}

    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
