"""Surface distances at bench shape: 128 pairs of ``mesh.ellipsoid_pair(i, 39)`` (15 212 vertices, 30 420 triangles), in
the bench configuration ``SpectralBatch(3, 3, 5000, 300, 40)`` with identity registration.  Prints one JSON line with
the GPU's name and power limit.

    python tools/surface_distance_bench.py --out profiles/r8_surface_distance_bench.json

  * ``SpectralBatch.run`` pairs/s with ``surface_distances`` off and ``"weighted"``, alternated in one process, and the
    ``surface`` stage of ``record_events``;
  * ``focusr_closest_points`` alone in each direction (transformed sources -> target surfaces, targets -> transformed
    source surfaces, on the run's own positions) and ``focusr_surface_distance_stats``: device time by CUDA events over
    warm repetitions;
  * exact (query, triangle) evaluations per query in each direction, home-tile seeds included, from a build of
    surface.cu with ``-DFB_SURFACE_COUNT`` made in a temporary directory and run in a child process;
  * the brute force (no workspace) on a few pairs, its time against the pruned search on the same pairs, and whether
    their outputs are equal.
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
CSRC = os.path.join(ROOT, "pyfocusr_b200", "csrc")
NVCC = "/usr/local/cuda/bin/nvcc"
BENCH_CONFIG = (3, 3, 5000, 300, 40)


def make_batch(n_pairs):
    from pyfocusr_b200 import mesh as fmesh
    from pyfocusr_b200.batch import SpectralBatch

    base = fmesh.icosphere(39)
    targets, sources = zip(*(fmesh.ellipsoid_pair(i, 39, base=base) for i in range(n_pairs)))
    targets, sources = list(targets), list(sources)
    pts, tris, off, P = SpectralBatch.pack_meshes(targets, sources)
    toff = np.cumsum([0] + [m.tris.shape[0] for m in targets + sources]).astype(np.int32)
    return targets, sources, pts, tris, off, toff


def searches(out, toff):
    """the two searches of the surface stage on a run's own positions and triangles, as closures, and their layouts"""
    import torch

    from pyfocusr_b200 import surface

    g, off = out["graph"], out["pair_mesh_off"]
    P = out["surface_distance_stats"].shape[0]
    X = out["weighted_avg_transformed_points"]
    src_off, tgt_off = (off[P:] - off[P]).astype(np.int32), off[:P + 1]
    s_tri_off = (toff[P:] - toff[P]).astype(np.int32)
    shift = np.repeat(src_off[:-1].astype(np.int64) - g.mesh_off_host[P:2 * P], np.diff(s_tri_off))
    s_tris = (g.tris[toff[P]:].to(torch.int64) + torch.from_numpy(shift).cuda()[:, None]).to(torch.int32).contiguous()

    def s2t(pairs=None, brute=False):
        n = P if pairs is None else pairs
        return surface.closest_points(g.points, g.tris, g.mesh_off_host, toff, X[:src_off[n]], src_off[:n + 1],
                                      np.arange(n), brute_force=brute)

    def t2s(pairs=None, brute=False):
        n = P if pairs is None else pairs
        return surface.closest_points(X, s_tris, src_off, s_tri_off, g.points[:tgt_off[n]], tgt_off[:n + 1], np.arange(n),
                                      want_closest=False, brute_force=brute)

    return s2t, t2s, src_off, tgt_off


def event_ms(fn, reps):
    import torch

    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def run_weighted(pts, tris, off, toff, P):
    from pyfocusr_b200.batch import SpectralBatch

    sb = SpectralBatch(*BENCH_CONFIG, registration="identity", surface_distances="weighted")
    return sb.run(pts, tris, off, P, tri_off_host=toff)


def child(args):
    """evaluations per query with the library named by FOCUSR_B200_LIB (a -DFB_SURFACE_COUNT build)"""
    import torch

    from pyfocusr_b200 import _lib

    _, _, pts, tris, off, toff = make_batch(args.pairs)
    out = run_weighted(pts.cuda(), tris, off, toff, args.pairs)
    s2t, t2s, src_off, tgt_off = searches(out, toff)
    res = {}
    for name, fn, n in (("source_to_target", s2t, src_off[-1]), ("target_to_source", t2s, tgt_off[-1])):
        torch.cuda.synchronize()
        _lib.load().focusr_profile_reset()
        fn()
        out4 = np.zeros(4)
        _lib.load().focusr_profile_get_kind(6, out4.ctypes.data)
        res["evals_per_query_" + name] = float(out4[0]) / float(n)
    print(json.dumps(res))


def build_count_variant(tmp):
    objs = [o for o in glob.glob(os.path.join(CSRC, "build", "*.o")) if os.path.basename(o) != "surface.o"]
    obj, so = os.path.join(tmp, "surface_count.o"), os.path.join(tmp, "libfocusr_b200_count.so")
    flags = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-Xcompiler", "-fopenmp"]
    subprocess.check_call([NVCC] + flags + ["-fmad=false", "-DFB_SURFACE_COUNT", "-c", os.path.join(CSRC, "surface.cu"), "-o", obj])
    subprocess.check_call([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", so] + objs + [obj, "-lcudart", "-lgomp"])
    return so


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=128)
    ap.add_argument("--reps", type=int, default=3, help="alternating timed runs of each configuration")
    ap.add_argument("--search-reps", type=int, default=10)
    ap.add_argument("--brute-pairs", type=int, default=2)
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.child:
        return child(args)
    import torch

    from pyfocusr_b200.batch import SpectralBatch

    assert torch.cuda.is_available(), "surface_distance_bench needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    P = args.pairs
    targets, sources, pts, tris, off, toff = make_batch(P)
    res = dict(gpu=smi, pairs=P, config=list(BENCH_CONFIG), vertices_per_mesh=int(targets[0].points.shape[0]),
               triangles_per_mesh=int(targets[0].tris.shape[0]))
    dp = pts.cuda()

    # the step with the option off and on, alternated
    sbs = {k: SpectralBatch(*BENCH_CONFIG, registration="identity", surface_distances=v)
           for k, v in (("off", None), ("weighted", "weighted"))}
    for sb in sbs.values():
        sb.run(dp, tris, off, P, tri_off_host=toff)
    secs = {k: [] for k in sbs}
    for _ in range(args.reps):
        for k, sb in sbs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sb.run(dp, tris, off, P, tri_off_host=toff)
            torch.cuda.synchronize()
            secs[k].append(time.perf_counter() - t0)
    for k in sbs:
        res["pairs_per_s_" + k] = [P / s for s in secs[k]]
        res["best_pairs_per_s_" + k] = P / min(secs[k])
    sbs["weighted"].run(dp, tris, off, P, tri_off_host=toff, record_events=True)
    res["stage_ms_weighted"] = sbs["weighted"].timings

    # the searches and the stats call alone, on the run's own positions
    out = run_weighted(dp, tris, off, toff, P)
    s2t, t2s, src_off, tgt_off = searches(out, toff)
    res["queries_source_to_target"], res["queries_target_to_source"] = int(src_off[-1]), int(tgt_off[-1])
    res["closest_points_ms_source_to_target"] = event_ms(s2t, args.search_reps)
    res["closest_points_ms_target_to_source"] = event_ms(t2s, args.search_reps)
    from pyfocusr_b200 import surface

    a, b = out["source_to_target_surface_dist"], out["target_to_source_surface_dist"]
    res["stats_ms"] = event_ms(lambda: surface.distance_stats(a, src_off, b, tgt_off), args.search_reps)
    same_as_run = all(torch.equal(x, y) for x, y in zip(s2t(), (out["source_to_target_closest_points"],
                                                                out["source_to_target_closest_tri"], a)))
    res["search_equals_run_keys"] = bool(same_as_run and torch.equal(t2s()[2], b))

    # brute force on a few pairs, against the pruned search on the same pairs
    nb = args.brute_pairs
    res["brute_pairs"] = nb
    equal = True
    for name, fn in (("source_to_target", s2t), ("target_to_source", t2s)):
        res["brute_ms_" + name] = event_ms(lambda: fn(nb, True), 1)
        res["pruned_ms_" + name + "_same_pairs"] = event_ms(lambda: fn(nb), args.search_reps)
        pr, br = fn(nb), fn(nb, True)
        equal &= all((x is None and y is None) or torch.equal(x, y) for x, y in zip(pr, br))
        res["brute_over_pruned_" + name] = res["brute_ms_" + name] / res["pruned_ms_" + name + "_same_pairs"]
    res["pruned_equals_brute_force"] = bool(equal)

    if not args.no_variants:
        with tempfile.TemporaryDirectory() as tmp:
            so = build_count_variant(tmp)
            env = dict(os.environ, FOCUSR_B200_LIB=so)
            line = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--pairs", str(P)], env=env,
                                  capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1]
            res.update(json.loads(line))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
