#!/usr/bin/env python
"""Headline benchmark: spectral-embed pairs/sec @15k vertices (BASELINE.json `metric`).

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): synthetic
perturbed-ellipsoid pairs, geodesic frequency nu=39 -> 15 212 vertices / 30 420 triangles per mesh,
Focusr defaults (n_spectral_features=3 + 3 extra -> k=7, 5000 ordering samples, 300 + 40 smoothing
passes), CPD = identity (out of scope, BASELINE.md section 3).  One "step" = the whole hot path
(Laplacian assembly -> eigensolve -> normalise -> eigsort -> spectral coords -> KNN -> smoothing ->
KNN -> k=3 weighted positions) over `--pairs-per-gpu` pairs on every GPU; ranks hold independent
pairs (no data-path collective), so scaling is weak and 8 GPUs x 128 pairs is the named 1024-pair batch.

  python bench.py --gpus N --steps K --warmup W            (torchrun for N > 1, one rank per GPU)
  python bench.py --impl reference ...                      the reference's CPU path (oracle port,
                                                            scipy ARPACK/SuperLU/cKDTree) on all host cores
  python bench.py ... --dump-outputs DIR                    also write the last timed step's results to DIR/*.npy

Prints ONE JSON line (rank 0).  `value` = pairs/s with the vertices already resident in HBM;
`e2e` = the same through the public API from pinned host buffers with the result read back.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NU = 39
N_SPECTRAL, N_EXTRA, N_SAMPLES, SMOOTH_T, SMOOTH_S = 3, 3, 5000, 300, 40
# --dump-outputs: the results of SpectralBatch.run that are written, and the number of vertices (per side) in the fixed
# sample that per-vertex results are written for (128 pairs x 15 212 vertices in full would exceed 64 MB)
DUMP_KEYS = ("eig_vals", "eig_vecs", "Q", "spectral_weights", "final_idx", "weighted_avg_transformed_points",
             "nearest_neighbor_transformed_points")
DUMP_ROWS = 1 << 17


def make_pairs(pair_ids, nu=NU):
    """Host arrays for the given pair ids: points [2P*N,3] (targets then sources), global tris, offsets."""
    from pyfocusr_b200.mesh import icosphere, perturbed_ellipsoid

    base = icosphere(nu)
    n, f = base.points.shape[0], base.tris.shape[0]
    n_pairs = len(pair_ids)
    pts = np.empty((2 * n_pairs, n, 3))
    for p, i in enumerate(pair_ids):
        pts[p] = perturbed_ellipsoid(nu, 2 * i, base=base).points            # target seed 2i
        pts[n_pairs + p] = perturbed_ellipsoid(nu, 2 * i + 1, base=base).points  # source seed 2i+1
    off = (np.arange(2 * n_pairs + 1, dtype=np.int64) * n).astype(np.int32)
    tris = (base.tris.astype(np.int64)[None] + off[:-1, None, None]).reshape(-1, 3).astype(np.int32)
    return pts.reshape(-1, 3), tris, off, n, f, base


def cpu_pair(args):
    """One pair through the CPU oracle (reference algorithm; see oracle/port.py header)."""
    i, nu = args
    from oracle import port
    from pyfocusr_b200.mesh import icosphere, perturbed_ellipsoid

    base = icosphere(nu)
    t, s = perturbed_ellipsoid(nu, 2 * i, base=base), perturbed_ellipsoid(nu, 2 * i + 1, base=base)
    np.random.seed(i)
    t0 = time.perf_counter()
    port.spectral_stage(t.points, t.tris, s.points, s.tris, N_SPECTRAL, N_EXTRA, N_SAMPLES,
                        graph_smoothing_iterations=SMOOTH_T, projection_smooth_iterations=SMOOTH_S)
    return time.perf_counter() - t0


def config_dict(pairs_per_gpu, nu, n):
    """The workload, in the same words for both arms (how each arm steps through it is in the line's `run` key)."""
    return {"workload": "configs[2]: synthetic perturbed-ellipsoid pairs, nu=%d (%d vertices/mesh), Focusr defaults "
                        "(k=7, 5000 samples, smoothing 300/40), CPD=identity" % (nu, n),
            "workload_pairs_per_gpu": pairs_per_gpu, "vertices_per_mesh": n,
            "l2": "GPU arm: working set >> L2 (batched CSR + blocks ~ %.1f GB per GPU), no flush needed; CPU arm: n/a"
                  % (pairs_per_gpu * 2 * 12e6 / 1e9)}


def dump_outputs(outs, n_eig, out_dir):
    """Write what one step returned -- `outs`: the DUMP_KEYS of SpectralBatch.run per sub-batch, sub-batches in pair
    order -- to out_dir/<name>.npy, all float64.  Per-pair results are written whole (`*_target` / `*_source`: the two
    meshes of each pair); per-vertex results for a fixed, seeded sample of DUMP_ROWS vertex positions, the same for
    targets and sources, so that two builds given the same arguments can be compared output for output."""
    import torch

    def cat(fn):
        return torch.cat([fn(o, o["spectral_weights"].shape[0]) for o in outs])

    n_vert = outs[0]["final_idx"].shape[0] // outs[0]["spectral_weights"].shape[0]   # every mesh has n_vert vertices
    tgt_vecs = cat(lambda o, p: o["eig_vecs"][:p * n_vert, :n_eig])
    rows = np.sort(np.random.RandomState(0).choice(tgt_vecs.shape[0], min(DUMP_ROWS, tgt_vecs.shape[0]), replace=False))
    rows_d = torch.from_numpy(rows).to(tgt_vecs.device)
    arrays = {"eig_vals_target": cat(lambda o, p: o["eig_vals"][:p, :n_eig]),
              "eig_vals_source": cat(lambda o, p: o["eig_vals"][p:, :n_eig]),
              "Q": cat(lambda o, p: o["Q"]),
              "spectral_weights": cat(lambda o, p: o["spectral_weights"]),
              "sample_vertex_rows": torch.from_numpy(rows),
              "eig_vecs_target": tgt_vecs[rows_d],
              "eig_vecs_source": cat(lambda o, p: o["eig_vecs"][p * n_vert:, :n_eig])[rows_d]}
    for key in ("final_idx", "weighted_avg_transformed_points", "nearest_neighbor_transformed_points"):
        arrays[key] = cat(lambda o, p: o[key])[rows_d]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float64))


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp

    from pyfocusr_b200.mesh import icosphere

    cores = os.cpu_count() or 1
    n = icosphere(a.nu).points.shape[0]
    pairs_per_step = cores
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        for w in range(a.warmup):  # full steps: every worker imports scipy and touches its pages before the clock starts
            pool.map(cpu_pair, [(w * pairs_per_step + j, a.nu) for j in range(pairs_per_step)])
        t0 = time.perf_counter()
        for s in range(a.steps):
            pool.map(cpu_pair, [(1000 + s * pairs_per_step + j, a.nu) for j in range(pairs_per_step)])
        dt = time.perf_counter() - t0
    value = a.steps * pairs_per_step / dt
    sample = ("bounded sample of the workload: %d pairs per step (not the %d of the GPU arm's step), one pair per process on "
              "%d host cores (scipy eigs/cKDTree are single-threaded)" % (pairs_per_step, a.pairs_per_gpu, cores))
    line = {"impl": "reference", "metric": "spectral-embed pairs/sec @15k verts", "value": value, "unit": "pairs/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(a.pairs_per_gpu, a.nu, n),
            "run": {"pairs_per_step": pairs_per_step, "processes": cores},
            "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for ln in self.f.read().strip().splitlines():
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        os.unlink(self.f.name)
        return out


def run_ours(a):
    import torch

    from pyfocusr_b200 import SpectralBatch, _lib
    from pyfocusr_b200 import dist as fdist

    rank, local, world = fdist.world()
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    fdist.init("nccl")
    P = a.pairs_per_gpu
    # pair i of the global batch lives on rank i mod world (SURVEY.md section 8d-3); no data-path collective.  On a GPU
    # the rank's pairs are processed as S sub-batches in flight at once (SpectralBatch.run_concurrent: one host thread +
    # CUDA stream each), so that the ALU-/latency-bound tail of one (eigsort, KNN) hides under the HBM-bound filter of another
    my_pairs = fdist.pair_shard(P * world, rank, world)
    sb = SpectralBatch(N_SPECTRAL, N_EXTRA, N_SAMPLES, SMOOTH_T, SMOOTH_S, seed=rank)
    # A/B knobs (per-call options, no process-wide state): FOCUSR_EIGS_OPTS="filter_policy=3,filter_min_blocks=6"
    if os.environ.get("FOCUSR_EIGS_OPTS"):
        sb.eigs_options = {kv.split("=")[0]: int(kv.split("=")[1]) for kv in os.environ["FOCUSR_EIGS_OPTS"].split(",") if "=" in kv}
    rng = np.random.RandomState(rank)
    jobs, jobs_e2e, h2d, n, f = [], [], 0, 0, 0
    groups = fdist.sub_batches(my_pairs, a.sub_batches)
    S = len(groups)
    for ids in groups:
        pts, tris, off, n, f, _ = make_pairs(ids, a.nu)
        pts_pin = torch.from_numpy(pts).pin_memory()
        tris_pin = torch.from_numpy(tris).pin_memory()
        sizes = np.diff(off)
        p_sub = len(ids)
        idx_t, idx_s = sb.sample_indices(sizes[:p_sub], rng), sb.sample_indices(sizes[p_sub:], rng)
        common = dict(mesh_off_host=off, n_pairs=p_sub, idx_t=idx_t, idx_s=idx_s)
        jobs.append(dict(points=pts_pin.cuda(), tris=tris_pin.cuda(), **common))
        # e2e: the whole mesh (vertices AND triangles) goes host -> device inside the timed region, as a real call does
        jobs_e2e.append(dict(points=pts_pin, tris=tris_pin, **common))
        h2d += pts_pin.numel() * 8 + tris_pin.numel() * 4
    lib = _lib.load()

    barrier = fdist.barrier
    D = max(1, a.in_flight)
    last = {}

    def certify(infos):
        """The timed run's own outputs: every mesh of the step converged (status 0) with its fp64 residual
        ||L v - theta v|| <= 1e-10 ||v||.  Raises otherwise: a throughput number from a step that did not solve its
        problems is not a number."""
        worst, fp32_steps, steps = 0.0, 0, 0
        for info in infos:
            if not (np.all(info["status"] == 0) and np.all(info["n_found"] >= sb.n)):
                raise RuntimeError("bench: a mesh of the timed step did not converge: status %s" % info["status"].tolist())
            worst = max(worst, float(info["max_residual"].max()))
            fp32_steps = max(fp32_steps, int(info["fp32_filter_degree"].max()))
            steps = max(steps, int(info["filter_degree"].max()))
        if not worst <= 1e-10:
            raise RuntimeError("bench: max residual %.3e of the timed step exceeds the tolerance 1e-10" % worst)
        return worst, fp32_steps, steps

    d2h = [0]

    def keep_info(out, k):      # resident run: nothing is read back but the solver's per-mesh report (host arrays)
        return out["eigs_info"]

    def fetch_results(out, k):  # e2e run: correspondences + weighted positions -> pinned host memory, per step
        d2h[0] = S * sum(v.nbytes for v in sb.fetch(out, slot=None).values())
        return out["eigs_info"]

    def run_steps(steps, e2e, keep_outputs=False):
        """`steps` steps of the hot path over this rank's pairs.  A step is either ONE batch of all P pairs (S = 1) with
        up to D steps in flight (SpectralBatch.run_pipelined: kernels keep their full size, the tail of a step hides under
        the filter of the next), or S sub-batches of P / S pairs run concurrently (SpectralBatch.run_concurrent).
        keep_outputs: the last step's results (device tensors) stay referenced in last["outputs"] for --dump-outputs."""
        js, consume = (jobs_e2e if e2e else jobs), (fetch_results if e2e else keep_info)
        if S == 1:
            if keep_outputs:
                def consume(out, k, base=consume):
                    if k == steps - 1:
                        last["outputs"] = [{key: out[key] for key in DUMP_KEYS}]
                    return base(out, k)
            infos = sb.run_pipelined([js[0]] * steps, depth=D, consume=consume)
            last["infos"] = infos[-1:]
        else:
            for _ in range(steps):
                outs = sb.run_concurrent(js)
                last["infos"] = [consume(o, k) for k, o in enumerate(outs)]
            if keep_outputs:
                last["outputs"] = [{key: o[key] for key in DUMP_KEYS} for o in outs]

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(steps)
        e1.record()
        barrier()
        return fdist.all_reduce_max(e0.elapsed_time(e1))  # device time, slowest rank

    run_steps(max(a.warmup, D), False)
    sampler = ClockSampler(local) if rank == 0 else None
    lib.focusr_profile_reset()
    l0 = _lib.launch_count()
    ms = timed(lambda k: run_steps(k, False, keep_outputs=bool(a.dump_outputs)), a.steps)
    launches = _lib.launch_count() - l0
    max_residual, fp32_steps, filter_steps = certify(last["infos"])
    if a.dump_outputs:
        outputs = last.pop("outputs")
        if rank == 0:
            dump_outputs(outputs, sb.n, a.dump_outputs)
        del outputs
    max_residual = fdist.all_reduce_max(max_residual)
    # With several streams in flight (steps, sub-batches, the smoothing side stream) launches interleave and a kernel's
    # duration is not defined; the per-kernel numbers (roofline) come from the same K steps run again right away, still
    # under the clock sampler, on ONE stream: steps / sub-batches one after the other, smoothing in line -- same launches,
    # same sizes, nothing else on the GPU.
    lib.focusr_profile_reset()
    ov, sb.overlap_smoothing = sb.overlap_smoothing, False
    [sb.run(**job) for job in jobs]   # warm-up of this form (the caching allocator keeps a pool per stream)
    lib.focusr_profile_reset()
    ms_kernels = timed(lambda k: [sb.run(**job) for _ in range(k) for job in jobs], a.steps)
    sb.overlap_smoothing = ov
    kernel_pass = "a second pass of the same %d steps on one stream (%d pairs per launch, smoothing in line: %.1f ms per step)" % (
        a.steps, P // S, ms_kernels / a.steps)
    prof = np.zeros(4)
    lib.focusr_profile_get(prof.ctypes.data)
    prof32, profc = np.zeros(4), np.zeros(4)
    lib.focusr_profile_get_kind(1, prof32.ctypes.data)  # filter passes on fp32 blocks (k_spmm_f32)
    lib.focusr_profile_get_kind(2, profc.ctypes.data)   # filter passes in fp32 correction form (k_spmm_corr)
    clocks = sampler.stop() if sampler else None
    run_steps(D, True)
    ms_e2e = timed(lambda k: run_steps(k, True), a.steps)
    certify(last["infos"])
    # the same steps with every filter pass in fp64 (options.mixed_precision = 0): what the fp32 inner iterations buy
    opts = dict(sb.eigs_options or {})
    sb.eigs_options = dict(opts, mixed_precision=0)
    run_steps(D, False)
    k64 = min(a.steps, 6)
    ms_fp64 = timed(lambda k: run_steps(k, False), k64) * a.steps / k64
    res_fp64, _, steps_fp64 = certify(last["infos"])
    sb.eigs_options = opts or None
    # per-stage breakdown (one extra, untimed step on one stream: sub-batches one after the other, smoothing in line;
    # times summed)
    stages = {}
    ov, sb.overlap_smoothing = sb.overlap_smoothing, False
    for job in jobs:
        sb.run(**job, record_events=True)
        for k, v in sb.timings.items():
            stages[k] = round(stages.get(k, 0.0) + v, 3)
    sb.overlap_smoothing = ov
    total_launches = fdist.all_reduce_sum(launches)
    dense = None
    if world == 1 and not a.no_dense:
        try:
            dense = dense_side_evidence(jobs[0]["points"], P // S, n)
        except Exception as exc:  # a reporting extra must never cost the bench line
            dense = {"error": repr(exc)}
    # BASELINE.json configs[3] (SURVEY.md section 8e-ii), outside the timed region: ONE 998 562-vertex icosphere, k = 10
    # smallest eigenpairs (+1 null).  N > 1: row-partitioned over all N GPUs (halo fused into the kernels over NVLink, the
    # filter passes as persistent kernels, dot products all-reduced) -- a strong-scaling number; N = 1: the single-GPU solve.
    rowpart = None
    if not a.no_rowpart:
        del jobs, jobs_e2e, last
        torch.cuda.empty_cache()
        try:
            rowpart = rowpart_1m(world)
        except Exception as exc:  # a reporting extra must never cost the bench line
            rowpart = {"error": repr(exc)}
    if rank != 0:
        fdist.finalize()
        return 0

    value = world * P * a.steps / (ms / 1e3)
    e2e = world * P * a.steps / (ms_e2e / 1e3)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    # The Chebyshev filter step exists in three forms (DESIGN.md section 4): fp64 on CSR (k_spmm), and fp32 blocks / the
    # fp32 correction form on the sliced-ELL fp32 copy of the matrix (k_filter_sell modes 0 and 3).  Each is timed live by
    # the library (CUDA events around every filter application, on the launching stream); the roofline line is the one
    # that holds the largest share of the step.
    kinds = [("fp64", "k_spmm<16,8,0> (Chebyshev filter step: CSR SpMM + three-term update, fp64 blocks)", prof),
             ("fp32", "k_filter_sell<16,4,0> (same step on fp32 blocks, sliced-ELL matrix: spectrum probe + first pass)", prof32),
             ("fp32_correction", "k_filter_sell<16,4,3> (same step in fp32 correction form: z = p(L)x - x driven by the fp64 "
                                 "residual; the pass that reaches the tolerance)", profc)]
    tpath = os.path.join(ROOT, "profiles", "filter_traffic.json")
    traffic = json.load(open(tpath)) if os.path.exists(tpath) else {}

    def kind_stats(tag, name, pr):
        ach = pr[2] / (pr[0] / 1e3) / 1e9 if pr[0] > 0 else None
        d = {"kernel": name, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
             "frac": (ach / peak) if ach else None, "traffic": None, "peak_source": peak_src, "launches": int(pr[1]),
             "avg_launch_ms": (pr[0] / pr[1]) if pr[1] else None, "bytes_per_launch": (pr[2] / pr[1]) if pr[1] else None,
             "share_of_step": (pr[0] / ms_kernels) if ms_kernels else None, "measured_in": kernel_pass}
        # DRAM traffic of the same kernel from an `ncu --set full` capture of this command (committed under
        # profiles/): dram__bytes_read.sum + dram__bytes_write.sum per launch
        rec = traffic.get("%s@%d" % (tag, 128))
        if rec:  # captured at 128 pairs per launch; a launch of a sub-batch moves the same bytes per pair
            d["traffic"] = rec["dram_bytes_per_launch"] * (P / S) / 128.0
            d["traffic_source"] = rec["source"] + ("" if P == 128 and S == 1 else "; scaled to %g pairs per launch" % (P / S))
        return d

    stats = {tag: kind_stats(tag, name, pr) for tag, name, pr in kinds}
    dominant = max(stats, key=lambda t: stats[t]["share_of_step"] or 0.0)
    roofline = stats[dominant]
    achieved = roofline["achieved"]
    knn_q = P * n  # queries per KNN call and GPU
    secondary = {"spmv_filter_hbm_gbs": achieved,
                 "filter_step_forms": {t: {k: v for k, v in st.items() if k not in ("peak", "peak_source", "bound", "unit")}
                                       for t, st in stats.items() if t != dominant},
                 "filter_share_of_step": sum(st["share_of_step"] or 0.0 for st in stats.values()),
                 "knn_queries_per_s": {"initial_k1_d3": knn_q / (stages["knn_initial"] / 1e3) if stages.get("knn_initial") else None,
                                       "final_k3_d3": knn_q / (stages["knn_final"] / 1e3) if stages.get("knn_final") else None}}
    # SURVEY.md section 8d: the other two HBM streams of the path by their compulsory bytes over the one-stream stage
    # times -- Laplacian build (read 24 N + 12 F, write adjacency + degree arrays: 12 nnz + 4 N + 16 N per mesh; the
    # row sort in between is not counted) and the smoothing passes (12 nnz + 12 N + 48 N per pass and mesh, 3 columns)
    try:
        nnz_mesh, meshes = 3.0 * f, 2.0 * P
        lap_bytes = meshes * (24.0 * n + 12.0 * f + 12.0 * nnz_mesh + 20.0 * n)
        smooth_bytes = P * (SMOOTH_T + SMOOTH_S) * (12.0 * nnz_mesh + 60.0 * n)
        secondary["other_hbm_streams"] = {
            "laplacian_build_gbs": lap_bytes / (stages["laplacian"] / 1e3) / 1e9 if stages.get("laplacian") else None,
            "smoothing_gbs": smooth_bytes / (stages["smoothing"] / 1e3) / 1e9 if stages.get("smoothing") else None,
            "smoothing_frac_of_peak": smooth_bytes / (stages["smoothing"] / 1e3) / 1e9 / peak if stages.get("smoothing") else None}
    except Exception as exc:  # a reporting extra must never cost the bench line
        secondary["other_hbm_streams"] = {"error": repr(exc)}
    secondary["rowpart_1m"] = rowpart
    if dense is not None:
        secondary["knn_frac_fp64_peak"] = dense.pop("knn_frac_fp64_peak", None)
        secondary["knn_pruned"] = dense.pop("knn_pruned", None)
        secondary["config5_k65"] = dense.pop("config5_k65", None)
        secondary["fp64_peaks"] = dense.pop("fp64_peaks", None)
        if dense:
            secondary["dense_evidence_error"] = dense
    if world == 1 and not a.no_nonsym:
        try:
            secondary["nonsym_batch"] = nonsym_batch_leg()
        except Exception as exc:  # a reporting extra must never cost the bench line
            secondary["nonsym_batch"] = {"error": repr(exc)}
        try:
            secondary["single_pair_ms"] = single_pair_leg()
        except Exception as exc:
            secondary["single_pair_ms"] = {"error": repr(exc)}
    if world == 1 and not a.no_cpu_baseline:
        secondary["widened_rows_ms"] = widened_rows_timing(a.nu)
    cpu = None
    if world == 1 and not a.no_cpu_baseline:
        t0 = time.perf_counter()
        times = [cpu_pair((5000 + j, a.nu)) for j in range(a.cpu_pairs)]
        cpu = {"value": len(times) / sum(times), "unit": "pairs/s", "cores": 1, "kind": "port",
               "sample": "%d pairs of the same workload, oracle/port.py (reference algorithm: scipy eigs shift-invert, "
                         "cKDTree, sparse smoothing) in one process, %.1f s" % (len(times), time.perf_counter() - t0)}
    secondary["value_fp64_only"] = {"value": world * P * a.steps / (ms_fp64 / 1e3), "unit": "pairs/s",
                                    "ms_per_step": ms_fp64 / a.steps, "filter_steps": steps_fp64, "max_residual": res_fp64,
                                    "note": "same step with options.mixed_precision = 0: every filter pass in fp64"}
    line = {"metric": "spectral-embed pairs/sec @15k verts", "value": value, "unit": "pairs/s", "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64 (fp32 inner filter)", "data": "synthetic",
            "max_residual": max_residual,
            "certified": "every mesh of the last timed step: status 0 and ||L v - theta v|| <= 1e-10 ||v|| in fp64 "
                         "(%d of its %d filter steps iterate in fp32)" % (fp32_steps, filter_steps),
            "precision": "results fp64 (every returned eigenpair meets ||Lv - theta v|| <= 1e-10 ||v|| in fp64; Laplacian, smoothing, "
                         "KNN, positions fp64 bit-exact); inside the eigensolver the filter passes iterate in fp32 (see "
                         "secondary_metrics.filter_step_forms), Rayleigh-Ritz and residuals in fp64",
            "config": config_dict(P, a.nu, n),
            "run": {"pairs_per_step": P, "steps_in_flight": D if S == 1 else 1, "sub_batches_in_flight": S,
                    "pairs_per_launch": P // S}, "clocks": clocks,
            "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h[0] * world,
                    "ms_per_step": ms_e2e / a.steps},
            "gpu_launches": int(total_launches), "roofline": roofline, "cpu_baseline": cpu, "stage_ms": stages, "secondary_metrics": secondary}
    print(json.dumps(line))
    fdist.finalize()
    return 0


def rowpart_1m(world, nu=316, k=11):
    """Collective: the 1M-vertex solve of BASELINE.json configs[3] on all `world` GPUs (tools/rowpart_solve.py has the
    multi-GPU driver); eigenvalues against tests/golden/large_eigs.npz (scipy, oracle/make_golden_large.py), residual
    ||L v - theta v|| recomputed on the assembled vectors.  Returns the report on rank 0."""
    import torch

    if world > 1:
        from tools.rowpart_solve import solve

        return solve(nu, k, p2p=True, shuffle=False, repeats=2, check_residual=True)
    from pyfocusr_b200._device import DeviceGraph
    from pyfocusr_b200.mesh import icosphere

    m = icosphere(nu)
    g = DeviceGraph([m.points], [m.tris])
    g.eigs_smallest(k=k, n_k_needed=k - 1)   # warm-up
    best = None
    for _ in range(2):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        vals, vecs, info = g.eigs_smallest(k=k, n_k_needed=k - 1)
        e1.record()
        torch.cuda.synchronize()
        best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
    nn = int(info["n_found"][0])
    v = vals[0, :nn].cpu().numpy()
    gold_path = os.path.join(ROOT, "tests", "golden", "large_eigs.npz")
    rel = None
    if nu == 316 and k == 11 and os.path.exists(gold_path):
        gold = np.load(gold_path)["nu316_k11"]
        rel = float(np.max(np.abs(v - gold) / gold))
    b = (nn + 7) // 8 * 8
    x = torch.zeros((g.n_points, b), dtype=torch.float64, device="cuda")
    x[:, :nn] = vecs[:, :nn]
    r = g.laplacian_apply(x)[:, :nn] - x[:, :nn] * vals[0, None, :nn]
    res = float(torch.linalg.vector_norm(r, dim=0).max())
    return {"config": "configs[3]: icosphere nu=%d (%d vertices), k=%d smallest, one GPU" % (nu, g.n_points, k), "n_gpus": 1,
            "halo": "none", "seconds": best / 1e3, "status": int(info["status"][0]), "n_found": nn,
            "outer_iterations": int(info["outer_iterations"][0]), "filter_degree": int(info["filter_degree"][0]),
            "fp32_filter_degree": int(info["fp32_filter_degree"][0]), "block": int(info["block_size"]),
            "max_residual_solver": float(info["max_residual"][0]), "max_residual_global": res,
            "max_rel_err_vs_scipy": rel, "within_1e-6": None if rel is None else bool(rel <= 1e-6)}


def dense_side_evidence(points, n_pairs, n):
    """The FP64-ALU / FP64-tensor side of the path, outside the timed region (N = 1 only; SURVEY.md section 7.3-8):
      * fp64_peaks: the denominators, measured on THIS GPU by tools/micro/fp64_peak (hand DMMA / DFMA issue loops; built
        by __graft_entry__.build()), else the figures of profiles/r2_dense_evidence.json (same pool) -- `source` says which;
      * knn_pruned: the bench-shape KNN (n_pairs segments of n x n, d = 3, k = 1 and 3) with the live count of (query,
        reference) distance evaluations, hence FP64 instructions per second (3 DSUB + 3 DMUL + 2 DADD per evaluation: no
        FMA, the sums must round as numpy's do) as a fraction of the DFMA issue peak -> knn_frac_fp64_peak;
      * config5_k65: BASELINE.json configs[4] top end, k = 65 smallest eigenpairs of the 100 002-vertex perturbed sphere
        (block 96: Gram / rotation on the FP64 tensor pipe) against the scipy golden vector."""
    import torch

    from pyfocusr_b200 import _device, _lib
    from pyfocusr_b200._device import DeviceGraph
    from pyfocusr_b200.mesh import perturbed_ellipsoid

    lib = _lib.load()
    out = {}
    exe = os.path.join(ROOT, "tools", "micro", "fp64_peak")
    peaks = None
    if os.path.exists(exe):
        try:
            peaks = json.loads(subprocess.run([exe], capture_output=True, text=True, check=True, timeout=120).stdout.strip().splitlines()[-1])
            peaks["source"] = "tools/micro/fp64_peak on this GPU (of measured)"
        except Exception:
            peaks = None
    if peaks is None:
        rec = os.path.join(ROOT, "profiles", "r2_dense_evidence.json")
        if os.path.exists(rec):
            peaks = dict(json.load(open(rec))["fp64_peaks"], source="profiles/r2_dense_evidence.json (same pool, earlier box)")
    out["fp64_peaks"] = peaks
    refs, qs = points[: n_pairs * n], points[n_pairs * n: 2 * n_pairs * n]
    seg = torch.arange(n_pairs + 1, dtype=torch.int32, device="cuda") * n
    knn = {}
    for k in (1, 3):
        kw = dict(k=k, ref_off=seg, query_off=seg, max_queries=n, max_refs=n)
        _device.knn(refs, qs, **kw)
        lib.focusr_profile_reset()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _device.knn(refs, qs, **kw)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        pr = np.zeros(4)
        lib.focusr_profile_get_kind(4, pr.ctypes.data)
        evals = float(pr[0])
        rec = {"ms": ms, "queries_per_s": n_pairs * n / ms * 1e3, "evaluations_per_query": evals / (n_pairs * n),
               "of_brute_force": evals / (float(n_pairs) * n * n), "fp64_instructions_per_s": 8.0 * evals / ms * 1e3}
        if peaks:
            rec["frac_of_dfma_issue_peak"] = rec["fp64_instructions_per_s"] / (peaks["dfma_ginstr_per_s"] * 1e9)
        knn["k%d_d3" % k] = rec
    out["knn_pruned"] = knn
    out["knn_frac_fp64_peak"] = {k: v.get("frac_of_dfma_issue_peak") for k, v in knn.items()}
    m = perturbed_ellipsoid(100, seed=5, semi_axes=(1.0, 1.0, 1.0))
    g = DeviceGraph([m.points], [m.tris])
    k = 65
    g.eigs_smallest(k=k, n_k_needed=k - 1)
    best = None
    for _ in range(2):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        vals, vecs, info = g.eigs_smallest(k=k, n_k_needed=k - 1)
        e1.record()
        torch.cuda.synchronize()
        best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
    rec = {"seconds": best / 1e3, "vertices": int(g.n_points), "block": int(info["block_size"]),
           "outer_iterations": int(info["outer_iterations"][0]), "filter_degree": int(info["filter_degree"][0]),
           "max_residual": float(info["max_residual"][0]), "status": int(info["status"][0])}
    gold_path = os.path.join(ROOT, "tests", "golden", "large_eigs.npz")
    if os.path.exists(gold_path):
        gold = np.load(gold_path)["nu100_seed5_k65"]
        v = vals[0, : k - 1].cpu().numpy()
        rec["max_rel_err_vs_scipy"] = float(np.max(np.abs(v - gold[: k - 1]) / gold[: k - 1]))
    rec["fp64_tensor_pipe"] = ("ncu of this solve: profiles/r2_summary.md (k_gram_wide<96>, k_rotate<96>: "
                               "sm__inst_executed_pipe_tensor_subpipe_dmma / DMMA-active)")
    out["config5_k65"] = rec
    return out


def nonsym_batch_leg(n_pairs=32, reps=2):
    """BASELINE.json configs[0] as a batch, outside the timed region (N = 1 only): `n_pairs` jittered copies of the
    reference's own shipped 15k pair (tests/golden/meshes.npz; open meshes -> structurally NON-symmetric adjacency, 2
    unreferenced vertices in the source -> the retry contract ends at k = 14 with 11 pairs) through the same batched
    pipeline.  The eigensolve takes the non-symmetric path: Euclidean projection, fp64 filter steps on CSR, the general
    b x b Rayleigh-Ritz step on the device (one CTA per mesh), b = 48."""
    import torch

    from pyfocusr_b200 import SpectralBatch

    z = np.load(os.path.join(ROOT, "tests", "golden", "meshes.npz"))
    tp, tt = z["target_mesh_15k_points"], z["target_mesh_15k_tris"].astype(np.int64)
    sp, st = z["source_mesh_15k_points"], z["source_mesh_15k_tris"].astype(np.int64)
    rng = np.random.RandomState(7)
    pts, tris, off = [], [], [0]
    for base_p, base_t in ((tp, tt), (sp, st)):
        scale = 1e-4 * float(np.ptp(base_p, axis=0).max())
        for i in range(n_pairs):
            pts.append(base_p + (scale * rng.randn(*base_p.shape) if i else 0.0))   # copy 0 is the shipped mesh itself
            tris.append(base_t + off[-1])
            off.append(off[-1] + base_p.shape[0])
    pts_d = torch.from_numpy(np.ascontiguousarray(np.concatenate(pts))).cuda()
    tris_d = torch.from_numpy(np.concatenate(tris).astype(np.int32)).cuda()
    off = np.asarray(off, dtype=np.int32)
    sb = SpectralBatch(N_SPECTRAL, N_EXTRA, N_SAMPLES, SMOOTH_T, SMOOTH_S, seed=3)
    out = sb.run(pts_d, tris_d, off, n_pairs)   # warm-up
    best = None
    for _ in range(reps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = sb.run(pts_d, tris_d, off, n_pairs)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    info = out["eigs_info"]
    ok = bool(np.all(info["status"] == 0))
    # the same batch with every filter pass in fp64 (what the fp32 forms buy on the non-symmetric path)
    sb.eigs_options = dict(mixed_precision=0)
    sb.run(pts_d, tris_d, off, n_pairs)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out64 = sb.run(pts_d, tris_d, off, n_pairs)
    e1.record()
    torch.cuda.synchronize()
    ms64 = e0.elapsed_time(e1)
    return {"config": "configs[0] as a batch: %d jittered copies of the shipped 15k pair (non-symmetric adjacency)" % n_pairs,
            "pairs_per_s": n_pairs / (best / 1e3), "ms_per_batch": best, "block": int(info["block_size"]),
            "fp32_filter_degree": int(info["fp32_filter_degree"].max()),
            "pairs_per_s_fp64_only": n_pairs / (ms64 / 1e3), "filter_degree_fp64_only": int(out64["eigs_info"]["filter_degree"].max()),
            "all_converged": ok, "max_residual": float(info["max_residual"].max()),
            "k_final": [int(info["k_final"][0]), int(info["k_final"][n_pairs])],
            "pairs_found": [int(info["n_found"][0]), int(info["n_found"][n_pairs])],
            "outer_iterations": int(info["outer_iterations"].max()), "filter_degree": int(info["filter_degree"].max())}


def single_pair_leg(reps=5):
    """BASELINE.json configs[0] and configs[1] through the drop-in API, outside the timed region (N = 1 only): the
    reference's own shipped meshes (tests/golden/meshes.npz), `Focusr(target, source, ...)` + `align_maps()` with ICP off
    and CPD = identity (BASELINE.md section 3), wall-clock with the device synchronised, median of `reps` after one
    warm-up call.  Latency of ONE pair, not throughput: the batched numbers are the headline."""
    import torch

    import pyfocusr_b200 as pyfocusr
    from pyfocusr_b200.mesh import PolyData

    z = np.load(os.path.join(ROOT, "tests", "golden", "meshes.npz"))
    out = {}
    for tag, (tn, sn), kw in (("configs0_15k_pair_defaults", ("target_mesh_15k", "source_mesh_15k"), {}),
                              ("configs1_5k_pair_n_spectral_features_10", ("target_mesh", "source_mesh"), dict(n_spectral_features=10))):
        mt, ms = PolyData(z[tn + "_points"], z[tn + "_tris"]), PolyData(z[sn + "_points"], z[sn + "_tris"])
        times = []
        for rep in range(reps + 1):
            np.random.seed(0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f = pyfocusr.Focusr(mt, ms, icp_register_first=False, list_features_to_calc=[], registration="identity", **kw)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            f.align_maps()
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            if rep:
                times.append(((t1 - t0) * 1e3, (t2 - t1) * 1e3))
        ctor, align = np.median([t[0] for t in times]), np.median([t[1] for t in times])
        out[tag] = {"constructor_ms": float(ctor), "align_maps_ms": float(align), "total_ms": float(ctor + align),
                    "vertices": [int(mt.points.shape[0]), int(ms.points.shape[0])],
                    "eigenpairs_kept": [int(f.graph_target.eig_vals.size), int(f.graph_source.eig_vals.size)],
                    "correspondences": int(np.asarray(f.corresponding_target_idx_for_each_source_pt).size)}
    return out


def widened_rows_timing(nu):
    """SURVEY.md section 8f rows, outside the timed region (N = 1 only): one CPD registration at the reference's
    default sizes on the spectral-coordinate-like synthetic problem of tools/cpd_bench.py, ICP and curvatures on one
    synthetic pair.  Wall-clock with device synchronisation, second run of each (the first warms the allocator)."""
    import torch

    from pyfocusr_b200 import _device
    from pyfocusr_b200.cpd import affine_registration, deformable_registration
    from pyfocusr_b200.mesh import ellipsoid_pair
    from tools.cpd_bench import problem

    def timed(fn):
        out = None
        for _ in range(2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) * 1e3
        return dt, out

    x, y = problem(0, 5000, 5000, 3)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    res = {}

    def run_affine():
        reg = affine_registration(X=xd, Y=yd, max_iterations=100, tolerance=1e-8)
        reg.register()
        return reg

    res["cpd_affine_5000x5000"], aff = timed(run_affine)
    ty = aff.transform_point_cloud(yd)

    def run_def():
        reg = deformable_registration(X=xd, Y=ty, max_iterations=1000, tolerance=1e-8, alpha=0.5, beta=3.0, num_eig=100)
        reg.register()
        return reg

    res["cpd_deformable_5000x5000_num_eig100"], dreg = timed(run_def)
    res["cpd_iterations"] = [int(aff.iteration), int(dreg.iteration)]
    t, s_ = ellipsoid_pair(0, nu)
    res["icp_100it_1000_landmarks"], _ = timed(lambda: _device.icp(t.points, t.tris, s_.points))
    res["curvatures_one_mesh"], _ = timed(lambda: _device.curvatures(t.points, t.tris))
    # the 'hungarian' correspondence (focusr.py:340-349): N x N assignment on the GPU next to scipy's on one host core,
    # on a geometric instance with long augmenting paths (4000 points of an ellipsoid matched to displaced copies)
    from scipy.optimize import linear_sum_assignment
    rng = np.random.RandomState(11)
    p = rng.randn(4000, 3)
    p = p / np.linalg.norm(p, axis=1)[:, None] * np.array([1.0, 0.8, 0.6])
    q = p[rng.permutation(4000)] + 0.3 * rng.randn(4000, 3)
    cost = _device.cdist(q, p)
    res["hungarian_lsap_4000x4000"], (_, col) = timed(lambda: _device.linear_sum_assignment(cost))
    t0 = time.perf_counter()
    _, col_ref = linear_sum_assignment(cost.cpu().numpy())
    res["hungarian_lsap_4000x4000_scipy_1core"] = (time.perf_counter() - t0) * 1e3
    res["hungarian_lsap_equal_to_scipy"] = bool(np.array_equal(col, col_ref))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs-per-gpu", type=int, default=128)
    ap.add_argument("--in-flight", type=int, default=2, help="steps in flight at once (whole batches, one stream each)")
    ap.add_argument("--sub-batches", type=int, default=1,
                    help="> 1: split a step's pairs into sub-batches run concurrently instead of pipelining whole steps")
    ap.add_argument("--nu", type=int, default=NU)
    ap.add_argument("--cpu-pairs", type=int, default=24)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-rowpart", action="store_true", help="skip the 1M-vertex solve reported under secondary_metrics")
    ap.add_argument("--no-dense", action="store_true", help="skip the KNN / k = 65 FP64 evidence reported under secondary_metrics")
    ap.add_argument("--no-nonsym", action="store_true", help="skip the non-symmetric batch reported under secondary_metrics")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0's pairs) to DIR/<name>.npy in float64")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results; the reference arm has none to write")
    return run_reference(a) if a.impl == "reference" else run_ours(a)


if __name__ == "__main__":
    sys.exit(main())
