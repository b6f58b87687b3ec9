"""Batched ICP at bench shape: 128 pairs of ``mesh.ellipsoid_pair(i, 39)`` (15 212 vertices, 30 420 triangles), every
source misaligned by a seeded random rigid motion (rotation up to 20 degrees, translation up to 5 mm), 100 iterations x
1000 landmarks (the reference's ICP).  Prints one JSON line with the GPU's name and power limit.

    python tools/batch_icp_bench.py --parent HEAD^            # in a git checkout
    git archive HEAD^ | tar -x -C /tmp/parent && python tools/batch_icp_bench.py --parent-src /tmp/parent


  * batched ICP of the 128 pairs (``focusr_icp_batch``, one call), device time, warm;
  * the same pairs through ``_device.icp``, one call each (wall clock, each call reads its matrix back), and through the
    library's ``focusr_icp`` one call after the other on resident inputs (device time), for this build and -- with
    ``--parent REV`` or ``--parent-src DIR`` -- for the library of another source tree, built by this script into a
    temporary directory (alternating), with a bit-for-bit comparison of their matrices on these pairs and on the inputs
    of tests/test_icp.py;
  * ``SpectralBatch.run`` pairs/s with ICP on and off (``registration="identity"``);
  * exact closest-point evaluations per landmark and iteration, and the batched time with 64-triangle tiles, each from a
    build of icp.cu with ``-DFB_ICP_COUNT`` / ``-DFB_ICP_TILE=64`` made in a temporary directory and run in a child
    process (``--no-variants`` skips them).
"""
from __future__ import annotations

import argparse
import ctypes as C
import glob
import hashlib
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


def _rot(rv):
    from scipy.spatial.transform import Rotation

    return Rotation.from_rotvec(rv).as_matrix()


def make_batch(n_pairs, seed=0):
    """targets then sources (SpectralBatch's order); sources misaligned by rotations <= 20 deg, translations <= 5 mm"""
    from pyfocusr_b200 import mesh as fmesh
    from pyfocusr_b200.batch import SpectralBatch

    base = fmesh.icosphere(39)
    rng = np.random.RandomState(seed)
    targets, sources = [], []
    for i in range(n_pairs):
        t, s = fmesh.ellipsoid_pair(i, 39, base=base)
        axis = rng.normal(size=3)
        axis /= np.linalg.norm(axis)
        shift = rng.normal(size=3)
        shift *= rng.uniform(0.0, 5.0) / np.linalg.norm(shift)
        r = _rot(axis * np.deg2rad(rng.uniform(0.0, 20.0)))
        targets.append(t)
        sources.append(fmesh.PolyData(s.points @ r.T + shift, s.tris))
    pts, tris, off, P = SpectralBatch.pack_meshes(targets, sources)
    toff = np.zeros(2 * P + 1, dtype=np.int32)
    toff[1:] = np.cumsum([m.tris.shape[0] for m in targets + sources])
    return targets, sources, pts, tris, off, toff


class OnePair:
    """``focusr_icp`` of one library (this build or another) on device tensors, no read-back"""

    def __init__(self, lib):
        self.lib = lib
        lib.focusr_icp_workspace_bytes.restype = C.c_size_t
        lib.focusr_icp_workspace_bytes.argtypes = [C.c_int, C.c_int]
        lib.focusr_icp.restype = C.c_int
        lib.focusr_icp.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        lib.focusr_last_error.restype = C.c_char_p

    def __call__(self, tp, tt, sp, mat, moved, ws, iters=100, landmarks=1000, similarity=0, match=1):
        import torch

        rc = self.lib.focusr_icp(tp.data_ptr(), tp.shape[0], tt.data_ptr(), tt.shape[0], sp.data_ptr(), sp.shape[0],
                                 landmarks, iters, similarity, match, mat.data_ptr(), moved.data_ptr(), ws.data_ptr(),
                                 ws.numel(), torch.cuda.current_stream().cuda_stream)
        if rc != 0:
            raise RuntimeError(self.lib.focusr_last_error().decode())

    def ws(self, ns, nf):
        import torch

        return torch.empty(int(self.lib.focusr_icp_workspace_bytes(ns, nf)), dtype=torch.uint8, device="cuda")


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


def batched(args, pts, tris, off, toff, P):
    """ms of one batched call, its matrices, and the evaluations per landmark and iteration (counting builds only)"""
    import torch

    from pyfocusr_b200 import _device, _lib

    dp, dt = pts.cuda(), tris.cuda()
    fixed, moving = np.arange(P, dtype=np.int32), np.arange(P, 2 * P, dtype=np.int32)

    def run():
        return _device.icp_batch_device(dp, dt, off, toff, fixed, moving, max_iterations=args.iters,
                                        max_landmarks=args.landmarks)

    ms = timed(run, args.reps)
    out4 = np.zeros(4)
    _lib.load().focusr_profile_reset()
    mats, _ = run()
    _lib.load().focusr_profile_get_kind(5, out4.ctypes.data)
    n_lm = sum(_device.icp_landmarks(int(off[P + p + 1] - off[P + p]), args.landmarks)[1] for p in range(P))
    return ms, mats.cpu().numpy(), float(out4[0]) / (n_lm * args.iters)


def build_variant(defines, tmp):
    objs = [o for o in glob.glob(os.path.join(CSRC, "build", "*.o")) if os.path.basename(o) != "icp.o"]
    tag = "_".join(d.lstrip("-D").replace("=", "") for d in defines)
    obj, so = os.path.join(tmp, "icp_%s.o" % tag), os.path.join(tmp, "libfocusr_b200_%s.so" % tag)
    flags = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-Xcompiler", "-fopenmp"]
    subprocess.check_call([NVCC] + flags + defines + ["-c", os.path.join(CSRC, "icp.cu"), "-o", obj])
    subprocess.check_call([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", so] + objs + [obj, "-lcudart", "-lgomp"])
    return so


def build_parent(args, tmp):
    """the other tree's csrc/ and include/ copied to tmp and built there with its own build.sh; returns the library"""
    import shutil

    src = args.parent_src
    if args.parent:
        src = os.path.join(tmp, "tree")
        os.makedirs(src)
        archive = subprocess.run(["git", "-C", ROOT, "archive", args.parent], check=True, capture_output=True).stdout
        subprocess.run(["tar", "-x", "-C", src], input=archive, check=True)
    dst = os.path.join(tmp, "parent")
    shutil.copytree(os.path.join(src, "pyfocusr_b200", "csrc"), os.path.join(dst, "pyfocusr_b200", "csrc"),
                    ignore=shutil.ignore_patterns("build", "*.so", "*.o"))
    shutil.copytree(os.path.join(src, "include"), os.path.join(dst, "include"))
    subprocess.check_call(["sh", os.path.join(dst, "pyfocusr_b200", "csrc", "build.sh")], stdout=subprocess.DEVNULL)
    return os.path.join(dst, "pyfocusr_b200", "csrc", "libfocusr_b200.so")


def child(args):
    """one batched measurement with the library named by FOCUSR_B200_LIB (a variant build)"""
    _, _, pts, tris, off, toff = make_batch(args.pairs)
    ms, mats, evals = batched(args, pts, tris, off, toff, args.pairs)
    print(json.dumps(dict(ms=ms, evals_per_landmark_iteration=evals, matrices_sha1=hashlib.sha1(mats.tobytes()).hexdigest())))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=128)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--landmarks", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent", default=None, help="git revision whose library focusr_icp is compared with (git archive)")
    ap.add_argument("--parent-src", default=None, help="source tree whose library focusr_icp is compared with")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.child:
        return child(args)
    import torch

    from pyfocusr_b200 import _device, _lib
    from pyfocusr_b200.batch import SpectralBatch

    assert torch.cuda.is_available(), "batch_icp_bench needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    P = args.pairs
    targets, sources, pts, tris, off, toff = make_batch(P)
    res = dict(gpu=smi, pairs=P, iterations=args.iters, landmarks=args.landmarks, triangles_per_target=int(targets[0].tris.shape[0]))

    ms, mats_batch, _ = batched(args, pts, tris, off, toff, P)
    res["batched_ms"] = ms

    # one call per pair through the Python wrapper (uploads, launches, matrix read-back)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mats_loop = np.stack([_device.icp(t.points, t.tris, s.points)[0] for t, s in zip(targets, sources)])
    torch.cuda.synchronize()
    res["device_icp_loop_ms"] = 1e3 * (time.perf_counter() - t0)
    res["device_icp_loop_equals_batched"] = bool(np.array_equal(mats_loop, mats_batch))

    # focusr_icp one pair after the other on resident inputs: this build and, alternating, the other one
    libs = {"new": OnePair(_lib.load())}
    scratch = tempfile.TemporaryDirectory()
    if args.parent or args.parent_src:
        libs["parent"] = OnePair(C.CDLL(build_parent(args, scratch.name)))
    dev = [(torch.from_numpy(t.points).cuda(), torch.from_numpy(t.tris.astype(np.int32)).cuda(), torch.from_numpy(s.points).cuda())
           for t, s in zip(targets, sources)]
    outs = {k: (torch.empty((P, 16), dtype=torch.float64, device="cuda"), torch.empty_like(dev[0][2]),
                f.ws(dev[0][2].shape[0], dev[0][1].shape[0])) for k, f in libs.items()}
    loops = {k: [] for k in libs}
    for rep in range(3):
        for k, f in libs.items():
            mat, moved, ws = outs[k]
            loops[k].append(timed(lambda: [f(tp, tt, sp, mat[p], moved, ws) for p, (tp, tt, sp) in enumerate(dev)], 1))
    for k in libs:
        res["focusr_icp_loop_ms_" + k] = loops[k]
        res["focusr_icp_one_pair_ms_" + k] = min(loops[k]) / P
    res["focusr_icp_new_equals_batched"] = bool(np.array_equal(outs["new"][0].cpu().numpy().reshape(P, 4, 4), mats_batch))
    if "parent" in libs:
        res["parent_equals_new_bench_pairs"] = bool(np.array_equal(outs["parent"][0].cpu().numpy(), outs["new"][0].cpu().numpy()))
        res["batched_speedup_over_parent_loop"] = min(loops["parent"]) / ms
        # tests/test_icp.py's inputs
        from pyfocusr_b200 import mesh as fmesh

        tm = fmesh.perturbed_ellipsoid(8, 0, semi_axes=(43.0, 25.0, 33.0))
        sm = fmesh.perturbed_ellipsoid(8, 1, semi_axes=(43.0, 25.0, 33.0))
        same, worst = True, 0.0
        for similarity in (0, 1):
            src = (1.08 if similarity else 1.0) * (sm.points @ _rot([0.12, -0.1, 0.2]).T) + np.array([4.0, -3.0, 2.0])
            tp, tt, sp = torch.from_numpy(tm.points).cuda(), torch.from_numpy(tm.tris.astype(np.int32)).cuda(), torch.from_numpy(src).cuda()
            for iters, lm, match in ((1, 1000, 1), (12, 100, 1), (40, 57, 1), (3, 80, 0), (100, 1000, 1)):
                got = {}
                for k, f in libs.items():
                    mat, moved = torch.empty(16, dtype=torch.float64, device="cuda"), torch.empty_like(sp)
                    f(tp, tt, sp, mat, moved, f.ws(sp.shape[0], tt.shape[0]), iters, lm, similarity, match)
                    got[k] = (mat.cpu().numpy(), moved.cpu().numpy())
                same &= all(np.array_equal(got["new"][i], got["parent"][i]) for i in range(2))
                worst = max(worst, float(np.max(np.abs(got["new"][0] - got["parent"][0]))))
        res["parent_equals_new_test_icp_inputs"] = bool(same)
        res["parent_new_max_abs_diff_test_icp_inputs"] = worst

    # the spectral stage with and without ICP
    dp = pts.cuda()
    for on in (False, True):
        sb = SpectralBatch(registration="identity", icp_register_first=on)
        run = lambda: sb.run(dp, tris, off, P, tri_off_host=toff)  # noqa: E731
        run()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(2):
            run()
        torch.cuda.synchronize()
        res["spectral_pairs_per_s_icp_" + ("on" if on else "off")] = 2 * P / (time.perf_counter() - t0)

    if not args.no_variants:
        with tempfile.TemporaryDirectory() as tmp:
            for name, defines in (("count", ["-DFB_ICP_COUNT"]), ("tile64", ["-DFB_ICP_TILE=64", "-DFB_ICP_COUNT"]),
                                  ("tile32", ["-DFB_ICP_TILE=32", "-DFB_ICP_COUNT"])):
                so = build_variant(defines, tmp)
                env = dict(os.environ, FOCUSR_B200_LIB=so)
                line = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--pairs", str(P), "--iters",
                                       str(args.iters), "--landmarks", str(args.landmarks), "--reps", str(args.reps)],
                                      env=env, capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1]
                res["variant_" + name] = json.loads(line)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
