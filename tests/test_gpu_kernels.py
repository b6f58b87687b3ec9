"""The eigensolver's kernels one step at a time against a high-precision reference of the same formula.

The solver checks its Ritz pairs in fp64, so a wrong fp32 filter step only costs it extra passes; these tests look at
every kernel output instead.  tests/kernel_probe builds a test-only library that launches k_filter_sell (sell.cu),
k_spmm (spmm.cu) and the Gram / rotation steps of eigs.cu on arrays this file owns.  Every element must lie within the
rounding bound of its formula,

    |got - ref| <= (len_r + 8) * u * S_r,

where ref is the formula in float64 (fp32 kernels) or long double (fp64 kernels) on exactly the inputs the kernel sees
(fp32-rounded weights, degrees and blocks for the fp32 forms), S_r is the same formula with every term replaced by its
absolute value, len_r the number of stored entries of the row (for the Gram pair: the rows of the mesh) and u the unit
roundoff of the kernel's arithmetic.  This is a rounding bound, not a tuned tolerance: one matrix entry dropped or moved
to the neighbouring column exceeds it (test_rounding_bound_flags_a_wrong_entry, which needs no GPU).

Each sweep runs on two batches: a small one, which the filter and SpMM launchers give one pass per CTA, and the same
meshes followed by enough others that the launchers switch to CTAs of 256 rows (sell.cu launch_fs_b, spmm.cu
launch_spmm_b).  A row's arithmetic does not depend on that choice, so the rows the two batches share must be
bit-identical, and so must every cache-policy / prefetch / launch / occupancy variant of the fp32 filter step.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import sparse

from oracle import port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROBE_DIR = os.path.join(ROOT, "tests", "kernel_probe")
CSRC = os.path.join(ROOT, "pyfocusr_b200", "csrc")

BLOCKS = list(range(8, 97, 8))
U32, U64 = 2.0 ** -24, 2.0 ** -53
SELL_ROWS, FS_ROWS, GRAM_ROWS = 64, 256, 1024
N_STEPS, STEP = 3, 2
# (mode, has_prev) of the fp32 filter step, sell.cu:232-237.  0: plain fp32 step; 1: first step of a pass (fp64 y, no
# x_prev term, also writes the fp32 copy of y); 2: last plain step (fp64 out); 3: correction step (per-column tables, r,
# z_prev when has_prev); 4: last correction step (fp64 x += the step).
FILTER_RUNS = [(0, 1), (1, 0), (2, 1), (3, 1), (3, 0), (4, 1)]


# ------------------------------------------------------------------------------------------------ reference helpers
def csr_apply(rp, cols, w, y, dtype):
    """(A y, |A| |y|) in `dtype`, row by row in entry order (a loop over the k-th entries of all rows)."""
    n = rp.size - 1
    lens = np.diff(rp)
    y = y.astype(dtype)
    ay = np.abs(y)
    acc = np.zeros((n, y.shape[1]), dtype=dtype)
    aacc = np.zeros_like(acc)
    wd = w.astype(dtype)
    for k in range(int(lens.max()) if n else 0):
        rows = np.nonzero(lens > k)[0]
        p = rp[rows] + k
        acc[rows] += wd[p, None] * y[cols[p]]
        aacc[rows] += np.abs(wd[p, None]) * ay[cols[p]]
    return acc, aacc


def block_apply(db, b, fp32):
    """csr_apply of the first b columns of db's y block, made once per (b, form): (fp32-rounded y and weights, float64)
    for the fp32 steps, (y, weights, long double) for the fp64 ones."""
    cache = db.__dict__.setdefault("_applied", {})
    if (b, fp32) not in cache:
        if any(k[0] != b for k in cache):
            cache.clear()
        h = db.h
        if fp32:
            y = db.y[:, :b].astype(np.float32).astype(np.float64)
            cache[b, fp32] = csr_apply(h.rp, h.cols, h.w.astype(np.float32).astype(np.float64), y, np.float64)
        else:
            cache[b, fp32] = csr_apply(h.rp, h.cols, h.w, db.y[:, :b], np.longdouble)
    return cache[b, fp32]


def step_ref(acc, aacc, y, d, di, cc, al, ga=None, xp=None, r=None):
    """al ((L - cc) y [+ r]) [- ga xp] and its absolute-value twin; L y = di (d y - acc).  al, ga, cc broadcast per row."""
    lap = di * (d * y - acc)
    s_lap = np.abs(di) * (np.abs(d * y) + aacc)
    v = lap - cc * y
    s = s_lap + np.abs(cc * y)
    if r is not None:
        v = v + r
        s = s + np.abs(r)
    v = al * v
    s = np.abs(al) * s
    if ga is not None:
        v = v - ga * xp
        s = s + np.abs(ga * xp)
    return v, s


def rounding_bound(s, lens, u):
    """(len + 8) u S elementwise, len per row (the first axis)."""
    lens = np.asarray(lens, dtype=np.float64).reshape(-1, *([1] * (np.ndim(s) - 1)))
    return (lens + 8.0) * u * np.asarray(s, dtype=np.float64)


def bound_ratio(got, ref, bound):
    """|got - ref| / bound elementwise; > 1 is a violation."""
    err = np.abs(np.asarray(got, dtype=np.float64) - np.asarray(ref, dtype=np.float64))
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(err == 0.0, 0.0, err / bound)


def assert_within(ratios, key, got, ref, bound):
    rt = bound_ratio(got, ref, bound)
    assert np.all(np.isfinite(np.asarray(got, dtype=np.float64))), key
    worst = float(rt.max()) if rt.size else 0.0
    if worst > 1.0:
        idx = np.unravel_index(int(np.argmax(rt)), rt.shape)
        pytest.fail("%s: |got - ref| exceeds the rounding bound %.3g times at %s (got %r, ref %r)"
                    % (key, worst, idx, np.asarray(got)[idx], np.asarray(ref)[idx]))
    k = key.split(" b=")[0]
    ratios[k] = max(ratios.get(k, 0.0), worst)


# ------------------------------------------------------------------------------------------------ graphs
def artificial_graph(n, seed, long_row=None, zero_rows=(), one_way=0.1):
    """CSR of n rows: ring and random neighbours, random weights; the pattern is symmetric except a fraction `one_way`
    of the entries whose mirror is dropped; `long_row` gets >= 320 entries; `zero_rows` have no entries either way."""
    rng = np.random.default_rng(seed)
    src = [np.arange(n), np.arange(n)]
    dst = [(np.arange(n) + 1) % n, (np.arange(n) + 2) % n]
    extra = rng.integers(0, n, size=(2 * n,))
    src.append(rng.integers(0, n, size=extra.size))
    dst.append(extra)
    s, t = np.concatenate(src), np.concatenate(dst)
    keep = s != t
    s, t = s[keep], t[keep]
    mirror = rng.random(s.size) >= one_way
    s, t = np.concatenate([s, t[mirror]]), np.concatenate([t, s[mirror]])
    if long_row is not None:
        others = np.setdiff1d(rng.choice(n, size=min(n, 340), replace=False), [long_row])
        s = np.concatenate([s, np.full(others.size, long_row)])
        t = np.concatenate([t, others])
    for z in zero_rows:
        keep = (s != z) & (t != z)
        s, t = s[keep], t[keep]
    a = sparse.csr_matrix((rng.uniform(0.05, 3.0, size=s.size), (s, t)), shape=(n, n))
    a.sum_duplicates()
    a.sort_indices()
    return a


def icosphere_graph(nu):
    from pyfocusr_b200.mesh import icosphere

    m = icosphere(nu)
    return port.adjacency(m.points, m.tris)


class Batch:
    """Block-diagonal batch of graphs with the host arrays the references need."""

    def __init__(self, graphs):
        a = sparse.block_diag(graphs, format="csr")
        a.sort_indices()
        self.sizes = np.array([g.shape[0] for g in graphs])
        self.off = np.zeros(len(graphs) + 1, dtype=np.int32)
        self.off[1:] = np.cumsum(self.sizes)
        self.n, self.m = int(self.off[-1]), len(graphs)
        self.max_rows = int(self.sizes.max())
        self.rp, self.cols, self.w = a.indptr.astype(np.int32), a.indices.astype(np.int32), a.data.astype(np.float64)
        self.lens = np.diff(self.rp)
        self.deg = port.row_sums_sequential(a)
        self.dinv = port.degree_inv(self.deg)
        self.mesh_of_row = np.repeat(np.arange(self.m), self.sizes)
        self.info = np.zeros((self.m, 8), dtype=np.int32)  # FOCUSR_MESH_INFO_INTS; [4] = longest row
        for k in range(self.m):
            self.info[k, 4] = int(self.lens[self.off[k]:self.off[k + 1]].max(initial=0))
        pattern = (a != 0).astype(np.int8)
        self.one_way = int((pattern != pattern.T).nnz)


def small_graphs():
    """Row counts 1024, 2049, 1023, 37, 642 and 300: n mod 64 in {0, 1, 63} and n mod 1024 in {0, 1, 1023}, a mesh
    smaller than one slice, meshes smaller than one Gram chunk; a row of >= 320 entries inside a slice of short rows,
    zero-degree rows (one of them alone in the last slice of its mesh), one-way entries."""
    return [
        artificial_graph(1024, 1),
        artificial_graph(2049, 2, long_row=100, zero_rows=(5, 2048)),
        artificial_graph(1023, 3, zero_rows=(1022,)),
        artificial_graph(37, 4, zero_rows=(0,)),
        icosphere_graph(8),
        artificial_graph(300, 5, long_row=299, one_way=0.5),
    ]


def takes_256_row_form(batch, sms):
    # sell.cu launch_fs_b / spmm.cu launch_spmm_b: one pass per CTA when a batch gives fewer than two waves of 256-row CTAs
    return -(-batch.max_rows // FS_ROWS) * batch.m >= 2 * sms


# ------------------------------------------------------------------------------------------------ CPU-only self-check
def test_rounding_bound_flags_a_wrong_entry():
    """The bound is tight enough to see one wrong matrix entry: a correctly rounded result passes, a reference with one
    entry of the longest row dropped or moved to the neighbouring column fails on that row (fp32 and fp64 forms)."""
    b = Batch([artificial_graph(2049, 2, long_row=100, zero_rows=(5, 2048))])
    rng = np.random.default_rng(7)
    y = rng.standard_normal((b.n, 16))
    w32 = b.w.astype(np.float32).astype(np.float64)
    row = int(np.argmax(b.lens))
    assert b.lens[row] >= 300
    p = b.rp[row] + b.lens[row] // 2

    for u, w, dtype, rnd in ((U32, w32, np.float64, np.float32), (U64, b.w, np.longdouble, np.float64)):
        d, di = b.deg[:, None], b.dinv[:, None]
        if rnd is np.float32:
            y_in = y.astype(np.float32).astype(np.float64)
            d, di = d.astype(np.float32).astype(np.float64), di.astype(np.float32).astype(np.float64)
        else:
            y_in = y
        acc, aacc = csr_apply(b.rp, b.cols, w, y_in, dtype)
        ref, s = step_ref(acc, aacc, y_in.astype(dtype), d, di, 0.9, 1.3, 0.4, y_in.astype(dtype))
        got = ref.astype(rnd)
        assert bound_ratio(got, ref, rounding_bound(s, b.lens, u)).max() <= 1.0
        for mutate in ("drop", "move"):
            cols = b.cols.copy()
            w_m = w.copy()
            if mutate == "drop":
                w_m[p] = 0.0
            else:
                cols[p] = cols[p] + 1 if cols[p] + 1 < b.n else cols[p] - 1
            acc_m, aacc_m = csr_apply(b.rp, cols, w_m, y_in, dtype)
            ref_m, s_m = step_ref(acc_m, aacc_m, y_in.astype(dtype), d, di, 0.9, 1.3, 0.4, y_in.astype(dtype))
            bad = bound_ratio(got, ref_m, rounding_bound(s_m, b.lens, u)) > 1.0
            assert bad[row].mean() >= 0.9, (u, mutate, bad[row].mean())
            assert not np.any(np.delete(bad, row, axis=0)), (u, mutate)


# ------------------------------------------------------------------------------------------------ GPU: the probe
@pytest.fixture(scope="module")
def torch():
    import torch

    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module")
def probe(torch):
    """tests/kernel_probe/libfocusr_probe.so, built when it is missing or older than its sources or the product's."""
    so = os.path.join(PROBE_DIR, "libfocusr_probe.so")
    srcs = [os.path.join(PROBE_DIR, f) for f in ("probe.cu", "build.sh")]
    srcs += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h", ".hpp"))]
    srcs.append(os.path.join(ROOT, "include", "focusr_b200.h"))
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(f) for f in srcs):
        subprocess.check_call(["sh", os.path.join(PROBE_DIR, "build.sh")])
    lib = C.CDLL(so)
    vp, i = C.c_void_p, C.c_int
    lib.probe_last_error.restype = C.c_char_p
    lib.probe_sell_entries_cap.restype = C.c_longlong
    lib.probe_sell_entries_cap.argtypes = [vp, vp, i]
    lib.probe_scan_tmp_ints.argtypes = [i]
    lib.probe_sell_build.argtypes = [vp] * 7 + [i, i] + [vp] * 7
    lib.probe_filter_sell.argtypes = [i, i] + [vp] * 5 + [i, i] + [vp] * 8 + [i] * 7 + [vp]
    lib.probe_spmm.argtypes = [i, i] + [vp] * 6 + [i, i] + [vp] * 6 + [i, i, vp]
    lib.probe_gram.argtypes = [i, i] + [vp] * 6 + [i, i] + [vp] * 3 + [vp]
    lib.probe_rotate.argtypes = [i] + [vp] * 7 + [i, i] + [vp] * 3 + [vp]
    return lib


@pytest.fixture(scope="module")
def ratios():
    """Largest |got - ref| / bound per kernel and mode, printed when the module is done (pytest -s shows it)."""
    r = {}
    yield r
    print("\nlargest |got - ref| / rounding bound:")
    for k in sorted(r):
        print("  %-40s %.3g" % (k, r[k]))


def call(lib, name, *args):
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RuntimeError("%s -> %d: %s" % (name, rc, lib.probe_last_error().decode("utf-8", "replace")))


def bits(t):
    import torch

    return t.contiguous().view({torch.float32: torch.int32, torch.float64: torch.int64}[t.dtype])


class DevBatch:
    """A Batch on the device with its SELL copy (built by sell_build_f32) and the blocks and tables of one sweep."""

    def __init__(self, torch, probe, batch, seed):
        self.t, self.h = torch, batch
        dev = torch.device("cuda", torch.cuda.current_device())
        self.dev = dev
        self.stream = torch.cuda.current_stream().cuda_stream
        h = batch
        i32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)
        f64 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
        self.i32, self.f64 = i32, f64
        self.rp, self.cols, self.w = i32(h.rp), i32(h.cols), f64(h.w)
        self.deg, self.dinv, self.mesh_off = f64(h.deg), f64(h.dinv), i32(h.off)
        n_slices = int(sum(-(-int(s) // SELL_ROWS) for s in h.sizes))
        self.n_slices = n_slices
        self.cap = int(probe.probe_sell_entries_cap(h.off.ctypes.data, h.info.ctypes.data, h.m))
        self.mso = torch.full((h.m + 1,), -1, dtype=torch.int32, device=dev)
        self.slice_ptr = torch.full((n_slices + 1,), -1, dtype=torch.int32, device=dev)
        self.entries = torch.full((self.cap, 2), -7, dtype=torch.int32, device=dev)
        self.ddi = torch.full((h.n, 2), float("nan"), dtype=torch.float32, device=dev)
        cnt = torch.empty(n_slices + 1, dtype=torch.int32, device=dev)
        tmp = torch.empty(max(int(probe.probe_scan_tmp_ints(n_slices + 1)), 1), dtype=torch.int32, device=dev)
        call(probe, "probe_sell_build", self.rp.data_ptr(), self.cols.data_ptr(), self.w.data_ptr(), self.deg.data_ptr(),
             self.dinv.data_ptr(), self.mesh_off.data_ptr(), h.off.ctypes.data, h.m, h.n, self.mso.data_ptr(),
             self.slice_ptr.data_ptr(), self.entries.data_ptr(), self.ddi.data_ptr(), cnt.data_ptr(), tmp.data_ptr(),
             self.stream)
        ddi = self.ddi.cpu().numpy().astype(np.float64)
        self.d32, self.di32 = ddi[:, :1], ddi[:, 1:]
        # blocks (full width; a sweep at block size b uses the first b columns) and tables
        rng = np.random.default_rng(seed)
        self.y = rng.standard_normal((h.n, 96))
        self.xp = rng.standard_normal((h.n, 96))
        self.r = rng.standard_normal((h.n, 96)) * 0.1
        self.x = rng.standard_normal((h.n, 96))
        self.z = rng.standard_normal((h.n, 96))
        self.al_d = rng.uniform(0.5, 2.0, (h.m, N_STEPS))
        self.ga_d = rng.uniform(0.2, 1.0, (h.m, N_STEPS))
        self.al_f = rng.uniform(0.5, 2.0, (h.m, N_STEPS, 96)).astype(np.float32)
        self.ga_f = rng.uniform(0.2, 1.0, (h.m, N_STEPS, 96)).astype(np.float32)
        self.center = rng.uniform(0.5, 1.5, h.m)
        self.theta = rng.uniform(0.0, 2.0, (h.m, 96))
        self.wrot = rng.standard_normal((h.m, 96, 96)) / np.sqrt(96.0)
        self._inputs = {}

    def inputs(self, b):
        """Device copies of the first b columns of the blocks and of the tables (made once per block size)."""
        if b not in self._inputs:
            t = self.t
            f32 = lambda a: t.from_numpy(np.ascontiguousarray(a[:, :b], dtype=np.float32)).to(self.dev)
            self._inputs[b] = dict(
                y32=f32(self.y), y64=self.f64(self.y[:, :b]), xp32=f32(self.xp), r32=f32(self.r), x64=self.f64(self.x[:, :b]),
                xp64=self.f64(self.xp[:, :b]), al_d=self.f64(self.al_d), ga_d=self.f64(self.ga_d), center=self.f64(self.center),
                al_f=t.from_numpy(np.ascontiguousarray(self.al_f[:, :, :b])).to(self.dev),
                ga_f=t.from_numpy(np.ascontiguousarray(self.ga_f[:, :, :b])).to(self.dev))
        return self._inputs[b]


# ------------------------------------------------------------------------------------------------ GPU fixtures
@pytest.fixture(scope="module")
def batches(torch, probe):
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    graphs = small_graphs()
    small = Batch(graphs)
    # the same meshes followed by meshes of 250-330 rows: enough CTAs of 256 rows for two waves
    per_mesh = -(-small.max_rows // FS_ROWS)
    n_fill = max(2, -(-2 * sms // per_mesh) - small.m + 2)
    rng = np.random.default_rng(11)
    big = Batch(graphs + [artificial_graph(int(rng.integers(250, 331)), 100 + k) for k in range(n_fill)])
    assert not takes_256_row_form(small, sms), "the small batch must take the one-pass form"
    assert takes_256_row_form(big, sms), "the large batch must take the 256-row form"
    assert small.one_way > 0 and np.any(small.deg == 0) and small.lens.max() >= 300
    assert np.array_equal(big.rp[:small.n + 1], small.rp) and np.array_equal(big.cols[:small.rp[-1]], small.cols)
    s, g = DevBatch(torch, probe, small, 3), DevBatch(torch, probe, big, 3)
    # the small batch's blocks are the first rows of the large batch's
    for name in ("y", "xp", "r", "x", "z"):
        setattr(g, name, np.concatenate([getattr(s, name), getattr(g, name)[small.n:]]))
    for name in ("al_d", "ga_d", "al_f", "ga_f", "center", "theta", "wrot"):
        setattr(g, name, np.concatenate([getattr(s, name), getattr(g, name)[small.m:]]))
    return dict(small=s, big=g)


# ------------------------------------------------------------------------------------------------ SELL layout
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["small", "big"])
def test_sell_layout_matches_a_numpy_build(batches, which):
    """Each slice is as wide as its longest row; entry k of row r of slice s at slice_ptr[s] + 64 k + r; padding
    {first row of the slice, +0.0f}; the entry count within sell_entries_cap; ddi = fp32 (degree, 1/(degree + 1e-8))."""
    db = batches[which]
    h = db.h
    mso, sp = db.mso.cpu().numpy(), db.slice_ptr.cpu().numpy()
    ent = db.entries.cpu().numpy()
    w_bits = h.w.astype(np.float32).view(np.int32)
    exp_mso = np.concatenate([[0], np.cumsum([-(-int(s) // SELL_ROWS) for s in h.sizes])])
    assert np.array_equal(mso, exp_mso)
    exp_sp = [0]
    exp = []
    for m in range(h.m):
        for r0 in range(int(h.off[m]), int(h.off[m + 1]), SELL_ROWS):
            r1 = min(int(h.off[m + 1]), r0 + SELL_ROWS)
            width = int(h.lens[r0:r1].max())
            blk = np.empty((width, SELL_ROWS, 2), dtype=np.int32)
            blk[:, :, 0], blk[:, :, 1] = r0, 0   # padding: first row of the slice, +0.0f
            for rl in range(r1 - r0):
                p0, ln = h.rp[r0 + rl], h.lens[r0 + rl]
                blk[:ln, rl, 0] = h.cols[p0:p0 + ln]
                blk[:ln, rl, 1] = w_bits[p0:p0 + ln]
            exp.append(blk.reshape(-1, 2))
            exp_sp.append(exp_sp[-1] + width * SELL_ROWS)
    assert np.array_equal(sp, np.array(exp_sp))
    assert sp[-1] <= db.cap
    assert np.array_equal(ent[:sp[-1]], np.concatenate(exp))
    ddi = db.ddi.cpu().numpy()
    assert np.array_equal(ddi[:, 0], h.deg.astype(np.float32)) and np.array_equal(ddi[:, 1], h.dinv.astype(np.float32))


# ------------------------------------------------------------------------------------------------ fp32 filter step
def run_filter(torch, probe, db, b, mode, has_prev, policy=3, prefetch=1, pdl=2, min_blocks=8):
    """One k_filter_sell launch; returns (out, y_copy) on the device."""
    t, h, dev, a = torch, db.h, db.dev, db.inputs(b)
    y = a["y64"] if mode == 1 else a["y32"]
    xp, r, center = a["xp32"], a["r32"], a["center"]
    if mode in (2, 4):
        out = a["x64"].clone() if mode == 4 else t.full((h.n, b), float("nan"), dtype=t.float64, device=dev)
    else:
        out = t.full((h.n, b), float("nan"), dtype=t.float32, device=dev)
    y_copy = t.full((h.n, b), float("nan"), dtype=t.float32, device=dev)
    al, ga = (a["al_f"], a["ga_f"]) if mode >= 3 else (a["al_d"], a["ga_d"])
    call(probe, "probe_filter_sell", mode, b, db.entries.data_ptr(), db.slice_ptr.data_ptr(), db.mso.data_ptr(),
         db.ddi.data_ptr(), db.mesh_off.data_ptr(), h.m, h.max_rows, y.data_ptr(), xp.data_ptr(), r.data_ptr(),
         out.data_ptr(), y_copy.data_ptr(), al.data_ptr(), ga.data_ptr(), center.data_ptr(), STEP, N_STEPS, has_prev,
         policy, prefetch, pdl, min_blocks, db.stream)
    return out, y_copy


def filter_ref(db, b, mode, has_prev):
    h = db.h
    rnd = lambda a: a[:, :b].astype(np.float32).astype(np.float64)
    y, xp, r = rnd(db.y), rnd(db.xp), rnd(db.r)
    acc, aacc = block_apply(db, b, True)
    mr = h.mesh_of_row
    cc = db.center.astype(np.float32).astype(np.float64)[mr, None]
    if mode >= 3:
        al = db.al_f[mr, STEP, :b].astype(np.float64)
        ga = db.ga_f[mr, STEP, :b].astype(np.float64)
        v, s = step_ref(acc, aacc, y, db.d32, db.di32, cc, al, ga if has_prev else None, xp if has_prev else None, r)
    else:
        al = db.al_d[mr, STEP].astype(np.float32).astype(np.float64)[:, None]
        ga = db.ga_d[mr, STEP].astype(np.float32).astype(np.float64)[:, None]
        v, s = step_ref(acc, aacc, y, db.d32, db.di32, cc, al, None if mode == 1 else ga, None if mode == 1 else xp)
    if mode == 4:
        v, s = db.x[:, :b] + v, np.abs(db.x[:, :b]) + s
    return v, s


@pytest.mark.gpu
@pytest.mark.parametrize("b", BLOCKS)
def test_filter_sell_step_within_rounding_bound(torch, probe, batches, ratios, b):
    """Every mode of k_filter_sell at block size b on both CTA shapes: within the fp32 rounding bound of the step's
    formula; bit-identical when repeated, across the two CTA shapes, and (256-row form) across every cache policy,
    prefetch and launch form; for b = 16 also across the 8 / 6 / 5 resident-CTA builds of modes 0 and 3."""
    small, big = batches["small"], batches["big"]
    for mode, hp in FILTER_RUNS:
        base = {}
        for which, db in (("small", small), ("big", big)):
            out, y_copy = run_filter(torch, probe, db, b, mode, hp)
            ref, s = filter_ref(db, b, mode, hp)
            got = out.cpu().numpy()
            assert_within(ratios, "k_filter_sell mode %d%s b=%d" % (mode, "" if hp or mode == 1 else " (no z_prev)", b),
                          got, ref, rounding_bound(s, db.h.lens, U32))
            if mode == 1:
                assert np.array_equal(y_copy.cpu().numpy(), db.y[:, :b].astype(np.float32))
            again, _ = run_filter(torch, probe, db, b, mode, hp)
            assert torch.equal(bits(again), bits(out)), (which, mode, "repeat")
            base[which] = out
            variants = []
            if which == "big":
                variants += [dict(policy=p, prefetch=f, pdl=d) for p in range(4) for f in (0, 1) for d in (0, 1, 2)]
            if b == 16 and mode in (0, 3):
                variants += [dict(min_blocks=mb) for mb in (8, 6, 5)]
            for v in variants:
                o, _ = run_filter(torch, probe, db, b, mode, hp, **v)
                assert torch.equal(bits(o), bits(out)), (which, mode, v)
        # a row's arithmetic does not depend on the rows per CTA
        assert torch.equal(bits(base["big"][:small.h.n]), bits(base["small"])), (mode, "one-pass vs 256-row")


# ------------------------------------------------------------------------------------------------ fp64 SpMM
def run_spmm(torch, probe, db, b, mode):
    t, a = torch, db.inputs(b)
    y, xp, al, ga, center = a["y64"], a["xp64"], a["al_d"], a["ga_d"], a["center"]
    out = t.full((db.h.n, b), float("nan"), dtype=t.float64, device=db.dev)
    call(probe, "probe_spmm", mode, b, db.rp.data_ptr(), db.cols.data_ptr(), db.w.data_ptr(), db.deg.data_ptr(),
         db.dinv.data_ptr(), db.mesh_off.data_ptr(), db.h.m, db.h.max_rows, y.data_ptr(), xp.data_ptr(), out.data_ptr(),
         al.data_ptr(), ga.data_ptr(), center.data_ptr(), STEP, N_STEPS, db.stream)
    return out, y


def spmm_ref(db, b, mode):
    h, ld = db.h, np.longdouble
    y = db.y[:, :b].astype(ld)
    acc, aacc = block_apply(db, b, False)
    d, di = h.deg.astype(ld)[:, None], h.dinv.astype(ld)[:, None]
    if mode == 1:
        return d * y - acc, np.abs(d * y) + aacc
    if mode == 2:
        return di * (d * y - acc), np.abs(di) * (np.abs(d * y) + aacc)
    mr = h.mesh_of_row
    return step_ref(acc, aacc, y, d, di, db.center.astype(ld)[mr, None], db.al_d[mr, STEP].astype(ld)[:, None],
                    db.ga_d[mr, STEP].astype(ld)[:, None], db.xp[:, :b].astype(ld))


@pytest.mark.gpu
@pytest.mark.parametrize("b", BLOCKS)
def test_spmm_f64_within_rounding_bound(torch, probe, batches, ratios, b):
    """k_spmm modes 0..2 at block size b on both CTA shapes: within the fp64 rounding bound; bit-identical when repeated
    and across the two CTA shapes; mode 2 bit-identical with focusr_laplacian_apply of the product library."""
    from pyfocusr_b200 import _lib

    small, big = batches["small"], batches["big"]
    for mode in (0, 1, 2):
        base = {}
        for which, db in (("small", small), ("big", big)):
            out, y = run_spmm(torch, probe, db, b, mode)
            ref, s = spmm_ref(db, b, mode)
            assert_within(ratios, "k_spmm mode %d b=%d" % (mode, b), out.cpu().numpy(), ref, rounding_bound(s, db.h.lens, U64))
            again, _ = run_spmm(torch, probe, db, b, mode)
            assert torch.equal(bits(again), bits(out)), (which, mode, "repeat")
            if mode == 2:
                lap = torch.empty_like(y)
                _lib.call("focusr_laplacian_apply", db.rp.data_ptr(), db.cols.data_ptr(), db.w.data_ptr(), db.deg.data_ptr(),
                          db.dinv.data_ptr(), db.mesh_off.data_ptr(), db.h.m, db.h.max_rows, y.data_ptr(), lap.data_ptr(),
                          b, _lib.stream_ptr())
                assert torch.equal(bits(lap), bits(out)), (which, "focusr_laplacian_apply")
            base[which] = out
        assert torch.equal(bits(base["big"][:small.h.n]), bits(base["small"])), (mode, "one-pass vs 256-row")


# ------------------------------------------------------------------------------------------------ Gram and rotation
@pytest.mark.gpu
@pytest.mark.parametrize("b", BLOCKS)
def test_gram_and_rotation_within_rounding_bound(torch, probe, batches, ratios, b):
    """Per mesh, G = X^T g X and H = X^T h Z (k_gram for b < 64, k_gram_wide for b >= 64, then k_reduce_gh) with
    g = degree + 1e-8, h = 1 (sym = 1) or g = 1, h = 1/(degree + 1e-8) (sym = 0); then X W, the fp32 residual block
    dinv Z W - X W theta and the residual norms ||dinv Z W - X W theta|| / ||X W|| per column (k_rotate, k_residual).
    Within the fp64 rounding bounds; bit-identical when repeated.  Meshes of 1024 k + {0, 1, 1023} rows and smaller
    than one chunk of 1024."""
    db = batches["small"]
    h, t, ld = db.h, torch, np.longdouble
    chunks_max = int(max(-(-int(s) // GRAM_ROWS) for s in h.sizes))
    x, z = db.inputs(b)["x64"], db.f64(db.z[:, :b])
    partial = t.empty(h.m * chunks_max * 2 * b * b, dtype=t.float64, device=db.dev)
    xl, zl = db.x[:, :b].astype(ld), db.z[:, :b].astype(ld)
    for sym in (1, 0):
        outs = []
        for _ in range(2):
            g = t.full((h.m, b, b), float("nan"), dtype=t.float64, device=db.dev)
            hh = t.full((h.m, b, b), float("nan"), dtype=t.float64, device=db.dev)
            call(probe, "probe_gram", b, sym, x.data_ptr(), z.data_ptr(), db.deg.data_ptr(), db.dinv.data_ptr(),
                 db.mesh_off.data_ptr(), h.off.ctypes.data, h.m, chunks_max, partial.data_ptr(), g.data_ptr(),
                 hh.data_ptr(), db.stream)
            outs.append((g, hh))
        assert torch.equal(bits(outs[0][0]), bits(outs[1][0])) and torch.equal(bits(outs[0][1]), bits(outs[1][1]))
        g, hh = outs[0][0].cpu().numpy(), outs[0][1].cpu().numpy()
        gw = (h.deg + 1e-8) if sym else np.ones(h.n)
        hw = np.ones(h.n) if sym else h.dinv
        name = "gram%s sym=%d" % ("_wide" if b >= 64 else "", sym)
        for m in range(h.m):
            o0, o1 = h.off[m], h.off[m + 1]
            xm, zm = xl[o0:o1], zl[o0:o1]
            gm, hm = gw[o0:o1].astype(ld)[:, None], hw[o0:o1].astype(ld)[:, None]
            rg, sg = xm.T @ (gm * xm), np.abs(xm).T @ (np.abs(gm * xm))
            rh, sh = xm.T @ (hm * zm), np.abs(xm).T @ (np.abs(hm * zm))
            n_r = np.full(b, int(o1 - o0))
            assert_within(ratios, "%s G b=%d" % (name, b), g[m], rg, rounding_bound(sg, n_r, U64))
            assert_within(ratios, "%s H b=%d" % (name, b), hh[m], rh, rounding_bound(sh, n_r, U64))

    w = db.f64(db.wrot[:, :b, :b])
    theta = db.f64(db.theta[:, :b])
    partial_res = t.empty(h.m * chunks_max * 2 * b, dtype=t.float64, device=db.dev)
    outs = []
    for _ in range(2):
        xr = x.clone()
        res = t.full((h.m, b), float("nan"), dtype=t.float64, device=db.dev)
        r_out = t.full((h.n, b), float("nan"), dtype=t.float32, device=db.dev)
        call(probe, "probe_rotate", b, xr.data_ptr(), z.data_ptr(), w.data_ptr(), theta.data_ptr(), db.dinv.data_ptr(),
             db.mesh_off.data_ptr(), h.off.ctypes.data, h.m, chunks_max, partial_res.data_ptr(), res.data_ptr(),
             r_out.data_ptr(), db.stream)
        outs.append((xr, res, r_out))
    for a, c in zip(outs[0], outs[1]):
        assert torch.equal(bits(a), bits(c))
    xr, res, r_out = (o.cpu().numpy() for o in outs[0])
    for m in range(h.m):
        o0, o1 = h.off[m], h.off[m + 1]
        wm = db.wrot[m, :b, :b].astype(ld)
        xm, zm = xl[o0:o1], zl[o0:o1]
        xw, sxw = xm @ wm, np.abs(xm) @ np.abs(wm)
        zw, szw = zm @ wm, np.abs(zm) @ np.abs(wm)
        di, th = h.dinv[o0:o1].astype(ld)[:, None], db.theta[m, :b].astype(ld)[None, :]
        e, se = di * zw - th * xw, np.abs(di) * szw + np.abs(th) * sxw
        n_b = np.full(o1 - o0, b)
        assert_within(ratios, "rotate X W b=%d" % b, xr[o0:o1], xw, rounding_bound(sxw, n_b, U64))
        assert_within(ratios, "rotate fp32 residual block b=%d" % b, r_out[o0:o1], e, rounding_bound(se, n_b, U32))
        # residual norms sqrt(num / den): num and den are sums of n squares of values that are each within (b + 8) u S
        # of the reference, so |num - ref| <= (n + 2 (b + 8) + 1) u sum S^2; the quotient and the root add 2 u
        num, den = (e * e).sum(axis=0), (xw * xw).sum(axis=0)
        ref = np.sqrt(num / den)
        k = int(o1 - o0) + 2 * b + 24
        rel = 0.5 * k * U64 * ((se * se).sum(axis=0) / num + (sxw * sxw).sum(axis=0) / den) + 2 * U64
        assert_within(ratios, "k_residual b=%d" % b, res[m], ref, ref * rel)
