"""Device-resident batch graph: the host-side owner of everything the CUDA library works on.

A :class:`DeviceGraph` holds one block-diagonal graph made of ``n_meshes`` meshes (their
vertices concatenated, triangle ids made global) and exposes the C-ABI operations on it as
methods.  ``Graph`` (one mesh) and ``SpectralBatch`` (many pairs) are thin users of this class.
All arrays are ``torch`` CUDA tensors; nothing here computes on the host.
"""
from __future__ import annotations

import numpy as np

from . import _lib

EIG_STATUS = {0: "ok", 1: "not converged", 2: "block too small", 3: "numerical breakdown", 4: "ldv too small"}


def _torch():
    return _lib.require_cuda()


def _dev_i32(a):
    torch = _torch()
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).cuda(non_blocking=True)


class DeviceGraph:
    def __init__(self, points_list, tris_list, edge_points_list=None):
        """``edge_points_list`` (optional): per mesh [n][3+f] coordinates the edge weights are measured
        in (xyz followed by range-scaled node features, reference graph.py:166-175); default = xyz."""
        torch = _torch()
        self.n_meshes = len(points_list)
        sizes = [int(np.asarray(p).shape[0]) for p in points_list]
        self.mesh_off_host = np.zeros(self.n_meshes + 1, dtype=np.int32)
        self.mesh_off_host[1:] = np.cumsum(sizes)
        self.n_points = int(self.mesh_off_host[-1])
        self.max_mesh_points = int(max(sizes))
        pts = np.ascontiguousarray(np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1, 3) for p in points_list]))
        tris = np.concatenate(
            [np.asarray(t, dtype=np.int64).reshape(-1, 3) + int(o) for t, o in zip(tris_list, self.mesh_off_host[:-1])]
        ).astype(np.int32)
        edge_pts = None
        if edge_points_list is not None:
            edge_pts = torch.from_numpy(np.ascontiguousarray(np.concatenate(
                [np.asarray(p, dtype=np.float64).reshape(len(p), -1) for p in edge_points_list])))
        self._init_from_host(torch.from_numpy(pts), torch.from_numpy(np.ascontiguousarray(tris)), edge_pts)

    @classmethod
    def from_device(cls, points, tris, mesh_off_host, edge_points=None):
        """Build from tensors that are already resident in HBM (``tris`` hold global ids).  ``edge_points`` (optional,
        [n_points][3+f]): the coordinates the edge weights are measured in (``node_features``); ``points`` stays xyz."""
        self = cls.__new__(cls)
        self.mesh_off_host = np.ascontiguousarray(mesh_off_host, dtype=np.int32)
        self.n_meshes = self.mesh_off_host.size - 1
        self.n_points = int(self.mesh_off_host[-1])
        self.max_mesh_points = int(np.max(np.diff(self.mesh_off_host)))
        self._init_from_host(points, tris, edge_points)
        return self

    def _init_from_host(self, points, tris, edge_points=None):
        torch = _torch()
        dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        self.points = points.to(dev, non_blocking=True).contiguous()
        self.tris = tris.to(dev, non_blocking=True).contiguous()
        self.n_tris = int(self.tris.shape[0])
        self.mesh_off = torch.from_numpy(self.mesh_off_host).to(dev, non_blocking=True)
        n, f, m = self.n_points, self.n_tris, self.n_meshes
        self.row_ptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
        self.cols = torch.empty(max(3 * f, 1), dtype=torch.int32, device=dev)
        self.weights = torch.empty(max(3 * f, 1), dtype=torch.float64, device=dev)
        self.degree = torch.empty(n, dtype=torch.float64, device=dev)
        self.degree_inv = torch.empty(n, dtype=torch.float64, device=dev)
        mesh_info = torch.empty((m, _lib.MESH_INFO_INTS), dtype=torch.int32, device=dev)
        lib = _lib.load()
        ws_bytes = int(lib.focusr_laplacian_workspace_bytes(n, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        ep = self.points if edge_points is None else edge_points.to(dev, non_blocking=True).contiguous()
        _lib.call("focusr_laplacian_build", _lib.ptr(ep), int(ep.shape[1]), _lib.ptr(self.tris), n, f, _lib.ptr(self.mesh_off), m,
                  _lib.ptr(self.row_ptr), _lib.ptr(self.cols), _lib.ptr(self.weights), _lib.ptr(self.degree),
                  _lib.ptr(self.degree_inv), _lib.ptr(mesh_info), _lib.ptr(ws), ws_bytes, _lib.stream_ptr())
        # {nnz, one-way entries, zero-degree rows, non-finite weights, longest row, 0, 0, 0} per mesh
        self.mesh_info_host = np.ascontiguousarray(mesh_info.cpu().numpy())
        self.nnz = int(self.mesh_info_host[:, 0].sum())
        self._lap = None

    # --- K1 -----------------------------------------------------------------------------------
    def adjacency_host(self):
        """(indptr, indices, data) of A on the host (canonical CSR)."""
        nnz = self.nnz
        return (self.row_ptr.cpu().numpy(), self.cols[:nnz].cpu().numpy(), self.weights[:nnz].cpu().numpy())

    def laplacian_device(self):
        if self._lap is None:
            torch = _torch()
            n = self.n_points
            l_rp = torch.empty(n + 1, dtype=torch.int32, device=self.device)
            l_cols = torch.empty(self.nnz + n, dtype=torch.int32, device=self.device)
            l_vals = torch.empty(self.nnz + n, dtype=torch.float64, device=self.device)
            ws_bytes = 8 * (n + 1) + 8 * ((n + 1) // 2048 + 8) + 4096
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
            _lib.call("focusr_laplacian_csr", _lib.ptr(self.row_ptr), _lib.ptr(self.cols), _lib.ptr(self.weights),
                      _lib.ptr(self.degree), _lib.ptr(self.degree_inv), n, _lib.ptr(l_rp), _lib.ptr(l_cols),
                      _lib.ptr(l_vals), _lib.ptr(ws), ws_bytes, _lib.stream_ptr())
            self._lap = (l_rp, l_cols, l_vals)
        return self._lap

    def laplacian_host(self):
        l_rp, l_cols, l_vals = self.laplacian_device()
        rp = l_rp.cpu().numpy()
        nnz = int(rp[-1])
        return rp, l_cols[:nnz].cpu().numpy(), l_vals[:nnz].cpu().numpy()

    # --- K2 -----------------------------------------------------------------------------------
    def eigs_smallest(self, k, n_k_needed, k_buffer=1, min_eig_val=1e-10, tol=1e-10, max_outer=60,
                      block_size=0, ldv=None, spectrum_upper_bound=0.0, options=None):
        """Batched ``recursive_eig``.  Returns ``(vals [M][ldv], vecs [N][ldv], info)`` on the
        device; ``info`` is a dict of host arrays (``n_found``, ``k_final``, ...).  ``options``: an
        ``_lib.EigsOptions`` (or a dict of its fields); default = the library's defaults."""
        import ctypes as C
        torch = _torch()
        lib = _lib.load()
        n, m = self.n_points, self.n_meshes
        max_oneway = int(self.mesh_info_host[:, 1].max())
        max_zero = int(self.mesh_info_host[:, 2].max())
        b = int(block_size) if block_size else int(lib.focusr_eigs_block_size(k, n_k_needed, k_buffer, max_oneway, max_zero))
        res_i = np.zeros((m, 8), dtype=np.int32)
        res_d = np.zeros((m, 2), dtype=np.float64)
        restarts = 0
        if isinstance(options, dict):
            options = _lib.EigsOptions(**options)
        opt_ptr = C.byref(options) if options is not None else None
        sell_cap = int(lib.focusr_sell_entries_cap(_lib.ptr(self.mesh_off_host), _lib.ptr(self.mesh_info_host), m))
        # columns of the output block: one retry of the reference's recursion by default; the
        # solver reports status 4 if a mesh needs more and the call is repeated with ldv = block
        ldv_use = int(ldv) if ldv else int(k + k_buffer + n_k_needed)
        while True:
            vals = torch.zeros((m, ldv_use), dtype=torch.float64, device=self.device)
            vecs = torch.zeros((n, ldv_use), dtype=torch.float64, device=self.device)
            ws_bytes = int(lib.focusr_eigs_workspace_bytes_mixed(n, sell_cap, m, self.max_mesh_points, b))
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
            try:
                _lib.call("focusr_eigs_smallest", _lib.ptr(self.row_ptr), _lib.ptr(self.cols), _lib.ptr(self.weights),
                          _lib.ptr(self.degree), _lib.ptr(self.degree_inv), _lib.ptr(self.points), n,
                          _lib.ptr(self.mesh_off_host), m, _lib.ptr(self.mesh_info_host), int(k), int(n_k_needed),
                          int(k_buffer), float(min_eig_val), float(tol), int(max_outer), b, float(spectrum_upper_bound), _lib.ptr(vals),
                          _lib.ptr(vecs), ldv_use, _lib.ptr(res_i), _lib.ptr(res_d), _lib.ptr(ws), ws_bytes,
                          opt_ptr, _lib.stream_ptr())
                break
            except _lib.FocusrB200Error as e:
                status = int(res_i[:, 0].max()) if e.code < 100 else -1
                # a multiplet cut by the block / a large null space: enlarge the block and retry
                if status == 2 and b < 96 and restarts < 6:
                    b = min(96, b + 16)
                    restarts += 1
                    continue
                if status == 4 and ldv_use < b:
                    ldv_use = b
                    restarts += 1
                    continue
                if e.code < 100:   # a solver status, not a CUDA / argument error: say which meshes
                    e.eigs_info = dict(status=res_i[:, 0].copy(), n_found=res_i[:, 1].copy(), max_residual=res_d[:, 0].copy())
                raise
            finally:
                del ws
        info = dict(status=res_i[:, 0].copy(), n_found=res_i[:, 1].copy(), k_final=res_i[:, 2].copy(),
                    outer_iterations=res_i[:, 3].copy(), filter_degree=res_i[:, 4].copy(), block_size=b,
                    symmetric=res_i[:, 6].copy(), restarts=restarts, max_residual=res_d[:, 0].copy(),
                    spectrum_bound=res_d[:, 1].copy(), fp32_filter_degree=res_i[:, 7].copy())
        return vals, vecs, info

    def laplacian_apply(self, x):
        torch = _torch()
        y = torch.empty_like(x)
        _lib.call("focusr_laplacian_apply", _lib.ptr(self.row_ptr), _lib.ptr(self.cols), _lib.ptr(self.weights),
                  _lib.ptr(self.degree), _lib.ptr(self.degree_inv), _lib.ptr(self.mesh_off), self.n_meshes,
                  self.max_mesh_points, _lib.ptr(x), _lib.ptr(y), int(x.shape[1]), _lib.stream_ptr())
        return y

    # --- B2 / C5 / D1 ---------------------------------------------------------------------------
    def normalize_columns(self, vecs, n_cols):
        n_cols_dev = _dev_i32(n_cols)
        _lib.call("focusr_normalize_columns", _lib.ptr(vecs), self.n_points, int(vecs.shape[1]), _lib.ptr(self.mesh_off),
                  self.n_meshes, _lib.ptr(n_cols_dev), _lib.stream_ptr())

    def flip_permute(self, vecs, dst, src, sign):
        """dst/src/sign: int arrays [n_meshes][n_moves], host (numpy) or device (torch int32, e.g. from
        ``eigsort_decide``)."""
        torch = _torch()
        if isinstance(dst, torch.Tensor):
            d, s, g = dst, src, sign
            n_moves = int(d.shape[1])
        else:
            dst = np.ascontiguousarray(dst, dtype=np.int32).reshape(self.n_meshes, -1)
            n_moves = dst.shape[1]
            d, s, g = _dev_i32(dst), _dev_i32(np.asarray(src).reshape(self.n_meshes, -1)), _dev_i32(np.asarray(sign).reshape(self.n_meshes, -1))
        _lib.call("focusr_flip_permute_columns", _lib.ptr(vecs), self.n_points, int(vecs.shape[1]), _lib.ptr(self.mesh_off),
                  self.n_meshes, self.max_mesh_points, _lib.ptr(d), _lib.ptr(s), _lib.ptr(g), n_moves, _lib.stream_ptr())

    def spectral_coords(self, vecs, weights, ns):
        """weights: [n_meshes][ns], host (numpy) or device (torch float64) -> device [n_points][ns]."""
        torch = _torch()
        if isinstance(weights, torch.Tensor):
            w = weights
        else:
            w = torch.from_numpy(np.ascontiguousarray(weights, dtype=np.float64).reshape(self.n_meshes, ns)).to(self.device)
        out = torch.empty((self.n_points, ns), dtype=torch.float64, device=self.device)
        _lib.call("focusr_spectral_coords", _lib.ptr(vecs), self.n_points, int(vecs.shape[1]), _lib.ptr(self.mesh_off),
                  self.n_meshes, self.max_mesh_points, _lib.ptr(w), int(ns), _lib.ptr(out), _lib.stream_ptr())
        return out

    # --- K5 -----------------------------------------------------------------------------------
    def mean_filter(self, values, iterations, row_begin=0, row_end=None):
        """values: device [n_points][c]; rows [row_begin, row_end) must be whole meshes (rows outside are ignored).
        Returns a new tensor.  One launch per pass, chained by programmatic dependent launch."""
        torch = _torch()
        lib = _lib.load()
        row_end = self.n_points if row_end is None else row_end
        c = int(values.shape[1])
        out = torch.empty_like(values)
        off = self.mesh_off_host
        mb, me = int(np.searchsorted(off, row_begin)), int(np.searchsorted(off, row_end))
        if not (mb < me <= self.n_meshes and off[mb] == row_begin and off[me] == row_end):
            raise ValueError("mean_filter: the row range must cover whole meshes")
        ws_bytes = int(lib.focusr_mean_filter_workspace_bytes(int(row_end - row_begin), c))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        _lib.call("focusr_mean_filter", _lib.ptr(self.row_ptr), _lib.ptr(self.cols), _lib.ptr(self.weights),
                  _lib.ptr(self.degree), int(row_begin), int(row_end), _lib.ptr(values), _lib.ptr(out),
                  c, int(iterations), _lib.ptr(ws), ws_bytes, _lib.stream_ptr())
        return out

    def mean_filter_mapped(self, values, iterations, seg_mesh):
        """``focusr_mean_filter_mapped``: segment s of ``values`` (device [rows][c]; the segments' rows one after the
        other, each as many as its mesh has) is smoothed on graph mesh ``seg_mesh[s]`` (host ints).  A mesh may serve
        several segments or none.  Returns a new tensor, equal to :meth:`mean_filter` on a batch holding a copy of mesh
        ``seg_mesh[s]`` for every segment."""
        torch = _torch()
        lib = _lib.load()
        seg_host = np.ascontiguousarray(seg_mesh, dtype=np.int32).reshape(-1)
        if seg_host.size and 0 <= seg_host.min() and seg_host.max() < self.n_meshes:  # otherwise the library says which
            n_rows = int(np.diff(self.mesh_off_host.astype(np.int64))[seg_host].sum())
            if int(values.shape[0]) != n_rows:
                raise ValueError("mean_filter_mapped: the segments hold %d rows, values has %d" % (n_rows, values.shape[0]))
        c = int(values.shape[1])
        out = torch.empty_like(values)
        ws_bytes = int(lib.focusr_mean_filter_mapped_workspace_bytes(int(values.shape[0]), c, int(seg_host.size)))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        seg_dev = torch.from_numpy(seg_host).to(self.device, non_blocking=True)
        _lib.call("focusr_mean_filter_mapped", _lib.ptr(self.row_ptr), _lib.ptr(self.cols), _lib.ptr(self.weights),
                  _lib.ptr(self.degree), _lib.ptr(self.mesh_off), _lib.ptr(self.mesh_off_host), self.n_meshes,
                  _lib.ptr(seg_dev), _lib.ptr(seg_host), int(seg_host.size), _lib.ptr(values), _lib.ptr(out), c,
                  int(iterations), _lib.ptr(ws), ws_bytes, _lib.stream_ptr())
        return out


# ---------------------------------------------------------------------------------------------
# free functions on device tensors
# ---------------------------------------------------------------------------------------------
def knn(refs, queries, k=1, ref_off=None, query_off=None, max_queries=None, max_refs=None, want_dist=True,
        brute_force=False):
    """Exact k-NN of ``queries`` in ``refs`` (device [n][dim] float64, row-major, contiguous).
    Optional segment offset tensors (device int32) make it batched; indices are segment-local.
    ``brute_force=True`` skips the (bit-identical) bounding-box pruning."""
    torch = _torch()
    lib = _lib.load()
    dev = refs.device
    nq, dim, nr = int(queries.shape[0]), int(queries.shape[1]), int(refs.shape[0])
    if ref_off is None:
        ref_off = torch.tensor([0, nr], dtype=torch.int32, device=dev)
        query_off = torch.tensor([0, nq], dtype=torch.int32, device=dev)
        max_queries, max_refs = nq, nr
    if max_refs is None:
        max_refs = int(torch.diff(ref_off).max().item())
    n_seg = int(ref_off.shape[0]) - 1
    idx = torch.empty((nq, k), dtype=torch.int64, device=dev)
    dist = torch.empty((nq, k), dtype=torch.float64, device=dev) if want_dist else None
    ws, ws_bytes = None, 0
    if not brute_force:
        ws_bytes = int(lib.focusr_knn_workspace_bytes(nr, nq, n_seg, dim))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    _lib.call("focusr_knn", _lib.ptr(refs), int(refs.stride(0)), _lib.ptr(ref_off), nr, int(max_refs),
              _lib.ptr(queries), int(queries.stride(0)), _lib.ptr(query_off), nq, int(max_queries), n_seg, dim,
              int(k), _lib.ptr(idx), _lib.ptr(dist), _lib.ptr(ws), ws_bytes, _lib.stream_ptr())
    return idx, dist


def knn_mapped(refs, queries, ref_off, query_off, ref_seg, k=1, max_queries=None, max_refs=None, want_dist=True,
               brute_force=False):
    """Exact k-NN against shared reference segments (``focusr_knn_mapped``): query segment s (``query_off``, device
    int32) searches reference segment ``ref_seg[s]`` (``ref_off``, device int32; ``ref_seg`` host ints).  Indices are
    local to the reference segment; the result equals :func:`knn` on a copy of reference segment ``ref_seg[s]`` for
    every query segment.  ``max_refs`` must bound every reference segment."""
    torch = _torch()
    lib = _lib.load()
    dev = refs.device
    nq, dim, nr = int(queries.shape[0]), int(queries.shape[1]), int(refs.shape[0])
    seg_host = np.ascontiguousarray(ref_seg, dtype=np.int32).reshape(-1)
    n_ref_seg, n_q_seg = int(ref_off.shape[0]) - 1, int(query_off.shape[0]) - 1
    if seg_host.size != n_q_seg:
        raise ValueError("knn_mapped: ref_seg needs one entry per query segment (%d), got %d" % (n_q_seg, seg_host.size))
    if max_refs is None:
        max_refs = int(torch.diff(ref_off).max().item())
    if max_queries is None:
        max_queries = int(torch.diff(query_off).max().item())
    seg_dev = torch.from_numpy(seg_host).to(dev, non_blocking=True)
    idx = torch.empty((nq, k), dtype=torch.int64, device=dev)
    dist = torch.empty((nq, k), dtype=torch.float64, device=dev) if want_dist else None
    ws, ws_bytes = None, 0
    if not brute_force:
        ws_bytes = int(lib.focusr_knn_mapped_workspace_bytes(nr, nq, n_ref_seg, dim))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    _lib.call("focusr_knn_mapped", _lib.ptr(refs), int(refs.stride(0)), _lib.ptr(ref_off), nr, n_ref_seg, int(max_refs),
              _lib.ptr(queries), int(queries.stride(0)), _lib.ptr(query_off), nq, int(max_queries), n_q_seg,
              _lib.ptr(seg_dev), _lib.ptr(seg_host), dim, int(k), _lib.ptr(idx), _lib.ptr(dist), _lib.ptr(ws), ws_bytes,
              _lib.stream_ptr())
    return idx, dist


def cdist(a, b):
    """scipy.spatial.distance.cdist(a, b) (euclidean) on the device: [n_a][n_b] float64."""
    torch = _torch()
    a = torch.as_tensor(a, dtype=torch.float64, device="cuda").contiguous()
    b = torch.as_tensor(b, dtype=torch.float64, device="cuda").contiguous()
    out = torch.empty((a.shape[0], b.shape[0]), dtype=torch.float64, device=a.device)
    _lib.call("focusr_cdist", _lib.ptr(a), int(a.shape[0]), _lib.ptr(b), int(b.shape[0]), int(a.shape[1]),
              _lib.ptr(out), _lib.stream_ptr())
    return out


def linear_sum_assignment(cost):
    """scipy.optimize.linear_sum_assignment(cost) for a device matrix: (row_ind, col_ind) as numpy int64 arrays, the
    assignment scipy itself returns (same algorithm, same tie rules; ``focusr_lsap``).  Raises ValueError for a matrix
    without a finite assignment, as scipy does."""
    import ctypes as C

    torch = _torch()
    cost = torch.as_tensor(cost, dtype=torch.float64, device="cuda")
    if cost.ndim != 2:
        raise ValueError("expected a matrix (2-D array), got a %d array" % cost.ndim)
    nr, nc = int(cost.shape[0]), int(cost.shape[1])
    if nr == 0 or nc == 0:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    transposed = nr > nc
    m = (cost.t() if transposed else cost).contiguous()
    rows, cols = int(m.shape[0]), int(m.shape[1])
    col4row = torch.empty(rows, dtype=torch.int32, device=m.device)
    ws_bytes = int(_lib.load().focusr_lsap_workspace_bytes(rows))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=m.device)
    status = C.c_int(0)
    _lib.call("focusr_lsap", _lib.ptr(m), rows, cols, _lib.ptr(col4row), C.addressof(status), _lib.ptr(ws), ws_bytes,
              _lib.stream_ptr())
    if status.value != 0:
        raise ValueError("cost matrix is infeasible")
    a = col4row.cpu().numpy().astype(np.int64)
    if not transposed:
        return np.arange(rows, dtype=np.int64), a
    order = np.argsort(a, kind="stable")   # scipy: rows of the original matrix in ascending order
    return a[order], order.astype(np.int64)


def gather_rows(values, idx, idx_base=None):
    torch = _torch()
    n, c = int(idx.shape[0]), int(values.shape[1])
    out = torch.empty((n, c), dtype=torch.float64, device=values.device)
    _lib.call("focusr_gather_rows", _lib.ptr(values), _lib.ptr(idx), _lib.ptr(idx_base), n, c, _lib.ptr(out),
              _lib.stream_ptr())
    return out


def weighted_positions(idx3, dist3, target_points, point_base=None):
    torch = _torch()
    n = int(idx3.shape[0])
    out = torch.empty((n, 3), dtype=torch.float64, device=target_points.device)
    _lib.call("focusr_weighted_positions", _lib.ptr(idx3), _lib.ptr(dist3), _lib.ptr(target_points),
              _lib.ptr(point_base), n, _lib.ptr(out), _lib.stream_ptr())
    return out


def icp(target_points, target_tris, source_points, max_iterations=100, max_landmarks=1000, similarity=False,
        start_by_matching_centroids=True):
    """vtkIterativeClosestPointTransform on the device (vtk_functions.py:12-37).  Returns ``(matrix, moved)``:
    the accumulated 4x4 matrix (host numpy, acting on column vectors) and the transformed source points
    (device tensor)."""
    torch = _torch()
    lib = _lib.load()

    def dev(a, dt):
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
        return t.to(device="cuda", dtype=dt).contiguous()

    tp, sp, tt = dev(target_points, torch.float64), dev(source_points, torch.float64), dev(target_tris, torch.int32)
    ns = int(sp.shape[0])
    mat = torch.empty(16, dtype=torch.float64, device=sp.device)
    moved = torch.empty_like(sp)
    nbytes = int(lib.focusr_icp_workspace_bytes(ns, int(tt.shape[0])))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=sp.device)
    _lib.call("focusr_icp", _lib.ptr(tp), int(tp.shape[0]), _lib.ptr(tt), int(tt.shape[0]), _lib.ptr(sp), ns,
              int(max_landmarks), int(max_iterations), int(bool(similarity)), int(bool(start_by_matching_centroids)),
              _lib.ptr(mat), _lib.ptr(moved), _lib.ptr(ws), nbytes, _lib.stream_ptr())
    return mat.cpu().numpy().reshape(4, 4), moved


def icp_landmarks(n_points, max_landmarks):
    """The landmark rule of ``focusr_icp`` / ``focusr_icp_batch`` (vtkIterativeClosestPointTransform::InternalUpdate):
    every ``step``-th point of a moving mesh of ``n_points`` is a landmark.  Returns ``(step, count)``."""
    n, ml = int(n_points), int(max_landmarks)
    step = n // ml if n > ml else 1
    return step, n // step


def icp_batch_device(points, tris, mesh_off_host, tri_off_host, fixed_mesh, moving_mesh, max_iterations=100,
                     max_landmarks=1000, similarity=False, start_by_matching_centroids=True):
    """``focusr_icp_batch`` on device tensors; returns ``(matrices (P, 4, 4) float64, moved (N, 3) float64)``, both on
    the device, without synchronising.  ``points`` is not modified."""
    torch = _torch()
    lib = _lib.load()
    dev = points.device
    off = np.ascontiguousarray(mesh_off_host, dtype=np.int32)
    toff = np.ascontiguousarray(tri_off_host, dtype=np.int32)
    fm = np.ascontiguousarray(fixed_mesh, dtype=np.int32).reshape(-1)
    mm = np.ascontiguousarray(moving_mesh, dtype=np.int32).reshape(-1)
    m, P, n = off.size - 1, int(fm.size), int(points.shape[0])
    if toff.size != off.size or mm.size != P:
        raise ValueError("icp_batch: tri_off_host needs n_meshes + 1 entries and every pair a fixed and a moving mesh")
    nbytes = int(lib.focusr_icp_batch_workspace_bytes(_lib.ptr(off), _lib.ptr(toff), m, _lib.ptr(fm), _lib.ptr(mm), P,
                                                      int(max_landmarks)))
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
    off_d, toff_d, fm_d, mm_d = (torch.from_numpy(a).to(dev, non_blocking=True) for a in (off, toff, fm, mm))
    mats = torch.empty((P, 4, 4), dtype=torch.float64, device=dev)
    moved = torch.empty_like(points)
    _lib.call("focusr_icp_batch", _lib.ptr(points), n, _lib.ptr(tris), _lib.ptr(off_d), _lib.ptr(off), _lib.ptr(toff_d),
              _lib.ptr(toff), m, _lib.ptr(fm_d), _lib.ptr(mm_d), _lib.ptr(fm), _lib.ptr(mm), P, int(max_landmarks),
              int(max_iterations), int(bool(similarity)), int(bool(start_by_matching_centroids)), _lib.ptr(mats),
              _lib.ptr(moved), _lib.ptr(ws), nbytes, _lib.stream_ptr())
    return mats, moved


def icp_batch(points, tris, mesh_off_host, tri_off_host, fixed_mesh, moving_mesh, max_iterations=100,
              max_landmarks=1000, similarity=False, start_by_matching_centroids=True):
    """vtkIterativeClosestPointTransform for many pairs at once (``focusr_icp_batch``): pair p moves mesh
    ``moving_mesh[p]`` onto the surface of mesh ``fixed_mesh[p]`` of the batch (``points`` (N, 3) float64, ``tris``
    (F, 3) int32 with global vertex ids grouped by mesh, host or device; ``mesh_off_host`` / ``tri_off_host`` the
    per-mesh row and triangle ranges).  Each pair's result is that of :func:`icp` on the pair alone.  Returns
    ``(matrices (P, 4, 4) host numpy, moved points (N, 3) device tensor)``: the rows of meshes that do not move are
    copied unchanged."""
    torch = _torch()

    def dev(a, dt):
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
        return t.to(device="cuda", dtype=dt).contiguous()

    mats, moved = icp_batch_device(dev(points, torch.float64), dev(tris, torch.int32), mesh_off_host, tri_off_host,
                                   fixed_mesh, moving_mesh, max_iterations, max_landmarks, similarity,
                                   start_by_matching_centroids)
    return mats.cpu().numpy(), moved


def procrustes_fit(configs, reference, similarity, want_aligned=True):
    """``focusr_procrustes_fit``: every configuration of ``configs`` (P, N, 3) fitted onto ``reference`` (N, 3), both
    contiguous float64 device tensors.  Returns ``(matrices (P, 4, 4), aligned (P, N, 3) or None)`` on the device."""
    torch = _torch()
    P, N = int(configs.shape[0]), int(configs.shape[1])
    mats = torch.empty((P, 4, 4), dtype=torch.float64, device=configs.device)
    aligned = torch.empty_like(configs) if want_aligned else None
    _lib.call("focusr_procrustes_fit", _lib.ptr(configs), P, N, _lib.ptr(reference), int(bool(similarity)), _lib.ptr(mats),
              _lib.ptr(aligned), _lib.stream_ptr())
    return mats, aligned


def procrustes_mean(aligned, reference, similarity, prev_mean, mean_out, change_out, ws=None):
    """``focusr_procrustes_mean``: the mean of ``aligned`` (P, N, 3) fitted onto ``reference`` into ``mean_out`` (N, 3),
    its RMS change against ``prev_mean`` into ``change_out`` (a one-element device tensor).  ``ws``: a workspace of at
    least ``focusr_procrustes_mean_workspace_bytes(N)`` bytes (allocated when None).  Returns the workspace."""
    torch = _torch()
    P, N = int(aligned.shape[0]), int(aligned.shape[1])
    nbytes = int(_lib.load().focusr_procrustes_mean_workspace_bytes(N))
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(nbytes, dtype=torch.uint8, device=aligned.device)
    _lib.call("focusr_procrustes_mean", _lib.ptr(aligned), P, N, _lib.ptr(reference), int(bool(similarity)),
              _lib.ptr(prev_mean), _lib.ptr(mean_out), _lib.ptr(change_out), _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
    return ws


def shape_gram(aligned, mean):
    """``focusr_shape_gram``: (P, P) float64 device tensor D D^T, D = ``aligned`` (P, N, 3) - ``mean`` (N, 3) as [P][3N]."""
    torch = _torch()
    P, N = int(aligned.shape[0]), int(aligned.shape[1])
    nbytes = int(_lib.load().focusr_shape_gram_workspace_bytes(P, N))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=aligned.device)
    gram = torch.empty((P, P), dtype=torch.float64, device=aligned.device)
    _lib.call("focusr_shape_gram", _lib.ptr(aligned), _lib.ptr(mean), P, N, _lib.ptr(gram), _lib.ptr(ws), nbytes,
              _lib.stream_ptr())
    return gram


def shape_modes(aligned, mean, weights):
    """``focusr_shape_modes``: (K, N, 3) float64 device tensor D^T W for ``weights`` (P, K), D as in :func:`shape_gram`."""
    torch = _torch()
    P, N, K = int(aligned.shape[0]), int(aligned.shape[1]), int(weights.shape[1])
    w = weights.to(device=aligned.device, dtype=torch.float64).contiguous()
    modes = torch.empty((K, N, 3), dtype=torch.float64, device=aligned.device)
    _lib.call("focusr_shape_modes", _lib.ptr(aligned), _lib.ptr(mean), P, N, _lib.ptr(w), K, _lib.ptr(modes),
              _lib.stream_ptr())
    return modes


def curvatures(points, tris):
    """vtkCurvatures on the device (vtk_functions.py:40-74).  ``points`` (N, 3) f64, ``tris`` (F, 3) i32, host or
    device.  Returns a dict of device tensors ``gauss``, ``mean``, ``minimum``, ``maximum``, each (N,)."""
    torch = _torch()
    lib = _lib.load()
    pts = points if isinstance(points, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(points, dtype=np.float64))
    tr = tris if isinstance(tris, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(tris, dtype=np.int32))
    pts = pts.to(device="cuda", dtype=torch.float64).contiguous()
    tr = tr.to(device="cuda", dtype=torch.int32).contiguous()
    n, f = int(pts.shape[0]), int(tr.shape[0])
    out = torch.empty((4, n), dtype=torch.float64, device=pts.device)
    nbytes = int(lib.focusr_curvature_workspace_bytes(n, f))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=pts.device)
    _lib.call("focusr_curvatures", _lib.ptr(pts), _lib.ptr(tr), n, f, _lib.ptr(out[0]), _lib.ptr(out[1]), _lib.ptr(out[2]),
              _lib.ptr(out[3]), _lib.ptr(ws), nbytes, _lib.stream_ptr())
    return dict(gauss=out[0], mean=out[1], minimum=out[2], maximum=out[3])


def node_features(raw, points, mesh_off, norm_std=True, cap=3, norm_0_1=True, want_edge_points=False):
    """Graph.norm_node_features (graph.py:121-142) for every (mesh, column) of a batch (``focusr_node_features``).
    ``raw`` device [n_points][f] float64, ``points`` device [n_points][3], ``mesh_off`` device int32 [n_meshes + 1].
    ``cap``: any value but ``False`` caps at +-cap, as the reference does.  Returns ``(features [n_points][f],
    edge_points [n_points][3 + f] or None)``: xyz followed by the features times each mesh's mean xyz range
    (graph.py:166-175).  Does not synchronise."""
    torch = _torch()
    lib = _lib.load()
    n, f, m = int(raw.shape[0]), int(raw.shape[1]), int(mesh_off.shape[0]) - 1
    out = torch.empty((n, f), dtype=torch.float64, device=raw.device)
    ep = torch.empty((n, 3 + f), dtype=torch.float64, device=raw.device) if want_edge_points else None
    ws_bytes = int(lib.focusr_node_features_workspace_bytes(n, m, f))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=raw.device)
    has_cap = cap is not False
    _lib.call("focusr_node_features", _lib.ptr(raw), _lib.ptr(points), n, _lib.ptr(mesh_off), m, f, int(norm_std is True),
              int(has_cap), float(cap) if has_cap else 0.0, int(norm_0_1 is True), _lib.ptr(out), _lib.ptr(ep), _lib.ptr(ws),
              ws_bytes, _lib.stream_ptr())
    return out, ep


def feature_coords(spectral, smoothed, points, mesh_off, include_points=False, norm_physical_and_spectral=True):
    """The extended correspondence coordinates of focusr.py:218-295 for every mesh of a batch (``focusr_feature_coords``):
    ``spectral`` device [n_points][ns], then the smoothed features ``smoothed`` [n_points][f] (or None) rescaled to each
    mesh's spectral range, then, with ``include_points``, the normed (or raw) xyz of ``points``.  Returns a new device
    tensor [n_points][ns + f + 3 * include_points]."""
    torch = _torch()
    n, ns = int(spectral.shape[0]), int(spectral.shape[1])
    f = 0 if smoothed is None else int(smoothed.shape[1])
    m = int(mesh_off.shape[0]) - 1
    out = torch.empty((n, ns + f + (3 if include_points else 0)), dtype=torch.float64, device=spectral.device)
    _lib.call("focusr_feature_coords", _lib.ptr(spectral), ns, _lib.ptr(smoothed), f, _lib.ptr(points), n,
              _lib.ptr(mesh_off), m, int(bool(include_points)), int(bool(norm_physical_and_spectral)), _lib.ptr(out),
              _lib.stream_ptr())
    return out


def eigsort_decide(graph, vals, n_found, t_mesh, s_mesh, costs, n_features, ns, target_as_reference=True, weighted=True):
    """The n x n decisions of eigsort for every pair on the device (``focusr_eigsort_decide``): no host visit.
    ``vals`` device [n_meshes][ldv]; ``n_found`` host ints [n_meshes]; ``costs`` = (c_hist, c_hist_f, c_spatial,
    c_spatial_f) device tensors [n_pairs][n][n].  Returns device tensors: Q [n_pairs][n], dst / src / sign int32
    [n_meshes][n], weights [n_meshes][ns], status int32 [1] (non-zero: an assignment was infeasible)."""
    torch = _torch()
    lib = _lib.load()
    dev = graph.device
    n, m = int(n_features), graph.n_meshes
    tm, sm, nf = _dev_i32(t_mesh), _dev_i32(s_mesh), _dev_i32(n_found)
    n_pairs = int(tm.shape[0])
    q = torch.empty((n_pairs, n), dtype=torch.float64, device=dev)
    ident = torch.arange(n, dtype=torch.int32, device=dev).repeat(m, 1)
    dst, src = ident.clone(), ident
    sign = torch.ones((m, n), dtype=torch.int32, device=dev)
    w = torch.ones((m, int(ns)), dtype=torch.float64, device=dev)
    status = torch.empty(1, dtype=torch.int32, device=dev)
    ws_bytes = int(lib.focusr_eigsort_decide_workspace_bytes(n_pairs, n))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    ch, chf, cs, csf = costs
    _lib.call("focusr_eigsort_decide", _lib.ptr(vals), int(vals.shape[1]), _lib.ptr(nf), _lib.ptr(tm), _lib.ptr(sm), n_pairs,
              _lib.ptr(ch), _lib.ptr(chf), _lib.ptr(cs), _lib.ptr(csf), n, int(ns), int(bool(target_as_reference)),
              int(bool(weighted)), _lib.ptr(q), _lib.ptr(dst), _lib.ptr(src), _lib.ptr(sign), _lib.ptr(w), _lib.ptr(status),
              _lib.ptr(ws), ws_bytes, _lib.stream_ptr())
    return q, dst, src, sign, w, status


def sample_rows(idx):
    """Ordering samples of a batch, as ``eigsort_costs`` takes them: a 2-D [P][n] array (every pair the same count) stays
    a 2-D int64 array; anything else is read as a sequence of P 1-D arrays (a count per pair) and returned as a list of
    1-D int64 arrays."""
    if getattr(idx, "ndim", None) == 2:
        return np.ascontiguousarray(idx, dtype=np.int64)
    return [np.asarray(r, dtype=np.int64).reshape(-1) for r in idx]


def eigsort_costs(graph, vecs, t_mesh, s_mesh, idx_t, idx_s, n_features):
    """Cost matrices of eigsort for pairs (t_mesh[p], s_mesh[p]) of ``graph``.
    idx_t / idx_s: host int arrays [n_pairs][n_samples] (Graph.rand_idxs), or sequences of n_pairs 1-D arrays (a sample
    count per pair: ``focusr_eigsort_costs_ragged``).  Returns device tensors (c_hist, c_hist_f, c_spatial, c_spatial_f)
    each [n_pairs][n][n] and nn_idx: [n_pairs][n_samp_t] for 2-D input, else a list of per-pair [n_t] views."""
    torch = _torch()
    lib = _lib.load()
    dev = graph.device
    idx_t, idx_s = sample_rows(idx_t), sample_rows(idx_s)
    n = int(n_features)
    tm, sm = _dev_i32(t_mesh), _dev_i32(s_mesh)
    n_pairs = int(tm.shape[0])
    outs = [torch.empty((n_pairs, n, n), dtype=torch.float64, device=dev) for _ in range(4)]
    if isinstance(idx_t, np.ndarray) and isinstance(idx_s, np.ndarray):
        n_t, n_s = idx_t.shape[1], idx_s.shape[1]
        it = torch.from_numpy(idx_t).to(dev)
        is_ = torch.from_numpy(idx_s).to(dev)
        nn = torch.empty((n_pairs, n_t), dtype=torch.int64, device=dev)
        ws_bytes = int(lib.focusr_eigsort_workspace_bytes(n_pairs, n_t, n_s, n))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.call("focusr_eigsort_costs", _lib.ptr(vecs), int(vecs.shape[1]), _lib.ptr(graph.points), _lib.ptr(graph.mesh_off),
                  _lib.ptr(tm), _lib.ptr(sm), n_pairs, _lib.ptr(it), _lib.ptr(is_), n_t, n_s, n, _lib.ptr(outs[0]),
                  _lib.ptr(outs[1]), _lib.ptr(outs[2]), _lib.ptr(outs[3]), _lib.ptr(nn), _lib.ptr(ws), ws_bytes,
                  _lib.stream_ptr())
        return outs[0], outs[1], outs[2], outs[3], nn
    rows_t, rows_s = list(idx_t), list(idx_s)
    if len(rows_t) != n_pairs or len(rows_s) != n_pairs:
        raise ValueError("eigsort_costs: %d pairs, but %d target and %d source sample arrays" % (n_pairs, len(rows_t), len(rows_s)))
    cnt_t = np.array([r.size for r in rows_t], dtype=np.int64)
    off_t = np.zeros(n_pairs + 1, dtype=np.int32)
    off_t[1:] = np.cumsum(cnt_t)
    off_s = np.zeros(n_pairs + 1, dtype=np.int32)
    off_s[1:] = np.cumsum([r.size for r in rows_s])
    it = torch.from_numpy(np.concatenate(rows_t)).to(dev)
    is_ = torch.from_numpy(np.concatenate(rows_s)).to(dev)
    ot, os_ = torch.from_numpy(off_t).to(dev), torch.from_numpy(off_s).to(dev)
    nn = torch.empty(int(off_t[-1]), dtype=torch.int64, device=dev)
    ws_bytes = int(lib.focusr_eigsort_ragged_workspace_bytes(_lib.ptr(off_t), _lib.ptr(off_s), n_pairs, n))
    if ws_bytes == 0:
        raise ValueError("eigsort_costs: every pair needs at least one target and one source sample")
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    _lib.call("focusr_eigsort_costs_ragged", _lib.ptr(vecs), int(vecs.shape[1]), _lib.ptr(graph.points),
              _lib.ptr(graph.mesh_off), _lib.ptr(tm), _lib.ptr(sm), n_pairs, _lib.ptr(it), _lib.ptr(is_), _lib.ptr(ot),
              _lib.ptr(os_), _lib.ptr(off_t), _lib.ptr(off_s), n, _lib.ptr(outs[0]), _lib.ptr(outs[1]), _lib.ptr(outs[2]),
              _lib.ptr(outs[3]), _lib.ptr(nn), _lib.ptr(ws), ws_bytes, _lib.stream_ptr())
    return outs[0], outs[1], outs[2], outs[3], list(torch.split(nn, cnt_t.tolist()))
