"""Batched spectral-correspondence stage: many (target, source) mesh pairs per launch.

This is the throughput path of BASELINE.json config 3 ("batch of 1024 synthetic 15k-vertex mesh
pairs sharded across 1/2/4/8 B200").  It is the same sequence ``Focusr.__init__`` +
``Focusr.align_maps`` run for one pair (reference focusr.py:134-169, 514-562, CPD = identity as
in BASELINE.md section 3), but every kernel works on the block-diagonal graph of all 2P meshes, so
one SpMM launch streams gigabytes instead of 1.3 MB and nothing visits the host between the upload
of the vertices and the download of the correspondences except the eigensolver's convergence test
(a few hundred Ritz values and residuals per outer iteration) and, with node features on, the one synchronise of
``focusr_curvatures`` (its triangle-index check).

Mesh order inside the batch graph: targets 0..P-1, then sources 0..P-1.  With ``run(..., target_of_pair=...)`` (many
sources against a few templates) the batch graph holds T distinct targets, then the P sources, and pair p is target
``target_of_pair[p]`` with source p: each target is built, solved and smoothed once, and the results are returned in the
pair layout (target copy p, then source p) of the batch with every target repeated once per pair.  With
``run(..., mesh_pairs=...)`` (all-vs-all, one subject against several atlases, both directions of a pair) the batch graph
holds M meshes in any order and pair p is mesh ``mesh_pairs[p][0]`` with mesh ``mesh_pairs[p][1]``: each mesh is built
and solved once, each target smoothed once, and every pair's projection smoothed on the one copy of its source's graph
(``focusr_mean_filter_mapped``).  ``target_of_pair`` runs as ``mesh_pairs = [(target_of_pair[p], T + p)]``.
"""
from __future__ import annotations

import os
import threading

import numpy as np

from . import _device, _lib
from ._device import DeviceGraph
from .shape import ALIGN_TYPES

__all__ = ["SpectralBatch"]

# graph.py:11-15 (features_dictionary): the focusr_curvatures outputs each name contributes, in order
CURVATURE_FEATURES = {"curvature": ("minimum", "maximum"), "min_curvature": ("minimum",), "max_curvature": ("maximum",)}
MAX_KNN_DIM, MAX_CPD_DIM = 32, 16  # focusr_knn, focusr_cpd_*
# SpectralBatch(surface_distances=...): the transformed source positions whose surface is measured, by the names of
# build_shape_model's align_type
SURFACE_POSITIONS = ALIGN_TYPES


def shared_targets(target_of_pair, n_meshes, n_pairs):
    """Checks ``target_of_pair`` of a batch of ``n_meshes`` meshes (T targets, then ``n_pairs`` sources) and returns it as
    int32 [P] with T.  ``ValueError`` unless it has one integer per pair, T >= 1, every value lies in [0, T) and every
    target is used by some pair."""
    P = int(n_pairs)
    T = int(n_meshes) - P
    top = np.asarray(target_of_pair)
    if top.ndim != 1 or top.size != P:
        raise ValueError("target_of_pair needs one entry per pair (%d), got shape %s" % (P, top.shape))
    if P < 1 or T < 1:
        raise ValueError("a batch with target_of_pair needs at least one pair and one target (mesh layout: T targets, then "
                         "%d sources; %d meshes given)" % (P, n_meshes))
    if top.dtype.kind not in "iu":
        if top.dtype.kind != "f" or not np.all(np.isfinite(top)) or not np.all(top == np.round(top)):
            raise ValueError("target_of_pair must hold integers")
    top = top.astype(np.int64)
    bad = np.nonzero((top < 0) | (top >= T))[0]
    if bad.size:
        raise ValueError("target_of_pair[%d] = %d lies outside [0, %d)" % (bad[0], top[bad[0]], T))
    unused = np.setdiff1d(np.arange(T), top)
    if unused.size:
        raise ValueError("target(s) %s are used by no pair: a batch holds only the targets its pairs use" % unused[:16].tolist())
    return top.astype(np.int32), T


def mesh_pairs_checked(mesh_pairs, n_meshes, n_pairs=None):
    """Checks ``mesh_pairs`` ((target mesh, source mesh) per pair) of a batch of ``n_meshes`` meshes and returns it as
    int32 [P][2].  ``ValueError`` unless it is [P][2] with P >= 1 (and P == ``n_pairs`` when given), every value is an
    integer in [0, n_meshes) and every mesh is used by some pair."""
    mp = np.asarray(mesh_pairs)
    if mp.ndim != 2 or mp.shape[1] != 2:
        raise ValueError("mesh_pairs must be [P][2] (target mesh, source mesh), got shape %s" % (mp.shape,))
    P, M = mp.shape[0], int(n_meshes)
    if P < 1:
        raise ValueError("mesh_pairs needs at least one pair")
    if n_pairs is not None and int(n_pairs) != P:
        raise ValueError("n_pairs (%d) must equal the number of mesh_pairs (%d)" % (int(n_pairs), P))
    if mp.dtype.kind not in "iu":
        if mp.dtype.kind != "f" or not np.all(np.isfinite(mp)) or not np.all(mp == np.round(mp)):
            raise ValueError("mesh_pairs must hold integers")
    mp = mp.astype(np.int64)
    bad = np.argwhere((mp < 0) | (mp >= M))
    if bad.size:
        p, c = bad[0]
        raise ValueError("mesh_pairs[%d][%d] = %d lies outside [0, %d)" % (p, c, mp[p, c], M))
    unused = np.setdiff1d(np.arange(M), mp)
    if unused.size:
        raise ValueError("mesh(es) %s are used by no pair: a batch holds only the meshes its pairs use" % unused[:16].tolist())
    return mp.astype(np.int32)


def check_icp_moving(mesh_pairs, target_to_source):
    """ICP moves one mesh of every pair, and the batch graph is built from the moved points: ``ValueError`` unless every
    moving mesh is in exactly one pair and is not that pair's fixed mesh."""
    fixed, moving = (mesh_pairs[:, 1], mesh_pairs[:, 0]) if target_to_source else (mesh_pairs[:, 0], mesh_pairs[:, 1])
    for p, m in enumerate(moving):
        pairs = np.nonzero((mesh_pairs == m).any(axis=1))[0]
        if pairs.size != 1 or fixed[p] == m:
            raise ValueError("ICP moves mesh %d (the %s of pair %d) onto mesh %d, but mesh %d is in pairs %s: a moving mesh "
                             "must be in exactly one pair and not be that pair's fixed mesh" % (
                                 m, "target" if target_to_source else "source", p, fixed[p], m, pairs.tolist()))


def sample_indices_checked(idx, sizes, name):
    """Checks user-supplied ordering samples of one side of a batch (``idx_t`` or ``idx_s``) against the sizes of that
    side's meshes in pair order, and returns them in the form ``eigsort_costs`` takes (a 2-D array, or a list of 1-D
    arrays).  ``ValueError`` unless there is one non-empty array of integers per pair, each in [0, size of its mesh)."""
    if idx is None:
        raise ValueError("give idx_t and idx_s together")
    rows = _device.sample_rows(idx)
    if len(rows) != len(sizes):
        raise ValueError("%s needs one sample array per pair (%d), got %d" % (name, len(sizes), len(rows)))
    for p, (r, sz) in enumerate(zip(rows, sizes)):
        if r.size == 0:
            raise ValueError("%s[%d] is empty: every pair needs at least one ordering sample" % (name, p))
        lo, hi = int(r.min()), int(r.max())
        if lo < 0 or hi >= sz:
            raise ValueError("%s[%d] holds index %d outside [0, %d) (its mesh has %d vertices)" % (
                name, p, lo if lo < 0 else hi, sz, sz))
    return rows


def layout_rows(src_off, mesh_of, dev):
    """A layout holding a copy of mesh ``mesh_of[i]`` of a batch with mesh offsets ``src_off`` (host), one after the
    other: its mesh offsets (host int32) and the batch row of every one of its rows (device int64)."""
    torch = _lib.require_cuda()
    src_off = np.asarray(src_off, dtype=np.int64)
    sizes = np.diff(src_off)[mesh_of]
    off = np.zeros(sizes.size + 1, dtype=np.int32)
    off[1:] = np.cumsum(sizes)
    # each mesh's shift, repeated over the mesh's rows, plus the row itself
    shift = torch.from_numpy(src_off[mesh_of] - off[:-1]).to(dev, non_blocking=True)
    row_map = torch.arange(int(off[-1]), dtype=torch.int64, device=dev) + torch.repeat_interleave(
        shift, torch.from_numpy(sizes).to(dev, non_blocking=True), output_size=int(off[-1]))
    return off, row_map


class PairLayout:
    """A layout of copies of batch meshes: mesh i is a copy of batch mesh ``mesh_of[i]``.  As the pair layout of a batch
    with shared meshes (``mesh_of`` = the P targets, then the P sources of the pairs) it stands in for the batch's
    ``DeviceGraph`` in the stages that work pair by pair (eigsort, spectral and feature coordinates, CPD, the first
    KNN): same attributes (``mesh_off`` / ``mesh_off_host``, ``n_meshes``, ``n_points``, ``max_mesh_points``,
    ``points``, ``device``) and the same column methods, but no Laplacian of its own.  ``rows`` gathers per-vertex rows
    of the batch graph into this layout (``focusr_gather_rows``)."""

    flip_permute = DeviceGraph.flip_permute
    spectral_coords = DeviceGraph.spectral_coords

    def __init__(self, g, mesh_of):
        torch = _lib.require_cuda()
        self.mesh_of = np.asarray(mesh_of, dtype=np.int64)
        self.device = dev = g.device
        self.mesh_off_host, self.row_map = layout_rows(g.mesh_off_host, self.mesh_of, dev)
        self.n_meshes = int(self.mesh_of.size)
        self.n_points = int(self.mesh_off_host[-1])
        self.max_mesh_points = int(np.diff(self.mesh_off_host).max())
        self.mesh_off = torch.from_numpy(self.mesh_off_host).to(dev, non_blocking=True)
        self.mesh_map = torch.from_numpy(self.mesh_of).to(dev, non_blocking=True)
        self.points = self.rows(g.points)

    def rows(self, values, n_rows=None):
        """Per-vertex rows [n_points of the batch][c] -> the first ``n_rows`` rows of this layout (default: all)."""
        idx = self.row_map if n_rows is None else self.row_map[:n_rows]
        return _device.gather_rows(values.contiguous(), idx)

    def meshes(self, values):
        """Per-mesh rows [batch meshes][c] -> [2P][c]."""
        return _device.gather_rows(values.contiguous(), self.mesh_map)


def mesh_point_scalars(mesh, name):
    """graph.py:88-119: the point scalars called ``name`` of a mesh (PolyData or vtkPolyData) as float64."""
    pd = mesh.GetPointData()
    for idx in range(pd.GetNumberOfArrays()):
        if pd.GetArray(idx).GetName() == name:
            return np.array(np.asarray(pd.GetArray(idx)), dtype=np.float64)
    raise Exception("NO SCALARS WITH SPECIFIED NAME: %s" % name)


class SpectralBatch:
    def __init__(self, n_spectral_features=3, n_extra_spectral=3, n_coords_spectral_ordering=5000,
                 graph_smoothing_iterations=300, projection_smooth_iterations=40,
                 target_eigenmap_as_reference=True, get_weighted_spectral_coords=True, tol=1e-10,
                 block_size=0, seed=0, registration="identity", n_coords_spectral_registration=5000,
                 rigid_before_non_rigid_reg=True, rigid_reg_max_iterations=100, rigid_tolerance=1e-8,
                 non_rigid_max_iterations=1000, non_rigid_tolerance=1e-8, non_rigid_alpha=0.5, non_rigid_beta=3.0,
                 non_rigid_n_eigens=100, cpd_streams=8, icp_register_first=False, icp_registration_mode="rigid",
                 icp_reg_target_to_source=False, list_features_to_calc=("curvature",), list_features_to_get_from_mesh=(),
                 include_features_in_adj_matrix=False, use_features_as_coords=False, feature_smoothing_iterations=40,
                 norm_node_features_std=True, norm_node_features_cap_std=3, norm_node_features_0_1=True,
                 include_points_as_features=False, norm_physical_and_spectral=True, surface_distances=None):
        """The keyword names and defaults of ``Focusr`` where the two share a setting.  ``surface_distances``: None (the
        default: no extra work, no extra keys), or ``"weighted"`` / ``"nearest"`` to have ``run`` measure, for every
        pair, the distances between its transformed source (``weighted_avg_transformed_points`` or
        ``nearest_neighbor_transformed_points`` on the source mesh's triangles) and its target surface, both ways.  The
        keys this adds to ``run``'s result: ``source_to_target_surface_dist``, ``source_to_target_closest_points``,
        ``source_to_target_closest_tri``, ``target_to_source_surface_dist``, ``target_to_source_closest_tri`` and
        ``surface_distance_stats`` (see ``run``); ``build_shape_model`` then reports ``surface_distance_stats`` per
        round.  ``ValueError`` for any other value."""
        if surface_distances is not None and not (isinstance(surface_distances, str) and surface_distances in SURFACE_POSITIONS):
            raise ValueError("surface_distances must be None, 'weighted' or 'nearest', got %r" % (surface_distances,))
        self.surface_distances = surface_distances
        self.ns = int(n_spectral_features)
        self.n = int(n_spectral_features + n_extra_spectral)
        self.n_samples = int(n_coords_spectral_ordering)
        self.graph_smoothing_iterations = int(graph_smoothing_iterations)
        self.projection_smooth_iterations = int(projection_smooth_iterations)
        self.target_as_reference = bool(target_eigenmap_as_reference)
        self.weighted = bool(get_weighted_spectral_coords)
        self.tol = float(tol)
        self.block_size = int(block_size)
        self.seed = int(seed)
        # focusr.py:297-334, 537-543: "identity" (BASELINE.json's throughput configuration) or "b200" = affine +
        # deformable CPD on the GPU, one pair after the other (pyfocusr_b200.cpd; Focusr's keyword names)
        if registration not in ("identity", "b200"):
            raise ValueError("registration must be 'identity' or 'b200'")
        self.registration = registration
        self.n_coords_spectral_registration = int(n_coords_spectral_registration)
        self.rigid_before_non_rigid_reg = bool(rigid_before_non_rigid_reg)
        self.cpd_streams = max(1, int(cpd_streams))
        self.cpd_kwargs = dict(rigid_reg_max_iterations=rigid_reg_max_iterations, rigid_tolerance=rigid_tolerance,
                               non_rigid_max_iterations=non_rigid_max_iterations, non_rigid_tolerance=non_rigid_tolerance,
                               non_rigid_alpha=non_rigid_alpha, non_rigid_beta=non_rigid_beta,
                               non_rigid_n_eigens=non_rigid_n_eigens)
        # focusr.py:106-131 with Focusr's keyword names: rigid ("rigid") or similarity ("similarity") ICP, 100 iterations x
        # 1000 landmarks, of every pair's source onto its target (or the target onto its source), before the Laplacian
        # build; off by default
        if icp_registration_mode not in ("rigid", "similarity"):
            raise TypeError("icp_registration_mode must be 'rigid' or 'similarity', got %r" % (icp_registration_mode,))
        self.icp_register_first = bool(icp_register_first)
        self.icp_registration_mode = icp_registration_mode
        self.icp_reg_target_to_source = bool(icp_reg_target_to_source)
        # graph.py:84-142,166-175 and focusr.py:218-295 with Focusr's keyword names and meanings: node features (curvature
        # columns, then mesh point scalars), normalised per mesh, in the edge weights and / or smoothed and appended to the
        # correspondence coordinates; xyz appended to the coordinates.  The features are computed only when one of the
        # two flags that consume them is set (otherwise the reference discards them), so the default call does no extra
        # work.
        unknown = [f for f in list_features_to_calc if f not in CURVATURE_FEATURES]
        if unknown:
            raise ValueError("unknown feature(s) %s: list_features_to_calc takes %s" % (unknown, sorted(CURVATURE_FEATURES)))
        self.list_features_to_calc = list(list_features_to_calc)
        self.list_features_to_get_from_mesh = list(list_features_to_get_from_mesh)
        self.curvature_columns = [c for f in self.list_features_to_calc for c in CURVATURE_FEATURES[f]]
        self.n_node_features = len(self.curvature_columns) + len(self.list_features_to_get_from_mesh)
        self.include_features_in_adj_matrix = include_features_in_adj_matrix is True
        self.use_features_as_coords = use_features_as_coords is True
        self.feature_smoothing_iterations = int(feature_smoothing_iterations)
        self.norm_node_features_std = norm_node_features_std
        self.norm_node_features_cap_std = norm_node_features_cap_std
        self.norm_node_features_0_1 = norm_node_features_0_1
        self.include_points_as_features = include_points_as_features is True
        self.norm_physical_and_spectral = norm_physical_and_spectral is True
        self.features_in_adjacency = self.n_node_features > 0 and self.include_features_in_adj_matrix
        self.features_as_coords = self.n_node_features > 0 and self.use_features_as_coords
        self.features_on = self.features_in_adjacency or self.features_as_coords
        self.n_coords = self.ns + (self.n_node_features if self.features_as_coords else 0) + \
            (3 if self.include_points_as_features else 0)
        if self.n_coords > MAX_KNN_DIM:
            raise ValueError("correspondence coordinates of %d columns: the KNN stages take at most %d" % (self.n_coords, MAX_KNN_DIM))
        if self.registration == "b200" and self.n_coords > MAX_CPD_DIM:
            raise ValueError("correspondence coordinates of %d columns: registration='b200' (CPD) takes at most %d" % (
                self.n_coords, MAX_CPD_DIM))
        self._tls = threading.local()
        self._pool = None
        self.eigs_options = None  # _lib.EigsOptions or dict: per-call options of the eigensolver (A/B measurements)
        # The smoothing of the target vertices (graph.py:349-354, 300 passes) depends only on the target graphs, not on
        # the spectral stages: with overlap_smoothing it is enqueued on a second CUDA stream right after the Laplacian
        # build and joined where its result is first read; its CTAs fill the gaps the latency-bound filter steps leave
        # (B200, 128 pairs: 1059 -> 1127 pairs/s).  Same kernels, same results; `timings` then attributes the overlapped
        # passes to the eigensolve stage.
        self.overlap_smoothing = os.environ.get("FOCUSR_OVERLAP_SMOOTHING", "1") == "1"
        self.timings = {}

    # ------------------------------------------------------------------------------------------
    def sample_indices(self, sizes, rng=None):
        """Graph.get_list_rand_idxs (graph.py:274-290) for every mesh, in order: ``n_samples`` distinct rows of a mesh, or
        all of its rows when it has fewer.  Returns a 2-D int64 array [len(sizes)][count] when every mesh yields the same
        count, else a list of 1-D int64 arrays (``run`` and ``eigsort_costs`` take both)."""
        rng = rng or np.random.RandomState(self.seed)
        out = []
        for sz in sizes:
            if self.n_samples > sz:
                out.append(np.arange(sz, dtype=np.int64))
            else:
                out.append(rng.choice(sz, size=self.n_samples, replace=False).astype(np.int64))
        if len({len(o) for o in out}) == 1:
            return np.stack(out)
        return out

    # ------------------------------------------------------------------------------------------
    def run(self, points, tris, mesh_off_host, n_pairs, idx_t=None, idx_s=None, record_events=False,
            keep_presort=False, tri_off_host=None, node_features=None, target_of_pair=None, mesh_pairs=None):
        """points: torch tensor [n_points_total, 3] float64 (host pinned or device), meshes in the
        order targets then sources; tris: int32 [n_tris_total, 3] with GLOBAL vertex ids;
        mesh_off_host: int32 [2P+1].  Returns a dict of device tensors + host metadata.

        With ``icp_register_first`` every pair's source is moved onto its target (or the target onto its source) in a
        new device tensor before anything else; ``points`` is never modified and ``icp_matrices`` holds the (P, 4, 4)
        matrices.  ICP needs each mesh's triangle range: ``tri_off_host`` int [2P+1], or else it is derived from
        ``tris``, which must then be grouped by mesh in mesh order as ``pack_meshes`` makes them (``ValueError``
        otherwise; for device ``tris`` the check reads one small result back to the host).

        ``node_features``: the mesh point scalars named by ``list_features_to_get_from_mesh``, host or device
        [n_points_total][len(list_features_to_get_from_mesh)] in the column order of the names (``run_meshes`` fills it);
        required when names are given.  With features on, ``node_features`` in the result is the normalised [n_points]
        [f] block (curvature columns first) and ``coords`` the extended coordinates.

        ``target_of_pair`` (int [P]): many sources against shared targets.  The mesh layout is then T targets, then the P
        sources (T = len(mesh_off_host) - 1 - n_pairs), and pair p is target ``target_of_pair[p]`` with source p.  Each
        target's Laplacian, eigenpairs, features and 300 smoothing passes are computed once; the results are gathered
        into the pair layout (target copy p, then source p), and every key equals, bit for bit, that of ``run`` on the
        batch with each target repeated once per pair, except ``graph`` and ``eigs_info``, which describe the T + P meshes
        built and solved.  ``pair_mesh_off`` holds the pair layout's mesh offsets (with ``target_of_pair=None``: those of
        ``graph``).  ``node_features`` and ``tri_off_host`` follow the T + P layout.  ``ValueError`` for a target outside
        [0, T), a target no pair uses, or ``icp_reg_target_to_source`` with ICP on and a target shared by two pairs.

        ``mesh_pairs`` (int [P][2]): any (target mesh, source mesh) pairs over the M meshes of ``mesh_off_host``, in any
        order; a mesh may be the target of some pairs and the source of others, in any number of pairs, and ``(m, m)``
        is a pair.  Each mesh's Laplacian, eigenpairs and features are computed once, each target's 300 smoothing passes
        once, and each pair's 40 projection passes run on the one copy of its source's graph.  Every key equals, bit for
        bit, that of ``run`` on the pair layout (``run_meshes([meshes[t] for t, _ in mesh_pairs], [meshes[s] for _, s
        in mesh_pairs])``), except ``graph`` and ``eigs_info``, which describe the M meshes; ``pair_mesh_off`` holds the
        pair layout's offsets.  ``ValueError`` for a malformed list, a mesh outside [0, M) or used by no pair, ``n_pairs
        != P``, ``target_of_pair`` given too, or, with ICP on, a moving mesh that is not in exactly one pair or is that
        pair's fixed mesh.  ``target_of_pair`` is the case ``mesh_pairs = [(target_of_pair[p], T + p)]``.

        With ``surface_distances`` set (``SpectralBatch(surface_distances="weighted" | "nearest")``) the result gains, on
        the rows of the pair layout: ``source_to_target_surface_dist`` [source rows] (each transformed source vertex to
        its pair's target surface: the batch graph's target points, after ICP when it is on, and triangles),
        ``source_to_target_closest_points`` [source rows][3] (the point on that surface), ``source_to_target_closest_tri``
        [source rows] int64 (the triangle, local to the target mesh), ``target_to_source_surface_dist`` [target rows]
        (each target vertex to its pair's transformed source surface: the source mesh's triangles on the pair's
        transformed positions), ``target_to_source_closest_tri`` [target rows] int64 (local to the source mesh) and
        ``surface_distance_stats`` (P, 6) (mean and max source -> target, mean and max target -> source, ASSD, Hausdorff;
        ``surface.STATS_COLUMNS``).  The triangle ranges come from ``tri_off_host``, or from ``tris`` as for ICP.  Every
        other key is unchanged, and with shared meshes every new key equals that of the repeated-mesh batch, bit for
        bit.  ``record_events`` then times a ``surface`` stage."""
        P = int(n_pairs)
        mp = None  # (target mesh, source mesh) of every pair when meshes are shared, else None (mesh p with mesh P + p)
        if target_of_pair is not None and mesh_pairs is not None:
            raise ValueError("give mesh_pairs or target_of_pair, not both (target_of_pair is mesh_pairs [(t, T + p)])")
        if target_of_pair is not None:
            top, T = shared_targets(target_of_pair, np.asarray(mesh_off_host).size - 1, P)
            if self.icp_register_first and self.icp_reg_target_to_source and np.unique(top).size < P:
                raise ValueError("icp_reg_target_to_source moves each pair's target onto its source: a target shared by "
                                 "several pairs would move differently for each of them")
            mp = np.stack([top, np.arange(T, T + P, dtype=np.int32)], axis=1)
        elif mesh_pairs is not None:
            mp = mesh_pairs_checked(mesh_pairs, np.asarray(mesh_off_host).size - 1, P)
        if mp is not None and self.icp_register_first:
            check_icp_moving(mp, self.icp_reg_target_to_source)
        if idx_t is not None:  # the pair layout's target and source sizes, from the host offsets
            sizes = np.diff(np.asarray(mesh_off_host, dtype=np.int64))
            t_sizes, s_sizes = (sizes[:P], sizes[P:2 * P]) if mp is None else (sizes[mp[:, 0]], sizes[mp[:, 1]])
            idx_t = sample_indices_checked(idx_t, t_sizes, "idx_t")
            idx_s = sample_indices_checked(idx_s, s_sizes, "idx_s")
        n_mesh_feats = len(self.list_features_to_get_from_mesh)
        if n_mesh_feats:
            n_total = int(np.asarray(mesh_off_host)[-1])
            if node_features is None:
                raise ValueError("list_features_to_get_from_mesh names %d mesh scalar(s): pass them as node_features "
                                 "[n_points][%d] (run_meshes does)" % (n_mesh_feats, n_mesh_feats))
            if tuple(node_features.shape) != (n_total, n_mesh_feats):
                raise ValueError("node_features must be [%d][%d], got %s" % (n_total, n_mesh_feats, tuple(node_features.shape)))
        torch = _lib.require_cuda()
        ev = []

        def mark(name):
            if record_events:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                ev.append((name, e))

        mark("start")
        icp_mats = None
        if self.icp_register_first:
            points, tris, icp_mats = self._icp(points, tris, mesh_off_host, P, tri_off_host, mp)
            mark("icp")
        feats, edge_points = None, None
        if self.features_on:
            points, tris, feats, edge_points = self._node_features(points, tris, mesh_off_host, node_features)
            mark("features")
        g = DeviceGraph.from_device(points, tris, mesh_off_host, edge_points)
        mark("laplacian")
        n, ns = self.n, self.ns
        if mp is None:
            nt_total = int(g.mesh_off_host[P])

            def smooth_targets():
                return g.mean_filter(g.points, self.graph_smoothing_iterations, 0, nt_total)
        else:  # the compact target block: the distinct targets in mesh order, cb_of[p] = pair p's target in it.  Mesh order
            # makes the block the contiguous graph rows of consecutive targets (target_of_pair, all-vs-all), which
            # focusr_mean_filter_mapped smooths with the identity form
            tb = PairLayout(g, np.unique(mp[:, 0]))
            cb_index = np.zeros(g.n_meshes, dtype=np.int32)
            cb_index[tb.mesh_of] = np.arange(tb.n_meshes)
            cb_of = cb_index[mp[:, 0]]

            def smooth_targets():
                return g.mean_filter_mapped(tb.points, self.graph_smoothing_iterations, tb.mesh_of)
        smoothed_t, side = None, None
        if self.overlap_smoothing:
            main = torch.cuda.current_stream()
            if getattr(self._tls, "side_stream", None) is None:  # one stream per host thread for the life of the object:
                self._tls.side_stream = torch.cuda.Stream(device=g.device)  # the caching allocator keeps a pool per stream
            side = self._tls.side_stream
            side.wait_stream(main)
            with torch.cuda.stream(side):
                smoothed_t = smooth_targets()
            smoothed_t.record_stream(main)
        try:
            vals, vecs, info = g.eigs_smallest(k=n + 1, n_k_needed=n, k_buffer=1, tol=self.tol,
                                               block_size=self.block_size, options=self.eigs_options)
        except _lib.FocusrB200Error as exc:
            info = getattr(exc, "eigs_info", None)
            if info is None:
                raise
            bad = np.nonzero(info["status"] != 0)[0]
            if mp is None:
                raise RuntimeError("eigensolve failed for %d of %d meshes: %s (mesh m is the %s of pair m %% %d); the other "
                                   "meshes of the batch were solved -- drop the named pairs and rerun" % (
                                       bad.size, 2 * P, ", ".join("mesh %d: %s" % (m, _device.EIG_STATUS.get(int(info["status"][m]), "?"))
                                                                  for m in bad[:16]), "target if m < %d else source" % P, P)) from exc
            raise RuntimeError("eigensolve failed for %d of %d meshes: %s; the other meshes of the batch were solved -- drop "
                               "the named pairs and rerun" % (bad.size, g.n_meshes, ", ".join(
                                   "%s: %s" % (self._mesh_pairs(m, mp), _device.EIG_STATUS.get(int(info["status"][m]), "?"))
                                   for m in bad[:16]))) from exc
        n_found = info["n_found"]
        if int(n_found.min()) < n:
            short = np.nonzero(n_found < n)[0]
            if mp is None:
                raise RuntimeError("meshes %s returned fewer than %d eigenpairs (pairs %s)" % (
                    short[:16].tolist(), n, sorted(set(int(m) % P for m in short[:16]))))
            raise RuntimeError("fewer than %d eigenpairs for %s" % (n, "; ".join(self._mesh_pairs(m, mp) for m in short[:16])))
        g.normalize_columns(vecs, n_found)
        mark("eigensolve")
        pg = g  # the graph of the pair stages: the batch graph itself, or its pair layout
        if mp is not None:  # gather the rows of every pair's target, then of every pair's source, into the pair layout
            pg = PairLayout(g, np.concatenate([mp[:, 0], mp[:, 1]]))
            vecs, vals, n_found = pg.rows(vecs), pg.meshes(vals), n_found[pg.mesh_of]
            mark("pair_layout")

        off = pg.mesh_off_host
        sizes = np.diff(off)
        if idx_t is None:
            rng = np.random.RandomState(self.seed)
            idx_t = self.sample_indices(sizes[:P], rng)
            idx_s = self.sample_indices(sizes[P:], rng)
        t_mesh = np.arange(P, dtype=np.int32)
        s_mesh = np.arange(P, 2 * P, dtype=np.int32)
        ch, chf, cs, csf, _ = _device.eigsort_costs(pg, vecs, t_mesh, s_mesh, idx_t, idx_s, n)
        # n x n decisions per pair (eigsort.py:66-122, 142-160; focusr.py:459-490) on the device: c_lambda, min(c, c_f),
        # the assignment (scipy's algorithm and tie rules), flips, column moves and spectral weights -- no host visit
        Q, dst, src, sign, weights, decide_status = _device.eigsort_decide(
            pg, vals, n_found, t_mesh, s_mesh, (ch, chf, cs, csf), n, ns, self.target_as_reference, self.weighted)
        costs = (ch, chf, cs, csf)
        presort = vecs.clone() if keep_presort else None
        pg.flip_permute(vecs, dst, src, sign)
        coords = pg.spectral_coords(vecs, weights, ns)
        mark("eigsort")
        if self.features_as_coords or self.include_points_as_features:  # focusr.py:218-295, in Focusr's order
            smoothed_f = None
            if self.features_as_coords:  # focusr_mean_filter smooths up to 8 columns per call
                parts = [g.mean_filter(feats[:, a:a + 8].contiguous(), self.feature_smoothing_iterations)
                         for a in range(0, self.n_node_features, 8)]
                smoothed_f = parts[0] if len(parts) == 1 else torch.cat(parts, dim=1)
                if mp is not None:
                    smoothed_f = pg.rows(smoothed_f)
            coords = _device.feature_coords(coords, smoothed_f, pg.points, pg.mesh_off, self.include_points_as_features,
                                            self.norm_physical_and_spectral)
            mark("feature_coords")

        dev = g.device
        nt_pair = int(off[P])
        ref_off = pg.mesh_off[: P + 1].contiguous()
        qry_off = (pg.mesh_off[P:] - nt_pair).contiguous()
        max_q, max_r = int(sizes[P:].max()), int(sizes[:P].max())
        cpd_idx, coords_b4_reg = None, None
        if self.registration == "b200":  # register every pair's target coordinates onto its source's
            coords_b4_reg = coords.clone()
            cpd_idx = self._register_pairs(coords, off, P, sizes)
            mark("cpd")
        idx0, _ = _device.knn(coords[:nt_pair], coords[nt_pair:], k=1, ref_off=ref_off, query_off=qry_off,
                              max_queries=max_q, max_refs=max_r, want_dist=False)
        mark("knn_initial")
        if side is not None:
            torch.cuda.current_stream().wait_stream(side)
        else:
            smoothed_t = smooth_targets()
        if mp is None:
            base_q = torch.repeat_interleave(g.mesh_off[:P], torch.from_numpy(sizes[P:].astype(np.int64)).to(dev)).to(torch.int32)
            staged = torch.empty_like(g.points)
            _lib.call("focusr_gather_rows", _lib.ptr(smoothed_t), _lib.ptr(idx0), _lib.ptr(base_q), g.n_points - nt_total, 3,
                      _lib.ptr(staged[nt_total:]), _lib.stream_ptr())
            src_proj = g.mean_filter(staged, self.projection_smooth_iterations, nt_total, g.n_points)[nt_total:]
        else:  # every pair's smoothed target, at idx0, smoothed on the one copy of its source's graph
            q_sizes = torch.from_numpy(sizes[P:].astype(np.int64)).to(dev, non_blocking=True)
            staged = _device.gather_rows(smoothed_t, idx0, torch.repeat_interleave(
                torch.from_numpy(tb.mesh_off_host[cb_of]).to(dev, non_blocking=True), q_sizes, output_size=pg.n_points - nt_pair))
            src_proj = g.mean_filter_mapped(staged, self.projection_smooth_iterations, mp[:, 1])
        mark("smoothing")
        # one k=3 search serves both focusr.py:391-392 (k=1: its first column, same distances and tie
        # rule) and focusr.py:409-413 (k=3)
        if mp is None:
            idx3, dist3 = _device.knn(smoothed_t[:nt_total], src_proj, k=3, ref_off=ref_off, query_off=qry_off,
                                      max_queries=max_q, max_refs=max_r)
        else:  # each target's Morton sort and tiles serve all of its pairs
            idx3, dist3 = _device.knn_mapped(smoothed_t, src_proj, tb.mesh_off, qry_off, cb_of, k=3, max_queries=max_q,
                                             max_refs=tb.max_mesh_points)
            # the first row of each pair's target in the batch graph
            base_q = torch.repeat_interleave(torch.from_numpy(g.mesh_off_host[mp[:, 0]]).to(dev, non_blocking=True),
                                             q_sizes, output_size=pg.n_points - nt_pair)
        idx1 = idx3[:, :1]
        weighted = _device.weighted_positions(idx3, dist3, g.points, base_q)
        nearest = _device.gather_rows(g.points, idx1[:, 0].contiguous(), base_q)
        mark("knn_final")
        if mp is None:
            smoothed_tc = smoothed_t[:nt_total]
        else:
            smoothed_tc = _device.gather_rows(smoothed_t, layout_rows(tb.mesh_off_host, cb_of, dev)[1])
            if feats is not None:
                feats = pg.rows(feats)
        surf = {}
        if self.surface_distances is not None:
            positions = weighted if self.surface_distances == "weighted" else nearest
            surf = self._surface(g, pg, positions, tri_off_host, mp, P)
            mark("surface")
        if record_events:
            torch.cuda.synchronize()
            self.timings = {ev[i][0]: ev[i - 1][1].elapsed_time(ev[i][1]) for i in range(1, len(ev))}
        return dict(graph=g, eig_vals=vals, eig_vecs=vecs, eigs_info=info, Q=Q, spectral_weights=weights[:P],
                    eigsort_status=decide_status, pair_mesh_off=off,
                    coords=coords, initial_idx=idx0[:, 0], smoothed_target_coords=smoothed_tc,
                    source_projected_on_target=src_proj, final_idx=idx1[:, 0], knn3_idx=idx3,
                    knn3_dist=dist3, weighted_avg_transformed_points=weighted,
                    nearest_neighbor_transformed_points=nearest, idx_t=idx_t, idx_s=idx_s, costs=costs,
                    eig_vecs_presort=presort, cpd_idx=cpd_idx, coords_b4_reg=coords_b4_reg, icp_matrices=icp_mats,
                    node_features=feats, **surf)

    def _surface(self, g, pg, positions, tri_off_host, mesh_pairs, P):
        """The surface-distance keys of ``run``: every pair's transformed source rows (``positions``, the source rows of
        the pair layout ``pg``) against its target mesh of the batch graph ``g`` (each distinct target tiled once), and
        the pair layout's target rows against the pair's source triangles re-based onto the pair's rows of
        ``positions``."""
        from . import surface

        torch = _lib.require_cuda()
        dev = g.device
        if tri_off_host is None:
            tri_off = self.tri_offsets(g.tris, g.mesh_off_host)
        else:
            tri_off = np.ascontiguousarray(tri_off_host, dtype=np.int32).reshape(-1)
            if tri_off.size != g.n_meshes + 1 or tri_off[0] != 0 or tri_off[-1] != g.n_tris or np.any(np.diff(tri_off) < 0):
                raise ValueError("tri_off_host must hold %d non-decreasing triangle offsets from 0 to %d" % (
                    g.n_meshes + 1, g.n_tris))
        t_mesh, s_mesh = (np.arange(P), np.arange(P, 2 * P)) if mesh_pairs is None else (mesh_pairs[:, 0], mesh_pairs[:, 1])
        off = pg.mesh_off_host
        nt_pair = int(off[P])
        src_off, tgt_off = (off[P:] - nt_pair).astype(np.int32), off[:P + 1]
        closest, s_tri, s_dist = surface.closest_points(g.points, g.tris, g.mesh_off_host, tri_off, positions, src_off, t_mesh)
        # pair p's source triangles, their ids moved from the source mesh's rows of g to pair p's rows of `positions`
        s_tri_off, tri_rows = layout_rows(tri_off, s_mesh, dev)
        shift = torch.from_numpy(src_off[:-1].astype(np.int64) - g.mesh_off_host[s_mesh]).to(dev, non_blocking=True)
        shift = torch.repeat_interleave(shift, torch.from_numpy(np.diff(s_tri_off).astype(np.int64)).to(dev, non_blocking=True),
                                        output_size=int(s_tri_off[-1]))
        s_tris = (g.tris.index_select(0, tri_rows) + shift[:, None]).to(torch.int32).contiguous()
        _, t_tri, t_dist = surface.closest_points(positions, s_tris, src_off, s_tri_off, pg.points[:nt_pair], tgt_off,
                                                  np.arange(P), want_closest=False)
        return dict(source_to_target_surface_dist=s_dist, source_to_target_closest_points=closest,
                    source_to_target_closest_tri=s_tri, target_to_source_surface_dist=t_dist,
                    target_to_source_closest_tri=t_tri,
                    surface_distance_stats=surface.distance_stats(s_dist, src_off, t_dist, tgt_off))

    @staticmethod
    def _mesh_pairs(m, mesh_pairs):
        """Mesh m of a batch graph with shared meshes named by every pair it serves."""
        t, s = (np.nonzero(mesh_pairs[:, c] == m)[0].tolist() for c in (0, 1))
        return "mesh %d (%s)" % (m, ", ".join((["target of pairs %s" % t] if t else []) + (["source of pairs %s" % s] if s else [])))

    def _node_features(self, points, tris, mesh_off_host, node_features):
        """graph.py:84-142,166-175 for every mesh at once: curvature of the (moved) points in one focusr_curvatures call
        over the whole batch (it synchronises once, for its index check), the mesh scalars behind it, then
        focusr_node_features.  Returns the device points and triangles, the normalised features [n_points][f] and the
        edge points [n_points][3 + f] (None unless the features go into the edge weights)."""
        torch = _lib.require_cuda()
        lib = _lib.load()
        dev = torch.device("cuda", torch.cuda.current_device())
        pts = points.to(dev, non_blocking=True).contiguous()
        tr = tris.to(dev, non_blocking=True).contiguous()
        n, nf = int(pts.shape[0]), int(tr.shape[0])
        raw = torch.empty((n, self.n_node_features), dtype=torch.float64, device=dev)
        nc = len(self.curvature_columns)
        if nc:
            curv = torch.empty((2, n), dtype=torch.float64, device=dev)
            ws_bytes = int(lib.focusr_curvature_workspace_bytes(n, nf))
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            _lib.call("focusr_curvatures", _lib.ptr(pts), _lib.ptr(tr), n, nf, None, None, _lib.ptr(curv[0]),
                      _lib.ptr(curv[1]), _lib.ptr(ws), ws_bytes, _lib.stream_ptr())
            for k, c in enumerate(self.curvature_columns):
                raw[:, k] = curv[0 if c == "minimum" else 1]
        if nc < self.n_node_features:
            raw[:, nc:] = torch.as_tensor(node_features, dtype=torch.float64).to(dev, non_blocking=True)
        mesh_off = torch.from_numpy(np.ascontiguousarray(mesh_off_host, dtype=np.int32)).to(dev, non_blocking=True)
        feats, edge_points = _device.node_features(raw, pts, mesh_off, self.norm_node_features_std,
                                                   self.norm_node_features_cap_std, self.norm_node_features_0_1,
                                                   want_edge_points=self.features_in_adjacency)
        return pts, tr, feats, edge_points

    def _icp(self, points, tris, mesh_off_host, P, tri_off_host, mesh_pairs=None):
        """focusr.py:110-131 for every pair at once (``focusr_icp_batch``): returns the device points with each pair's
        moving mesh registered onto its fixed one (a new tensor), the device triangles and the (P, 4, 4) matrices.  With
        ``mesh_pairs`` pair p is batch mesh ``mesh_pairs[p][0]`` with mesh ``mesh_pairs[p][1]``."""
        torch = _lib.require_cuda()
        off = np.ascontiguousarray(mesh_off_host, dtype=np.int32)
        if tri_off_host is None:
            tri_off_host = self.tri_offsets(tris, off)
        dev = torch.device("cuda", torch.cuda.current_device())
        pts = points.to(dev, non_blocking=True).contiguous()
        tr = tris.to(dev, non_blocking=True).contiguous()
        targets, sources = np.arange(P, dtype=np.int32), np.arange(P, 2 * P, dtype=np.int32)
        if mesh_pairs is not None:
            targets, sources = mesh_pairs[:, 0].copy(), mesh_pairs[:, 1].copy()
        fixed, moving = (sources, targets) if self.icp_reg_target_to_source else (targets, sources)
        mats, moved = _device.icp_batch_device(pts, tr, off, tri_off_host, fixed, moving, max_iterations=100,
                                               max_landmarks=1000, similarity=self.icp_registration_mode == "similarity")
        return moved, tr, mats

    @staticmethod
    def tri_offsets(tris, mesh_off_host):
        """Per-mesh triangle ranges int32 [M+1] of ``tris`` (torch int [F, 3], global vertex ids, host or device), which
        must be grouped by mesh in mesh order (every triangle's vertices in one mesh, meshes non-decreasing), as
        ``pack_meshes`` makes them; ``ValueError`` otherwise.  Device ``tris`` cost one small read back to the host."""
        import torch

        off = np.ascontiguousarray(mesh_off_host, dtype=np.int64)
        m = off.size - 1
        t = torch.as_tensor(tris).reshape(-1, 3).to(torch.int64)
        mesh = torch.bucketize(t, torch.from_numpy(off[1:-1].copy()).to(t.device), right=True)  # mesh of every vertex id
        m0 = mesh[:, 0]
        ok = (mesh == m0[:, None]).all() & (t >= int(off[0])).all() & (t < int(off[-1])).all() & (m0[1:] >= m0[:-1]).all()
        res = torch.cat([ok.reshape(1).to(torch.int64), torch.bincount(m0, minlength=m)[:m]]).cpu().numpy()
        if not res[0]:
            raise ValueError("tris must be grouped by mesh in mesh order (as pack_meshes makes them) to derive the "
                             "per-mesh triangle ranges; pass tri_off_host otherwise")
        tri_off = np.zeros(m + 1, dtype=np.int32)
        tri_off[1:] = np.cumsum(res[1:])
        return tri_off

    # ------------------------------------------------------------------------------------------
    def run_concurrent(self, sub_batches, **kw):
        """Several independent sub-batches at once, one host thread and one CUDA stream each: ``sub_batches`` is a list
        of ``(points, tris, mesh_off_host, n_pairs)`` or of dicts of ``run`` keyword arguments.  A batch is a chain of
        HBM-bound stages (Laplacian, filter steps, smoothing) followed by FP64-ALU / latency-bound ones (eigsort costs,
        KNN) with a few host visits in between; two sub-batches in flight let one's KNN and host visits hide under the
        other's filter steps (B200, 128 pairs as 2 x 64: 1186 -> see DESIGN.md).  Results are those of ``run`` on each
        sub-batch (deterministic kernels, no shared state); returns the list of result dicts in order."""
        from concurrent.futures import ThreadPoolExecutor

        torch = _lib.require_cuda()
        jobs = [dict(zip(("points", "tris", "mesh_off_host", "n_pairs"), b)) if not isinstance(b, dict) else dict(b)
                for b in sub_batches]
        if len(jobs) == 1:
            return [self.run(**jobs[0], **kw)]
        if self._pool is None or self._pool._max_workers < len(jobs):
            self._pool = ThreadPoolExecutor(max_workers=len(jobs))  # kept: workers own pinned pools and streams
        main = torch.cuda.current_stream()
        device = torch.cuda.current_device()

        def work(job):
            with torch.cuda.device(device):
                if getattr(self._tls, "stream", None) is None:
                    self._tls.stream = torch.cuda.Stream(device=device)
                st = self._tls.stream
                st.wait_stream(main)
                with torch.cuda.stream(st):
                    out = self.run(**job, **kw)
                return out, st

        def hand_over(obj):  # results were allocated on the worker's stream and are used on the caller's from here on
            for v in (obj.values() if isinstance(obj, dict) else vars(obj).values()):
                if isinstance(v, torch.Tensor) and v.is_cuda:
                    v.record_stream(main)
                elif isinstance(v, (tuple, list)):
                    for w in v:
                        if isinstance(w, torch.Tensor) and w.is_cuda:
                            w.record_stream(main)

        results = []
        for out, st in self._pool.map(work, jobs):
            main.wait_stream(st)
            hand_over(out)
            if out.get("graph") is not None:
                hand_over(out["graph"])
            results.append(out)
        return results

    # ------------------------------------------------------------------------------------------
    def run_pipelined(self, jobs, depth=2, consume=None, **kw):
        """A stream of independent batches with at most ``depth`` of them in flight, one host thread and one CUDA stream
        each: ``jobs`` is an iterable of dicts of ``run`` keyword arguments (successive steps of a production queue).
        Unlike ``run_concurrent`` the launches keep their full size -- every kernel works on a whole batch -- while the
        FP64-ALU / latency-bound tail of one batch (eigsort, KNN, host visits) hides under the HBM-bound filter steps of
        the next.  ``consume(out, k)`` runs in the worker thread right after batch k has been enqueued, with its stream
        current (read results back there, keep what is needed); what it returns is collected in order.  Default: the
        whole result dict is kept (its tensors are handed over to the caller's stream)."""
        from concurrent.futures import ThreadPoolExecutor

        torch = _lib.require_cuda()
        jobs = [dict(j) for j in jobs]
        depth = max(1, min(int(depth), len(jobs)))
        main = torch.cuda.current_stream()
        device = torch.cuda.current_device()
        if depth == 1:
            return [consume(self.run(**j, **kw), k) if consume else self.run(**j, **kw) for k, j in enumerate(jobs)]
        if self._pool is None or self._pool._max_workers < depth:
            self._pool = ThreadPoolExecutor(max_workers=depth)  # kept: workers own pinned pools and streams
        streams = set()
        lock = threading.Lock()

        def work(item):
            k, job = item
            with torch.cuda.device(device):
                if getattr(self._tls, "stream", None) is None:
                    self._tls.stream = torch.cuda.Stream(device=device)
                st = self._tls.stream
                with lock:
                    streams.add(st)
                st.wait_stream(main)
                with torch.cuda.stream(st):
                    out = self.run(**job, **kw)
                    if consume is not None:
                        return consume(out, k)
                    for obj in (out, out.get("graph")):
                        if obj is None:
                            continue
                        for v in (obj.values() if isinstance(obj, dict) else vars(obj).values()):
                            if isinstance(v, torch.Tensor) and v.is_cuda:
                                v.record_stream(main)
                    return out

        # ThreadPoolExecutor hands items to idle workers in order: at most `depth` batches are in flight
        results = list(self._pool.map(work, list(enumerate(jobs))))
        for st in streams:
            main.wait_stream(st)
        return results

    # ------------------------------------------------------------------------------------------
    def _register_pairs(self, coords, off, P, sizes):
        """focusr.py:537-543 per pair: affine on fresh random subsets, transform all target coordinates, then
        deformable on fresh subsets, transform again.  Returns the index draws [(s_aff, t_aff, s_def, t_def)].

        The pairs are independent, and one registration leaves most of the GPU idle during its latency-bound
        steps (the r x r solve, the host Rayleigh-Ritz of the low-rank set-up), so ``cpd_streams`` host threads
        run registrations concurrently, one CUDA stream each (ctypes releases the GIL inside the library).  All
        random draws are made up front in pair order: the result does not depend on the thread schedule."""
        from concurrent.futures import ThreadPoolExecutor

        from .cpd import affine_registration, deformable_registration

        torch = _lib.require_cuda()
        rng = np.random.RandomState(self.seed + 7919)
        kw = self.cpd_kwargs
        stages = (["affine"] if self.rigid_before_non_rigid_reg else []) + ["deformable"]

        def draw(n):  # Graph.get_list_rand_idxs (graph.py:274-290)
            if self.n_coords_spectral_registration > n:
                return np.arange(n, dtype=np.int64)
            return rng.choice(n, size=self.n_coords_spectral_registration, replace=False).astype(np.int64)

        draws = []
        for p in range(P):
            nt, ns = int(off[p + 1] - off[p]), int(off[P + p + 1] - off[P + p])
            rec = []
            for _ in stages:
                rec += [draw(ns), draw(nt)]   # source first, as the reference's dict literal evaluates
            draws.append(tuple(rec))

        main = torch.cuda.current_stream()
        device = coords.device

        def work(pairs):
            st = torch.cuda.Stream(device=device)
            st.wait_stream(main)
            with torch.cuda.device(device), torch.cuda.stream(st):
                for p in pairs:
                    t0, t1, s0, s1 = int(off[p]), int(off[p + 1]), int(off[P + p]), int(off[P + p + 1])
                    tgt, src = coords[t0:t1], coords[s0:s1]
                    for k, stage in enumerate(stages):
                        i_s, i_t = draws[p][2 * k], draws[p][2 * k + 1]
                        x = src[torch.from_numpy(i_s).to(device)]
                        y = tgt[torch.from_numpy(i_t).to(device)]
                        if stage == "affine":
                            reg = affine_registration(X=x, Y=y, max_iterations=kw["rigid_reg_max_iterations"],
                                                      tolerance=kw["rigid_tolerance"])
                        else:
                            reg = deformable_registration(X=x, Y=y, num_eig=kw["non_rigid_n_eigens"],
                                                          max_iterations=kw["non_rigid_max_iterations"],
                                                          tolerance=kw["non_rigid_tolerance"], alpha=kw["non_rigid_alpha"],
                                                          beta=kw["non_rigid_beta"])
                        reg.register()
                        tgt.copy_(reg.transform_point_cloud(tgt.contiguous()))
            st.synchronize()
            return st

        n_workers = min(self.cpd_streams, P)
        chunks = [list(range(w, P, n_workers)) for w in range(n_workers)]
        if n_workers == 1:
            work(chunks[0])
        else:
            with ThreadPoolExecutor(max_workers=n_workers) as pool:
                for st in pool.map(work, chunks):
                    main.wait_stream(st)
        return draws

    def fetch(self, out, keys=("final_idx", "weighted_avg_transformed_points"), slot=0):
        """Device -> host read-back of the per-vertex results into reusable pinned buffers (one
        asynchronous copy each, then a single synchronisation).  Returns numpy views that stay valid
        until the next ``fetch`` with the same ``slot`` (one slot per sub-batch of ``run_concurrent``; ``slot=None`` =
        one slot per calling thread, for the workers of ``run_pipelined``)."""
        torch = _lib.require_cuda()
        if slot is None:
            slot = ("thread", threading.get_ident())
        if not hasattr(self, "_pinned"):
            self._pinned = {}
        res = {}
        for k in keys:
            t = out[k]
            buf = self._pinned.get((slot, k))
            if buf is None or buf.shape != t.shape or buf.dtype != t.dtype:
                buf = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
                self._pinned[(slot, k)] = buf
            buf.copy_(t, non_blocking=True)
            res[k] = buf
        torch.cuda.current_stream().synchronize()
        return {k: v.numpy() for k, v in res.items()}

    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _pack(meshes):
        """A list of PolyData-like meshes (``.points``, ``.tris``) -> host ``(points, tris, mesh_off_host)``, the meshes
        in list order, triangle vertex ids made global."""
        import torch

        sizes = [m.points.shape[0] for m in meshes]
        off = np.zeros(len(meshes) + 1, dtype=np.int32)
        off[1:] = np.cumsum(sizes)
        pts = torch.from_numpy(np.ascontiguousarray(np.concatenate([m.points for m in meshes])))
        tris = torch.from_numpy(np.ascontiguousarray(np.concatenate(
            [m.tris.astype(np.int64) + int(o) for m, o in zip(meshes, off[:-1])]).astype(np.int32)))
        return pts, tris, off

    @staticmethod
    def pack_meshes(targets, sources, target_of_pair=None):
        """Lists of PolyData-like meshes (``.points``, ``.tris``) -> ``(points, tris, mesh_off_host, n_pairs)`` of ``run``
        (host tensors; targets first, then sources; triangle vertex ids made global).  With ``target_of_pair`` (int [P],
        one entry per source) the targets are the T shared ones, pair p being ``targets[target_of_pair[p]]`` with
        ``sources[p]``; without it, pair p is ``targets[p]`` with ``sources[p]``."""
        if target_of_pair is None:
            if len(targets) != len(sources) or not targets:
                raise ValueError("need as many source meshes as target meshes (at least one pair)")
        else:
            shared_targets(target_of_pair, len(targets) + len(sources), len(sources))
        return SpectralBatch._pack(list(targets) + list(sources)) + (len(sources),)

    def _run_packed(self, meshes, pts, tris, off, n_pairs, kw):
        """``run`` on meshes packed by ``_pack``, with their point scalars (``list_features_to_get_from_mesh``) and
        triangle ranges filled in unless given."""
        if self.list_features_to_get_from_mesh and "node_features" not in kw:
            import torch

            kw["node_features"] = torch.from_numpy(np.ascontiguousarray(np.stack(
                [np.concatenate([mesh_point_scalars(m, name).reshape(-1) for m in meshes])
                 for name in self.list_features_to_get_from_mesh], axis=1)))
        tri_off = np.zeros(len(meshes) + 1, dtype=np.int32)
        tri_off[1:] = np.cumsum([m.tris.shape[0] for m in meshes])
        kw.setdefault("tri_off_host", tri_off)
        return self.run(pts, tris, off, n_pairs, **kw)

    def run_meshes(self, targets, sources, target_of_pair=None, **kw):
        """Convenience: lists of PolyData-like meshes (``.points``, ``.tris``); the point scalars named by
        ``list_features_to_get_from_mesh`` are read from the meshes (``Exception`` for a missing name, as graph.py).
        ``target_of_pair``: as in ``pack_meshes`` and ``run`` (many sources against shared targets)."""
        pts, tris, off, n_pairs = self.pack_meshes(targets, sources, target_of_pair)
        if target_of_pair is not None:
            kw["target_of_pair"] = target_of_pair
        return self._run_packed(list(targets) + list(sources), pts, tris, off, n_pairs, kw)

    def run_mesh_pairs(self, meshes, mesh_pairs, **kw):
        """Convenience for ``run(..., mesh_pairs=...)``: a list of M PolyData-like meshes, each packed once in list order,
        and ``mesh_pairs`` [P][2] of (target, source) indices into it (all-vs-all, one subject against several atlases,
        both directions of a pair...).  Point scalars and triangle ranges are filled in as by ``run_meshes``."""
        meshes = list(meshes)
        mp = mesh_pairs_checked(mesh_pairs, len(meshes))
        pts, tris, off = self._pack(meshes)
        return self._run_packed(meshes, pts, tris, off, mp.shape[0], dict(kw, mesh_pairs=mp))

    def build_shape_model(self, subjects, template, rounds=5, template_tolerance=1e-3, procrustes="similarity",
                          align_type="weighted", n_modes=10, **run_kw):
        """A statistical shape model of the cohort ``subjects`` (PolyData-like meshes, any sizes) on the vertices of
        ``template``.  Round k runs ``run_mesh_pairs(subjects + [template_k], [(m, P) for m in range(P)], **run_kw)`` with
        this object's settings (the subjects are the targets, the template the shared source), takes the P
        configurations [P][N_T][3] (every template vertex located on every subject) from
        ``weighted_avg_transformed_points`` (``align_type="weighted"``) or ``nearest_neighbor_transformed_points``
        (``"nearest"``), runs ``shape.procrustes`` on them (``procrustes``: "rigid" or "similarity") with template_k's
        points as the reference, and makes template_{k+1} = the GPA mean on the template's triangles.  Rounds stop when
        RMS(template_{k+1} - template_k) <= ``template_tolerance`` (in the units of the points) or after ``rounds``;
        ``shape.pca`` then runs on the last round's aligned configurations.

        Returns a dict: ``mean_points`` (N_T, 3) and ``mean_mesh`` (the last template_{k+1}); ``aligned`` (P, N_T, 3) and
        ``procrustes_matrices`` (P, 4, 4) of the last GPA; ``modes``, ``variances``, ``scores`` of ``shape.pca`` with
        ``n_modes``; ``rounds``, one dict per round with ``template_change``, ``gpa_iterations``, ``gpa_changes``,
        with ICP on ``icp_matrices`` and, with ``surface_distances`` set, ``surface_distance_stats`` ((P, 6) host numpy,
        row m for subject m: the template is the source).  ``ValueError`` before any device work for no subjects, a bad ``procrustes`` or
        ``align_type``, ``n_modes`` < 1, ``rounds`` < 1, or ``icp_register_first`` without ``icp_reg_target_to_source``
        (the shared template would be every pair's moving mesh).  A failed registration (an eigensolve, a zero-length
        edge in an averaged template) raises ``RuntimeError`` naming the round and the subjects or template."""
        from .shape import build_shape_model

        return build_shape_model(self, subjects, template, rounds=rounds, template_tolerance=template_tolerance,
                                 procrustes_mode=procrustes, align_type=align_type, n_modes=n_modes, **run_kw)
