"""Surface distances on the device: how far every vertex of a registered mesh lies from the surface it was registered
onto, and the reverse, per pair summarised as means, the average symmetric surface distance (ASSD) and the Hausdorff
distance.

The closest point of a query on a triangle surface is the exact one of a scan over all the surface's triangles (the
lowest triangle index wins a tie), found by the tile-pruned search of ``csrc/surface.cu`` (K14), which ICP's search
(K10) generalises to whole meshes of queries.  ``SpectralBatch(surface_distances="weighted" | "nearest")`` adds these
measures to every pair of a batch; :func:`surface_distances` computes them for lists of meshes, for instance one
``Focusr`` result: ``surface_distances([reg.get_source_mesh_transformed_weighted_avg()], [target])``.
"""
from __future__ import annotations

import numpy as np

from . import _lib

__all__ = ["closest_points", "distance_stats", "surface_distances"]

STATS_COLUMNS = ("mean_source_to_target", "max_source_to_target", "mean_target_to_source", "max_target_to_source",
                 "assd", "hausdorff")


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32).reshape(-1)


def closest_points(surf_points, tris, surf_point_off, surf_tri_off, queries, query_off, surf_of_segment,
                   want_closest=True, brute_force=False):
    """``focusr_closest_points``: query segment s (rows ``query_off[s] .. [s+1]`` of ``queries``) against surface
    ``surf_of_segment[s]`` (points ``surf_point_off[m] .. [m+1]`` of ``surf_points``, triangles ``surf_tri_off[m] ..
    [m+1]`` of ``tris``, whose vertex ids are global rows of ``surf_points``).  ``surf_points`` / ``queries`` are
    contiguous float64 device tensors [..][3], ``tris`` a contiguous int32 device tensor [..][3]; the offsets and the map
    are host integer arrays.  Triangle ids must lie in range (not checked here).

    Returns device tensors indexed like ``queries``: ``(closest [n][3] float64 or None without want_closest, tri [n]
    int64 local to the surface's triangle range, dist [n] float64)``.  ``brute_force=True`` scans every triangle in index
    order (the bit-identical on-device reference of the pruned search)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = queries.device
    poff, toff, qoff, seg = _i32(surf_point_off), _i32(surf_tri_off), _i32(query_off), _i32(surf_of_segment)
    n_surf, n_seg = poff.size - 1, qoff.size - 1
    if toff.size != poff.size or seg.size != n_seg:
        raise ValueError("closest_points: surf_tri_off needs %d entries and surf_of_segment one per segment (%d), got %d "
                         "and %d" % (poff.size, n_seg, toff.size, seg.size))
    n = int(queries.shape[0])
    closest = torch.empty((n, 3), dtype=torch.float64, device=dev) if want_closest else None
    tri = torch.empty(n, dtype=torch.int32, device=dev)
    dist = torch.empty(n, dtype=torch.float64, device=dev)
    ws, ws_bytes = None, 0
    if not brute_force:
        ws_bytes = int(lib.focusr_closest_points_workspace_bytes(_lib.ptr(poff), _lib.ptr(toff), n_surf, _lib.ptr(qoff),
                                                                 n_seg, _lib.ptr(seg)))
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
    poff_d, toff_d, qoff_d, seg_d = (torch.from_numpy(a).to(dev, non_blocking=True) for a in (poff, toff, qoff, seg))
    _lib.call("focusr_closest_points", _lib.ptr(surf_points), _lib.ptr(tris), _lib.ptr(poff_d), _lib.ptr(toff_d),
              _lib.ptr(poff), _lib.ptr(toff), n_surf, _lib.ptr(queries), _lib.ptr(qoff_d), _lib.ptr(qoff), n_seg,
              _lib.ptr(seg_d), _lib.ptr(seg), _lib.ptr(closest), _lib.ptr(tri), _lib.ptr(dist), _lib.ptr(ws), ws_bytes,
              _lib.stream_ptr())
    return closest, tri.to(torch.int64), dist


def distance_stats(a_dist, a_off, b_dist, b_off):
    """``focusr_surface_distance_stats``: per pair p, from the distances ``a_dist[a_off[p] .. [p+1]]`` (a -> b) and
    ``b_dist[b_off[p] .. [p+1]]`` (b -> a), a (P, 6) float64 device tensor of the columns ``STATS_COLUMNS``: mean and max
    a -> b, mean and max b -> a, ASSD = (sum a -> b + sum b -> a) / (n_a + n_b), Hausdorff = the larger maximum."""
    torch = _lib.require_cuda()
    ao, bo = _i32(a_off), _i32(b_off)
    if ao.size != bo.size or ao.size < 2:
        raise ValueError("distance_stats: a_off and b_off need the same number (>= 2) of entries")
    dev = a_dist.device
    out = torch.empty((ao.size - 1, 6), dtype=torch.float64, device=dev)
    ao_d, bo_d = (torch.from_numpy(a).to(dev, non_blocking=True) for a in (ao, bo))
    _lib.call("focusr_surface_distance_stats", _lib.ptr(a_dist), _lib.ptr(ao_d), _lib.ptr(b_dist), _lib.ptr(bo_d),
              int(ao.size - 1), _lib.ptr(out), _lib.stream_ptr())
    return out


def check_triangles(meshes, what):
    """``ValueError`` unless every mesh of ``meshes`` has triangles [F][3], F >= 1, with vertex ids in [0, its points)."""
    for i, m in enumerate(meshes):
        t = np.asarray(m.tris)
        n = int(np.asarray(m.points).shape[0])
        if t.ndim != 2 or t.shape[1] != 3 or t.shape[0] == 0:
            raise ValueError("%s[%d] needs triangles [F][3] with F >= 1, got shape %s" % (what, i, t.shape))
        lo, hi = int(t.min()), int(t.max())
        if lo < 0 or hi >= n:
            raise ValueError("%s[%d] has triangle vertex id %d outside [0, %d)" % (what, i, lo if lo < 0 else hi, n))


def surface_distances(sources, targets):
    """Surface distances of the pairs (``sources[p]``, ``targets[p]``) of two equal-length lists of PolyData-like meshes
    (``.points``, ``.tris``), e.g. registered sources and their targets.

    Returns a dict of device tensors: ``source_to_target_surface_dist`` [source vertices of all pairs] (each source vertex
    to its target's surface), ``source_to_target_closest_points`` [..][3] and ``source_to_target_closest_tri`` [..] int64
    (local to the target mesh), ``target_to_source_surface_dist`` [target vertices of all pairs] and
    ``target_to_source_closest_tri`` (local to the source mesh), ``surface_distance_stats`` (P, 6) (``STATS_COLUMNS``,
    source = a, target = b), and the host row offsets ``source_off`` / ``target_off`` [P + 1] of each pair's vertices.
    ``ValueError`` for lists of different lengths or no pair, and for a mesh without triangles or with a triangle vertex
    id outside its points."""
    from .batch import SpectralBatch

    sources, targets = list(sources), list(targets)
    if len(sources) != len(targets) or not sources:
        raise ValueError("surface_distances needs as many targets as sources (at least one pair), got %d and %d" % (
            len(sources), len(targets)))
    check_triangles(sources, "sources")
    check_triangles(targets, "targets")
    torch = _lib.require_cuda()
    P = len(sources)
    pts, tris, off = SpectralBatch._pack(sources + targets)  # meshes 0..P-1 the sources, P..2P-1 the targets
    tri_off = np.zeros(2 * P + 1, dtype=np.int32)
    tri_off[1:] = np.cumsum([m.tris.shape[0] for m in sources + targets])
    dev = torch.device("cuda", torch.cuda.current_device())
    pts = pts.to(dev, non_blocking=True).contiguous()
    tris = tris.to(dev, non_blocking=True).contiguous()
    ns = int(off[P])
    src_off, tgt_off = off[:P + 1].copy(), (off[P:] - ns).astype(np.int32)
    closest, s_tri, s_dist = closest_points(pts, tris, off, tri_off, pts[:ns], src_off, np.arange(P, 2 * P))
    _, t_tri, t_dist = closest_points(pts, tris, off, tri_off, pts[ns:], tgt_off, np.arange(P), want_closest=False)
    return dict(source_to_target_surface_dist=s_dist, source_to_target_closest_points=closest,
                source_to_target_closest_tri=s_tri, target_to_source_surface_dist=t_dist,
                target_to_source_closest_tri=t_tri, surface_distance_stats=distance_stats(s_dist, src_off, t_dist, tgt_off),
                source_off=src_off, target_off=tgt_off)
