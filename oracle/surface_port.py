"""Closest points on a triangle surface by brute force in numpy: the reference the K14 search (csrc/surface.cu) is
tested against.  Test infrastructure only.

A triangle is scored by Ericson's region test (``icp_port.closest_points_on_triangles``); one whose region solve divides
by zero -- it has collapsed to a segment or a point, and the test returns a non-finite point -- is scored as the
closest of its edges ab, bc, ca instead, a tie keeping the earlier edge and a zero-length edge scoring as its end
point.  The winner of a query is the lowest-index triangle of least squared distance.
"""
from __future__ import annotations

import numpy as np

from oracle.icp_port import closest_points_on_triangles


def closest_points_on_segments(p, a, b):
    """Closest point of segment (a, b) to p, broadcasting; a zero-length segment gives a.  Returns (point, dist2)."""
    ab = b - a
    l2 = np.sum(ab * ab, -1)
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.clip(np.sum((p - a) * ab, -1) / l2, 0.0, 1.0)
    t = np.where(l2 == 0.0, 0.0, t)
    out = a + t[..., None] * ab
    d = p - out
    return out, np.sum(d * d, -1)


def closest_points_on_triangles_or_edges(p, a, b, c):
    """``closest_points_on_triangles`` with the edge rule for collapsed triangles; returns (point, dist2)."""
    with np.errstate(invalid="ignore", over="ignore"):
        out, d2 = closest_points_on_triangles(p, a, b, c)
    bad = ~np.all(np.isfinite(out), axis=-1)
    if np.any(bad):
        best, bd = closest_points_on_segments(p, a, b)
        for u, v in ((b, c), (c, a)):
            e, ed = closest_points_on_segments(p, u, v)
            take = ed < bd
            best, bd = np.where(take[..., None], e, best), np.where(take, ed, bd)
        out = np.where(bad[..., None], best, out)
        d2 = np.where(bad, bd, d2)
    return out, d2


def closest_points(queries, points, tris, chunk=64):
    """Every query against every triangle of one surface (``tris`` local vertex ids into ``points``).  Returns
    (closest point [n][3], d2 [n], winning triangle [n] (the lowest index on ties), second-best d2 [n] (inf for a
    one-triangle surface))."""
    queries = np.asarray(queries, dtype=np.float64).reshape(-1, 3)
    a, b, c = (np.asarray(points, dtype=np.float64)[np.asarray(tris)[:, k]] for k in range(3))
    n = queries.shape[0]
    cl, d2, win, second = np.empty((n, 3)), np.empty(n), np.empty(n, dtype=np.int64), np.empty(n)
    for s in range(0, n, chunk):
        q = queries[s:s + chunk, None, :]
        cp, dd = closest_points_on_triangles_or_edges(q, a[None], b[None], c[None])
        best = np.argmin(dd, axis=1)  # first minimum = lowest triangle index
        rows = np.arange(cp.shape[0])
        cl[s:s + chunk], d2[s:s + chunk], win[s:s + chunk] = cp[rows, best], dd[rows, best], best
        if dd.shape[1] > 1:
            second[s:s + chunk] = np.partition(dd, 1, axis=1)[:, 1]
        else:
            second[s:s + chunk] = np.inf
    return cl, d2, win, second
