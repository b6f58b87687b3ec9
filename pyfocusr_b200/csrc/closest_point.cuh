// Closest point on a triangle and the box bound that prunes a search for it, shared by the ICP closest-point search
// (K10, icp.cu) and the surface-distance search (K14, surface.cu), so both score a (point, triangle) pair alike.
// The numpy restatements are oracle/icp_port.py::closest_points_on_triangles and oracle/surface_port.py.
#pragma once
#include <cuda_runtime.h>

namespace fb {

struct P3 {
  double x, y, z;
};
__device__ __forceinline__ P3 p3(const double* __restrict__ p, long long i) { return P3{p[3 * i], p[3 * i + 1], p[3 * i + 2]}; }
__device__ __forceinline__ P3 operator-(P3 a, P3 b) { return P3{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ P3 operator+(P3 a, P3 b) { return P3{a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ P3 operator*(P3 a, double s) { return P3{a.x * s, a.y * s, a.z * s}; }
__device__ __forceinline__ double dot3(P3 a, P3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }

// closest point of segment (a, b) to p; a zero-length segment gives a
__device__ __forceinline__ P3 closest_on_segment(P3 p, P3 a, P3 b) {
  const P3 ab = b - a;
  const double l2 = dot3(ab, ab);
  if (l2 == 0.0) return a;
  const double t = fmin(fmax(dot3(p - a, ab) / l2, 0.0), 1.0);
  return a + ab * t;
}

// closest point of the edges ab, bc, ca to p, tried in that order; a tie keeps the earlier edge
__device__ __forceinline__ P3 closest_on_edges(P3 p, P3 a, P3 b, P3 c) {
  P3 best = closest_on_segment(p, a, b);
  P3 d = p - best;
  double bd = dot3(d, d);
  const P3 e1 = closest_on_segment(p, b, c);
  d = p - e1;
  const double d1 = dot3(d, d);
  if (d1 < bd) best = e1, bd = d1;
  const P3 e2 = closest_on_segment(p, c, a);
  d = p - e2;
  if (dot3(d, d) < bd) best = e2;
  return best;
}

// closest point of triangle (a, b, c) to p: Ericson, "Real-Time Collision Detection", 5.1.5.  With EDGES, a triangle
// whose region solve would divide by zero (va + vb + vc == 0 for the interior, a zero-length edge for an edge region:
// only a triangle collapsed to a segment or a point has one) is scored as the closest of its edges; without it the
// division is left as ICP has always done it.
template <bool EDGES>
__device__ __forceinline__ P3 closest_on_triangle_t(P3 p, P3 a, P3 b, P3 c) {
  const P3 ab = b - a, ac = c - a, ap = p - a;
  const double d1 = dot3(ab, ap), d2 = dot3(ac, ap);
  if (d1 <= 0.0 && d2 <= 0.0) return a;
  const P3 bp = p - b;
  const double d3 = dot3(ab, bp), d4 = dot3(ac, bp);
  if (d3 >= 0.0 && d4 <= d3) return b;
  const double vc = d1 * d4 - d3 * d2;
  if (vc <= 0.0 && d1 >= 0.0 && d3 <= 0.0) {
    if (!EDGES || d1 - d3 != 0.0) return a + ab * (d1 / (d1 - d3));
  } else {
    const P3 cp = p - c;
    const double d5 = dot3(ab, cp), d6 = dot3(ac, cp);
    if (d6 >= 0.0 && d5 <= d6) return c;
    const double vb = d5 * d2 - d1 * d6;
    if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) {
      if (!EDGES || d2 - d6 != 0.0) return a + ac * (d2 / (d2 - d6));
    } else {
      const double va = d3 * d6 - d5 * d4;
      if (va <= 0.0 && (d4 - d3) >= 0.0 && (d5 - d6) >= 0.0) {
        if (!EDGES || (d4 - d3) + (d5 - d6) != 0.0) return b + (c - b) * ((d4 - d3) / ((d4 - d3) + (d5 - d6)));
      } else if (!EDGES || va + vb + vc != 0.0) {
        const double denom = 1.0 / (va + vb + vc);
        return a + ab * (vb * denom) + ac * (vc * denom);
      }
    }
  }
  return closest_on_edges(p, a, b, c);  // reached only with EDGES, for a collapsed triangle
}

__device__ __forceinline__ P3 closest_on_triangle(P3 p, P3 a, P3 b, P3 c) { return closest_on_triangle_t<false>(p, a, b, c); }

// squared distance from q to an axis-aligned box, rounded down
__device__ __forceinline__ double box_lb(P3 q, const double* __restrict__ lo, const double* __restrict__ hi) {
  const double g0 = fmax(fmax(lo[0] - q.x, q.x - hi[0]), 0.0);
  const double g1 = fmax(fmax(lo[1] - q.y, q.y - hi[1]), 0.0);
  const double g2 = fmax(fmax(lo[2] - q.z, q.z - hi[2]), 0.0);
  return (g0 * g0 + g1 * g1 + g2 * g2) * (1.0 - 1e-12);
}

}  // namespace fb
