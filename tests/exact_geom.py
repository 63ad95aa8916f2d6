"""Exact-rational footprint predicates and boundary-hugging pose generators shared by the footprint tests.

Every predicate works on ``fractions.Fraction`` points made from the very same float64 inputs the float code sees
(``F``), so its answer is the set-theoretic truth for those inputs, with no rounding anywhere:

  * rectangle meets closed convex polygon  <=>  a vertex of one lies in the other (closed) or two edges meet;
  * rectangle inside a closed simple polygon  <=>  every piece of the rectangle's boundary, cut at all crossings
    with polygon edges, has its midpoint inside the closed polygon;
  * rectangle inside a UNION of convex polygons  <=>  every boundary piece is inside some polygon AND no piece of a
    polygon's boundary inside the open rectangle is left uncovered by the other polygons, i.e. no hole of the union
    inside the rectangle."""
import math
from fractions import Fraction as Fr

import numpy as np

from oracle import geometry as geo


# ------------------------------------------------------------------ exact primitives
def F(a):
    return [(Fr(float(x)), Fr(float(y))) for x, y in np.asarray(a, dtype=np.float64).reshape(-1, 2)]


def orient(a, b, c):
    return (b[0] - a[0]) * (c[1] - a[1]) - (b[1] - a[1]) * (c[0] - a[0])


def on_segment(a, b, p):
    return min(a[0], b[0]) <= p[0] <= max(a[0], b[0]) and min(a[1], b[1]) <= p[1] <= max(a[1], b[1]) and orient(a, b, p) == 0


def in_closed_polygon(p, poly):
    """winding number by exact crossing count; boundary counts as inside"""
    inside = False
    n = len(poly)
    for i in range(n):
        a, b = poly[i], poly[(i + 1) % n]
        if on_segment(a, b, p):
            return True
        if (a[1] > p[1]) != (b[1] > p[1]):
            xint = a[0] + (b[0] - a[0]) * (p[1] - a[1]) / (b[1] - a[1])
            if p[0] < xint:
                inside = not inside
    return inside


def in_open_convex(p, poly_ccw):
    return all(orient(poly_ccw[i], poly_ccw[(i + 1) % len(poly_ccw)], p) > 0 for i in range(len(poly_ccw)))


def in_closed_convex(p, poly_ccw):
    return all(orient(poly_ccw[i], poly_ccw[(i + 1) % len(poly_ccw)], p) >= 0 for i in range(len(poly_ccw)))


def boxes_apart(a, b, c, d):
    """the closed bounding boxes of segments a-b and c-d are disjoint (then the segments share no point)"""
    return (max(a[0], b[0]) < min(c[0], d[0]) or max(c[0], d[0]) < min(a[0], b[0]) or
            max(a[1], b[1]) < min(c[1], d[1]) or max(c[1], d[1]) < min(a[1], b[1]))


def segs_meet(a, b, c, d):
    """closed segments share a point"""
    if boxes_apart(a, b, c, d):
        return False
    o1, o2, o3, o4 = orient(a, b, c), orient(a, b, d), orient(c, d, a), orient(c, d, b)
    if ((o1 > 0) != (o2 > 0)) and o1 != 0 and o2 != 0 and ((o3 > 0) != (o4 > 0)) and o3 != 0 and o4 != 0:
        return True
    return on_segment(a, b, c) or on_segment(a, b, d) or on_segment(c, d, a) or on_segment(c, d, b)


def seg_params_with(a, b, c, d):
    """parameters t in [0, 1] on a->b where the closed segment c->d touches it (finite list)"""
    if boxes_apart(a, b, c, d):
        return []
    r = (b[0] - a[0], b[1] - a[1])
    s = (d[0] - c[0], d[1] - c[1])
    den = r[0] * s[1] - r[1] * s[0]
    qp = (c[0] - a[0], c[1] - a[1])
    out = []
    if den != 0:
        t = (qp[0] * s[1] - qp[1] * s[0]) / den
        u = (qp[0] * r[1] - qp[1] * r[0]) / den
        if 0 <= t <= 1 and 0 <= u <= 1:
            out.append(t)
    else:                                             # parallel: endpoints of c-d that lie on a-b
        rr = r[0] * r[0] + r[1] * r[1]
        for p in (c, d):
            if orient(a, b, p) == 0:
                t = ((p[0] - a[0]) * r[0] + (p[1] - a[1]) * r[1]) / rr
                if 0 <= t <= 1:
                    out.append(t)
    return out


def pieces_midpoints(a, b, edges):
    ts = {Fr(0), Fr(1)}
    for c, d in edges:
        ts.update(seg_params_with(a, b, c, d))
    ts = sorted(ts)
    return [(a[0] + (b[0] - a[0]) * (t0 + t1) / 2, a[1] + (b[1] - a[1]) * (t0 + t1) / 2) for t0, t1 in zip(ts[:-1], ts[1:])]


def ring_edges(poly):
    return [(poly[i], poly[(i + 1) % len(poly)]) for i in range(len(poly))]


# ------------------------------------------------------------------ exact definitions
def x_rect_hits_convex(rect, poly_ccw):
    if any(in_closed_convex(p, poly_ccw) for p in rect) or any(in_closed_convex(p, rect) for p in poly_ccw):
        return True
    return any(segs_meet(a, b, c, d) for a, b in ring_edges(rect) for c, d in ring_edges(poly_ccw))


def x_rect_in_polygon(rect, poly):
    pe = ring_edges(poly)
    for a, b in ring_edges(rect):
        if not all(in_closed_polygon(m, poly) for m in pieces_midpoints(a, b, pe)):
            return False
    return True                                       # simple polygon: boundary inside => region inside


def x_rect_in_union(rect, polys_ccw):
    all_edges = [e for P in polys_ccw for e in ring_edges(P)]
    for a, b in ring_edges(rect):                     # the rectangle's boundary is covered
        for m in pieces_midpoints(a, b, all_edges):
            if not any(in_closed_convex(m, P) for P in polys_ccw):
                return False
    redges = ring_edges(rect)                         # no hole of the union inside the rectangle
    rbox = (rect[0], rect[0])
    for p in rect:
        rbox = ((min(rbox[0][0], p[0]), min(rbox[0][1], p[1])), (max(rbox[1][0], p[0]), max(rbox[1][1], p[1])))
    for i, P in enumerate(polys_ccw):
        others = [e for j, Q in enumerate(polys_ccw) if j != i for e in ring_edges(Q)]
        for a, b in ring_edges(P):
            if boxes_apart(a, b, *rbox):              # no piece of this edge lies in the open rectangle
                continue
            for m in pieces_midpoints(a, b, redges + others):
                if in_open_convex(m, rect) and not any(in_open_convex(m, Q) or
                                                       any(on_segment(c, d, m) for c, d in ring_edges(Q))
                                                       for j, Q in enumerate(polys_ccw) if j != i):
                    return False
    return True


# ------------------------------------------------------------------ pose generators
EXT = geo.body_extent(0.55, 3.0, 1.48)
DELTAS = (1e-9, -1e-9, 1e-7, -1e-7, 1e-6, -1e-6, 3e-4, -3e-4)


def _poses_near(rng, boundary_pts, normals, n, deltas=DELTAS, ext=EXT, with_deltas=False):
    """poses whose k-th footprint corner (of the local rectangle ``ext``) lies at boundary point + delta * normal;
    ``with_deltas`` also returns the delta of every pose"""
    lx = np.array([ext[0], ext[0], ext[1], ext[1]])
    ly = np.array([ext[3], ext[2], ext[2], ext[3]])
    out, ds = [], []
    for _ in range(n):
        j = rng.integers(len(boundary_pts))
        k = rng.integers(4)
        yaw = rng.uniform(-math.pi, math.pi)
        d = deltas[rng.integers(len(deltas))]
        q = boundary_pts[j] + d * normals[j]
        c, s = math.cos(yaw), math.sin(yaw)
        out.append([q[0] - (c * lx[k] - s * ly[k]), q[1] - (s * lx[k] + c * ly[k]), yaw])
        ds.append(d)
    return (np.array(out), np.array(ds)) if with_deltas else np.array(out)


def _edge_samples(rng, poly, per_edge=3):
    pts, nrm = [], []
    for a, b in zip(poly, np.roll(poly, -1, axis=0)):
        e = b - a
        n = np.array([e[1], -e[0]]) / np.hypot(*e)
        for t in list(rng.uniform(0.02, 0.98, per_edge)) + [0.0]:
            pts.append(a + t * e)
            nrm.append(n)
    return np.array(pts), np.array(nrm)
