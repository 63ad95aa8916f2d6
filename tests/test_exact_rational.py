"""CPU: exact-rational cross-check of the oracle's footprint predicates (``oracle/geometry.py``).

shapely / GEOS cannot be installed here, so the oracle's float64 predicates DEFINE parity for the CUDA kernels.
This file checks them against brute-force set-theoretic definitions evaluated in exact rational arithmetic
(``fractions.Fraction`` on the very same float64 inputs) with ALGORITHMS THAT SHARE NOTHING with the oracle's:

  * rectangle meets closed convex polygon  <=>  a vertex of one lies in the other (closed) or two edges meet
    (the oracle uses separating axes);
  * rectangle inside a closed simple polygon  <=>  every piece of the rectangle's boundary, cut at all crossings
    with polygon edges, has its midpoint inside the closed polygon (the oracle tests corners + "no polygon edge
    meets the open rectangle");
  * rectangle inside a UNION of convex polygons  <=>  every boundary piece is inside some polygon AND no piece of a
    polygon's boundary inside the open rectangle is left uncovered by the other polygons, i.e. no hole of the union
    inside the rectangle (the oracle uses clip intervals + precomputed union-boundary vertices).

Poses are placed so that a footprint corner (or edge) sits within 1e-9 .. 1e-6 m of an obstacle edge, a field edge
or a lane-capsule boundary -- where a wrong strict/non-strict comparison or a missed case would show."""
import math

import numpy as np

import hl_helpers as H
from exact_geom import EXT, F, _edge_samples, _poses_near, x_rect_hits_convex, x_rect_in_polygon, x_rect_in_union
from oracle import geometry as geo
from oracle import planner as OP


def test_rect_vs_convex_obstacles_exact():
    rng = np.random.default_rng(1)
    rows = H.canonical_rows(l_std=0.5)
    env = OP.OrchardGeometryEnvironment(rows, [(-3.0, 6.0)], tree_width=0.3, headland_width=6.0)
    quads = [geo.ccw(q) for q in env.obs_poly_list]
    n_checked = 0
    for q in quads[:4] + quads[-1:]:
        pts, nrm = _edge_samples(rng, q)
        poses = _poses_near(rng, pts, nrm, 60)
        corners = geo.rect_corners(poses, EXT)
        got = geo.rects_hit_convex(poses, EXT, q, corners)
        for p in range(len(poses)):
            assert got[p] == x_rect_hits_convex(F(corners[p]), F(q)), (poses[p], q)
            n_checked += 1
        assert 0.1 < got.mean() < 0.9
    assert n_checked == 300


def test_rect_in_field_polygon_exact():
    rng = np.random.default_rng(2)
    for l_std in (0.0, 1.0):
        rows = H.canonical_rows(l_std=l_std)
        env = OP.OrchardGeometryEnvironment(rows, [], tree_width=0.3, headland_width=6.0)
        poly = geo.ccw(env.field_poly)
        pts, nrm = _edge_samples(rng, poly)
        poses = _poses_near(rng, pts, nrm, 150)
        corners = geo.rect_corners(poses, EXT)
        got = geo.rects_inside_polygon(poses, EXT, poly, corners)
        fp = F(poly)
        for p in range(len(poses)):
            assert got[p] == x_rect_in_polygon(F(corners[p]), fp), (l_std, poses[p])
        assert 0.05 < got.mean() < 0.95


def test_rect_in_lane_union_exact():
    rng = np.random.default_rng(3)
    way = np.array([[0.0, 3.75], [-4.5, 5.0], [-4.06, 7.5], [-3.62, 10.0], [-1.5, 11.0]])
    lane = geo.Lane(way)
    polys = [F(p) for p in lane.polys]
    # boundary samples of the UNION: capsule boundary points that are not strictly inside another capsule
    pts, nrm = [], []
    for i, P in enumerate(lane.polys):
        bp, bn = _edge_samples(rng, P, per_edge=1)
        for q, n in zip(bp, bn):
            if not any(lane.points_in(k, np.array([q[0]]), np.array([q[1]]), strict=True)[0] for k in range(len(lane.polys)) if k != i):
                pts.append(q); nrm.append(n)
    poses = _poses_near(rng, np.array(pts), np.array(nrm), 70)
    # plus footprints straddling the junctions between capsules (the union, not a single capsule, contains them)
    extra = np.stack([rng.uniform(-6, -2, 40), rng.uniform(4, 10.5, 40), rng.uniform(-math.pi, math.pi, 40)], axis=1)
    poses = np.concatenate([poses, extra])
    corners = geo.rect_corners(poses, EXT)
    got = lane.rects_inside(poses, EXT, corners)
    for p in range(len(poses)):
        assert got[p] == x_rect_in_union(F(corners[p]), polys), poses[p]
    assert 0.1 < got.mean() < 0.95


def test_capsule_polygon_is_the_published_buffer_shape():
    """GEOS OffsetSegmentGenerator, quad_segs = 16: 66 vertices, the two offset segments exact, every fillet vertex ON the
    radius-6 circle about its end point at multiples of pi/32 from the segment normal, polygon inside the true capsule
    and containing the inscribed radius 6 cos(pi/64)."""
    rng = np.random.default_rng(4)
    for _ in range(20):
        p0, p1 = rng.uniform(-10, 10, 2), rng.uniform(-10, 10, 2)
        P = geo.capsule_polygon(p0, p1)
        assert P.shape == (66, 2)
        d = p1 - p0
        ang = math.atan2(d[1], d[0])
        r0 = np.hypot(*(P - p0).T)
        r1 = np.hypot(*(P - p1).T)
        on = np.minimum(np.abs(r0 - 6.0), np.abs(r1 - 6.0))
        assert on.max() < 1e-12                                  # every vertex on one of the two circles
        near1 = np.abs(r1 - 6.0) < 1e-12
        a1 = np.arctan2(*(P[near1] - p1).T[::-1]) - ang
        k = (a1 / (math.pi / 32))
        assert np.abs(k - np.round(k)).max() < 1e-9
        dist = geo.Lane(np.array([p0, p1]))._seg_dist(0, P[:, 0], P[:, 1])
        assert dist.max() <= 6.0 + 1e-12
        mids = 0.5 * (P + np.roll(P, -1, axis=0))
        dm = geo.Lane(np.array([p0, p1]))._seg_dist(0, mids[:, 0], mids[:, 1])
        assert dm.min() >= geo.LANE_INSCRIBED - 1e-12
