"""Footprint checks at the boundary: K1 (hl_collision_check) and K7 (hl_grid_footprint_check) on poses whose corner
sits 1e-12 .. 1e-3 m from an edge, against the CPU oracle and against exact rational arithmetic (``exact_geom``).

K1: the float32 filter decides a pose outright only outside its error band (``D.eps``, about 1e-4 m on the canonical
field) and hands the rest to the float64 predicates, queued per CTA.  The deltas below bracket that band from both
sides, so both verdict paths and the float64 queue (including its overflow) see real geometry.  Three environments
reach code that the canonical scene does not: non-rectangular obstacle quads (the generic-quad branch, and the per-pose
path because ``all_rect`` is 0), a 40-vertex field (more than 32 field edges: the ``overflow`` bit and the per-pose
path) and the canonical scene in UTM-sized coordinates (the float32 frame is relative to the environment's origin).

K7: a pose hits iff its closed float64 rectangle meets the closed square [fl(i*res), fl((i+1)*res)] x
[fl(j*res), fl((j+1)*res)] of an occupied cell.  Exact ties are placed at yaw 0 only (cos 0 = 1 and sin 0 = 0 on both
sides); general headings keep 1e-9 m or more from a tie, since CUDA's cos / sin may differ from numpy's in the last
bit."""
import math

import numpy as np
import pytest

import hl_helpers as H
from exact_geom import F, _edge_samples, _poses_near, x_rect_hits_convex, x_rect_in_polygon, x_rect_in_union
from oracle import geometry as geo

pytestmark = pytest.mark.gpu

WAY = np.array([[0.0, 3.75], [-4.5, 5.0], [-4.06, 7.5], [-3.62, 10.0], [-1.5, 11.0]])
GOAL = np.array([-1.5, 11.0, 0.3])
OBSTACLES = [(-3.0, 6.0), (24.0, 11.0)]
SHIFT = np.array([431250.0, 5291730.0])          # UTM-sized easting / northing: one ulp is 9.3e-10 m
MAGS = (1e-12, 1e-9, 1e-7, 1e-6, 1e-5, 5e-5, 1e-4, 2e-4, 5e-4, 1e-3)
N_SMALL, N_LARGE = 2560, 1536                    # per set: |delta| <= 1e-5 first (2.5 tiles of 1024 poses), then the rest
N_TRUTH = 1500                                   # per set: poses checked in exact arithmetic


def _signed(mags):
    return tuple(s * m for m in mags for s in (1.0, -1.0))


# ------------------------------------------------------------------ K1 scenes
def _scene(kind):
    """(oracle env, oracle car, oracle heuristic, EnvRecord, smallest |delta|).  All scenes carry the sprayer's three
    implement rectangles and the canonical lane."""
    from headland_trajectory_planning_b200.env_batch import EnvRecord, make_record
    sh = SHIFT if kind == "utm" else np.zeros(2)
    rows = H.canonical_rows(l_std=0.5) + sh
    (o_env, o_car, o_h), (g_env, g_car, g_h) = H.make_pair(
        rows, obstacles=[tuple(np.array(p) + sh) for p in OBSTACLES], axle_to_front=2.85, aux=H.SPRAYER_AUX,
        waypoints=WAY + sh, goal=GOAL + np.r_[sh, 0.0])
    rec = make_record(g_env, g_car, g_h)
    quads, field = [np.asarray(q) for q in o_env.obs_poly_list], np.asarray(o_env.field_poly)
    if kind == "quads":
        # a trapezoid in the headland and a kite next to the row ends: convex, counter-clockwise, not rectangles
        quads = [np.array([[-4.2, 7.1], [-2.6, 7.1], [-2.9, 8.05], [-3.85, 8.05]]),
                 np.array([[-1.3, 12.3], [-0.55, 12.9], [-1.3, 14.6], [-2.05, 12.9]])] + quads
    elif kind == "field40":
        # the canonical ring, every edge cut into pieces whose inner vertices are pushed out by up to 2 cm
        rng = np.random.default_rng(40)
        ring = []
        for a, b in zip(field, np.roll(field, -1, axis=0)):
            e = b - a
            nrm = np.array([e[1], -e[0]]) / np.hypot(*e) * _outward_sign(field)
            k = 3 if np.hypot(*e) > 3.0 else 2
            ring.append(a)
            for t in np.arange(1, k) / k:
                ring.append(a + t * e + rng.uniform(0.0, 0.02) * nrm)
        field = np.array(ring)
        assert 36 <= len(field) <= 48
    if kind in ("quads", "field40"):
        o_env.obs_poly_list = quads
        o_env.field_poly = field
        rec = EnvRecord(np.array(quads), field, rec.body_ext, rec.aux, seg_xy=rec.seg_xy, seg_polys=rec.seg_polys,
                        seg_len=rec.seg_len, crit_xy=rec.crit, guide=rec.guide,
                        default_search_length=rec.default_search_length)
    assert np.array_equal(rec.obs, np.array(o_env.obs_poly_list)) and np.array_equal(rec.field, o_env.field_poly)
    return o_env, o_car, o_h, rec, (1e-6 if kind == "utm" else 1e-12)


def _outward_sign(poly):
    """+1 when the (e_y, -e_x) normals of the ring point outwards (counter-clockwise ring), else -1"""
    area2 = np.sum(poly[:, 0] * np.roll(poly[:, 1], -1) - np.roll(poly[:, 0], -1) * poly[:, 1])
    return 1.0 if area2 > 0 else -1.0


def _samples(rng, poly, per_edge):
    """_edge_samples, with the normal at each vertex sample (t = 0) replaced by the bisector of the normals of its two
    edges.  Moved along one edge's normal, a corner at a vertex would stay ON the line of the other edge at every
    delta (exactly so at a right angle), a tie whose verdict rests on the last bit of cos / sin."""
    pts, nrm = _edge_samples(rng, poly, per_edge)
    v = np.arange(per_edge, len(nrm), per_edge + 1)                    # the vertex sample of every edge
    b = nrm[v] + np.roll(nrm[v], 1, axis=0)                            # this edge's normal + the previous edge's
    nrm[v] = b / np.hypot(b[:, 0], b[:, 1])[:, None]
    return pts, nrm


def _lane_boundary(rng, lane):
    """boundary samples of the lane UNION: capsule boundary points not strictly inside another capsule"""
    pts, nrm = [], []
    for i, P in enumerate(lane.polys):
        bp, bn = _samples(rng, P, per_edge=1)
        for q, n in zip(bp, bn):
            if not any(lane.points_in(k, np.array([q[0]]), np.array([q[1]]), strict=True)[0]
                       for k in range(len(lane.polys)) if k != i):
                pts.append(q); nrm.append(n)
    return np.array(pts), np.array(nrm)


def _boundary(rng, kind, o_env, o_h):
    """boundary points and unit normals pointing to the FREE side: out of an obstacle, into the field or the lane"""
    if kind == "obstacles":
        parts = [_samples(rng, geo.ccw(q), 3) for q in o_env.obs_poly_list]
        return np.concatenate([p for p, _ in parts]), np.concatenate([n for _, n in parts])
    if kind == "field":
        pts, nrm = _samples(rng, np.asarray(o_env.field_poly), 3)        # t = 0: the vertices
        return pts, -nrm * _outward_sign(np.asarray(o_env.field_poly))
    pts, nrm = _lane_boundary(rng, o_h.lane)
    return pts, -nrm


FAR = 3e-3          # a candidate is kept when its rectangle is free with the corner moved this far to the free side


def _near_free(rng, pts, nrm, n, deltas, ext, is_bad):
    """n poses from _poses_near whose rectangle only touches the boundary near the placed corner: the same pose with
    the corner moved FAR to the free side is free (``is_bad`` says it is not).  Both signs of a delta then decide the
    verdict, and a small |delta| lies inside the float32 band."""
    out, ds = [], []
    while sum(map(len, out)) < n:
        state = rng.bit_generator.state
        p, d = _poses_near(rng, pts, nrm, n, deltas=deltas, ext=ext, with_deltas=True)
        twin = np.random.default_rng()
        twin.bit_generator.state = state                                   # the same draws, corner moved to FAR
        far = _poses_near(twin, pts, nrm, n, deltas=(FAR,) * len(deltas), ext=ext)
        keep = ~is_bad(far)
        out.append(p[keep]); ds.append(d[keep])
    return np.concatenate(out)[:n], np.concatenate(ds)[:n]


def _make_set(rng, kind, o_env, o_car, o_h, min_mag):
    """N_SMALL poses with |delta| <= 1e-5, then N_LARGE with |delta| > 1e-5.  kind "aux": the corner of an implement
    rectangle at the even indices (against obstacle and field edges), a body corner at the odd ones."""
    mags = [m for m in MAGS if m >= min_mag]
    small, large = _signed([m for m in mags if m <= 1e-5]), _signed([m for m in mags if m > 1e-5])
    body = o_car.body_ext
    if kind != "aux":
        pts, nrm = _boundary(rng, kind, o_env, o_h)
        is_bad = {"obstacles": lambda q: o_env.pose_flags(o_car, q, boundary_check=False),
                  "field": lambda q: ~geo.rects_inside_polygon(q, body, o_env.field_poly),
                  "lane": lambda q: o_h.pose_flags(o_car, q)}[kind]
        blocks = [_near_free(rng, pts, nrm, n, d, body, is_bad) for n, d in ((N_SMALL, small), (N_LARGE, large))]
        return np.concatenate([b[0] for b in blocks]), np.concatenate([b[1] for b in blocks])
    po, no = _boundary(rng, "obstacles", o_env, o_h)
    pf, nf = _boundary(rng, "field", o_env, o_h)
    pts, nrm = np.concatenate([po, pf]), np.concatenate([no, nf])
    body_bad = lambda q: o_env._part_flags(q, body, True)
    out, ds = [], []
    for n, d in ((N_SMALL, small), (N_LARGE, large)):
        poses, dd = np.zeros((n, 3)), np.zeros(n)
        for a, ext in enumerate(o_car.aux_exts):
            sel = np.arange(0, n, 2)[a::len(o_car.aux_exts)]
            poses[sel], dd[sel] = _near_free(rng, pts, nrm, len(sel), d, ext,
                                             lambda q, ext=ext: o_env._part_flags(q, ext, True) | body_bad(q))
        poses[1::2], dd[1::2] = _near_free(rng, pts, nrm, n // 2, d, body, body_bad)
        out.append(poses); ds.append(dd)
    return np.concatenate(out), np.concatenate(ds)


def _oracle_flags(o_env, o_car, o_h, poses, flags):
    bad = np.zeros(len(poses), dtype=bool)
    if flags & 1:
        bad |= o_env.pose_flags(o_car, poses, boundary_check=bool(flags & 2), aux_check=bool(flags & 4))
    if flags & 8:
        bad |= o_h.pose_flags(o_car, poses)
    return bad


def _apart(cor, poly):
    """the float bounding boxes are disjoint (compared exactly): the closed shapes share no point"""
    return (cor[:, 0].max() < poly[:, 0].min() or poly[:, 0].max() < cor[:, 0].min() or
            cor[:, 1].max() < poly[:, 1].min() or poly[:, 1].max() < cor[:, 1].min())


def _exact_parts(job):
    """exact (obstacle hit, outside the field, outside the lane) for rectangles given by their float corners; runs in
    a worker process"""
    cors, quads, field, lane_polys = job
    fq, ff, fl = [F(q) for q in quads], F(field), [F(P) for P in lane_polys]
    out = []
    for cor in cors:
        r = F(cor)
        hit = any(x_rect_hits_convex(r, q) for q, Q in zip(fq, quads) if not _apart(cor, Q))
        out_f = not x_rect_in_polygon(r, ff)
        near = [P for P, Q in zip(fl, lane_polys) if not _apart(cor, Q)]
        out.append((hit, out_f, not (near and x_rect_in_union(r, near))))
    return out


@pytest.fixture(scope="module")
def exact_pool():
    """worker processes for the exact checks (spawned: they never touch CUDA)"""
    import multiprocessing as mp
    import os
    from concurrent.futures import ProcessPoolExecutor
    with ProcessPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1)), mp_context=mp.get_context("spawn")) as ex:
        yield ex


def _exact_many(pool, cors, o_env, lane=None):
    quads = [geo.ccw(q) for q in o_env.obs_poly_list]
    field, polys = np.asarray(o_env.field_poly), (list(lane.polys) if lane is not None else [])
    chunks = [cors[k:k + 50] for k in range(0, len(cors), 50)]
    return np.array([r for part in pool.map(_exact_parts, [(c, quads, field, polys) for c in chunks]) for r in part])


def _check_truth(pool, o_env, o_car, o_h, poses, sample, what, aux):
    """the oracle's per-part verdicts equal the exact ones on ``sample``; with ``aux`` also those of the implement
    rectangles (obstacles and field) at the even indices"""
    body = geo.rect_corners(poses[sample], o_car.body_ext)
    want = _exact_many(pool, body, o_env, o_h.lane)
    got = np.stack([o_env.pose_flags(o_car, poses[sample], boundary_check=False),
                    ~geo.rects_inside_polygon(poses[sample], o_car.body_ext, o_env.field_poly, body),
                    o_h.pose_flags(o_car, poses[sample])], axis=1)
    bad = np.nonzero((want != got).any(axis=1))[0]
    assert len(bad) == 0, f"{what}: oracle differs from the exact reference at poses {poses[sample[bad[:5]]].tolist()}"
    even = sample[sample % 2 == 0]
    for ext in (o_car.aux_exts if aux else []):
        cor = geo.rect_corners(poses[even], ext)
        want = _exact_many(pool, cor, o_env)[:, :2]
        got = np.stack([o_env._part_flags(poses[even], ext, False),
                        ~geo.rects_inside_polygon(poses[even], ext, o_env.field_poly, cor)], axis=1)
        bad = np.nonzero((want != got).any(axis=1))[0]
        assert len(bad) == 0, f"{what}, aux {ext}: oracle differs from the exact reference at {poses[even[bad[:5]]].tolist()}"


SETS = {"canonical": ("obstacles", "field", "lane", "aux"), "quads": ("obstacles",), "field40": ("field",),
        "utm": ("obstacles", "field", "lane")}
REACH_FLAGS = {"obstacles": 1, "field": 2, "lane": 8, "aux": 7}


@pytest.mark.parametrize("scene", list(SETS))
def test_k1_boundary_poses_equal_oracle_and_exact(built_library, exact_pool, scene):
    """K1 == oracle on every pose, through the staged path (one environment) and the per-pose path (two copies,
    alternating env_id); oracle == exact on a sample of every set; the float64 predicates are really reached."""
    import torch
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.env_batch import EnvBatch
    o_env, o_car, o_h, rec, min_mag = _scene(scene)
    rng = np.random.default_rng(sum(map(ord, scene)))
    sets = [(kind,) + _make_set(rng, kind, o_env, o_car, o_h, min_mag) for kind in SETS[scene]]
    poses = np.concatenate([p for _, p, _ in sets])
    n = len(poses)
    one, two = EnvBatch([rec]), EnvBatch([rec, rec])
    d_poses = torch.from_numpy(poses).cuda()
    idx = torch.arange(n, dtype=torch.int32, device="cuda")
    alt = (idx & 1).to(torch.int32)
    for flags in (1, 3, 8, 11, 15):
        want = _oracle_flags(o_env, o_car, o_h, poses, flags)
        for path, got in (("staged", ops.collision_check(one, d_poses, pose_idx=idx, flags=flags)),
                          ("per-pose", ops.collision_check(two, d_poses, env_id=alt, pose_idx=idx, flags=flags))):
            g = got.cpu().numpy().astype(bool)
            bad = np.nonzero(g != want)[0]
            assert len(bad) == 0, (f"{scene}, {path} path, flags={flags}: {len(bad)} of {n} booleans differ from the "
                                   f"oracle, first poses {poses[bad[:3]].tolist()} (K1 says {g[bad[:3]].tolist()})")
        assert 0.01 < want.mean() < 0.995, (flags, want.mean())
    off = 0
    for kind, p, d in sets:
        m = len(p)
        # reach: the poses within 1e-5 m of an edge go to the float64 predicates
        small = np.nonzero(np.abs(d) <= 1e-5)[0] + off
        sel = torch.from_numpy(small).cuda()
        _, n_exact = ops.collision_check(one, d_poses[sel], pose_idx=idx[sel].contiguous(), flags=REACH_FLAGS[kind],
                                         count_exact=True)
        assert int(n_exact.item()) >= len(small) // 2, (scene, kind, int(n_exact.item()), len(small))
        sample = np.sort(rng.choice(m, N_TRUTH, replace=False)) + off
        _check_truth(exact_pool, o_env, o_car, o_h, poses, sample, f"{scene}/{kind}", kind == "aux")
        off += m


# ------------------------------------------------------------------ K7
def _k7_reference(occ, res, poses, ext):
    """exact: a non-finite pose hits; else the closed float64 rectangle meets the closed square of an occupied cell"""
    W, Hh = occ.shape
    ex, ey = np.arange(W + 1) * res, np.arange(Hh + 1) * res          # fl(i*res), as the kernel rounds it
    out = np.zeros(len(poses), dtype=bool)
    fin = np.isfinite(poses).all(axis=1)
    out[~fin] = True
    cors = geo.rect_corners(np.where(fin[:, None], poses, 0.0), ext)
    for p in np.nonzero(fin)[0]:
        c = cors[p]
        cols = np.nonzero((ex[:-1] <= c[:, 0].max()) & (ex[1:] >= c[:, 0].min()))[0]
        rows = np.nonzero((ey[:-1] <= c[:, 1].max()) & (ey[1:] >= c[:, 1].min()))[0]
        if len(cols) == 0 or len(rows) == 0:
            continue
        ii, jj = np.nonzero(occ[cols[0]:cols[-1] + 1, rows[0]:rows[-1] + 1])
        r = F(c)
        for i, j in zip(ii + cols[0], jj + rows[0]):
            sq = np.array([[ex[i], ey[j]], [ex[i + 1], ey[j]], [ex[i + 1], ey[j + 1]], [ex[i], ey[j + 1]]])
            if x_rect_hits_convex(r, F(sq)):
                out[p] = True
                break
    return out


def _k7(occ, res, poses, ext):
    from headland_trajectory_planning_b200 import ops
    bits = ops.grid_pack(occ)
    return ops.grid_footprint_check(bits, occ.shape, res, np.asarray(poses, dtype=np.float64), ext).cpu().numpy().astype(bool)


def _k7_cmp(occ, res, poses, ext, what):
    got = _k7(occ, res, poses, ext)
    want = _k7_reference(occ, res, poses, ext)
    bad = np.nonzero(got != want)[0]
    assert len(bad) == 0, (f"{what}: {len(bad)} of {len(poses)} differ, first poses {np.asarray(poses)[bad[:3]].tolist()} "
                           f"(K7 says {got[bad[:3]].tolist()}, exact {want[bad[:3]].tolist()})")
    return want


def _touch_below(res, n):
    """i < n where floor(fl(i*res) / res) < i: an edge exactly at fl(i*res) divides to just below i"""
    return [i for i in range(1, n) if math.floor((i * res) / res) < i]


def _ulp_overlap(res, n):
    """i < n where an edge one ulp below fl(i*res) still divides to i"""
    return [i for i in range(1, n) if math.floor(math.nextafter(i * res, -math.inf) / res) == i]


@pytest.mark.parametrize("res", [0.1, 0.05, 0.3, 0.25])
def test_k7_yaw0_ties_exact(built_library, res):
    """Yaw-0 rectangles with an edge exactly at fl(i*res) or one ulp either side, on both axes, from both sides,
    against a single occupied cell.  The tie cells come from the loops above (at res = 0.1: touch at i = 43, one-ulp
    overlap at i = 17); every case is also checked against what it must be."""
    touch, ulp = _touch_below(res, 5000), _ulp_overlap(res, 5000)
    assert (43 in touch and 17 in ulp) if res == 0.1 else True
    assert (not touch and not ulp) if res == 0.25 else (touch and ulp)
    idx = sorted(set(touch[:6] + ulp[:6] + [1, 2, 7, 40, 97]))
    idx = [i for i in idx if i < 120]
    n_cells = 124
    w = 2.5 * res                                     # rectangle length across the edge, half a cell wide the other way
    cases = []                                        # (axis, i, side, ulps, cell index across, expected hit)
    for axis in (0, 1):
        for i in idx:
            X = i * res
            for ulps in (-1, 0, 1):
                e = X if ulps == 0 else math.nextafter(X, ulps * math.inf)
                cases.append((axis, e, "below", i, ulps >= 0))         # rectangle below the edge, cell i above it
                cases.append((axis, e, "above", i - 1, ulps <= 0))     # rectangle above the edge, cell i-1 below it
    results, wrong = [], []
    for axis, e, side, cell, expect in cases:
        occ = np.zeros((n_cells, 7) if axis == 0 else (7, n_cells), dtype=bool)
        if axis == 0:
            occ[cell, 3] = True
        else:
            occ[3, cell] = True
        # the tied edge is a corner coordinate of exactly 0 + e; the other side of the rectangle is w away
        ext_along = (-w, 0.0) if side == "below" else (0.0, w)
        if axis == 0:
            ext, pose = (ext_along[0], ext_along[1], -0.25 * res, 0.25 * res), [e, 3.5 * res, 0.0]
        else:
            ext, pose = (-0.25 * res, 0.25 * res, ext_along[0], ext_along[1]), [3.5 * res, e, 0.0]
        got, want = _k7(occ, res, [pose], ext)[0], _k7_reference(occ, res, np.array([pose]), ext)[0]
        assert want == expect, (res, axis, e, side, cell)
        if got != want:
            wrong.append(f"axis={axis} edge={e!r} rectangle {side} cell {cell}: K7 {got}, exact {want}")
        results.append(want)
    assert not wrong, f"res={res}: {len(wrong)} of {len(cases)} ties wrong: " + "; ".join(wrong[:8])
    assert any(results) and not all(results)


def _random_grid(rng, W, Hh, p):
    return rng.random((W, Hh)) < p


@pytest.mark.parametrize("res", [0.1, 0.05, 0.3, 0.25])
def test_k7_general_yaw_near_cell_edges(built_library, res):
    """Random headings with a footprint corner 1e-9, 1e-6 or 1e-3 m from a cell edge or a cell corner."""
    rng = np.random.default_rng(int(res * 1000))
    W, Hh = 61, 45
    occ = _random_grid(rng, W, Hh, 0.12)
    ext = (-1.3 * res, 2.1 * res, -0.7 * res, 0.9 * res)
    lx = np.array([ext[0], ext[0], ext[1], ext[1]])
    ly = np.array([ext[3], ext[2], ext[2], ext[3]])
    poses = []
    for _ in range(1200):
        i, j = int(rng.integers(0, W + 1)), int(rng.integers(0, Hh + 1))
        q = np.array([i * res, j * res])
        if rng.random() < 0.5:                                         # a point on a cell edge, not a corner
            q[rng.integers(2)] += rng.uniform(0.05, 0.95) * res
        ang = rng.uniform(-math.pi, math.pi)
        q = q + rng.choice([1e-9, 1e-6, 1e-3]) * np.array([math.cos(ang), math.sin(ang)])
        yaw, k = rng.uniform(-math.pi, math.pi), int(rng.integers(4))
        c, s = math.cos(yaw), math.sin(yaw)
        poses.append([q[0] - (c * lx[k] - s * ly[k]), q[1] - (s * lx[k] + c * ly[k]), yaw])
    want = _k7_cmp(occ, res, np.array(poses), ext, f"res={res}")
    assert 0.2 < want.mean() < 0.9


def test_k7_grid_shapes_and_word_masks(built_library):
    """Shapes whose H and W*H are not multiples of 32 (W = 1 and H = 1 included), random poses on and around them;
    then column runs j0..j1 that start at bit 0, end at bit 31, or span two or three 32-bit words, each with one
    occupied cell at the first / last cell of the run (hit) or just outside it (free)."""
    rng = np.random.default_rng(7)
    res = 0.1
    for W, Hh in ((1, 1), (1, 37), (37, 1), (3, 33), (5, 70), (7, 100), (11, 97)):
        occ = _random_grid(rng, W, Hh, 0.15)
        ext = (-0.12, 0.21, -0.07, 0.09)
        n = 400
        poses = np.stack([rng.uniform(-0.4, W * res + 0.4, n), rng.uniform(-0.4, Hh * res + 0.4, n),
                          rng.uniform(-math.pi, math.pi, n)], 1)
        _k7_cmp(occ, res, poses, ext, f"{W}x{Hh}")
        _k7_cmp(np.ones_like(occ), res, poses, ext, f"{W}x{Hh} full")
    W, Hh = 9, 99                                      # 99 = 3*32 + 3: the words of column i start at bit (i*99) % 32
    n_runs = 0
    for i in range(W):
        base = i * Hh
        for j0 in range(Hh):
            for span in (32, 45, 70):                  # one word, two words, three words
                j1 = j0 + span - 1
                if j1 >= Hh:
                    continue
                first_bit, last_bit = (base + j0) % 32 == 0, (base + j1) % 32 == 31
                if not (first_bit or last_bit):
                    continue
                n_runs += 1
                ext = (-0.25 * res, 0.25 * res, 0.0, (j1 - j0) * res)
                pose = [[(i + 0.5) * res, (j0 + 0.5) * res, 0.0]]
                for cell, expect in ((j0, True), (j1, True), (j0 - 1, False), (j1 + 1, False)):
                    if not 0 <= cell < Hh:
                        continue
                    occ = np.zeros((W, Hh), dtype=bool)
                    occ[i, cell] = True
                    got = _k7(occ, res, pose, ext)[0]
                    assert got == expect == _k7_reference(occ, res, np.array(pose), ext)[0], (i, j0, j1, cell)
    assert n_runs >= 20


def test_k7_off_grid_huge_and_non_finite(built_library):
    """Poses partly off the grid on each side, fully off it, at +-1e12 m (the double-to-int conversion of the cell
    range saturates), and with NaN / +-inf in x, y or yaw: those always hit, even on an empty grid."""
    rng = np.random.default_rng(12)
    res, W, Hh = 0.1, 40, 30
    occ = _random_grid(rng, W, Hh, 0.3)
    occ[0, :] = occ[-1, :] = occ[:, 0] = occ[:, -1] = True
    ext = (-0.55, 3.0, -0.74, 0.74)
    side = []
    for x, y in ((-1.0, 1.5), (W * res + 1.0, 1.5), (2.0, -1.0), (2.0, Hh * res + 1.0),
                 (-0.2, -0.2), (W * res + 0.2, Hh * res + 0.2)):
        for yaw in np.linspace(-math.pi, math.pi, 16, endpoint=False):
            side.append([x, y, yaw])
    far = [[x, y, yaw] for x in (-1e12, 1e12, 2.0) for y in (-1e12, 1e12, 1.5) for yaw in (0.0, 1.1) if (x, y) != (2.0, 1.5)]
    far += [[-50.0, 1.5, 0.3], [2.0, 80.0, -2.0], [1e6, -1e6, 0.7]]
    want = _k7_cmp(occ, res, np.array(side + far), ext, "off grid")
    assert want[:len(side)].any() and not want[len(side):].any()
    nf = []
    for k in range(3):
        for v in (np.nan, np.inf, -np.inf):
            p = [2.0, 1.5, 0.3]
            p[k] = v
            nf.append(p)
    for grid in (np.zeros((W, Hh), dtype=bool), np.ones((W, Hh), dtype=bool)):
        got = _k7(grid, res, np.array(nf), ext)
        assert got.all(), f"non-finite poses reported free: {np.array(nf)[~got].tolist()}"


def test_k7_grid_pack_matches_packbits(built_library):
    """hl_grid_pack == numpy's little-endian bit packing of the row-major grid, tail word zero-padded."""
    rng = np.random.default_rng(3)
    for W, Hh in ((1, 1), (3, 7), (37, 29), (5, 70), (101, 33)):
        assert (W * Hh) % 32 != 0
        occ = rng.random((W, Hh)) < 0.5
        from headland_trajectory_planning_b200 import ops
        got = ops.grid_pack(occ).cpu().numpy().view(np.uint32)
        b = np.packbits(occ.ravel(), bitorder="little")
        b = np.concatenate([b, np.zeros((-len(b)) % 4, dtype=np.uint8)])
        assert np.array_equal(got, b.view("<u4")), (W, Hh)
