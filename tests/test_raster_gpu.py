"""K12 (hl_env_rasterize / ops.rasterize): occupancy grids from environment geometry, and K7's grid origin
(hl_grid_footprint_check_at).

A cell is the closed square [fl(g*res), fl((g+1)*res)] of its global indices; it is occupied when K1's float64
predicates at the identity pose find it meeting an obstacle quad (flag 1) or not contained in the field polygon
(flag 2).  The raster must equal the CPU oracle (``raster_oracle``: ``oracle.geometry``'s predicates per cell) on every
byte, the oracle must equal exact rational arithmetic on boundary cells, and the grid check K7 on a raster must be
conservative against K1: a pose K1 finds infeasible is infeasible on the grid.  Tests without the ``gpu`` marker run
on the CPU."""
import ctypes
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

import raster_oracle as RO
from exact_geom import F, x_rect_hits_convex, x_rect_in_polygon
from oracle import geometry as geo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLAG_SETS = (1, 2, 3)


# ------------------------------------------------------------------ helpers
def _exact_cell(job):
    """exact (meets an obstacle, not contained in the field) of cell squares; runs in a worker process"""
    squares, quads, field = job
    fq, ff = [F(q) for q in quads], F(field)
    out = []
    for sq in squares:
        r = F(sq)
        hit = any(x_rect_hits_convex(r, q) for q, Q in zip(fq, quads)
                  if not (sq[:, 0].max() < Q[:, 0].min() or Q[:, 0].max() < sq[:, 0].min() or
                          sq[:, 1].max() < Q[:, 1].min() or Q[:, 1].max() < sq[:, 1].min()))
        out.append((hit, (not x_rect_in_polygon(r, ff)) if len(field) else True))
    return out


def _oracle_job(job):
    quads, field, i0, j0, w, h, res = job
    return RO.raster_parts(quads, field, i0, j0, w, h, res)


@pytest.fixture(scope="module")
def pool():
    """worker processes for the oracle and the exact checks (spawned: they never touch CUDA)"""
    import multiprocessing as mp
    from concurrent.futures import ProcessPoolExecutor
    with ProcessPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1)), mp_context=mp.get_context("spawn")) as ex:
        yield ex


def _exact_cells(pool, quads, field, squares):
    quads = [np.asarray(q, dtype=np.float64) for q in quads]
    field = np.asarray(field, dtype=np.float64)
    chunks = [squares[k:k + 40] for k in range(0, len(squares), 40)]
    return np.array([r for part in pool.map(_exact_cell, [(c, quads, field) for c in chunks]) for r in part]).reshape(-1, 2)


def _cmp(got, want, what):
    got = got.cpu().numpy() if hasattr(got, "cpu") else np.asarray(got)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.argwhere(got != want)
    assert len(bad) == 0, f"{what}: {len(bad)} of {want.size} cells differ, first {bad[:5].tolist()}"


def _config5(k):
    """(EnvRecord with the scenario's car, oracle quads, field ring) of config-5 scenario k"""
    from headland_trajectory_planning_b200 import scenarios
    from headland_trajectory_planning_b200.car_model import CarModel
    from headland_trajectory_planning_b200.env_batch import make_record
    from headland_trajectory_planning_b200.orchard_geometry_environment import OrchardGeometryEnvironment
    sp = scenarios.scenario_spec(k)
    env = OrchardGeometryEnvironment(sp["rows"], [], tree_width=sp["tree_width"], headland_width=sp["headland_width"])
    rec = make_record(env, CarModel(**sp["car"]))
    return rec, rec.obs, rec.field


def _ccw_checked(quads):
    for q in quads:
        assert np.array_equal(geo.ccw(q), q), "obstacle quads must be counter-clockwise"


# ------------------------------------------------------------------ CPU only
def test_raster_window_hand_computed():
    from headland_trajectory_planning_b200 import ops
    ring = np.array([[0.0, 0.0], [1.0, 0.0], [1.0, 0.5], [0.0, 0.5]])
    # box [-0.25, 1.25] x [-0.25, 0.75] at res 0.5: cells -1 .. 2 (edge 1.0 and 1.5 straddle 1.25), rows -1 .. 1
    assert ops.raster_window(ring, 0.5, 0.25) == (-1, -1, 4, 3)
    # the box edges fall exactly on cell edges: the cells on both sides meet the closed interval
    assert ops.raster_window(ring, 0.5, 0.0) == (-1, -1, 4, 3)
    assert ops.raster_window(ring, 0.25, 0.0) == (-1, -1, 6, 4)
    # res = 0.1: fl(3*0.1) = 0.30000000000000004 > 0.3 and fl(7*0.1) = 0.7000000000000001 > 0.7, so x in [0.3, 0.7]
    # meets cells 2 .. 6 (cell 7 starts after 0.7); fl(6*0.1) = 0.6000000000000001 > 0.6: y in [0.3, 0.6] meets 2 .. 5
    tri = np.array([[0.3, 0.3], [0.7, 0.3], [0.5, 0.6]])
    assert ops.raster_window(tri, 0.1, 0.0) == (2, 2, 5, 4)
    for vmin, vmax, res in ((0.3, 0.7, 0.1), (0.3, 0.6, 0.1), (-4.35, 17.05, 0.05), (1e3 / 3, 1e3 / 3, 0.3)):
        lo, hi = ops._cell_range(vmin, vmax, res)
        meets = [i for i in range(lo - 5, hi + 6) if i * res <= vmax and (i + 1) * res >= vmin]
        assert meets == list(range(lo, hi + 1)), (vmin, vmax, res)
    # negative coordinates and a margin
    i0, j0, w, h = ops.raster_window(ring - 5.0, 1.0, 0.5)
    assert (i0, j0, w, h) == (-6, -6, 3, 3)                    # [-5.5, -3.5] x [-5.5, -4.0]
    with pytest.raises(Exception):
        ops.raster_window(ring, 0.0, 1.0)


def test_indices_beyond_int32_are_rejected_before_the_abi():
    """ctypes would wrap 2**31 + 5 into -2147483643 in an int32 slot, so the C side's range checks could not see it:
    ops rejects such values (naming the grid and the field) before anything reaches the library."""
    from headland_trajectory_planning_b200 import HeadlandError, ops
    ext = (-0.5, 1.0, -0.4, 0.4)
    for bad in ((0, 2**31 + 5, 0, 4, 4), (0, 0, -2**31 - 1, 4, 4), (2**32, 0, 0, 4, 4), (0, 0, 0, 2**32 + 4, 4)):
        with pytest.raises(HeadlandError, match="grid 1: .*int32"):
            ops.rasterize(None, [(0, 0, 0, 4, 4), bad], 0.1)
    with pytest.raises(HeadlandError, match="uint32"):
        ops.rasterize(None, [(0, 0, 0, 4, 4)], 0.1, flags=2**32 + 1)
    # a UTM northing at a millimetre grid gives indices beyond int32: raster_window computes them, rasterize refuses
    ring = np.array([[431250.0, 5291730.0], [431260.0, 5291730.0], [431260.0, 5291740.0]])
    win = ops.raster_window(ring, 0.001, 1.0)
    assert win[1] > 2**31
    with pytest.raises(HeadlandError, match="j0 = .*int32"):
        ops.rasterize(None, [(0,) + win], 0.001)
    for origin in ((2**31, 0), (0, -2**31 - 7)):
        with pytest.raises(HeadlandError, match="origin .*int32"):
            ops.grid_footprint_check(None, (4, 4), 0.1, np.zeros((1, 3)), ext, origin=origin)
    with pytest.raises(HeadlandError, match="w = .*int32"):
        ops.grid_footprint_check(None, (2**32 + 4, 4), 0.1, np.zeros((1, 3)), ext)


def test_oracle_equals_exact_on_small_grids():
    """The vectorised oracle rasteriser equals exact rational arithmetic on every cell of small grids with edges and
    vertices placed on, and one ulp beside, cell edges."""
    res = 0.1
    g = lambda i: i * res
    up = lambda v: math.nextafter(v, math.inf)
    dn = lambda v: math.nextafter(v, -math.inf)
    quads = [np.array([[g(3), g(3)], [g(5), g(3)], [g(5), g(5)], [g(3), g(5)]]),                 # on cell edges
             np.array([[up(g(8)), dn(g(2))], [dn(g(10)), dn(g(2))], [dn(g(10)), up(g(4))], [up(g(8)), up(g(4))]]),
             np.array([[g(6), g(7)], [0.75, 0.78], [g(6), 0.86], [0.45, 0.78]])]             # vertex on a corner
    field = np.array([[g(1), g(1)], [g(11), g(1)], [g(11), g(9)], [0.65, up(0.95)], [g(1), g(9)]])
    i0, j0, w, h = 0, 0, 13, 11
    parts = RO.raster_parts(quads, field, i0, j0, w, h, res)
    squares = [RO.cell_square(i0, j0, i, j, res) for i in range(w) for j in range(h)]
    want = np.array(_exact_cell((squares, quads, field)))
    assert np.array_equal(parts[0].reshape(-1), want[:, 0]) and np.array_equal(parts[1].reshape(-1), want[:, 1])
    assert parts[0].any() and not parts[0].all() and parts[1].any() and not parts[1].all()


# ------------------------------------------------------------------ GPU: scenes
def _boundary_scenes():
    from test_footprint_boundary_gpu import _scene
    out = {}
    for kind in ("canonical", "quads", "field40", "utm"):
        rec = _scene(kind)[3]
        out[kind] = rec
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("res", [0.1, 0.3])
def test_boundary_scenes_equal_oracle(built_library, pool, res):
    """The footprint-boundary scenes (canonical, non-rectangular quads, a field of more than 32 edges, UTM-sized
    coordinates with cell indices around 4.3 M at 0.1 m), flags 1, 2 and 3, byte for byte."""
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.env_batch import EnvBatch
    scenes = _boundary_scenes()
    recs = list(scenes.values())
    envs = EnvBatch(recs)
    wins = [ops.raster_window(r.field, res, 2.0) for r in recs]
    assert wins[-1][0] > 4_000_000 or res != 0.1
    jobs = [(r.obs, r.field) + tuple(win) + (res,) for r, win in zip(recs, wins)]
    parts = list(pool.map(_oracle_job, jobs))
    for flags in FLAG_SETS:
        got = ops.rasterize(envs, [(e,) + tuple(win) for e, win in enumerate(wins)], res, flags)
        for kind, g, p in zip(scenes, got, parts):
            _cmp(g, RO.combine(p, flags), f"{kind} res={res} flags={flags}")


@pytest.mark.gpu
@pytest.mark.parametrize("res", [0.1, 0.05, 0.3, 0.25])
def test_config5_batch_equals_oracle(built_library, pool, res):
    """32 config-5 environments in one batch, every grid side by side in one pooled buffer, flags 1, 2 and 3."""
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.env_batch import EnvBatch
    items = [_config5(k) for k in range(32)]
    for _, q, _ in items:
        _ccw_checked(q)
    envs = EnvBatch([r for r, _, _ in items])
    wins = [ops.raster_window(f, res, 2.0) for _, _, f in items]
    parts = list(pool.map(_oracle_job, [(q, f) + tuple(w) + (res,) for (_, q, f), w in zip(items, wins)]))
    for flags in FLAG_SETS:
        got, n_exact = ops.rasterize(envs, [(e,) + tuple(w) for e, w in enumerate(wins)], res, flags, count_exact=True)
        for k, (g, p) in enumerate(zip(got, parts)):
            want = RO.combine(p, flags)
            _cmp(g, want, f"env {k} res={res} flags={flags}")
            assert 0.0 < want.mean() < 1.0
        assert int(n_exact.item()) < sum(g.numel() for g in got) // 20


@pytest.mark.gpu
def test_odd_grids_equal_oracle(built_library):
    """w = 1 and h = 1 grids, a grid wholly outside the field, a grid inside one tree row, negative origins; several
    grids of one environment in one call."""
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.env_batch import EnvBatch
    rec, quads, field = _config5(3)
    envs = EnvBatch([rec, _config5(4)[0]])
    res = 0.05
    i0, j0, w, h = ops.raster_window(field, res, 2.0)
    row = quads[2]
    ri, rj = int(row[:, 0].mean() / res), int(row[:, 1].mean() / res)
    grids = [(0, i0, j0, 1, h), (0, i0 + w // 2, j0, 1, h), (0, i0, j0 + h // 2, w, 1), (0, i0 + 7, j0 + 9, 1, 1),
             (0, i0 - 500, j0 - 400, 37, 29),                  # wholly outside the field
             (0, ri - 1, rj, 2, 2), (0, ri, rj, 1, 1),         # inside one tree row
             (0, -37, -45, 300, 260), (1, -20, -30, 70, 80), (0, i0, j0, w, h)]
    for flags in FLAG_SETS:
        got = ops.rasterize(envs, grids, res, flags)
        for k, (e, a, b, ww, hh) in enumerate(grids):
            q, f = (quads, field) if e == 0 else _config5(4)[1:]
            _cmp(got[k], RO.rasterize(q, f, a, b, ww, hh, res, flags), f"grid {k} flags={flags}")
    got = ops.rasterize(envs, grids, res, 3)
    assert got[4].cpu().numpy().all()                          # outside the field: all occupied
    assert not ops.rasterize(envs, grids[4:5], res, 1)[0].cpu().numpy().any()   # ... and no obstacle there
    assert got[6].cpu().numpy().all() and ops.rasterize(envs, grids[6:7], res, 1)[0].cpu().numpy().all()


def _exact_scene():
    """obstacle squares with edges at fl(g*res) and one ulp either side, a quad with a vertex on a cell corner, rotated
    quads, a field whose edges lie on cell edges and whose other vertices sit 1e-12 .. 1e-3 m from cell edges"""
    res = 0.1
    g = lambda i: i * res
    up = lambda v: math.nextafter(v, math.inf)
    dn = lambda v: math.nextafter(v, -math.inf)
    quads = []
    for k, (f0, f1) in enumerate(((lambda v: v, lambda v: v), (up, dn), (dn, up), (up, up), (dn, dn))):
        a, b = 4 + 6 * k, 8
        quads.append(np.array([[f0(g(a)), f0(g(b))], [f1(g(a + 3)), f0(g(b))], [f1(g(a + 3)), f1(g(b + 2))],
                               [f0(g(a)), f1(g(b + 2))]]))
    quads.append(np.array([[g(12), g(16)], [g(14) - 0.03, g(15) + 0.04], [g(14), g(17)], [g(13), g(18) - 0.02]]))
    rng = np.random.default_rng(5)
    for k in range(6):                                         # rotated squares with a vertex near a cell edge
        c = np.array([g(4 + 5 * k) + 0.25, g(22) + 0.2])
        ang = rng.uniform(0.1, 1.4)
        v = c + 0.17 * np.array([[math.cos(ang + m * math.pi / 2), math.sin(ang + m * math.pi / 2)] for m in range(4)])
        d = (1e-12, 1e-9, 1e-6, 1e-4, 1e-3, -1e-9)[k]
        v[0, 0] = g(round(v[0, 0] / res)) + d
        quads.append(geo.ccw(v))
    ring = [[g(2), g(2)], [g(34), g(2)], [g(34), g(26)]]
    for k, d in enumerate((1e-12, -1e-12, 1e-9, -1e-6, 1e-4, -1e-3, 1e-3)):
        ring.append([g(34 - 4 * k) - 0.013, g(26) + d])          # near the row edge fl(26*res), both sides
    ring += [[g(2), g(28)]]
    field = geo.ccw(np.array(ring))
    return res, quads, field


@pytest.mark.gpu
def test_exact_cells(built_library, pool):
    """On the exact scene: raster == oracle on every cell, oracle == exact rational arithmetic on every cell, and the
    float64 predicates are reached (d_n_exact > 0)."""
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.env_batch import EnvRecord, EnvBatch
    res, quads, field = _exact_scene()
    _ccw_checked(quads)
    envs = EnvBatch([EnvRecord(np.array(quads), field, (-0.5, 1.0, -0.4, 0.4))])
    i0, j0, w, h = -1, -2, 38, 33
    parts = RO.raster_parts(quads, field, i0, j0, w, h, res)
    for flags in FLAG_SETS:
        got, n_exact = ops.rasterize(envs, [(0, i0, j0, w, h)], res, flags, count_exact=True)
        _cmp(got[0], RO.combine(parts, flags), f"exact scene flags={flags}")
        assert int(n_exact.item()) > 0, flags
    squares = [RO.cell_square(i0, j0, i, j, res) for i in range(w) for j in range(h)]
    want = _exact_cells(pool, quads, field, squares)
    assert np.array_equal(parts[0].reshape(-1), want[:, 0]) and np.array_equal(parts[1].reshape(-1), want[:, 1])
    # the touching cases: a cell touching the field's bottom edge from inside is free, from outside occupied
    bi, bj = 10 - i0, 2 - j0
    assert not parts[1][bi, bj] and parts[1][bi, bj - 1]
    # the square on cell edges hits the cells that touch it; the one-ulp-shrunk square does not reach them
    assert parts[0][3 - i0, 8 - j0] and parts[0][7 - i0, 10 - j0]


# ------------------------------------------------------------------ GPU: against K1
def _poses_in(rng, n, lo, hi, ext):
    """n poses whose body lies wholly inside the box [lo, hi] (corners checked with the oracle's corner formula)"""
    out = []
    while sum(map(len, out)) < n:
        p = np.stack([rng.uniform(lo[0], hi[0], 2 * n), rng.uniform(lo[1], hi[1], 2 * n), rng.uniform(-math.pi, math.pi, 2 * n)], 1)
        c = geo.rect_corners(p, ext)
        ok = (c[..., 0].min(1) > lo[0]) & (c[..., 0].max(1) < hi[0]) & (c[..., 1].min(1) > lo[1]) & (c[..., 1].max(1) < hi[1])
        out.append(p[ok])
    return np.concatenate(out)[:n]


@pytest.mark.gpu
def test_grid_check_conservative_against_k1(built_library):
    """K1 hit => K7 hit on the raster, with no exception, for 2e5 random poses per scene and the near-boundary pose
    sets of test_footprint_boundary_gpu (|delta| >= 1e-9 m), flags 1, 2 and 3; and K7 hit => K1 hit for the body grown
    by 1.5 res on every side (the raster is not trivially occupied)."""
    import torch
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.env_batch import EnvBatch, EnvRecord
    from test_footprint_boundary_gpu import _make_set, _scene
    rng = np.random.default_rng(99)
    scenes = []
    for kind in ("canonical", "quads", "field40", "utm"):
        o_env, o_car, o_h, rec, min_mag = _scene(kind)
        near = [_make_set(rng, k, o_env, o_car, o_h, max(min_mag, 1e-9))[0] for k in ("obstacles", "field")]
        scenes.append((kind, rec, np.concatenate(near)))
    for k in (0, 1):
        rec = _config5(k)[0]
        scenes.append((f"config5-{k}", rec, np.zeros((0, 3))))
    for kind, rec, near in scenes:
        ext = tuple(rec.body_ext)
        for res in (0.1, 0.25):
            i0, j0, w, h = ops.raster_window(rec.field, res, 2.0)
            lo, hi = (i0 * res, j0 * res), ((i0 + w) * res, (j0 + h) * res)
            poses = _poses_in(rng, 200_000, lo, hi, ext)
            c = geo.rect_corners(near, ext)
            inside = (c[..., 0].min(1) > lo[0]) & (c[..., 0].max(1) < hi[0]) & (c[..., 1].min(1) > lo[1]) & (c[..., 1].max(1) < hi[1])
            poses = np.concatenate([poses, near[inside]])
            grown = (ext[0] - 1.5 * res, ext[1] + 1.5 * res, ext[2] - 1.5 * res, ext[3] + 1.5 * res)
            envs = EnvBatch([rec])
            envs_g = EnvBatch([EnvRecord(rec.obs, rec.field, grown)])
            d_poses = torch.from_numpy(poses).cuda()
            for flags in FLAG_SETS:
                grid = ops.rasterize(envs, [(0, i0, j0, w, h)], res, flags)[0]
                k7 = ops.grid_footprint_check(ops.grid_pack(grid), (w, h), res, d_poses, ext, origin=(i0, j0)).cpu().numpy().astype(bool)
                k1 = ops.collision_check(envs, d_poses, flags=flags).cpu().numpy().astype(bool)
                k1g = ops.collision_check(envs_g, d_poses, flags=flags).cpu().numpy().astype(bool)
                miss = np.nonzero(k1 & ~k7)[0]
                assert len(miss) == 0, f"{kind} res={res} flags={flags}: K1 hit but grid free at {poses[miss[:3]].tolist()}"
                over = np.nonzero(k7 & ~k1g)[0]
                assert len(over) == 0, f"{kind} res={res} flags={flags}: grid hit but grown K1 free at {poses[over[:3]].tolist()}"
                assert k1.any() and not k7.all()
            if kind.startswith("config5"):
                occ = ops.rasterize(envs, [(0, i0, j0, w, h)], res, 3)[0].cpu().numpy()
                assert 0.0 < occ.mean() < 1.0


# ------------------------------------------------------------------ GPU: into K6
@pytest.mark.gpu
def test_rasters_into_distance_fields(built_library):
    """With the boundary test and a margin of at least 2 res every border cell is occupied; distance fields of 16
    rasterised config-5 scenes (goal = the cell holding the scenario's goal) through distance_field_batch on the raster
    views equal distance_field per grid, and one 0.3 m field equals the oracle."""
    from headland_trajectory_planning_b200 import ops, scenarios
    from headland_trajectory_planning_b200.env_batch import EnvBatch
    from oracle import distance_field as DF
    scns = scenarios.make_scenarios_gpu(range(16))
    items = [_config5(k) for k in range(16)]
    envs = EnvBatch([r for r, _, _ in items])
    for res in (0.1, 0.3):
        wins = [ops.raster_window(f, res, 2 * res) for _, _, f in items]
        grids = ops.rasterize(envs, [(e,) + tuple(w) for e, w in enumerate(wins)], res, ops.CHECK_OBSTACLES | ops.CHECK_BOUNDARY)
        goals = []
        for s, (i0, j0, w, h), g in zip(scns, wins, grids):
            a = g.cpu().numpy()
            assert a[0, :].all() and a[-1, :].all() and a[:, 0].all() and a[:, -1].all()
            gi, gj = ops._cell_range(s["goal"][0], s["goal"][0], res)[0] - i0, ops._cell_range(s["goal"][1], s["goal"][1], res)[0] - j0
            assert 0 <= gi < w and 0 <= gj < h
            goals.append((gi, gj))
        fields, sweeps = ops.distance_field_batch(grids, goals, "King")
        assert sweeps > 0
        for k, (g, goal, f) in enumerate(zip(grids, goals, fields)):
            single, _ = ops.distance_field(g, goal, "King")
            assert np.array_equal(single.cpu().numpy(), f.cpu().numpy()), (res, k)
            assert np.isfinite(f.cpu().numpy()).sum() > 100
        if res == 0.3:
            want = DF.holonomic_costs_with_obstacles(goals[0], grids[0].cpu().numpy().astype(bool), "King")
            assert np.array_equal(want, fields[0].cpu().numpy())


# ------------------------------------------------------------------ GPU: K7 origin
def _k7_at(occ, origin, res, poses, ext):
    from headland_trajectory_planning_b200 import ops
    return ops.grid_footprint_check(ops.grid_pack(occ), occ.shape, res, np.asarray(poses, dtype=np.float64), ext,
                                    origin=origin).cpu().numpy().astype(bool)


def _k7_shifted_reference(occ, origin, res, poses, ext):
    """exact: the closed float64 rectangle meets the closed square [fl(g*res), fl((g+1)*res)] of an occupied cell"""
    W, Hh = occ.shape
    ex, ey = RO.cell_edges(origin[0], W, res), RO.cell_edges(origin[1], Hh, res)
    out = np.zeros(len(poses), dtype=bool)
    cors = geo.rect_corners(poses, ext)
    for p, c in enumerate(cors):
        cols = np.nonzero((ex[:-1] <= c[:, 0].max()) & (ex[1:] >= c[:, 0].min()))[0]
        rows = np.nonzero((ey[:-1] <= c[:, 1].max()) & (ey[1:] >= c[:, 1].min()))[0]
        if len(cols) == 0 or len(rows) == 0:
            continue
        r = F(c)
        for i, j in zip(*np.nonzero(occ[cols[0]:cols[-1] + 1, rows[0]:rows[-1] + 1])):
            i, j = i + cols[0], j + rows[0]
            sq = np.array([[ex[i], ey[j]], [ex[i + 1], ey[j]], [ex[i + 1], ey[j + 1]], [ex[i], ey[j + 1]]])
            if x_rect_hits_convex(r, F(sq)):
                out[p] = True
                break
    return out


@pytest.mark.gpu
def test_k7_origin_zero_equals_plain_call(built_library):
    import torch
    from headland_trajectory_planning_b200 import _lib, ops
    lib = _lib.load_library()
    rng = np.random.default_rng(4)
    for W, Hh, res, p in ((160, 120, 0.1, 0.02), (61, 45, 0.05, 0.12), (37, 1, 0.3, 0.3), (1, 37, 0.25, 0.3)):
        occ = rng.random((W, Hh)) < p
        ext = (-0.55, 3.0, -0.74, 0.74) if res == 0.1 else (-1.3 * res, 2.1 * res, -0.7 * res, 0.9 * res)
        n = 4000
        poses = torch.from_numpy(np.stack([rng.uniform(-1, W * res + 1, n), rng.uniform(-1, Hh * res + 1, n),
                                           rng.uniform(-math.pi, math.pi, n)], 1)).cuda()
        bits = ops.grid_pack(occ)
        e = (ctypes.c_double * 4)(*ext)
        a = torch.empty(n, dtype=torch.uint8, device="cuda")
        b = torch.empty_like(a)
        _lib.check(lib.hl_grid_footprint_check(_lib.get_ctx(), _lib.ptr(bits), W, Hh, res, _lib.ptr(poses), n, e,
                                               _lib.ptr(a), _lib.stream_ptr()), "plain")
        _lib.check(lib.hl_grid_footprint_check_at(_lib.get_ctx(), _lib.ptr(bits), W, Hh, 0, 0, res, _lib.ptr(poses), n, e,
                                                  _lib.ptr(b), _lib.stream_ptr()), "at")
        assert torch.equal(a, b) and 0 < int(a.sum()) < n


@pytest.mark.gpu
@pytest.mark.parametrize("res", [0.1, 0.3])
def test_k7_origin_offsets_exact(built_library, res):
    """Offsets (-37, 12345) and (4_312_500, -52_917): random headings against a brute force over the shifted cell
    squares, and yaw-0 rectangles with an edge at fl(g*res) and one ulp either side."""
    rng = np.random.default_rng(int(res * 100))
    for origin in ((-37, 12345), (4_312_500, -52_917)):
        W, Hh = 41, 33
        occ = rng.random((W, Hh)) < 0.12
        ext = (-1.3 * res, 2.1 * res, -0.7 * res, 0.9 * res)
        x0, y0 = origin[0] * res, origin[1] * res
        n = 800
        poses = np.stack([x0 + rng.uniform(-0.5, W * res + 0.5, n), y0 + rng.uniform(-0.5, Hh * res + 0.5, n),
                          rng.uniform(-math.pi, math.pi, n)], 1)
        want = _k7_shifted_reference(occ, origin, res, poses, ext)
        assert np.array_equal(_k7_at(occ, origin, res, poses, ext), want), origin
        assert 0.1 < want.mean() < 0.95
        # yaw-0 ties: a rectangle whose right edge sits at fl(g*res) or one ulp beside it, one occupied cell g
        one = np.zeros((W, Hh), dtype=bool)
        one[20, 10] = True
        ties, exp = [], []
        for gi in (20, 21):
            X = float(origin[0] + gi) * res
            for ulps in (-1, 0, 1):
                e = X if ulps == 0 else math.nextafter(X, ulps * math.inf)
                y = (float(origin[1] + 10) + 0.5) * res
                ties.append([e, y, 0.0])
        ext0 = (-0.6 * res, 0.0, -0.2 * res, 0.2 * res)
        want = _k7_shifted_reference(one, origin, res, np.array(ties), ext0)
        assert np.array_equal(_k7_at(one, origin, res, ties, ext0), want), origin
        assert want.any() and not want.all()


# ------------------------------------------------------------------ plumbing
def test_raster_grid_layout_matches_header(built_library):
    from headland_trajectory_planning_b200 import _lib
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "headland_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(HlRasterGrid), offsetof(HlRasterGrid, out_offset),
         offsetof(HlRasterGrid, env_id), offsetof(HlRasterGrid, w), offsetof(HlRasterGrid, h),
         offsetof(HlRasterGrid, i0), offsetof(HlRasterGrid, j0));
  return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        out = [int(v) for v in subprocess.check_output([exe], text=True).split()]
    G = _lib.HlRasterGrid
    assert out == [ctypes.sizeof(G), G.out_offset.offset, G.env_id.offset, G.w.offset, G.h.offset, G.i0.offset, G.j0.offset]


@pytest.mark.gpu
def test_rejections_and_determinism(built_library):
    import torch
    from headland_trajectory_planning_b200 import HeadlandError, _lib, ops
    from headland_trajectory_planning_b200.env_batch import EnvBatch
    items = [_config5(k) for k in range(3)]
    envs = EnvBatch([r for r, _, _ in items])
    res = 0.1
    wins = [ops.raster_window(f, res, 2.0) for _, _, f in items]
    grids = [(e,) + tuple(w) for e, w in enumerate(wins)]
    a = ops.rasterize(envs, grids, res)
    b = ops.rasterize(envs, grids, res)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert ops.rasterize(envs, [], res) == []
    with pytest.raises(HeadlandError, match="grid 1"):
        ops.rasterize(envs, [grids[0], (3, 0, 0, 4, 4)], res)
    with pytest.raises(HeadlandError, match="grid 0"):
        ops.rasterize(envs, [(0, 0, 0, 0, 4)], res)
    with pytest.raises(HeadlandError, match="grid 1"):
        ops.rasterize(envs, [grids[0], (0, 2**31 - 3, 0, 4, 4)], res)
    with pytest.raises(HeadlandError, match="grid 0"):
        ops.rasterize(envs, [(0, 2**31 - 8, 0, 4, 4)], 1e300)
    for bad_res in (0.0, -0.1, math.inf, math.nan):
        with pytest.raises(HeadlandError, match="res"):
            ops.rasterize(envs, grids, bad_res)
    for bad_flags in (0, 4, 8, 7):
        with pytest.raises(HeadlandError, match="flags"):
            ops.rasterize(envs, grids, res, bad_flags)

    lib = _lib.load_library()
    out = torch.zeros(3 * 100, dtype=torch.uint8, device="cuda")

    def call(entries, out_elems=out.numel(), flags=3, n=None):
        t = (_lib.HlRasterGrid * max(len(entries), 1))(*[_lib.HlRasterGrid(*e) for e in entries])
        rc = lib.hl_env_rasterize(envs.ctx, envs.handle, t, len(entries) if n is None else n, res, flags, _lib.ptr(out),
                                  out_elems, None, _lib.stream_ptr())
        return rc, _lib.last_error()

    ok = [(0, 0, 10, 10, 0, 0), (100, 1, 10, 10, 5, 5), (200, 2, 10, 10, -5, -5)]
    assert call(ok)[0] == 0
    rc, msg = call([ok[0], (50, 1, 10, 10, 0, 0)])
    assert rc != 0 and "grids 0 and 1" in msg and "overlap" in msg
    rc, msg = call([ok[0], ok[1], (250, 2, 10, 10, 0, 0)])
    assert rc != 0 and "grid 2" in msg
    rc, msg = call([ok[0], (100, 1, 10, 10, 0, 2**31 - 5)])
    assert rc != 0 and "grid 1" in msg
    rc, msg = call([(0, 0, 10, 10, 0, 0), (100, 0, 10, -1, 0, 0)])
    assert rc != 0 and "grid 1" in msg
    rc, msg = call([(0, -1, 10, 10, 0, 0)])
    assert rc != 0 and "grid 0" in msg and "env_id" in msg
    rc, msg = call(ok, flags=8)
    assert rc != 0 and "flags" in msg
    out.fill_(7)
    rc, msg = call([], n=0)
    assert rc == 0 and bool((out == 7).all())



@pytest.mark.gpu
def test_occupancy_grid_of_the_mirror(built_library):
    """OrchardGeometryEnvironment.occupancy_grid needs no car, and its grid is the raster of its own quads and ring."""
    from headland_trajectory_planning_b200 import scenarios
    from headland_trajectory_planning_b200.orchard_geometry_environment import OrchardGeometryEnvironment
    sp = scenarios.scenario_spec(7)
    env = OrchardGeometryEnvironment(sp["rows"], [(3.0, 4.0)], tree_width=sp["tree_width"], headland_width=sp["headland_width"])
    grid, (i0, j0) = env.occupancy_grid(0.2, margin=1.0)
    w, h = grid.shape
    _cmp(grid, RO.rasterize(env.obstacle_quads(), env.field_ring(), i0, j0, w, h, 0.2, 3), "mirror")
    g1, o1 = env.occupancy_grid(0.2, margin=1.0, flags=1)
    assert o1 == (i0, j0) and int(g1.sum()) < int(grid.sum())
