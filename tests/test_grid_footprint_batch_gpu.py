"""K7 batch (hl_grid_pack_batch / hl_grid_footprint_check_batch, ops.grid_pack_batch / grid_footprint_check_batch /
grid_check_sweep): many grids packed in one launch, many (grid, vehicle) maps checked in one launch, implement
rectangles at even path indices.

Every verdict is compared with the exact references of the single-grid K7 tests (``_k7_reference``,
``_k7_shifted_reference``: closed float64 rectangles against closed cell squares in rational arithmetic), and with the
single-grid calls, which are batches of one of the same kernels."""
import ctypes
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

import hl_helpers as H
from test_footprint_boundary_gpu import _make_set, _scene, _touch_below, _ulp_overlap
from test_raster_gpu import _config5, _k7_shifted_reference, _poses_in

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MOWER_AUX = [[[-1.84, 0.5], 1.0, 1.1]]


def _exts(aux_features):
    """CarModel's implement extents (x0, x1, y0, y1) of aux_poly_features"""
    return np.array([[f[0][0], f[0][0] + f[2], f[0][1] - f[1], f[0][1]] for f in aux_features], dtype=np.float64).reshape(-1, 4)


def _packbits(occ):
    b = np.packbits(np.asarray(occ, dtype=bool).ravel(), bitorder="little")
    return np.concatenate([b, np.zeros((-len(b)) % 4, dtype=np.uint8)]).view("<u4")


# ------------------------------------------------------------------ layout
def test_grid_pack_and_map_layout_matches_header(built_library):
    from headland_trajectory_planning_b200 import _lib
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "headland_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu\n", sizeof(HlGridPack), offsetof(HlGridPack, occ_offset), offsetof(HlGridPack, bits_offset),
         offsetof(HlGridPack, w), offsetof(HlGridPack, h));
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(HlGridMap), offsetof(HlGridMap, bits_offset),
         offsetof(HlGridMap, w), offsetof(HlGridMap, h), offsetof(HlGridMap, i0), offsetof(HlGridMap, j0),
         offsetof(HlGridMap, body_ext), offsetof(HlGridMap, aux_first), offsetof(HlGridMap, n_aux));
  return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        out = [int(v) for v in subprocess.check_output([exe], text=True).split()]
    P, M = _lib.HlGridPack, _lib.HlGridMap
    assert out == [ctypes.sizeof(P), P.occ_offset.offset, P.bits_offset.offset, P.w.offset, P.h.offset,
                   ctypes.sizeof(M), M.bits_offset.offset, M.w.offset, M.h.offset, M.i0.offset, M.j0.offset,
                   M.body_ext.offset, M.aux_first.offset, M.n_aux.offset]


# ------------------------------------------------------------------ pack
SENTINEL = 0x5A5A5A5A


@pytest.mark.gpu
def test_pack_batch_interleaved_slices(built_library):
    """One call over five grids whose byte grids and bit slices are interleaved with gaps, one slice at word 0: each
    slice equals numpy's little-endian packbits with a zero tail and ops.grid_pack, the words between slices keep their
    sentinel; ops.grid_pack_batch on rasterize's views (packed in place) equals the same grids uploaded from the host."""
    import torch
    from headland_trajectory_planning_b200 import _lib, ops
    from headland_trajectory_planning_b200.env_batch import EnvBatch
    rng = np.random.default_rng(3)
    shapes = ((1, 1), (3, 7), (37, 29), (5, 70), (101, 33))
    occs = [rng.random(s) < 0.5 for s in shapes]
    order = [2, 0, 4, 1, 3]                           # slice order in the buffers; grid 2 starts at word 0
    occ_off, bits_off, ob, wb = {}, {}, 0, 0
    for k in order:
        w, h = shapes[k]
        occ_off[k], bits_off[k] = ob, wb
        ob += w * h + 5
        wb += (w * h + 31) // 32 + 2                  # two sentinel words after every slice
    occ_host = np.full(ob, 9, dtype=np.uint8)         # gap bytes are non-zero: a read past a grid would show
    for k, (w, h) in enumerate(shapes):
        occ_host[occ_off[k]:occ_off[k] + w * h] = occs[k].ravel()
    occ = torch.from_numpy(occ_host).cuda()
    bits = torch.full((wb,), SENTINEL, dtype=torch.int32, device="cuda")
    table = (_lib.HlGridPack * 5)(*[_lib.HlGridPack(occ_off[k], bits_off[k], w, h) for k, (w, h) in enumerate(shapes)])
    lib = _lib.load_library()
    _lib.check(lib.hl_grid_pack_batch(_lib.get_ctx(), _lib.ptr(occ), ob, table, 5, _lib.ptr(bits), wb, _lib.stream_ptr()),
               "hl_grid_pack_batch")
    got = bits.cpu().numpy().view(np.uint32)
    touched = np.zeros(wb, dtype=bool)
    for k, (w, h) in enumerate(shapes):
        nw = (w * h + 31) // 32
        s = got[bits_off[k]:bits_off[k] + nw]
        assert np.array_equal(s, _packbits(occs[k])), shapes[k]
        assert np.array_equal(s, ops.grid_pack(occs[k]).cpu().numpy().view(np.uint32)), shapes[k]
        touched[bits_off[k]:bits_off[k] + nw] = True
    assert (got[~touched] == SENTINEL).all()

    items = [_config5(k) for k in range(3)]
    envs = EnvBatch([r for r, _, _ in items])
    wins = [(e,) + tuple(ops.raster_window(f, 0.2, 2.0)) for e, (_, _, f) in enumerate(items)]
    views = ops.rasterize(envs, wins, 0.2, 3)
    a, oa = ops.grid_pack_batch(views)
    b, ob_ = ops.grid_pack_batch([v.cpu().numpy() for v in views])
    c, oc = ops.grid_pack_batch([v.clone() for v in views])           # CUDA tensors of separate storages: one copy
    assert torch.equal(a, b) and torch.equal(a, c) and np.array_equal(oa, ob_) and np.array_equal(oa, oc)
    for v, o in zip(views, oa):
        single = ops.grid_pack(v)
        assert torch.equal(a[o:o + single.numel()], single)
    empty, eo = ops.grid_pack_batch([])
    assert empty.numel() == 0 and len(eo) == 0


# ------------------------------------------------------------------ body, exact
def _tie_maps(res):
    """the yaw-0 tie constructions of test_k7_yaw0_ties_exact as (occ, origin, ext, pose): one occupied cell per map"""
    touch, ulp = _touch_below(res, 200), _ulp_overlap(res, 200)
    idx = sorted({i for i in touch[:3] + ulp[:3] + [1, 7, 40, 97] if i < 120})
    w = 2.5 * res
    out = []
    for axis in (0, 1):
        for i in idx:
            X = i * res
            for ulps in (-1, 0, 1):
                e = X if ulps == 0 else math.nextafter(X, ulps * math.inf)
                for side, cell in (("below", i), ("above", i - 1)):
                    occ = np.zeros((124, 7) if axis == 0 else (7, 124), dtype=bool)
                    occ[(cell, 3) if axis == 0 else (3, cell)] = True
                    along = (-w, 0.0) if side == "below" else (0.0, w)
                    if axis == 0:
                        ext, pose = (along[0], along[1], -0.25 * res, 0.25 * res), [e, 3.5 * res, 0.0]
                    else:
                        ext, pose = (-0.25 * res, 0.25 * res, along[0], along[1]), [3.5 * res, e, 0.0]
                    out.append((occ, (0, 0), ext, np.array([pose])))
    return out


def _near_edge_poses(rng, W, Hh, origin, res, ext, n):
    """test_k7_general_yaw_near_cell_edges' poses: a footprint corner 1e-9, 1e-6 or 1e-3 m from a cell edge or corner"""
    lx = np.array([ext[0], ext[0], ext[1], ext[1]])
    ly = np.array([ext[3], ext[2], ext[2], ext[3]])
    poses = []
    for _ in range(n):
        i, j = int(rng.integers(0, W + 1)) + origin[0], int(rng.integers(0, Hh + 1)) + origin[1]
        q = np.array([i * res, j * res])
        if rng.random() < 0.5:
            q[rng.integers(2)] += rng.uniform(0.05, 0.95) * res
        ang = rng.uniform(-math.pi, math.pi)
        q = q + rng.choice([1e-9, 1e-6, 1e-3]) * np.array([math.cos(ang), math.sin(ang)])
        yaw, k = rng.uniform(-math.pi, math.pi), int(rng.integers(4))
        c, s = math.cos(yaw), math.sin(yaw)
        poses.append([q[0] - (c * lx[k] - s * ly[k]), q[1] - (s * lx[k] + c * ly[k]), yaw])
    return np.array(poses)


def _body_maps(rng, res):
    """(occ, origin, ext, poses): shapes with W = 1, H = 1 and H, W*H not multiples of 32, negative and large origins,
    different vehicles; then the tie maps"""
    maps = []
    for (W, Hh), origin, ext in (
            ((61, 45), (0, 0), (-1.3 * res, 2.1 * res, -0.7 * res, 0.9 * res)),
            ((1, 37), (-5, 3), (-0.12, 0.21, -0.07, 0.09)),
            ((37, 1), (4, -9), (-0.2 * res, 0.6 * res, -0.1 * res, 0.3 * res)),
            ((11, 97), (-37, 12345), (-0.55 * res, 3.0 * res, -0.74 * res, 0.74 * res)),
            ((41, 33), (4_312_500, -52_917), (-1.3 * res, 2.1 * res, -0.7 * res, 0.9 * res))):
        occ = rng.random((W, Hh)) < 0.15
        near = _near_edge_poses(rng, W, Hh, origin, res, ext, 150)
        x0, y0 = origin[0] * res, origin[1] * res
        rnd = np.stack([x0 + rng.uniform(-0.4, W * res + 0.4, 150), y0 + rng.uniform(-0.4, Hh * res + 0.4, 150),
                        rng.uniform(-math.pi, math.pi, 150)], 1)
        maps.append((occ, origin, ext, np.concatenate([near, rnd])))
    return maps + _tie_maps(res)


def _pool(maps, rng):
    """pack every map's grid in one batch; pool all poses, shuffled across maps.  Returns (bits, table rows, poses,
    map ids)"""
    from headland_trajectory_planning_b200 import ops
    bits, offs = ops.grid_pack_batch([m[0] for m in maps])
    poses = np.concatenate([m[3] for m in maps])
    ids = np.concatenate([np.full(len(m[3]), k, dtype=np.int32) for k, m in enumerate(maps)])
    perm = rng.permutation(len(poses))
    return bits, offs, poses[perm], ids[perm]


@pytest.mark.gpu
@pytest.mark.parametrize("res", [0.1, 0.05, 0.3, 0.25])
def test_body_batch_exact_and_equal_to_single_calls(built_library, res):
    from headland_trajectory_planning_b200 import ops
    rng = np.random.default_rng(int(res * 1000) + 1)
    maps = _body_maps(rng, res)
    bits, offs, poses, ids = _pool(maps, rng)
    table = [(o, m[0].shape, m[1], m[2], None) for o, m in zip(offs, maps)]
    got = ops.grid_footprint_check_batch(bits, table, res, poses, map_id=ids).cpu().numpy().astype(bool)
    n_ties = 0
    for k, (occ, origin, ext, _) in enumerate(maps):
        sel = np.nonzero(ids == k)[0]
        want = _k7_shifted_reference(occ, origin, res, poses[sel], ext)
        bad = np.nonzero(got[sel] != want)[0]
        assert len(bad) == 0, (f"res={res} map {k} {occ.shape} at {origin}: {len(bad)} of {len(sel)} differ, first "
                               f"{poses[sel[bad[:3]]].tolist()}")
        single = ops.grid_footprint_check(ops.grid_pack(occ), occ.shape, res, poses[sel], ext, origin=origin)
        assert np.array_equal(single.cpu().numpy().astype(bool), got[sel]), (res, k)
        n_ties += k >= 5
    assert n_ties >= 48 and 0.05 < got.mean() < 0.95


# ------------------------------------------------------------------ implements, exact
@pytest.mark.gpu
@pytest.mark.parametrize("res", [0.1, 0.3])
def test_implements_exact(built_library, res):
    """Vehicles with 0, 1 and 3 implement rectangles in one batch: verdict = body or (pose_idx even and some
    implement), each term from the exact reference; yaw-0 implement edges on fl(i*res) and one ulp either side, odd
    indices there are free; check_aux=False ignores implements."""
    from headland_trajectory_planning_b200 import ops
    rng = np.random.default_rng(int(res * 100) + 7)
    body = (-0.5, 1.2, -0.35, 0.35)
    vehicles = [np.zeros((0, 4)), _exts(MOWER_AUX), _exts(H.SPRAYER_AUX)]
    maps = []                                         # (occ, origin, body, aux, poses, pose_idx)
    for v, aux in enumerate(vehicles):
        W, Hh = 70 + 9 * v, 53
        origin = (-20 + 7 * v, 11 - 5 * v)
        occ = rng.random((W, Hh)) < 0.03
        x0, y0 = origin[0] * res, origin[1] * res
        n = 400
        poses = np.stack([x0 + rng.uniform(0, W * res, n), y0 + rng.uniform(0, Hh * res, n), rng.uniform(-math.pi, math.pi, n)], 1)
        maps.append((occ, origin, body, aux, poses, rng.integers(0, 1000, n).astype(np.int32)))
    # ties: an implement whose right edge x1 = 0 sits, at yaw 0, exactly on px = fl(i*res) or one ulp beside it, with
    # one occupied cell just right (hit iff the edge reaches it) or left of the edge; the body is 1 m further right
    tie_aux = np.array([[-2.5 * res, 0.0, -0.25 * res, 0.25 * res]])
    tie_body = (1.0, 1.5, -0.25 * res, 0.25 * res)
    for i in sorted({i for i in _touch_below(res, 120)[:2] + _ulp_overlap(res, 120)[:2] + [7, 40]}):
        X = i * res
        occ = np.zeros((124, 7), dtype=bool)
        occ[i, 3] = True
        poses = [[X if u == 0 else math.nextafter(X, u * math.inf), 3.5 * res, 0.0] for u in (-1, 0, 1)]
        maps.append((occ, (0, 0), tie_body, tie_aux, np.array(poses * 2), np.array([0, 2, 4, 1, 3, 5], dtype=np.int32)))
    bits, offs = ops.grid_pack_batch([m[0] for m in maps])
    poses = np.concatenate([m[4] for m in maps])
    pidx = np.concatenate([m[5] for m in maps])
    ids = np.concatenate([np.full(len(m[4]), k, dtype=np.int32) for k, m in enumerate(maps)])
    perm = rng.permutation(len(poses))
    poses, pidx, ids = poses[perm], pidx[perm], ids[perm]
    table = [(o, m[0].shape, m[1], m[2], m[3]) for o, m in zip(offs, maps)]
    got = ops.grid_footprint_check_batch(bits, table, res, poses, map_id=ids, pose_idx=pidx, check_aux=True).cpu().numpy().astype(bool)
    body_only = ops.grid_footprint_check_batch(bits, table, res, poses, map_id=ids, pose_idx=pidx).cpu().numpy().astype(bool)
    aux_hits = 0
    for k, (occ, origin, b, aux, _, _) in enumerate(maps):
        sel = np.nonzero(ids == k)[0]
        want_body = _k7_shifted_reference(occ, origin, res, poses[sel], b)
        want_aux = np.zeros(len(sel), dtype=bool)
        for e in aux:
            want_aux |= _k7_shifted_reference(occ, origin, res, poses[sel], tuple(e))
        want = want_body | ((pidx[sel] % 2 == 0) & want_aux)
        assert np.array_equal(got[sel], want), (res, k, poses[sel][got[sel] != want][:3].tolist())
        assert np.array_equal(body_only[sel], want_body), (res, k)
        aux_hits += int((want & ~want_body).sum())
        if k >= 3:                                    # tie map: the even copies hit where the edge reaches the cell
            assert not want_body.any()
            assert not got[sel][pidx[sel] % 2 == 1].any()
            ev = pidx[sel] % 2 == 0
            assert got[sel][ev].any() and not got[sel][ev].all()
    assert aux_hits > 5


# ------------------------------------------------------------------ conservative against K1
@pytest.mark.gpu
def test_batch_conservative_against_k1_with_implements(built_library):
    """The four boundary scenes (sprayer implements) and two config-5 environments (with the mower's implement),
    rasterised at 0.1 and 0.25 m with flags 3 in one call, checked in one grid_check_sweep call: a K1 hit with
    flags 3 | HL_CHECK_AUX implies a grid hit, for 2e5 random poses per scene and the canonical scene's implement
    near-boundary set."""
    import torch
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.env_batch import EnvBatch, EnvRecord
    rng = np.random.default_rng(77)
    recs, extra = [], []
    for kind in ("canonical", "quads", "field40", "utm"):
        o_env, o_car, o_h, rec, min_mag = _scene(kind)
        recs.append(rec)
        extra.append(_make_set(rng, "aux", o_env, o_car, o_h, max(min_mag, 1e-9))[0] if kind == "canonical" else np.zeros((0, 3)))
    for k in (0, 1):
        rec = _config5(k)[0]
        recs.append(EnvRecord(rec.obs, rec.field, rec.body_ext, _exts(MOWER_AUX)))
        extra.append(np.zeros((0, 3)))
    envs = EnvBatch(recs)
    for res in (0.1, 0.25):
        wins = [(e,) + tuple(ops.raster_window(r.field, res, 2.0)) for e, r in enumerate(recs)]
        grids = ops.rasterize(envs, wins, res, 3)
        poses, ids, pidx = [], [], []
        for e, ((_, i0, j0, w, h), rec, near) in enumerate(zip(wins, recs, extra)):
            allr = np.vstack([rec.body_ext[None], rec.aux])
            hull = (allr[:, 0].min(), allr[:, 1].max(), allr[:, 2].min(), allr[:, 3].max())
            lo, hi = (i0 * res, j0 * res), ((i0 + w) * res, (j0 + h) * res)
            p = _poses_in(rng, 200_000, lo, hi, hull)
            q = np.arange(len(p), dtype=np.int32)
            if len(near):
                from oracle import geometry as geo
                c = geo.rect_corners(near, hull)
                inside = (c[..., 0].min(1) > lo[0]) & (c[..., 0].max(1) < hi[0]) & (c[..., 1].min(1) > lo[1]) & (c[..., 1].max(1) < hi[1])
                p = np.concatenate([p, near[inside]])
                q = np.concatenate([q, np.nonzero(inside)[0].astype(np.int32)])       # the set's own path indices
            poses.append(p); pidx.append(q); ids.append(np.full(len(p), e, dtype=np.int32))
        poses, pidx, ids = np.concatenate(poses), np.concatenate(pidx), np.concatenate(ids)
        d_poses, d_ids, d_pidx = (torch.from_numpy(a).cuda() for a in (poses, ids, pidx))
        grid = ops.grid_check_sweep(recs, wins, grids, res, d_poses, map_id=d_ids, pose_idx=d_pidx,
                                    check_aux=True).cpu().numpy().astype(bool)
        k1 = ops.collision_check(envs, d_poses, env_id=d_ids, pose_idx=d_pidx, flags=3 | ops.CHECK_AUX).cpu().numpy().astype(bool)
        k1_body = ops.collision_check(envs, d_poses, env_id=d_ids, pose_idx=d_pidx, flags=3).cpu().numpy().astype(bool)
        miss = np.nonzero(k1 & ~grid)[0]
        assert len(miss) == 0, f"res={res}: K1 hit but grid free at {poses[miss[:3]].tolist()} (maps {ids[miss[:3]].tolist()})"
        assert (k1 & ~k1_body).any() and not grid.all()
        for e in range(len(recs)):
            assert k1[ids == e].any(), (res, e)


# ------------------------------------------------------------------ non-finite, far, bad map ids
@pytest.mark.gpu
def test_non_finite_far_and_bad_map_ids(built_library):
    import torch
    from headland_trajectory_planning_b200 import ops
    res, W, Hh = 0.1, 40, 30
    rng = np.random.default_rng(12)
    border = rng.random((W, Hh)) < 0.3
    border[0, :] = border[-1, :] = border[:, 0] = border[:, -1] = True
    empty = np.zeros((W, Hh), dtype=bool)
    ext = (-0.55, 3.0, -0.74, 0.74)
    bits, offs = ops.grid_pack_batch([empty, border])
    table = [(offs[0], (W, Hh), (0, 0), ext, _exts(MOWER_AUX)), (offs[1], (W, Hh), (0, 0), ext, None)]
    nf = []
    for k in range(3):
        for v in (np.nan, np.inf, -np.inf):
            p = [2.0, 1.5, 0.3]
            p[k] = v
            nf.append(p)
    far = [[x, y, yaw] for x in (-1e12, 1e12, 2.0) for y in (-1e12, 1e12, 1.5) for yaw in (0.0, 1.1) if (x, y) != (2.0, 1.5)]
    far += [[-50.0, 1.5, 0.3], [2.0, 80.0, -2.0], [1e6, -1e6, 0.7]]
    poses = np.array(nf + far + [[2.0, 1.5, 0.3]] * 3)
    n_nf, n_far = len(nf), len(far)
    for m in (0, 1):
        ids = np.full(len(poses), m, dtype=np.int32)
        ids[-2:] = (-1, 2)                            # outside [0, n_maps): hit whatever the grid holds
        got = ops.grid_footprint_check_batch(bits, table, res, poses, map_id=ids, pose_idx=np.zeros(len(poses), np.int32),
                                             check_aux=True).cpu().numpy().astype(bool)
        assert got[:n_nf].all(), f"map {m}: non-finite poses reported free"
        occ = empty if m == 0 else border
        single = ops.grid_footprint_check(ops.grid_pack(occ), (W, Hh), res, poses[n_nf:n_nf + n_far], ext).cpu().numpy().astype(bool)
        assert np.array_equal(got[n_nf:n_nf + n_far], single) and not single.any()
        assert got[-2:].all()
        assert got[-3] == (m == 1)                    # the in-range copy: free on the empty grid, on the border grid not
    d_ids = torch.tensor([0, -1, 2, 1], dtype=torch.int32, device="cuda")
    got = ops.grid_footprint_check_batch(bits, table, res, np.array([[2.0, 1.5, 0.3]] * 4), map_id=d_ids)
    assert got.cpu().tolist() == [0, 1, 1, 1]


# ------------------------------------------------------------------ rejections
@pytest.mark.gpu
def test_rejections_before_launch_and_empty_batches(built_library):
    import torch
    from headland_trajectory_planning_b200 import HeadlandError, _lib, ops
    lib = _lib.load_library()
    ctx, st = _lib.get_ctx(), _lib.stream_ptr()
    res = 0.1
    occ = np.zeros((10, 10), dtype=bool)
    bits, offs = ops.grid_pack_batch([occ, occ])
    ext = (-0.3, 0.3, -0.2, 0.2)
    good = (0, (10, 10), (0, 0), ext, None)
    poses = np.array([[0.5, 0.5, 0.0]] * 4)
    d_poses = torch.from_numpy(poses).cuda()
    out = torch.full((4,), 7, dtype=torch.uint8, device="cuda")
    aux = np.zeros((3, 4))

    def check(maps, res=res, flags=0, pose_idx=None, n_aux=3):
        t = (_lib.HlGridMap * len(maps))()
        for k, (off, w, h, i0, j0, a0, na) in enumerate(maps):
            t[k].bits_offset, t[k].w, t[k].h, t[k].i0, t[k].j0, t[k].aux_first, t[k].n_aux = off, w, h, i0, j0, a0, na
            t[k].body_ext[:] = ext
        rc = lib.hl_grid_footprint_check_batch(ctx, _lib.ptr(bits), bits.numel(), t, len(maps), _lib.dptr(aux), n_aux, res,
                                               None, _lib.ptr(d_poses), _lib.ptr(pose_idx), 4, flags, _lib.ptr(out), st)
        torch.cuda.synchronize()
        assert rc == 0 or bool((out == 7).all()), "a rejected call wrote its output"
        return rc, _lib.last_error()

    ok = (0, 10, 10, 0, 0, 0, 3)
    for bad, name in (((0, 10, 0, 0, 0, 0, 0), "w and h"), ((0, 10, 10, 2**31 - 3, 0, 0, 0), "int32"),
                      ((0, 10, 10, 0, 2**31 - 9, 0, 0), "int32"), ((int(bits.numel()) - 1, 10, 10, 0, 0, 0, 0), "bit slice"),
                      ((-1, 10, 10, 0, 0, 0, 0), "bit slice"), ((0, 10, 10, 0, 0, 2, 2), "implement"),
                      ((0, 10, 10, 0, 0, -1, 1), "implement"), ((0, 10, 10, 0, 0, 0, -1), "implement")):
        rc, msg = check([ok, bad])
        assert rc != 0 and "map 1" in msg and name in msg, msg
    rc, msg = check([(0, 10, 10, 2**31 - 20, 0, 0, 0)], res=1e300)
    assert rc != 0 and "map 0" in msg and "not finite" in msg, msg
    for bad_res in (0.0, -0.1, math.inf, math.nan):
        rc, msg = check([ok], res=bad_res)
        assert rc != 0 and "res" in msg, msg
    idx = torch.zeros(4, dtype=torch.int32, device="cuda")
    for flags in (1, 2, 8, 4 | 1):
        rc, msg = check([ok], flags=flags, pose_idx=idx)
        assert rc != 0 and "flags" in msg, msg
    rc, msg = check([ok], flags=4)
    assert rc != 0 and "HL_CHECK_AUX" in msg and "d_pose_idx" in msg, msg
    assert check([ok], flags=4, pose_idx=idx)[0] == 0
    out.fill_(7)
    # through ops: the same messages, and tensors of another device
    with pytest.raises(HeadlandError, match="map 1"):
        ops.grid_footprint_check_batch(bits, [good, (0, (0, 10), (0, 0), ext, None)], res, poses)
    with pytest.raises(HeadlandError, match="HL_CHECK_AUX"):
        ops.grid_footprint_check_batch(bits, [good], res, poses, check_aux=True)
    with pytest.raises(HeadlandError, match="i0 = .*int32"):
        ops.grid_footprint_check_batch(bits, [(0, (10, 10), (2**31, 0), ext, None)], res, poses)
    with pytest.raises(HeadlandError, match="tensor on cpu"):
        ops.grid_footprint_check_batch(bits, [good], res, torch.from_numpy(poses))
    with pytest.raises(HeadlandError, match="tensor on cpu"):
        ops.grid_pack_batch([torch.from_numpy(occ)])
    if torch.cuda.device_count() > 1:
        with pytest.raises(HeadlandError, match="cuda:1"):
            ops.grid_footprint_check_batch(bits, [good], res, d_poses.to("cuda:1"))
    # empty batches
    assert ops.grid_footprint_check_batch(bits, [good], res, np.zeros((0, 3))).numel() == 0
    t0 = (_lib.HlGridMap * 1)()
    assert lib.hl_grid_footprint_check_batch(ctx, None, 0, t0, 0, None, 0, res, None, None, None, 0, 0, None, st) == 0
    rc = lib.hl_grid_footprint_check_batch(ctx, None, 0, t0, 0, None, 0, res, None, _lib.ptr(d_poses), None, 4, 0, _lib.ptr(out), st)
    assert rc != 0 and "no maps" in _lib.last_error()

    # the pack's table
    src = torch.zeros(300, dtype=torch.uint8, device="cuda")
    dst = torch.full((20,), SENTINEL, dtype=torch.int32, device="cuda")

    def pack(entries, occ_bytes=300, words=20):
        t = (_lib.HlGridPack * max(len(entries), 1))(*[_lib.HlGridPack(*e) for e in entries])
        rc = lib.hl_grid_pack_batch(ctx, _lib.ptr(src), occ_bytes, t, len(entries), _lib.ptr(dst), words, st)
        torch.cuda.synchronize()
        assert bool((dst == SENTINEL).all()) or rc == 0
        return rc, _lib.last_error()

    okp = (0, 0, 10, 10)                                   # 100 cells = 4 words
    for bad, name in (((100, 3, 10, 10), "overlap"), ((100, 4, 0, 10), "w and h"), ((250, 4, 10, 10), "grid bytes"),
                      ((100, 17, 10, 10), "bit slice"), ((-1, 4, 10, 10), "grid bytes")):
        rc, msg = pack([okp, bad])
        assert rc != 0 and ("grids 0 and 1" in msg if name == "overlap" else "grid 1" in msg) and name in msg, msg
    assert pack([], occ_bytes=0, words=0)[0] == 0 and bool((dst == SENTINEL).all())
    assert pack([okp, (100, 4, 10, 10)])[0] == 0


# ------------------------------------------------------------------ mirror
@pytest.mark.gpu
def test_check_poses_on_grid_aux(built_library):
    """utils.occupancy_grid_utils.check_poses_on_grid with aux_check equals the batched call with pose_idx = path index;
    without it, the single-grid call as before."""
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.car_model import CarModel
    from headland_trajectory_planning_b200.utils import occupancy_grid_utils as OG
    rng = np.random.default_rng(21)
    grid = (rng.random((200, 150)) < 0.0015).astype(np.uint8) * 100
    res = 0.1
    f = OG.get_grid_map_features(grid, res)
    car = CarModel(aux_poly_features=H.SPRAYER_AUX, with_aux=True)
    assert len(car.aux_exts) == 3
    path = np.stack([rng.uniform(3, 17, 3000), rng.uniform(3, 12, 3000), rng.uniform(-math.pi, math.pi, 3000)], 1)
    with_aux = OG.check_poses_on_grid(f, car, path, aux_check=True)
    maps = [(0, f.obstacles_boolean.shape, (0, 0), car.body_ext, car.aux_exts)]
    want = ops.grid_footprint_check_batch(f.device_bits, maps, res, path, pose_idx=np.arange(len(path), dtype=np.int32),
                                          check_aux=True)
    body = OG.check_poses_on_grid(f, car, path)
    today = ops.grid_footprint_check(f.device_bits, f.obstacles_boolean.shape, res, path, car.body_ext)
    assert np.array_equal(with_aux.cpu().numpy(), want.cpu().numpy())
    assert np.array_equal(body.cpu().numpy(), today.cpu().numpy())
    a, b = with_aux.cpu().numpy().astype(bool), body.cpu().numpy().astype(bool)
    assert (a >= b).all() and (a & ~b)[0::2].any() and not (a & ~b)[1::2].any() and not b.all()
