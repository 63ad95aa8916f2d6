"""K6 batch: hl_distance_field_batch / ops.distance_field_batch.  Every field of a batch is bit-identical to the pinned
oracle and to the single-field call on the same grid and goal (wrap-around included), whatever the batch around it;
malformed batches are rejected before anything launches."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import distance_field as DF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_grid_field_layout_matches_header(built_library):
    from headland_trajectory_planning_b200 import _lib
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "headland_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(HlGridField), offsetof(HlGridField, occ_offset),
         offsetof(HlGridField, out_offset), offsetof(HlGridField, w), offsetof(HlGridField, h),
         offsetof(HlGridField, gi), offsetof(HlGridField, gj));
  return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        out = [int(v) for v in subprocess.check_output([exe], text=True).split()]
    F = _lib.HlGridField
    assert out == [ctypes.sizeof(F), F.occ_offset.offset, F.out_offset.offset, F.w.offset, F.h.offset,
                   F.gi.offset, F.gj.offset]


def _mixed_batch(seed):
    """About 40 (grid, goal) pairs: synthetic maps, random grids with free and occupied borders, 1 x N / N x 1 / 1 x 1
    grids, an occupied goal, a goal on the border and a fully occupied grid."""
    rng = np.random.default_rng(seed)
    items = []
    for n in (16, 64, 200, 333):
        items.append(DF.synthetic_grid(n, seed=n))
    for k in range(24):
        w, h = int(rng.integers(3, 41)), int(rng.integers(3, 41))
        occ = rng.random((w, h)) < rng.choice([0.0, 0.1, 0.25])
        if k % 2:
            occ[0, :] = occ[-1, :] = occ[:, 0] = occ[:, -1] = True
        free = np.argwhere(~occ[1:-1, 1:-1]) + 1
        cells = free if len(free) else np.argwhere(np.ones_like(occ))
        items.append((occ, tuple(int(v) for v in cells[rng.integers(len(cells))])))
    for shape, goal in (((1, 37), (0, 5)), ((29, 1), (28, 0)), ((1, 1), (0, 0)), ((1, 2), (0, 1)), ((2, 1), (0, 0))):
        items.append((rng.random(shape) < 0.2, goal))
    occ, goal = DF.synthetic_grid(64, seed=7)
    items.append((occ, (0, 0)))                           # occupied goal on the (occupied) border
    items.append((occ, (0, 17)))                          # goal on the border
    occ2 = occ.copy()
    occ2[goal] = True
    items.append((occ2, goal))                            # occupied goal inside a closed map
    items.append((np.ones((12, 9), dtype=bool), (5, 4)))  # fully occupied grid
    half = DF.synthetic_grid(96, seed=3)
    half[0][0, :] = False
    half[0][:, -1] = False
    items.append(half)                                    # half-open map
    items.append((np.zeros((8, 8), dtype=bool), (1, 1)))  # free map: 11.31 at the goal in King mode
    return items


@pytest.mark.gpu
@pytest.mark.parametrize("motion", ["King", "Pawn"])
def test_batch_equals_oracle_and_single_call(built_library, motion):
    from headland_trajectory_planning_b200 import ops
    items = _mixed_batch(1 if motion == "King" else 2)
    assert len(items) >= 38
    outs, sweeps = ops.distance_field_batch([o for o, _ in items], [g for _, g in items], motion)
    assert len(outs) == len(items) and sweeps > 0
    for k, ((occ, goal), got) in enumerate(zip(items, outs)):
        got = got.cpu().numpy()
        assert got.shape == occ.shape and got.dtype == np.float64
        want = DF.holonomic_costs_with_obstacles(goal, occ, motion)
        assert np.array_equal(np.isinf(want), np.isinf(got)), k
        assert np.array_equal(want, got), k
        single, _ = ops.distance_field(occ, goal, motion)
        assert np.array_equal(single.cpu().numpy(), got), k


@pytest.mark.gpu
def test_one_grid_many_goals(built_library):
    from headland_trajectory_planning_b200 import ops
    from headland_trajectory_planning_b200.utils import a_star_utils
    rng = np.random.default_rng(11)
    closed, _ = DF.synthetic_grid(128, seed=4)
    open_ = rng.random((48, 48)) < 0.15                   # free border cells: every field takes the extended grid
    for occ in (closed, open_):
        free, busy = np.argwhere(~occ), np.argwhere(occ)
        goals = [tuple(int(v) for v in free[rng.integers(len(free))]) for _ in range(56)]
        goals += [tuple(int(v) for v in busy[rng.integers(len(busy))]) for _ in range(8)]
        got = a_star_utils.holonomic_costs_with_obstacles_batch(goals, occ, "King")
        assert len(got) == 64
        for g, d in zip(goals, got):
            single, _ = ops.distance_field(occ, g, "King")
            assert np.array_equal(single.cpu().numpy(), d), g
        assert np.array_equal(got[0], DF.holonomic_costs_with_obstacles(goals[0], occ, "King"))


@pytest.mark.gpu
def test_order_and_determinism(built_library):
    import torch
    from headland_trajectory_planning_b200 import ops
    items = _mixed_batch(3)
    occs = [torch.from_numpy(o.astype(np.uint8)).cuda() for o, _ in items]      # device grids are accepted too
    goals = [g for _, g in items]
    a, sa = ops.distance_field_batch(occs, goals, "King")
    b, sb = ops.distance_field_batch(occs, goals, "King")
    r, _ = ops.distance_field_batch(occs[::-1], goals[::-1], "King")
    assert sa == sb
    for x, y, z in zip(a, b, r[::-1]):
        assert torch.equal(x, y) and torch.equal(x, z)


@pytest.mark.gpu
def test_deep_fields_next_to_shallow_ones(built_library):
    """Two 1024^2 fields (a long frontier) share their launches with 200 fields of 64^2 that finish early."""
    from headland_trajectory_planning_b200 import ops
    items = [DF.synthetic_grid(1024, seed=s) for s in (1, 2)] + [DF.synthetic_grid(64, seed=s) for s in range(200)]
    outs, sweeps = ops.distance_field_batch([o for o, _ in items], [g for _, g in items], "King")
    _, deep = ops.distance_field(*items[0], "King")
    assert sweeps >= deep
    for k, ((occ, goal), got) in enumerate(zip(items, outs)):
        single, _ = ops.distance_field(occ, goal, "King")
        assert np.array_equal(single.cpu().numpy(), got.cpu().numpy()), k


@pytest.mark.gpu
def test_rejections(built_library):
    import torch
    from headland_trajectory_planning_b200 import HeadlandError, _lib, ops
    occ, goal = DF.synthetic_grid(32, seed=1)
    with pytest.raises(HeadlandError, match="field 2"):
        ops.distance_field_batch([occ, occ, occ], [goal, goal, (32, 3)])
    with pytest.raises(HeadlandError, match="field 1"):
        ops.distance_field_batch(occ, [goal, (-1, 0)])
    with pytest.raises(HeadlandError):
        ops.distance_field_batch([occ, occ], [goal])
    with pytest.raises(HeadlandError):
        ops.distance_field_batch(occ, [goal], "Bishop")
    assert ops.distance_field_batch(occ, []) == ([], 0)
    assert ops.distance_field_batch([], []) == ([], 0)

    lib = _lib.load_library()
    d_occ = torch.from_numpy(occ.astype(np.uint8)).cuda()
    d_out = torch.empty(3 * 32 * 32, dtype=torch.float64, device="cuda")

    def call(offsets, out_elems=d_out.numel(), motion=0):
        fields = (_lib.HlGridField * len(offsets))(*[_lib.HlGridField(0, o, 32, 32, goal[0], goal[1]) for o in offsets])
        sweeps = ctypes.c_int32(-1)
        rc = lib.hl_distance_field_batch(_lib.get_ctx(), _lib.ptr(d_occ), d_occ.numel(), fields, len(offsets), motion,
                                         _lib.ptr(d_out), out_elems, ctypes.byref(sweeps), _lib.stream_ptr())
        return rc, _lib.last_error(), sweeps.value

    assert call([0, 1024, 2048])[0] == 0
    rc, msg, _ = call([0, 2048, 1500])
    assert rc != 0 and "fields 1 and 2" in msg
    rc, msg, _ = call([0, 2048 + 1], out_elems=3 * 1024)
    assert rc != 0 and "field 1" in msg
    rc, msg, _ = call([0], motion=2)
    assert rc != 0 and "motion_type" in msg
    rc, _, sweeps = call([])
    assert rc == 0 and sweeps == 0
