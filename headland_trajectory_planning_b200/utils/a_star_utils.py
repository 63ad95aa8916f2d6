"""Mirror of ``path_planner/utils/a_star_utils.py``'s public entry point backed by the
tiled-wavefront kernel ``hl_distance_field``."""
import numpy as np

from .. import ops

BLOCK_COST = 100


def holonomic_motion_commands():
    return [[-1, 0], [-1, 1], [0, 1], [1, 1], [1, 0], [1, -1], [0, -1], [-1, -1]]


def forward_holonomic_motion_commands():
    return [[-1, 0], [0, 1], [-1, 1], [1, 1], [1, 0]]


def holonomic_costs_with_obstacles(goal_index, obstacles, motion_type="King"):
    """a_star_utils.py:75-142, INCLUDING the reference's index wrap-around on grids whose border is not fully
    occupied (validity is ``abs(index) < dim`` and the occupancy / cost arrays are read and written with Python's
    negative indexing, :49-64,138-140): e.g. a free 8 x 8 grid with goal (1, 1) returns 11.3137... at the goal cell,
    like the reference does.  ``hl_distance_field`` detects the open border and runs the extended-grid formulation."""
    out, _ = ops.distance_field(np.asarray(obstacles), goal_index, motion_type)
    return out.cpu().numpy()


def holonomic_costs_with_obstacles_batch(goal_indices, obstacles, motion_type="King"):
    """``holonomic_costs_with_obstacles`` for many goals in one call (``ops.distance_field_batch``): ``obstacles`` is
    one grid shared by every goal or a sequence of grids, one per goal.  Returns float64 arrays in input order."""
    import torch
    outs, _ = ops.distance_field_batch(obstacles, goal_indices, motion_type)
    if not outs:
        return []
    host = torch.cat([o.reshape(-1) for o in outs]).cpu().numpy()      # one download instead of one per field
    ends = np.cumsum([o.numel() for o in outs])
    return [host[e - o.numel():e].reshape(tuple(o.shape)) for o, e in zip(outs, ends)]
