"""Mirror of the grid container of ``path_planner/utils/occupancy_grid_utils.py`` without
its ROS / cv2 imports (the reference module cannot be imported outside ROS, :2-8): same
grid layout -- 1-cell free padding, obstacle = cells equal to the map maximum, cell
centres at ``idx*res + res/2`` (:70-101) -- plus the bit-packed device copy the footprint
kernel reads."""
import numpy as np

from .. import ops


class GridMapFeatures:
    def __init__(self):
        self.obstacles_boolean = np.array([])
        self.obstacles_xs = np.array([])
        self.obstacles_ys = np.array([])
        self.obstacle_field_map = None
        self.resolution = None
        self.device_bits = None


def shrink_grid_map(occupancy_map, old_resolution, new_resolution):
    """occupancy_grid_utils.py:43-61 with nearest-neighbour index selection in numpy."""
    if new_resolution < old_resolution:
        return occupancy_map
    w, h = occupancy_map.shape
    rw, rh = int(w * (old_resolution / new_resolution)), int(h * (old_resolution / new_resolution))
    ii = np.minimum((np.arange(rw) * (w / rw)).astype(int), w - 1)
    jj = np.minimum((np.arange(rh) * (h / rh)).astype(int), h - 1)
    return occupancy_map[np.ix_(ii, jj)]


def get_grid_map_features(occupancy_map, resolution, map_2d_position=(0.0, 0.0), upload=True):
    """occupancy_grid_utils.py:70-101."""
    obstacle_value = np.max(occupancy_map)
    padded = np.pad(occupancy_map, 1, mode="constant", constant_values=0)      # padder=0: free border (:77)
    idx = np.where(padded == obstacle_value)
    f = GridMapFeatures()
    f.obstacles_xs = idx[0] * resolution + resolution / 2.0
    f.obstacles_ys = idx[1] * resolution + resolution / 2.0
    f.obstacles_boolean = np.zeros(padded.shape, dtype=bool)
    f.obstacles_boolean[idx] = True
    f.obstacle_field_map = padded
    f.resolution = resolution
    if upload:
        f.device_bits = ops.grid_pack(f.obstacles_boolean)
    return f


def check_poses_on_grid(features, car_model, path, aux_check=False):
    """Grid footprint check (the reference's commented-out
    ``check_path_feasibility_with_grid_map``): uint8 CUDA tensor, 1 = body meets an occupied cell.  With
    ``aux_check`` the implement rectangles count too, at the even indices of ``path`` (car_model.py:58)."""
    poses = np.asarray(path, dtype=np.float64)[:, :3]
    if not aux_check:
        return ops.grid_footprint_check(features.device_bits, features.obstacles_boolean.shape, features.resolution,
                                        poses, car_model.body_ext)
    maps = [(0, features.obstacles_boolean.shape, (0, 0), car_model.body_ext, car_model.aux_exts)]
    return ops.grid_footprint_check_batch(features.device_bits, maps, features.resolution, poses,
                                          pose_idx=np.arange(len(poses), dtype=np.int32), check_aux=True)


def synthetic_grid(n, seed=1, n_rows=None, n_blocks=None):
    """BASELINE config-4 occupancy grid (SURVEY.md 8d), n x n cells of 0.05 m: occupied 1-cell border, tree rows as
    8-cell-wide bars with headland gaps, random 6 x 6 blocks.  Returns (bool grid, goal cell = the free cell nearest
    the centre).  Workload generator of ``bench.py``'s distance-field line and of the grid tests."""
    rng = np.random.default_rng(seed)
    occ = np.zeros((n, n), dtype=bool)
    occ[0, :] = occ[-1, :] = occ[:, 0] = occ[:, -1] = True
    n_rows = n_rows if n_rows is not None else max(2, n // 64)
    gap = max(8, n // 10)
    pitch = max(16, (n - 2 * gap) // n_rows)
    for r in range(n_rows):
        j = gap + r * pitch
        occ[gap:n - gap, j:j + min(8, max(1, pitch // 3))] = True
    n_blocks = n_blocks if n_blocks is not None else max(4, (n * n) // 8192)
    for _ in range(n_blocks):
        a, b = rng.integers(1, n - 7, 2)
        occ[a:a + 6, b:b + 6] = True
    c = n // 2
    free = np.argwhere(~occ)
    goal = tuple(int(v) for v in free[np.argmin(np.abs(free[:, 0] - c) + np.abs(free[:, 1] - c))])
    return occ, goal
