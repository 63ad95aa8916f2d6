"""Mirror of ``path_planner/orchard_geometry_environment.py``: same class name,
constructor and ``check_path_feasibility`` signature; geometry is built once as
vertex arrays and lives in HBM, every footprint test runs in ``hl_collision_check``
(no shapely, no CPU predicate)."""
import math

import numpy as np

from . import ops
from .env_batch import EnvBatch, EnvRecord, make_record
from .geometry_host import flat_line_buffer, square_point_buffer, Poly


class OrchardGeometryEnvironment(object):
    NEAR_SIDE = 1
    FAR_SIDE = -1

    def __init__(self, map_tree_rows, obstacles, contour_points=[], tree_width=0.2, headland_width=7,
                 obstacle_dim=0.3):
        self.map_tree_rows = np.asarray(map_tree_rows, dtype=np.float64)
        self.tree_width = tree_width
        self.headland_width = headland_width
        self.obstacle_dim = obstacle_dim
        self.obstacles = obstacles
        self._tree_quads = self.create_row_polygons(tree_width)
        self._obstacle_quads = self.create_obstacle_polygons(obstacles, obstacle_dim)
        self.contour_points = contour_points
        self._field = self.create_field_polygon(headland_width, contour_points)
        # the reference builds its STRtree once here (:31); update_tree_width never
        # rebuilds it, so collision geometry is frozen at construction (Appendix A, 8)
        self._collision_quads = np.array(self._obstacle_quads + self._tree_quads).reshape(-1, 4, 2)
        self._uploads = {}

    # ---- geometry (orchard_geometry_environment.py:277-353, 463-472) -----------
    def create_row_polygons(self, tree_width):
        return [flat_line_buffer(r[0], r[1], tree_width / 2) for r in self.map_tree_rows]

    def create_obstacle_polygons(self, obstacles, obstacle_dim):
        return [square_point_buffer(o[0], o[1], obstacle_dim) for o in obstacles] if len(obstacles) > 0 else []

    def update_tree_width(self, new_tree_width):
        self._tree_quads = self.create_row_polygons(new_tree_width)   # checks keep the old STRtree

    def get_headland_angle(self, side):
        side_idx = 0 if side == self.NEAR_SIDE else 1
        xs = self.map_tree_rows[:, side_idx, 0]
        if np.std(xs) < 0.01:
            return np.pi / 2
        k = np.polyfit(xs, self.map_tree_rows[:, side_idx, 1], deg=1)[0]
        return math.atan(k)

    def get_map_exterior_pts(self, headland_width):
        rows = self.map_tree_rows
        row_width = np.mean(np.diff(rows[:, 0, 1]))
        near_angle = self.get_headland_angle(self.NEAR_SIDE)
        far_angle = self.get_headland_angle(self.FAR_SIDE)
        dnear = abs(headland_width / math.sin(near_angle))
        dfar = abs(headland_width / math.sin(far_angle))
        near = np.array([r[0] for r in rows])
        near[:, 0] -= dnear
        shift = 0 if np.abs(np.sin(near_angle)) < 1e-5 else row_width / np.tan(near_angle)
        hi = np.argmax(near[:, 1]); near[hi, 1] += row_width; near[hi, 0] += shift
        lo = np.argmin(near[:, 1]); near[lo, 1] -= row_width; near[lo, 0] -= shift
        far = np.array([r[1] for r in rows][::-1])
        far[:, 0] += dfar
        shift = 0 if np.abs(np.sin(far_angle)) < 1e-5 else row_width / np.tan(far_angle)
        hi = np.argmax(far[:, 1]); far[hi, 1] += row_width; far[hi, 0] += shift
        lo = np.argmin(far[:, 1]); far[lo, 1] -= row_width; far[lo, 0] -= shift
        return np.concatenate((near, far))

    def create_field_polygon(self, headland_width, contour_points):
        pts = self.get_map_exterior_pts(headland_width) if len(contour_points) == 0 else np.asarray(contour_points, dtype=np.float64)
        if len(pts) > 1 and (pts[0] == pts[-1]).all():
            pts = pts[:-1]
        return np.ascontiguousarray(pts, dtype=np.float64)

    # shapely-like views for plotting / OBCA code
    @property
    def tree_polys(self):
        return [Poly(q) for q in self._tree_quads]

    @property
    def obstacle_polys(self):
        return [Poly(q) for q in self._obstacle_quads]

    @property
    def field_range_poly(self):
        return Poly(self._field)

    def obstacle_quads(self):
        return self._collision_quads

    def field_ring(self):
        return self._field

    # ---- the collision predicate (:423-458) -> GPU -------------------------------
    def _env_batch(self, car_model):
        key = car_model.footprint_key()
        if key not in self._uploads:
            self._uploads[key] = EnvBatch([make_record(self, car_model)])
        return self._uploads[key]

    def pose_flags(self, car_model, path, boundary_check=True, aux_check=False):
        """uint8 CUDA tensor, 1 = infeasible pose."""
        path = np.asarray(path, dtype=np.float64)
        flags = ops.CHECK_OBSTACLES | (ops.CHECK_BOUNDARY if boundary_check else 0)
        pose_idx = None
        if aux_check and len(car_model.aux_exts) > 0:
            flags |= ops.CHECK_AUX
            pose_idx = np.arange(len(path), dtype=np.int32)
        return ops.collision_check(self._env_batch(car_model), path[:, :3], pose_idx=pose_idx, flags=flags)

    def check_path_feasibility(self, car_model, path, boundary_check=True, aux_check=False):
        return not bool(self.pose_flags(car_model, path, boundary_check, aux_check).any().item())

    def get_min_distance_to_boundary(self, car_model, path, with_aux=True):
        """orchard_geometry_environment.py:393-412: smallest signed distance of the swept footprint unions' exterior
        vertices to the field boundary (negative outside) -- K10 ``hl_min_boundary_distance``, a batch of one path."""
        path = np.asarray(path, dtype=np.float64)
        d = ops.min_boundary_distance(self._env_batch(car_model), path[:, :3], np.array([0, len(path)], dtype=np.int64),
                                      with_aux=with_aux)
        return float(d[0].item())

    # ---- occupancy grid (the grid path the reference left commented out, :8,35-43,460-461) -> GPU
    def occupancy_grid(self, res, margin=2.0, flags=ops.CHECK_OBSTACLES | ops.CHECK_BOUNDARY):
        """(uint8 CUDA tensor [w, h], (i0, j0)): K12 raster of the obstacle / tree-row quads and the field polygon on
        the cells that meet the field ring's bounding box grown by ``margin``; cell (i, j) is the closed square
        [fl((i0+i)*res), fl((i0+i+1)*res)] x [fl((j0+j)*res), fl((j0+j+1)*res)], 1 = occupied.  Pass (i0, j0) as the
        ``origin`` of ``ops.grid_footprint_check``.  Needs no car model."""
        if "raster" not in self._uploads:
            self._uploads["raster"] = EnvBatch([EnvRecord(self.obstacle_quads(), self.field_ring(), (0.0, 0.0, 0.0, 0.0))])
        i0, j0, w, h = ops.raster_window(self.field_ring(), res, margin)
        grid = ops.rasterize(self._uploads["raster"], [(0, i0, j0, w, h)], res, flags)[0]
        return grid, (i0, j0)

    # ---- host-side topology helpers used by the orchestration (:49-64, 93-127, 199-248)
    def check_side_of_a_point(self, point):
        row_centers = np.mean(self.map_tree_rows[:, :, :], axis=1)
        epsilon = np.random.uniform(-0.5, 0.5, size=(len(row_centers),))
        self._center_line_coeff = np.polyfit(row_centers[:, 0] + epsilon, row_centers[:, 1], deg=1)
        k, b = self._center_line_coeff[0], self._center_line_coeff[1]
        origin_sign = np.sign(0 * k + b - 0)
        judge = np.sign(point[0] * k + b - point[1])
        return self.NEAR_SIDE if origin_sign == judge else self.FAR_SIDE

    def get_row_ids_between_start_and_end(self, start_pose, end_pose):
        near_xs, near_ys = self.map_tree_rows[:, 0, 0], self.map_tree_rows[:, 0, 1]
        far_xs, far_ys = self.map_tree_rows[:, 1, 0], self.map_tree_rows[:, 1, 1]
        row_id = np.argmin(np.abs(start_pose[1] - near_ys))
        near = abs(start_pose[0] - near_xs[row_id]) < abs(start_pose[0] - far_xs[row_id])
        ys = np.copy(near_ys) if near else np.copy(far_ys)
        xs = np.copy(near_xs) if near else np.copy(far_xs)
        sy, ey = start_pose[1], end_pose[1]
        idx = np.where((ys > ey) & (ys < sy))[0] if sy > ey else np.where((ys > sy) & (ys < ey))[0]
        return xs, ys, idx

    def get_intermediate_contour_points(self, safety_distance, start_point, xs, ys):
        side = self.check_side_of_a_point(start_point)
        offset = -safety_distance if side == self.NEAR_SIDE else safety_distance
        return np.vstack((xs[:] + offset, ys[:])).T

    def get_topology_waypoints(self, start_pose, end_pose, drive_row_offset):
        xs, ys, idx = self.get_row_ids_between_start_and_end(start_pose, end_pose)
        iys, ixs = ys[idx], xs[idx]
        order = np.argsort(np.abs(iys - start_pose[1]))
        contour = self.get_intermediate_contour_points(drive_row_offset, start_pose[:2], ixs[order], iys[order])
        return np.vstack((start_pose[:2], contour, end_pose[:2]))

    def plot_field_geometry(self, plt, color="skyblue", with_range=True):
        for row in self.map_tree_rows:
            plt.plot(row[:, 0], row[:, 1], "*-", c="g")
        for q in self._tree_quads:
            plt.fill(q[:, 0], q[:, 1], color="g", alpha=0.5)
        for q in self._obstacle_quads:
            plt.fill(q[:, 0], q[:, 1], color="orange", alpha=0.9)
        if with_range:
            plt.fill(self._field[:, 0], self._field[:, 1], color=color, alpha=0.5)
