"""CPU reference rasteriser for K12 (``hl_env_rasterize``): ``oracle.geometry``'s footprint predicates applied to every
cell square at the identity pose (0, 0, 0), vectorised over cells.

Cell (i, j) of a grid with origin (i0, j0) is the closed square [fl((i0+i)*res), fl((i0+i+1)*res)] x
[fl((j0+j)*res), fl((j0+j+1)*res)].  At yaw 0 numpy's cos and sin are exactly 1 and 0, so ``rect_corners`` and
``to_local`` reproduce the edges bit for bit; the corners are handed in directly and the rectangle extent is an
array of per-cell edges.  Occupied: the square meets a closed obstacle quad (flag 1) or is not contained in the closed
field polygon (flag 2)."""
import numpy as np

from oracle import geometry as geo


def cell_edges(g0, n, res):
    """fl(g*res) for g = g0 .. g0+n (exact integers as float64, one rounded product each)"""
    return (np.arange(n + 1, dtype=np.float64) + float(g0)) * float(res)


def _cells(ex, ey, a, b):
    """edges and corners of the cells of rows a..b-1 (row-major, like the grid)"""
    h = len(ey) - 1
    X0, X1 = np.repeat(ex[a:b], h), np.repeat(ex[a + 1:b + 1], h)
    Y0, Y1 = np.tile(ey[:-1], b - a), np.tile(ey[1:], b - a)
    # vertex order (x0,y1),(x0,y0),(x1,y0),(x1,y1) of car_model.py:102-119
    cor = np.stack([np.stack([X0, Y1], 1), np.stack([X0, Y0], 1), np.stack([X1, Y0], 1), np.stack([X1, Y1], 1)], axis=1)
    return X0, X1, Y0, Y1, cor


def raster_parts(quads, field, i0, j0, w, h, res, chunk=1 << 15):
    """(obstacle part, boundary part): two bool [w, h] arrays, 1 = the cell meets an obstacle quad / is not contained
    in the field polygon.  ``quads`` [n][4][2] counter-clockwise, ``field`` [m][2]."""
    ex, ey = cell_edges(i0, w, res), cell_edges(j0, h, res)
    quads = [np.asarray(q, dtype=np.float64) for q in np.asarray(quads, dtype=np.float64).reshape(-1, 4, 2)]
    field = np.asarray(field, dtype=np.float64).reshape(-1, 2)
    obs = np.zeros((w, h), dtype=bool)
    bnd = np.zeros((w, h), dtype=bool)
    step = max(1, chunk // h)
    for a in range(0, w, step):
        b = min(w, a + step)
        X0, X1, Y0, Y1, cor = _cells(ex, ey, a, b)
        poses = np.zeros((len(X0), 3))
        hit = np.zeros(len(X0), dtype=bool)
        for q in quads:
            hit |= geo.rects_hit_convex(poses, (X0, X1, Y0, Y1), q, cor)
        obs[a:b] = hit.reshape(b - a, h)
        if len(field) == 0:
            bnd[a:b] = True
        else:
            col = lambda v: v[:, None]          # per-cell extent against the (cells, edges) arrays of the edge test
            inside = geo.rects_inside_polygon(poses, (col(X0), col(X1), col(Y0), col(Y1)), field, cor)
            bnd[a:b] = (~inside).reshape(b - a, h)
    return obs, bnd


def combine(parts, flags):
    """uint8 grid of the selected parts, 1 = occupied"""
    obs, bnd = parts
    occ = np.zeros(obs.shape, dtype=bool)
    if flags & 1:
        occ |= obs
    if flags & 2:
        occ |= bnd
    return occ.astype(np.uint8)


def rasterize(quads, field, i0, j0, w, h, res, flags=3):
    """uint8 [w, h] grid of one environment, 1 = occupied"""
    return combine(raster_parts(quads, field, i0, j0, w, h, res), flags)


def cell_square(i0, j0, i, j, res):
    """float64 corners (4, 2) of cell (i, j), counter-clockwise"""
    x0, x1 = (float(i0 + i)) * res, (float(i0 + i) + 1.0) * res
    y0, y1 = (float(j0 + j)) * res, (float(j0 + j) + 1.0) * res
    return np.array([[x0, y0], [x1, y0], [x1, y1], [x0, y1]])
