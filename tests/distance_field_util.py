"""Reference of obstacle clearance (occgrid_distance_field / occgrid_inflate, DESIGN §6g) for the tests
and the benchmark: the exact squared EDT from scipy's feature transform, a brute-force EDT that pins
it on small grids, and the inflation and footprint rules restated in NumPy."""
import numpy as np

from frontier_assign_util import robot_cell


def edt_reference(grid):
    """int32 [H, W]: squared distance in cells from every cell to the nearest cell > 50, -1 everywhere
    when there is none.  Formed in int64 from scipy's feature indices: ties may pick another
    obstacle, but the squared distance is unique."""
    from scipy.ndimage import distance_transform_edt
    grid = np.asarray(grid, np.int8)
    obstacle = grid > 50
    if not obstacle.any():
        return np.full(grid.shape, -1, np.int32)
    iy, ix = distance_transform_edt(~obstacle, return_distances=False, return_indices=True)
    y, x = np.indices(grid.shape)
    return ((iy.astype(np.int64) - y) ** 2 + (ix.astype(np.int64) - x) ** 2).astype(np.int32)


def edt_brute(grid):
    """O(N^2) squared EDT over every (cell, obstacle) pair, same conventions."""
    grid = np.asarray(grid, np.int8)
    oy, ox = np.nonzero(grid > 50)
    if len(oy) == 0:
        return np.full(grid.shape, -1, np.int32)
    y, x = np.indices(grid.shape)
    d = (y.reshape(-1, 1).astype(np.int64) - oy) ** 2 + (x.reshape(-1, 1).astype(np.int64) - ox) ** 2
    return d.min(axis=1).reshape(grid.shape).astype(np.int32)


def max_d2_of(robot_radius, res):
    """The documented radius conversion: floor((robot_radius / res) ** 2) in fp64."""
    return int(np.floor((float(robot_radius) / float(res)) ** 2))


def footprint_mask(shape, robot_xy, ox, oy, res, max_d2):
    """bool [H, W]: the cells within max_d2 of some robot's cell (robots outside the grid or at a
    non-finite position have none)."""
    h, w = shape
    mask = np.zeros(shape, bool)
    y, x = np.indices(shape)
    for wx, wy in np.asarray(robot_xy, np.float64).reshape(-1, 2):
        cell = robot_cell(wx, wy, ox, oy, res, w, h)
        if cell is not None:
            mask |= (x.astype(np.int64) - cell[0]) ** 2 + (y.astype(np.int64) - cell[1]) ** 2 <= max_d2
    return mask


def inflate_reference(grid, max_d2, robot_xy=(), ox=0.0, oy=0.0, res=0.05, d2=None):
    """int8 [H, W] navigation grid: OCCUPIED where the cell is FREE, 0 <= d2 <= max_d2 and outside
    every footprint, else the grid's value."""
    grid = np.asarray(grid, np.int8)
    d2 = edt_reference(grid) if d2 is None else d2
    block = (grid == 0) & (d2 >= 0) & (d2.astype(np.int64) <= max_d2)
    block &= ~footprint_mask(grid.shape, robot_xy, ox, oy, res, max_d2)
    return np.where(block, np.int8(100), grid).astype(np.int8)
