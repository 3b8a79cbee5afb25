"""NumPy reference of the fused occupancy map (MapMerger.fuse_occupancy / mapmerge_warp_fuse).

It restates the contract of include/occgrid_b200.h in float64, one rounded operation at a time
(NumPy does not contract a*b + c into an FMA):

    bx = (gox + 0.5*g) - tx            by = (goy + 0.5*g) - ty
    c0 = (R00*g)/r   c1 = (R10*g)/r   c2 = ((R00*bx + R10*by) - ox_a)/r
    c3 = (R01*g)/r   c4 = (R11*g)/r   c5 = ((R01*bx + R11*by) - oy_a)/r
    u = (c0*j) + ((c1*i) + c2)         v = (c3*j) + ((c4*i) + c5)
    out[i][j] = max(-1, max over agents with 0 <= u < W and 0 <= v < H of map_a[int(v)][int(u)])
"""
import math

import numpy as np


def se2(tx, ty, theta):
    c, s = math.cos(theta), math.sin(theta)
    T = np.eye(4)
    T[0, 0], T[0, 1], T[0, 3] = c, -s, tx
    T[1, 0], T[1, 1], T[1, 3] = s, c, ty
    return T


def coefficients(T, origin, res, out_ox, out_oy, out_res):
    R00, R01, R10, R11 = float(T[0][0]), float(T[0][1]), float(T[1][0]), float(T[1][1])
    tx, ty = float(T[0][3]), float(T[1][3])
    ox, oy = float(origin[0]), float(origin[1])
    g, r = float(out_res), float(res)
    bx = (float(out_ox) + 0.5 * g) - tx
    by = (float(out_oy) + 0.5 * g) - ty
    return ((R00 * g) / r, (R10 * g) / r, ((R00 * bx + R10 * by) - ox) / r,
            (R01 * g) / r, (R11 * g) / r, ((R01 * bx + R11 * by) - oy) / r)


def _candidates(T, origin, res, hw, out_ox, out_oy, out_res, out_w, out_h, margin=8):
    """Target rows and columns that can hold a covered cell: the agent map's corners taken to the
    global frame, widened by `margin` cells (only an optimisation of the reference)."""
    h, w = hw
    x0, y0 = float(origin[0]), float(origin[1])
    cx = np.array([x0, x0 + w * res, x0, x0 + w * res])
    cy = np.array([y0, y0, y0 + h * res, y0 + h * res])
    T = np.asarray(T, np.float64)
    gx = T[0, 0] * cx + T[0, 1] * cy + T[0, 3]
    gy = T[1, 0] * cx + T[1, 1] * cy + T[1, 3]
    if not (np.isfinite(gx).all() and np.isfinite(gy).all()):
        return None
    j0 = max(int(math.floor((gx.min() - out_ox) / out_res)) - margin, 0)
    j1 = min(int(math.ceil((gx.max() - out_ox) / out_res)) + margin, out_w - 1)
    i0 = max(int(math.floor((gy.min() - out_oy) / out_res)) - margin, 0)
    i1 = min(int(math.ceil((gy.max() - out_oy) / out_res)) + margin, out_h - 1)
    if j0 > j1 or i0 > i1:
        return None
    return i0, i1 + 1, j0, j1 + 1


def warp_fuse(maps, origins, res, transforms, out_ox, out_oy, out_res, out_w, out_h):
    """maps int8 [A, H, W], origins [A, 2], transforms [A, 4, 4] -> int8 [out_h, out_w]."""
    maps = np.asarray(maps, np.int8)
    A, H, W = maps.shape
    out = np.full((out_h, out_w), -1, np.int8)
    for a in range(A):
        box = _candidates(transforms[a], origins[a], res, (H, W), out_ox, out_oy, out_res, out_w, out_h)
        if box is None:
            continue
        i0, i1, j0, j1 = box
        c0, c1, c2, c3, c4, c5 = coefficients(transforms[a], origins[a], res, out_ox, out_oy, out_res)
        j = np.arange(j0, j1, dtype=np.float64)
        i = np.arange(i0, i1, dtype=np.float64)
        u = (c0 * j)[None, :] + ((c1 * i) + c2)[:, None]
        v = (c3 * j)[None, :] + ((c4 * i) + c5)[:, None]
        with np.errstate(invalid='ignore'):
            cov = (u >= 0) & (u < W) & (v >= 0) & (v < H)
        vals = maps[a][v[cov].astype(np.int64), u[cov].astype(np.int64)]
        sub = out[i0:i1, j0:j1]
        sub[cov] = np.maximum(sub[cov], vals)
    return out
