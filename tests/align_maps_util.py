"""Reference of correlative map alignment (mapmerge_align / MapMerger.align_maps, DESIGN §6h) for the
tests, the benchmark and smoke(): the contract restated in NumPy.  The coefficients are Python floats
computed as the header brackets them, every candidate is scored by an integer sum of weight lookups,
and the winner is the largest 64-bit key.  The reference's d2 comes from distance_field_util.edt_reference
(SciPy's EDT) and the clearance rule from max_d2_of."""
import math

import numpy as np

from distance_field_util import edt_reference, max_d2_of  # noqa: F401  (re-exported for the callers)

FAR = 2.0 ** 30


def rotation_table(max_angle, angle_step):
    """(theta [n], rot [n, 2]): θ = m * angle_step for m = 0, 1, -1, 2, -2, ... ±K0, K0 = round(max_angle /
    angle_step), and (math.cos θ, math.sin θ)."""
    k0 = round(float(max_angle) / float(angle_step))
    steps = [0] + [m for i in range(1, k0 + 1) for m in (i, -i)]
    theta = np.array([m * float(angle_step) for m in steps])
    return theta, np.array([[math.cos(t), math.sin(t)] for t in theta], np.float64)


def coefficients(prior, origin, r, width, height, cs, sn, gox, goy, g):
    """(e0, ..., e5) of one (agent, rotation), Python floats, each operation rounded on its own."""
    p = np.asarray(prior, np.float64)
    p00, p01, p03, p10, p11, p13 = (float(p[0, 0]), float(p[0, 1]), float(p[0, 3]), float(p[1, 0]), float(p[1, 1]),
                                    float(p[1, 3]))
    ox, oy, r, g, cs, sn = float(origin[0]), float(origin[1]), float(r), float(g), float(cs), float(sn)
    mx, my = ox + ((0.5 * width) * r), oy + ((0.5 * height) * r)
    ex, ey = -((p00 * mx) + (p01 * my)), -((p10 * mx) + (p11 * my))
    m00, m01 = (cs * p00) - (sn * p10), (cs * p01) - (sn * p11)
    m10, m11 = (sn * p00) + (cs * p10), (sn * p01) + (cs * p11)
    tx, ty = p03 + (((cs - 1.0) * ex) - (sn * ey)), p13 + ((sn * ex) + ((cs - 1.0) * ey))
    bx, by = ox + 0.5 * r, oy + 0.5 * r
    return ((m00 * r) / g, (m01 * r) / g, ((((m00 * bx) + (m01 * by)) + tx) - float(gox)) / g,
            (m10 * r) / g, (m11 * r) / g, ((((m10 * bx) + (m11 * by)) + ty) - float(goy)) / g)


def agent_points(grid):
    """(u, v) float64 of the occupied cells (> 50), row-major."""
    v, u = np.nonzero(np.asarray(grid, np.int8) > 50)
    return u.astype(np.float64), v.astype(np.float64)


def project(e, u, v):
    """(j, i, valid): the reference cell of every point, floor of X and Y; valid is False where |X| or
    |Y| >= 2^30 or NaN (such a point contributes nothing)."""
    X = e[0] * u + (e[1] * v + e[2])
    Y = e[3] * u + (e[4] * v + e[5])
    with np.errstate(invalid='ignore'):
        valid = (np.abs(X) < FAR) & (np.abs(Y) < FAR)
    j = np.where(valid, np.floor(np.where(valid, X, 0.0)), 0).astype(np.int64)
    i = np.where(valid, np.floor(np.where(valid, Y, 0.0)), 0).astype(np.int64)
    return j, i, valid


def weights(d2, max_d2):
    """int64 [Hr, Wr]: max_d2 + 1 - d2 where 0 <= d2 <= max_d2, else 0."""
    d2 = np.asarray(d2, np.int64)
    return np.where((d2 >= 0) & (d2 <= max_d2), max_d2 + 1 - d2, 0)


def o(v):
    return np.where(v > 0, 2 * v - 1, -2 * v)


def rank(k, dx, dy, rc):
    d = 2 * rc + 1
    return (k * d + o(np.asarray(dy))) * d + o(np.asarray(dx))


def key(score, rnk):
    return (np.asarray(score, np.uint64) << np.uint64(32)) | (np.uint64(2 ** 32 - 1) - np.asarray(rnk, np.uint64))


def score_grid(j, i, valid, w, rc):
    """int64 [2rc+1, 2rc+1] indexed [dy + rc, dx + rc]: the score of every offset."""
    hr, wr = w.shape
    d, pad = 2 * rc + 1, 2 * rc + 1
    keep = valid & (j >= -rc) & (j < wr + rc) & (i >= -rc) & (i < hr + rc)
    j, i = j[keep], i[keep]
    wp = np.zeros((hr + 2 * pad, wr + 2 * pad), np.int64)
    wp[pad:pad + hr, pad:pad + wr] = w
    win = np.lib.stride_tricks.sliding_window_view(wp, (d, d))
    out = np.zeros((d, d), np.int64)
    for c in range(0, j.size, 2048):
        out += win[i[c:c + 2048] + pad - rc, j[c:c + 2048] + pad - rc].sum(axis=0, dtype=np.int64)
    return out


def score_at(grid, origin, r, prior, d2, gox, goy, g, cs, sn, dx, dy, max_d2):
    """The score of one candidate (rotation (cs, sn), offset (dx, dy))."""
    grid = np.asarray(grid)
    u, v = agent_points(grid)
    e = coefficients(prior, origin, r, grid.shape[1], grid.shape[0], cs, sn, gox, goy, g)
    j, i, valid = project(e, u, v)
    w = weights(d2, max_d2)
    jj, ii = j + dx, i + dy
    inside = valid & (jj >= 0) & (jj < w.shape[1]) & (ii >= 0) & (ii < w.shape[0])
    return int(w[ii[inside], jj[inside]].sum())


def align_reference(grids, origins, r, priors, d2, gox, goy, g, rot, rc, max_d2):
    """int64 [A, 6] rows (score, k, dx, dy, prior_score, n_points) of the exhaustive search."""
    grids = np.asarray(grids)
    A, h, wd = grids.shape
    w = weights(d2, max_d2)
    d = 2 * rc + 1
    off = np.arange(-rc, rc + 1)
    dyy, dxx = np.meshgrid(off, off, indexing='ij')
    out = np.zeros((A, 6), np.int64)
    for a in range(A):
        u, v = agent_points(grids[a])
        if u.size == 0:
            continue
        best, prior_score = None, 0
        for k, (cs, sn) in enumerate(np.asarray(rot, np.float64)):
            e = coefficients(priors[a], origins[a], r, wd, h, cs, sn, gox, goy, g)
            sc = score_grid(*project(e, u, v), w, rc)
            if k == 0:
                prior_score = int(sc[rc, rc])
            keys = key(sc, rank(k, dxx, dyy, rc))
            m = int(keys.max())
            if best is None or m > best:
                best = m
        score, rk = best >> 32, (2 ** 32 - 1) - (best & (2 ** 32 - 1))
        odx, rest = rk % d, rk // d
        ody, k = rest % d, rest // d
        inv = (lambda x: (x + 1) // 2 if x % 2 else -(x // 2))
        out[a] = (score, k, inv(odx), inv(ody), prior_score, u.size)
    return out


def align_brute(grids, origins, r, priors, d2, gox, goy, g, rot, rc, max_d2):
    """The same rows from plain Python loops over points and candidates (pins align_reference)."""
    d2 = np.asarray(d2)
    hr, wr = d2.shape
    A, h, wd = np.asarray(grids).shape
    out = np.zeros((A, 6), np.int64)
    for a in range(A):
        vs, us = np.nonzero(np.asarray(grids[a]) > 50)
        if us.size == 0:
            continue
        best = None
        prior_score = 0
        for k, (cs, sn) in enumerate(rot):
            e = coefficients(priors[a], origins[a], r, wd, h, cs, sn, gox, goy, g)
            cells = []
            for u, v in zip(us.tolist(), vs.tolist()):
                X = e[0] * float(u) + (e[1] * float(v) + e[2])
                Y = e[3] * float(u) + (e[4] * float(v) + e[5])
                if abs(X) < FAR and abs(Y) < FAR:
                    cells.append((math.floor(X), math.floor(Y)))
            for dy in range(-rc, rc + 1):
                for dx in range(-rc, rc + 1):
                    s = 0
                    for j, i in cells:
                        jj, ii = j + dx, i + dy
                        if 0 <= jj < wr and 0 <= ii < hr and 0 <= d2[ii, jj] <= max_d2:
                            s += max_d2 + 1 - int(d2[ii, jj])
                    if k == 0 and dx == 0 and dy == 0:
                        prior_score = s
                    kk = (s << 32) | (2 ** 32 - 1 - int(rank(k, dx, dy, rc)))
                    if best is None or kk > best[0]:
                        best = (kk, s, k, dx, dy)
        out[a] = (best[1], best[2], best[3], best[4], prior_score, us.size)
    return out
