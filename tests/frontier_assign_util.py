"""Reference of the frontier assignment (occgrid_frontier_assign, DESIGN §6e) for the tests and the
benchmark: geodesic fields from the plain C BFS in tests/geodesic_oracle.c, clusters from the
frontier oracle, and the cost, goal and greedy rule restated in NumPy.

The C file is compiled with gcc into a per-user directory under the system temporary directory,
keyed by the source's hash, so that the repository tree is never written."""
import ctypes as C
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'geodesic_oracle.c')
_lib = None


def lib():
    global _lib
    if _lib is None:
        with open(SRC, 'rb') as f:
            tag = hashlib.sha1(f.read()).hexdigest()[:12]
        out_dir = os.path.join(tempfile.gettempdir(), f'occgrid_geodesic_{os.getuid()}')
        os.makedirs(out_dir, exist_ok=True)
        so = os.path.join(out_dir, f'libgeodesic_{tag}.so')
        if not os.path.exists(so):
            tmp = f'{so}.{os.getpid()}.tmp'
            subprocess.run(['gcc', '-O2', '-std=c11', '-fPIC', '-shared', '-Wall', '-Wextra', '-o', tmp, SRC], check=True)
            os.replace(tmp, so)
        _lib = C.CDLL(so)
        _lib.oracle_geodesic.restype = C.c_int
        _lib.oracle_geodesic.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]
    return _lib


def oracle_geodesic(grid, sx, sy):
    """int32 [H, W] BFS distances from cell (sx, sy) over FREE cells, -1 where unreachable."""
    g = np.ascontiguousarray(grid, np.int8)
    h, w = g.shape
    dist = np.empty((h, w), np.int32)
    rc = lib().oracle_geodesic(g.ctypes.data_as(C.c_void_p), w, h, int(sx), int(sy), dist.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise MemoryError('oracle_geodesic: out of memory')
    return dist


def robot_cell(wx, wy, ox, oy, res, w, h):
    """world_to_grid (int((w - o) / res), truncation) or None outside the grid / not finite."""
    if not (math.isfinite(wx) and math.isfinite(wy)):
        return None
    qx, qy = (wx - ox) / res, (wy - oy) / res
    if not (math.isfinite(qx) and math.isfinite(qy)):
        return None
    gx, gy = int(qx), int(qy)
    return (gx, gy) if 0 <= gx < w and 0 <= gy < h else None


def clusters(grid, ox, oy, res):
    """The frontier oracle's clusters (frontier_centroids() order) and centroids."""
    from oracle import occgrid_oracle as O
    cl = O.cluster_frontiers(O.get_frontiers_fast(grid))
    return cl, [O.cluster_centroid_world(c, ox, oy, res) for c in cl]


def assign_reference(grid, ox, oy, res, robot_xy, fields=None):
    """-> dict(cluster, cost, goal, target_xy, costs, goals [A, K, 2], targets_all = every cluster's
    centroid) by the DESIGN §6e rules.  ``fields``
    (optional): a callable robot index -> its field, else oracle_geodesic is run per robot."""
    grid = np.ascontiguousarray(grid, np.int8)
    h, w = grid.shape
    robot_xy = np.asarray(robot_xy, np.float64).reshape(-1, 2)
    A = robot_xy.shape[0]
    cl, cents = clusters(grid, ox, oy, res)
    K = len(cl)
    costs = np.full((A, K), -1, np.int32)
    goals = np.full((A, K, 2), -1, np.int32)
    if K:
        xs = np.concatenate([np.array([c[0] for c in cc], np.int64) for cc in cl])
        ys = np.concatenate([np.array([c[1] for c in cc], np.int64) for cc in cl])
        starts = np.concatenate([[0], np.cumsum([len(cc) for cc in cl])[:-1]])
        lin = ys * w + xs
    for a in range(A):
        cell = robot_cell(robot_xy[a, 0], robot_xy[a, 1], ox, oy, res, w, h)
        if cell is None or K == 0:
            continue
        field = fields(a) if fields is not None else oracle_geodesic(grid, *cell)
        d = field[ys, xs].astype(np.int64)
        key = np.where(d >= 0, (d << 32) | lin, np.iinfo(np.int64).max)
        best = np.minimum.reduceat(key, starts)
        ok = best != np.iinfo(np.int64).max
        costs[a, ok] = (best[ok] >> 32).astype(np.int32)
        gl = best[ok] & 0xffffffff
        goals[a, ok, 0] = gl % w
        goals[a, ok, 1] = gl // w
    cluster = np.full(A, -1, np.int32)
    cost = np.full(A, -1, np.int32)
    goal = np.full((A, 2), -1, np.int32)
    target = np.full((A, 2), np.nan)
    claimed = np.zeros(K, bool)
    for a in range(A):
        c = np.where((costs[a] >= 0) & ~claimed, costs[a].astype(np.int64), np.iinfo(np.int64).max)
        if K == 0 or c.min() == np.iinfo(np.int64).max:
            continue
        k = int(np.argmin(c))                      # first index of the minimum: ties to the lowest k
        claimed[k] = True
        cluster[a], cost[a], goal[a] = k, costs[a, k], goals[a, k]
        target[a] = cents[k]
    return {'cluster': cluster, 'cost': cost, 'goal': goal, 'target_xy': target, 'costs': costs, 'goals': goals,
            'targets_all': np.asarray(cents, np.float64).reshape(K, 2)}


def assert_same(result, want):
    """Bit-for-bit comparison of a FrontierAssignment with assign_reference's dict."""
    np.testing.assert_array_equal(result.costs, want['costs'])
    np.testing.assert_array_equal(result.cluster, want['cluster'])
    np.testing.assert_array_equal(result.cost, want['cost'])
    np.testing.assert_array_equal(result.goal, want['goal'])
    got, ref = result.target_xy, want['target_xy']
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    assert np.array_equal(got.view(np.int64)[~np.isnan(ref)], ref.view(np.int64)[~np.isnan(ref)])
