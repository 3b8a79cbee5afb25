"""Frontier assignment (OccupancyGrid.assign_frontiers / occgrid_frontier_assign) and the dense
geodesic field (geodesic_distance / occgrid_geodesic_field).

Every GPU case compares fields, costs, goals, clusters and targets bit for bit with the reference in
frontier_assign_util: the plain C BFS of tests/geodesic_oracle.c, the frontier oracle's clusters and
the cost, goal and greedy rule restated in NumPy.  The C BFS is itself pinned against
scipy.sparse.csgraph on the host."""
import math
import struct
from types import SimpleNamespace

import numpy as np
import pytest

from frontier_assign_util import assert_same, assign_reference, oracle_geodesic, robot_cell

torch = pytest.importorskip('torch')

TILE_BYTES = 64 * 64 * 4


def align(v):
    return (v + 255) // 256 * 256


def layout_bytes(w, h, A, K, pool):
    """The workspace layout of frontier_assign.cu, summed: control words, robot cells, slot and
    mark tables, two worklists, free mask, cost keys, claimed bitmap, tile pool."""
    nt = ((w + 63) // 64) * ((h + 63) // 64)
    parts = [48, 4 * A, 4 * A * nt, 4 * A * nt, 8 * pool, 8 * pool, 8 * h * ((w + 63) // 64), 8 * A * K,
             4 * ((K + 31) // 32), TILE_BYTES * pool]
    return sum(align(p) for p in parts)


# ---- host only ---------------------------------------------------------------------------------

def _assign_args(**kw):
    a = dict(grid=16, w=8, h=8, res=0.05, xy=16, A=2, fxy=16, count=16, label=16, root=16, cent=16, ncl=16, K=4, pool=8,
             cluster=16, cost=16, goal=16, target=16, costs=16, status=16, ws=16, ws_bytes=1 << 40)
    a.update(kw)
    return a


def _assign_call(lib, a):
    return lib.occgrid_frontier_assign(a['grid'], a['w'], a['h'], 0.0, 0.0, a['res'], a['xy'], a['A'], a['fxy'], a['count'],
                                       a['label'], a['root'], a['cent'], a['ncl'], a['K'], a['pool'], a['cluster'], a['cost'],
                                       a['goal'], a['target'], a['costs'], a['status'], None, a['ws'], a['ws_bytes'], None)


def _field_call(lib, a):
    return lib.occgrid_geodesic_field(a['grid'], a['w'], a['h'], 0.0, 0.0, a['res'], a['xy'], a['pool'], a['costs'],
                                      a['status'], None, a['ws'], a['ws_bytes'], None)


def test_bad_arguments_host_only():
    from occgrid_b200 import _native
    lib = _native.lib()
    null = ['grid', 'xy', 'fxy', 'count', 'label', 'root', 'cent', 'ncl', 'cluster', 'cost', 'goal', 'target', 'costs',
            'status', 'ws']
    cases = [(dict(**{k: None}), 'NULL pointer') for k in null]
    cases += [(dict(A=0), 'n_robots'), (dict(A=-3), 'n_robots'), (dict(A=65536), 'n_robots'),
              (dict(w=2), 'width x height'), (dict(h=2), 'width x height'), (dict(w=-1), 'width x height'),
              (dict(w=65536, h=32768), 'width x height'),
              (dict(res=0.0), 'resolution'), (dict(res=-0.1), 'resolution'), (dict(res=math.nan), 'resolution'),
              (dict(res=math.inf), 'resolution'),
              (dict(K=0), 'capacity'), (dict(pool=0), 'capacity'), (dict(pool=-1), 'capacity'), (dict(pool=1 << 31), 'capacity')]
    for kw, word in cases:
        assert _assign_call(lib, _assign_args(**kw)) == -1, kw
        assert word in _native.last_error(), (kw, _native.last_error())
    for kw, word in [(dict(grid=None), 'NULL pointer'), (dict(xy=None), 'NULL pointer'), (dict(costs=None), 'NULL pointer'),
                     (dict(status=None), 'NULL pointer'), (dict(ws=None), 'NULL pointer'), (dict(w=1), 'width x height'),
                     (dict(res=0.0), 'resolution'), (dict(pool=0), 'capacity')]:
        assert _field_call(lib, _assign_args(**kw)) == -1, kw
        assert word in _native.last_error(), (kw, _native.last_error())
    for w, h, A, K, pool in ((8, 8, 2, 4, 8), (3, 3, 1, 1, 1), (4099, 77, 300, 1000, 5000)):
        need = lib.occgrid_frontier_assign_workspace_bytes(w, h, A, K, pool)
        rc = _assign_call(lib, _assign_args(w=w, h=h, A=A, K=K, pool=pool, ws_bytes=need - 1))
        assert rc == -2 and 'workspace too small' in _native.last_error()
        need = lib.occgrid_frontier_assign_workspace_bytes(w, h, 1, 1, pool)
        assert _field_call(lib, _assign_args(w=w, h=h, pool=pool, ws_bytes=need - 1)) == -2
        assert 'workspace too small' in _native.last_error()


def test_workspace_bytes_host_only():
    from occgrid_b200 import _native
    lib = _native.lib()
    for w, h, A, K, pool in ((3, 3, 1, 1, 1), (64, 64, 1, 1, 1), (65, 64, 2, 33, 7), (4096, 4096, 64, 4096, 8192),
                             (2053, 1000, 300, 100, 12345), (8, 8, 65535, 1, 1)):
        assert lib.occgrid_frontier_assign_workspace_bytes(w, h, A, K, pool) == layout_bytes(w, h, A, K, pool)
    for args, word in (((2, 8, 1, 1, 1), 'width x height'), ((8, 8, 0, 1, 1), 'n_robots'), ((8, 8, 1, 0, 1), 'capacity'),
                       ((8, 8, 1, 1, 0), 'capacity')):
        assert lib.occgrid_frontier_assign_workspace_bytes(*args) == 0
        assert word in _native.last_error()
    # the "overflows size_t" check guards 32-bit size_t: with a 64-bit one the largest legal
    # arguments need under 2^51 bytes, and the size is exact
    big = (46340, 46340, 65535, (1 << 31) - 1, (1 << 31) - 1)
    assert lib.occgrid_frontier_assign_workspace_bytes(*big) == layout_bytes(*big) < 1 << 51


def test_python_argument_errors_host_only():
    from occgrid_b200 import dual_bot_mapper as M
    g = M.OccupancyGrid.__new__(M.OccupancyGrid)     # no device needed: every case fails before any upload
    g.size, g.window = 16, (0, 0, 16, 16)
    for bad in (np.zeros((2, 3)), np.zeros(3), np.zeros((0, 2)), np.zeros((65536, 2)), np.zeros((1, 2, 2))):
        with pytest.raises(ValueError, match='robot'):
            g.assign_frontiers(bad)
    with pytest.raises(ValueError, match='robot'):
        g.geodesic_distance([1.0, 2.0, 3.0])
    g.window = (0, 0, 16, 8)
    with pytest.raises(M.OccGridError, match='window'):
        g.assign_frontiers(np.zeros((1, 2)))
    a = M.AgentGrids.__new__(M.AgentGrids)
    for name in ('assign_frontiers', 'geodesic_distance'):
        with pytest.raises(M.OccGridError, match='single-map'):
            getattr(a, name)(np.zeros((1, 2)))


@pytest.mark.parametrize('seed', range(6))
def test_oracle_geodesic_matches_scipy_host_only(seed):
    """The C BFS against scipy's unweighted shortest paths on a directed graph whose edges enter
    FREE cells only, from every kind of source cell."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import shortest_path
    rng = np.random.default_rng(seed)
    h, w = int(rng.integers(1, 23)), int(rng.integers(1, 23))
    grid = rng.choice(np.array([-1, 0, 100], np.int8), size=(h, w), p=[0.15, 0.65, 0.2])
    idx = np.arange(h * w).reshape(h, w)
    src, dst = [], []
    for dy, dx in ((0, 1), (0, -1), (1, 0), (-1, 0)):
        a = idx[max(0, -dy):h - max(0, dy), max(0, -dx):w - max(0, dx)]
        b = idx[max(0, dy):h + min(0, dy), max(0, dx):w + min(0, dx)]
        ok = grid.ravel()[b.ravel()] == 0
        src.append(a.ravel()[ok])
        dst.append(b.ravel()[ok])
    src, dst = np.concatenate(src), np.concatenate(dst)
    graph = coo_matrix((np.ones(len(src)), (src, dst)), shape=(h * w, h * w)).tocsr()
    for _ in range(8):
        sx, sy = int(rng.integers(0, w)), int(rng.integers(0, h))
        d = shortest_path(graph, directed=True, unweighted=True, indices=sy * w + sx)
        want = np.where(np.isinf(d), -1, d).astype(np.int32).reshape(h, w)
        assert np.array_equal(oracle_geodesic(grid, sx, sy), want)
    assert (oracle_geodesic(grid, -1, 0) == -1).all() and (oracle_geodesic(grid, w, 0) == -1).all()


def test_reference_rules_and_target_packets_host_only():
    """The NumPy rule on a hand map, and TARG datagrams from a result."""
    from occgrid_b200 import dual_bot_mapper as M
    grid = np.full((7, 9), -1, np.int8)
    grid[1:6, 1:8] = 0
    grid[1:6, 4] = 100                        # a wall with no door: left and right halves
    xy = [(1.5 * 0.1, 3.5 * 0.1), (6.5 * 0.1, 3.5 * 0.1), (2.5 * 0.1, 3.5 * 0.1), (math.nan, 0.0), (-0.3, 0.1)]
    want = assign_reference(grid, 0.0, 0.0, 0.1, xy)
    assert want['costs'].shape == (5, 2)
    assert want['cluster'].tolist() == [0, 1, -1, -1, -1]
    assert robot_cell(math.nan, 0.0, 0.0, 0.0, 0.1, 9, 7) is None and robot_cell(-0.05, 0.0, 0.0, 0.0, 0.1, 9, 7) == (0, 0)
    res = M.FrontierAssignment(want['cluster'], want['cost'], want['goal'], want['target_xy'], want['costs'], {})
    pk = M.target_packets(res)
    assert sorted(pk) == [1, 2]
    tag, x, y = struct.unpack(M.TARGET_FMT, pk[2])
    assert tag == b'TARG' and (x, y) == tuple(np.float32(want['target_xy'][1]).tolist())


# ---- GPU cases ---------------------------------------------------------------------------------

@pytest.fixture(scope='module')
def M():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper
    return dual_bot_mapper


def on_device(M, grid, res=0.05, ox=0.0, oy=0.0):
    g = M.OccupancyGrid(grid.shape[0], res, ox, oy, lazy_workspace=True)
    g.grid_tensor.copy_(torch.from_numpy(np.ascontiguousarray(grid, np.int8)))
    return g


def check(M, grid, xy, res=0.05, ox=0.0, oy=0.0):
    g = on_device(M, grid, res, ox, oy)
    got = g.assign_frontiers(np.asarray(xy, np.float64).reshape(-1, 2))
    want = assign_reference(grid, ox, oy, res, xy)
    assert_same(got, want)
    return got, want


def centre(x, y, res=0.05, ox=0.0, oy=0.0):
    return ox + (x + 0.5) * res, oy + (y + 0.5) * res


def room(n):
    grid = np.full((n, n), 100, np.int8)
    grid[1:-1, 1:-1] = 0
    return grid


@pytest.mark.gpu
def test_corridor_with_a_door(M):
    grid = room(40)
    grid[:, 20] = 100
    grid[30, 20] = 0                          # the door
    grid[5:10, 35:39] = -1                    # unknown pocket in the right room
    got, _ = check(M, grid, [centre(5, 5)])
    assert got.cluster[0] >= 0 and got.cost[0] > 15 + 25 + 14        # through the door, not through the wall


@pytest.mark.gpu
def test_straight_line_nearest_frontier_behind_a_wall(M):
    grid = room(64)
    grid[:, 30] = 100                         # wall right of the robot; the only door is far down
    grid[60, 30] = 0
    grid[10:13, 33:36] = -1                   # cluster 0: 4 cells away in a straight line, behind the wall
    grid[40:43, 3:6] = -1                     # cluster 1: farther away, same side
    got, want = check(M, grid, [centre(27, 11)])
    rx, ry = centre(27, 11)
    nearest = int(np.argmin(np.hypot(want['targets_all'][:, 0] - rx, want['targets_all'][:, 1] - ry)))
    assert want['costs'].shape[1] > 1
    assert want['targets_all'][nearest][0] > 30 * 0.05 and got.target_xy[0, 0] < 30 * 0.05   # stays on its side


@pytest.mark.gpu
def test_sealed_robot_occupied_unknown_outside_nan_and_shared_cells(M):
    grid = room(50)
    grid[20:30, 20:30] = 100
    grid[22:28, 22:28] = 0                    # sealed cell block, with its own frontier-free inside
    grid[3:6, 40:43] = -1
    grid[40:43, 3:6] = -1
    grid[12, 12] = 100
    grid[14, 14] = -1
    xy = [centre(24, 24), centre(12, 12), centre(14, 14), (-1.0, 0.5), (math.nan, 0.5), (0.5, math.inf),
          centre(2, 2), centre(2, 2), centre(45, 45)]
    got, _ = check(M, grid, xy)
    assert got.cluster[0] == -1 and (got.costs[0] == -1).all() and np.isnan(got.target_xy[0]).all()
    assert got.cluster[1] >= 0 and got.cluster[2] >= 0       # occupied and unknown source cells: 0, then moves on
    assert all(got.cluster[a] == -1 and (got.costs[a] == -1).all() for a in (3, 4, 5))
    assert np.array_equal(got.costs[6], got.costs[7]) and got.cluster[6] != got.cluster[7]


@pytest.mark.gpu
def test_zero_frontiers_and_ties(M):
    got, _ = check(M, room(20), [centre(3, 3), centre(5, 5)])
    assert got.costs.shape == (2, 0) and (got.cluster == -1).all()
    grid = room(41)
    grid[1, 10:13] = -1                       # two clusters at the same path length from the robot
    grid[1, 28:31] = -1
    grid[39, 10:13] = -1
    got, want = check(M, grid, [centre(20, 20), centre(20, 20), centre(5, 20), centre(5, 20), centre(35, 20)])
    assert want['costs'].shape[1] == 3 and (want['costs'][0] == want['costs'][0, 0]).all()
    assert got.cluster.tolist() == [0, 1, 2, -1, -1]     # three-way tie to the lowest k; more robots than clusters
    # goal-cell ties: the cluster's cells at equal distance resolve to the lowest y * W + x
    assert tuple(got.goal[0]) == tuple(want['goals'][0, 0])


def random_map(rng, n, p_free=0.7):
    grid = rng.choice(np.array([-1, 0, 100], np.int8), size=(n, n), p=[(1 - p_free) / 2, p_free, (1 - p_free) / 2])
    for _ in range(max(1, n // 16)):                                     # walls with gaps
        if rng.random() < 0.5:
            grid[int(rng.integers(0, n)), :] = np.where(rng.random(n) < 0.9, 100, grid[0, 0])
        else:
            grid[:, int(rng.integers(0, n))] = np.where(rng.random(n) < 0.9, 100, grid[0, 0])
    return grid


RANDOM_CASES = [(3, 0.2, 1), (5, 0.03, 3), (63, 0.05, 7), (64, 0.1, 2), (65, 0.07, 40), (130, 0.05, 300),
                (200, 0.15, 64), (511, 0.05, 17), (1000, 0.12, 64), (2053, 0.05, 9)]


@pytest.mark.gpu
@pytest.mark.parametrize('case', range(len(RANDOM_CASES)))
def test_random_maps(M, case):
    n, res, A = RANDOM_CASES[case]
    rng = np.random.default_rng(100 + case)
    grid = random_map(rng, n, p_free=0.85 if n > 500 else 0.7)
    ox, oy = float(rng.uniform(-20, 20)), float(rng.uniform(-20, 20))
    xy = np.stack([ox + rng.uniform(-0.05, 1.05, A) * n * res, oy + rng.uniform(-0.05, 1.05, A) * n * res], axis=1)
    got, want = check(M, grid, xy, res, ox, oy)
    if n >= 64:
        assert (want['cluster'] >= 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize('w,h', [(3, 200), (200, 3), (129, 1000), (1000, 70)])
def test_non_square_grids_through_the_c_entry(M, w, h):
    rng = np.random.default_rng(w * 7 + h)
    grid = rng.choice(np.array([-1, 0, 100], np.int8), size=(h, w), p=[0.1, 0.8, 0.1])
    xy = np.stack([rng.uniform(0, w * 0.05, 20), rng.uniform(0, h * 0.05, 20)], axis=1)
    out, status, ws, _ = c_assign(grid, 0.05, xy, tile_pool=20 * ((w + 63) // 64) * ((h + 63) // 64))
    assert status == 0
    want = assign_reference(grid, 0.0, 0.0, 0.05, xy)
    assert_same(out, want)


def c_assign(grid, res, xy, tile_pool, guard=0, kmax=4096):
    """frontiers -> clusters -> occgrid_frontier_assign through the C ABI on a [h, w] grid."""
    from occgrid_b200 import _native
    from occgrid_b200.dual_bot_mapper import FrontierAssignment
    lib = _native.lib()
    h, w = grid.shape
    A = len(xy)
    dev = torch.device('cuda', torch.cuda.current_device())
    st = torch.cuda.current_stream().cuda_stream
    d_grid = torch.from_numpy(np.ascontiguousarray(grid)).to(dev)
    cap = w * h
    fws = torch.empty(lib.occgrid_frontier_workspace_bytes(w * h, cap), dtype=torch.uint8, device=dev)
    fxy = torch.empty((cap, 2), dtype=torch.int32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    fst = torch.zeros(1, dtype=torch.int32, device=dev)
    label, root, size = (torch.empty(cap, dtype=torch.int32, device=dev) for _ in range(3))
    cent = torch.empty((cap, 2), dtype=torch.float64, device=dev)
    ncl = torch.zeros(1, dtype=torch.int64, device=dev)
    _native.check(lib.occgrid_frontiers(d_grid.data_ptr(), w, h, fxy.data_ptr(), cap, cnt.data_ptr(), fst.data_ptr(),
                                        fws.data_ptr(), fws.numel(), st), 'occgrid_frontiers')
    _native.check(lib.occgrid_frontier_clusters(fxy.data_ptr(), cnt.data_ptr(), cap, w, 3, 0.0, 0.0, res, label.data_ptr(),
                                                root.data_ptr(), size.data_ptr(), cent.data_ptr(), ncl.data_ptr(),
                                                fws.data_ptr(), fws.numel(), st), 'occgrid_frontier_clusters')
    need = lib.occgrid_frontier_assign_workspace_bytes(w, h, A, kmax, tile_pool)
    ws = torch.full((need + guard,), 0xA5, dtype=torch.uint8, device=dev)
    d_xy = torch.from_numpy(np.ascontiguousarray(xy, np.float64)).to(dev)
    o = [torch.full((A,), 77, dtype=torch.int32, device=dev) for _ in range(2)]
    goal = torch.full((A, 2), 77, dtype=torch.int32, device=dev)
    target = torch.zeros((A, 2), dtype=torch.float64, device=dev)
    costs = torch.full((A, kmax), 77, dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    stats = torch.zeros(3, dtype=torch.int64, device=dev)
    _native.check(lib.occgrid_frontier_assign(d_grid.data_ptr(), w, h, 0.0, 0.0, res, d_xy.data_ptr(), A, fxy.data_ptr(),
                                              cnt.data_ptr(), label.data_ptr(), root.data_ptr(), cent.data_ptr(), ncl.data_ptr(),
                                              kmax, tile_pool, o[0].data_ptr(), o[1].data_ptr(), goal.data_ptr(),
                                              target.data_ptr(), costs.data_ptr(), status.data_ptr(), stats.data_ptr(),
                                              ws.data_ptr(), need, st), 'occgrid_frontier_assign')
    k = int(ncl.item())
    out = FrontierAssignment(o[0].cpu().numpy(), o[1].cpu().numpy(), goal.cpu().numpy(), target.cpu().numpy(),
                             costs[:, :k].cpu().numpy(), dict(zip(('rounds', 'items', 'tile_slots'), stats.cpu().tolist())))
    return out, int(status.item()), ws[need:].cpu().numpy(), need


@pytest.mark.gpu
def test_pool_overflow_sets_the_status_bit_and_grows_in_python(M):
    rng = np.random.default_rng(9)
    grid = random_map(rng, 700, p_free=0.9)
    xy = np.stack([rng.uniform(0, 35, 5), rng.uniform(0, 35, 5)], axis=1)
    out, status, tail, _ = c_assign(grid, 0.05, xy, tile_pool=3, guard=1 << 16)
    assert status & 1
    assert (tail == 0xA5).all()                                   # nothing beyond the workspace is written
    assert (out.cluster == -1).all() and np.isnan(out.target_xy).all() and out.stats['tile_slots'] <= 3
    g = on_device(M, grid)
    g._fa_sizes['pool'] = 1                                       # start tiny: assign_frontiers grows it
    got = g.assign_frontiers(xy)
    assert got.stats['tile_pool'] > 5 * 16
    assert_same(got, assign_reference(grid, 0.0, 0.0, 0.05, xy))
    g._fa_sizes['kmax'] = 1                                       # fewer cluster columns than clusters: widened
    assert_same(g.assign_frontiers(xy), assign_reference(grid, 0.0, 0.0, 0.05, xy))


def serpentine(n, pitch):
    """Vertical corridors joined alternately at the top and the bottom: one path crosses every tile
    row n / pitch times.  Unknown cells at the far end make the frontier."""
    grid = np.full((n, n), 100, np.int8)
    for i, x in enumerate(range(1, n - 1, pitch)):
        grid[1:n - 1, x] = 0
        if x + pitch < n - 1:
            y = n - 2 if i % 2 == 0 else 1
            grid[y, x:x + pitch + 1] = 0
    grid[n // 2, n - 3:n - 1] = -1
    return grid


def spiral(n, gap):
    grid = np.full((n, n), 100, np.int8)
    x0, y0, x1, y1 = 1, 1, n - 2, n - 2
    while x1 - x0 > 2 * gap and y1 - y0 > 2 * gap:
        grid[y0, x0:x1 + 1] = 0
        grid[y0:y1 + 1, x1] = 0
        grid[y1, x0:x1 + 1] = 0
        grid[y0 + gap:y1 + 1, x0] = 0
        grid[y0 + gap, x0:x0 + gap + 1] = 0
        x0, y0, x1, y1 = x0 + gap, y0 + gap, x1 - gap, y1 - gap
    grid[(y0 + y1) // 2, (x0 + x1) // 2] = -1
    grid[(y0 + y1) // 2, (x0 + x1) // 2 - 1] = -1
    return grid


@pytest.mark.gpu
@pytest.mark.parametrize('shape', ['serpentine', 'spiral'])
def test_long_paths(M, shape):
    n = 1024
    grid = serpentine(n, 8) if shape == 'serpentine' else spiral(n, 4)
    starts = [(1, 1), (1, n - 2), (n // 2, 1)]
    xy = [centre(x, y) for x, y in starts]
    got, want = check(M, grid, xy)
    g = on_device(M, grid)
    for x, y in starts:
        want_f = oracle_geodesic(grid, x, y)
        assert want_f.max() > 50_000
        assert np.array_equal(g.geodesic_distance(centre(x, y)), want_f)
    assert got.stats['rounds'] > 1000


def last_poses(packets, agent_idx, offsets):
    """World position of every agent's last record: its (x, y) in its own frame + its offset."""
    pk = np.asarray(packets, np.uint8)
    A = offsets.shape[0] - 1
    xy = np.full((A, 2), np.nan)
    for a in range(1, A + 1):
        rows = np.nonzero(agent_idx == a)[0]
        if len(rows):
            r = pk[rows[-1]]
            xy[a - 1] = (float(r[5:9].view('<f4')[0]) + offsets[a, 0], float(r[9:13].view('<f4')[0]) + offsets[a, 1])
    return xy


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', ['tiled', 'global_atomic'])
def test_golden_dual_session_end_to_end(M, strategy):
    from conftest import normalise_datagrams, session_packets
    from occgrid_b200.map_merger import MapMerger
    pk, _ = session_packets(time_sorted=True)
    maps = M.AgentGrids(2, strategy=strategy, size=200, resolution=0.05, origin_x=-5.0, origin_y=-5.0)
    maps.update_packets(pk)
    tf = [(0.0, 0.0, 0.0), (-2.5, 0.0, 0.0)]
    target = M.OccupancyGrid(300, 0.05, -10.0, -7.5)
    MapMerger().fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, tf, target)
    arr, _ = normalise_datagrams(pk)
    xy = last_poses(arr, arr[:, 4].astype(np.int32), np.array([[0.0, 0.0], [0.0, 0.0], [-2.5, 0.0]]))
    got = target.assign_frontiers(xy)
    assert_same(got, assign_reference(target.grid, -10.0, -7.5, 0.05, xy))
    assert (got.cluster >= 0).all()
    assert len(M.target_packets(got)) == 2


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', ['tiled', 'global_atomic'])
def test_swarm_prefix_end_to_end_and_dense_fields(M, strategy):
    """configs[1] prefix: 64 agents in their own 256^2 frames -> the shared 4096^2 map -> one
    target per robot from its last pose; dense fields of a few robots."""
    from occgrid_b200 import simulation_tools as st
    from occgrid_b200.map_merger import MapMerger
    s = st.generate_session(n_agents=64, n_packets=200_000, seed=42)
    z = np.zeros((65, 2))
    maps = M.AgentGrids(64, strategy=strategy, max_batch=200_000, size=256, resolution=0.05, origin_x=-4.0, origin_y=-6.4)
    maps.update_packets(s['packets'], agent_offsets=z)
    tf = np.concatenate([s['agent_offsets'][1:], np.zeros((64, 1))], axis=1)
    G = s['grid']
    target = M.OccupancyGrid(G['size'], G['resolution'], G['origin_x'], G['origin_y'])
    MapMerger().fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, tf, target)
    xy = last_poses(s['packets'], s['agent_idx'], s['agent_offsets'])
    fused = target.grid
    fields = {}

    def field(a):
        if a not in fields:
            fields[a] = oracle_geodesic(fused, *robot_cell(xy[a, 0], xy[a, 1], target.ox, target.oy, target.res, 4096, 4096))
        return fields[a]

    got = target.assign_frontiers(xy)
    assert_same(got, assign_reference(fused, target.ox, target.oy, target.res, xy, fields=field))
    assert (got.cluster >= 0).sum() >= 32
    if strategy == 'tiled':
        for a in (0, 1, 31, 63):
            assert np.array_equal(target.geodesic_distance(xy[a]), field(a))
