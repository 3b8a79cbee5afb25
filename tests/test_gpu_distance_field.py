"""Obstacle clearance: the exact squared distance field (OccupancyGrid.distance_field /
occgrid_distance_field), the navigation grid of a robot radius (navigation_grid / occgrid_inflate) and
radius-aware frontier assignment (assign_frontiers / geodesic_distance with robot_radius).

Every GPU case is bit for bit: the EDT against scipy's feature transform (distance_field_util, itself
pinned against a brute-force EDT on the host) or a closed form, the inflation against its NumPy
restatement, and the assignment against frontier_assign_util.assign_reference with the clusters of the
raw grid and the C BFS over the reference navigation grid."""
import math

import numpy as np
import pytest

from distance_field_util import edt_brute, edt_reference, footprint_mask, inflate_reference, max_d2_of
from frontier_assign_util import assert_same, assign_reference, oracle_geodesic, robot_cell
from test_gpu_frontier_assign import centre, last_poses, random_map, room

torch = pytest.importorskip('torch')

MAX_SIDE = 32768


def align(v):
    return (v + 255) // 256 * 256


def layout_bytes(w, h):
    """The workspace layout of distance_field.cu, summed: band masks, band links, d2, stacks."""
    nb = (h + 31) // 32
    return align(4 * w * nb) + align(8 * w * nb) + align(4 * w * h) + align(8 * w * h)


# ---- host only ---------------------------------------------------------------------------------

def _args(**kw):
    a = dict(grid=16, w=8, h=8, res=0.05, max_d2=4, xy=16, A=2, out=16, d2=16, ws=16, ws_bytes=1 << 40)
    a.update(kw)
    return a


def _df_call(lib, a):
    return lib.occgrid_distance_field(a['grid'], a['w'], a['h'], a['d2'], a['ws'], a['ws_bytes'], None)


def _inflate_call(lib, a):
    return lib.occgrid_inflate(a['grid'], a['w'], a['h'], 0.0, 0.0, a['res'], a['max_d2'], a['xy'], a['A'], a['out'],
                               a['ws'], a['ws_bytes'], None)


def test_bad_arguments_host_only():
    from occgrid_b200 import _native
    lib = _native.lib()
    sides = [(dict(w=0), 'width x height'), (dict(h=0), 'width x height'), (dict(w=-1), 'width x height'),
             (dict(w=MAX_SIDE + 1), 'width x height'), (dict(h=MAX_SIDE + 1), 'width x height')]
    for kw, word in [(dict(grid=None), 'NULL pointer'), (dict(d2=None), 'NULL pointer'), (dict(ws=None), 'NULL pointer')] + sides:
        assert _df_call(lib, _args(**kw)) == -1, kw
        assert word in _native.last_error(), (kw, _native.last_error())
    cases = [(dict(grid=None), 'NULL pointer'), (dict(out=None), 'NULL pointer'), (dict(ws=None), 'NULL pointer'),
             (dict(xy=None), 'NULL pointer'), (dict(xy=None, A=65535), 'NULL pointer'),
             (dict(max_d2=-1), 'max_d2'), (dict(max_d2=-(1 << 62)), 'max_d2'),
             (dict(A=-1), 'n_robots'), (dict(A=65536), 'n_robots'),
             (dict(res=0.0), 'resolution'), (dict(res=-0.05), 'resolution'), (dict(res=math.nan), 'resolution'),
             (dict(res=math.inf), 'resolution')] + sides
    for kw, word in cases:
        assert _inflate_call(lib, _args(**kw)) == -1, kw
        assert word in _native.last_error(), (kw, _native.last_error())
    for w, h in ((1, 1), (8, 8), (33, 65), (4099, 77)):
        need = lib.occgrid_distance_field_workspace_bytes(w, h)
        assert _df_call(lib, _args(w=w, h=h, ws_bytes=need - 1)) == -2 and 'workspace too small' in _native.last_error()
        assert _inflate_call(lib, _args(w=w, h=h, ws_bytes=need - 1)) == -2 and 'workspace too small' in _native.last_error()
        assert _inflate_call(lib, _args(w=w, h=h, xy=None, A=0, ws_bytes=need - 1)) == -2


def test_workspace_bytes_host_only():
    from occgrid_b200 import _native
    lib = _native.lib()
    for w, h in ((1, 1), (1, MAX_SIDE), (MAX_SIDE, 1), (3, 3), (63, 64), (65, 33), (1000, 1001), (4096, 4096), (4803, 4803),
                 (16384, 16384), (MAX_SIDE, MAX_SIDE)):
        assert lib.occgrid_distance_field_workspace_bytes(w, h) == layout_bytes(w, h), (w, h)
    assert layout_bytes(MAX_SIDE, MAX_SIDE) == 12 * MAX_SIDE ** 2 + 12 * MAX_SIDE * 1024
    for w, h in ((0, 1), (1, 0), (-5, 8), (MAX_SIDE + 1, 8), (8, MAX_SIDE + 1)):
        assert lib.occgrid_distance_field_workspace_bytes(w, h) == 0
        assert 'width x height' in _native.last_error()


def test_python_argument_errors_host_only():
    from occgrid_b200 import dual_bot_mapper as M
    g = M.OccupancyGrid.__new__(M.OccupancyGrid)     # no device needed: every case fails before any upload
    g.size, g.window, g.res = 16, (0, 0, 16, 16), 0.05
    for bad in (-0.01, -math.inf, math.inf, math.nan):
        with pytest.raises(ValueError, match='robot_radius'):
            g.navigation_grid(bad)
        with pytest.raises(ValueError, match='robot_radius'):
            g.assign_frontiers(np.zeros((1, 2)), robot_radius=bad)
        with pytest.raises(ValueError, match='robot_radius'):
            g.geodesic_distance([0.0, 0.0], robot_radius=bad)
    # fp64 as documented: 0.15 / 0.05 = 2.9999999999999996, so 0.15 m blocks up to d2 = 8, not 9
    assert g._max_d2(0.0, 'x') == 0 and g._max_d2(0.15, 'x') == max_d2_of(0.15, 0.05) == 8
    assert g._max_d2(0.1, 'x') == math.floor((0.1 / 0.05) ** 2) and g._max_d2(1e300, 'x') == 1 << 62
    a = M.AgentGrids.__new__(M.AgentGrids)
    with pytest.raises(M.OccGridError, match='single-map'):
        a.distance_field()
    with pytest.raises(M.OccGridError, match='single-map'):
        a.navigation_grid(0.1)


@pytest.mark.parametrize('seed', range(8))
def test_reference_against_brute_force_host_only(seed):
    """scipy's feature transform, the NumPy inflation and the footprint rule against brute force."""
    rng = np.random.default_rng(seed)
    h, w = int(rng.integers(1, 40)), int(rng.integers(1, 40))
    p = [0.0, 0.003, 0.05, 0.3, 0.7, 0.85, 0.1, 0.02][seed]
    grid = rng.choice(np.array([-1, 0, 50, 51, 100], np.int8), size=(h, w), p=[0.1, 0.88 - p, 0.01, 0.01, p])
    want = edt_brute(grid)
    assert np.array_equal(edt_reference(grid), want)
    xy = rng.uniform(-0.2, 0.05 * max(h, w) + 0.2, (3, 2))
    max_d2 = int(rng.integers(0, 20))
    nav = inflate_reference(grid, max_d2, xy)
    cells = [c for c in (robot_cell(rx, ry, 0.0, 0.0, 0.05, w, h) for rx, ry in xy) if c is not None]
    for y in range(h):
        for x in range(w):
            near = any((x - cx) ** 2 + (y - cy) ** 2 <= max_d2 for cx, cy in cells)
            blocked = grid[y, x] == 0 and 0 <= want[y, x] <= max_d2 and not near
            assert nav[y, x] == (100 if blocked else grid[y, x])


# ---- GPU cases ---------------------------------------------------------------------------------

@pytest.fixture(scope='module')
def M():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper
    return dual_bot_mapper


def c_edt(grid, device_out=False):
    """occgrid_distance_field through the C ABI on a [h, w] grid; guard values around d2 must survive."""
    from occgrid_b200 import _native
    lib = _native.lib()
    h, w = grid.shape
    dev = torch.device('cuda', torch.cuda.current_device())
    d_grid = torch.from_numpy(np.ascontiguousarray(grid, np.int8)).to(dev)
    ws = torch.empty(lib.occgrid_distance_field_workspace_bytes(w, h), dtype=torch.uint8, device=dev)
    guard = 64
    buf = torch.full((w * h + 2 * guard,), 0x5A5A5A5A, dtype=torch.int32, device=dev)
    d2 = buf[guard:guard + w * h]
    _native.check(lib.occgrid_distance_field(d_grid.data_ptr(), w, h, d2.data_ptr(), ws.data_ptr(), ws.numel(),
                                             torch.cuda.current_stream().cuda_stream), 'occgrid_distance_field')
    assert (buf[:guard] == 0x5A5A5A5A).all() and (buf[guard + w * h:] == 0x5A5A5A5A).all()
    d2 = d2.view(h, w)
    return d2 if device_out else d2.cpu().numpy()


def c_inflate(grid, max_d2, xy, res=0.05, ox=0.0, oy=0.0):
    from occgrid_b200 import _native
    lib = _native.lib()
    h, w = grid.shape
    dev = torch.device('cuda', torch.cuda.current_device())
    d_grid = torch.from_numpy(np.ascontiguousarray(grid, np.int8)).to(dev)
    ws = torch.empty(lib.occgrid_distance_field_workspace_bytes(w, h), dtype=torch.uint8, device=dev)
    out = torch.full((h, w), 77, dtype=torch.int8, device=dev)
    xy = np.asarray(xy, np.float64).reshape(-1, 2)
    d_xy = torch.from_numpy(np.ascontiguousarray(xy)).to(dev) if len(xy) else None
    _native.check(lib.occgrid_inflate(d_grid.data_ptr(), w, h, ox, oy, res, int(max_d2), d_xy.data_ptr() if len(xy) else None,
                                      len(xy), out.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream),
                  'occgrid_inflate')
    return out.cpu().numpy()


def density_grid(rng, h, w, density):
    if density == 'none':
        return np.zeros((h, w), np.int8)
    if density == 'one':
        g = np.zeros((h, w), np.int8)
        g[int(rng.integers(0, h)), int(rng.integers(0, w))] = 100
        return g
    if density == 'all':
        return np.full((h, w), 100, np.int8)
    return np.where(rng.random((h, w)) < density, 100, rng.choice(np.array([-1, 0], np.int8), size=(h, w))).astype(np.int8)


SMALL_SHAPES = [(1, 1), (1, 777), (777, 1), (3, 3), (63, 63), (64, 64), (65, 65), (1000, 1001)]
DENSITIES = ['none', 'one', 0.001, 0.1, 0.5, 'all']


@pytest.mark.gpu
@pytest.mark.parametrize('shape', SMALL_SHAPES)
@pytest.mark.parametrize('density', DENSITIES)
def test_edt_shapes_and_densities(M, shape, density):
    rng = np.random.default_rng(16 * SMALL_SHAPES.index(shape) + DENSITIES.index(density))
    grid = density_grid(rng, *shape, density)
    got = c_edt(grid)
    assert np.array_equal(got, edt_reference(grid))
    if density == 'none':
        assert (got == -1).all()
    if density == 'all':
        assert (got == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize('n', [4096, 4803])
@pytest.mark.parametrize('density', ['one', 0.001, 0.1])
def test_edt_large_grids(M, n, density):
    grid = density_grid(np.random.default_rng(n), n, n, density)
    assert np.array_equal(c_edt(grid), edt_reference(grid))


@pytest.mark.gpu
def test_edt_every_int8_value(M):
    """Only cells > 50 are obstacles: 50 is not, 51 is, and so is every value up to 127."""
    rng = np.random.default_rng(3)
    vals = np.arange(-128, 128, dtype=np.int16).astype(np.int8)
    grid = rng.choice(vals, size=(300, 257))
    grid[grid > 50] = 0
    grid[::7, ::5] = rng.choice(vals, size=grid[::7, ::5].shape)
    assert np.array_equal(c_edt(grid), edt_reference(grid))
    for v in range(-128, 128):
        g = np.zeros((5, 9), np.int8)
        g[2, 4] = v
        want = edt_reference(g)
        assert np.array_equal(c_edt(g), want), v
        assert (want[2, 4] == 0) == (v > 50)


@pytest.mark.gpu
def test_edt_walls_with_one_cell_gaps(M):
    n = 257
    grid = np.zeros((n, n), np.int8)
    for x in range(8, n, 16):
        grid[:, x] = 100
        grid[(x * 37) % n, x] = 0
    for y in range(13, n, 32):
        grid[y, :] = 100
        grid[y, (y * 11) % n] = -1
    assert np.array_equal(c_edt(grid), edt_reference(grid))


@pytest.mark.gpu
def test_edt_long_rows_and_columns_closed_form(M):
    for h, w in ((2, MAX_SIDE), (MAX_SIDE, 2)):
        for at_start in (True, False):
            grid = np.zeros((h, w), np.int8)
            oy, ox = (0, 0) if at_start else (h - 1, w - 1)
            grid[oy, ox] = 100
            y, x = np.indices((h, w))
            want = ((x - ox).astype(np.int64) ** 2 + (y - oy).astype(np.int64) ** 2).astype(np.int32)
            assert np.array_equal(c_edt(grid), want), (h, w, at_start)


@pytest.mark.gpu
def test_edt_largest_grid_closed_form(M):
    """32768^2 with one obstacle at (0, 0): d2 = x^2 + y^2, up to 2 * 32767^2, compared on the device."""
    n = MAX_SIDE
    grid = np.zeros((n, n), np.int8)
    grid[0, 0] = 100
    d2 = c_edt(grid, device_out=True)
    del grid
    x = torch.arange(n, device=d2.device, dtype=torch.int64)
    for y0 in range(0, n, 1024):
        y = torch.arange(y0, y0 + 1024, device=d2.device, dtype=torch.int64).view(-1, 1)
        assert torch.equal(d2[y0:y0 + 1024].to(torch.int64), x.view(1, -1) ** 2 + y ** 2), y0
    assert int(d2[-1, -1]) == 2 * 32767 ** 2 == 2_147_352_578


# ---- inflation ---------------------------------------------------------------------------------

def mixed_map(rng, h, w):
    return rng.choice(np.array([-1, 0, 100], np.int8), size=(h, w), p=[0.1, 0.85, 0.05])


@pytest.mark.gpu
def test_inflate_zero_radius_returns_the_grid(M):
    rng = np.random.default_rng(11)
    grid = mixed_map(rng, 301, 203)
    assert np.array_equal(c_inflate(grid, 0, []), grid)
    assert np.array_equal(c_inflate(grid, 0, [(1.0, 1.0), (3.0, 7.0)]), grid)


@pytest.mark.gpu
def test_inflate_huge_radius_blocks_every_free_cell_outside_the_footprints(M):
    rng = np.random.default_rng(12)
    grid = mixed_map(rng, 150, 170)
    outside = [(-1.0, 2.0), (2.0, 1e6), (math.nan, 1.0), (math.inf, 0.5), (1.0, -math.inf)]
    for xy in ([], outside):
        got = c_inflate(grid, 1 << 62, xy)
        assert np.array_equal(got, np.where(grid == 0, 100, grid))
    # a robot inside: its footprint (the whole grid at this radius) keeps every cell
    assert np.array_equal(c_inflate(grid, 1 << 62, [(4.0, 4.0)]), grid)
    got = c_inflate(grid, 200, [(4.0, 4.0)] + outside)
    assert np.array_equal(got, inflate_reference(grid, 200, [(4.0, 4.0)] + outside))


@pytest.mark.gpu
@pytest.mark.parametrize('seed', range(6))
def test_inflate_random_maps_robots_and_overlapping_footprints(M, seed):
    rng = np.random.default_rng(40 + seed)
    h, w = int(rng.integers(20, 700)), int(rng.integers(20, 700))
    grid = mixed_map(rng, h, w)
    res, ox, oy = 0.05, float(rng.uniform(-5, 5)), float(rng.uniform(-5, 5))
    max_d2 = [0, 1, 2, 9, 50, 400][seed]
    A = [0, 1, 3, 64, 300, 7][seed]
    xy = np.stack([ox + rng.uniform(-0.1, 1.1, A) * w * res, oy + rng.uniform(-0.1, 1.1, A) * h * res], axis=1)
    if A >= 3:
        xy[1] = xy[0] + 0.04                            # overlapping footprints
        xy[2] = (math.nan, oy)
    got = c_inflate(grid, max_d2, xy, res, ox, oy)
    assert np.array_equal(got, inflate_reference(grid, max_d2, xy, ox, oy, res))


@pytest.mark.gpu
def test_python_surface_matches_the_c_entries(M):
    rng = np.random.default_rng(5)
    grid = mixed_map(rng, 256, 256)
    g = M.OccupancyGrid(256, 0.05, -3.0, 2.0, lazy_workspace=True)
    g.grid_tensor.copy_(torch.from_numpy(grid))
    assert np.array_equal(g.distance_field(), edt_reference(grid))
    xy = np.array([(-2.0, 4.0), (1.0, 5.0)])
    for r in (0.0, 0.05, 0.1, 0.15, 0.33):
        want = inflate_reference(grid, max_d2_of(r, 0.05), xy, -3.0, 2.0, 0.05)
        assert np.array_equal(g.navigation_grid(r, xy), want)
        assert np.array_equal(g.navigation_grid(r, np.zeros((0, 2))), inflate_reference(grid, max_d2_of(r, 0.05)))
    assert np.array_equal(g.navigation_grid(0.1), inflate_reference(grid, 4))
    assert g.distance_field(to_host=False).dtype == torch.int32 and g.navigation_grid(0.1, to_host=False).dtype == torch.int8


# ---- radius-aware assignment ------------------------------------------------------------------

def radius_reference(grid, ox, oy, res, xy, radius):
    """Clusters of the raw grid, BFS over the reference navigation grid."""
    xy = np.asarray(xy, np.float64).reshape(-1, 2)
    h, w = grid.shape
    nav = inflate_reference(grid, max_d2_of(radius, res), xy, ox, oy, res)

    def field(a):
        return oracle_geodesic(nav, *robot_cell(xy[a, 0], xy[a, 1], ox, oy, res, w, h))
    return assign_reference(grid, ox, oy, res, xy, fields=field), nav


def assert_clearance(grid, xy, ox, oy, res, radius, fields):
    """Every reachable cell of every field outside the footprints keeps d2 > max_d2."""
    max_d2 = max_d2_of(radius, res)
    d2 = edt_reference(grid)
    fp = footprint_mask(grid.shape, xy, ox, oy, res, max_d2)
    for f in fields:
        cells = (f >= 0) & ~fp
        assert ((d2[cells] > max_d2) | (d2[cells] < 0)).all()


def on_grid(M, grid, res=0.05, ox=0.0, oy=0.0):
    g = M.OccupancyGrid(grid.shape[0], res, ox, oy, lazy_workspace=True)
    g.grid_tensor.copy_(torch.from_numpy(np.ascontiguousarray(grid, np.int8)))
    return g


def check_radius(M, grid, xy, radius, res=0.05, ox=0.0, oy=0.0):
    g = on_grid(M, grid, res, ox, oy)
    xy = np.asarray(xy, np.float64).reshape(-1, 2)
    got = g.assign_frontiers(xy, robot_radius=radius)
    want, nav = radius_reference(grid, ox, oy, res, xy, radius)
    assert_same(got, want)
    return g, got, want, nav


@pytest.mark.gpu
def test_radius_zero_is_the_default_call(M):
    rng = np.random.default_rng(21)
    grid = random_map(rng, 300)
    xy = rng.uniform(0, 15, (12, 2))
    g = on_grid(M, grid)
    a, b = g.assign_frontiers(xy), g.assign_frontiers(xy, robot_radius=0)
    for k in ('cluster', 'cost', 'goal', 'costs'):
        assert np.array_equal(getattr(a, k), getattr(b, k))
    assert np.array_equal(a.target_xy.view(np.int64), b.target_xy.view(np.int64))
    assert np.array_equal(g.geodesic_distance(xy[0]), g.geodesic_distance(xy[0], robot_radius=0.0))


@pytest.mark.gpu
def test_one_cell_doorway_closes_at_one_cell(M):
    """Two rooms joined by a 1-cell door: open for a point robot, closed for a radius of one cell."""
    grid = room(40)
    grid[:, 20] = 100
    grid[20, 20] = 0                                   # the door
    grid[10:30, 35:38] = -1                            # the unknown beyond the door: the only frontier
    xy = [centre(5, 20)]
    for radius, reachable in ((0.0, True), (0.049, True), (0.05, False), (0.12, False)):
        g, got, want, nav = check_radius(M, grid, xy, radius)
        assert (got.cluster[0] >= 0) == reachable, radius
        f = g.geodesic_distance(xy[0], robot_radius=radius)
        assert np.array_equal(f, oracle_geodesic(nav, 5, 20))
        assert (f[20, 25] >= 0) == reachable
        assert_clearance(grid, xy, 0.0, 0.0, 0.05, radius, [f])


@pytest.mark.gpu
def test_robot_against_a_wall_escapes_through_its_footprint(M):
    grid = room(60)
    grid[20:40, 45:50] = -1
    xy = [centre(1, 30)]                               # next to the left wall, inside the inflated band
    for radius in (0.1, 0.15, 0.2):
        g, got, want, nav = check_radius(M, grid, xy, radius)
        assert nav[30, 1] == 0 and got.cluster[0] >= 0, radius
        f = g.geodesic_distance(xy[0], robot_radius=radius)
        assert np.array_equal(f, oracle_geodesic(nav, 1, 30))
        assert_clearance(grid, xy, 0.0, 0.0, 0.05, radius, [f])
    # without the footprint rule the robot would be sealed in
    nav = inflate_reference(grid, max_d2_of(0.2, 0.05))
    assert (oracle_geodesic(nav, 1, 30) >= 0).sum() == 1


@pytest.mark.gpu
@pytest.mark.parametrize('case', range(5))
def test_random_maps_with_radius(M, case):
    n, A, radius = [(64, 3, 0.05), (130, 20, 0.1), (300, 64, 0.15), (700, 9, 0.25), (1000, 64, 0.12)][case]
    rng = np.random.default_rng(200 + case)
    grid = random_map(rng, n, p_free=0.85)
    ox, oy = float(rng.uniform(-20, 20)), float(rng.uniform(-20, 20))
    xy = np.stack([ox + rng.uniform(-0.05, 1.05, A) * n * 0.05, oy + rng.uniform(-0.05, 1.05, A) * n * 0.05], axis=1)
    g, got, want, nav = check_radius(M, grid, xy, radius, 0.05, ox, oy)
    fields = [g.geodesic_distance(xy[a], robot_radius=radius) for a in range(min(A, 3))]
    for a, f in enumerate(fields):
        cell = robot_cell(xy[a, 0], xy[a, 1], ox, oy, 0.05, n, n)
        want_f = oracle_geodesic(inflate_reference(grid, max_d2_of(radius, 0.05), xy[a:a + 1], ox, oy, 0.05), *cell) \
            if cell is not None else np.full((n, n), -1, np.int32)
        assert np.array_equal(f, want_f)
    assert_clearance(grid, xy, ox, oy, 0.05, radius,
                     [oracle_geodesic(nav, *robot_cell(x, y, ox, oy, 0.05, n, n)) for x, y in xy
                      if robot_cell(x, y, ox, oy, 0.05, n, n) is not None])


@pytest.mark.gpu
def test_swarm_prefix_with_radius(M):
    """configs[1] prefix: 64 agent maps fused into the 4096^2 map, robots at their last poses."""
    from occgrid_b200 import simulation_tools as st
    from occgrid_b200.map_merger import MapMerger
    s = st.generate_session(n_agents=64, n_packets=200_000, seed=42)
    maps = M.AgentGrids(64, max_batch=200_000, size=256, resolution=0.05, origin_x=-4.0, origin_y=-6.4)
    maps.update_packets(s['packets'], agent_offsets=np.zeros((65, 2)))
    tf = np.concatenate([s['agent_offsets'][1:], np.zeros((64, 1))], axis=1)
    G = s['grid']
    target = M.OccupancyGrid(G['size'], G['resolution'], G['origin_x'], G['origin_y'])
    MapMerger().fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, tf, target)
    xy = last_poses(s['packets'], s['agent_idx'], s['agent_offsets'])
    fused = target.grid
    assert np.array_equal(target.distance_field(), edt_reference(fused))
    radius = 0.15
    got = target.assign_frontiers(xy, robot_radius=radius)
    want, nav = radius_reference(fused, target.ox, target.oy, target.res, xy, radius)
    assert_same(got, want)
    assert np.array_equal(target.navigation_grid(radius, xy), nav)
    fields = [oracle_geodesic(nav, *robot_cell(xy[a, 0], xy[a, 1], target.ox, target.oy, target.res, 4096, 4096))
              for a in (0, 31, 63) if robot_cell(xy[a, 0], xy[a, 1], target.ox, target.oy, target.res, 4096, 4096) is not None]
    assert_clearance(fused, xy, target.ox, target.oy, target.res, radius, fields)
