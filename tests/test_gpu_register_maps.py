"""Batched map registration (MapMerger.register_maps, mapmerge_icp_register_batch; DESIGN §6f).

Host-only: every error code and key word of the two C functions, the exact workspace arithmetic
and the Python argument errors.  GPU: bit for bit against A separate
mapmerge_extract_transform(prior) + mapmerge_icp_register calls (the registration of each agent
with the same cell list), against oracle/icp_oracle.py within the tolerances of test_icp.py, and
the pipeline maps -> register_maps -> fuse_occupancy -> assign_frontiers on a configs[1] prefix."""
import math
from types import SimpleNamespace

import numpy as np
import pytest

from map_fuse_util import se2, warp_fuse
from merge_util import synth_agent_grid
from oracle import icp_oracle as IO
from oracle import merge_oracle as MO

E_ARG, E_WORKSPACE = -1, -2


@pytest.fixture(scope='module')
def lib():
    from occgrid_b200 import _native
    return _native.lib()


def _err(lib):
    return lib.occgrid_last_error().decode()


# ---- host only ------------------------------------------------------------------------------------
def _align(v):
    return (v + 255) // 256 * 256


def _workspace(n_target, points, A, cw, ch):
    cells = cw * ch
    vbs = (points + 255) // 256 + A
    fixed = 3 * _align((cells + 1) * 4) + 2 * _align(n_target * 8) + _align(n_target * 4) + \
        _align(((cells + 16383) // 16384 + 1) * 4) + _align(A * 328) + _align((A + 1) * 4) + 256
    return fixed + 2 * _align(points * 8) + _align(points * 4) + _align(vbs * 48) + _align(vbs * 16) + _align(vbs * 4)


@pytest.mark.parametrize('n_target,points,A,cw,ch', [(1, 0, 1, 1, 1), (1000, 1, 1, 40, 30), (123457, 654321, 64, 1999, 2001),
                                                     (5, 257, 65535, 3, 7), (2 ** 32 - 2, 2 ** 39, 300, 46341, 46341)])
def test_workspace_arithmetic(lib, n_target, points, A, cw, ch):
    assert lib.mapmerge_icp_register_batch_workspace_bytes(n_target, points, A, cw, ch) == _workspace(n_target, points, A, cw, ch)


@pytest.mark.parametrize('args,key', [((0, 10, 1, 4, 4), 'n_target'), ((2 ** 32 - 1, 10, 1, 4, 4), 'n_target'),
                                      ((10, -1, 1, 4, 4), 'total_source_points'), ((10, 2 ** 39 + 1, 1, 4, 4), 'total_source_points'),
                                      ((10, 10, 0, 4, 4), 'n_agents'), ((10, 10, 65536, 4, 4), 'n_agents'),
                                      ((10, 10, 1, 0, 4), 'cells'), ((10, 10, 1, 4, -1), 'cells'),
                                      ((10, 10, 1, 2 ** 31 - 1, 2 ** 31 - 1), 'overflows size_t')])
def test_workspace_query_rejects(lib, args, key):
    assert lib.mapmerge_icp_register_batch_workspace_bytes(*args) == 0
    assert key in _err(lib)


def _call(lib, **kw):
    a = dict(sx=256, sy=256, off=256, A=2, tx=256, ty=256, n_target=100, min_x=0.0, min_y=0.0, cell=0.25, cw=8, ch=8,
             thr=1.0, it=30, rf=1e-6, rr=1e-6, res=256, ws=256, ws_bytes=1 << 40)
    a.update(kw)
    return lib.mapmerge_icp_register_batch(a['sx'], a['sy'], a['off'], a['A'], a['tx'], a['ty'], a['n_target'], a['min_x'],
                                           a['min_y'], a['cell'], a['cw'], a['ch'], a['thr'], a['it'], a['rf'], a['rr'],
                                           a['res'], a['ws'], a['ws_bytes'], None)


@pytest.mark.parametrize('kw,key', [(dict(sx=None), 'NULL pointer'), (dict(sy=None), 'NULL pointer'), (dict(off=None), 'NULL pointer'),
                                    (dict(tx=None), 'NULL pointer'), (dict(ty=None), 'NULL pointer'), (dict(res=None), 'NULL pointer'),
                                    (dict(ws=None), 'NULL pointer'), (dict(A=0), 'n_agents'), (dict(A=65536), 'n_agents'),
                                    (dict(n_target=0), 'n_target'), (dict(n_target=2 ** 32 - 1), 'n_target'),
                                    (dict(cell=0.0), 'cell'), (dict(cell=math.nan), 'cell'), (dict(cell=math.inf), 'cell'),
                                    (dict(cw=0), 'cells'), (dict(ch=-3), 'cells'),
                                    (dict(cw=2 ** 31 - 1, ch=2 ** 31 - 1), 'overflows size_t'),
                                    (dict(thr=0.0), 'threshold'), (dict(thr=-1.0), 'threshold'), (dict(thr=math.nan), 'threshold'),
                                    (dict(it=-1), 'max_iteration')])
def test_call_rejects(lib, kw, key):
    assert _call(lib, **kw) == E_ARG
    assert key in _err(lib)


def test_short_workspace(lib):
    need = lib.mapmerge_icp_register_batch_workspace_bytes(100, 0, 2, 8, 8)
    assert need == _workspace(100, 0, 2, 8, 8)
    assert _call(lib, ws_bytes=need - 1) == E_WORKSPACE
    assert 'workspace' in _err(lib)
    assert lib.mapmerge_icp_batch_set_max_ctas(-1) == E_ARG and 'ctas' in _err(lib)


def _bare_merger():
    """A MapMerger whose argument checks can run without a device (they come before any launch)."""
    from occgrid_b200 import map_merger as MM
    m = object.__new__(MM.MapMerger)
    m.device, m._n_global = 'cuda:0', 10
    return m


def test_python_argument_errors():
    from occgrid_b200._native import OccGridError
    m = _bare_merger()
    g = np.zeros((3, 8, 8), np.int8)
    org = np.zeros((3, 2))
    with pytest.raises(ValueError, match='origins'):
        m.register_maps(g, np.zeros((2, 2)), 0.05, None)
    with pytest.raises(ValueError, match='2 priors for 3'):
        m.register_maps(g, org, 0.05, np.tile(np.eye(4), (2, 1, 1)))
    with pytest.raises(ValueError, match='prior 1 must be'):
        m.register_maps(g, org, 0.05, [np.eye(4), np.eye(3), np.eye(4)])
    with pytest.raises(ValueError, match=r'\[A, H, W\]'):
        m.register_maps(np.zeros((8, 8), np.int8), org, 0.05, None)
    bad = np.tile(np.eye(4), (3, 1, 1))
    bad[2, 0, 0] = 1.0 + 1e-8
    with pytest.raises(OccGridError, match='prior 2 is not rigid'):
        m.register_maps(g, org, 0.05, bad)
    bad[2, 0, 0] = math.nan
    with pytest.raises(OccGridError, match='prior 2 has a non-finite'):
        m.register_maps(g, org, 0.05, bad)
    ok = np.tile(np.eye(4), (3, 1, 1))
    ok[1, :2, :2] = [[math.cos(1.0), -math.sin(1.0)], [math.sin(1.0), math.cos(1.0)]]
    win = SimpleNamespace(size=64, window=(0, 0, 32, 64), device='cuda:0')
    with pytest.raises(OccGridError, match='whole grid'):
        m.register_maps(g, org, 0.05, ok, reference=win)
    other = SimpleNamespace(size=64, window=(0, 0, 64, 64), device='cuda:1')
    with pytest.raises(OccGridError, match='cuda:1'):
        m.register_maps(g, org, 0.05, [(0.0, 0.0, 0.1)] * 3, reference=other)
    m._n_global = 0
    with pytest.raises(OccGridError, match='global cloud is empty'):
        m.register_maps(g, org, 0.05, None)


# ---- GPU ------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def gpu():
    torch = pytest.importorskip('torch')
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper as M
    from occgrid_b200 import map_merger as MM
    return SimpleNamespace(torch=torch, M=M, MM=MM)


def _world(n=320, seed=3):
    """A wall-like world map and agent crops of it (each in its own frame at the world's origin)."""
    return synth_agent_grid(n, seed, occ_segments=60)


def _scene(A, seed, size=96, n_world=320, res=0.05, empty=(), far=()):
    """A crops of one world map: agent a sees the window at (x_a, y_a) cells and maps it in a frame
    whose origin is that window's corner, so its true agent->global transform is the identity with
    origin (ox + x_a res, oy + y_a res).  Priors perturb it by up to 0.1 m and 2 degrees; agents in
    `far` are moved 100 m away (no overlap), agents in `empty` see nothing."""
    world = _world(n_world)
    r = np.random.default_rng(seed)
    ox = oy = -n_world * res / 2
    grids = np.full((A, size, size), -1, np.int8)
    org = np.zeros((A, 2))
    priors = np.zeros((A, 4, 4))
    for a in range(A):
        x0, y0 = (int(v) for v in r.integers(0, n_world - size, 2))
        if a not in empty:
            grids[a] = world[y0:y0 + size, x0:x0 + size]
            grids[a][r.random((size, size)) < 0.02] = -1               # every agent misses a few cells
        org[a] = (ox + x0 * res, oy + y0 * res)
        c = org[a] + size * res / 2                                       # perturb about the map's centre
        d = se2(*r.uniform(-0.1, 0.1, 2), math.radians(r.uniform(-2, 2)))
        priors[a] = se2(c[0], c[1], 0) @ d @ se2(-c[0], -c[1], 0)
        if a in far:
            priors[a] = se2(100.0, 0.0, 0.0) @ priors[a]
    return world, ox, oy, grids, org, priors


def _reference_grid(gpu, world, ox, oy, res=0.05):
    g = gpu.M.OccupancyGrid(world.shape[0], res, ox, oy, lazy_workspace=True)
    g.grid_tensor.copy_(gpu.torch.from_numpy(world))
    g._host_cache = None
    return g


def _ref_cloud(gpu, m, reference):
    """(x, y) device tensors of the reference cloud register_maps uses."""
    if reference is None:
        return m._cloud.x[:m._n_global].clone(), m._cloud.y[:m._n_global].clone()
    x, y = MO.grid_to_points(reference.grid.ravel(), reference.size, reference.size, reference.res, reference.ox, reference.oy)
    return gpu.torch.from_numpy(x).cuda(), gpu.torch.from_numpy(y).cuda()


def _single(gpu, lib, grids, org, res, priors, tx, ty, threshold=1.0, max_iteration=30):
    """Per agent: mapmerge_extract_transform(prior), then mapmerge_icp_register with the cell list
    MapMerger.register builds -> [A, 20]."""
    torch, MM = gpu.torch, gpu.MM
    from occgrid_b200 import _native
    st = torch.cuda.current_stream().cuda_stream
    n_t = tx.numel()
    bb = [tx.min().item(), ty.min().item(), tx.max().item(), ty.max().item()]
    cell = threshold / 4.0
    cw, ch = int((bb[2] - bb[0]) / cell) + 2, int((bb[3] - bb[1]) / cell) + 2
    A, h, w = grids.shape
    out = np.zeros((A, 20))
    cloud = MM._Cloud(h * w + 16, 'cuda')
    last = torch.zeros(1, dtype=torch.int64, device='cuda')
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    ews = torch.empty(lib.mapmerge_extract_workspace_bytes(h * w), dtype=torch.uint8, device='cuda')
    res_d = torch.empty(20, dtype=torch.float64, device='cuda')
    for a in range(A):
        g = torch.from_numpy(np.ascontiguousarray(grids[a])).cuda()
        cloud.count.zero_()
        T = np.ascontiguousarray(priors[a], np.float64)
        _native.check(lib.mapmerge_extract_transform(g.data_ptr(), w, h, res, float(org[a, 0]), float(org[a, 1]), T.ctypes.data,
                                                     cloud.x.data_ptr(), cloud.y.data_ptr(), cloud.capacity, cloud.count.data_ptr(),
                                                     last.data_ptr(), status.data_ptr(), ews.data_ptr(), ews.numel(), st), 'extract')
        k = int(cloud.count.item())
        if k == 0:
            out[a, :16] = np.eye(4).ravel()
            continue
        ws = torch.empty(lib.mapmerge_icp_workspace_bytes(n_t, k, cw, ch), dtype=torch.uint8, device='cuda')
        _native.check(lib.mapmerge_icp_register(cloud.x.data_ptr(), cloud.y.data_ptr(), k, tx.data_ptr(), ty.data_ptr(), n_t,
                                                bb[0], bb[1], cell, cw, ch, threshold, max_iteration, 1e-6, 1e-6,
                                                res_d.data_ptr(), ws.data_ptr(), ws.numel(), st), 'icp')
        out[a] = res_d.cpu().numpy()
    assert int(status.item()) == 0
    return out


def _rows(got):
    return np.concatenate([got.refinement.reshape(-1, 16), got.fitness[:, None], got.inlier_rmse[:, None],
                           got.iterations[:, None].astype(np.float64), got.correspondences[:, None].astype(np.float64)], axis=1)


def _assert_bitwise(got, want):
    rows = _rows(got)
    assert rows.shape == want.shape
    bad = np.flatnonzero((rows.view(np.int64) != want.view(np.int64)).any(axis=1))
    assert bad.size == 0, f'agents {bad[:10]} differ: {rows[bad[0]]} vs {want[bad[0]]}' if bad.size else ''


def _merger_with_cloud(gpu, world, ox, oy, res=0.05):
    """A merger whose global cloud is the world map's occupied cells (the reference None)."""
    m = gpu.MM.MapMerger()
    x, y = MO.grid_to_points(world.ravel(), world.shape[1], world.shape[0], res, ox, oy)
    m._ensure_capacity(x.size + 16)
    m._cloud.x[:x.size].copy_(gpu.torch.from_numpy(x))
    m._cloud.y[:x.size].copy_(gpu.torch.from_numpy(y))
    m._cloud.count.fill_(x.size)
    m._n_global = x.size
    return m


@pytest.mark.gpu
@pytest.mark.parametrize('A,ref_kind', [(1, 'grid'), (2, 'cloud'), (7, 'grid'), (7, 'cloud'), (64, 'grid'), (300, 'cloud')])
def test_batch_equals_single_calls(gpu, lib, A, ref_kind):
    empty = (3, 5) if A >= 7 else ()
    far = (1,) if A >= 2 else ()
    world, ox, oy, grids, org, priors = _scene(A, seed=A, empty=empty, far=far)
    if ref_kind == 'grid':
        m, ref = gpu.MM.MapMerger(), _reference_grid(gpu, world, ox, oy)
    else:
        m, ref = _merger_with_cloud(gpu, world, ox, oy), None
    tx, ty = _ref_cloud(gpu, m, ref)
    got = m.register_maps(gpu.torch.from_numpy(grids).cuda(), org, 0.05, priors, reference=ref)
    want = _single(gpu, lib, grids, org, 0.05, priors, tx, ty)
    _assert_bitwise(got, want)
    for a in empty:
        assert got.iterations[a] == 0 and got.fitness[a] == 0 and got.correspondences[a] == 0
        assert np.array_equal(got.refinement[a], np.eye(4)) and not got.accepted[a]
        assert np.array_equal(got.transformation[a], priors[a])
    for a in far:
        assert got.fitness[a] == 0 and got.iterations[a] == 1 and not got.accepted[a]
    live = [a for a in range(A) if a not in empty and a not in far]
    assert got.accepted[live].all()
    if A >= 7:
        assert len(set(got.iterations[live].tolist())) > 1               # agents converge at different iterations
    acc = got.accepted
    assert np.array_equal(got.transformation[acc], np.matmul(got.refinement[acc], priors[acc]))


@pytest.mark.gpu
@pytest.mark.parametrize('max_iteration', [0, 1])
def test_max_iteration_zero_and_one(gpu, lib, max_iteration):
    world, ox, oy, grids, org, priors = _scene(9, seed=11, empty=(4,), far=(2,))
    m, ref = gpu.MM.MapMerger(), _reference_grid(gpu, world, ox, oy)
    tx, ty = _ref_cloud(gpu, m, ref)
    got = m.register_maps(grids, org, 0.05, priors, reference=ref, max_iteration=max_iteration)
    _assert_bitwise(got, _single(gpu, lib, grids, org, 0.05, priors, tx, ty, max_iteration=max_iteration))
    assert (got.iterations <= max_iteration).all()
    if max_iteration == 0:
        assert np.array_equal(got.refinement, np.tile(np.eye(4), (9, 1, 1)))


@pytest.mark.gpu
def test_grid_size_does_not_change_the_result(gpu, lib):
    """Total virtual blocks below the resident grid (default), and far above a forced grid of 1, 3
    and 7 CTAs: the results are the same bits."""
    world, ox, oy, grids, org, priors = _scene(12, seed=5, empty=(6,), far=(9,))
    m, ref = gpu.MM.MapMerger(), _reference_grid(gpu, world, ox, oy)
    tx, ty = _ref_cloud(gpu, m, ref)
    want = _single(gpu, lib, grids, org, 0.05, priors, tx, ty)
    try:
        for cap in (0, 1, 3, 7):
            assert lib.mapmerge_icp_batch_set_max_ctas(cap) == 0
            _assert_bitwise(m.register_maps(grids, org, 0.05, priors, reference=ref), want)
    finally:
        lib.mapmerge_icp_batch_set_max_ctas(0)


@pytest.mark.gpu
def test_dense_agent_with_more_blocks_than_resident_ctas(gpu, lib):
    """One 2048^2 agent with ~600 k occupied cells (~2 400 virtual blocks, over 5x the CTAs a B200
    keeps resident) next to two small agents."""
    n, res = 2048, 0.05
    r = np.random.default_rng(17)
    dense = np.where(r.random((n, n)) < 0.145, 100, 0).astype(np.int8)
    ox = oy = -n * res / 2
    ref = gpu.M.OccupancyGrid(n, res, ox, oy, lazy_workspace=True)
    ref.grid_tensor.copy_(gpu.torch.from_numpy(dense))
    grids = np.full((3, n, n), -1, np.int8)
    grids[0] = dense
    grids[2, 100:300, 100:300] = dense[100:300, 100:300]
    org = np.tile([[ox, oy]], (3, 1))
    priors = np.stack([se2(0.011, -0.007, 0.0004), se2(0.0, 0.0, 0.0), se2(-0.01, 0.02, -0.0003)])
    m = gpu.MM.MapMerger()
    tx, ty = _ref_cloud(gpu, m, ref)
    got = m.register_maps(grids, org, res, priors, reference=ref, max_iteration=6)
    assert got.correspondences[0] > 444 * 256 * 5 * 0.9
    _assert_bitwise(got, _single(gpu, lib, grids, org, res, priors, tx, ty, max_iteration=6))


@pytest.mark.gpu
def test_against_the_oracle(gpu):
    """A few agents against oracle/icp_oracle.py, with test_icp.py's tolerances."""
    world, ox, oy, grids, org, priors = _scene(4, seed=23)
    m, ref = gpu.MM.MapMerger(), _reference_grid(gpu, world, ox, oy)
    got = m.register_maps(grids, org, 0.05, priors, reference=ref)
    gx, gy = MO.grid_to_points(world.ravel(), world.shape[1], world.shape[0], 0.05, ox, oy)
    for a in range(4):
        lx, ly = MO.grid_to_points(grids[a].ravel(), 96, 96, 0.05, *org[a])
        sx, sy = MO.transform_points(lx, ly, priors[a])
        Tw, fw, rw, iw = IO.registration_icp(sx, sy, gx, gy)
        assert got.correspondences[a] == round(fw * sx.shape[0])
        assert got.fitness[a] == fw and got.iterations[a] == iw
        assert abs(got.inlier_rmse[a] - rw) < 1e-9
        assert np.allclose(got.refinement[a], Tw, atol=1e-9)


# Recovered error of the pipeline test, from the CPU oracle (oracle/icp_oracle.py run on the same
# agent maps, fused reference and priors): all 64 agents are accepted and the worst ends 0.0293 m and
# 6.3e-14 degrees off (the residual is the reference's resampling to 5 cm cells, not the angle).  The
# device follows the oracle to 1e-9 (test_icp.py), so it must stay within these plus 1e-6.
PIPE_ORACLE_M = 0.0294
PIPE_ORACLE_DEG = 6.3e-14


def _pose_error(T, T_true):
    d = np.linalg.inv(T_true) @ T
    return math.hypot(d[0, 3], d[1, 3]), abs(math.atan2(d[1, 0], d[0, 0]))


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', ['tiled', 'global_atomic'])
def test_pipeline_register_fuse_assign(gpu, strategy):
    """configs[1] prefix: 64 agent maps, fused with the true room offsets into the reference; the
    agents are registered from priors off by up to 0.15 m and 3 degrees (about their frame), fused
    with the result and given frontier targets."""
    from agent_maps_util import integrate_packets_agent_maps
    from occgrid_b200 import simulation_tools as st
    M, MM = gpu.M, gpu.MM
    s = st.generate_session(n_agents=64, n_packets=200_000, seed=42)
    z = np.zeros((65, 2))
    geom = dict(size=256, resolution=0.05, origin_x=-4.0, origin_y=-6.4)
    maps = M.AgentGrids(64, strategy=strategy, max_batch=200_000, **geom)
    maps.update_packets(s['packets'], agent_offsets=z)
    want_maps = np.full((64, 256, 256), -1, np.int8)
    integrate_packets_agent_maps(s['packets'], want_maps, -4.0, -6.4, 0.05, agent_offsets=z)
    assert np.array_equal(maps.grids, want_maps)
    tf = np.concatenate([s['agent_offsets'][1:], np.zeros((64, 1))], axis=1)
    truth = np.stack([se2(*t) for t in tf])
    G = s['grid']
    merger = MM.MapMerger()
    reference = M.OccupancyGrid(G['size'], G['resolution'], G['origin_x'], G['origin_y'])
    merger.fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, truth, reference)
    r = np.random.default_rng(1)
    pert = np.stack([r.uniform(-0.15, 0.15, 64), r.uniform(-0.15, 0.15, 64), np.radians(r.uniform(-3, 3, 64))], 1)
    priors = np.stack([truth[a] @ se2(*pert[a]) for a in range(64)])
    reg = merger.register_maps(maps.grids_tensor, maps.origins, maps.res, priors, reference=reference)
    assert reg.accepted.all()
    worst_t = worst_a = 0.0
    for a in np.flatnonzero(reg.accepted):
        e, e0 = _pose_error(reg.transformation[a], truth[a]), _pose_error(priors[a], truth[a])
        assert e[0] < e0[0] and e[1] < e0[1], (a, e, e0)
        worst_t, worst_a = max(worst_t, e[0]), max(worst_a, e[1])
    assert worst_t <= PIPE_ORACLE_M + 1e-6 and math.degrees(worst_a) <= PIPE_ORACLE_DEG + 1e-6
    fused = M.OccupancyGrid(G['size'], G['resolution'], G['origin_x'], G['origin_y'])
    merger.fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, reg.transformation, fused)
    want = warp_fuse(want_maps, maps.origins, 0.05, reg.transformation, G['origin_x'], G['origin_y'], G['resolution'],
                     G['size'], G['size'])
    assert np.array_equal(fused.grid, want)
    ys, xs = np.nonzero(want == 0)
    pick = np.random.default_rng(2).choice(xs.size, 64, replace=False)
    xy = np.stack([G['origin_x'] + (xs[pick] + 0.5) * G['resolution'], G['origin_y'] + (ys[pick] + 0.5) * G['resolution']], 1)
    targets = fused.assign_frontiers(xy)
    assert (targets.cluster >= 0).sum() >= 16
