"""Fused occupancy map (MapMerger.fuse_occupancy / mapmerge_warp_fuse): agent maps resampled into one
target grid under rigid transforms, combined with an int8 max so that free space survives.

Identity and whole-cell cases are checked against expectations built without the coefficient formula
(slices, np.rot90, integer geometry); random SE(2) cases against the NumPy restatement of the
formula in map_fuse_util, bit for bit."""
import math
from types import SimpleNamespace

import numpy as np
import pytest

from map_fuse_util import se2, warp_fuse

torch = pytest.importorskip('torch')

PREFILL = 55            # a target value the fuse never produces from -1/0/100 maps: catches unwritten tiles


def _args(**kw):
    """Valid host-side arguments of mapmerge_warp_fuse with fake device pointers (never launched:
    the cases below fail in the argument checks)."""
    A = kw.pop('A', 2)
    n = min(max(A, 1), 65535)
    a = dict(d_maps=16, A=A, w=8, h=8, res=0.05, org=np.zeros((n, 2)), T=np.tile(np.eye(4), (n, 1, 1)),
             gox=0.0, goy=0.0, g=0.05, ow=8, oh=8, d_out=16, d_ws=16, ws=1 << 20)
    a.update(kw)
    return a


def _call(lib, a):
    org = np.ascontiguousarray(a['org'], np.float64)
    T = np.ascontiguousarray(a['T'], np.float64)
    return lib.mapmerge_warp_fuse(a['d_maps'], a['A'], a['w'], a['h'], a['res'],
                                  org.ctypes.data if a['org'] is not None else None,
                                  T.ctypes.data if a['T'] is not None else None, a['gox'], a['goy'], a['g'],
                                  a['ow'], a['oh'], a['d_out'], a['d_ws'], a['ws'], None)


# ---- host only ---------------------------------------------------------------------------------

def test_bad_arguments_host_only():
    from occgrid_b200 import _native
    lib = _native.lib()
    shear = np.eye(4)
    shear[0, 1] = 0.5
    nan_t = np.eye(4)
    nan_t[0, 3] = math.nan
    inf_t = np.eye(4)
    inf_t[3, 3] = math.inf
    cases = [
        (dict(d_maps=None), 'NULL'), (dict(d_out=None), 'NULL'), (dict(d_ws=None), 'NULL'),
        (dict(org=None), 'NULL'), (dict(T=None), 'NULL'),
        (dict(A=0), 'n_agents'), (dict(A=-1), 'n_agents'), (dict(A=65536), 'n_agents'),
        (dict(w=0), 'size'), (dict(h=-5), 'size'), (dict(ow=0), 'size'), (dict(oh=0), 'size'),
        (dict(res=0.0), 'resolution'), (dict(res=-0.05), 'resolution'), (dict(res=math.inf), 'resolution'),
        (dict(res=math.nan), 'resolution'), (dict(g=0.0), 'resolution'), (dict(g=math.nan), 'resolution'),
        (dict(A=65535, w=(1 << 31) - 1, h=(1 << 31) - 1), 'overflow'),
        (dict(T=np.stack([np.eye(4), nan_t])), 'non-finite'), (dict(T=np.stack([inf_t, np.eye(4)])), 'non-finite'),
        (dict(T=np.stack([np.eye(4), 2 * np.eye(4)])), 'rigid'), (dict(T=np.stack([shear, np.eye(4)])), 'rigid'),
        (dict(T=np.stack([np.eye(4), se2(0, 0, 0.3) * (1 + 1e-8)])), 'rigid'),
    ]
    for kw, word in cases:
        a = _args(**kw)
        assert _call(lib, a) == -1, kw
        assert word in _native.last_error(), (kw, _native.last_error())
    # a workspace below the size asked for: E_WORKSPACE (every argument above passed its check)
    near_rigid = se2(1.0, -2.0, 0.7)
    near_rigid[:2, :2] *= 1 + 1e-12
    for A in (1, 2, 1000):
        need = lib.mapmerge_warp_fuse_workspace_bytes(A, 8, 8)
        T = np.tile(near_rigid, (A, 1, 1))
        assert _call(lib, _args(A=A, org=np.zeros((A, 2)), T=T, ws=need - 1)) == -2
        assert 'workspace' in _native.last_error()


def test_workspace_bytes_host_only():
    from occgrid_b200 import _native
    lib = _native.lib()
    sizes = [lib.mapmerge_warp_fuse_workspace_bytes(a, 4096, 4096) for a in range(1, 2100)]
    assert all(s > 0 for s in sizes) and all(x <= y for x, y in zip(sizes, sizes[1:]))
    assert sizes[1023] >= 1024 * 64
    assert lib.mapmerge_warp_fuse_workspace_bytes(65535, 1, 1) >= 65535 * 64
    for a, w, h, word in ((0, 8, 8, 'n_agents'), (65536, 8, 8, 'n_agents'), (1, 0, 8, 'size'), (1, 8, -1, 'size')):
        assert lib.mapmerge_warp_fuse_workspace_bytes(a, w, h) == 0
        assert word in _native.last_error()


def test_fuse_occupancy_argument_errors_before_launch_host_only():
    from occgrid_b200 import _native
    from occgrid_b200.map_merger import MapMerger, OccGridError
    m = MapMerger.__new__(MapMerger)             # no device needed: every case fails before the launch
    m.device, m._lib, m._ws = torch.device('cuda', 0), _native.lib(), {}
    target = SimpleNamespace(size=16, window=(0, 0, 16, 16), device=torch.device('cuda', 0))
    maps = np.full((2, 8, 8), -1, np.int8)
    org = np.zeros((2, 2))
    with pytest.raises(OccGridError, match='window'):
        m.fuse_occupancy(maps, org, 0.05, None, SimpleNamespace(**dict(vars(target), window=(0, 0, 8, 16))))
    with pytest.raises(OccGridError, match='cuda:1'):
        m.fuse_occupancy(maps, org, 0.05, None, SimpleNamespace(**dict(vars(target), device=torch.device('cuda', 1))))
    for bad in (maps[0], maps[None], np.zeros((0, 8, 8), np.int8), np.zeros((2, 0, 8), np.int8)):
        with pytest.raises(ValueError, match='A, H, W'):
            m.fuse_occupancy(bad, org, 0.05, None, target)
    with pytest.raises(ValueError, match='int8'):
        m.fuse_occupancy(torch.zeros((2, 8, 8)), org, 0.05, None, target)
    with pytest.raises(ValueError, match='origins'):
        m.fuse_occupancy(maps, np.zeros((3, 2)), 0.05, None, target)
    with pytest.raises(ValueError, match='transforms'):
        m.fuse_occupancy(maps, org, 0.05, [(0.0, 0.0, 0.0)], target)


# ---- GPU cases ---------------------------------------------------------------------------------

@pytest.fixture(scope='module')
def M():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper
    return dual_bot_mapper


def fuse(M, maps, origins, res, transforms, size, out_res, gox, goy):
    """fuse_occupancy into a fresh OccupancyGrid pre-filled with PREFILL; -> host int8 [size, size]."""
    from occgrid_b200.map_merger import MapMerger
    target = M.OccupancyGrid(size, out_res, gox, goy, lazy_workspace=True)
    target.grid_tensor.fill_(PREFILL)
    assert (target.grid == PREFILL).all()
    out = MapMerger().fuse_occupancy(maps, origins, res, transforms, target)
    assert out is target
    return target.grid


def rand_maps(rng, A, h, w, lo=-1, hi=127):
    return rng.integers(lo, hi + 1, size=(A, h, w)).astype(np.int8)


def occ_maps(rng, A, h, w):
    """-1 / 0 / 100 maps."""
    return rng.choice(np.array([-1, 0, 100], np.int8), size=(A, h, w), p=[0.4, 0.45, 0.15])


@pytest.mark.gpu
def test_identity_one_agent_returns_the_map(M):
    rng = np.random.default_rng(1)
    m = rand_maps(rng, 1, 300, 300, lo=-128)
    got = fuse(M, torch.from_numpy(m).cuda(), [(-4.0, -6.4)], 0.05, None, 300, 0.05, -4.0, -6.4)
    assert np.array_equal(got, np.maximum(m[0], -1))        # values >= -1 bit for bit, the rest clamped
    keep = m[0] >= -1
    assert np.array_equal(got[keep], m[0][keep])


@pytest.mark.gpu
def test_identity_many_agents_is_the_max_in_any_order(M):
    rng = np.random.default_rng(2)
    m = rand_maps(rng, 5, 200, 200, lo=-128)
    want = np.maximum(m.max(0), -1)
    org = np.tile([[-5.0, -5.0]], (5, 1))
    for perm in [range(5), range(4, -1, -1)] + [rng.permutation(5) for _ in range(3)]:
        perm = list(perm)
        got = fuse(M, m[perm], org[perm], 0.05, np.tile(np.eye(4), (5, 1, 1)), 200, 0.05, -5.0, -5.0)
        assert np.array_equal(got, want), perm


def _rot(k):
    c, s = [(1, 0), (0, 1), (-1, 0), (0, -1)][k % 4]
    return np.array([[c, -s], [s, c]], np.int64)


def exact_reference(m, origin_cells, k, t_cells, size, target_cells):
    """Integer geometry in half-cell units (no floating point): target cell centre -> agent frame by
    R^T (x - t) -> agent cell."""
    H, W = m.shape
    R = _rot(k)
    out = np.full((size, size), -1, np.int8)
    i, j = np.mgrid[0:size, 0:size]
    X = 2 * (target_cells[0] + j) + 1 - 2 * t_cells[0]
    Y = 2 * (target_cells[1] + i) + 1 - 2 * t_cells[1]
    xa = R[0, 0] * X + R[1, 0] * Y - 2 * origin_cells[0]
    ya = R[0, 1] * X + R[1, 1] * Y - 2 * origin_cells[1]
    gx, gy = xa // 2, ya // 2
    cov = (gx >= 0) & (gx < W) & (gy >= 0) & (gy < H)
    out[cov] = m[gy[cov], gx[cov]]
    return out, cov


@pytest.mark.gpu
@pytest.mark.parametrize('k', [0, 1, 2, 3])
@pytest.mark.parametrize('t_cells', [(0, 0), (7, -3), (-20, 11)])
def test_right_angle_rotations_and_whole_cell_shifts(M, k, t_cells):
    r = 0.0625
    rng = np.random.default_rng(10 + k)
    m = rand_maps(rng, 1, 48, 80)[0]
    origin_cells, target_cells, size = (-24, 12), (-100, -100), 200
    T = np.eye(4)
    T[:2, :2] = _rot(k)
    T[0, 3], T[1, 3] = t_cells[0] * r, t_cells[1] * r
    got = fuse(M, m[None], [(origin_cells[0] * r, origin_cells[1] * r)], r, [T], size, r,
               target_cells[0] * r, target_cells[1] * r)
    want, cov = exact_reference(m, origin_cells, k, t_cells, size, target_cells)
    assert np.array_equal(got, want)
    ys, xs = np.nonzero(cov)
    block = got[ys.min():ys.max() + 1, xs.min():xs.max() + 1]
    assert cov.sum() == m.size and np.array_equal(block, np.rot90(m, -k))
    assert (got[~cov] == -1).all()


RANDOM_CASES = [
    # A, (H, W), target size, target res / agent res, footprint spread in metres
    (1, (1, 1), 1, 1.0, 0.0),
    (2, (1, 1), 3, 1.0, 0.05),
    (2, (3, 257), 3, 1.0, 0.5),
    (1, (131, 257), 1000, 1.0, 10.0),
    (2, (3, 257), 1000, 2.0, 30.0),
    (64, (131, 257), 1000, 1.0, 30.0),
    (64, (131, 257), 1000, 0.5, 15.0),
    (300, (64, 64), 1000, 2.0, 60.0),           # many footprints partly or wholly outside
    (2, (131, 257), 4099, 1.0, 80.0),
    (3, (257, 131), 4099, 0.5, 40.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', RANDOM_CASES, ids=lambda c: f'A{c[0]}_{c[1][0]}x{c[1][1]}_T{c[2]}_g{c[3]}')
def test_random_se2_matches_reference(M, case):
    A, (H, W), size, ratio, spread = case
    rng = np.random.default_rng(hash(case) % (1 << 32))
    r = 0.05
    g = r * ratio
    m = occ_maps(rng, A, H, W)
    org = rng.uniform(-3, 3, (A, 2))
    T = np.stack([se2(*rng.uniform(-spread, spread, 2), rng.uniform(-math.pi, math.pi)) for _ in range(A)])
    gox = goy = -0.5 * size * g
    got = fuse(M, m, org, r, T, size, g, gox, goy)
    want = warp_fuse(m, org, r, T, gox, goy, g, size, size)
    assert np.array_equal(got, want)
    if size >= 1000:
        assert (want == 100).any() and (want == 0).any() and (want == -1).any()


@pytest.mark.gpu
def test_1024_agents_on_the_same_cells(M):
    rng = np.random.default_rng(1024)
    A = 1024
    m = rand_maps(rng, A, 40, 40, lo=-128)
    org = np.tile([[0.0, 0.0]], (A, 1))
    T = np.tile(se2(0.3, -0.2, 0.4), (A, 1, 1))
    got = fuse(M, m, org, 0.05, T, 64, 0.05, -1.6, -1.6)
    assert np.array_equal(got, warp_fuse(m, org, 0.05, T, -1.6, -1.6, 0.05, 64, 64))
    same = fuse(M, m, org, 0.05, None, 40, 0.05, 0.0, 0.0)
    assert np.array_equal(same, np.maximum(m.max(0), -1))


def call_c(maps, origins, res, T, gox, goy, g, out):
    """mapmerge_warp_fuse on torch tensors (maps int8 [A, H, W], out int8 [out_h, out_w] on the device)."""
    from occgrid_b200 import _native
    lib = _native.lib()
    A, H, W = maps.shape
    oh, ow = out.shape
    org = np.ascontiguousarray(origins, np.float64)
    Tm = np.ascontiguousarray(T, np.float64)
    ws = torch.empty(lib.mapmerge_warp_fuse_workspace_bytes(A, ow, oh), dtype=torch.uint8, device=out.device)
    rc = lib.mapmerge_warp_fuse(maps.data_ptr(), A, W, H, res, org.ctypes.data, Tm.ctypes.data, gox, goy, g, ow, oh,
                                out.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    _native.check(rc, 'mapmerge_warp_fuse')


@pytest.mark.gpu
@pytest.mark.parametrize('oh,ow', [(37, 300), (300, 37), (64, 1), (1, 129)])
def test_non_square_targets_through_the_c_entry(M, oh, ow):
    rng = np.random.default_rng(oh * 1000 + ow)
    m = occ_maps(rng, 3, 131, 257)
    org = rng.uniform(-3, 3, (3, 2))
    T = np.stack([se2(*rng.uniform(-2, 2, 2), rng.uniform(-math.pi, math.pi)) for _ in range(3)])
    out = torch.full((oh, ow), PREFILL, dtype=torch.int8, device='cuda')
    call_c(torch.from_numpy(m).cuda(), org, 0.05, T, -7.0, -6.0, 0.05, out)
    assert np.array_equal(out.cpu().numpy(), warp_fuse(m, org, 0.05, T, -7.0, -6.0, 0.05, ow, oh))


@pytest.mark.gpu
def test_stack_above_2_31_bytes(M):
    """3 maps of 27 000^2 (2.19e9 bytes): whole-cell translations view the far corner of each map."""
    r, S, P = 0.0625, 27_000, 96
    rng = np.random.default_rng(31)
    maps = torch.full((3, S, S), -1, dtype=torch.int8, device='cuda')
    patches = rand_maps(rng, 3, P, P)
    corners = [(S - P, S - P - 5), (S - 2 * P, S - P), (S - P - 7, S - P - 3)]      # (x0, y0) of each patch
    for a, (x0, y0) in enumerate(corners):
        maps[a, y0:y0 + P, x0:x0 + P] = torch.from_numpy(patches[a]).cuda()
    # agent a's patch lands on target cells [0, P)^2: t = -(x0, y0) cells, agent origin 0
    T = np.tile(np.eye(4), (3, 1, 1))
    for a, (x0, y0) in enumerate(corners):
        T[a, 0, 3], T[a, 1, 3] = -x0 * r, -y0 * r
    out = torch.full((P + 32, P + 32), PREFILL, dtype=torch.int8, device='cuda')
    call_c(maps, np.zeros((3, 2)), r, T, 0.0, 0.0, r, out)
    got = out.cpu().numpy()
    assert np.array_equal(got[:P, :P], patches.max(0))
    # beyond the patches: the rest of each map (-1) up to the map edge, then uncovered (-1)
    assert (got[P:, :] == -1).all() and (got[:, P:] == -1).all()
    assert 2 * S * S + corners[2][1] * S > 1 << 31          # agent 2's patch lies beyond byte 2^31


@pytest.mark.gpu
def test_target_above_2_31_cells(M):
    """A 46 341^2 target (2.147e9 cells): one agent on its last rows, partly beyond cell 2^31."""
    r, N = 0.0625, 46_341
    rng = np.random.default_rng(46)
    m = torch.from_numpy(rand_maps(rng, 1, 50, 600)).cuda()
    x0, y0 = 45_000, N - 50
    assert (N - 1) * N + x0 + 599 > 1 << 31
    out = torch.full((N, N), PREFILL, dtype=torch.int8, device='cuda')
    call_c(m, [(x0 * r, y0 * r)], r, np.eye(4)[None], 0.0, 0.0, r, out)
    assert torch.equal(out[y0:, x0:x0 + 600], m[0])
    written = int((out == -1).sum().item()) + int((out[y0:, x0:x0 + 600] != -1).sum().item())
    assert written == N * N
    del out


# ---- end to end: packets -> agent maps -> fused map -> frontiers ---------------------------------

def frontier_checks(target, fused):
    from oracle import occgrid_oracle as O
    fr = O.get_frontiers(fused) if fused.shape[0] <= 512 else O.get_frontiers_fast(fused)
    assert target.get_frontiers() == fr
    cl = O.cluster_frontiers(fr)
    got = target.cluster_frontiers()
    assert [sorted(c) for c in got] == [sorted(c) for c in cl]
    cent = target.frontier_centroids()
    assert cent == [O.cluster_centroid_world(c, target.ox, target.oy, target.res) for c in cl]
    assert len(cent) > 0
    return cent


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', ['tiled', 'global_atomic'])
def test_golden_dual_session_fused_and_explored(M, strategy):
    from agent_maps_util import integrate_packets_agent_maps
    from conftest import normalise_datagrams, session_packets
    from occgrid_b200.map_merger import MapMerger
    pk, _ = session_packets(time_sorted=True)
    maps = M.AgentGrids(2, strategy=strategy, size=200, resolution=0.05, origin_x=-5.0, origin_y=-5.0)
    maps.update_packets(pk)
    want_maps = np.full((2, 200, 200), -1, np.int8)
    arr, _ = normalise_datagrams(pk)
    integrate_packets_agent_maps(arr, want_maps, -5.0, -5.0, 0.05)
    assert np.array_equal(maps.grids, want_maps)
    tf = [(0.0, 0.0, 0.0), (-2.5, 0.0, 0.0)]                 # bot 2's start offset in the shared frame
    target = M.OccupancyGrid(300, 0.05, -10.0, -7.5)
    MapMerger().fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, tf, target)
    fused = warp_fuse(want_maps, maps.origins, 0.05, np.stack([se2(*t) for t in tf]), -10.0, -7.5, 0.05, 300, 300)
    assert np.array_equal(target.grid, fused)
    assert (fused == 0).sum() > 1000 and (fused == 100).sum() > 100
    frontier_checks(target, fused)
    # the reference-faithful merge of the same maps publishes no free cell, hence no frontier
    published, _ = MapMerger().merge(maps.grids_tensor, maps.origins, maps.res, tf)
    assert not (published == 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', ['tiled', 'global_atomic'])
def test_swarm_prefix_fused_into_the_shared_map(M, strategy):
    """configs[1] prefix: 64 agents in their own 256^2 frames, fused into the shared 4096^2 map with
    the room offsets."""
    from agent_maps_util import integrate_packets_agent_maps
    from occgrid_b200 import simulation_tools as st
    from occgrid_b200.map_merger import MapMerger
    s = st.generate_session(n_agents=64, n_packets=200_000, seed=42)
    z = np.zeros((65, 2))
    geom = dict(size=256, resolution=0.05, origin_x=-4.0, origin_y=-6.4)
    maps = M.AgentGrids(64, strategy=strategy, max_batch=200_000, **geom)
    maps.update_packets(s['packets'], agent_offsets=z)
    want_maps = np.full((64, 256, 256), -1, np.int8)
    integrate_packets_agent_maps(s['packets'], want_maps, -4.0, -6.4, 0.05, agent_offsets=z)
    assert np.array_equal(maps.grids, want_maps)
    tf = np.concatenate([s['agent_offsets'][1:], np.zeros((64, 1))], axis=1)
    G = s['grid']
    target = M.OccupancyGrid(G['size'], G['resolution'], G['origin_x'], G['origin_y'])
    MapMerger().fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, tf, target)
    fused = warp_fuse(want_maps, maps.origins, 0.05, np.stack([se2(*t) for t in tf]), G['origin_x'], G['origin_y'],
                      G['resolution'], G['size'], G['size'])
    assert np.array_equal(target.grid, fused)
    cent = frontier_checks(target, fused)
    assert len(cent) >= 32
