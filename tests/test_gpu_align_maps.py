"""Correlative map alignment (MapMerger.align_maps, mapmerge_align; DESIGN §6h).

Host-only: the exact workspace arithmetic, every rejection by key word from the query and the call, a
short workspace, the Python argument errors, and the NumPy reference (align_maps_util) pinned against
plain loops.  GPU: [A][6] rows bit for bit against the NumPy reference on scenes, shapes, resolutions,
parameters, edge cases and hand-built ties; the same rows for every pruning block size; the winner's
and the prior's score at the configs[2] scale; and the recovery align_maps -> register_maps from priors
off by up to 1 m and 20 degrees on a configs[1] prefix."""
import math
from types import SimpleNamespace

import numpy as np
import pytest

import align_maps_util as AU
from distance_field_util import edt_reference, max_d2_of
from map_fuse_util import se2
from merge_util import synth_agent_grid

E_ARG, E_WORKSPACE = -1, -2


@pytest.fixture(scope='module')
def lib():
    from occgrid_b200 import _native
    return _native.lib()


def _err(lib):
    return lib.occgrid_last_error().decode()


# ---- host only ------------------------------------------------------------------------------------
def _a(v):
    return (v + 255) // 256 * 256


def _workspace(A, W, H, Wr, Hr, rc, n, points, s=8):
    cpa = -(-(W * H) // 4096)
    nb = (-(-(2 * rc + 1) // s)) ** 2
    pad = 2 * rc + 64
    np_ = (Wr + 2 * pad) * (Hr + 2 * pad)
    return (_a(48 * A * n) + _a(4 * A * cpa) + _a(8 * (A + 1)) + _a(4 * A * n * nb) + 3 * _a(8 * A) + _a(65536) + 256
            + 3 * _a(np_) + _a(8 * points))


WS_CASES = [(1, 1, 1, 1, 1, 0, 1, 0), (3, 96, 80, 320, 300, 17, 51, 1000), (64, 256, 256, 4096, 4096, 24, 101, 200000),
            (65535, 7, 3, 5, 9, 0, 1, 1), (5, 2048, 2048, 32768, 32768, 2048, 255, 10 ** 7)]


@pytest.mark.parametrize('block', [0, 1, 3, 64])
@pytest.mark.parametrize('case', WS_CASES)
def test_workspace_arithmetic(lib, case, block):
    A, W, H, Wr, Hr, rc, n, pts = case
    try:
        assert lib.mapmerge_align_set_block(block) == 0
        assert lib.mapmerge_align_workspace_bytes(A, W, H, Wr, Hr, 0, rc, n, pts) == \
            _workspace(A, W, H, Wr, Hr, rc, n, pts, block or 8)
    finally:
        lib.mapmerge_align_set_block(0)


QUERY_REJECTS = [((0, 8, 8, 8, 8, 0, 1, 1, 0), 'n_agents'), ((65536, 8, 8, 8, 8, 0, 1, 1, 0), 'n_agents'),
                 ((1, 0, 8, 8, 8, 0, 1, 1, 0), 'width x height'), ((1, 8, -1, 8, 8, 0, 1, 1, 0), 'width x height'),
                 ((1, 2 ** 31 - 1, 1, 8, 8, 1, 1, 1, 0), 'width x height'), ((1, 65536, 32768, 8, 8, 0, 1, 1, 0), 'width x height'),
                 ((1, 4096, 4096, 8, 8, 127, 1, 1, 0), 'width x height'),
                 ((1, 8, 8, 0, 8, 0, 1, 1, 0), 'reference size'), ((1, 8, 8, 8, 32769, 0, 1, 1, 0), 'reference size'),
                 ((1, 8, 8, 8, 8, -1, 1, 1, 0), 'max_d2'), ((1, 8, 8, 8, 8, 255, 1, 1, 0), 'max_d2'),
                 ((1, 8, 8, 8, 8, 0, -1, 1, 0), 'max_offset'), ((1, 8, 8, 8, 8, 0, 2049, 1, 0), 'max_offset'),
                 ((1, 8, 8, 8, 8, 0, 1, 0, 0), 'n_angles'), ((1, 8, 8, 8, 8, 0, 1, 65536, 0), 'n_angles'),
                 ((1, 8, 8, 8, 8, 0, 2048, 256, 0), 'candidates'),
                 ((2, 8, 8, 8, 8, 0, 1, 1, -1), 'total_points'), ((2, 8, 8, 8, 8, 0, 1, 1, 129), 'total_points')]


@pytest.mark.parametrize('args,key', QUERY_REJECTS)
def test_workspace_query_rejects(lib, args, key):
    assert lib.mapmerge_align_workspace_bytes(*args) == 0
    assert key in _err(lib)


def test_limits_accepted(lib):
    assert lib.mapmerge_align_workspace_bytes(1, 2 ** 31 - 1, 1, 8, 8, 0, 1, 1, 0) > 0                 # W*H*(0+1) = 2^31-1
    assert lib.mapmerge_align_workspace_bytes(1, 8, 8, 8, 8, 0, 2048, 255, 0) > 0                      # 255 * 4097^2 < 2^32
    assert lib.mapmerge_align_workspace_bytes(65535, 1, 1, 32768, 32768, 254, 0, 65535, 65535) > 0


def _host(a):
    a = np.ascontiguousarray(a, np.float64)
    return a, a.ctypes.data


def _call(lib, **kw):
    org, org_p = _host(np.zeros((2, 2)))
    pri, pri_p = _host(np.tile(np.eye(4), (2, 1, 1)))
    rot, rot_p = _host([[1.0, 0.0], [0.0, 1.0]])
    a = dict(grids=256, A=2, W=8, H=8, res=0.05, org=org_p, pri=pri_p, d2=256, Wr=16, Hr=16, gox=0.0, goy=0.0, g=0.05,
             rot=rot_p, n=2, rc=3, max_d2=4, out=256, diag=None, ws=256, ws_bytes=1 << 40)
    for k, v in kw.items():
        if k in ('pri', 'rot', 'org') and v is not None and not isinstance(v, int):
            kw[k] = _host(v)
            v = kw[k][1]
        a[k] = v
    return lib.mapmerge_align(a['grids'], a['A'], a['W'], a['H'], a['res'], a['org'], a['pri'], a['d2'], a['Wr'], a['Hr'],
                              a['gox'], a['goy'], a['g'], a['rot'], a['n'], a['rc'], a['max_d2'], a['out'], a['diag'],
                              a['ws'], a['ws_bytes'], None)


def _rot_bad(k):
    r = np.array([[1.0, 0.0], [0.0, 1.0]])
    r[k] = (1.0 + 1e-8, 0.0)
    return r


def _prior_bad(v):
    p = np.tile(np.eye(4), (2, 1, 1))
    p[1, 0, 0] = v
    return p


CALL_REJECTS = [(dict(grids=None), 'NULL pointer'), (dict(org=None), 'NULL pointer'), (dict(pri=None), 'NULL pointer'),
                (dict(d2=None), 'NULL pointer'), (dict(rot=None), 'NULL pointer'), (dict(out=None), 'NULL pointer'),
                (dict(ws=None), 'NULL pointer'), (dict(A=0), 'n_agents'), (dict(A=65536), 'n_agents'),
                (dict(W=0), 'width x height'), (dict(W=4096, H=4096, max_d2=128), 'width x height'),
                (dict(Wr=32769), 'reference size'), (dict(Hr=0), 'reference size'),
                (dict(max_d2=-1), 'max_d2'), (dict(max_d2=255), 'max_d2'), (dict(rc=-1), 'max_offset'),
                (dict(rc=2049), 'max_offset'), (dict(n=0), 'n_angles'), (dict(n=65536), 'n_angles'),
                (dict(rc=2048, n=256), 'candidates'),
                (dict(res=0.0), 'resolution'), (dict(res=math.nan), 'resolution'), (dict(g=-0.05), 'resolution'),
                (dict(g=math.inf), 'resolution'),
                (dict(pri=_prior_bad(math.nan)), 'prior'), (dict(pri=_prior_bad(1.0 + 1e-8)), 'prior'),
                (dict(rot=_rot_bad(1)), 'rotation'), (dict(rot=np.array([[1.0, 0.0], [math.nan, 0.0]])), 'rotation')]


@pytest.mark.parametrize('kw,key', CALL_REJECTS)
def test_call_rejects(lib, kw, key):
    assert _call(lib, **kw) == E_ARG
    assert key in _err(lib)


def test_short_workspace(lib):
    need = lib.mapmerge_align_workspace_bytes(2, 8, 8, 16, 16, 4, 3, 2, 0)
    assert need == _workspace(2, 8, 8, 16, 16, 3, 2, 0)
    assert _call(lib, ws_bytes=need - 1) == E_WORKSPACE
    assert 'workspace' in _err(lib)
    for s in (-1, 65):
        assert lib.mapmerge_align_set_block(s) == E_ARG and 'block' in _err(lib)


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
    ref = SimpleNamespace(size=64, window=(0, 0, 64, 64), device='cuda:0', res=0.05)
    with pytest.raises(ValueError, match='align_maps: origins'):
        m.align_maps(g, np.zeros((2, 2)), 0.05, None, ref)
    with pytest.raises(ValueError, match='2 priors for 3'):
        m.align_maps(g, org, 0.05, np.tile(np.eye(4), (2, 1, 1)), ref)
    with pytest.raises(ValueError, match='prior 1 must be'):
        m.align_maps(g, org, 0.05, [np.eye(4), np.eye(3), np.eye(4)], ref)
    with pytest.raises(ValueError, match=r'\[A, H, W\]'):
        m.align_maps(np.zeros((8, 8), np.int8), org, 0.05, None, ref)
    bad = np.tile(np.eye(4), (3, 1, 1))
    bad[2, 0, 0] = 1.0 + 1e-8
    with pytest.raises(OccGridError, match='align_maps: prior 2 is not rigid'):
        m.align_maps(g, org, 0.05, bad, ref)
    bad[2, 0, 0] = math.nan
    with pytest.raises(OccGridError, match='prior 2 has a non-finite'):
        m.align_maps(g, org, 0.05, bad, ref)
    with pytest.raises(OccGridError, match='whole grid'):
        m.align_maps(g, org, 0.05, None, SimpleNamespace(size=64, window=(0, 0, 32, 64), device='cuda:0', res=0.05))
    with pytest.raises(OccGridError, match='cuda:1'):
        m.align_maps(g, org, 0.05, None, SimpleNamespace(size=64, window=(0, 0, 64, 64), device='cuda:1', res=0.05))
    for kw, key in ((dict(max_offset=-0.1), 'max_offset'), (dict(max_offset=math.inf), 'max_offset'),
                    (dict(max_angle=math.nan), 'max_angle'), (dict(angle_step=0.0), 'angle_step'),
                    (dict(clearance=-1.0), 'clearance'), (dict(max_offset=102.5), 'more than 2048'),
                    (dict(max_angle=1.0, angle_step=1e-5), 'more than 65 535'), (dict(clearance=0.8), 'more than 254')):
        with pytest.raises(ValueError, match=key):
            m.align_maps(g, org, 0.05, None, ref, **kw)


def _tiny_case(seed, A=2, h=6, w=5, n_ref=12, rc=2, n_angles=3, max_d2=2, g=0.05, shift=(0.0, 0.0)):
    r = np.random.default_rng(seed)
    grids = np.where(r.random((A, h, w)) < 0.3, 100, 0).astype(np.int8)
    grids[r.random((A, h, w)) < 0.2] = 51
    grids[r.random((A, h, w)) < 0.2] = 50
    ref = np.where(r.random((n_ref, n_ref)) < 0.15, 100, -1).astype(np.int8)
    org = r.uniform(-0.2, 0.2, (A, 2)) + np.array(shift)
    priors = np.stack([se2(*r.uniform(-0.2, 0.2, 2), r.uniform(-0.5, 0.5)) for _ in range(A)])
    _, rot = AU.rotation_table(math.radians(3) * (n_angles // 2), math.radians(3))
    return grids, org, priors, edt_reference(ref), rot, rc, max_d2, g


@pytest.mark.parametrize('seed', range(4))
def test_reference_against_brute_force(seed):
    grids, org, priors, d2, rot, rc, max_d2, g = _tiny_case(seed)
    args = (grids, org, 0.05, priors, d2, -0.1, -0.15, g, rot, rc, max_d2)
    assert np.array_equal(AU.align_reference(*args), AU.align_brute(*args))


def test_reference_floor_of_negative_x():
    """A map that hangs over the reference's low edge: X < 0 for most points, floor differs from
    truncation, and the scores near the edge pin it."""
    grids, org, priors, d2, rot, rc, max_d2, g = _tiny_case(7, shift=(-0.3, -0.3))
    args = (grids, org, 0.05, priors, d2, 0.0, 0.0, g, rot, rc, max_d2)
    u, v = AU.agent_points(grids[0])
    j, i, ok = AU.project(AU.coefficients(priors[0], org[0], 0.05, 5, 6, 1.0, 0.0, 0.0, 0.0, g), u, v)
    assert (j < 0).any() and ok.all()
    assert np.array_equal(AU.align_reference(*args), AU.align_brute(*args))


def test_reference_rank_order():
    """Two equidistant obstacles either side of a single point: dx = +2 (rank 3) beats dx = -2 (rank 4)."""
    grid = np.zeros((1, 1, 1), np.int8)
    grid[0, 0, 0] = 100
    ref = np.full((5, 9), -1, np.int8)
    ref[2, 2] = ref[2, 6] = 100
    d2 = edt_reference(ref)
    org = np.array([[0.0, 0.0]])
    prior = se2(4 * 0.05, 2 * 0.05, 0.0)[None]
    rows = AU.align_reference(grid, org, 0.05, prior, d2, 0.0, 0.0, 0.05, np.array([[1.0, 0.0]]), 2, 0)
    assert rows.tolist() == [[1, 0, 2, 0, 0, 1]]
    assert np.array_equal(rows, AU.align_brute(grid, org, 0.05, prior, d2, 0.0, 0.0, 0.05, [[1.0, 0.0]], 2, 0))


def test_reference_far_cut_off():
    """Points at |X| >= 2^30 contribute nothing: the reference marks them, and no candidate scores."""
    grid = np.full((1, 3, 3), 100, np.int8)
    d2 = np.zeros((4, 4), np.int32)
    for far in (2.0 ** 30, -(2.0 ** 30) - 3.0):
        prior = se2(far * 0.05, 0.0, 0.0)[None]
        e = AU.coefficients(prior[0], (0.0, 0.0), 0.05, 3, 3, 1.0, 0.0, 0.0, 0.0, 0.05)
        assert not AU.project(e, *AU.agent_points(grid[0]))[2].any()
        args = (grid, np.zeros((1, 2)), 0.05, prior, d2, 0.0, 0.0, 0.05, np.array([[1.0, 0.0]]), 1, 0)
        assert AU.align_reference(*args).tolist() == [[0, 0, 0, 0, 0, 9]] == AU.align_brute(*args).tolist()


# ---- GPU ------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def gpu():
    torch = pytest.importorskip('torch')
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper as M
    from occgrid_b200 import map_merger as MM
    return SimpleNamespace(torch=torch, M=M, MM=MM)


def _run(gpu, lib, grids, org, r, priors, d2, gox, goy, g, rot, rc, max_d2, block=0):
    """mapmerge_align through the C ABI with the given block size -> (rows [A, 6], diag [2])."""
    from occgrid_b200 import _native
    torch = gpu.torch
    grids = np.ascontiguousarray(grids, np.int8)
    A, h, w = grids.shape
    dg = torch.from_numpy(grids).cuda()
    dd = torch.from_numpy(np.ascontiguousarray(d2, np.int32)).cuda()
    org = np.ascontiguousarray(org, np.float64)
    pri = np.ascontiguousarray(priors, np.float64)
    rot = np.ascontiguousarray(rot, np.float64)
    pts = int((grids > 50).sum())
    assert lib.mapmerge_align_set_block(block) == 0
    try:
        nb = lib.mapmerge_align_workspace_bytes(A, w, h, d2.shape[1], d2.shape[0], max_d2, rc, len(rot), pts)
        assert nb > 0, _err(lib)
        ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
        out = torch.full((A, 6), 7, dtype=torch.int64, device='cuda')
        diag = torch.zeros(2, dtype=torch.int64, device='cuda')
        _native.check(lib.mapmerge_align(dg.data_ptr(), A, w, h, r, org.ctypes.data, pri.ctypes.data, dd.data_ptr(), d2.shape[1],
                                         d2.shape[0], gox, goy, g, rot.ctypes.data, len(rot), rc, max_d2, out.data_ptr(),
                                         diag.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream),
                      'mapmerge_align')
        return out.cpu().numpy(), diag.cpu().numpy()
    finally:
        lib.mapmerge_align_set_block(0)


def _assert_rows(got, want):
    bad = np.flatnonzero((got != want).any(axis=1))
    assert bad.size == 0, f'agents {bad[:10].tolist()} differ: {got[bad[0]].tolist()} vs {want[bad[0]].tolist()}' if bad.size else ''


def _check(gpu, lib, *args, blocks=(0,)):
    want = AU.align_reference(*args)
    for b in blocks:
        got, diag = _run(gpu, lib, *args, block=b)
        _assert_rows(got, want)
        live = int((want[:, 5] > 0).sum())
        assert diag[0] == live * len(args[8]) * (2 * args[9] + 1) ** 2 and diag[1] >= live
    return want


def _world(n=320, seed=3):
    return synth_agent_grid(n, seed, occ_segments=60)


def _scene(A, seed, size=(96, 96), n_world=320, res=0.05, empty=(), far=(), max_t=1.0, max_deg=20.0):
    """A crops of one world map (as test_gpu_register_maps._scene), priors rotated by up to max_deg
    and shifted by up to max_t metres about each map's centre; agents in `far` moved 100 m away,
    agents in `empty` see nothing.  Returns the world, its origin, grids, origins, priors and truths."""
    world = _world(n_world)
    r = np.random.default_rng(seed)
    ox = oy = -n_world * res / 2
    h, w = size
    grids = np.full((A, h, w), -1, np.int8)
    org = np.zeros((A, 2))
    priors = np.zeros((A, 4, 4))
    for a in range(A):
        x0, y0 = int(r.integers(0, n_world - w)), int(r.integers(0, n_world - h))
        if a not in empty:
            grids[a] = world[y0:y0 + h, x0:x0 + w]
            grids[a][r.random((h, w)) < 0.02] = -1
        org[a] = (ox + x0 * res, oy + y0 * res)
        c = org[a] + np.array([w, h]) * res / 2
        d = se2(*r.uniform(-max_t, max_t, 2), math.radians(r.uniform(-max_deg, max_deg)))
        priors[a] = se2(c[0], c[1], 0) @ d @ se2(-c[0], -c[1], 0)
        if a in far:
            priors[a] = se2(100.0, 0.0, 0.0) @ priors[a]
    return world, ox, oy, grids, org, priors


@pytest.mark.gpu
@pytest.mark.parametrize('A,rc,deg,step', [(1, 17, 25, 1.0), (7, 17, 25, 1.0), (64, 8, 10, 2.0)])
def test_scenes(gpu, lib, A, rc, deg, step):
    empty, far = ((3,), (5,)) if A >= 7 else ((), ())
    world, ox, oy, grids, org, priors = _scene(A, seed=A, empty=empty, far=far)
    _, rot = AU.rotation_table(math.radians(deg), math.radians(step))
    want = _check(gpu, lib, grids, org, 0.05, priors, edt_reference(world), ox, oy, 0.05, rot, rc, 2)
    for a in empty + far:
        assert want[a, 0] == 0 and want[a, 1:4].tolist() == [0, 0, 0]
    assert (want[:, 0] > want[:, 4]).sum() >= A // 2            # most agents find something better than the prior


@pytest.mark.gpu
def test_non_square_maps(gpu, lib):
    world, ox, oy, grids, org, priors = _scene(5, seed=9, size=(64, 112), max_t=0.5, max_deg=10)
    _, rot = AU.rotation_table(math.radians(12), math.radians(3))
    _check(gpu, lib, grids, org, 0.05, priors, edt_reference(world[:250, :]), ox, oy, 0.05, rot, 9, 4)


@pytest.mark.gpu
@pytest.mark.parametrize('ratio', [1, 2])
def test_reference_resolution(gpu, lib, ratio):
    """g = r and g = 2r: the reference is the world max-pooled 2 x 2 (occupied wins) at 0.10 m."""
    world, ox, oy, grids, org, priors = _scene(6, seed=13, max_t=0.6, max_deg=12)
    ref = world if ratio == 1 else world.reshape(160, 2, 160, 2).max(axis=(1, 3))
    _, rot = AU.rotation_table(math.radians(15), math.radians(1.5))
    _check(gpu, lib, grids, org, 0.05, priors, edt_reference(ref), ox, oy, 0.05 * ratio, rot, 12 // ratio, 3, blocks=(0, 1))


@pytest.mark.gpu
@pytest.mark.parametrize('max_d2', [0, 8, 254])
@pytest.mark.parametrize('rc', [0, 1, 17])
@pytest.mark.parametrize('n_angles', [1, 2, 51])
def test_parameters(gpu, lib, max_d2, rc, n_angles):
    world, ox, oy, grids, org, priors = _scene(3, seed=rc * 7 + n_angles, size=(48, 64), max_t=0.4, max_deg=8)
    theta = np.radians(0.4) * np.array([0] + [m for i in range(1, 26) for m in (i, -i)])[:n_angles]
    rot = np.stack([np.cos(theta), np.sin(theta)], 1)
    _check(gpu, lib, grids, org, 0.05, priors, edt_reference(world), ox, oy, 0.05, rot, rc, max_d2)


@pytest.mark.gpu
def test_unknown_reference_keeps_the_prior(gpu, lib):
    world, ox, oy, grids, org, priors = _scene(4, seed=2)
    d2 = np.full((200, 180), -1, np.int32)
    _, rot = AU.rotation_table(math.radians(10), math.radians(2))
    want = _check(gpu, lib, grids, org, 0.05, priors, d2, ox, oy, 0.05, rot, 6, 8, blocks=(0, 1, 32))
    assert (want[:, :5] == 0).all() and (want[:, 5] > 0).all()


@pytest.mark.gpu
def test_maps_over_the_reference_edges(gpu, lib):
    """Maps that hang over the low and the high edge of a 64^2 reference (negative X and Y, and cells
    beyond the last column), and one 100 m away."""
    world = _world(64, seed=4)
    ox = oy = 0.0
    grids = np.stack([_world(96, seed=s)[:80, :] for s in (5, 6, 7, 8)])
    org = np.array([[-1.2, -0.9], [1.5, 1.8], [-0.7, 1.9], [100.0, -100.0]])
    priors = np.stack([se2(0.05, -0.08, 0.2), se2(-0.1, 0.03, -0.3), se2(0.0, 0.0, 0.5), se2(0.0, 0.0, 0.0)])
    _, rot = AU.rotation_table(math.radians(20), math.radians(4))
    want = _check(gpu, lib, grids, org, 0.05, priors, edt_reference(world), ox, oy, 0.05, rot, 10, 4, blocks=(0, 1))
    assert want[3, 0] == 0


@pytest.mark.gpu
def test_cells_50_51_60(gpu, lib):
    """Values 50 (free by the > 50 rule), 51 and 60 (occupied) in the maps and in the reference, whose
    d2 comes from the device's own distance field and must equal SciPy's."""
    r = np.random.default_rng(21)
    vals = np.array([-1, 0, 50, 51, 60, 100], np.int8)
    world = vals[r.integers(0, 6, (120, 140))] * (r.random((120, 140)) < 0.2).astype(np.int8)
    world[world == 0] = 50
    grids = vals[r.integers(0, 6, (3, 40, 30))]
    org = np.array([[0.5, 0.5], [1.2, 2.0], [3.0, 1.0]])
    priors = np.stack([se2(0.1, 0.0, 0.1), se2(0.0, -0.1, -0.2), se2(0.02, 0.03, 0.0)])
    ref = gpu.M.OccupancyGrid(140, 0.05, 0.0, 0.0, lazy_workspace=True)
    full = np.full((140, 140), -1, np.int8)
    full[:120] = world
    ref.grid_tensor.copy_(gpu.torch.from_numpy(full))
    ref._host_cache = None
    d2 = ref.distance_field()
    assert np.array_equal(d2, edt_reference(full))
    _, rot = AU.rotation_table(math.radians(6), math.radians(2))
    want = _check(gpu, lib, grids, org, 0.05, priors, d2, 0.0, 0.0, 0.05, rot, 5, 0, blocks=(0, 1))
    assert want[:, 5].tolist() == [int((g > 50).sum()) for g in grids]


@pytest.mark.gpu
def test_hand_built_ties(gpu, lib):
    """Agent 0: one point between two obstacles 2 cells either side: dx = +2 (rank 3) beats dx = -2
    (rank 4).  Agent 1: the same along y.  Agent 2: two points and a symmetric pair of obstacle
    columns, so that (dx, dy) = (+3, 0) and (-3, 0) tie; agent 3: a tie between rotations k = 1 and 2."""
    ref = np.full((21, 21), -1, np.int8)
    ref[10, 8] = ref[10, 12] = 100                   # agent 0
    ref[3, 3] = ref[7, 3] = 100                      # agent 1
    ref[15:18, 14] = ref[15:18, 20] = 100            # agent 2
    grids = np.full((4, 3, 3), -1, np.int8)
    grids[0, 1, 1] = grids[1, 1, 1] = 100
    grids[2, 0, 1] = grids[2, 2, 1] = 100
    grids[3, 1, 0] = grids[3, 1, 2] = 100            # a bar through the centre: ±90 degrees give the same cells
    org = np.full((4, 2), -0.075)
    priors = np.stack([se2(10.5 * 0.05, 10.5 * 0.05, 0.0), se2(3.5 * 0.05, 5.5 * 0.05, 0.0),
                       se2(17.5 * 0.05, 16.5 * 0.05, 0.0), se2(10.5 * 0.05, 3.5 * 0.05, 0.0)])
    ref[3, 10] = 100                                  # agent 3: the bar rotated upright hits it at dx = 0, dy = -1
    ref[2, 10] = ref[4, 10] = 100
    rot = np.array([[1.0, 0.0], [0.0, 1.0], [0.0, -1.0]])
    want = _check(gpu, lib, grids, org, 0.05, priors, edt_reference(ref), 0.0, 0.0, 0.05, rot, 3, 0, blocks=(0, 1, 2))
    assert want[0, :4].tolist() == [1, 0, 2, 0]
    assert want[1, :4].tolist() == [1, 0, 0, 2]
    assert want[2, :4].tolist() == [2, 0, 3, 0]
    assert want[3, 1] == 1


@pytest.mark.gpu
@pytest.mark.parametrize('flat', [False, True])
def test_block_size_invariance(gpu, lib, flat):
    """s = 1, 2, 8, 32 and the default give the same rows; `flat`: a reference that is all obstacle, so
    every candidate that keeps the points inside scores the same and nothing prunes."""
    world, ox, oy, grids, org, priors = _scene(9, seed=31, empty=(4,), far=(7,), max_t=0.5, max_deg=10)
    if flat:
        world = np.full_like(world, 100)
    _, rot = AU.rotation_table(math.radians(9), math.radians(1.5))
    want = _check(gpu, lib, grids, org, 0.05, priors, edt_reference(world), ox, oy, 0.05, rot, 11, 3, blocks=(0, 1, 2, 8, 32))
    if flat:
        live = [a for a in range(9) if a not in (4, 7)]
        assert (want[live, 1:4] == 0).all() and (want[live, 0] == want[live, 4]).all()


@pytest.mark.gpu
def test_align_maps_equals_the_reference(gpu):
    """The Python entry: conversions (Rc, the rotation table, max_d2), the device distance field and the
    transformation of the winner."""
    world, ox, oy, grids, org, priors = _scene(5, seed=41, empty=(2,), max_t=0.5, max_deg=10)
    ref = gpu.M.OccupancyGrid(world.shape[0], 0.05, ox, oy, lazy_workspace=True)
    ref.grid_tensor.copy_(gpu.torch.from_numpy(world))
    ref._host_cache = None
    m = gpu.MM.MapMerger()
    got = m.align_maps(gpu.torch.from_numpy(grids).cuda(), org, 0.05, priors, ref, max_offset=0.6, max_angle=math.radians(12),
                       angle_step=math.radians(1.5), clearance=0.1)
    theta, rot = AU.rotation_table(math.radians(12), math.radians(1.5))
    want = AU.align_reference(grids, org, 0.05, priors, edt_reference(world), ox, oy, 0.05, rot, 12, max_d2_of(0.1, 0.05))
    assert got.score.tolist() == want[:, 0].tolist() and got.prior_score.tolist() == want[:, 4].tolist()
    assert got.points.tolist() == want[:, 5].tolist() and got.offset.tolist() == want[:, 2:4].tolist()
    assert np.array_equal(got.angle, theta[want[:, 1]])
    assert np.array_equal(got.improved, want[:, 0] > want[:, 4])
    assert np.array_equal(got.transformation[2], priors[2])
    for a in (0, 1, 3, 4):
        T = gpu.MM.align_transform(priors[a], org[a], 0.05, 96, 96, *rot[want[a, 1]], want[a, 2], want[a, 3], 0.05)
        assert np.array_equal(got.transformation[a], T)
    T0 = gpu.MM.align_transform(priors[0], org[0], 0.05, 96, 96, 1.0, 0.0, 0, 0, 0.05)
    assert np.array_equal(np.abs(T0[:2]), np.abs(priors[0][:2]))          # the prior, up to the sign of a zero


def _scale_check(gpu, lib, grids_t, org, res, priors, d2, gox, goy, g, rot, rc, max_d2, sample):
    """Rows equal for s = 1 and the default; the winner's and the prior's score equal NumPy's."""
    rows = {}
    for b in (0, 1):
        rows[b] = _run_device(gpu, lib, grids_t, org, res, priors, d2, gox, goy, g, rot, rc, max_d2, b)
    _assert_rows(rows[1], rows[0])
    d2h = d2.cpu().numpy()
    for a in sample:
        grid = grids_t[a].cpu().numpy()
        k, dx, dy = (int(v) for v in rows[0][a, 1:4])
        assert rows[0][a, 0] == AU.score_at(grid, org[a], res, priors[a], d2h, gox, goy, g, *rot[k], dx, dy, max_d2)
        assert rows[0][a, 4] == AU.score_at(grid, org[a], res, priors[a], d2h, gox, goy, g, 1.0, 0.0, 0, 0, max_d2)
        assert rows[0][a, 5] == int((grid > 50).sum())
    return rows[0]


def _run_device(gpu, lib, grids_t, org, res, priors, d2, gox, goy, g, rot, rc, max_d2, block):
    from occgrid_b200 import _native
    torch = gpu.torch
    A, h, w = grids_t.shape
    org = np.ascontiguousarray(org, np.float64)
    pri = np.ascontiguousarray(priors, np.float64)
    rot = np.ascontiguousarray(rot, np.float64)
    pts = int((grids_t > 50).sum().item())
    assert lib.mapmerge_align_set_block(block) == 0
    try:
        nb = lib.mapmerge_align_workspace_bytes(A, w, h, d2.shape[1], d2.shape[0], max_d2, rc, len(rot), pts)
        ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
        out = torch.empty((A, 6), dtype=torch.int64, device='cuda')
        _native.check(lib.mapmerge_align(grids_t.data_ptr(), A, w, h, res, org.ctypes.data, pri.ctypes.data, d2.data_ptr(),
                                         d2.shape[1], d2.shape[0], gox, goy, g, rot.ctypes.data, len(rot), rc, max_d2,
                                         out.data_ptr(), None, ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream),
                      'mapmerge_align')
        return out.cpu().numpy()
    finally:
        lib.mapmerge_align_set_block(0)


@pytest.mark.gpu
def test_scale_2048_maps_against_4803_reference(gpu, lib):
    """16 maps of 2048^2 (bench_merge.device_grids) against their 4803^2 fusion, priors off by up to
    0.5 m and 5 degrees; a ±0.6 m, ±6 degree window at 1.5 degrees."""
    from bench_merge import device_grids
    torch = gpu.torch
    A, S, res = 16, 2048, 0.05
    stack = torch.stack(device_grids(torch, torch.device('cuda'), A, S))
    rng = np.random.default_rng(0)
    origins = np.tile(np.array([[-S * res / 2, -S * res / 2]]), (A, 1))
    tf = np.stack([se2(*rng.uniform(-50, 50, 2), rng.uniform(-math.pi, math.pi)) for _ in range(A)])
    n = 4803
    gox = goy = -n * res / 2
    ref = gpu.M.OccupancyGrid(n, res, gox, goy, lazy_workspace=True)
    gpu.MM.MapMerger().fuse_occupancy(stack, origins, res, tf, ref)
    d2 = ref.distance_field(to_host=False)
    r = np.random.default_rng(1)
    priors = np.stack([tf[a] @ se2(*r.uniform(-0.5, 0.5, 2), math.radians(r.uniform(-5, 5))) for a in range(A)])
    _, rot = AU.rotation_table(math.radians(6), math.radians(1.5))
    rows = _scale_check(gpu, lib, stack, origins, res, priors, d2, gox, goy, res, rot, 12, 2, sample=(0, 5, 11, 15))
    assert (rows[:, 0] > rows[:, 4]).all()


# Agents of the configs[1] prefix (seed 42, 200 000 packets) with the recovery priors below that
# align_maps -> register_maps does not bring within the pipeline bounds; each needs its own reason.
UNRECOVERABLE = {}


def _configs1(gpu, strategy='tiled'):
    from agent_maps_util import integrate_packets_agent_maps
    from occgrid_b200 import simulation_tools as st
    M = gpu.M
    s = st.generate_session(n_agents=64, n_packets=200_000, seed=42)
    z = np.zeros((65, 2))
    maps = M.AgentGrids(64, strategy=strategy, max_batch=200_000, size=256, resolution=0.05, origin_x=-4.0, origin_y=-6.4)
    maps.update_packets(s['packets'], agent_offsets=z)
    want_maps = np.full((64, 256, 256), -1, np.int8)
    integrate_packets_agent_maps(s['packets'], want_maps, -4.0, -6.4, 0.05, agent_offsets=z)
    assert np.array_equal(maps.grids, want_maps)
    tf = np.concatenate([s['agent_offsets'][1:], np.zeros((64, 1))], axis=1)
    truth = np.stack([se2(*t) for t in tf])
    G = s['grid']
    reference = M.OccupancyGrid(G['size'], G['resolution'], G['origin_x'], G['origin_y'])
    merger = gpu.MM.MapMerger()
    merger.fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, truth, reference)
    return maps, truth, reference, merger


def _far_priors(truth, maps, seed=1):
    """truth perturbed by U(-1, 1) m and U(-20, 20) degrees about each map's centre."""
    r = np.random.default_rng(seed)
    A = len(truth)
    c = maps.origins + 256 * 0.05 / 2
    out = []
    for a in range(A):
        d = se2(*r.uniform(-1.0, 1.0, 2), math.radians(r.uniform(-20, 20)))
        out.append(truth[a] @ se2(c[a, 0], c[a, 1], 0) @ d @ se2(-c[a, 0], -c[a, 1], 0))
    return np.stack(out)


@pytest.mark.gpu
def test_recovery_align_then_register(gpu, lib):
    """configs[1] prefix: priors off by up to 1 m and 20 degrees; align_maps with a ±1.2 m / ±25 degree
    window at 0.5 degrees, then register_maps.  Every agent must be accepted and end within the
    bounds test_pipeline_register_fuse_assign holds from ±0.15 m / 3 degrees."""
    from test_gpu_register_maps import PIPE_ORACLE_DEG, PIPE_ORACLE_M, _pose_error
    maps, truth, reference, merger = _configs1(gpu)
    priors = _far_priors(truth, maps)
    al = merger.align_maps(maps.grids_tensor, maps.origins, maps.res, priors, reference, max_offset=1.2,
                           max_angle=math.radians(25), angle_step=math.radians(0.5), clearance=0.1)
    theta, rot = AU.rotation_table(math.radians(25), math.radians(0.5))
    rows = _scale_check(gpu, lib, maps.grids_tensor, maps.origins, 0.05, priors, reference.distance_field(to_host=False),
                        reference.ox, reference.oy, 0.05, rot, 24, max_d2_of(0.1, 0.05), sample=(0, 17, 42, 63))
    assert rows[:, 0].tolist() == al.score.tolist() and rows[:, 2:4].tolist() == al.offset.tolist()
    assert np.array_equal(theta[rows[:, 1]], al.angle)
    reg = merger.register_maps(maps.grids_tensor, maps.origins, maps.res, al.transformation, reference=reference)
    alone = merger.register_maps(maps.grids_tensor, maps.origins, maps.res, priors, reference=reference)
    bad = []
    for a in range(64):
        e = _pose_error(reg.transformation[a], truth[a])
        if not (reg.accepted[a] and e[0] <= PIPE_ORACLE_M + 1e-6 and math.degrees(e[1]) <= PIPE_ORACLE_DEG + 1e-6):
            bad.append(a)
    ok_alone = sum(1 for a in range(64) if alone.accepted[a] and _pose_error(alone.transformation[a], truth[a])[0] <= PIPE_ORACLE_M + 1e-6
                   and math.degrees(_pose_error(alone.transformation[a], truth[a])[1]) <= PIPE_ORACLE_DEG + 1e-6)
    print(f'recovered: align_maps -> register_maps {64 - len(bad)} of 64, register_maps alone {ok_alone} of 64')
    assert sorted(bad) == sorted(UNRECOVERABLE), [(a, al.score[a], al.prior_score[a], al.offset[a].tolist(),
                                                   math.degrees(al.angle[a])) for a in bad]
