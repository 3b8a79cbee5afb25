"""Argument checks of the integration entry points, host only.

Every call here is rejected (or returns early) before the library touches the CUDA runtime, so the
test needs no GPU.  Device pointers are made-up addresses: they are never dereferenced because each
case fails a check first.  A case that got past the checks would launch on them, which is why no
case may be fully valid (and why `occgrid_route_packets` with n == 0, which clears the band counts,
and `occgrid_accumulate_packets` under GLOBAL_ATOMIC, which has no workspace check, are not called
with otherwise valid arguments).

The expected codes, the key word of each message, the order of the checks (`n == 0` returns before
the strategy is looked at, for example) and the workspace byte counts callers allocate from are
pinned here.
"""
import ctypes as C

import pytest

from occgrid_b200 import _native

OK, E_ARG, E_WORKSPACE, E_RANGE = 0, -1, -2, -4
AUTO, GLOBAL, TILED = -1, 0, 1
FAKE = 0x10000          # a 256-byte aligned address that is never dereferenced
N = 1000


@pytest.fixture(scope='module')
def lib():
    return _native.lib()


def geom(res=0.05, size=200, win=None):
    x0, y0, w, h = win if win else (0, 0, size, size)
    return _native.Geom(-5.0, -5.0, res, size, size, x0, y0, w, h)


GOOD = geom()
BAD = geom(win=(0, 0, 300, 10))              # window outside the grid
SUB = geom(win=(10, 10, 100, 100))           # valid, but not the whole grid
FINE = geom(res=0.01, size=64)               # 1 cm cells: the TILED window does not fit in shared memory


def ws_bytes(lib, g, n, strategy):
    return lib.occgrid_workspace_bytes(g, n, strategy)


def maps_ws_bytes(lib, g, n_agents, n, strategy):
    return lib.occgrid_agent_maps_workspace_bytes(g, n_agents, n, strategy)


def check(lib, rc, want, key):
    assert rc == want, (rc, lib.occgrid_last_error())
    if key is not None:
        assert key.encode() in lib.occgrid_last_error(), lib.occgrid_last_error()


# ---- occgrid_integrate_packets / _agent_maps / occgrid_accumulate_packets -------------------------
# (overrides, expected code, key word); the defaults are a valid call of N records at stride 42.
PACKET_CASES = [
    (dict(geom=BAD), E_ARG, 'window'),
    (dict(n=-1), E_ARG, '2^29'),
    (dict(n=1 << 29), E_ARG, '2^29'),
    (dict(rec_len=40), E_ARG, 'rec_len'),
    (dict(stride=41), E_ARG, 'stride'),
    (dict(stride=65), E_ARG, 'stride'),
    (dict(rec_len=41, stride=40), E_ARG, 'stride'),
    (dict(n_agents=0), E_ARG, 'n_agents'),
    (dict(agent_off=None), E_ARG, 'agent offset table'),
    (dict(out=None), E_ARG, 'NULL'),
    (dict(ws=None), E_ARG, 'NULL'),
    (dict(pkts=None), E_ARG, 'packets'),
    (dict(strategy=7), E_ARG, 'unknown strategy'),
    (dict(geom=FINE, strategy=TILED), E_RANGE, 'TILED'),
    # order: n == 0 returns before the packets and the strategy are looked at, not before the rest
    (dict(n=0, strategy=7), OK, None),
    (dict(n=0, pkts=None), OK, None),
    (dict(n=0, geom=FINE, strategy=TILED), OK, None),
    (dict(n=0, out=None), E_ARG, 'NULL'),
    (dict(n=0, rec_len=40), E_ARG, 'rec_len'),
    (dict(n=0, n_agents=0), E_ARG, 'n_agents'),
    (dict(n=0, geom=BAD), E_ARG, 'window'),
]


def call_packets(lib, fn, g, n_agents=4, **kw):
    a = dict(geom=g, pkts=FAKE, n=N, stride=42, rec_len=42, agent_idx=None, drift=None, agent_off=FAKE,
             n_agents=n_agents, out=FAKE, ws=FAKE, ws_bytes=1 << 40, strategy=GLOBAL)
    a.update(kw)
    return fn(a['geom'], a['pkts'], a['n'], a['stride'], a['rec_len'], a['agent_idx'], a['drift'], a['agent_off'],
              a['n_agents'], a['out'], a['ws'], a['ws_bytes'], None, a['strategy'], None)


@pytest.mark.parametrize('kw,want,key', PACKET_CASES)
def test_integrate_packets_rejects(lib, kw, want, key):
    check(lib, call_packets(lib, lib.occgrid_integrate_packets, GOOD, **kw), want, key)


@pytest.mark.parametrize('kw,want,key', PACKET_CASES + [
    (dict(geom=SUB), E_ARG, 'whole grid'),
    (dict(n=0, geom=SUB), E_ARG, 'whole grid'),
])
def test_integrate_agent_maps_rejects(lib, kw, want, key):
    check(lib, call_packets(lib, lib.occgrid_integrate_packets_agent_maps, GOOD, **kw), want, key)


def test_agent_maps_stack_overflow(lib):
    huge = _native.Geom(0.0, 0.0, 0.05, 1 << 30, 1 << 30, 0, 0, 1 << 30, 1 << 30)
    check(lib, call_packets(lib, lib.occgrid_integrate_packets_agent_maps, huge, n_agents=1 << 20), E_ARG, 'overflow')
    assert lib.occgrid_agent_maps_workspace_bytes(huge, 1 << 20, N, GLOBAL) == 0


@pytest.mark.parametrize('kw,want,key', PACKET_CASES + [
    (dict(out=FAKE + 4), E_ARG, '8-byte'),
])
def test_accumulate_packets_rejects(lib, kw, want, key):
    # GLOBAL_ATOMIC count mode has no workspace check: every case here returns before the launch.
    check(lib, call_packets(lib, lib.occgrid_accumulate_packets, GOOD, **kw), want, key)


@pytest.mark.parametrize('strategy', [GLOBAL, TILED, AUTO])
def test_packet_workspace_one_byte_short(lib, strategy):
    need = ws_bytes(lib, GOOD, N, strategy)
    assert need > 0
    check(lib, call_packets(lib, lib.occgrid_integrate_packets, GOOD, ws_bytes=need - 1, strategy=strategy),
          E_WORKSPACE, 'workspace')
    need = maps_ws_bytes(lib, GOOD, 4, N, strategy)
    assert need > 0
    check(lib, call_packets(lib, lib.occgrid_integrate_packets_agent_maps, GOOD, ws_bytes=need - 1, strategy=strategy),
          E_WORKSPACE, 'workspace')


def test_accumulate_tiled_workspace_one_byte_short(lib):
    need = ws_bytes(lib, GOOD, N, TILED)
    check(lib, call_packets(lib, lib.occgrid_accumulate_packets, GOOD, ws_bytes=need - 1, strategy=TILED),
          E_WORKSPACE, 'workspace')


# ---- occgrid_integrate_poses: no record checks, 16-byte aligned pose records ------------------------
POSE_CASES = [
    (dict(geom=BAD), E_ARG, 'window'),
    (dict(n=-1), E_ARG, '2^29'),
    (dict(n=1 << 29), E_ARG, '2^29'),
    (dict(out=None), E_ARG, 'NULL'),
    (dict(ws=None), E_ARG, 'NULL'),
    (dict(recs=None), E_ARG, '16-byte'),
    (dict(recs=FAKE + 8), E_ARG, '16-byte'),
    (dict(strategy=7), E_ARG, 'unknown strategy'),
    (dict(geom=FINE, strategy=TILED), E_RANGE, 'TILED'),
    (dict(n=0, strategy=7), OK, None),
    (dict(n=0, recs=None), OK, None),
    (dict(n=0, out=None), E_ARG, 'NULL'),
]


def call_poses(lib, **kw):
    a = dict(geom=GOOD, recs=FAKE, n=2048, out=FAKE, ws=FAKE, ws_bytes=1, strategy=GLOBAL)
    a.update(kw)
    return lib.occgrid_integrate_poses(a['geom'], a['recs'], a['n'], 1, a['out'], a['ws'], a['ws_bytes'], None,
                                       a['strategy'], None)


@pytest.mark.parametrize('kw,want,key', POSE_CASES)
def test_integrate_poses_rejects(lib, kw, want, key):
    check(lib, call_poses(lib, **kw), want, key)


def test_integrate_poses_workspace_one_byte_short(lib):
    need = ws_bytes(lib, GOOD, 2048, GLOBAL)
    check(lib, call_poses(lib, ws_bytes=need - 1, strategy=GLOBAL), E_WORKSPACE, 'workspace')
    # the pose-record layout of TILED is that of one band segment of the same size
    need = lib.occgrid_band_workspace_bytes(GOOD, 1, 2048)
    assert need > 0
    check(lib, call_poses(lib, ws_bytes=need - 1, strategy=TILED), E_WORKSPACE, 'workspace')
    check(lib, call_poses(lib, ws_bytes=need - 1, strategy=AUTO), E_WORKSPACE, 'workspace')


# ---- occgrid_update_rays: the strategy argument is ignored ------------------------------------------
@pytest.mark.parametrize('kw,want,key', [
    (dict(geom=BAD), E_ARG, 'window'),
    (dict(n=-1), E_ARG, '2^31'),
    (dict(n=(1 << 31) - 1), E_ARG, '2^31'),
    (dict(out=None), E_ARG, 'NULL'),
    (dict(ws=None), E_ARG, 'NULL'),
    (dict(rays=None), E_ARG, 'NULL'),
    (dict(hit=None), E_ARG, 'NULL'),
    (dict(rays=FAKE + 8), E_ARG, '16-byte'),
    (dict(ws_bytes=200 * 200 * 4 - 1), E_WORKSPACE, 'workspace'),
    (dict(ws_bytes=200 * 200 * 4 - 1, strategy=7), E_WORKSPACE, 'workspace'),
    (dict(n=0, strategy=7), OK, None),
])
def test_update_rays_rejects(lib, kw, want, key):
    a = dict(geom=GOOD, rays=FAKE, hit=FAKE, n=N, out=FAKE, ws=FAKE, ws_bytes=1, strategy=GLOBAL)
    a.update(kw)
    rc = lib.occgrid_update_rays(a['geom'], a['rays'], a['hit'], a['n'], a['out'], a['ws'], a['ws_bytes'], None,
                                 a['strategy'], None)
    check(lib, rc, want, key)


# ---- occgrid_route_packets (n > 0 throughout: with n == 0 it clears the band counts) -----------------
@pytest.mark.parametrize('kw,want,key', [
    (dict(geom=BAD), E_ARG, 'window'),
    (dict(n_bands=0), E_ARG, 'n_bands'),
    (dict(n_bands=33), E_ARG, 'n_bands'),
    (dict(band_y0=None), E_ARG, 'n_bands'),
    (dict(n=-1), E_ARG, '2^29'),
    (dict(n=1 << 29), E_ARG, '2^29'),
    (dict(rec_len=40), E_ARG, 'rec_len'),
    (dict(stride=41), E_ARG, 'stride'),
    (dict(stride=65), E_ARG, 'stride'),
    (dict(n_agents=0), E_ARG, None),
    (dict(agent_off=None), E_ARG, None),
    (dict(send=None), E_ARG, None),
    (dict(band_counts=None), E_ARG, None),
    (dict(status=None), E_ARG, None),
    (dict(ws=None), E_ARG, None),
    (dict(send=FAKE + 8), E_ARG, '16-byte'),
    (dict(capacity=1 << 32), E_ARG, 'capacity'),
    (dict(ws_bytes='short'), E_WORKSPACE, 'workspace'),
])
def test_route_packets_rejects(lib, kw, want, key):
    a = dict(geom=GOOD, n_bands=2, band_y0=(C.c_int32 * 3)(0, 100, 200), pkts=FAKE, n=N, stride=42, rec_len=42,
             agent_off=FAKE, n_agents=4, send=FAKE, capacity=4 * N, band_counts=FAKE, status=FAKE, ws=FAKE,
             ws_bytes=1 << 40)
    a.update(kw)
    if a['ws_bytes'] == 'short':
        a['ws_bytes'] = lib.occgrid_route_workspace_bytes(a['n'], a['n_bands']) - 1
    rc = lib.occgrid_route_packets(a['geom'], a['n_bands'], a['band_y0'], a['pkts'], a['n'], a['stride'], a['rec_len'],
                                   None, None, a['agent_off'], a['n_agents'], a['send'], a['capacity'],
                                   a['band_counts'], a['status'], None, a['ws'], a['ws_bytes'], None)
    check(lib, rc, want, key)


# ---- occgrid_band_raycast_route with a bad route job ---------------------------------------------
# The workspace is 1 byte: a job that passed every check would stop at E_WORKSPACE, before any launch.
def route_job(**kw):
    j = _native.RouteJob()
    a = dict(pkts=FAKE, n=N, stride=42, rec_len=42, agent_off=FAKE, n_agents=4, ordinal_base=0, res=0.05,
             size_x=200, n_bands=2, src_rank=0, peer_recs=FAKE, peer_tiles=FAKE, seg_capacity=2048, resv=FAKE,
             status=FAKE)
    a.update(kw)
    j.d_packets, j.n, j.stride, j.rec_len = a['pkts'], a['n'], a['stride'], a['rec_len']
    j.d_agent_off, j.n_agents, j.ordinal_base = a['agent_off'], a['n_agents'], a['ordinal_base']
    j.ox, j.oy, j.res, j.size_x = -5.0, -5.0, a['res'], a['size_x']
    j.n_bands, j.src_rank = a['n_bands'], a['src_rank']
    for b in range(33):
        j.band_y0[b] = min(b, a['n_bands']) * 100
    j.d_peer_recs, j.d_peer_tiles, j.seg_capacity = a['peer_recs'], a['peer_tiles'], a['seg_capacity']
    j.d_resv, j.d_status = a['resv'], a['status']
    return j


@pytest.mark.parametrize('kw,want,key', [
    (dict(pkts=None), E_ARG, 'band_raycast_route'),
    (dict(agent_off=None), E_ARG, 'band_raycast_route'),
    (dict(n_agents=0), E_ARG, 'band_raycast_route'),
    (dict(peer_recs=None), E_ARG, 'band_raycast_route'),
    (dict(peer_tiles=None), E_ARG, 'band_raycast_route'),
    (dict(resv=None), E_ARG, 'band_raycast_route'),
    (dict(status=None), E_ARG, 'band_raycast_route'),
    (dict(n_bands=0), E_ARG, 'n_bands'),
    (dict(n_bands=33), E_ARG, 'n_bands'),
    (dict(src_rank=2), E_ARG, 'n_bands'),
    (dict(src_rank=-1), E_ARG, 'n_bands'),
    (dict(rec_len=40), E_ARG, 'rec_len'),
    (dict(stride=41), E_ARG, 'stride'),
    (dict(stride=65), E_ARG, 'stride'),
    (dict(n=1 << 29), E_ARG, '2^29'),
    (dict(ordinal_base=(1 << 29) - N), E_ARG, '2^29'),
    (dict(seg_capacity=4096), E_ARG, 'segment capacity'),
    (dict(res=0.01), E_RANGE, 'thinner'),                # 100-row bands; reach 122 cells at 1 cm, 26 at 5 cm
    (dict(n_bands=4, src_rank=3), E_WORKSPACE, None),
    (dict(n=0, pkts=None), E_WORKSPACE, None),           # an empty job is no job
    (dict(ordinal_base=(1 << 29) - 1 - N), E_WORKSPACE, None),
    (dict(), E_WORKSPACE, None),
])
def test_band_route_job_rejects(lib, kw, want, key):
    j = route_job(**kw)
    rc = lib.occgrid_band_raycast_route(GOOD, FAKE, 2, 2048, 1, C.byref(j), FAKE, FAKE, 1, None, None)
    check(lib, rc, want, key)


@pytest.mark.parametrize('kw,want,key', [
    (dict(geom=BAD), E_ARG, 'window'),
    (dict(grid=None), E_ARG, 'NULL'),
    (dict(ws=None), E_ARG, 'NULL'),
    (dict(slot=None), E_ARG, 'NULL'),
    (dict(n_segs=0), E_ARG, 'segments'),
    (dict(n_segs=33), E_ARG, 'segments'),
    (dict(seg_cap=1000), E_ARG, 'segments'),
])
def test_band_raycast_route_rejects(lib, kw, want, key):
    a = dict(geom=GOOD, slot=FAKE, n_segs=2, seg_cap=2048, grid=FAKE, ws=FAKE)
    a.update(kw)
    rc = lib.occgrid_band_raycast_route(a['geom'], a['slot'], a['n_segs'], a['seg_cap'], 1, None, a['grid'], a['ws'], 1,
                                        None, None)
    check(lib, rc, want, key)


# ---- workspace sizes --------------------------------------------------------------------------------
@pytest.mark.parametrize('args,key', [
    ((BAD, N, GLOBAL), 'window'),
    ((GOOD, -1, GLOBAL), 'max_packets'),
    ((GOOD, N, 7), 'unknown strategy'),
    ((FINE, N, TILED), 'TILED'),
])
def test_workspace_bytes_rejects(lib, args, key):
    assert lib.occgrid_workspace_bytes(*args) == 0
    assert key.encode() in lib.occgrid_last_error()


@pytest.mark.parametrize('args,key', [
    ((BAD, 4, N, GLOBAL), 'window'),
    ((SUB, 4, N, GLOBAL), 'whole grid'),
    ((GOOD, 0, N, GLOBAL), 'n_agents'),
    ((GOOD, 4, -1, GLOBAL), 'max_packets'),
    ((GOOD, 4, N, 7), 'unknown strategy'),
    ((FINE, 4, N, TILED), 'TILED'),
])
def test_agent_maps_workspace_bytes_rejects(lib, args, key):
    assert lib.occgrid_agent_maps_workspace_bytes(*args) == 0
    assert key.encode() in lib.occgrid_last_error()


@pytest.mark.parametrize('args', [(BAD, 2, 2048), (GOOD, 0, 2048), (GOOD, 33, 2048), (GOOD, 2, 1000), (GOOD, 2, 0),
                                  (GOOD, 2, 1 << 31)])
def test_band_workspace_bytes_rejects(lib, args):
    assert lib.occgrid_band_workspace_bytes(*args) == 0


# Byte counts callers allocate from (0: the strategy does not support the geometry).
GEOMS = {
    'g200': geom(),
    'g4096': _native.Geom(-102.4, -102.4, 0.05, 4096, 4096, 0, 0, 4096, 4096),
    'win': _native.Geom(-10.0, -10.0, 0.05, 1000, 800, 100, 50, 700, 600),
    'fine': FINE,
    'coarse': _native.Geom(0.0, 0.0, 0.2, 333, 77, 0, 0, 333, 77),
}
WS_PINNED = {                 # (geometry, max_packets): bytes under (AUTO, GLOBAL_ATOMIC, TILED)
    ('g200', 0): (162816, 160000, 162816),
    ('g200', 2_049): (294400, 160000, 294400),
    ('g200', 2_500_000): (160323584, 160000, 160323584),
    ('g4096', 0): (67181312, 67108864, 67181312),
    ('g4096', 2_049): (67345152, 67108864, 67345152),
    ('g4096', 2_500_000): (227411200, 67108864, 227411200),
    ('win', 0): (1684992, 1680128, 1684992),
    ('win', 2_049): (1818624, 1680128, 1818624),
    ('win', 2_500_000): (161847808, 1680128, 161847808),
    ('fine', 0): (16384, 16384, 0),
    ('fine', 2_049): (16384, 16384, 0),
    ('fine', 2_500_000): (16384, 16384, 0),
}
MAPS_WS_PINNED = {            # (geometry, n_agents, max_packets): bytes under (AUTO, GLOBAL_ATOMIC, TILED)
    ('g200', 1, 1): (162816, 160000, 162816),
    ('g200', 1, 100_000): (6568704, 160000, 6568704),
    ('g200', 64, 1): (10279680, 10240000, 10279680),
    ('g200', 64, 100_000): (16721920, 10240000, 16721920),
    ('g200', 300, 1): (48174848, 48000000, 48174848),
    ('g200', 300, 100_000): (54753024, 48000000, 54753024),
    ('coarse', 1, 1): (105472, 102656, 105472),
    ('coarse', 1, 100_000): (6511360, 102656, 6511360),
    ('coarse', 64, 1): (6599680, 6564096, 6599680),
    ('coarse', 64, 100_000): (13037824, 6564096, 13037824),
    ('coarse', 300, 1): (30925824, 30769408, 30925824),
    ('coarse', 300, 100_000): (37484800, 30769408, 37484800),
    ('fine', 1, 1): (16384, 16384, 0),
    ('fine', 1, 100_000): (16384, 16384, 0),
    ('fine', 64, 1): (1048576, 1048576, 0),
    ('fine', 64, 100_000): (1048576, 1048576, 0),
    ('fine', 300, 1): (4915200, 4915200, 0),
    ('fine', 300, 100_000): (4915200, 4915200, 0),
    ('g4096', 3851, 1): (258704636672, 258436235264, 258704636672),   # 3851 * 66^2 tile keys <= 2^24
    ('g4096', 3852, 1): (258503344128, 258503344128, 0),              # one agent more: TILED runs out of keys
}
BAND_WS_PINNED = {            # (geometry, n_segs, seg_capacity): bytes
    ('g200', 1, 2048): 178432,
    ('g200', 1, 65536): 690432,
    ('g200', 8, 2048): 294144,
    ('g200', 8, 65536): 4389120,
    ('win', 1, 2048): 1702656,
    ('win', 1, 65536): 2214400,
    ('win', 8, 2048): 1818112,
    ('win', 8, 65536): 5913088,
}


def test_workspace_bytes_pinned(lib):
    got = {k: tuple(lib.occgrid_workspace_bytes(GEOMS[k[0]], k[1], s) for s in (AUTO, GLOBAL, TILED)) for k in WS_PINNED}
    assert got == WS_PINNED


def test_agent_maps_workspace_bytes_pinned(lib):
    got = {k: tuple(lib.occgrid_agent_maps_workspace_bytes(GEOMS[k[0]], k[1], k[2], s) for s in (AUTO, GLOBAL, TILED))
           for k in MAPS_WS_PINNED}
    assert got == MAPS_WS_PINNED


def test_band_workspace_bytes_pinned(lib):
    got = {k: lib.occgrid_band_workspace_bytes(GEOMS[k[0]], k[1], k[2]) for k in BAND_WS_PINNED}
    assert got == BAND_WS_PINNED
