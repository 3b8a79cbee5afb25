"""Per-agent maps (occgrid_integrate_packets_agent_maps / AgentGrids): one packet batch into a stack
of agent grids.  Grid a - 1 must equal the single-grid loop run over agent a's records alone (the
C oracle, per agent) bit for bit, and every counter slot must equal those of the single-grid call
on the whole batch, under both strategies."""
import struct

import numpy as np
import pytest

from agent_maps_util import default_agent_offsets, integrate_packets_agent_maps
from conftest import load_packet_stream, normalise_datagrams, session_packets

torch = pytest.importorskip('torch')

STRATEGIES = ['tiled', 'global_atomic']
ORACLE_SLOTS = ('packets', 'accepted', 'dropped', 'bad_pose', 'beams', 'hits', 'updates')
GEOM_DEFAULT = dict(size=200, resolution=0.05, origin_x=-5.0, origin_y=-5.0)
GEOM_ROOM = dict(size=256, resolution=0.05, origin_x=-4.0, origin_y=-6.4)     # room + 1.2 m reach, own frames


# ---- host-only ABI checks (no GPU) ---------------------------------------------------------------

def test_workspace_bytes_host_only():
    from occgrid_b200 import _native
    lib = _native.lib()
    g = _native.Geom(-5.0, -5.0, 0.05, 200, 200, 0, 0, 200, 200)
    for name in ('global_atomic', 'tiled', 'auto'):
        s = _native.STRATEGY[name]
        one, two, many = (lib.occgrid_agent_maps_workspace_bytes(g, a, 1000, s) for a in (1, 2, 64))
        assert 0 < one < two < many, name
        assert many >= 64 * 200 * 200 * 4
    assert lib.occgrid_agent_maps_workspace_bytes(g, 64, 1000, _native.STRATEGY['auto']) == \
        lib.occgrid_agent_maps_workspace_bytes(g, 64, 1000, _native.STRATEGY['tiled'])
    # a single map costs what the single-grid call costs
    assert lib.occgrid_agent_maps_workspace_bytes(g, 1, 1000, 1) == lib.occgrid_workspace_bytes(g, 1000, 1)
    sub = _native.Geom(-5.0, -5.0, 0.05, 200, 200, 0, 0, 100, 200)
    assert lib.occgrid_agent_maps_workspace_bytes(sub, 2, 1000, 0) == 0
    assert b'whole grid' in lib.occgrid_last_error()
    for bad_agents in (0, -3):
        assert lib.occgrid_agent_maps_workspace_bytes(g, bad_agents, 1000, 0) == 0
        assert b'n_agents' in lib.occgrid_last_error()
    huge = _native.Geom(0.0, 0.0, 0.05, 1 << 30, 1 << 30, 0, 0, 1 << 30, 1 << 30)
    assert lib.occgrid_agent_maps_workspace_bytes(huge, 64, 1000, 0) == 0
    assert b'overflow' in lib.occgrid_last_error()


def test_auto_falls_back_when_keys_exceed_2_24_host_only():
    """n_agents * tiles > 2^24: AUTO sizes the GLOBAL_ATOMIC workspace, explicit TILED is refused."""
    from occgrid_b200 import _native
    lib = _native.lib()
    g = _native.Geom(0.0, 0.0, 0.05, 8192, 8192, 0, 0, 8192, 8192)        # 130^2 = 16 900 tiles
    auto = lib.occgrid_agent_maps_workspace_bytes(g, 1000, 1, _native.STRATEGY['auto'])
    assert auto == lib.occgrid_agent_maps_workspace_bytes(g, 1000, 1, _native.STRATEGY['global_atomic']) > 0
    assert lib.occgrid_agent_maps_workspace_bytes(g, 1000, 1, _native.STRATEGY['tiled']) == 0
    assert lib.occgrid_agent_maps_workspace_bytes(g, 900, 1, _native.STRATEGY['tiled']) > 0


# ---- GPU cases -----------------------------------------------------------------------------------

@pytest.fixture(scope='module')
def M():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper
    return dual_bot_mapper


def synthetic(n_packets, seed=3, n_agents=64):
    from occgrid_b200 import simulation_tools as st
    return st.generate_session(n_agents=n_agents, n_packets=n_packets, seed=seed)


def check(M, strategy, n_agents, geom, calls, max_batch=None):
    """`calls`: list of (packets, kwargs) fed to AgentGrids.update_packets one after another; the
    same calls go to the oracle helper (host records; datagram lists normalised like the device
    path) and to one shared OccupancyGrid for the counters.  Returns the AgentGrids."""
    n_max = max(len(p) for p, _ in calls)
    maps = M.AgentGrids(n_agents, strategy=strategy, max_batch=max_batch or n_max, **geom)
    shared = M.OccupancyGrid(strategy=strategy, max_batch=max_batch or n_max, **geom)
    want = np.full((n_agents, geom['size'], geom['size']), -1, np.int8)
    total = dict.fromkeys(ORACLE_SLOTS, 0)
    for pk, kw in calls:
        tab = kw.get('agent_offsets')
        if tab is None:                      # AgentGrids' default: zero but row 2 = (separation, 0)
            tab = default_agent_offsets(n_agents, kw.get('separation', 0.0))
        maps.update_packets(pk, **kw)
        shared.update_packets(pk, **dict(kw, agent_offsets=tab))
        host, drift = pk, kw.get('drift')
        if isinstance(pk, list):
            host, drift = normalise_datagrams(pk, drift)
        elif isinstance(pk, torch.Tensor):
            host = pk.cpu().numpy()
        c = integrate_packets_agent_maps(host, want, geom['origin_x'], geom['origin_y'], geom['resolution'],
                                         rec_len=kw.get('rec_len', 42), drift=drift, agent_offsets=tab,
                                         agent_idx=kw.get('agent_idx'))
        for k in ORACLE_SLOTS:
            total[k] += c[k]
    got = maps.grids
    assert got.shape == want.shape and got.dtype == np.int8
    for a in range(n_agents):
        assert np.array_equal(got[a], want[a]), f'map of agent {a + 1} differs from the oracle'
    k_maps, k_shared = maps.counters(), shared.counters()
    assert k_maps == k_shared
    # TILED counts the cells of packets it bins, i.e. whose robot lies within reach of the grid (the
    # beams of the others cannot touch it); its 'updates' equals the oracle's only when every robot does
    slots = ORACLE_SLOTS if strategy == 'global_atomic' else ORACLE_SLOTS[:-1]
    for name in slots:
        assert k_maps[name] == total[name], name
    return maps


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_golden_dual_session_with_slam(M, strategy):
    """The seeded two-bot session in the reference geometry, SLAM drift on: each bot in its own
    map (bot 2's beams past x = 5 m fall off the 200^2 grid and are clipped cell by cell)."""
    pk, _ = session_packets(time_sorted=True)
    drift, _ = M.slam_drift_table(pk, separation=0.0)
    maps = check(M, strategy, 2, GEOM_DEFAULT, [(pk, dict(drift=drift))])
    assert (maps.grid(1) != -1).sum() > 1000 and (maps.grid(2) != -1).sum() > 1000
    assert np.array_equal(maps.grid(2), maps.grids[1])


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_golden_dual_session_through_ingest_batcher(M, strategy):
    """IngestBatcher drives AgentGrids unchanged: frames of 100 datagrams, SLAM state carried over."""
    pk, _ = session_packets(time_sorted=True)
    maps = M.AgentGrids(2, strategy=strategy, **GEOM_DEFAULT)
    b = M.IngestBatcher(maps, separation=0.0, use_slam=True, capacity=100)
    for d in pk:
        b.push(d)
    b.flush()
    drift, _ = M.slam_drift_table(pk, separation=0.0)
    want = np.full((2, 200, 200), -1, np.int8)
    arr, d = normalise_datagrams(pk, drift)
    c = integrate_packets_agent_maps(arr, want, -5.0, -5.0, 0.05, drift=d)
    assert np.array_equal(maps.grids, want)
    assert maps.counters()['updates'] == c['updates']


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
@pytest.mark.parametrize('name', ['mixed_a', 'mixed_b_sep', 'mixed_c_4096', 'mixed_d_edge'])
def test_adversarial_packet_streams(M, golden, strategy, name):
    """Bad magic, foreign agents, v1/junk datagram sizes, NaN/inf poses, the 96^2 edge geometry."""
    want = golden['packet_streams'][name]
    pk, ref_drift = load_packet_stream(name)
    geom = dict(GEOM_DEFAULT, **want['grid_kwargs'])
    kw = dict(separation=want['separation'])
    if want['slam']:
        kw['drift'] = ref_drift
    check(M, strategy, 2, geom, [(pk, kw)])


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_synthetic_swarm_64_maps(M, strategy):
    """64 agents, 2e5 packets, every agent in its own frame, 256^2 maps."""
    s = synthetic(200_000)
    maps = check(M, strategy, 64, GEOM_ROOM, [(s['packets'], dict(agent_offsets=np.zeros((65, 2))))])
    assert all((maps.grids[a] != -1).any() for a in range(64))


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_more_than_255_agents_through_agent_idx(M, strategy):
    """300 agents on 96^2 maps: the wire byte saturates at 255, agent_idx carries the real id."""
    s = synthetic(60_000, seed=9, n_agents=300)
    assert (s['packets'][:, 4] == 255).any() and s['agent_idx'].max() == 300
    geom = dict(size=96, resolution=0.05, origin_x=-1.6, origin_y=-2.4)
    maps = check(M, strategy, 300, geom, [(s['packets'], dict(agent_offsets=np.zeros((301, 2)), agent_idx=s['agent_idx']))])
    assert (maps.grids[299] != -1).any()


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
@pytest.mark.parametrize('n', [1, 255, 2047, 2049])
def test_batch_sizes(M, strategy, n):
    s = synthetic(3000, seed=17)
    check(M, strategy, 64, GEOM_ROOM, [(s['packets'][:n], dict(agent_offsets=np.zeros((65, 2))))])


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_large_then_small_batches_in_one_workspace(M, strategy):
    s = synthetic(60_000, seed=19)
    z = dict(agent_offsets=np.zeros((65, 2)))
    pk = s['packets']
    check(M, strategy, 64, GEOM_ROOM, [(pk[:40_000], z), (pk[45_000:48_000], z), (pk[50_000:50_001], z)])


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_dropped_and_nan_poses_interleaved_with_drift(M, strategy):
    from occgrid_b200.simulation_tools import PACKET_DTYPE
    s = synthetic(4396, seed=23)
    rec = s['packets'].copy().view(PACKET_DTYPE).reshape(-1)
    raw = rec.view(np.uint8).reshape(-1, 42)
    raw[::7, 0] = ord('X')                       # bad magic
    raw[3::11, 4] = 250                          # agent beyond the table
    rec['x'][5::13] = np.float32('nan')
    rec['y'][6::17] = np.float32('inf')
    rec['yaw'][9::19] = np.float32('nan')
    drift = np.random.default_rng(3).normal(0, 0.05, (len(raw), 2))
    maps = check(M, strategy, 64, GEOM_ROOM, [(raw, dict(agent_offsets=np.zeros((65, 2)), drift=drift))])
    k = maps.counters()
    assert k['dropped'] > 0 and k['bad_pose'] > 0


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_v1_records_and_padded_stride(M, strategy):
    s = synthetic(20_000, seed=11)
    z = np.zeros((65, 2))
    v1 = np.ascontiguousarray(s['packets'][:, :41])
    check(M, strategy, 64, GEOM_ROOM, [(v1, dict(agent_offsets=z, rec_len=41))])
    padded = np.zeros((20_000, 48), np.uint8)
    padded[:, :42] = s['packets']
    check(M, strategy, 64, GEOM_ROOM, [(padded, dict(agent_offsets=z))])


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_one_agent_only_leaves_the_other_maps_unknown(M, strategy):
    s = synthetic(40_000, seed=29)
    pk = s['packets'][s['agent_idx'] == 7]
    z = np.zeros((65, 2))
    maps = check(M, strategy, 64, GEOM_ROOM, [(pk, dict(agent_offsets=z))])
    g = M.OccupancyGrid(strategy=strategy, max_batch=len(pk), **GEOM_ROOM)
    g.update_packets(pk, agent_offsets=z)
    assert np.array_equal(maps.grid(7), g.grid)
    others = np.delete(maps.grids, 6, axis=0)
    assert (others == -1).all()


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_two_agents_on_the_same_cells(M, strategy):
    """Both bots of a room in one frame: the shared grid mixes their beams (last writer wins across
    agents), the agent maps keep them apart."""
    s = synthetic(30_000, seed=31)
    sel = s['agent_idx'] <= 2
    pk = s['packets'][sel]
    z = np.zeros((3, 2))
    maps = check(M, strategy, 2, GEOM_ROOM, [(pk, dict(agent_offsets=z))])
    shared = M.OccupancyGrid(strategy=strategy, max_batch=len(pk), **GEOM_ROOM)
    shared.update_packets(pk, agent_offsets=z)
    g1, g2 = maps.grid(1), maps.grid(2)
    assert ((g1 != -1) & (g2 != -1)).sum() > 1000
    assert not np.array_equal(g1, g2)
    assert not np.array_equal(g1, shared.grid) and not np.array_equal(g2, shared.grid)


@pytest.mark.gpu
def test_streamed_host_batch_full_config(M):
    """The full 2.5e6-packet BASELINE configs[1] batch from host memory into 64 maps (chunked,
    double-buffered H2D)."""
    s = synthetic(2_500_000, seed=42)
    z = np.zeros((65, 2))
    maps = M.AgentGrids(64, max_batch=M.OccupancyGrid.h2d_chunk, **GEOM_ROOM)
    maps.update_packets(s['packets'], agent_offsets=z)
    want = np.full((64, 256, 256), -1, np.int8)
    c = integrate_packets_agent_maps(s['packets'], want, -4.0, -6.4, 0.05, agent_offsets=z)
    assert np.array_equal(maps.grids, want)
    k = maps.counters()
    for name in ORACLE_SLOTS:
        assert k[name] == c[name], name


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_fusion_with_map_merger(M, strategy):
    """The stack goes to MapMerger.merge as is (device views, no copy) and publishes what a fresh
    merger publishes from the oracle's host maps."""
    from occgrid_b200.map_merger import MapMerger
    s = synthetic(100_000, seed=37, n_agents=8)
    z = np.zeros((9, 2))
    maps = check(M, strategy, 8, GEOM_ROOM, [(s['packets'], dict(agent_offsets=z))])
    want = np.full((8, 256, 256), -1, np.int8)
    integrate_packets_agent_maps(s['packets'], want, -4.0, -6.4, 0.05, agent_offsets=z)
    rel = s['agent_offsets'][1:] - s['agent_offsets'][1]
    tf = np.concatenate([rel, np.zeros((8, 1))], axis=1)                      # (tx, ty, theta)
    got, origin = MapMerger().merge(maps.grids_tensor, maps.origins, maps.res, tf)
    ref, ref_origin = MapMerger().merge(want, maps.origins, maps.res, tf)
    assert got is not None and (got == 100).sum() > 100
    assert np.array_equal(got, ref) and origin == ref_origin


@pytest.mark.gpu
def test_fine_resolution_falls_back_to_global_atomics(M):
    """At 1 cm cells the TILED window does not fit: 'tiled' is refused, 'auto' runs GLOBAL_ATOMIC."""
    s = synthetic(8_000, seed=41, n_agents=4)
    geom = dict(size=700, resolution=0.01, origin_x=-1.0, origin_y=-2.5)
    with pytest.raises(M.OccGridError):
        M.AgentGrids(4, strategy='tiled', **geom)
    maps = check(M, 'auto', 4, geom, [(s['packets'], dict(agent_offsets=np.zeros((5, 2))))])
    assert (maps.grids != -1).any()


@pytest.mark.gpu
def test_single_map_methods_raise_and_table_rows_checked(M):
    maps = M.AgentGrids(3, **GEOM_DEFAULT)
    for call in (lambda: maps.update_ray(0, 0, 1, 1, True), lambda: maps.update_rays(np.zeros((1, 4)), np.ones(1)),
                 lambda: maps.update_poses(torch.zeros((1, 48), dtype=torch.uint8, device='cuda')),
                 lambda: maps.accumulate_packets(b''), lambda: maps.log_odds(), lambda: maps.counts_tensor,
                 lambda: maps.get_frontiers(), lambda: maps.frontier_centroids(), lambda: maps.render_overlay()):
        with pytest.raises(M.OccGridError):
            call()
    good = struct.pack(M.PACKET_FMT, b'QSRL', 3, 0.0, 0.0, 0.0, 0, 0, 0.5, 0.5, 0.5, 0.5, 0)
    with pytest.raises(ValueError):
        maps.update_packets([good], agent_offsets=np.zeros((3, 2)))        # 3 agents need 4 rows
    maps.update_packets([good])
    assert (maps.grid(3) != -1).sum() > 0 and (maps.grid(1) == -1).all()
    assert maps.origins.shape == (3, 2) and (maps.origins == [-5.0, -5.0]).all()
    maps.clear()
    assert (maps.grids == -1).all()
