"""The packet path at the limits its entry points accept, against the C oracle bit for bit.

(a) Batches of 2^29 - 1 records, the most one call takes.  A beam's stamp is (4k + s + 1) << 1 in
    32 bits, so near k = 2^29 it sets bits 24..31; a stamp or an ordinal cut short anywhere on the
    way would let an early record beat a late one.  The batch is built on the device: zero records
    (dropped on the magic) with groups of accepted records at its start, around a segment the
    TILED bin pass claims late, just below 2^28 and at its end, all in the same rooms.
(b) A 65536 x 65536 grid (2^32 cells) on one GPU, the BASELINE configs[3] geometry, with poses
    over the whole map: linear cell indices above 2^31 in the raycast flush, k_home_resolve and the
    global-atomic walk, a window whose first cell lies beyond 2^31, count planes and an agent-map
    stack of more than 2^31 cells.
(c) Decoded pose records ordered by the ordinal they carry (occgrid_integrate_poses with
    ordinals_in_records = 1), ordinals just below 2^29 - 1 interleaved with small ones.

Every case needs tens of GiB of device memory and skips, saying how much, when the device (or for
(b) the host) has less free."""
import ctypes as C
import gc
import os

import numpy as np
import pytest

from agent_maps_util import integrate_packets_agent_maps

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

GiB = 1 << 30
COUNTERS = ('accepted', 'bad_pose', 'beams', 'hits', 'updates')
N_MAX = (1 << 29) - 1
GROUP = 1 << 16
SMALL = 1024                    # 51.2 m grid: 8 rooms, 16 agents
SMALL_ORIGIN = -25.6
N_AGENTS = 16


@pytest.fixture(scope='module')
def M():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper
    return dual_bot_mapper


@pytest.fixture(autouse=True)
def release_device_memory():
    yield
    if torch.cuda.is_available():
        gc.collect()                # a grid held by a reference cycle would keep its workspace
        torch.cuda.empty_cache()


def need_device(nbytes, what):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes + GiB:
        pytest.skip(f'{what}: needs {nbytes / GiB:.1f} GiB of device memory (+1 GiB spare), {free / GiB:.1f} GiB free')


def need_host(nbytes, what):
    avail = os.sysconf('SC_AVPHYS_PAGES') * os.sysconf('SC_PAGE_SIZE')
    if avail < nbytes + 2 * GiB:
        pytest.skip(f'{what}: needs {nbytes / GiB:.1f} GiB of host memory (+2 GiB spare), {avail / GiB:.1f} GiB available')


def workspace_bytes(M, size, window, n, strategy, n_maps=None):
    """occgrid_workspace_bytes (or the agent-map one) of a geometry, without allocating anything."""
    from occgrid_b200 import _native
    x0, y0, w, h = window if window is not None else (0, 0, size, size)
    geom = _native.Geom(-102.4, -102.4, 0.05, size, size, x0, y0, w, h)
    lib, s = _native.lib(), _native.STRATEGY[strategy]
    if n_maps is None:
        return lib.occgrid_workspace_bytes(C.byref(geom), n, s)
    return lib.occgrid_agent_maps_workspace_bytes(C.byref(geom), n_maps, n, s)


def assert_rows_equal(dev, want, rows=1024):
    """Whole-array comparison of a device tensor with a host array, a slice of rows at a time."""
    assert tuple(dev.shape) == want.shape
    for y in range(0, want.shape[0], rows):
        got = dev[y:y + rows].cpu().numpy()
        if not np.array_equal(got, want[y:y + rows]):
            at = np.argwhere(got != want[y:y + rows])[0]
            raise AssertionError(f'first difference at index {(y + at[0],) + tuple(at[1:])}: '
                                 f'device {got[tuple(at)]}, oracle {want[y:y + rows][tuple(at)]}')


def assert_counters(k, c, n, updates=True):
    """k: device counters of a batch of n records; c: oracle counters over its non-zero records.
    updates=False for TILED on a window: it counts only the beams of packets homed in the window."""
    for name in COUNTERS:
        if name != 'updates' or updates:
            assert k[name] == c[name], name
    assert k['packets'] == n
    assert k['dropped'] == n - c['accepted'] - c['bad_pose']


# ---- (b) 2^32 cells ---------------------------------------------------------------------------

HUGE = 65536


@pytest.fixture(scope='module')
def huge_session(M):
    """BASELINE configs[3] geometry: 1024 agents (ids from agent_idx) on 65536^2, poses anywhere."""
    from occgrid_b200 import simulation_tools as st
    s = st.generate_session(n_agents=1024, n_packets=2_000_000, grid_size=HUGE, seed=31)
    s = st.disperse_poses(s, seed=32)
    s['dev_packets'] = torch.from_numpy(s['packets']).cuda()
    s['dev_agent_idx'] = torch.from_numpy(s['agent_idx']).cuda()
    return s


@pytest.mark.parametrize('strategy,window', [
    pytest.param(strategy, window, id=f'{strategy}-{name}') for strategy in ('tiled', 'global_atomic')
    for name, window in (('full', None), ('window_beyond_2_31', (0, 40000, HUGE, 20000)))])   # 40000 * 65536 > 2^31
def test_grid_above_2_31_cells(M, huge_session, strategy, window):
    from oracle import c_oracle
    s = huge_session
    n = s['packets'].shape[0]
    x0, y0, w, h = window if window is not None else (0, 0, HUGE, HUGE)
    need_device(w * h + workspace_bytes(M, HUGE, window, n, strategy), f'{strategy} on a {w} x {h} window of 65536^2')
    need_host(w * h + (1 << 26), f'oracle grid of {w} x {h}')
    g = M.OccupancyGrid(strategy=strategy, window=window, max_batch=n, **s['grid'])
    g.update_packets(s['dev_packets'], agent_offsets=s['agent_offsets'], agent_idx=s['dev_agent_idx'])
    want = np.full((h, w), -1, np.int8)
    c = c_oracle.integrate_packets(s['packets'], want, -102.4, -102.4, 0.05, agent_offsets=s['agent_offsets'],
                                   agent_idx=s['agent_idx'], window=(x0, y0), size_x=HUGE, size_y=HUGE)
    assert (want[max(0, 32768 - y0):] != -1).any()          # cells beyond linear index 2^31 were written
    assert_rows_equal(g.grid_tensor, want)
    assert_counters(g.counters(), c, n, updates=window is None or strategy == 'global_atomic')


def test_counts_window_above_2_31_cells(M, huge_session):
    from oracle import c_oracle
    s = huge_session
    n = s['packets'].shape[0]
    x0, y0, w, h = 0, 16384, HUGE, 32800            # 2^31 + 15 * 2^17 cells, the last beyond global index 2^31 too
    need_device(w * h * 9 + workspace_bytes(M, HUGE, (x0, y0, w, h), n, 'tiled'), 'count planes of a 65536 x 32800 window')
    need_host(w * h * 8 + (1 << 26), 'oracle count planes of 65536 x 32800')
    g = M.OccupancyGrid(strategy='tiled', window=(x0, y0, w, h), max_batch=n, **s['grid'])
    g.accumulate_packets(s['dev_packets'], agent_offsets=s['agent_offsets'], agent_idx=s['dev_agent_idx'])
    want = np.zeros((h, w, 2), np.int32)
    c = c_oracle.accumulate_packets(s['packets'], want, -102.4, -102.4, 0.05, agent_offsets=s['agent_offsets'],
                                    agent_idx=s['agent_idx'], window=(x0, y0), size_x=HUGE, size_y=HUGE)
    assert want[h // 2 + 1:].any()
    assert_rows_equal(g.counts_tensor, want)
    assert_counters(g.counters(), c, n, updates=False)


@pytest.mark.parametrize('strategy', ['tiled', 'global_atomic'])
def test_agent_map_stack_above_2_31_cells(M, strategy):
    """70 maps of 8192^2 (4.7 G cells, keys below 2^24): maps 32.. start beyond cell 2^31."""
    from occgrid_b200 import simulation_tools as st
    A, S = 70, 8192
    cells = A * S * S
    need_device(cells + workspace_bytes(M, S, None, 1_000_000, strategy, A), f'{strategy} stack of {A} maps of {S}^2')
    need_host(cells + (1 << 27), f'oracle stack of {A} maps of {S}^2')
    s = st.disperse_poses(st.generate_session(n_agents=A, n_packets=1_000_000, grid_size=S, seed=37), seed=38)
    g = M.AgentGrids(n_agents=A, strategy=strategy, max_batch=1_000_000, **s['grid'])
    g.update_packets(torch.from_numpy(s['packets']).cuda(), agent_offsets=s['agent_offsets'])
    want = np.full((A, S, S), -1, np.int8)
    c = integrate_packets_agent_maps(s['packets'], want, -102.4, -102.4, 0.05, agent_offsets=s['agent_offsets'])
    assert (want[A - 1] != -1).any()
    for a in range(A):
        assert_rows_equal(g.grids_tensor[a], want[a], rows=S)
    assert_counters(g.counters(), c, s['packets'].shape[0])


# ---- (c) ordinals carried in decoded records ----------------------------------------------------

POSE_REC = np.dtype([('rx', '<f8'), ('ry', '<f8'), ('yaw', '<f4'), ('d', '<f4', (4,)), ('k', '<u4'),
                     ('tile', '<i4'), ('pad', '<u4')])          # occgrid_pose_rec, include/occgrid_b200.h
assert POSE_REC.itemsize == 48


@pytest.mark.parametrize('strategy', ['tiled', 'global_atomic'])
def test_pose_records_ordered_by_ordinal(M, strategy):
    """4096 records: the first half of the stream carries ordinals 0..2047, the second half ordinals
    ending at 2^29 - 2; in the buffer they alternate, the late ones first.  Applied by ordinal they
    must give the packet path's result for the stream in order."""
    from occgrid_b200 import simulation_tools as st
    from oracle import c_oracle
    n = 4096
    s = st.generate_session(n_agents=N_AGENTS, n_packets=n, grid_size=SMALL, origin=(SMALL_ORIGIN, SMALL_ORIGIN), seed=41)
    pk = s['packets'].view(st.PACKET_DTYPE).reshape(-1)
    off = s['agent_offsets'][pk['agent']]
    rec = np.zeros(n, POSE_REC)
    rec['rx'] = pk['x'].astype(np.float64) + off[:, 0]      # decode_packet: wire pose + agent offset
    rec['ry'] = pk['y'].astype(np.float64) + off[:, 1]
    rec['yaw'] = pk['yaw']
    rec['d'] = np.stack([pk['front'], pk['left'], pk['back'], pk['right']], axis=1)
    r = np.arange(n)
    rec['k'] = np.where(r < n // 2, r, (N_MAX - 1) - (n - 1 - r))
    order = np.empty(n, np.int64)
    order[0::2] = np.arange(n // 2, n)
    order[1::2] = np.arange(n // 2)
    g = M.OccupancyGrid(size=SMALL, resolution=0.05, origin_x=SMALL_ORIGIN, origin_y=SMALL_ORIGIN, strategy=strategy,
                        max_batch=n)
    g.update_poses(torch.from_numpy(rec[order].view(np.uint8).reshape(n, 48)).cuda(), ordinals_in_records=True)
    want = np.full((SMALL, SMALL), -1, np.int8)
    c = c_oracle.integrate_packets(s['packets'], want, SMALL_ORIGIN, SMALL_ORIGIN, 0.05, agent_offsets=s['agent_offsets'])
    assert c['accepted'] == n
    assert np.array_equal(g.grid, want)
    assert_counters(g.counters(), c, n)


# ---- (a) 2^29 - 1 records (last in the module: the batch holds 21.5 GiB until it ends) ----------



def group_starts():
    late_seg = N_MAX // 2048 - 600                 # the bin pass claims segments in order: one of the last
    return [0, (1 << 28) - GROUP, late_seg * 2048 - GROUP // 2, N_MAX - GROUP]   # k order; the last ends at 2^29 - 2


@pytest.fixture(scope='module')
def big_batch(M):
    """(device uint8 [N_MAX, 42], host uint8 [4 * GROUP, 42] = its non-zero records in k order,
    agent offsets)."""
    from occgrid_b200 import simulation_tools as st
    need_device(N_MAX * 42 + workspace_bytes(M, SMALL, None, N_MAX, 'tiled'), '2^29 - 1 records and the TILED workspace')
    s = st.generate_session(n_agents=N_AGENTS, n_packets=4 * GROUP, grid_size=SMALL,
                            origin=(SMALL_ORIGIN, SMALL_ORIGIN), seed=29)
    host = s['packets'].copy()
    # dropped on the agent id with a valid magic: 0 and n_agents + 1
    host[5::13, 4] = 0
    host[11::13, 4] = N_AGENTS + 1
    host[7::101, 5:9] = np.frombuffer(np.float32(np.nan).tobytes(), np.uint8)   # bad poses
    dev = torch.zeros((N_MAX, 42), dtype=torch.uint8, device='cuda')
    foreign = torch.arange(1000, N_MAX, 999_983, device='cuda')                  # also between the groups
    dev[foreign, :4] = torch.tensor(list(b'QSRL'), dtype=torch.uint8, device='cuda')
    dev[foreign[0::2], 4] = N_AGENTS + 1
    for j, lo in enumerate(group_starts()):
        dev[lo:lo + GROUP] = torch.from_numpy(host[j * GROUP:(j + 1) * GROUP]).cuda()
    torch.cuda.synchronize()
    return dev, host, s['agent_offsets']


@pytest.mark.parametrize('mode', ['tiled', 'global_atomic', 'counts', 'agent_maps'])
def test_largest_batch(M, big_batch, mode):
    from oracle import c_oracle
    dev, host, off = big_batch
    kw = dict(resolution=0.05, origin_x=SMALL_ORIGIN, origin_y=SMALL_ORIGIN)
    strategy = 'global_atomic' if mode == 'global_atomic' else 'tiled'
    maps = N_AGENTS if mode == 'agent_maps' else None
    need_device(workspace_bytes(M, SMALL, None, N_MAX, strategy, maps), f'{mode} workspace for 2^29 - 1 records')
    if mode == 'agent_maps':
        g = M.AgentGrids(n_agents=N_AGENTS, size=SMALL, strategy='tiled', max_batch=N_MAX, **kw)
        g.update_packets(dev, agent_offsets=off)
        want = np.full((N_AGENTS, SMALL, SMALL), -1, np.int8)
        c = integrate_packets_agent_maps(host, want, SMALL_ORIGIN, SMALL_ORIGIN, 0.05, agent_offsets=off)
        got = g.grids
    elif mode == 'counts':
        g = M.OccupancyGrid(size=SMALL, strategy='tiled', max_batch=N_MAX, **kw)
        g.accumulate_packets(dev, agent_offsets=off)
        want = np.zeros((SMALL, SMALL, 2), np.int32)
        c = c_oracle.accumulate_packets(host, want, SMALL_ORIGIN, SMALL_ORIGIN, 0.05, agent_offsets=off)
        got = g.counts_tensor.cpu().numpy()
    else:
        g = M.OccupancyGrid(size=SMALL, strategy=strategy, max_batch=N_MAX, **kw)
        g.update_packets(dev, agent_offsets=off)
        want = np.full((SMALL, SMALL), -1, np.int8)
        c = c_oracle.integrate_packets(host, want, SMALL_ORIGIN, SMALL_ORIGIN, 0.05, agent_offsets=off)
        got = g.grid
    assert c['accepted'] > 3 * GROUP and c['bad_pose'] > 0 and c['dropped'] > 0
    assert np.array_equal(got, want)
    assert_counters(g.counters(), c, N_MAX)
