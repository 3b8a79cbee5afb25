"""Count mode on the GPU (occgrid_accumulate_packets, occgrid_counts_to_logodds) against the C count
reference (oracle/occgrid_oracle.c: oracle_accumulate_packets), under both strategies, bit for bit:
random geometry and streams, every line shape of a long beam (TILED's recurrence walk, taken by
beams of more than 33 cells), windows, cells that collect hundreds of thousands of counts from
hundreds of work items, the full configs[1] batch, several kinds of input stream, and log-odds
equal to a float64 NumPy evaluation, bit for bit."""
import math

import numpy as np
import pytest

from oracle import c_oracle
from test_count_reference import RECORD, fma_sensitive_counts, logodds_reference, make_packets

pytestmark = pytest.mark.gpu
torch = pytest.importorskip('torch')
hyp = pytest.importorskip('hypothesis')
from hypothesis import given, settings, strategies as st_, HealthCheck

STRATEGIES = ('global_atomic', 'tiled')
PACKET_COUNTERS = ('packets', 'accepted', 'dropped', 'bad_pose', 'beams', 'hits')
SENSOR_ANGLES = (0.0, math.pi / 2, math.pi, -math.pi / 2)
LOGODDS_PARAMS = [
    (0.85, -0.4, -2.0, 3.5),          # the defaults
    (0.9, -0.35, -4.0, 4.0),
    (0.85, -0.4, 1.25, 1.25),         # l_min == l_max: every cell is the bound
    (-0.7, 0.3, -3.0, 3.0),           # negative l_occ
    (0.85, -0.4, -1e30, 1e30),        # nothing clamped
    (0.0, 0.0, -2.0, 3.5),            # zero weights
]


@pytest.fixture(scope='module')
def M():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper
    return dual_bot_mapper


def planes(g):
    """int32 [h, w, 2] = {miss, hit}, the layout of the C reference."""
    return g.counts_tensor.cpu().numpy()


def reference(pk, size, res, ox, oy, window=None, counts=None, **kw):
    x0, y0, w, h = window if window is not None else (0, 0, size, size)
    if counts is None:
        counts = np.zeros((h, w, 2), np.int32)
    c = c_oracle.accumulate_packets(pk, counts, ox, oy, res, window=(x0, y0), size_x=size, size_y=size, **kw)
    return counts, c


def assert_packet_counters(g, c):
    got = g.counters()
    assert {k: got[k] for k in PACKET_COUNTERS} == {k: c[k] for k in PACKET_COUNTERS}


def assert_log_odds(g, counts):
    """The kernel rounds h * l_occ and m * l_free to float64, adds, clamps, rounds to float32: the
    same operations as NumPy, so the result must be identical to the bit."""
    for p in LOGODDS_PARAMS:
        got = g.log_odds(*p)
        want = logodds_reference(counts, *p)
        assert got.dtype == np.float32 and np.array_equal(got.view(np.uint32), want.view(np.uint32)), p


def posed_packets(x, y, yaw, dists):
    """v2 records of agent 1 at float32 poses (x, y, yaw) with the four ranges `dists`."""
    n = len(x)
    out = np.zeros((n, 42), np.uint8)
    rec = out.view(RECORD)[:, 0]
    rec['magic'] = b'QSRL'
    rec['agent'] = 1
    rec['x'], rec['y'], rec['yaw'] = x, y, yaw
    rec['d'] = np.asarray(dists, np.float32)
    return out


# ---- a. random geometry and streams ----------------------------------------------------------

@settings(max_examples=30, deadline=None, suppress_health_check=[HealthCheck.too_slow])
@given(seed=st_.integers(0, 2 ** 31 - 1), size=st_.integers(8, 700), res=st_.sampled_from([0.03, 0.035, 0.05, 0.1, 0.2]),
       stride=st_.sampled_from([42, 48, 64]), windowed=st_.booleans(), use_drift=st_.booleans())
def test_random_geometry_and_streams(M, seed, size, res, stride, windowed, use_drift):
    rng = np.random.default_rng(seed)
    ox, oy = float(rng.uniform(-50, 10)), float(rng.uniform(-50, 10))
    n_agents = int(rng.integers(1, 6))
    offs = np.zeros((n_agents + 1, 2))
    offs[1:] = rng.uniform(-1, 1, (n_agents, 2))
    n = int(rng.integers(1, 6000))
    buf = np.zeros((n, stride), np.uint8)
    buf[:, :42] = make_packets(rng, n, size * res, ox, oy, n_agents)
    drift = rng.normal(0, 0.05, (n, 2)) if use_drift else None
    window = None
    if windowed:
        x0, y0 = int(rng.integers(0, size)), int(rng.integers(0, size))
        window = (x0, y0, int(rng.integers(1, size - x0 + 1)), int(rng.integers(1, size - y0 + 1)))
    want, c = reference(buf, size, res, ox, oy, window, agent_offsets=offs, drift=drift)
    half = n // 2
    for strategy in STRATEGIES:
        try:
            g = M.OccupancyGrid(size, res, ox, oy, window=window, strategy=strategy, max_batch=n)
        except M.OccGridError:
            assert strategy == 'tiled'
            continue                    # TILED refuses this geometry (never for these resolutions: see below)
        g.accumulate_packets(buf[:half], agent_offsets=offs, drift=None if drift is None else drift[:half])
        g.accumulate_packets(buf[half:], agent_offsets=offs, drift=None if drift is None else drift[half:])
        assert np.array_equal(planes(g), want), strategy
        assert_packet_counters(g, c)
        if strategy == 'global_atomic':
            assert g.counters()['updates'] == c['updates']


@pytest.mark.parametrize('res', [0.03, 0.035, 0.028])
def test_tiled_accepts_long_beam_resolutions(M, res):
    """Below 0.0375 m a 1.2 m beam spans more than 33 cells and TILED walks it with the recurrence
    instead of the mask table; the tests above and below only reach that walk if TILED takes them."""
    g = M.OccupancyGrid(700, res, strategy='tiled')          # raises OccGridError if TILED refuses
    pk = posed_packets(np.array([g.ox + 350.5 * res]), np.array([g.oy + 350.5 * res]), np.array([0.1]), [[3.0] * 4])
    g.accumulate_packets(pk)
    want, c = reference(pk, 700, res, g.ox, g.oy)
    assert np.array_equal(planes(g), want) and want[350, 350, 0] == 4 and c['updates'] > 4 * 34


# ---- b. long beams ---------------------------------------------------------------------------

def line_shape_packets(res, ox, oy, reach=40):
    """One packet per integer offset (dx, dy), max(|dx|, |dy|) <= reach and at most 1.19 m: the
    front beam aimed from a cell centre at the centre of the cell (dx, dy) away, as a hit and as a
    1.2 m miss; the other three beams come along (a hit, a miss below MIN_DIST, a hit)."""
    xs, ys, yaws, d0, lengths = [], [], [], [], []
    slot = 0
    for dy in range(-reach, reach + 1):
        for dx in range(-reach, reach + 1):
            r = math.hypot(dx, dy) * res
            if r > 1.19 or (dx == 0 and dy == 0):
                continue
            cx, cy = 50 + 30 * (slot % 90), 50 + 30 * (slot // 90)
            slot += 1
            for d in (r, 3.0):
                xs.append(ox + (cx + 0.5) * res)
                ys.append(oy + (cy + 0.5) * res)
                yaws.append(math.atan2(dy, dx))
                d0.append(d)
            lengths.append(max(abs(dx), abs(dy)) + 1)
    n = len(xs)
    dists = np.stack([d0, 0.3 + 0.01 * (np.arange(n) % 50), np.zeros(n), np.ones(n)], axis=1)
    return posed_packets(np.array(xs), np.array(ys), np.array(yaws), dists), max(lengths), 50 + 30 * (slot // 90) + 100


@pytest.mark.parametrize('res', [0.03, 0.028])
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_long_beams_all_line_shapes(M, strategy, res):
    ox = oy = -20.0
    pk, longest, extent = line_shape_packets(res, ox, oy)
    assert longest > 33 + 6                         # hit beams of up to 40 cells, not only the mask table's 33
    size = max(extent, 2800)
    want, c = reference(pk, size, res, ox, oy)
    g = M.OccupancyGrid(size, res, ox, oy, strategy=strategy, max_batch=len(pk))
    g.accumulate_packets(pk)
    assert np.array_equal(planes(g), want)
    assert_packet_counters(g, c)
    assert g.counters()['updates'] == c['updates'] and c['packets'] > 9000


# ---- c. windows ------------------------------------------------------------------------------

WIN_SIZE, WIN_RES, WIN_O = 300, 0.05, -7.5


@pytest.fixture(scope='module')
def window_stream():
    rng = np.random.default_rng(21)
    offs = np.array([[0.0, 0.0], [0.0, 0.0], [0.4, -0.3], [-0.2, 0.1]])
    pk = make_packets(rng, 30_000, WIN_SIZE * WIN_RES, WIN_O, WIN_O, 3)
    drift = rng.normal(0, 0.05, (len(pk), 2))
    kw = dict(agent_offsets=offs, drift=drift)
    full, _ = reference(pk, WIN_SIZE, WIN_RES, WIN_O, WIN_O, **kw)
    assert (full[..., 0] > 0).mean() > 0.99 and full[..., 1].any()     # nearly every cell is crossed,
    assert full[0, :, 0].all() and full[-1, :, 0].all() and full[:, 0, 0].all() and full[:, -1, 0].all()  # every edge cell
    return pk, kw, full


def windowed_planes(M, strategy, window, pk, kw):
    g = M.OccupancyGrid(WIN_SIZE, WIN_RES, WIN_O, WIN_O, window=window, strategy=strategy, max_batch=len(pk))
    g.accumulate_packets(pk, **kw)
    return planes(g)


@pytest.mark.parametrize('strategy', STRATEGIES)
def test_windows_equal_crops(M, window_stream, strategy):
    """Windows of every shape the clips have to get right: not aligned to 64 cells, narrower and
    lower than a tile, one cell wide, one cell high, one cell, touching each edge of the grid."""
    pk, kw, full = window_stream
    assert np.array_equal(windowed_planes(M, strategy, None, pk, kw), full)
    for (x0, y0, w, h) in [(37, 51, 64, 80), (100, 10, 20, 280), (5, 130, 290, 9), (149, 0, 1, 300),
                           (0, 201, 300, 1), (7, 9, 1, 1), (250, 250, 50, 50), (0, 0, 63, 65), (299, 299, 1, 1)]:
        got = windowed_planes(M, strategy, (x0, y0, w, h), pk, kw)
        assert np.array_equal(got, full[y0:y0 + h, x0:x0 + w]), (x0, y0, w, h)


@pytest.mark.parametrize('strategy', STRATEGIES)
def test_window_layouts_sum_to_full_planes(M, window_stream, strategy):
    """Row bands (the multi-GPU layout) and column strips of uneven sizes, placed side by side,
    give the full planes: no count is lost or doubled at a band edge."""
    pk, kw, full = window_stream
    for cuts, axis in (([0, 64, 70, 171, 300], 0), ([0, 1, 100, 229, 300], 1)):
        out = np.zeros_like(full)
        for a, b in zip(cuts[:-1], cuts[1:]):
            win = (0, a, WIN_SIZE, b - a) if axis == 0 else (a, 0, b - a, WIN_SIZE)
            got = windowed_planes(M, strategy, win, pk, kw)
            if axis == 0:
                out[a:b] += got
            else:
                out[:, a:b] += got
        assert np.array_equal(out, full), axis


# ---- d. dense cells --------------------------------------------------------------------------

DENSE_SIZE, DENSE_RES, DENSE_O = 256, 0.05, -6.4
DENSE_DISTS = (0.7, 3.0, 0.45, 0.0)                   # front and back hit; left and right miss 1.2 m out
DENSE_YAW = 0.3


def dense_packets(n, jitter=None):
    """n packets at the centre of cell (150, 140), which lies in the 64 x 64 home tile of cells
    128..191 (the 5 cm pad is one tile); `jitter` spreads the poses over that tile instead."""
    x = np.full(n, DENSE_O + 150.5 * DENSE_RES)
    y = np.full(n, DENSE_O + 140.5 * DENSE_RES)
    if jitter is not None:
        x = DENSE_O + jitter.uniform(128.5, 191.5, n) * DENSE_RES
        y = DENSE_O + jitter.uniform(128.5, 191.5, n) * DENSE_RES
    return posed_packets(x, y, np.full(n, DENSE_YAW), np.tile(DENSE_DISTS, (n, 1)))


def dense_end_cells():
    """End cells of the two hit beams, with the reference's arithmetic (:142-143, :890-891)."""
    rec = dense_packets(1).view(RECORD)[0, 0]
    rx, ry, yaw = float(rec['x']), float(rec['y']), float(rec['yaw'])
    cells = []
    for s in (0, 2):
        d = float(rec['d'][s])
        cells.append((int((rx + d * math.cos(yaw + SENSOR_ANGLES[s]) - DENSE_O) / DENSE_RES),
                      int((ry + d * math.sin(yaw + SENSOR_ANGLES[s]) - DENSE_O) / DENSE_RES)))
    return cells


@pytest.mark.parametrize('n', [70_000, 2_500_000])
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_dense_start_cell(M, strategy, n):
    """Every packet at one pose: the start cell collects 4 n misses (far above 2^16, so the global
    plane has to add up the 16-bit window halves of many work items), each hit end cell n hits.
    70 000 packets of one tile make ~270 work items of 256 packets; 2.5e6 packets make the plan
    choose the largest, 2 048-packet items (8 192 misses of the start cell in one window word)."""
    pk = dense_packets(n)
    g = M.OccupancyGrid(DENSE_SIZE, DENSE_RES, DENSE_O, DENSE_O, strategy=strategy, max_batch=n)
    g.accumulate_packets(pk)
    got = planes(g)
    assert got[140, 150, 0] == 4 * n and got[140, 150, 1] == 0 and 4 * n > 2 ** 17
    for (ex, ey) in dense_end_cells():
        assert got[ey, ex, 1] == n and got[ey, ex, 0] == 0
    want, c = reference(pk, DENSE_SIZE, DENSE_RES, DENSE_O, DENSE_O)
    assert np.array_equal(got, want)
    assert_packet_counters(g, c)
    assert g.counters()['updates'] == c['updates']
    if n < 1_000_000:
        assert_log_odds(g, want)


@pytest.mark.parametrize('strategy', STRATEGIES)
def test_dense_tile_jittered(M, strategy):
    """70 000 poses spread over one 64 x 64 home tile: hundreds of work items of the same tile
    flush overlapping windows into the same cells."""
    n = 70_000
    pk = dense_packets(n, jitter=np.random.default_rng(4))
    g = M.OccupancyGrid(DENSE_SIZE, DENSE_RES, DENSE_O, DENSE_O, strategy=strategy, max_batch=n)
    g.accumulate_packets(pk)
    want, c = reference(pk, DENSE_SIZE, DENSE_RES, DENSE_O, DENSE_O)
    assert np.array_equal(planes(g), want)
    assert want[..., 0].max() > 2 ** 10 and want[..., 1].max() > 40
    assert_packet_counters(g, c)
    assert_log_odds(g, want)


# ---- e. the full configs[1] batch ------------------------------------------------------------

def test_configs1_batch(M):
    """BASELINE configs[1]: 2.5e6 packets of 64 agents into 4096^2 cells at 5 cm, both strategies
    against the C reference.  `updates` is compared too: every robot cell of this session lies
    within reach of the grid, the only packets whose cells TILED counts (DESIGN §7)."""
    from occgrid_b200 import simulation_tools as st
    s = st.generate_session(n_agents=64, n_packets=2_500_000, grid_size=4096, seed=5)
    kw = dict(agent_offsets=s['agent_offsets'], agent_idx=s['agent_idx'])
    geo = s['grid']
    size, res, ox, oy = geo['size'], geo['resolution'], geo['origin_x'], geo['origin_y']
    want, c = reference(s['packets'], size, res, ox, oy, **kw)
    rec = s['packets'].view(RECORD)[:, 0]
    reach = math.ceil(1.2 / res) + 2
    gx = np.trunc((rec['x'].astype(np.float64) + s['agent_offsets'][s['agent_idx'], 0] - ox) / res)
    gy = np.trunc((rec['y'].astype(np.float64) + s['agent_offsets'][s['agent_idx'], 1] - oy) / res)
    assert ((gx >= -reach) & (gx < size + reach) & (gy >= -reach) & (gy < size + reach)).all()
    for strategy in STRATEGIES:
        g = M.OccupancyGrid(strategy=strategy, max_batch=len(s['packets']), **geo)
        g.accumulate_packets(s['packets'], **kw)
        assert np.array_equal(planes(g), want), strategy
        assert_packet_counters(g, c)
        assert g.counters()['updates'] == c['updates']
        if strategy == 'tiled':
            assert_log_odds(g, want)
        del g
        torch.cuda.empty_cache()


# ---- f. streams ------------------------------------------------------------------------------

STREAM_SIZE, STREAM_RES, STREAM_O = 400, 0.05, -10.0


@pytest.fixture(scope='module')
def stream():
    rng = np.random.default_rng(33)
    offs = np.zeros((6, 2))
    offs[1:] = rng.uniform(-1, 1, (5, 2))
    pk = make_packets(rng, 40_000, STREAM_SIZE * STREAM_RES, STREAM_O, STREAM_O, 5)
    drift = rng.normal(0, 0.05, (len(pk), 2))
    return pk, offs, drift


def stream_grid(M, strategy, n=40_000):
    return M.OccupancyGrid(STREAM_SIZE, STREAM_RES, STREAM_O, STREAM_O, strategy=strategy, max_batch=n)


def stream_reference(pk, **kw):
    return reference(pk, STREAM_SIZE, STREAM_RES, STREAM_O, STREAM_O, **kw)


@pytest.mark.parametrize('strategy', STRATEGIES)
def test_stream_calls_accumulate_and_reset(M, stream, strategy):
    """Three calls of uneven size add up on one plane; after reset_counts() one call equals one
    reference call."""
    pk, offs, drift = stream
    g = stream_grid(M, strategy)
    for a, b in ((0, 1), (1, 17_000), (17_000, 40_000)):
        g.accumulate_packets(pk[a:b], agent_offsets=offs, drift=drift[a:b])
    want, c = stream_reference(pk, agent_offsets=offs, drift=drift)
    assert np.array_equal(planes(g), want)
    assert_packet_counters(g, c)
    g.reset_counts()
    g.accumulate_packets(pk[5_000:9_000], agent_offsets=offs)
    want, _ = stream_reference(pk[5_000:9_000], agent_offsets=offs)
    assert np.array_equal(planes(g), want)


@pytest.mark.parametrize('pinned', [False, True])
@pytest.mark.parametrize('strategy', STRATEGIES)
def test_stream_host_chunks(M, stream, strategy, pinned):
    """A host batch of at least two H2D chunks is copied chunk by chunk on a side stream; drift
    and agent_idx are sliced per chunk.  7 chunks through the 2 device slots."""
    pk, offs, drift = stream
    rng = np.random.default_rng(5)
    idx = rng.integers(1, 6, len(pk)).astype(np.int32)
    g = stream_grid(M, strategy, n=6_000)
    g.h2d_chunk = 6_000
    src = torch.from_numpy(pk)
    if pinned:
        src = src.pin_memory()
    g.accumulate_packets(src, agent_offsets=offs, agent_idx=idx, drift=drift)
    want, c = stream_reference(pk, agent_offsets=offs, agent_idx=idx, drift=drift)
    assert np.array_equal(planes(g), want)
    assert_packet_counters(g, c)


@pytest.mark.parametrize('strategy', STRATEGIES)
def test_stream_agent_idx_override_with_dropped_ids(M, stream, strategy):
    """The out-of-band agent index replaces the wire byte; ids 0, -1 and n_agents + 1 are dropped."""
    pk, offs, drift = stream
    rng = np.random.default_rng(6)
    idx = rng.integers(-1, 7, len(pk)).astype(np.int32)
    g = stream_grid(M, strategy)
    g.accumulate_packets(pk, agent_offsets=offs, agent_idx=idx, drift=drift)
    want, c = stream_reference(pk, agent_offsets=offs, agent_idx=idx, drift=drift)
    assert np.array_equal(planes(g), want)
    assert_packet_counters(g, c)
    assert c['dropped'] > len(pk) // 5


@pytest.mark.parametrize('strategy', STRATEGIES)
def test_stream_v1_records_and_slots(M, stream, strategy):
    """41-byte v1 records back to back (stride 41), and 42-byte records in 48-byte slots."""
    pk, offs, drift = stream
    v1 = np.ascontiguousarray(pk[:, :41])
    g = stream_grid(M, strategy)
    g.accumulate_packets(v1, agent_offsets=offs, drift=drift, rec_len=41)
    want, c = stream_reference(v1, agent_offsets=offs, drift=drift, rec_len=41)
    assert np.array_equal(planes(g), want)
    assert_packet_counters(g, c)
    slots = np.zeros((len(pk), 48), np.uint8)
    slots[:, :42] = pk
    slots[:, 42:] = 0xAB                                           # padding must not be read
    g2 = stream_grid(M, strategy)
    g2.accumulate_packets(slots, agent_offsets=offs, drift=drift)
    want2, _ = stream_reference(pk, agent_offsets=offs, drift=drift)
    assert np.array_equal(planes(g2), want2)


# ---- g. log-odds -----------------------------------------------------------------------------

@pytest.mark.parametrize('p', LOGODDS_PARAMS)
def test_log_odds_bit_exact_on_fma_sensitive_counts(M, p):
    """Counts written straight into the plane, chosen so that a fused multiply-add in the kernel
    would round some cells to a different float32 (tests/test_count_reference.py shows that it
    does); the float64 NumPy evaluation must come out bit for bit."""
    l_occ, l_free = p[0], p[1]
    if l_occ and l_free:
        c = fma_sensitive_counts(l_occ, l_free)
    else:
        c = np.random.default_rng(8).integers(0, 1 << 30, (4096, 2)).astype(np.int32)
    g = M.OccupancyGrid(64, 0.05, strategy='global_atomic', max_batch=1)
    g.counts_tensor.copy_(torch.from_numpy(c.reshape(64, 64, 2)))
    got = g.log_odds(*p)
    want = logodds_reference(c.reshape(64, 64, 2), *p)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
