"""Packet binning of the TILED strategy (k_home_bin / k_place_runs): every case below stresses one
way the per-CTA grouping of packets by home tile could go wrong.  Each compares the int8 grid and
the counters bit for bit against the C oracle and against strategy='global_atomic'."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

ORIGIN, RES, SIZE = -102.4, 0.05, 4096
PKT_PER_CTA = 2048          # packets per binning CTA (one segment of local bins)


@pytest.fixture(scope='module')
def M():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper
    return dual_bot_mapper


@pytest.fixture(scope='module')
def sess():
    from occgrid_b200 import simulation_tools as st
    return st.generate_session(n_agents=64, n_packets=40_000, seed=21)


def run(M, strategy, batches, agent_offsets, max_batch, drift=None):
    """Integrate `batches` (uint8 [n, 42] each) one call after another into one grid."""
    g = M.OccupancyGrid(size=SIZE, resolution=RES, origin_x=ORIGIN, origin_y=ORIGIN, strategy=strategy, max_batch=max_batch)
    for i, pk in enumerate(batches):
        g.update_packets(pk, agent_offsets=agent_offsets, drift=None if drift is None else drift[i])
    return g.grid.copy(), g.counters()


def oracle(batches, agent_offsets, drift=None):
    from oracle import c_oracle
    want = np.full((SIZE, SIZE), -1, np.int8)
    total = {}
    for i, pk in enumerate(batches):
        c = c_oracle.integrate_packets(pk, want, ORIGIN, ORIGIN, RES, agent_offsets=agent_offsets,
                                       drift=None if drift is None else drift[i])
        for k, v in c.items():
            total[k] = total.get(k, 0) + v
    return want, total


def check(M, batches, agent_offsets, drift=None):
    max_batch = max(len(b) for b in batches)
    want, c = oracle(batches, agent_offsets, drift)
    tiled, kt = run(M, 'tiled', batches, agent_offsets, max_batch, drift)
    glob, kg = run(M, 'global_atomic', batches, agent_offsets, max_batch, drift)
    assert np.array_equal(tiled, want)
    assert np.array_equal(glob, want)
    for name in ('packets', 'accepted', 'dropped', 'bad_pose', 'beams', 'hits', 'updates'):
        assert kt[name] == c[name] == kg[name], name
    assert kt['owned_updates'] == kg['owned_updates'] == c['updates']
    return c


def test_one_home_tile(M, sess):
    """Every packet in one 64x64-cell home tile: each binning CTA holds a single run covering its
    whole segment, and every CTA ranks itself inside the same bin."""
    from occgrid_b200.simulation_tools import PACKET_DTYPE
    n = 3 * PKT_PER_CTA + 77
    rng = np.random.default_rng(1)
    rec = sess['packets'][:n].copy().view(PACKET_DTYPE).reshape(-1)
    off = sess['agent_offsets'][sess['agent_idx'][:n]]
    # cells 2050..2110 of both axes: inside one tile for any tile origin that is a multiple of 64
    wx = rng.uniform(ORIGIN + 2050 * RES + 0.01, ORIGIN + 2110 * RES, n)
    wy = rng.uniform(ORIGIN + 2050 * RES + 0.01, ORIGIN + 2110 * RES, n)
    rec['x'] = (wx - off[:, 0]).astype(np.float32)
    rec['y'] = (wy - off[:, 1]).astype(np.float32)
    c = check(M, [rec.view(np.uint8).reshape(-1, 42)], sess['agent_offsets'])
    assert c['accepted'] == n


def test_dispersed_poses(M, sess):
    """Poses spread over the whole map: almost every run is one packet long."""
    from occgrid_b200 import simulation_tools as st
    d = st.disperse_poses(sess, seed=4)
    check(M, [d['packets']], sess['agent_offsets'])


@pytest.mark.parametrize('n', [1, 255, PKT_PER_CTA - 1, PKT_PER_CTA + 1])
def test_batch_sizes(M, sess, n):
    check(M, [sess['packets'][:n]], sess['agent_offsets'])


def test_dropped_and_bad_poses_interleaved(M, sess):
    """Packets that are never binned (bad magic, unknown agent, NaN / inf pose) between binned
    ones, with a drift table that must be applied to the right packet."""
    from occgrid_b200.simulation_tools import PACKET_DTYPE
    n = 2 * PKT_PER_CTA + 300
    rec = sess['packets'][:n].copy().view(PACKET_DTYPE).reshape(-1)
    raw = rec.view(np.uint8).reshape(-1, 42)
    raw[::7, 0] = ord('X')                       # bad magic
    raw[3::11, 4] = 250                          # agent beyond the offset table
    rec['x'][5::13] = np.float32('nan')
    rec['y'][6::17] = np.float32('inf')
    rec['yaw'][9::19] = np.float32('nan')
    drift = np.random.default_rng(3).normal(0, 0.05, (n, 2))
    c = check(M, [raw], sess['agent_offsets'], drift=[drift])
    assert c['dropped'] > 0 and c['bad_pose'] > 0 and c['accepted'] > n // 2


def test_large_then_small_batch(M, sess):
    """A smaller batch after a larger one in the same grid and workspace: the runs, local bins and
    segment counts the first batch left behind must not leak into the second."""
    pk = sess['packets']
    check(M, [pk[:20_000], pk[25_000:28_000], pk[30_000:30_001]], sess['agent_offsets'])
