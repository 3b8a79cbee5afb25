"""Hit/miss count planes and log-odds — an EXTENSION beyond the reference (north-star wording,
SURVEY §8c): the reference stores FREE / OCCUPIED (dual_bot_mapper.py:148-156), this mode counts
those stores instead.  Golden planes were produced by the UNMODIFIED reference's own
world_to_grid / _bresenham / in_bounds (oracle/make_golden_counts.py).  Integer planes must be
bit-exact; float32 log-odds equal to the float64 evaluation rounded once to float32."""
import os

import numpy as np
import pytest

from conftest import GOLD, load_packet_stream, session_packets
from oracle import occgrid_oracle as O


def _golden():
    return np.load(os.path.join(GOLD, 'session_counts.npz'))


@pytest.mark.parametrize('slam', [False, True])
def test_oracle_counts_equal_reference_enumeration(slam):
    pk, _ = session_packets(True)
    g = O.OracleCountGrid()
    O.replay(pk, grid=g, separation=0.0, slam=O.OracleSLAM() if slam else None)
    z = _golden()
    tag = 'slam_on' if slam else 'slam_off'
    assert np.array_equal(g.hit, z[f'hit_{tag}']) and np.array_equal(g.miss, z[f'miss_{tag}'])
    # cells that were ever touched are exactly the known cells of the last-writer-wins grid
    ref = O.OracleGrid()
    O.replay(pk, grid=ref, separation=0.0, slam=O.OracleSLAM() if slam else None)
    assert np.array_equal((g.hit + g.miss) > 0, ref.grid != -1)


torch = pytest.importorskip('torch')


@pytest.fixture(scope='module')
def M():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper
    return dual_bot_mapper


def _grid(M, strategy, **kw):
    try:
        return M.OccupancyGrid(strategy=strategy, **kw)
    except M.OccGridError as e:
        pytest.skip(f'{strategy}: {e}')


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', ['global_atomic', 'tiled'])
@pytest.mark.parametrize('slam', [False, True])
def test_gpu_counts_golden_session(M, strategy, slam):
    pk, _ = session_packets(True)
    z = _golden()
    tag = 'slam_on' if slam else 'slam_off'
    g = _grid(M, strategy)
    drift = M.slam_drift_table(pk, separation=0.0)[0] if slam else None
    g.accumulate_packets(pk, separation=0.0, drift=drift)
    assert g.hit_counts.dtype == np.int32 and g.hit_counts.shape == (200, 200)
    assert np.array_equal(g.hit_counts, z[f'hit_{tag}']) and np.array_equal(g.miss_counts, z[f'miss_{tag}'])
    assert (g.grid == -1).all()                                   # the int8 grid is a different product
    # log-odds from the integer planes: the float64 evaluation rounded to float32
    want = np.clip(z[f'hit_{tag}'].astype(np.float64) * 0.85 + z[f'miss_{tag}'].astype(np.float64) * -0.4, -2.0, 3.5)
    got = g.log_odds()
    assert got.dtype == np.float32 and np.array_equal(got, want.astype(np.float32))
    # counts accumulate: the same session again doubles every cell
    g.accumulate_packets(pk, separation=0.0, drift=drift)
    assert np.array_equal(g.hit_counts, 2 * z[f'hit_{tag}']) and np.array_equal(g.miss_counts, 2 * z[f'miss_{tag}'])
    g.reset_counts()
    assert not g.hit_counts.any() and not g.miss_counts.any()


@pytest.mark.gpu
@pytest.mark.parametrize('strategy', ['global_atomic', 'tiled'])
@pytest.mark.parametrize('name', ['mixed_a', 'mixed_b_sep', 'mixed_c_4096', 'mixed_d_edge'])
def test_gpu_counts_adversarial_streams(M, golden, strategy, name):
    """Bad magic, foreign agents, v1/junk sizes, NaN/inf ranges, out-of-grid rays, cell-boundary
    yaws: count planes vs the oracle replay of the same datagrams."""
    want = golden['packet_streams'][name]
    pk, ref_drift = load_packet_stream(name)
    kw = want['grid_kwargs']
    og = O.OracleCountGrid(**kw)
    O.replay(pk, grid=og, separation=want['separation'], slam=O.OracleSLAM() if want['slam'] else None)
    g = _grid(M, strategy, **kw)
    g.accumulate_packets(pk, separation=want['separation'], drift=ref_drift if want['slam'] else None)
    assert np.array_equal(g.hit_counts, og.hit) and np.array_equal(g.miss_counts, og.miss)
    assert np.array_equal(g.log_odds(0.9, -0.35, -4.0, 4.0), og.log_odds(0.9, -0.35, -4.0, 4.0))


@pytest.mark.gpu
def test_gpu_counts_full_size_properties(M):
    """BASELINE configs[1] scale (4096^2, 64 agents): both strategies give identical planes, the
    planes sum to the counters' beam-cell updates minus the untouched end cells, and the touched
    set equals the known cells of the last-writer-wins grid built from the same batch."""
    from occgrid_b200 import simulation_tools as st
    sess = st.generate_session(n_agents=64, n_packets=400_000, grid_size=4096, seed=5)
    kw = sess['grid']
    planes = []
    for strategy in ('tiled', 'global_atomic'):
        g = _grid(M, strategy, **kw)
        g.accumulate_packets(sess['packets'], agent_offsets=sess['agent_offsets'], agent_idx=sess['agent_idx'])
        planes.append((g.hit_counts, g.miss_counts, g.counters()))
    (h0, m0, c0), (h1, m1, c1) = planes
    assert np.array_equal(h0, h1) and np.array_equal(m0, m1)
    assert int(h0.sum()) == c0['hits']                                   # every valid hit lands in this grid
    assert int(m0.sum()) + c0['beams'] == c0['updates']                  # each beam's end cell is not a miss
    ref = _grid(M, 'tiled', **kw)
    ref.update_packets(sess['packets'], agent_offsets=sess['agent_offsets'], agent_idx=sess['agent_idx'])
    assert np.array_equal((h0 + m0) > 0, ref.grid != -1)
