"""The streamed TILED bin pass (k_home_bin): persistent CTAs that each take several 2048-packet
segments, with a ring of bulk copies running across segment boundaries.  The cases below reach
what smaller batches do not: a CTA's second and third segment, a last sub-batch whose byte count
is not a multiple of 16, record strides other than 42, a buffer that is not 16-byte aligned (no
bulk copies) and an agent-offset table too large for shared memory.  Each compares the int8 grid
and the counters bit for bit against the C oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

ORIGIN, RES, SIZE = -102.4, 0.05, 4096
N_BIG = 1_000_037           # > 148 SMs x 3 CTAs x 2048 packets: some CTAs bin more than one segment; 37 x 42 B % 16 != 0


@pytest.fixture(scope='module')
def M():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper
    return dual_bot_mapper


@pytest.fixture(scope='module')
def sess():
    from occgrid_b200 import simulation_tools as st
    return st.generate_session(n_agents=64, n_packets=N_BIG, seed=33)


def check(M, dev_packets, host_packets, agent_offsets, agent_idx=None):
    """dev_packets: uint8 cuda tensor [n, stride] handed to the library as is."""
    from oracle import c_oracle
    want = np.full((SIZE, SIZE), -1, np.int8)
    c = c_oracle.integrate_packets(host_packets, want, ORIGIN, ORIGIN, RES, agent_offsets=agent_offsets, agent_idx=agent_idx)
    g = M.OccupancyGrid(size=SIZE, resolution=RES, origin_x=ORIGIN, origin_y=ORIGIN, strategy='tiled',
                        max_batch=dev_packets.shape[0])
    g.update_packets(dev_packets, agent_offsets=agent_offsets, agent_idx=agent_idx)
    assert np.array_equal(g.grid, want)
    k = g.counters()
    for name in ('packets', 'accepted', 'dropped', 'bad_pose', 'beams', 'hits', 'updates'):
        assert k[name] == c[name], name
    return c


def test_several_segments_per_cta(M, sess):
    pk = sess['packets']
    c = check(M, torch.from_numpy(pk).cuda(), pk, sess['agent_offsets'])
    assert c['packets'] == N_BIG and c['accepted'] > N_BIG // 2


def test_stride_64(M, sess):
    """Wider record slots: fewer CTAs fit an SM, so each bins more segments."""
    pk = sess['packets']
    wide = torch.zeros((pk.shape[0], 64), dtype=torch.uint8)
    wide[:, :42] = torch.from_numpy(pk)
    wide[:, 42:] = 0xA5                            # padding the decode must not read
    check(M, wide.cuda(), wide.numpy(), sess['agent_offsets'])


@pytest.mark.parametrize('shift', [1, 8])
def test_unaligned_buffer(M, sess, shift):
    """A record buffer that starts off a 16-byte boundary is staged without bulk copies."""
    pk = sess['packets']
    n = pk.shape[0]
    flat = torch.empty(n * 42 + shift, dtype=torch.uint8, device='cuda')
    dev = flat[shift:].view(n, 42)
    dev.copy_(torch.from_numpy(pk))
    assert dev.data_ptr() % 16 == shift
    check(M, dev, pk, sess['agent_offsets'])


def test_agent_table_beyond_shared_memory():
    """300 agents (ids from agent_idx): the offset table is read from global memory."""
    from occgrid_b200 import dual_bot_mapper as M
    from occgrid_b200 import simulation_tools as st
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    s = st.generate_session(n_agents=300, n_packets=300_011, seed=9)
    c = check(M, torch.from_numpy(s['packets']).cuda(), s['packets'], s['agent_offsets'], agent_idx=s['agent_idx'])
    assert c['accepted'] > 300_011 // 2
