"""The streamed TILED bin pass (k_home_bin): persistent CTAs that each take several 2048-packet
segments, with a ring of bulk copies running across segment boundaries.  The cases below reach
what smaller batches do not: a CTA's second and third segment, batches one packet either side of
one segment per resident CTA (no segment claimed from bin_counter, or exactly one), a last
sub-batch whose byte count is not a multiple of 16 at every tail length, record strides other
than 42, a buffer that is not 16-byte aligned (no bulk copies) and the switch of the agent-offset
table from shared to global memory at 256 agents.  In every batch the last record is accepted and
all four of its beams hit cells no other record writes, so a last record staged wrongly changes
the grid.  Each compares the int8 grid (or the agent-map stack) and the counters bit for bit
against the C oracle."""
import numpy as np
import pytest

from agent_maps_util import integrate_packets_agent_maps

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

ORIGIN, RES, SIZE = -102.4, 0.05, 4096
N_BIG = 1_000_037           # > 148 SMs x 3 CTAs x 2048 packets: some CTAs bin more than one segment; 37 x 42 B % 16 != 0
SHORT = 3001                # one segment, a short last sub-batch


@pytest.fixture(scope='module')
def M():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper
    return dual_bot_mapper


@pytest.fixture(scope='module')
def resident(M):
    """Bin CTAs resident at once for 42-byte records: three per SM (__launch_bounds__(kTT, 3), and
    3 x 73 KB of shared memory fit an SM, DESIGN §3)."""
    return torch.cuda.get_device_properties(0).multi_processor_count * 3


@pytest.fixture(scope='module')
def sess(resident):
    from occgrid_b200 import simulation_tools as st
    return st.generate_session(n_agents=64, n_packets=max(N_BIG, 2048 * (resident + 1) + 1), seed=33)


def last_record_counts(pk, agent_offsets, agent_idx=None, rec_len=42, origin=ORIGIN):
    """Copies of pk [n, stride] (and agent_idx) whose last record is agent 1's, accepted, with four
    hits, placed 1.6 m inside the map's (origin, origin) corner, where no other record's beams go."""
    from occgrid_b200 import simulation_tools as st
    rec = np.zeros(1, st.PACKET_DTYPE)
    rec['magic'], rec['agent'], rec['yaw'] = b'QSRL', 1, 0.3
    rec['x'] = origin + 1.6 - agent_offsets[1, 0]
    rec['y'] = origin + 1.6 - agent_offsets[1, 1]
    rec['front'], rec['left'], rec['back'], rec['right'] = 0.61, 0.83, 0.47, 0.97     # all in (0.05, 1.2]: hits
    pk = pk.copy()
    pk[-1, :rec_len] = rec.view(np.uint8)[:rec_len]
    if agent_idx is not None:
        agent_idx = agent_idx.copy()
        agent_idx[-1] = 1
    return pk, agent_idx


def check(M, dev_packets, host_packets, agent_offsets, agent_idx=None, rec_len=42, maps=False, size=SIZE, origin=ORIGIN):
    """dev_packets: uint8 cuda tensor [n, stride] handed to the library as is."""
    from oracle import c_oracle
    n = dev_packets.shape[0]
    kw = dict(size=size, resolution=RES, origin_x=origin, origin_y=origin, strategy='tiled', max_batch=n)
    if maps:
        n_agents = agent_offsets.shape[0] - 1
        want = np.full((n_agents, size, size), -1, np.int8)
        c = integrate_packets_agent_maps(host_packets, want, origin, origin, RES, rec_len=rec_len,
                                         agent_offsets=agent_offsets, agent_idx=agent_idx)
        g = M.AgentGrids(n_agents=n_agents, **kw)
    else:
        want = np.full((size, size), -1, np.int8)
        c = c_oracle.integrate_packets(host_packets, want, origin, origin, RES, rec_len=rec_len,
                                       agent_offsets=agent_offsets, agent_idx=agent_idx)
        g = M.OccupancyGrid(**kw)
    g.update_packets(dev_packets, agent_offsets=agent_offsets, agent_idx=agent_idx, rec_len=rec_len)
    assert np.array_equal(g.grids if maps else g.grid, want)
    k = g.counters()
    for name in ('packets', 'accepted', 'dropped', 'bad_pose', 'beams', 'hits', 'updates'):
        assert k[name] == c[name], name
    return c


def test_several_segments_per_cta(M, sess):
    pk, _ = last_record_counts(sess['packets'][:N_BIG], sess['agent_offsets'])
    c = check(M, torch.from_numpy(pk).cuda(), pk, sess['agent_offsets'])
    assert c['packets'] == N_BIG and c['accepted'] > N_BIG // 2


@pytest.mark.parametrize('dm,dr', [pytest.param(dm, dr, id=f'2048x(resident{dm:+d}){dr:+d}')
                                   for dm in (-1, 0, 1) for dr in (-1, 0, 1)])
def test_one_segment_per_resident_cta(M, sess, resident, dm, dr):
    """2048 * m + r packets for m = resident CTAs - 1 .. resident + 1: every CTA takes one segment
    and claims none (m <= resident - 1, or m = resident with r <= 0), or the last segments are
    claimed by CTAs done with their first."""
    n = 2048 * (resident + dm) + dr
    pk, _ = last_record_counts(sess['packets'][:n], sess['agent_offsets'])
    c = check(M, torch.from_numpy(pk).cuda(), pk, sess['agent_offsets'])
    assert c['packets'] == n and c['accepted'] > n // 2


def test_stride_64(M, sess):
    """Wider record slots: fewer CTAs fit an SM, so each bins more segments."""
    pk, _ = last_record_counts(sess['packets'][:N_BIG], sess['agent_offsets'])
    wide = torch.zeros((pk.shape[0], 64), dtype=torch.uint8)
    wide[:, :42] = torch.from_numpy(pk)
    wide[:, 42:] = 0xA5                            # padding the decode must not read
    check(M, wide.cuda(), wide.numpy(), sess['agent_offsets'])


@pytest.mark.parametrize('tail', range(1, 17))
def test_v1_records_last_sub_batch(M, sess, tail):
    """41-byte (v1) records at stride 41, the last sub-batch `tail` records long: 41 * tail % 16
    bytes (every value 0..15) lie past the last whole 16 bytes the bulk copy brings and are loaded
    by hand; they end with the last record's right range."""
    n = 256 * 1171 + tail
    pk, _ = last_record_counts(np.ascontiguousarray(sess['packets'][:n, :41]), sess['agent_offsets'], rec_len=41)
    check(M, torch.from_numpy(pk).cuda(), pk, sess['agent_offsets'], rec_len=41)


@pytest.mark.parametrize('shift,n', [pytest.param(1, N_BIG, id='1'), pytest.param(8, N_BIG, id='8')] +
                         [pytest.param(s, SHORT, id=f'short-{s}') for s in range(1, 16)])
def test_unaligned_buffer(M, sess, shift, n):
    """A record buffer that starts off a 16-byte boundary is staged without bulk copies."""
    pk, _ = last_record_counts(sess['packets'][:n], sess['agent_offsets'])
    flat = torch.empty(n * 42 + shift, dtype=torch.uint8, device='cuda')
    dev = flat[shift:].view(n, 42)
    dev.copy_(torch.from_numpy(pk))
    assert dev.data_ptr() % 16 == shift
    check(M, dev, pk, sess['agent_offsets'])


def test_agent_table_beyond_shared_memory(M):
    """300 agents (ids from agent_idx): the offset table is read from global memory."""
    from occgrid_b200 import simulation_tools as st
    s = st.generate_session(n_agents=300, n_packets=300_011, seed=9)
    pk, agent_idx = last_record_counts(s['packets'], s['agent_offsets'], s['agent_idx'])
    c = check(M, torch.from_numpy(pk).cuda(), pk, s['agent_offsets'], agent_idx=agent_idx)
    assert c['accepted'] > 300_011 // 2


@pytest.mark.parametrize('maps', [False, True], ids=['grid', 'agent_maps'])
@pytest.mark.parametrize('ids', ['wire', 'agent_idx'])
@pytest.mark.parametrize('n_agents', [254, 255, 256, 257])
def test_agent_table_switch(M, n_agents, ids, maps):
    """Up to 255 agents the offset table is staged in shared memory, from 256 on it is read from
    global memory.  Every agent maps in its own frame (the room's coordinates, 256^2 maps) shifted
    by its own random offset, so a row read from the wrong place moves the beams; in one grid the
    agents overlap and overwrite each other's cells.  The highest id and a foreign one (n_agents + 1,
    or 0 where the wire byte cannot say n_agents + 1) are in the batch."""
    from occgrid_b200 import simulation_tools as st
    size, origin = 256, -6.4
    s = st.generate_session(n_agents=n_agents + 1 + (n_agents + 1) % 2, n_packets=300_011, seed=n_agents)
    highest, foreign = n_agents, n_agents + 1
    agent = np.minimum(s['agent_idx'], foreign)                   # the generated agents above n_agents: foreign
    pk = s['packets']
    if ids == 'wire':
        highest, foreign = min(n_agents, 255), (foreign if foreign <= 255 else 0)
        agent = np.where(agent > n_agents, foreign, np.minimum(agent, 255))
        pk = pk.copy()
        pk[:, 4] = agent
        agent_idx = None
    else:
        agent_idx = agent.astype(np.int32)
    assert (agent == highest).any() and (agent == foreign).any()
    off = np.random.default_rng(n_agents).uniform(-0.5, 0.5, (n_agents + 1, 2))
    pk, agent_idx = last_record_counts(pk, off, agent_idx, origin=origin)
    c = check(M, torch.from_numpy(pk).cuda(), pk, off, agent_idx=agent_idx, maps=maps, size=size, origin=origin)
    assert 0 < c['dropped'] < 300_011 // 50 and c['accepted'] > 300_011 // 2
