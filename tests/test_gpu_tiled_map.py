"""Multi-GPU integration path emulated on ONE GPU (SURVEY §4 'Multi-GPU without a cluster'):
N logical ranks each route their share with the CUDA routing kernel, the all-to-all is done by
concatenating segments in source-rank order, every band integrates what it receives, and the
assembled map must equal the untiled oracle result bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip('torch')


@pytest.mark.parametrize('world', [2, 4])
@pytest.mark.parametrize('strategy', ['global_atomic', 'tiled'])
def test_emulated_ranks_equal_single_grid(world, strategy):
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import simulation_tools as st
    from occgrid_b200.distributed import BandLayout, CudaBandOps
    from occgrid_b200.dual_bot_mapper import OccGridError
    from oracle import c_oracle
    size, origin = 1024, (-25.6, -25.6)
    sess = st.generate_session(n_agents=16, n_packets=60_000, grid_size=size, origin=origin, seed=9)
    n = sess['packets'].shape[0]
    offs = sess['agent_offsets'].copy()
    # park two rooms right on band boundaries so that packets go to two bands
    offs[1:3] = (-2.0, origin[1] + size * 0.05 / world - 1.0)
    offs[3:5] = (3.0, origin[1] + size * 0.05 / 2 + 0.2)
    drift = np.random.default_rng(1).normal(0, 0.02, (n, 2))
    layout = BandLayout(size, world)
    try:
        ops = [CudaBandOps(layout, r, size, 0.05, origin[0], origin[1], 'cuda', strategy, n) for r in range(world)]
    except OccGridError as e:
        pytest.skip(str(e))
    tab = torch.from_numpy(offs).cuda()
    routed = []
    for r in range(world):
        sl = slice(r * n // world, (r + 1) * n // world)
        pk = ops[r].stage(sess['packets'][sl])
        idx = torch.from_numpy(sess['agent_idx'][sl].copy()).cuda()
        dr = torch.from_numpy(drift[sl].copy()).cuda()
        send, counts = ops[r].route(pk, idx, dr, tab)
        offs_c = np.concatenate([[0], np.cumsum(counts)])
        routed.append([send[offs_c[b]:offs_c[b + 1]].clone() for b in range(world)])
    total_rows = 0
    bands = []
    for b in range(world):
        recv = torch.cat([routed[r][b] for r in range(world)])
        total_rows += recv.shape[0]
        ops[b].integrate(recv)
        bands.append(ops[b].band_tensor().cpu().numpy())
    got = np.concatenate(bands, axis=0)
    want = np.full((size, size), -1, np.int8)
    c = c_oracle.integrate_packets(sess['packets'], want, origin[0], origin[1], 0.05, agent_offsets=offs,
                                   agent_idx=sess['agent_idx'], drift=drift)
    assert np.array_equal(got, want)
    assert n < total_rows < 1.5 * n                      # boundary rooms are duplicated, the rest is not
    owned = sum(ops[b].grid.counters()['owned_updates'] for b in range(world))
    assert owned == c['updates']                         # every beam counted exactly once across bands


def test_fused_swarm_map_single_rank():
    """exchange='p2p' with world = 1: the fused band step end to end (route batch i+1 inside the
    persistent raycast kernel of batch i, per-source segments, device-side fill counts, publish):
    same map as the oracle after flush()."""
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import simulation_tools as st
    from occgrid_b200.distributed import TiledSwarmMap
    from oracle import c_oracle
    size, origin = 1024, (-25.6, -25.6)
    sess = st.generate_session(n_agents=16, n_packets=90_000, grid_size=size, origin=origin, seed=21)
    tmap = TiledSwarmMap(size, 0.05, origin[0], origin[1], max_batch=30_000, exchange='p2p')
    assert tmap.exchange == 'p2p' and tmap.band is not None
    drift = np.random.default_rng(2).normal(0, 0.02, (90_000, 2))
    for i in range(3):
        sl = slice(i * 30_000, (i + 1) * 30_000)
        tmap.update_packets(sess['packets'][sl], agent_offsets=sess['agent_offsets'], agent_idx=sess['agent_idx'][sl],
                            drift=drift[sl])
    got = tmap.gather_grid()            # flushes
    want = np.full((size, size), -1, np.int8)
    c = c_oracle.integrate_packets(sess['packets'], want, origin[0], origin[1], 0.05, agent_offsets=sess['agent_offsets'],
                                   agent_idx=sess['agent_idx'], drift=drift)
    assert np.array_equal(got, want)
    cn = tmap.counters()
    assert cn['owned_updates'] == c['updates'] and cn['packets'] == 90_000 and cn['beams'] == c['beams']
    # a second stream after a flush continues on the same map (later batches still win)
    tmap.update_packets(sess['packets'][:30_000], agent_offsets=sess['agent_offsets'], agent_idx=sess['agent_idx'][:30_000])
    c_oracle.integrate_packets(sess['packets'][:30_000], want, origin[0], origin[1], 0.05, agent_offsets=sess['agent_offsets'],
                               agent_idx=sess['agent_idx'][:30_000])
    assert np.array_equal(tmap.gather_grid(), want)
    with pytest.raises(Exception):
        tmap.update_packets(sess['packets'][:40_000], agent_offsets=sess['agent_offsets'], agent_idx=sess['agent_idx'][:40_000])


def test_fused_swarm_map_full_size_config2():
    """BASELINE config 2 at full size through the fused band step (world = 1): 2.5e6 packets in 5
    batches of 5e5 into 4096^2, equal to the C oracle, and the update count matches."""
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import simulation_tools as st
    from occgrid_b200.distributed import TiledSwarmMap
    from oracle import c_oracle
    size, origin, n, b = 4096, (-102.4, -102.4), 2_500_000, 500_000
    sess = st.generate_session(n_agents=64, n_packets=n, grid_size=size, origin=origin, seed=42)
    tmap = TiledSwarmMap(size, 0.05, origin[0], origin[1], max_batch=b, exchange='p2p')
    for i in range(n // b):
        sl = slice(i * b, (i + 1) * b)
        tmap.update_packets(sess['packets'][sl], agent_offsets=sess['agent_offsets'], agent_idx=sess['agent_idx'][sl])
    got = tmap.gather_grid()
    want = np.full((size, size), -1, np.int8)
    c = c_oracle.integrate_packets(sess['packets'], want, origin[0], origin[1], 0.05, agent_offsets=sess['agent_offsets'],
                                   agent_idx=sess['agent_idx'])
    assert np.array_equal(got, want)
    cn = tmap.counters()
    assert cn['owned_updates'] == c['updates'] and cn['beams'] == c['beams'] == 4 * n


def test_routed_poses_full_size_config2_tiled():
    """update_poses under TILED on the whole BASELINE config 2 batch (2.5e6 packets into 4096^2),
    routed to one band: the pose-record count and scatter passes walk 1 221 chunks of 2 048 records,
    more than their 8 CTAs per SM take in one pass, and the map equals the C oracle."""
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import simulation_tools as st
    from occgrid_b200.distributed import BandLayout, CudaBandOps
    from oracle import c_oracle
    size, origin, n = 4096, (-102.4, -102.4), 2_500_000
    sess = st.generate_session(n_agents=64, n_packets=n, grid_size=size, origin=origin, seed=42)
    ops = CudaBandOps(BandLayout(size, 1), 0, size, 0.05, origin[0], origin[1], 'cuda', 'tiled', n)
    pk = ops.stage(sess['packets'])
    idx = torch.from_numpy(sess['agent_idx'].copy()).cuda()
    send, counts = ops.route(pk, idx, None, torch.from_numpy(sess['agent_offsets']).cuda())
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert 8 * sms * 2048 < counts[0] <= n                # some persistent CTAs take a second chunk
    ops.integrate(send)
    got = ops.band_tensor().cpu().numpy()
    want = np.full((size, size), -1, np.int8)
    c = c_oracle.integrate_packets(sess['packets'], want, origin[0], origin[1], 0.05, agent_offsets=sess['agent_offsets'],
                                   agent_idx=sess['agent_idx'])
    assert np.array_equal(got, want)
    assert ops.grid.counters()['owned_updates'] == c['updates']


def _emulated_band_steps(world, size, origin, max_batch):
    """`world` logical ranks on ONE GPU: plain receive buffers linked by pointer (peer-mapped over
    NVLink in production), publish without the wait (the steps are issued one rank after another on
    one stream, so a spinning barrier would never be released)."""
    from occgrid_b200.distributed import BandBuffers, BandLayout, BandStep
    layout = BandLayout(size, world)
    steps = [BandStep(layout, r, size, 0.05, origin[0], origin[1], 'cuda', max_batch) for r in range(world)]
    BandBuffers.link([s.buf for s in steps])
    for s in steps:
        s.finish_init()
    return steps


@pytest.mark.parametrize('world', [2, 4])
def test_fused_band_step_emulated_ranks(world):
    """The fused raycast + route kernel on one GPU: every logical rank stores its records straight
    into the band owners' per-source segments in arbitrary arrival order; owners bin what arrived
    using the tile ids and ordinals carried by the records.  Three batches (so both receive slots
    are reused); assembled map == untiled oracle over the canonical stream."""
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import simulation_tools as st
    from oracle import c_oracle
    size, origin = 1024, (-25.6, -25.6)
    n_batches, per_rank = 3, 20_000
    sess = st.generate_session(n_agents=16, n_packets=n_batches * per_rank * world, grid_size=size, origin=origin, seed=9)
    n = sess['packets'].shape[0]
    offs = sess['agent_offsets'].copy()
    offs[1:3] = (-2.0, origin[1] + size * 0.05 / world - 1.0)     # rooms right on band boundaries: records go to two bands
    offs[3:5] = (3.0, origin[1] + size * 0.05 / 2 + 0.2)
    drift = np.random.default_rng(1).normal(0, 0.02, (n, 2))
    steps = _emulated_band_steps(world, size, origin, per_rank)
    tab = torch.from_numpy(offs).cuda()
    order = []
    for b in range(n_batches):
        base = b * per_rank * world
        for r in reversed(range(world)):                          # issue order must not matter
            sl = slice(base + r * per_rank, base + (r + 1) * per_rank)
            steps[r].step(torch.from_numpy(sess['packets'][sl]).cuda(), torch.from_numpy(sess['agent_idx'][sl].copy()).cuda(),
                          torch.from_numpy(drift[sl].copy()).cuda(), tab, wait=False)
        order.append(np.arange(base, base + per_rank * world))
    for s in steps:
        s.step(None, None, None, None)
        s.check_status()
    got = np.concatenate([s.grid.grid for s in steps], axis=0)
    o = np.concatenate(order)
    want = np.full((size, size), -1, np.int8)
    c = c_oracle.integrate_packets(sess['packets'][o], want, origin[0], origin[1], 0.05, agent_offsets=offs,
                                   agent_idx=sess['agent_idx'][o], drift=drift[o])
    assert np.array_equal(got, want)
    cn = [s.grid.counters() for s in steps]
    assert sum(x['owned_updates'] for x in cn) == c['updates']      # every beam counted exactly once across bands
    assert sum(x['packets'] for x in cn) == n and sum(x['beams'] for x in cn) == c['beams']
    assert n < sum(x['records'] for x in cn) < 1.5 * n              # boundary rooms are duplicated, the rest is not


def test_fused_band_step_reports_segment_overflow():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import simulation_tools as st
    from occgrid_b200.distributed import OccGridError
    size, origin = 512, (-12.8, -12.8)
    sess = st.generate_session(n_agents=4, n_packets=6000, grid_size=size, origin=origin, seed=4)
    steps = _emulated_band_steps(2, size, origin, 2048)
    tab = torch.from_numpy(sess['agent_offsets']).cuda()
    s = steps[0]
    s.seg_cap_saved = s.seg_cap
    pk = torch.from_numpy(sess['packets'][:2048]).cuda()
    idx = torch.from_numpy(sess['agent_idx'][:2048].copy()).cuda()
    s.step(pk, idx, None, tab, wait=False)
    s.step(pk, idx, None, tab, wait=False)          # fine: the reservation counters were reset by publish
    s.check_status()
    s._resv[:2].fill_(2040)                         # pretend the segments are nearly full
    s.step(pk, idx, None, tab, wait=False)
    with pytest.raises(OccGridError, match='overflow'):
        s.check_status()


@pytest.mark.parametrize('name', ['mixed_a', 'mixed_b_sep', 'mixed_c_4096', 'mixed_d_edge'])
def test_fused_band_step_on_adversarial_streams(name):
    """The router of the fused band step has its own decode (aligned word loads + funnel shifts from
    shared memory) and screened robot-cell evaluation: the reference-generated adversarial streams
    (bad magic, foreign agents, NaN/inf/sentinel ranges, SLAM drift, poses on cell boundaries) must
    give the reference's grid through it, on one band and split over two."""
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    import hashlib
    import json
    import os
    from conftest import GOLD, load_packet_stream, normalise_datagrams
    from occgrid_b200.distributed import BandBuffers, BandLayout, BandStep
    want = json.load(open(os.path.join(GOLD, 'golden.json')))['packet_streams'][name]
    pk, ref_drift = load_packet_stream(name)
    arr, drift = normalise_datagrams(pk, ref_drift if want['slam'] else None)
    kw = want['grid_kwargs']
    size, res = kw.get('size', 200), kw.get('resolution', 0.05)
    ox, oy = kw.get('origin_x', -5.0), kw.get('origin_y', -5.0)
    tab = torch.tensor([[0.0, 0.0], [0.0, 0.0], [float(want['separation']), 0.0]], dtype=torch.float64, device='cuda')
    import math
    for world in (1, 2):
        if world > 1 and size // world < 2 * (math.ceil(1.2 / res) + 2) + 1:
            continue                                             # bands thinner than two reaches are rejected by the library
        layout = BandLayout(size, world)
        steps = [BandStep(layout, r, size, res, ox, oy, 'cuda', arr.shape[0]) for r in range(world)]
        BandBuffers.link([s.buf for s in steps])
        for s in steps:
            s.finish_init()
        n = arr.shape[0]
        for r in range(world):                                   # rank r ingests the r-th part of the stream, in order
            sl = slice(r * n // world, (r + 1) * n // world)
            steps[r].step(torch.from_numpy(arr[sl].copy()).cuda(), None,
                          torch.from_numpy(drift[sl].copy()).cuda() if drift is not None else None, tab, wait=False)
        for s in steps:
            s.step(None, None, None, None)
            s.check_status()
        got = np.concatenate([s.grid.grid for s in steps], axis=0)
        assert hashlib.sha1(got.tobytes()).hexdigest() == want['sha1'], (name, world)
