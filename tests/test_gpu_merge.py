"""GPU parity of the map-fusion path (mapmerge_* kernels through the reference-shaped
MapMerger) against oracle/merge_oracle.py.  fp64 coordinates are compared BIT-EXACTLY (both
sides perform the same individually rounded fp64 operations in the same order); the published
int8 grids and origins must be identical."""
import math

import numpy as np
import pytest

from merge_util import load_merge_ref, synth_agent_grid

pytestmark = pytest.mark.gpu
torch = pytest.importorskip('torch')


@pytest.fixture(scope='module')
def MM():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import map_merger
    return map_merger


def run_pair(MM, n, n_agents, seed, res=0.05, origin=(-5.0, -5.0), span=4.0, check_every=True):
    from oracle import merge_oracle as MO
    r = np.random.default_rng(seed)
    m, o = MM.MapMerger(agent_ids=list(range(1, n_agents + 1))), MO.OracleMerger()
    got = want = None
    for a in range(n_agents):
        g = synth_agent_grid(n, seed * 100 + a)
        T = MO.se2_matrix(*r.uniform(-span, span, 2), r.uniform(-math.pi, math.pi))
        got = m.map_callback(MM.make_grid_msg(g.ravel(), n, n, res, *origin), a + 1, transform=T)
        want = o.map_callback(g.ravel(), n, n, res, origin[0], origin[1], T)
        if check_every or a == n_agents - 1:
            assert got is not None and want is not None
            assert (got.info.width, got.info.height) == (want[0].shape[1], want[0].shape[0])
            assert (got.info.origin.position.x, got.info.origin.position.y) == want[1]
            assert np.array_equal(got.data, want[0]), f'agent {a}'
            pc = m.global_pcd
            assert pc.shape[0] == o.gx.shape[0]
            assert np.array_equal(pc[:, 0], o.gx) and np.array_equal(pc[:, 1], o.gy)
    return m, o, got, want


def test_sequential_callbacks_match_oracle(MM):
    m, o, got, _ = run_pair(MM, 256, 6, seed=1)
    assert got.header.frame_id == 'map_global'
    assert got.data.dtype == np.int8 and set(np.unique(got.data)) == {-1, 100}
    assert m.map_resolution == 0.05 and m.map_origin == [-5.0, -5.0]


def test_other_resolution_and_offsets(MM):
    run_pair(MM, 300, 4, seed=2, res=0.1, origin=(12.3, -40.7), span=9.0)


def test_first_callback_empty_and_rejected(MM):
    from oracle import merge_oracle as MO
    m = MM.MapMerger()
    empty = np.full((32, 32), -1, np.int8)
    assert m.map_callback(MM.make_grid_msg(empty.ravel(), 32, 32, 0.05, 0, 0), 1) is None
    g = synth_agent_grid(96, 5)
    first = m.map_callback(MM.make_grid_msg(g.ravel(), 96, 96, 0.05, -2.4, -2.4), 1)
    o = MO.OracleMerger()
    want = o.map_callback(g.ravel(), 96, 96, 0.05, -2.4, -2.4)
    assert np.array_equal(first.data, want[0])          # adopted as is: no voxel filter (:40-43)
    n = m.global_pcd.shape[0]
    assert m.map_callback(MM.make_grid_msg(g.ravel(), 96, 96, 0.05, -2.4, -2.4), 2,
                          transform=(1.0, 0.5, 0.2), fitness=0.59) is None       # :54-56
    assert m.global_pcd.shape[0] == n
    assert m.map_callback(MM.make_grid_msg(empty.ravel(), 32, 32, 0.05, 0, 0), 2) is None
    pts = m.grid_to_pcd(MM.make_grid_msg(g.ravel(), 96, 96, 0.05, -2.4, -2.4))
    ox, oy = MO.grid_to_points(g.ravel(), 96, 96, 0.05, -2.4, -2.4)
    assert np.array_equal(pts[:, 0], ox) and np.array_equal(pts[:, 1], oy) and not pts[:, 2].any()


def test_identity_transform_property(MM):
    """Merging a grid with itself under the identity transform leaves the occupied set
    unchanged (every voxel averages two identical points)."""
    g = synth_agent_grid(128, 9)
    m = MM.MapMerger()
    a = m.map_callback(MM.make_grid_msg(g.ravel(), 128, 128, 0.5, -32.0, -32.0), 1)
    b = m.map_callback(MM.make_grid_msg(g.ravel(), 128, 128, 0.5, -32.0, -32.0), 2, transform=np.eye(4))
    assert np.array_equal(a.data, b.data)
    ys, xs = np.nonzero(g > 50)
    want = np.full_like(a.data, -1)
    want[ys - ys.min(), xs - xs.min()] = 100
    assert np.array_equal(a.data, want)


def test_batched_merge_equals_callbacks(MM):
    from oracle import merge_oracle as MO
    r = np.random.default_rng(4)
    grids = np.stack([synth_agent_grid(200, 40 + a) for a in range(5)])
    origins = np.tile(np.array([[-5.0, -5.0]]), (5, 1))
    tf = np.stack([MO.se2_matrix(*r.uniform(-3, 3, 2), r.uniform(-math.pi, math.pi)) for _ in range(5)])
    o = MO.OracleMerger()
    for a in range(5):
        want = o.map_callback(grids[a].ravel(), 200, 200, 0.05, -5.0, -5.0, tf[a])
    out, origin = MM.MapMerger().merge(grids, origins, 0.05, tf)
    assert np.array_equal(out, want[0]) and origin == want[1]
    out2, origin2 = MM.MapMerger().merge(torch.from_numpy(grids).cuda(), origins, 0.05, tf)
    assert np.array_equal(out2, want[0]) and origin2 == want[1]


def _oracle_chain(grids, n, res, origin, tf):
    from oracle import merge_oracle as MO
    o = MO.OracleMerger()
    want = None
    for a in range(len(grids)):
        out = o.map_callback(grids[a].ravel(), n, n, res, origin[0], origin[1], tf[a])
        want = out if out is not None else want
    return o, want


@pytest.mark.parametrize('span,rot,seed', [(3.0, math.pi, 21), (0.4, 0.05, 22), (0.0, 0.0, 23)])
def test_incremental_chain_is_bit_exact(MM, span, rot, seed):
    """merge() fuses equal-shaped grids with the incremental chain: while the voxel lattice stands
    still only the voxels a slice touches are re-averaged.  The cloud (coordinates AND order) and
    the published grid must equal the oracle's full filter per callback; heavy overlap (small
    span / rotation, or identical poses) makes most slice points land in occupied voxels."""
    from oracle import merge_oracle as MO
    r = np.random.default_rng(seed)
    A, n = 24, 160
    grids = np.stack([synth_agent_grid(n, seed * 50 + a) for a in range(A)])
    origins = np.tile(np.array([[-4.0, -4.0]]), (A, 1))
    tf = np.stack([MO.se2_matrix(*r.uniform(-span, span, 2), r.uniform(-rot, rot)) if (span or rot) else np.eye(4)
                   for _ in range(A)])
    o, want = _oracle_chain(grids, n, 0.05, (-4.0, -4.0), tf)
    m = MM.MapMerger()
    out, origin = m.merge(grids, origins, 0.05, tf)
    assert np.array_equal(out, want[0]) and origin == want[1]
    pc = m.global_pcd
    assert pc.shape[0] == o.gx.shape[0]
    assert np.array_equal(pc[:, 0], o.gx) and np.array_equal(pc[:, 1], o.gy)
    st = m.chain_stats
    assert st['callbacks'] == A - 1 and 1 <= st['rebuilds'] <= st['callbacks']
    if span == 3.0:
        assert st['rebuilds'] < st['callbacks'], st          # the incremental path did run


def test_chain_continues_an_existing_cloud(MM):
    """A second merge() (and callbacks in between) on the same merger continue the same cloud."""
    from oracle import merge_oracle as MO
    r = np.random.default_rng(31)
    A, n = 12, 128
    grids = np.stack([synth_agent_grid(n, 900 + a) for a in range(A)])
    origins = np.tile(np.array([[-3.2, -3.2]]), (A, 1))
    tf = np.stack([MO.se2_matrix(*r.uniform(-2, 2, 2), r.uniform(-math.pi, math.pi)) for _ in range(A)])
    o, want = _oracle_chain(grids, n, 0.05, (-3.2, -3.2), tf)
    m = MM.MapMerger()
    m.merge(grids[:5], origins[:5], 0.05, tf[:5])
    m.map_callback(MM.make_grid_msg(grids[5].ravel(), n, n, 0.05, -3.2, -3.2), 6, transform=tf[5])
    out, origin = m.merge(grids[6:], origins[6:], 0.05, tf[6:])
    assert np.array_equal(out, want[0]) and origin == want[1]
    pc = m.global_pcd
    assert np.array_equal(pc[:, 0], o.gx) and np.array_equal(pc[:, 1], o.gy)


def test_chain_deep_voxel_stacks(MM):
    """Transforms that shrink the slices (scale 0.3) put ~10 slice points into one voxel: the
    per-voxel stacks of the incremental chain get deep, sums still run in ascending index."""
    from oracle import merge_oracle as MO
    r = np.random.default_rng(77)
    A, n = 10, 128
    grids = np.stack([synth_agent_grid(n, 300 + a, occ_segments=40) for a in range(A)])
    origins = np.tile(np.array([[-3.2, -3.2]]), (A, 1))
    tf = []
    for a in range(A):
        T = MO.se2_matrix(*r.uniform(-0.5, 0.5, 2), r.uniform(-math.pi, math.pi))
        T[:2, :2] *= 0.3
        tf.append(T)
    tf = np.stack(tf)
    o, want = _oracle_chain(grids, n, 0.05, (-3.2, -3.2), tf)
    m = MM.MapMerger()
    out, origin = m.merge(grids, origins, 0.05, tf)
    assert np.array_equal(out, want[0]) and origin == want[1]
    pc = m.global_pcd
    assert pc.shape[0] == o.gx.shape[0]
    assert np.array_equal(pc[:, 0], o.gx) and np.array_equal(pc[:, 1], o.gy)


def test_chain_with_rejected_and_empty_agents(MM):
    """fitness < 0.6 (:54-56) and empty grids (:37-38) are skipped inside a batched merge."""
    from oracle import merge_oracle as MO
    r = np.random.default_rng(5)
    A, n = 9, 96
    grids = [synth_agent_grid(n, 500 + a) for a in range(A)]
    grids[0] = np.full((n, n), -1, np.int8)          # empty first grid: the next one is adopted
    grids[4] = np.full((n, n), -1, np.int8)
    grids = np.stack(grids)
    origins = np.tile(np.array([[-2.4, -2.4]]), (A, 1))
    tf = np.stack([MO.se2_matrix(*r.uniform(-1, 1, 2), r.uniform(-math.pi, math.pi)) for _ in range(A)])
    fit = np.ones(A)
    fit[1] = 0.1                                      # adopted anyway: the first cloud is never registered
    fit[3] = 0.59
    fit[7] = 0.2
    o = MO.OracleMerger()
    want = None
    for a in range(A):
        out = o.map_callback(grids[a].ravel(), n, n, 0.05, -2.4, -2.4, tf[a], accept=fit[a] >= 0.6)
        want = out if out is not None else want
    m = MM.MapMerger()
    out, origin = m.merge(grids, origins, 0.05, tf, fitness=fit)
    assert np.array_equal(out, want[0]) and origin == want[1]
    pc = m.global_pcd
    assert np.array_equal(pc[:, 0], o.gx) and np.array_equal(pc[:, 1], o.gy)
    assert m.chain_stats['callbacks'] == 4            # agents 2, 5, 6, 8


def test_chain_min_corner_moves_inwards(MM):
    """The point on the cloud's min corner is re-averaged inwards by an incremental callback: the
    chain has to recompute its bounds (stall reason 3) before the next decision, which then
    re-anchors the lattice (rebuild).  Agents 1 and 3 do not see the corner, agents 2 and 4 see it
    shifted by a fraction of a voxel."""
    n = 96
    g = synth_agent_grid(n, 41)
    g[0, :] = -1
    g[:, 0] = -1
    inner = g.copy()
    inner[:6, :] = -1
    inner[:, :6] = -1
    g[0, 0] = 100                                         # the only point on the min corner
    grids = np.stack([g, inner, g, inner, g, inner])
    A = len(grids)
    origins = np.tile(np.array([[-2.4, -2.4]]), (A, 1))
    tf = np.stack([np.eye(4) for _ in range(A)])
    for a in range(A):
        tf[a, 0, 3], tf[a, 1, 3] = 0.004 * a, 0.003 * a
    o, want = _oracle_chain(grids, n, 0.05, (-2.4, -2.4), tf)
    m = MM.MapMerger()
    out, origin = m.merge(grids, origins, 0.05, tf)
    assert np.array_equal(out, want[0]) and origin == want[1]
    pc = m.global_pcd
    assert pc.shape[0] == o.gx.shape[0]
    assert np.array_equal(pc[:, 0], o.gx) and np.array_equal(pc[:, 1], o.gy)
    assert m.chain_stats['rebounds'] >= 1 and m.chain_stats['rebuilds'] < m.chain_stats['callbacks'], m.chain_stats


def test_2048_grids(MM):
    """BASELINE config 3 grid size (2048^2, ~1.5 % occupied) on a few agents, 50 m translations."""
    run_pair(MM, 2048, 4, seed=7, span=50.0, origin=(-51.2, -51.2), check_every=False)


def test_grid_of_more_than_1024_scan_blocks(MM):
    """4160^2 cells = 1 057 blocks of 16 384: the single-CTA scans of the block counts (grid_to_pcd's
    and the batched merge's) take a second round, whose offsets carry the first round's total."""
    from oracle import merge_oracle as MO
    n, res, origin = 4160, 0.05, (-104.0, -104.0)
    assert (n * n + 16383) // 16384 > 1024
    g = np.full((n, n), -1, np.int8)
    g[np.random.default_rng(17).random((n, n)) < 0.003] = 100
    pts = MM.MapMerger().grid_to_pcd(MM.make_grid_msg(g.ravel(), n, n, res, *origin))
    ox, oy = MO.grid_to_points(g.ravel(), n, n, res, *origin)
    assert np.array_equal(pts[:, 0], ox) and np.array_equal(pts[:, 1], oy)
    o = MO.OracleMerger()
    want = o.map_callback(g.ravel(), n, n, res, *origin)
    m = MM.MapMerger()
    out, org = m.merge(g[None], np.array([origin]), res)
    assert np.array_equal(out, want[0]) and org == want[1]
    pc = m.global_pcd
    assert np.array_equal(pc[:, 0], o.gx) and np.array_equal(pc[:, 1], o.gy)


def test_sharded_merger_single_rank_equals_merge(MM):
    """ShardedMapMerger (agent blocks per rank, batched extraction sharded, ordered voxel chain
    replicated) with world = 1 must equal MapMerger.merge and the oracle; an empty first grid
    exercises the 'first NON-EMPTY grid is adopted untransformed' rule (map_merger.py:37-43), and a
    second merge on the same object continues the cloud (every agent transformed from then on)."""
    from occgrid_b200.distributed import ShardedMapMerger
    from oracle import merge_oracle as MO
    r = np.random.default_rng(12)
    grids = [np.full((160, 160), -1, np.int8)] + [synth_agent_grid(160, 70 + a) for a in range(6)]
    origins = np.tile(np.array([[-4.0, -4.0]]), (7, 1))
    tf = np.stack([MO.se2_matrix(*r.uniform(-3, 3, 2), r.uniform(-math.pi, math.pi)) for _ in range(7)])
    fit = np.array([1.0, 1.0, 1.0, 0.5, 1.0, 1.0, 0.59])
    o = MO.OracleMerger()
    want = None
    for a in range(5):
        out = o.map_callback(grids[a].ravel(), 160, 160, 0.05, -4.0, -4.0, tf[a], accept=fit[a] >= 0.6)
        want = out if out is not None else want
    sm = ShardedMapMerger()
    got, origin = sm.merge(grids[:5], origins[:5], 0.05, tf[:5], 5, fitness=fit[:5])
    assert np.array_equal(got, want[0]) and origin == want[1]
    got2, origin2 = MM.MapMerger().merge(grids[:5], origins[:5], 0.05, tf[:5], fitness=fit[:5])
    assert np.array_equal(got2, want[0]) and origin2 == want[1]
    for a in (5, 6):                                   # second call: the merger already holds a cloud
        out = o.map_callback(grids[a].ravel(), 160, 160, 0.05, -4.0, -4.0, tf[a], accept=fit[a] >= 0.6)
        want = out if out is not None else want
    got3, origin3 = sm.merge(grids[5:], origins[5:], 0.05, tf[5:], 2, fitness=fit[5:])
    assert np.array_equal(got3, want[0]) and origin3 == want[1]
    pc = sm.merger.global_pcd
    assert np.array_equal(pc[:, 0], o.gx) and np.array_equal(pc[:, 1], o.gy)


def test_raster_fuse_mode_single_rank_equals_merge(MM):
    """mode='raster_fuse' (per-rank chain + bounds all-reduce + max fuse of partial rasters, SURVEY
    §8e) degenerates to the exact merge when one rank holds every agent."""
    from occgrid_b200.distributed import ShardedMapMerger
    from oracle import merge_oracle as MO
    r = np.random.default_rng(13)
    grids = [synth_agent_grid(128, 170 + a) for a in range(4)]
    origins = np.tile(np.array([[-3.2, -3.2]]), (4, 1))
    tf = np.stack([MO.se2_matrix(*r.uniform(-2, 2, 2), r.uniform(-math.pi, math.pi)) for _ in range(4)])
    o = MO.OracleMerger()
    for a in range(4):
        want = o.map_callback(grids[a].ravel(), 128, 128, 0.05, -3.2, -3.2, tf[a])
    got, origin = ShardedMapMerger(mode='raster_fuse').merge(grids, origins, 0.05, tf, 4)
    assert np.array_equal(got, want[0]) and origin == want[1]


# ---- fixtures produced by EXECUTING the unmodified reference (oracle/make_golden_merge.py) --------
@pytest.mark.parametrize('seq', ['A', 'B', 'C'])
def test_callbacks_equal_reference_executed_fixture(MM, seq):
    """tests/golden/merge_ref.npz: the reference's own map_callback / grid_to_pcd /
    publish_global_map ran on these grids.  Every callback on the device must return early where
    the reference did, hold the same cloud (fp64 bit for bit, same order), keep the same
    map_resolution / map_origin and publish the same int8 grid and origin."""
    steps = load_merge_ref()[seq]
    m = MM.MapMerger()
    for k, s in enumerate(steps):
        g = s['grid']
        h, w = g.shape
        res, ox, oy = s['geom'].tolist()
        msg = MM.make_grid_msg(g.ravel(), w, h, res, ox, oy)
        pts = m.grid_to_pcd(msg)                                             # a10 (:64-85)
        assert np.array_equal(pts, s['pcd'].reshape(-1, 3)), k
        got = m.map_callback(msg, k + 1, transform=s['T'], fitness=float(s['fitness']))
        assert (got is not None) == bool(s['published']), k
        assert np.array_equal(m.global_pcd[:, :2], s['cloud']), k
        assert [m.map_resolution] + list(m.map_origin) == s['state'].tolist(), k
        if got is not None:                                                  # a12 (:87-127)
            assert got.header.frame_id == 'map_global'
            assert (got.info.height, got.info.width) == s['out'].shape and got.info.resolution == float(s['out_res'])
            assert np.array_equal(got.data, s['out']), k
            assert [got.info.origin.position.x, got.info.origin.position.y] == s['out_origin'].tolist(), k


@pytest.mark.parametrize('seq', ['A', 'C'])
def test_batched_merge_equals_reference_executed_fixture(MM, seq):
    """The batched entry (one extraction launch + incremental chain) must end where the
    reference's callback sequence ended."""
    steps = load_merge_ref()[seq]
    grids = np.stack([s['grid'] for s in steps])
    origins = np.stack([s['geom'][1:] for s in steps])
    tf = np.stack([s['T'] for s in steps])
    fit = np.array([float(s['fitness']) for s in steps])
    m = MM.MapMerger()
    out, origin = m.merge(grids, origins, float(steps[0]['geom'][0]), tf, fitness=fit)
    last = [s for s in steps if bool(s['published'])][-1]
    assert np.array_equal(out, last['out']) and list(origin) == last['out_origin'].tolist()
    assert np.array_equal(m.global_pcd[:, :2], steps[-1]['cloud'])


def test_publish_equals_reference_on_handmade_clouds(MM):
    """publish_global_map (:87-127) alone: ceil + 1 extents, astype(int) truncation and clipping
    on clouds that never went through a grid."""
    for case in load_merge_ref()['P']:
        pts = case['points']
        m = MM.MapMerger()
        m._ensure_capacity(len(pts))
        m._cloud.x[:len(pts)].copy_(torch.from_numpy(pts[:, 0].copy()))
        m._cloud.y[:len(pts)].copy_(torch.from_numpy(pts[:, 1].copy()))
        m._cloud.count.fill_(len(pts))
        m._n_global = len(pts)
        m.map_resolution = float(case['res'])
        got = m.publish_global_map('map')
        assert np.array_equal(got.data, case['out'])
        assert [got.info.origin.position.x, got.info.origin.position.y] == case['out_origin'].tolist()


def test_icp_callbacks_against_reference_driven_fixture(MM):
    """Sequence D: the reference's map_callback called registration_icp itself (restated Open3D
    algorithm) on partial views.  MapMerger(registration='icp') must accept the same callbacks,
    find the same correspondence counts, and publish the same map up to the cells a <= 1e-9 m
    difference in the estimated transform can move across a cell edge."""
    ref = load_merge_ref()
    steps, calls = ref['D'], ref['D_meta']['icp_calls']
    m = MM.MapMerger(registration='icp')
    j = 0
    for k, s in enumerate(steps):
        g = s['grid']
        h, w = g.shape
        res, ox, oy = s['geom'].tolist()
        got = m.map_callback(MM.make_grid_msg(g.ravel(), w, h, res, ox, oy), k + 1)
        assert (got is not None) == bool(s['published'])
        if k:
            reg = m.last_registration
            assert reg.fitness == calls[j, 3] and reg.correspondences == round(calls[j, 3] * calls[j, 0])
            j += 1
        pc = m.global_pcd[:, :2]
        assert pc.shape == s['cloud'].shape
        assert np.abs(pc - s['cloud']).max() < 1e-8
        assert got.data.shape == s['out'].shape
        assert (got.data != s['out']).mean() < 1e-3
        assert np.abs(np.array([got.info.origin.position.x, got.info.origin.position.y]) - s['out_origin']).max() < 1e-8
