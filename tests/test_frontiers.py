"""Frontier detection + clustering (SURVEY §8 row f1; reference dual_bot_mapper.py:181-237).
CPU part: the oracle restatement against the fixtures produced by the unmodified reference.
GPU part: the CUDA path (occgrid_frontiers / occgrid_frontier_clusters through the
reference-shaped OccupancyGrid methods) against fixtures and oracle.  Integer lists and cluster
membership must be identical; centroids are fp64 and must be bit-equal (integer sums, one division,
the reference's grid_to_world expression)."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLD, session_packets
from oracle import occgrid_oracle as O


def describe(fr, cl, ce):
    return {'n_frontiers': len(fr), 'frontiers_sha1': hashlib.sha1(np.asarray(fr, np.int32).tobytes()).hexdigest(),
            'n_clusters': len(cl), 'cluster_sizes': [len(c) for c in cl], 'cluster_first': [list(min(c, key=lambda t: (t[1], t[0]))) for c in cl],
            'centroids': [list(c) for c in ce],
            'cluster_sets_sha1': hashlib.sha1(json.dumps([sorted(map(list, c)) for c in cl]).encode()).hexdigest()}


def session_grid():
    pk, _ = session_packets(True)
    g, _ = O.replay(pk)
    return g.grid


def test_oracle_matches_reference_fixtures(golden):
    g = session_grid()
    fr = O.get_frontiers(g)
    assert fr == O.get_frontiers_fast(g)
    cl = O.cluster_frontiers(fr)
    got = describe(fr, cl, [O.cluster_centroid_world(c, -5.0, -5.0, 0.05) for c in cl])
    assert got == golden['frontiers_session_time_off']
    rg = np.load(os.path.join(GOLD, 'frontier_random_grid.npy'))
    fr = O.get_frontiers(rg)
    cl = O.cluster_frontiers(fr)
    got = describe(fr, cl, [O.cluster_centroid_world(c, -3.3, 7.7, 0.1) for c in cl])
    assert got == golden['frontiers_random96']
    # in the reference the first cell of a BFS cluster is also its first cell in scan order
    assert all(c[0] == min(c, key=lambda t: (t[1], t[0])) for c in cl)


torch = pytest.importorskip('torch')


def gpu_grid(arr, **kw):
    from occgrid_b200 import dual_bot_mapper as M
    g = M.OccupancyGrid(size=arr.shape[0], **kw)
    g.grid_tensor.copy_(torch.from_numpy(arr))
    return g


@pytest.mark.gpu
def test_gpu_frontiers_match_reference_fixtures(golden):
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    for arr, kw, key in ((session_grid(), {}, 'frontiers_session_time_off'),
                         (np.load(os.path.join(GOLD, 'frontier_random_grid.npy')),
                          dict(resolution=0.1, origin_x=-3.3, origin_y=7.7), 'frontiers_random96')):
        g = gpu_grid(arr, **kw)
        fr = g.get_frontiers()
        cl = g.cluster_frontiers(fr)
        ce = g.frontier_centroids()
        assert describe(fr, cl, ce) == golden[key]
        assert [g.cluster_centroid_world(c) for c in cl] == [tuple(c) for c in ce]


@pytest.mark.gpu
@pytest.mark.parametrize('seed', [0, 1])
def test_gpu_frontiers_large_grid_vs_oracle(seed):
    """4096^2 grid integrated from a synthetic swarm batch, plus random speckle: frontier list,
    cluster partition, order and centroids equal the oracle (vectorised stencil + the reference's
    BFS restated)."""
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper as M, simulation_tools as st
    s = st.generate_session(n_agents=64, n_packets=150_000, seed=60 + seed)
    g = M.OccupancyGrid(max_batch=150_000, **s['grid'])
    g.update_packets(s['packets'], agent_offsets=s['agent_offsets'])
    arr = g.grid.copy()
    rng = np.random.default_rng(seed)
    ys, xs = rng.integers(0, 4096, 20000), rng.integers(0, 4096, 20000)
    arr[ys, xs] = rng.choice(np.array([-1, 0, 100], np.int8), 20000)
    g.grid_tensor.copy_(torch.from_numpy(arr))
    fr = g.get_frontiers()
    want_fr = O.get_frontiers_fast(arr)
    assert fr == want_fr and len(fr) > 1000
    want_cl = O.cluster_frontiers(want_fr)
    cl = g.cluster_frontiers(fr)
    assert [sorted(c) for c in cl] == [sorted(c) for c in want_cl]
    assert g.frontier_centroids() == [O.cluster_centroid_world(c, g.ox, g.oy, g.res) for c in want_cl]


@pytest.mark.gpu
def test_gpu_frontiers_more_than_one_reserve_round():
    """8208^2 cells = 16 449 blocks of 4 096: the single-CTA scan of the block counts (16 per thread
    and round) takes a second round, whose offsets carry the first round's total."""
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    n = 8208
    assert (n * n + 4095) // 4096 > 1024 * 16
    rng = np.random.default_rng(3)
    arr = np.full((n, n), -1, np.int8)
    arr[rng.integers(0, n, 40000), rng.integers(0, n, 40000)] = 0
    g = gpu_grid(arr)
    fr = g.get_frontiers()
    want = O.get_frontiers_fast(arr)
    assert fr == want and sum(y * n + x >= 1024 * 16 * 4096 for x, y in want) > 50


@pytest.mark.gpu
def test_gpu_frontiers_edge_cases():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import dual_bot_mapper as M
    g = M.OccupancyGrid(size=16)
    assert g.get_frontiers() == [] and g.cluster_frontiers() == [] and g.frontier_centroids() == []
    a = np.zeros((16, 16), np.int8)                   # all free: no unknown neighbour anywhere
    g.grid_tensor.copy_(torch.from_numpy(a))
    assert g.get_frontiers() == []
    a[:, :] = -1
    a[5, 5:8] = 0                                     # one 3-cell cluster, one 2-cell cluster (dropped), border cells ignored
    a[9, 2:4] = 0
    a[0, 0:5] = 0
    g.grid_tensor.copy_(torch.from_numpy(a))
    assert g.get_frontiers() == [(5, 5), (6, 5), (7, 5), (2, 9), (3, 9)]
    assert g.cluster_frontiers() == [[(5, 5), (6, 5), (7, 5)]]
    assert g.frontier_centroids() == [g.grid_to_world(6.0, 5.0)]
    w = M.OccupancyGrid(size=64, window=(0, 0, 64, 32))
    with pytest.raises(M.OccGridError):
        w.get_frontiers()
