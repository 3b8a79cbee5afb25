"""ICP registration (map_merger.py:45-56): the oracle restatement on its own (CPU) and the CUDA
path against it (GPU).  Parity is UNPINNED (Open3D absent, see oracle/icp_oracle.py): tolerances
are stated per assertion; the correspondence COUNT (fitness) must be equal."""
import math

import numpy as np
import pytest

from merge_util import synth_agent_grid
from oracle import icp_oracle as IO
from oracle import merge_oracle as MO


def _cloud(n, seed, res=0.05, origin=(-6.4, -6.4), segs=40):
    g = synth_agent_grid(n, seed, occ_segments=segs)
    x, y = MO.grid_to_points(g.ravel(), n, n, res, origin[0], origin[1])
    return g, x, y


def test_oracle_recovers_a_known_transform():
    _, x, y = _cloud(256, 3)
    T = MO.se2_matrix(0.12, -0.08, 0.03)
    sx, sy = MO.transform_points(x, y, np.linalg.inv(T))
    Th, fit, rmse, its = IO.registration_icp(sx, sy, x, y)
    assert fit == 1.0 and rmse < 1e-12 and 1 <= its <= 30
    assert np.allclose(Th, T, atol=1e-12)


def test_oracle_planar_umeyama_equals_closed_form():
    """The CUDA path fits theta = atan2(sum cross, sum dot); the oracle keeps Eigen's 3-D Umeyama."""
    r = np.random.default_rng(0)
    src = np.vstack([r.uniform(-5, 5, (2, 500)), np.zeros((1, 500))])
    T = MO.se2_matrix(0.7, -1.3, 0.41)
    dst = (T[:3, :3] @ src) + T[:3, 3:4] + np.vstack([r.normal(0, 0.01, (2, 500)), np.zeros((1, 500))])
    U = IO._umeyama_rigid(src, dst)
    ms, md = src.mean(1), dst.mean(1)
    s, d = src - ms[:, None], dst - md[:, None]
    th = math.atan2((s[0] * d[1] - s[1] * d[0]).sum(), (s[0] * d[0] + s[1] * d[1]).sum())
    R = np.array([[math.cos(th), -math.sin(th)], [math.sin(th), math.cos(th)]])
    assert np.allclose(U[:2, :2], R, atol=1e-12)
    assert np.allclose(U[:2, 3], md[:2] - R @ ms[:2], atol=1e-12)
    assert U[2, 2] == pytest.approx(1.0, abs=1e-12)


def test_oracle_no_overlap_gives_zero_fitness():
    _, x, y = _cloud(128, 4)
    Th, fit, rmse, its = IO.registration_icp(x + 100.0, y, x, y)
    assert fit == 0.0 and rmse == 0.0 and its == 1 and np.array_equal(Th, np.eye(4))


@pytest.fixture(scope='module')
def MM():
    torch = pytest.importorskip('torch')
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import map_merger
    return map_merger


@pytest.mark.gpu
@pytest.mark.parametrize('tx,ty,th,seed', [(0.12, -0.08, 0.03, 3), (-0.3, 0.25, -0.06, 8), (0.0, 0.0, 0.0, 5), (0.6, 0.4, 0.1, 9)])
def test_gpu_registration_matches_oracle(MM, tx, ty, th, seed):
    n, res, origin = 256, 0.05, (-6.4, -6.4)
    g, x, y = _cloud(n, seed)
    g2 = synth_agent_grid(n, seed, occ_segments=40)
    g2[:, : n // 5] = -1                                   # the local map sees only part of the scene ...
    r = np.random.default_rng(seed)
    g2[r.random((n, n)) < 0.001] = 100                     # ... plus some clutter the global map lacks
    lx, ly = MO.grid_to_points(g2.ravel(), n, n, res, *origin)
    T = MO.se2_matrix(tx, ty, th)
    # global cloud = the scene moved by T (adopted as is); the local grid then has to be moved by ~T
    m = MM.MapMerger(registration='icp')
    gx, gy = MO.transform_points(x, y, T)
    m._ensure_capacity(gx.shape[0] + 16)
    import torch
    m._cloud.x[:gx.shape[0]].copy_(torch.from_numpy(gx))
    m._cloud.y[:gx.shape[0]].copy_(torch.from_numpy(gy))
    m._cloud.count.fill_(gx.shape[0])
    m._n_global = gx.shape[0]
    reg = m.register(MM.make_grid_msg(g2.ravel(), n, n, res, *origin))
    Tw, fw, rw, iw = IO.registration_icp(lx, ly, gx, gy)
    assert reg.correspondences == round(fw * lx.shape[0])          # same correspondence count
    assert reg.fitness == fw
    assert reg.iterations == iw
    assert abs(reg.inlier_rmse - rw) < 1e-9
    assert np.allclose(reg.transformation, Tw, atol=1e-9)
    if (tx, ty, th) != (0.6, 0.4, 0.1):                            # within the basin of a 1 m threshold
        assert np.allclose(reg.transformation, T, atol=0.02)


@pytest.mark.gpu
def test_gpu_callbacks_with_icp_match_oracle_chain(MM):
    """map_callback without a transform: register, gate on fitness, transform, fuse (:45-60)."""
    n, res, origin = 192, 0.05, (-4.8, -4.8)
    base = synth_agent_grid(n, 21, occ_segments=30)
    m = MM.MapMerger(registration='icp')
    o = MO.OracleMerger()
    r = np.random.default_rng(2)
    for a in range(4):
        g = base.copy()
        g[r.random((n, n)) < 0.02] = -1                    # every agent misses a few cells
        sh = (int(r.integers(-2, 3)), int(r.integers(-2, 3)))
        g = np.roll(g, sh, axis=(0, 1))                    # and is offset by a few cells (<= 0.1 m)
        got = m.map_callback(MM.make_grid_msg(g.ravel(), n, n, res, *origin), a + 1)
        if a == 0:
            want = o.map_callback(g.ravel(), n, n, res, origin[0], origin[1])
        else:
            lx, ly = MO.grid_to_points(g.ravel(), n, n, res, *origin)
            Tw, fw, _, _ = IO.registration_icp(lx, ly, o.gx, o.gy)
            assert m.last_registration.fitness == fw
            assert np.allclose(m.last_registration.transformation, Tw, atol=1e-9)
            # fuse with the DEVICE's transform so that the clouds stay bit-comparable downstream
            want = o.map_callback(g.ravel(), n, n, res, origin[0], origin[1], m.last_registration.transformation, accept=fw >= 0.6)
        assert (got is None) == (want is None)
        if got is not None:
            assert np.array_equal(got.data, want[0])
            pc = m.global_pcd
            assert np.array_equal(pc[:, 0], o.gx) and np.array_equal(pc[:, 1], o.gy)
    far = np.roll(base, (60, 60), axis=(0, 1))             # 3 m off: registration must fail the gate or stay consistent
    lx, ly = MO.grid_to_points(far.ravel(), n, n, res, origin[0] + 40.0, origin[1])
    got = m.map_callback(MM.make_grid_msg(far.ravel(), n, n, res, origin[0] + 40.0, origin[1]), 9)
    assert got is None and m.last_registration.fitness < 0.6


@pytest.mark.gpu
def test_gpu_no_overlap_is_rejected(MM):
    """No target within 1 m of any source point: zero correspondences, identity transform, one
    iteration (the second evaluation equals the first), and map_callback rejects the grid."""
    n, res = 128, 0.05
    g = synth_agent_grid(n, 4)
    m = MM.MapMerger(registration='icp')
    assert m.map_callback(MM.make_grid_msg(g.ravel(), n, n, res, -3.2, -3.2), 1) is not None
    k = m.global_pcd.shape[0]
    far = MM.make_grid_msg(g.ravel(), n, n, res, 100.0, -3.2)
    reg = m.register(far)
    assert reg.fitness == 0.0 and reg.inlier_rmse == 0.0 and reg.correspondences == 0 and reg.iterations == 1
    assert np.array_equal(reg.transformation, np.eye(4))
    assert m.map_callback(far, 2) is None and m.global_pcd.shape[0] == k
    assert m.register(MM.make_grid_msg(np.full(n * n, -1, np.int8), n, n, res, 0.0, 0.0)) is None


@pytest.mark.gpu
def test_gpu_registration_of_a_cloud_larger_than_the_resident_grid(MM):
    """150 k source points = ~590 virtual blocks of the loop kernel, more than the CTAs a B200 keeps
    resident (444): the persistent grid strides over them, and the result must not depend on it —
    same correspondences, iterations and transform as the oracle."""
    import torch
    n, res, origin = 1024, 0.05, (-25.6, -25.6)
    r = np.random.default_rng(11)
    g = np.where(r.random((n, n)) < 0.145, 100, 0).astype(np.int8)
    lx, ly = MO.grid_to_points(g.ravel(), n, n, res, *origin)
    assert lx.shape[0] > 444 * 256
    T = MO.se2_matrix(0.011, -0.007, 0.0004)               # well inside the basin of a dense random cloud
    gx, gy = MO.transform_points(lx, ly, T)
    m = MM.MapMerger(registration='icp')
    m._ensure_capacity(gx.shape[0] + 16)
    m._cloud.x[:gx.shape[0]].copy_(torch.from_numpy(gx))
    m._cloud.y[:gx.shape[0]].copy_(torch.from_numpy(gy))
    m._cloud.count.fill_(gx.shape[0])
    m._n_global = gx.shape[0]
    reg = m.register(MM.make_grid_msg(g.ravel(), n, n, res, *origin), max_iteration=6)
    Tw, fw, rw, iw = IO.registration_icp(lx, ly, gx, gy, max_iteration=6)
    assert reg.correspondences == round(fw * lx.shape[0]) and reg.fitness == fw and reg.iterations == iw
    assert abs(reg.inlier_rmse - rw) < 1e-9
    assert np.allclose(reg.transformation, Tw, atol=1e-9)


@pytest.mark.gpu
def test_gpu_registration_with_a_cell_index_of_more_than_1024_scan_blocks(MM):
    """A cluster 1 km below and left of the scene stretches the target's cell index past 1 024
    blocks of 16 384 cells: the single-CTA scan of the block sums takes a second round, and the
    scene's cells, all in that round, are found only if their offsets carry the first round's total."""
    import torch
    g, x, y = _cloud(256, 3)
    gx, gy = MO.transform_points(x, y, MO.se2_matrix(0.12, -0.08, 0.03))
    r = np.random.default_rng(4)
    gx = np.concatenate([r.uniform(-1040.0, -1030.0, 64), gx])
    gy = np.concatenate([r.uniform(-1040.0, -1030.0, 64), gy])
    cell = 1.0 / 4.0                                       # MapMerger.register's index cell for a 1 m threshold
    cw, ch = int((gx.max() - gx.min()) / cell) + 2, int((gy.max() - gy.min()) / cell) + 2
    assert (cw * ch + 16383) // 16384 > 1024
    m = MM.MapMerger(registration='icp')
    m._ensure_capacity(gx.shape[0] + 16)
    m._cloud.x[:gx.shape[0]].copy_(torch.from_numpy(gx))
    m._cloud.y[:gx.shape[0]].copy_(torch.from_numpy(gy))
    m._cloud.count.fill_(gx.shape[0])
    m._n_global = gx.shape[0]
    reg = m.register(MM.make_grid_msg(g.ravel(), 256, 256, 0.05, -6.4, -6.4))
    Tw, fw, rw, iw = IO.registration_icp(x, y, gx, gy)
    assert fw > 0.6
    assert reg.correspondences == round(fw * x.shape[0]) and reg.fitness == fw and reg.iterations == iw
    assert abs(reg.inlier_rmse - rw) < 1e-9
    assert np.allclose(reg.transformation, Tw, atol=1e-9)
