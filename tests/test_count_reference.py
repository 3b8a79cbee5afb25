"""The C count reference (oracle_accumulate_packets) pinned without a GPU: it must reproduce the
golden count planes of the unmodified reference, the Python OracleCountGrid on the adversarial
packet streams, and agree with itself and with the int8 integrate path on random streams
(windows are crops of the full grid; the touched cells are the known cells of the grid).  The GPU
count kernels are compared with this reference in tests/test_gpu_counts_reference.py."""
import os

import numpy as np
import pytest

from conftest import GOLD, load_packet_stream, normalise_datagrams, session_packets
from oracle import c_oracle
from oracle import occgrid_oracle as O


RECORD = np.dtype([('magic', 'S4'), ('agent', 'u1'), ('x', '<f4'), ('y', '<f4'), ('yaw', '<f4'), ('enc', '<i4'),
                   ('v2v', '<u4'), ('d', '<f4', 4), ('lm', 'u1')])       # the 42-byte v2 wire record


def make_packets(rng, n, span, ox, oy, n_agents):
    """Random 42-byte v2 records over a span x span m square at (ox, oy) and 2 m around it: bad
    magic, foreign agent ids, boundary / NaN / inf / out-of-range distances, cell-aligned x and
    15-degree yaws (the generator of tests/test_gpu_property.py)."""
    special = np.array([0.0, -1.0, 4.0, np.nan, np.inf, 0.05, 1.2, 1.2000001, 0.050000004, 0.01, 2.5], np.float32)
    out = np.zeros((n, 42), np.uint8)
    rec = out.view(RECORD)[:, 0]
    rec['magic'] = b'QSRL'
    rec['magic'][rng.random(n) < 0.03] = b'QSRX'
    rec['agent'] = rng.integers(0, n_agents + 2, n)
    rec['x'] = rng.uniform(ox - 2, ox + span + 2, n)
    rec['y'] = rng.uniform(oy - 2, oy + span + 2, n)
    q = rng.random(n) < 0.3
    rec['x'][q] = np.round(rec['x'][q] / 0.05) * 0.05
    rec['yaw'] = np.where(rng.random(n) < 0.5, np.radians(15.0 * rng.integers(-12, 13, n)), rng.uniform(-7, 7, n))
    d = rng.uniform(0, 1.5, (n, 4)).astype(np.float32)
    m = rng.random((n, 4)) < 0.2
    d[m] = special[rng.integers(0, len(special), int(m.sum()))]
    rec['d'] = d
    return out


def logodds_reference(counts, l_occ, l_free, l_min, l_max):
    """clamp(hits * l_occ + misses * l_free) from int32 {miss, hit} planes: each product and the sum
    rounded to float64 separately (NumPy does not contract), then one rounding to float32."""
    h = counts[..., 1].astype(np.float64)
    m = counts[..., 0].astype(np.float64)
    return np.clip(h * l_occ + m * l_free, l_min, l_max).astype(np.float32)


def fma_sensitive_counts(l_occ, l_free, n=4096, seed=0):
    """int32 [n, 2] {miss, hit} pairs whose log-odds change if h * l_occ + m * l_free is contracted
    into a fused multiply-add.  h is 2^24..2^26 and m makes the sum cancel to a few units, so the
    rounding error of one float64 product (up to 2^-29) is a visible fraction of the float32 spacing
    of the result: a few percent of these cells round to a different float32."""
    rng = np.random.default_rng(seed)
    h = rng.integers(1 << 24, 1 << 26, n)
    m = np.round(h * (l_occ / -l_free)).astype(np.int64) + rng.integers(-8, 9, n)
    assert (m >= 0).all() and (m < 2 ** 31).all()
    return np.stack([m, h], axis=1).astype(np.int32)


def _fused(a, x, p):
    """fl(a * x + p) with one rounding: what fma(a, x, p) returns."""
    from fractions import Fraction
    return float(Fraction(int(a)) * Fraction(x) + Fraction(p))      # int / int division rounds correctly


@pytest.mark.parametrize('l_occ, l_free', [(0.85, -0.4), (0.9, -0.35), (-0.7, 0.3)])
def test_fma_sensitive_counts_tell_a_contraction(l_occ, l_free):
    """The log-odds test on the GPU is bit-exact and feeds these cells: confirm here that both ways
    of contracting the expression into an FMA give a different float32 on many of them."""
    c = fma_sensitive_counts(l_occ, l_free)
    want = logodds_reference(c, l_occ, l_free, -1e30, 1e30)
    m, h = c[:, 0].astype(np.float64), c[:, 1].astype(np.float64)
    fused_occ = np.array([_fused(a, l_occ, p) for a, p in zip(c[:, 1], m * l_free)]).astype(np.float32)
    fused_free = np.array([_fused(a, l_free, p) for a, p in zip(c[:, 0], h * l_occ)]).astype(np.float32)
    assert (fused_occ != want).sum() >= 40 and (fused_free != want).sum() >= 40
    assert np.abs(want).max() < 8


@pytest.mark.parametrize('slam', [False, True])
def test_reference_equals_golden_session_counts(slam):
    pk, _ = session_packets(True)
    drift = np.load(os.path.join(GOLD, 'session_drift_time.npy')) if slam else None
    arr, d = normalise_datagrams(pk, drift)
    counts = np.zeros((200, 200, 2), np.int32)
    c = c_oracle.accumulate_packets(arr, counts, -5.0, -5.0, 0.05, drift=d)
    z = np.load(os.path.join(GOLD, 'session_counts.npz'))
    tag = 'slam_on' if slam else 'slam_off'
    assert np.array_equal(counts[..., 0], z[f'miss_{tag}']) and np.array_equal(counts[..., 1], z[f'hit_{tag}'])
    grid = np.full((200, 200), -1, np.int8)
    assert c == c_oracle.integrate_packets(arr, grid, -5.0, -5.0, 0.05, drift=d)     # same counters
    assert c['packets'] == 687 and c['beams'] == 2748


@pytest.mark.parametrize('name', ['mixed_a', 'mixed_b_sep', 'mixed_c_4096', 'mixed_d_edge'])
def test_reference_equals_python_count_oracle(golden, name):
    """Bad magic, foreign agents, v1/junk sizes, NaN/inf ranges, out-of-grid rays, cell-boundary
    yaws, agent separation and SLAM drift: the C planes equal the per-packet Python replay."""
    want = golden['packet_streams'][name]
    pk, ref_drift = load_packet_stream(name)
    og = O.OracleCountGrid(**want['grid_kwargs'])
    _, st = O.replay(pk, grid=og, separation=want['separation'], slam=O.OracleSLAM() if want['slam'] else None)
    arr, d = normalise_datagrams(pk, ref_drift if want['slam'] else None)
    counts = np.zeros((og.size, og.size, 2), np.int32)
    c = c_oracle.accumulate_packets(arr, counts, og.ox, og.oy, og.res, separation=want['separation'], drift=d)
    assert np.array_equal(counts[..., 0], og.miss) and np.array_equal(counts[..., 1], og.hit)
    assert (c['beams'], c['hits'], c['updates']) == (st['beams'], st['hits'], st['updates'])
    assert og.hit.any() and og.miss.any()


@pytest.mark.parametrize('seed', range(6))
def test_reference_windows_and_touched_cells(seed):
    rng = np.random.default_rng(1000 + seed)
    size = int(rng.integers(20, 160))
    res = float(rng.choice([0.03, 0.05, 0.1]))
    ox, oy = float(rng.uniform(-20, 5)), float(rng.uniform(-20, 5))
    n_agents = int(rng.integers(1, 6))
    offs = np.zeros((n_agents + 1, 2))
    offs[1:] = rng.uniform(-1, 1, (n_agents, 2))
    n = int(rng.integers(200, 1500))
    stride = int(rng.choice([42, 48, 64]))
    buf = np.zeros((n, stride), np.uint8)
    buf[:, :42] = make_packets(rng, n, size * res, ox, oy, n_agents)
    drift = rng.normal(0, 0.05, (n, 2)) if seed % 2 else None
    kw = dict(agent_offsets=offs, drift=drift)
    full = np.zeros((size, size, 2), np.int32)
    c = c_oracle.accumulate_packets(buf, full, ox, oy, res, **kw)
    grid = np.full((size, size), -1, np.int8)
    assert c == c_oracle.integrate_packets(buf, grid, ox, oy, res, **kw)
    assert np.array_equal(full.sum(axis=2) > 0, grid != -1)
    assert c['hits'] > 0 and full[..., 1].any() and full[..., 0].sum() > full[..., 1].sum()
    for _ in range(4):
        x0, y0 = int(rng.integers(0, size)), int(rng.integers(0, size))
        w, h = int(rng.integers(1, size - x0 + 1)), int(rng.integers(1, size - y0 + 1))
        win = np.full((h, w, 2), 7, np.int32)                        # adds to what is there
        cw = c_oracle.accumulate_packets(buf, win, ox, oy, res, window=(x0, y0), size_x=size, size_y=size, **kw)
        assert np.array_equal(win - 7, full[y0:y0 + h, x0:x0 + w])
        assert cw == c                                               # the window clips cells, not packets


def test_reference_single_packet_by_hand():
    """One packet at a cell centre of a 5 cm grid, yaw 0: front hits 10 cells east, left misses
    (1.2 m = 24 cells north), back is below MIN_DIST (a 1.2 m miss west), right hits 5 cells south."""
    import struct
    ox = oy = -5.0
    x, y = ox + 100.5 * 0.05, oy + 100.5 * 0.05
    pk = struct.pack(O.PACKET_FMT, b'QSRL', 1, x, y, 0.0, 0, 0, 0.5, 3.0, 0.01, 0.25, 0)
    counts = np.zeros((200, 200, 2), np.int32)
    c = c_oracle.accumulate_packets(np.frombuffer(pk, np.uint8)[None], counts, ox, oy, 0.05)
    assert counts[100, 100, 0] == 4 and counts[100, 100, 1] == 0       # every beam starts with a miss here
    assert counts[100, 110, 1] == 1 and counts[100, 110, 0] == 0       # front end cell: hit only
    assert counts[95, 100, 1] == 1 and counts[96:100, 100, 0].tolist() == [1, 1, 1, 1]
    assert counts[..., 1].sum() == 2 == c['hits']
    assert counts[..., 0].sum() + c['beams'] == c['updates']          # every end cell is not a miss
