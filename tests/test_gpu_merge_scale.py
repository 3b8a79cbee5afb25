"""The merge path at the scale of BASELINE configs[2] (256 grids of 2048^2 at 5 cm under random SE(2))
and at the shapes, values and argument edges the smaller merge tests never reach.

A. The batched extraction (mapmerge_extract_batch_count + _write) called through the C ABI and
   compared with NumPy's grid_to_points / transform_points: per-agent totals, the offset table, every
   point, bit for bit.  The bulk-copy (TMA) scan runs persistent CTAs with a ring of stages; the ring
   only wraps (stage refills, mbarrier parity 1, reused per-stage counters) when every CTA consumes
   several laps of chunks, so those cases assert that they do.
B. MapMerger.merge against OracleMerger across several bursts of the incremental chain, with stalls
   serviced in a later burst, on non-square, mixed-shape and non-aligned inputs and on the bench
   geometry itself.
C. Host-only argument checks of the older mapmerge_* entry points (no GPU needed).

fp64 coordinates are compared with np.array_equal, clouds in order, published grids and origins
exactly, as in test_gpu_merge.py.
"""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from occgrid_b200 import _native
from merge_util import synth_agent_grid

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MERGE_CU = os.path.join(ROOT, 'distributed-multi-agent-slam-swarm-robotics-system_b200', 'csrc', 'mapmerge.cu')

# k_batch_count_tma's geometry (mapmerge.cu): chunks of 16 384 cells, SCAN_CTAS_PER_SM persistent CTAs
# per SM, SCAN_STAGES stages each.  Pinned by test_scan_constants_match_the_kernel.
CHUNK = 16384
SCAN_CTAS_PER_SM = 3
SCAN_STAGES = 4
RING_LAPS = 2                 # every CTA goes round its ring twice: both parities, every stage refilled
BURST = 64                    # callbacks per mapmerge_chain_run in MapMerger._run_chain


@pytest.fixture(scope='module')
def lib():
    return _native.lib()


@pytest.fixture(scope='module')
def torch():
    t = pytest.importorskip('torch')
    if not t.cuda.is_available():
        pytest.skip('no CUDA device')
    return t


@pytest.fixture(scope='module')
def MM(torch):
    from occgrid_b200 import map_merger
    return map_merger


def test_scan_constants_match_the_kernel():
    src = open(MERGE_CU).read()
    assert re.search(r'constexpr int kScanStages = (\d+);', src).group(1) == str(SCAN_STAGES)
    assert re.search(r'constexpr int kScanCtasPerSm = (\d+);', src).group(1) == str(SCAN_CTAS_PER_SM)
    assert re.search(r'constexpr int kCellsPerThread = (\d+);', src).group(1) == '64'
    src = open(os.path.join(os.path.dirname(MERGE_CU), '..', 'map_merger.py')).read()
    assert re.search(r'cursor, burst = 0, (\d+)', src).group(1) == str(BURST)


# ---- A. batched extraction through the C ABI -------------------------------------------------------
def ring_chunks_needed(torch):
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    return RING_LAPS * SCAN_STAGES * SCAN_CTAS_PER_SM * sms


def batch_extract(torch, lib, ptrs, w, h, res, origins, T=None, use=None, bulk_ok=None):
    """mapmerge_extract_batch_count + _write on the grids at device addresses `ptrs`.
    -> (totals [A], offsets [A + 1], x, y, status); x / y are the whole output arrays, with a NaN tail."""
    A = len(ptrs)
    dev = torch.device('cuda', torch.cuda.current_device())
    stream = torch.cuda.current_stream().cuda_stream
    if bulk_ok is None:                                      # MapMerger._count_occupied's rule
        bulk_ok = 1 if all(p % 16 == 0 for p in ptrs) else 0
    d_ptrs = torch.tensor(list(ptrs), dtype=torch.int64, device=dev)
    nbytes = lib.mapmerge_extract_batch_workspace_bytes(h * w, A)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    total = torch.full((A,), -7, dtype=torch.int64, device=dev)
    rc = lib.mapmerge_extract_batch_count(d_ptrs.data_ptr(), A, w, h, total.data_ptr(), ws.data_ptr(), nbytes, bulk_ok, stream)
    assert rc == 0, _native.last_error()
    totals = total.cpu().numpy()
    use_h = np.ones(A, np.uint8) if use is None else np.ascontiguousarray(np.asarray(use, np.uint8))
    n = int(totals[use_h != 0].sum())
    cap = n + 16
    px = torch.full((cap,), float('nan'), dtype=torch.float64, device=dev)
    py = torch.full((cap,), float('nan'), dtype=torch.float64, device=dev)
    offs = torch.full((A + 1,), -7, dtype=torch.int64, device=dev)
    xf = torch.empty(A * 96, dtype=torch.uint8, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    org = torch.from_numpy(np.ascontiguousarray(np.asarray(origins, np.float64).reshape(A, 2))).to(dev)
    Th = None if T is None else np.ascontiguousarray(np.asarray(T, np.float64).reshape(A, 16))
    rc = lib.mapmerge_extract_batch_write(d_ptrs.data_ptr(), A, w, h, float(res), org.data_ptr(),
                                          None if Th is None else Th.ctypes.data, use_h.ctypes.data, xf.data_ptr(),
                                          px.data_ptr(), py.data_ptr(), cap, total.data_ptr(), offs.data_ptr(),
                                          status.data_ptr(), ws.data_ptr(), nbytes, stream)
    assert rc == 0, _native.last_error()
    out = (totals, offs.cpu().numpy(), px.cpu().numpy(), py.cpu().numpy(), int(status.item()))
    del d_ptrs, ws
    return out


def check_batch(torch, lib, host_grid, ptrs, w, h, res, origins, T=None, use=None, bulk_ok=None):
    """Compare the batched extraction with NumPy.  host_grid(a) -> int8 [h, w] of agent a."""
    from oracle import merge_oracle as MO
    A = len(ptrs)
    origins = np.asarray(origins, np.float64).reshape(A, 2)
    totals, offs, px, py, status = batch_extract(torch, lib, ptrs, w, h, res, origins, T, use, bulk_ok)
    assert status == 0
    used = np.ones(A, bool) if use is None else np.asarray(use).astype(bool)
    want_tot = np.zeros(A, np.int64)
    for a in range(A):
        g = host_grid(a)
        x, y = MO.grid_to_points(g.ravel(), w, h, res, origins[a, 0], origins[a, 1])
        want_tot[a] = x.size
        assert totals[a] == x.size, (a, totals[a], x.size)
        if not used[a]:
            continue
        if T is not None and not np.array_equal(np.asarray(T[a]).reshape(4, 4), np.eye(4)):
            x, y = MO.transform_points(x, y, T[a])
        b = offs[a]
        assert np.array_equal(px[b:b + x.size], x) and np.array_equal(py[b:b + x.size], y), f'agent {a}'
    want_offs = np.concatenate([[0], np.cumsum(np.where(used, want_tot, 0))])
    assert np.array_equal(offs, want_offs)
    assert np.isnan(px[offs[A]:]).all() and np.isnan(py[offs[A]:]).all()    # nothing written past the slices
    return totals


def random_stack(A, h, w, seed):
    """int8 [A, h, w]: every int8 value, a per-agent occupancy between 0 and ~50 %, so chunk counts vary."""
    r = np.random.default_rng(seed)
    out = np.empty((A, h, w), np.int8)
    for a in range(A):
        v = r.integers(-128, 128, (h, w), dtype=np.int16).astype(np.int8)
        v[r.random((h, w)) < r.uniform(0.0, 1.0)] = -1
        out[a] = v
    if A > 2:
        out[A // 2] = -1                                      # one empty agent inside the batch
    return out


def device_stack(torch, stack, offset=0):
    """The stack copied to the device at `offset` bytes into one buffer -> (buffer, [grid addresses])."""
    A, h, w = stack.shape
    buf = torch.zeros(A * h * w + 64, dtype=torch.int8, device='cuda')
    buf[offset:offset + A * h * w] = torch.from_numpy(stack.reshape(-1)).cuda()
    return buf, [buf.data_ptr() + offset + a * h * w for a in range(A)]


def se2_stack(A, seed, span=50.0):
    from oracle import merge_oracle as MO
    r = np.random.default_rng(seed)
    return np.stack([MO.se2_matrix(*r.uniform(-span, span, 2), r.uniform(-math.pi, math.pi)) for _ in range(A)])


@gpu
def test_tma_ring_laps_1024_grids_of_256(torch, lib):
    """1 024 x 256^2 = 4 096 chunks: every CTA of the bulk-copy scan consumes >= 8 chunks, i.e. goes
    round its 4-stage ring twice (stage refills, both mbarrier parities, per-stage counters reused)."""
    A, h, w, res = 1024, 256, 256, 0.05
    assert (h * w) % 16 == 0
    assert A * math.ceil(h * w / CHUNK) >= ring_chunks_needed(torch)
    stack = random_stack(A, h, w, 1)
    buf, ptrs = device_stack(torch, stack)
    origins = np.tile([[-6.4, -6.4]], (A, 1))
    T = se2_stack(A, 2, span=5.0)
    T[0] = np.eye(4)
    check_batch(torch, lib, lambda a: stack[a], ptrs, w, h, res, origins, T)


@gpu
def test_tma_ring_laps_configs2_stack(torch, lib):
    """The configs[2] stack itself (bench_merge.device_grids, 256 x 2048^2 = 1 GiB, 65 536 chunks)."""
    from bench_merge import device_grids
    A, S, res = 256, 2048, 0.05
    assert A * math.ceil(S * S / CHUNK) >= ring_chunks_needed(torch)
    grids = device_grids(torch, torch.device('cuda', torch.cuda.current_device()), A, S)
    ptrs = [g.data_ptr() for g in grids]
    assert all(p % 16 == 0 for p in ptrs)
    origins = np.tile([[-S * res / 2, -S * res / 2]], (A, 1))
    T = se2_stack(A, 0)
    T[0] = np.eye(4)                                          # adopted untransformed, as merge() passes it
    totals = check_batch(torch, lib, lambda a: grids[a].cpu().numpy(), ptrs, S, S, res, origins, T)
    assert totals.min() > 0


@gpu
def test_tma_partial_last_chunk(torch, lib):
    """h*w % 16 == 0 but not a multiple of 16 384: the last bulk copy of every grid is short."""
    A, h, w, res = 64, 1000, 1008, 0.05
    assert (h * w) % 16 == 0 and (h * w) % CHUNK != 0
    assert A * math.ceil(h * w / CHUNK) >= ring_chunks_needed(torch)
    stack = random_stack(A, h, w, 3)
    buf, ptrs = device_stack(torch, stack)
    origins = np.tile([[-25.2, -25.0]], (A, 1))
    T = se2_stack(A, 4, span=10.0)
    check_batch(torch, lib, lambda a: stack[a], ptrs, w, h, res, origins, T)


@gpu
@pytest.mark.parametrize('A,h,w', [(4, 999, 1001), (40, 3, 5)])
def test_fallback_kernel_odd_sizes(torch, lib, A, h, w):
    """h*w % 16 != 0: k_batch_count, whatever the alignment of the grids."""
    assert (h * w) % 16 != 0
    stack = random_stack(A, h, w, 5 + h)
    buf, ptrs = device_stack(torch, stack)
    origins = np.tile([[-1.5, 2.5]], (A, 1))
    check_batch(torch, lib, lambda a: stack[a], ptrs, w, h, 0.05, origins, se2_stack(A, 6))


@gpu
@pytest.mark.parametrize('offset', [1, 8])
def test_fallback_kernel_unaligned_stack(torch, lib, offset):
    """16-byte-multiple grids whose base sits `offset` bytes into a buffer: bulk_ok = 0 as
    MapMerger._count_occupied decides it, and k_batch_count reads them byte-wise."""
    A, h, w = 50, 64, 96
    stack = random_stack(A, h, w, 7 + offset)
    buf, ptrs = device_stack(torch, stack, offset)
    assert not any(p % 16 == 0 for p in ptrs)
    origins = np.tile([[0.0, -3.0]], (A, 1))
    check_batch(torch, lib, lambda a: stack[a], ptrs, w, h, 0.1, origins, se2_stack(A, 8))


@gpu
@pytest.mark.parametrize('h,w', [(1, 1), (1, 17), (17, 1)])
def test_tiny_shapes(torch, lib, h, w):
    A = 33
    stack = random_stack(A, h, w, 9 + w)
    stack[0] = 100                                            # never empty everywhere
    buf, ptrs = device_stack(torch, stack)
    origins = np.random.default_rng(10).uniform(-5, 5, (A, 2))
    check_batch(torch, lib, lambda a: stack[a], ptrs, w, h, 0.05, origins, se2_stack(A, 11))


@gpu
def test_65535_grids_of_one_cell(torch, lib):
    """n_agents at its limit, which is also gridDim.y of k_batch_count and k_batch_write."""
    A = 65535
    cells = np.random.default_rng(12).integers(-128, 128, A, dtype=np.int16).astype(np.int8)
    buf = torch.from_numpy(cells).cuda()
    ptrs = [buf.data_ptr() + a for a in range(A)]
    origins = np.stack([np.arange(A) * 0.25, -np.arange(A) * 0.125], 1)
    use = np.random.default_rng(13).random(A) < 0.8
    totals = check_batch(torch, lib, lambda a: cells[a:a + 1].reshape(1, 1), ptrs, 1, 1, 0.05, origins, None, use)
    assert totals.sum() == (cells > 50).sum()


def value_domain_stack(A, seed):
    """int8 [A, 272, 256]: rows 0..255 hold (c + r) mod 256 - 128, so every int8 value sits at every
    byte of a 16-byte word and of a thread's 64-cell group; rows 256..271 are runs of 50 next to 51
    of every length 1..16.  Each agent permutes the rows."""
    base = np.empty((272, 256), np.int16)
    r_, c_ = np.mgrid[0:256, 0:256]
    base[:256] = (c_ + r_) % 256 - 128
    for k in range(16):
        base[256 + k] = np.where((np.arange(256) // (k + 1)) % 2 == 0, 50, 51)
    base = base.astype(np.int8)
    r = np.random.default_rng(seed)
    return np.stack([base] + [base[r.permutation(272)] for _ in range(A - 1)])


@gpu
@pytest.mark.parametrize('path', ['tma', 'vector', 'bytes'])
def test_value_domain_every_byte_lane(torch, lib, path):
    """The `> 50` test of occupied_bits16 (bulk-copy scan), of occupied_mask16's 16-byte loads
    (aligned grids, bulk_ok = 0) and of its byte loop (grids 1 byte into the buffer)."""
    A, h, w = 8, 272, 256
    stack = value_domain_stack(A, 14)
    for lane in range(64):                                    # every value at every byte of a thread's 64 cells
        assert np.unique(stack[0, :256, lane::64]).size == 256
    assert ((stack[:, :, :-1] == 50) & (stack[:, :, 1:] == 51)).any(axis=(1, 2)).all()
    buf, ptrs = device_stack(torch, stack, 1 if path == 'bytes' else 0)
    bulk_ok = {'tma': 1, 'vector': 0, 'bytes': 0}[path]
    origins = np.tile([[-6.4, -6.8]], (A, 1))
    check_batch(torch, lib, lambda a: stack[a], ptrs, w, h, 0.05, origins, se2_stack(A, 15, span=3.0), bulk_ok=bulk_ok)


@gpu
@pytest.mark.parametrize('h,w', [(160, 200), (161, 199)])
def test_use_flags_and_transforms(torch, lib, h, w):
    """Skipped and used agents mixed; the identity short-cut takes only exact identities (1 + 2^-52
    in m[0] is transformed); a 0.3-scaled rotation; a projective bottom row (w != 1 divides)."""
    from oracle import merge_oracle as MO
    A = 12
    stack = np.stack([synth_agent_grid(max(h, w), 600 + a)[:h, :w] for a in range(A)])
    buf, ptrs = device_stack(torch, stack)
    T = se2_stack(A, 16, span=4.0)
    T[0] = np.eye(4)
    T[1] = np.eye(4)
    T[1, 0, 0] = 1.0 + 2.0 ** -52
    T[2] = MO.se2_matrix(0.3, -0.2, 1.1)
    T[2, :2, :2] *= 0.3
    T[3, 3, 0], T[3, 3, 1] = 1e-3, -2e-3
    T[5] = np.eye(4)                                          # an identity on a skipped agent
    use = np.array([1, 1, 1, 1, 0, 0, 1, 0, 1, 1, 0, 1], np.uint8)
    origins = np.random.default_rng(17).uniform(-5, 5, (A, 2))
    check_batch(torch, lib, lambda a: stack[a], ptrs, w, h, 0.05, origins, T, use)
    # the near-identity really moves points: a tolerance in the identity test would be caught
    x, y = MO.grid_to_points(stack[1].ravel(), w, h, 0.05, *origins[1])
    assert not np.array_equal(MO.transform_points(x, y, T[1])[0], x)


# ---- B. MapMerger.merge against OracleMerger ------------------------------------------------------
class ChainSpy:
    """Forwards to the library and records (cursor, stalled) of every mapmerge_chain_poll."""

    def __init__(self, lib):
        self._lib = lib
        self.polls = []

    def __getattr__(self, name):
        f = getattr(self._lib, name)
        if name != 'mapmerge_chain_poll':
            return f

        def poll(ws, dims, n_agents, state, stream):
            rc = f(ws, dims, n_agents, state, stream)
            self.polls.append((int(state[0]), int(state[1])))
            return rc
        return poll


def spied_merger(MM):
    m = MM.MapMerger()
    m._lib = ChainSpy(m._lib)
    return m


def oracle_merge(o, grids, res, origins, tf, fit=None):
    """OracleMerger callbacks over the grids; -> the last published (grid, origin) or None."""
    want = None
    for a, g in enumerate(grids):
        h, w = g.shape
        out = o.map_callback(g.ravel(), w, h, res, origins[a][0], origins[a][1], tf[a],
                             accept=True if fit is None else fit[a] >= 0.6)
        want = out if out is not None else want
    return want


def assert_same(m, o, got, want):
    out, origin = got
    assert want is not None and out is not None
    assert out.shape == want[0].shape and np.array_equal(out, want[0]) and tuple(origin) == tuple(want[1])
    pc = m.global_pcd
    assert pc.shape[0] == o.gx.shape[0]
    assert np.array_equal(pc[:, 0], o.gx) and np.array_equal(pc[:, 1], o.gy)


def burst_case(MM):
    """200 grids of 96 x 128 under random SE(2).  Empty grids at 0, 64 and 128, fitness-rejected
    agents at 63, 65 and 127.  Agent 1 is adopted far from the rest, so the first 64 callbacks
    never move the min corner.  Agent 100 (translation -50 m) moves the anchor: a rebuild in the
    second burst.  Agent 150 repeats agent 100's grid, shifted by a fraction of a voxel, and
    re-averages the only point on the min corner inwards: a rebound in the third burst."""
    from oracle import merge_oracle as MO
    A, h, w, res = 200, 96, 128, 0.05
    r = np.random.default_rng(18)
    grids = [synth_agent_grid(w, 1000 + a)[:h] for a in range(A)]
    origins = np.tile([[-3.2, -2.4]], (A, 1))
    tf = np.stack([MO.se2_matrix(*r.uniform(-3, 3, 2), r.uniform(-math.pi, math.pi)) for _ in range(A)])
    fit = np.ones(A)
    for a in (0, 64, 128):
        grids[a] = np.full((h, w), -1, np.int8)
    for a in (63, 65, 127):
        fit[a] = 0.3
    origins[1] = (-40.0, -40.0)
    corner = grids[100].copy()
    corner[0, :] = -1
    corner[:, 0] = -1
    corner[0, 0] = 100                                        # the only point on the new min corner
    grids[100], grids[150] = corner, corner.copy()
    tf[100], tf[150] = np.eye(4), np.eye(4)
    tf[100, 0, 3], tf[100, 1, 3] = -50.0, -50.0              # below agent 1's corner at (-40, -40)
    tf[150, 0, 3], tf[150, 1, 3] = -50.0 + 0.004, -50.0 + 0.003
    return np.stack(grids), origins, res, tf, fit


def assert_bursts(m, spy):
    st = m.chain_stats
    n = st['callbacks']
    assert n > 2 * BURST and st['polls'] >= 4 and st['rebuilds'] >= 1 and st['rebounds'] >= 1, st
    polls = spy.polls
    assert len(polls) == st['polls']
    # a burst that ran through without finishing the order: the cursor was carried into the next call
    carried = [i for i, (cur, stall) in enumerate(polls) if stall == 0 and cur < n]
    assert carried, polls
    late = [(cur, stall) for cur, stall in polls[carried[0] + 1:]]
    assert any(stall == 1 and cur >= BURST for cur, stall in late), polls     # rebuild serviced after callback 64
    assert any(stall == 3 and cur >= BURST for cur, stall in late), polls     # rebound serviced after callback 64


@gpu
def test_merge_across_bursts(MM):
    from oracle import merge_oracle as MO
    grids, origins, res, tf, fit = burst_case(MM)
    assert grids.shape[1] != grids.shape[2] and (grids.shape[1] * grids.shape[2]) % 16 == 0
    o = MO.OracleMerger()
    want = oracle_merge(o, grids, res, origins, tf, fit)
    m = spied_merger(MM)
    assert_same(m, o, m.merge(grids, origins, res, tf.copy(), fitness=fit), want)
    assert_bursts(m, m._lib)


@gpu
def test_merge_continues_a_cloud_of_many_bursts(MM):
    """A second merge() on the same merger continues a cloud built by more than 64 callbacks, and
    itself runs more than 64 callbacks."""
    from oracle import merge_oracle as MO
    grids, origins, res, tf, fit = burst_case(MM)
    o = MO.OracleMerger()
    oracle_merge(o, grids, res, origins, tf, fit)
    m = spied_merger(MM)
    m.merge(grids, origins, res, tf.copy(), fitness=fit)
    assert m.chain_stats['callbacks'] > BURST
    A2 = 90
    g2 = np.stack([synth_agent_grid(128, 2000 + a)[:96] for a in range(A2)])
    g2[0] = -1
    o2 = np.tile([[-3.2, -2.4]], (A2, 1))
    tf2 = se2_stack(A2, 19, span=3.0)
    want = oracle_merge(o, g2, res, o2, tf2)
    m._lib.polls.clear()
    assert_same(m, o, m.merge(g2, o2, res, tf2), want)
    assert m.chain_stats['callbacks'] == A2 - 1 > BURST and m.chain_stats['polls'] >= 2


MIXED_SHAPES = [(96, 128), (128, 96), (100, 100), (77, 131), (64, 64), (1, 200), (150, 3), (33, 47), (128, 128), (90, 110)]


@gpu
@pytest.mark.parametrize('with_cloud', [False, True])
def test_merge_mixed_shapes(MM, with_cloud):
    """Grids of different shapes: merge() counts, extracts and filters agent by agent.  Without a
    cloud the first grid is empty, so the second is adopted; with one, every grid is transformed."""
    from oracle import merge_oracle as MO
    r = np.random.default_rng(20 + with_cloud)
    grids = []
    for k, (h, w) in enumerate(MIXED_SHAPES):
        g = synth_agent_grid(max(h, w), 3000 + k)[:h, :w].copy()
        g[r.random((h, w)) < 0.02] = 100
        grids.append(g)
    if not with_cloud:
        grids[0] = np.full(MIXED_SHAPES[0], -1, np.int8)
    A = len(grids)
    origins = r.uniform(-3, 3, (A, 2))
    tf = se2_stack(A, 21 + with_cloud, span=2.0)
    fit = np.ones(A)
    fit[4] = 0.5
    o, m = MO.OracleMerger(), MM.MapMerger()
    if with_cloud:
        pre = np.stack([synth_agent_grid(120, 3100 + a) for a in range(3)])
        pre_o = np.tile([[-3.0, -3.0]], (3, 1))
        pre_t = se2_stack(3, 23, span=2.0)
        oracle_merge(o, pre, 0.05, pre_o, pre_t)
        m.merge(pre, pre_o, 0.05, pre_t)
    want = oracle_merge(o, grids, 0.05, origins, tf, fit)
    assert_same(m, o, m.merge(grids, origins, 0.05, tf, fitness=fit), want)
    assert m.chain_stats is None                              # the per-agent branch ran


@gpu
@pytest.mark.parametrize('as_stack', [False, True])
def test_merge_unaligned_sizes(MM, torch, as_stack):
    """h*w % 16 != 0 through merge(): separately allocated device tensors are each 16-byte aligned,
    so only the size can send the scan to k_batch_count; a stack's slices are not aligned at all."""
    from oracle import merge_oracle as MO
    A, h, w = 20, 37, 53
    assert (h * w) % 16 != 0
    host = np.stack([synth_agent_grid(w, 4000 + a)[:h] for a in range(A)])
    if as_stack:
        grids = torch.from_numpy(host).cuda()
    else:
        grids = [torch.from_numpy(g.copy()).cuda() for g in host]
        assert all(g.data_ptr() % 16 == 0 for g in grids)
    origins = np.tile([[-1.3, -0.9]], (A, 1))
    tf = se2_stack(A, 24, span=1.0)
    o = MO.OracleMerger()
    want = oracle_merge(o, host, 0.05, origins, tf)
    m = MM.MapMerger()
    assert_same(m, o, m.merge(grids, origins, 0.05, tf), want)
    assert m.chain_stats['callbacks'] == A - 1


@gpu
def test_merge_bench_geometry(MM, torch):
    """bench_merge's workload (device_grids, 2048^2 at 5 cm, +-50 m, bench's transforms) through
    merge() against OracleMerger.  The oracle filters the whole growing cloud on every callback, so
    its cost grows with the square of the agent count: 1-2 s per callback once the cloud holds 3e6 to
    5e6 points, about 70-150 s for 130 agents depending on the host.  This case therefore runs 130
    agents rather than 256, the fewest that still give 3 bursts (129 callbacks).  The full 256-grid
    stack is checked in test_tma_ring_laps_configs2_stack."""
    from bench_merge import device_grids
    from oracle import merge_oracle as MO
    A, S, res = 130, 2048, 0.05
    dev = torch.device('cuda', torch.cuda.current_device())
    grids = device_grids(torch, dev, A, S)
    rng = np.random.default_rng(0)
    origins = np.tile(np.array([[-S * res / 2, -S * res / 2]]), (A, 1))
    tf = np.stack([MO.se2_matrix(*rng.uniform(-50, 50, 2), rng.uniform(-math.pi, math.pi)) for _ in range(A)])
    m = spied_merger(MM)
    got = m.merge(grids, origins, res, tf)
    st = m.chain_stats
    assert st['callbacks'] == A - 1 > 2 * BURST and st['polls'] >= 3, st
    o = MO.OracleMerger()
    want = oracle_merge(o, [g.cpu().numpy() for g in grids], res, origins, tf)
    assert_same(m, o, got, want)


@gpu
def test_merge_leaves_the_callers_transforms_alone(MM):
    """merge() on a fresh merger adopts the first non-empty cloud untransformed; it must not do so
    by writing the identity into the caller's [A, 4, 4] array, which the caller passes on to
    fuse_occupancy or register_maps.  The merged result still ignores that agent's transform."""
    from occgrid_b200.distributed import ShardedMapMerger
    from oracle import merge_oracle as MO
    A, n = 6, 96
    grids = np.stack([synth_agent_grid(n, 5000 + a) for a in range(A)])
    grids[0] = -1                                             # agent 1 is the first non-empty one
    origins = np.tile([[-2.4, -2.4]], (A, 1))
    tf = se2_stack(A, 25, span=2.0)
    assert tf.dtype == np.float64 and tf.flags.c_contiguous and not np.array_equal(tf[1], np.eye(4))
    keep = tf.copy()
    o = MO.OracleMerger()
    want = oracle_merge(o, grids, 0.05, origins, tf)
    m = MM.MapMerger()
    assert_same(m, o, m.merge(grids, origins, 0.05, tf), want)
    assert np.array_equal(tf, keep)
    out, origin = ShardedMapMerger().merge(grids, origins, 0.05, tf, A)
    assert np.array_equal(tf, keep)
    assert np.array_equal(out, want[0]) and tuple(origin) == tuple(want[1])


# ---- C. host-only argument checks -----------------------------------------------------------------
OK, E_ARG, E_WORKSPACE = 0, -1, -2
FAKE = 0x10000          # a 256-byte aligned address that is never dereferenced: every case fails a check first
NAN = float('nan')


def check(lib, rc, want, key):
    assert rc == want, (rc, lib.occgrid_last_error())
    assert key.encode() in lib.occgrid_last_error(), lib.occgrid_last_error()


def _batch_count(lib, **kw):
    a = dict(grids=FAKE, n_agents=4, w=64, h=32, total=FAKE, ws=FAKE, ws_bytes=1 << 40, bulk=1)
    a.update(kw)
    return lib.mapmerge_extract_batch_count(a['grids'], a['n_agents'], a['w'], a['h'], a['total'], a['ws'], a['ws_bytes'],
                                            a['bulk'], None)


def _batch_write(lib, **kw):
    a = dict(grids=FAKE, n_agents=4, w=64, h=32, res=0.05, origins=FAKE, xf=FAKE, px=FAKE, py=FAKE, total=FAKE,
             offs=FAKE, status=FAKE, ws=FAKE, ws_bytes=1 << 40)
    a.update(kw)
    return lib.mapmerge_extract_batch_write(a['grids'], a['n_agents'], a['w'], a['h'], a['res'], a['origins'], None, None,
                                            a['xf'], a['px'], a['py'], 1000, a['total'], a['offs'], a['status'], a['ws'],
                                            a['ws_bytes'], None)


BATCH_CASES = [
    (dict(grids=None), E_ARG, 'NULL pointer'),
    (dict(total=None), E_ARG, 'NULL pointer'),
    (dict(ws=None), E_ARG, 'NULL pointer'),
    (dict(n_agents=0), E_ARG, 'n_agents'),
    (dict(n_agents=65536), E_ARG, 'n_agents'),
    (dict(n_agents=-1), E_ARG, 'n_agents'),
    (dict(w=0), E_ARG, 'width x height'),
    (dict(h=0), E_ARG, 'width x height'),
    (dict(w=-5), E_ARG, 'width x height'),
]


@pytest.mark.parametrize('kw,want,key', BATCH_CASES)
def test_extract_batch_count_rejects(lib, kw, want, key):
    check(lib, _batch_count(lib, **kw), want, key)


@pytest.mark.parametrize('kw,want,key', BATCH_CASES + [
    (dict(origins=None), E_ARG, 'NULL pointer'),
    (dict(xf=None), E_ARG, 'NULL pointer'),
    (dict(px=None), E_ARG, 'NULL pointer'),
    (dict(offs=None), E_ARG, 'NULL pointer'),
    (dict(status=None), E_ARG, 'NULL pointer'),
    (dict(res=0.0), E_ARG, 'res'),
    (dict(res=-0.05), E_ARG, 'res'),
    (dict(res=NAN), E_ARG, 'res'),
])
def test_extract_batch_write_rejects(lib, kw, want, key):
    check(lib, _batch_write(lib, **kw), want, key)


@pytest.mark.parametrize('n_agents,w,h', [(1, 1, 1), (7, 999, 1001), (256, 2048, 2048), (65535, 1, 1)])
def test_extract_batch_workspace_one_byte_short(lib, n_agents, w, h):
    need = lib.mapmerge_extract_batch_workspace_bytes(w * h, n_agents)
    blocks = -(-w * h // CHUNK)
    assert need >= blocks * n_agents * (4 + 256 * 8)          # block counts + one bit per cell, 64 cells per thread
    check(lib, _batch_count(lib, n_agents=n_agents, w=w, h=h, ws_bytes=need - 1), E_WORKSPACE, 'workspace')
    check(lib, _batch_write(lib, n_agents=n_agents, w=w, h=h, ws_bytes=need - 1), E_WORKSPACE, 'workspace')


@pytest.mark.parametrize('args,key', [
    (dict(sx=None), 'NULL pointer'), (dict(offs=None), 'NULL pointer'), (dict(count=None), 'NULL pointer'),
    (dict(status=None), 'NULL pointer'), (dict(agent=-1), 'agent'),
])
def test_append_slice_rejects(lib, args, key):
    a = dict(sx=FAKE, offs=FAKE, agent=0, count=FAKE, status=FAKE)
    a.update(args)
    rc = lib.mapmerge_append_slice(a['sx'], FAKE, a['offs'], a['agent'], FAKE, FAKE, 100, a['count'], a['status'], None, None)
    check(lib, rc, E_ARG, key)


@pytest.mark.parametrize('grid,n,out,key', [(None, 10, FAKE, 'NULL pointer'), (FAKE, 10, None, 'NULL pointer'),
                                            (FAKE, -1, FAKE, 'n_cells')])
def test_count_occupied_rejects(lib, grid, n, out, key):
    check(lib, lib.mapmerge_count_occupied(grid, n, out, None), E_ARG, key)


def test_count_occupied_empty_is_a_no_op(lib):
    assert lib.mapmerge_count_occupied(FAKE, 0, FAKE, None) == OK


def _voxel(lib, **kw):
    a = dict(px=FAKE, count=FAKE, bounds=FAKE, benc=None, out=FAKE, status=FAKE, ws=FAKE, voxel=0.05, lat=1000, pts=1000,
             ws_bytes=1 << 40)
    a.update(kw)
    return lib.mapmerge_voxel_downsample(a['px'], FAKE, a['count'], a['pts'], a['voxel'], a['bounds'], a['benc'], a['lat'],
                                         a['out'], FAKE, FAKE, a['status'], a['ws'], a['ws_bytes'], None)


@pytest.mark.parametrize('kw,want,key', [
    (dict(px=None), E_ARG, 'NULL pointer'), (dict(bounds=None), E_ARG, 'NULL pointer'),
    (dict(out=None), E_ARG, 'NULL pointer'), (dict(ws=None), E_ARG, 'NULL pointer'),
    (dict(voxel=0.0), E_ARG, 'voxel'), (dict(voxel=-0.05), E_ARG, 'voxel'), (dict(voxel=NAN), E_ARG, 'voxel'),
    (dict(lat=0), E_ARG, 'capacity'), (dict(pts=0), E_ARG, 'capacity'),
])
def test_voxel_downsample_rejects(lib, kw, want, key):
    check(lib, _voxel(lib, **kw), want, key)


@pytest.mark.parametrize('lat,pts', [(1, 1), (1000, 1000), (5000 * 5000, 3_000_000)])
def test_voxel_workspace_one_byte_short(lib, lat, pts):
    need = lib.mapmerge_voxel_workspace_bytes(lat, pts)
    check(lib, _voxel(lib, lat=lat, pts=pts, ws_bytes=need - 1), E_WORKSPACE, 'workspace')
    check(lib, _voxel(lib, lat=lat, pts=pts, bounds=None, benc=FAKE, ws_bytes=need - 1), E_WORKSPACE, 'workspace')


@pytest.mark.parametrize('kw,want,key', [
    (dict(px=None), E_ARG, 'NULL pointer'), (dict(count=None), E_ARG, 'NULL pointer'),
    (dict(bounds=None), E_ARG, 'NULL pointer'), (dict(ws=None), E_ARG, 'NULL pointer'),
    (dict(short=True), E_WORKSPACE, 'workspace'),
])
def test_bounds_rejects(lib, kw, want, key):
    a = dict(px=FAKE, count=FAKE, bounds=FAKE, ws=FAKE, short=False)
    a.update(kw)
    nbytes = lib.mapmerge_bounds_workspace_bytes() - (1 if a['short'] else 0)
    check(lib, lib.mapmerge_bounds(a['px'], FAKE, a['count'], a['bounds'], a['ws'], nbytes, None), want, key)


@pytest.mark.parametrize('kw,key', [
    (dict(px=None), 'NULL pointer'), (dict(bounds=None), 'NULL pointer'), (dict(out=None), 'NULL pointer'),
    (dict(w=0), 'width x height'), (dict(h=0), 'width x height'), (dict(w=-3), 'width x height'),
    (dict(res=0.0), 'res'), (dict(res=-1.0), 'res'), (dict(res=NAN), 'res'),
])
def test_rasterise_rejects(lib, kw, key):
    a = dict(px=FAKE, bounds=FAKE, out=FAKE, w=10, h=10, res=0.05)
    a.update(kw)
    check(lib, lib.mapmerge_rasterise(a['px'], FAKE, FAKE, a['res'], a['bounds'], a['w'], a['h'], a['out'], None), E_ARG, key)


@pytest.mark.parametrize('dst,src,n,key', [(None, FAKE, 10, 'NULL pointer'), (FAKE, None, 10, 'NULL pointer'),
                                           (FAKE, FAKE, -1, 'n ')])
def test_fuse_max_rejects(lib, dst, src, n, key):
    check(lib, lib.mapmerge_fuse_max(dst, src, n, None), E_ARG, key)


def test_fuse_max_empty_is_a_no_op(lib):
    assert lib.mapmerge_fuse_max(FAKE, FAKE, 0, None) == OK


# chain: dims = {lattice_w, lattice_h, point_capacity, slice_capacity}
DIMS = (500, 400, 100_000, 20_000)
CHAIN_DIMS_CASES = [
    (dict(n_agents=0), 'n_agents'), (dict(n_agents=65536), 'n_agents'),
    (dict(dims=(0, 400, 100_000, 20_000)), 'dims'), (dict(dims=(500, -1, 100_000, 20_000)), 'dims'),
    (dict(dims=(500, 400, 0, 20_000)), 'dims'), (dict(dims=(500, 400, 100_000, 0)), 'dims'),
    (dict(dims=(1 << 16, 1 << 16, 100_000, 20_000)), 'dims'), (dict(dims=None), 'NULL pointer'),
]


def _dims(d):
    return None if d is None else np.ascontiguousarray(np.asarray(d, np.int64))


def _chain_init(lib, **kw):
    a = dict(chain=FAKE, dims=DIMS, n_agents=8, sx=FAKE, offs=FAKE, order=[1, 2, 3], n_order=None, px=FAKE, count=FAKE,
             chain_bytes=1 << 40)
    a.update(kw)
    d = _dims(a['dims'])
    order = None if a['order'] is None else np.ascontiguousarray(np.asarray(a['order'], np.int32))
    n_order = len(a['order'] or []) if a['n_order'] is None else a['n_order']
    return lib.mapmerge_chain_init(a['chain'], a['chain_bytes'], None if d is None else d.ctypes.data, a['n_agents'], a['sx'],
                                   FAKE, a['offs'], None if order is None else order.ctypes.data, n_order, a['px'], FAKE,
                                   a['count'], None)


@pytest.mark.parametrize('kw,want,key', [(kw, E_ARG, k) for kw, k in CHAIN_DIMS_CASES] + [
    (dict(chain=None), E_ARG, 'NULL pointer'), (dict(sx=None), E_ARG, 'NULL pointer'), (dict(offs=None), E_ARG, 'NULL pointer'),
    (dict(order=None), E_ARG, 'NULL pointer'), (dict(px=None), E_ARG, 'NULL pointer'), (dict(count=None), E_ARG, 'NULL pointer'),
    (dict(n_order=-1), E_ARG, 'n_order'), (dict(n_order=9, order=list(range(9))), E_ARG, 'n_order'),
    (dict(order=[1, 8]), E_ARG, 'order entry'), (dict(order=[-1]), E_ARG, 'order entry'),
])
def test_chain_init_rejects(lib, kw, want, key):
    check(lib, _chain_init(lib, **kw), want, key)


@pytest.mark.parametrize('dims,n_agents', [(DIMS, 8), ((1, 1, 1, 1), 1), ((4000, 4000, 5_000_000, 70_000), 65535)])
def test_chain_workspace_one_byte_short(lib, dims, n_agents):
    d = _dims(dims)
    need = lib.mapmerge_chain_workspace_bytes(d.ctypes.data, n_agents)
    assert need > 0
    check(lib, _chain_init(lib, dims=dims, n_agents=n_agents, order=[0], chain_bytes=need - 1), E_WORKSPACE, 'workspace')


def test_chain_workspace_bytes_rejects_what_init_rejects(lib):
    for kw, _ in CHAIN_DIMS_CASES:
        d = _dims(kw.get('dims', DIMS))
        assert lib.mapmerge_chain_workspace_bytes(None if d is None else d.ctypes.data, kw.get('n_agents', 8)) == 0, kw


def _chain_run(lib, **kw):
    a = dict(chain=FAKE, dims=DIMS, n_agents=8, n_order=3, n_cb=2, sx=FAKE, offs=FAKE, voxel=0.05, px=FAKE, cap=100_000,
             count=FAKE, status=FAKE)
    a.update(kw)
    d = _dims(a['dims'])
    return lib.mapmerge_chain_run(a['chain'], None if d is None else d.ctypes.data, a['n_agents'], a['n_order'], a['n_cb'],
                                  a['sx'], FAKE, a['offs'], a['voxel'], a['px'], FAKE, a['cap'], a['count'], a['status'], None)


@pytest.mark.parametrize('kw,key', CHAIN_DIMS_CASES + [
    (dict(chain=None), 'NULL pointer'), (dict(sx=None), 'NULL pointer'), (dict(offs=None), 'NULL pointer'),
    (dict(px=None), 'NULL pointer'), (dict(count=None), 'NULL pointer'), (dict(status=None), 'NULL pointer'),
    (dict(n_order=-1), 'n_order'), (dict(n_order=9), 'n_order'), (dict(n_cb=-1), 'n_callbacks'),
    (dict(voxel=0.0), 'voxel'), (dict(voxel=NAN), 'voxel'), (dict(cap=100_001), 'capacity'),
])
def test_chain_run_rejects(lib, kw, key):
    check(lib, _chain_run(lib, **kw), E_ARG, key)


@pytest.mark.parametrize('kw,key', CHAIN_DIMS_CASES + [(dict(chain=None), 'NULL pointer'), (dict(state=False), 'NULL pointer')])
def test_chain_poll_rejects(lib, kw, key):
    a = dict(chain=FAKE, dims=DIMS, n_agents=8, state=True)
    a.update(kw)
    d = _dims(a['dims'])
    state = (C.c_int32 * 2)()
    rc = lib.mapmerge_chain_poll(a['chain'], None if d is None else d.ctypes.data, a['n_agents'], state if a['state'] else None,
                                 None)
    check(lib, rc, E_ARG, key)


@pytest.mark.parametrize('kw,key', CHAIN_DIMS_CASES + [(dict(chain=None), 'NULL pointer'), (dict(px=None), 'NULL pointer'),
                                                       (dict(count=None), 'NULL pointer')])
def test_chain_rebounds_rejects(lib, kw, key):
    a = dict(chain=FAKE, dims=DIMS, n_agents=8, px=FAKE, count=FAKE)
    a.update(kw)
    d = _dims(a['dims'])
    rc = lib.mapmerge_chain_rebounds(a['chain'], None if d is None else d.ctypes.data, a['n_agents'], a['px'], FAKE, a['count'],
                                     None)
    check(lib, rc, E_ARG, key)


def _chain_rebuild(lib, **kw):
    a = dict(chain=FAKE, dims=DIMS, n_agents=8, sx=FAKE, offs=FAKE, agent=2, voxel=0.05, px=FAKE, cap=100_000, count=FAKE,
             out=FAKE, status=FAKE, vws=FAKE, vws_bytes=1 << 40, lat=DIMS[0] * DIMS[1])
    a.update(kw)
    d = _dims(a['dims'])
    return lib.mapmerge_chain_rebuild(a['chain'], None if d is None else d.ctypes.data, a['n_agents'], a['sx'], FAKE, a['offs'],
                                      a['agent'], a['voxel'], a['px'], FAKE, a['cap'], a['count'], a['out'], FAKE, FAKE,
                                      a['status'], a['vws'], a['vws_bytes'], a['lat'], None)


@pytest.mark.parametrize('kw,want,key', [(kw, E_ARG, k) for kw, k in CHAIN_DIMS_CASES] + [
    (dict(chain=None), E_ARG, 'NULL pointer'), (dict(sx=None), E_ARG, 'NULL pointer'), (dict(out=None), E_ARG, 'NULL pointer'),
    (dict(status=None), E_ARG, 'NULL pointer'), (dict(agent=-1), E_ARG, 'agent'), (dict(agent=8), E_ARG, 'agent'),
    (dict(voxel=-0.05), E_ARG, 'voxel'), (dict(voxel=NAN), E_ARG, 'voxel'), (dict(cap=100_001), E_ARG, 'capacity'),
    (dict(vws=None), E_WORKSPACE, 'workspace'), (dict(lat=DIMS[0] * DIMS[1] - 1), E_WORKSPACE, 'workspace'),
])
def test_chain_rebuild_rejects(lib, kw, want, key):
    check(lib, _chain_rebuild(lib, **kw), want, key)


def test_chain_rebuild_voxel_workspace_one_byte_short(lib):
    lat = DIMS[0] * DIMS[1]
    need = lib.mapmerge_voxel_workspace_bytes(lat, DIMS[2])
    check(lib, _chain_rebuild(lib, vws_bytes=need - 1), E_WORKSPACE, 'workspace')
