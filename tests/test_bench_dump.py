"""bench.py --dump-outputs: what it writes, the size bound, and (on the GPU) that the dumped grid
and counters are those of the last timed step — the C oracle replays the same seeded batch sequence."""
import json
import os
import subprocess
import sys

import bench
import numpy as np
import pytest

from conftest import ROOT


def test_dump_rows_are_fixed_and_the_dump_fits_the_limit(tmp_path):
    rows = bench.dump_rows(4096)
    assert np.array_equal(rows, bench.dump_rows(4096))
    assert len(np.unique(rows)) == 2048 and np.all(np.diff(rows) > 0) and rows[-1] < 4096
    from occgrid_b200 import _native
    grid = np.random.default_rng(1).choice(np.array([-1, 0, 100], np.int8), (4096, 4096))
    counters = {k: 10 ** 10 + i for i, k in enumerate(_native.COUNTER_NAMES)}
    bench.dump_outputs(str(tmp_path / 'out'), grid[rows], rows, counters)
    files = sorted(os.listdir(tmp_path / 'out'))
    assert files == ['counters.npy', 'grid.npy', 'grid_rows.npy']
    assert sum(os.path.getsize(tmp_path / 'out' / f) for f in files) <= 64_000_000
    g, r, c = (np.load(tmp_path / 'out' / f) for f in ('grid.npy', 'grid_rows.npy', 'counters.npy'))
    assert g.dtype == np.float32 and np.array_equal(g, grid[rows])
    assert r.dtype == np.float64 and np.array_equal(r, rows)
    assert c.dtype == np.float64 and c.tolist() == [float(counters[k]) for k in _native.COUNTER_NAMES]


@pytest.mark.parametrize('extra', [['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'unused']])
def test_bench_rejects_bad_arguments(extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra, capture_output=True, text=True)
    assert r.returncode == 2, r.stderr


@pytest.mark.gpu
def test_dump_is_the_grid_and_counters_of_the_last_timed_step(tmp_path):
    torch = pytest.importorskip('torch')
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from occgrid_b200 import simulation_tools as st
    from oracle import c_oracle
    npk, warmup, steps = 20_000, 3, 3
    out = tmp_path / 'dump'
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', str(steps),
                        '--warmup', str(warmup), '--packets', str(npk), '--no-cpu', '--no-merge',
                        '--dump-outputs', str(out)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])['steps'] == steps
    # bench.py's sequence: warm-up steps 0 .. max(W, POOL) - 1, then timed steps W .. W + K - 1,
    # step i integrating batch i % POOL; every batch uses the first session's agent offsets
    sess = [st.generate_session(n_agents=bench.AGENTS_PER_GPU, n_packets=npk, seed=42 + i) for i in range(bench.POOL)]
    gk, offs = sess[0]['grid'], sess[0]['agent_offsets']
    want = np.full((gk['size'], gk['size']), -1, np.int8)
    seq = list(range(max(warmup, bench.POOL))) + list(range(warmup, warmup + steps))
    for i in seq:
        last = c_oracle.integrate_packets(sess[i % bench.POOL]['packets'], want, gk['origin_x'], gk['origin_y'],
                                          gk['resolution'], agent_offsets=offs)
    rows = np.load(out / 'grid_rows.npy').astype(np.int64)
    assert np.array_equal(rows, bench.dump_rows(gk['size']))
    assert np.array_equal(np.load(out / 'grid.npy'), want[rows].astype(np.float32))
    from occgrid_b200 import _native
    got = dict(zip(_native.COUNTER_NAMES, np.load(out / 'counters.npy').tolist()))
    assert last['packets'] == npk
    assert {k: got[k] for k in ('packets', 'beams', 'updates')} == {k: float(last[k]) for k in ('packets', 'beams', 'updates')}
