#!/usr/bin/env python
"""bench.py — throughput of the occupancy-grid integration hot path.

A "step" = one pass of the hot path over one batch of synthetic QuasarPackets:
decode -> pose correction -> 4 beams -> Bresenham -> last-writer-wins scatter into the int8
grid (reference: server_nodes/dual_bot_mapper.py:826-903, 136-179).

Workload (N=1) = BASELINE.json configs[1]: 64 synthetic agents, 4096^2 grid at 5 cm,
1e7 beams (2.5e6 packets) per batch.  At N>1 (weak scaling) the map grows to (4096*N)^2 cut
into N row bands (one per GPU), the swarm to 64*N agents, and every rank ingests its own
1e7-beam share of the stream, routes the records to the band owners (NCCL all-to-all) and
integrates what it receives.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = beam-cell updates/s with the packets resident in
HBM; `e2e` = the same metric through OccupancyGrid.update_packets() with HOST buffers (pinned
H2D copy of the batch and D2H read of the step's counters inside the timed region);
`roofline` = algorithmic bytes of the integrate kernel over its measured duration vs the
measured HBM peak, `scatter_roofline` = updates/s vs a same-run microkernel doing nothing but
random atomicMax(u32) on a same-size plane (SURVEY §8d); `cpu_baseline` = the reference's
algorithm (oracle port) timed on this box's host cores on a bounded sample.

`--dump-outputs DIR` (single GPU) also writes what the last timed step computed as .npy files under
DIR (see dump_outputs()).  The inputs are seeded, so two builds run with the same arguments can
be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

METRIC = 'beam_cell_updates_per_sec'
UNIT = 'updates/s'
PACKETS_PER_BATCH = 2_500_000          # 1e7 beams
AGENTS_PER_GPU = 64
GRID_PER_GPU = 4096
RESOLUTION = 0.05
POOL = 4                               # distinct batches cycled so packet reads come from HBM


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '25',
                 '-i', str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(',')]
            if len(f) < 8:
                continue
            try:
                smax = float(f[2])
                if t0 - 0.05 <= ts <= t1 + 0.15:
                    sm.append(float(f[1]))
                    for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[4:8]):
                        if v.lower().startswith('active'):
                            reasons.add(name)
            except ValueError:
                continue
        if not sm:   # region shorter than one sample: take the nearest rows
            for ts, line in self.rows[-3:]:
                f = [x.strip() for x in line.split(',')]
                try:
                    sm.append(float(f[1]))
                except (ValueError, IndexError):
                    pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': smax,
                'reasons': sorted(reasons), 'samples': len(sm)}


# ----------------------------------------------------------------------------------------------
#  CPU baseline (oracle port of the reference) — test infrastructure used only as the baseline
# ----------------------------------------------------------------------------------------------

def _cpu_worker(args):
    """One host core: the reference's algorithm (Python restatement of
    dual_bot_mapper.py:826-903 + OccupancyGrid.update_ray) on a private grid."""
    packets, offsets, grid_kw = args
    from oracle import occgrid_oracle as O
    g = O.OracleGrid(**grid_kw)
    offs = {a: (float(offsets[a, 0]), float(offsets[a, 1])) for a in range(1, offsets.shape[0])}
    t0 = time.perf_counter()
    _, st = O.replay([p.tobytes() for p in packets], grid=g, agent_offsets=offs)
    return st['updates'], st['beams'], time.perf_counter() - t0


def cpu_baseline(sess, cores, packets_per_core):
    """Bounded sample of the same workload on `cores` host processes (disjoint packet slices,
    private grids: an upper bound on what the host could do, SURVEY §8d / BASELINE.md §3)."""
    import multiprocessing as mp
    kw = dict(size=sess['grid']['size'], resolution=sess['grid']['resolution'],
              origin_x=sess['grid']['origin_x'], origin_y=sess['grid']['origin_y'])
    jobs = [(sess['packets'][i * packets_per_core:(i + 1) * packets_per_core], sess['agent_offsets'], kw)
            for i in range(cores)]
    t0 = time.perf_counter()
    if cores == 1:
        res = [_cpu_worker(jobs[0])]
    else:
        with mp.get_context('fork').Pool(cores) as pool:
            res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    upd = sum(r[0] for r in res)
    beams = sum(r[1] for r in res)
    busy = max(r[2] for r in res)
    return {'value': upd / busy, 'unit': UNIT, 'cores': cores, 'kind': 'port',
            'sample': f'{beams} beams ({packets_per_core} packets x {cores} core(s)) of the same synthetic batch, '
                      f'Python restatement of the reference loop (oracle/occgrid_oracle.py), {wall:.1f} s wall',
            'updates': upd, 'seconds': busy}


def c_port_rate(sess, n_packets=250_000):
    from oracle import c_oracle
    g = np.full((sess['grid']['size'],) * 2, -1, np.int8)
    t0 = time.perf_counter()
    c = c_oracle.integrate_packets(sess['packets'][:n_packets], g, sess['grid']['origin_x'], sess['grid']['origin_y'],
                                   sess['grid']['resolution'], agent_offsets=sess['agent_offsets'])
    dt = time.perf_counter() - t0
    return {'value': c['updates'] / dt, 'unit': UNIT, 'cores': 1, 'kind': 'port (C restatement, oracle/occgrid_oracle.c)',
            'sample': f'{c["beams"]} beams'}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (it is pure Python and
    single-threaded; its restatement runs on all host cores over disjoint slices)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from occgrid_b200 import simulation_tools as st
    cores = os.cpu_count() or 1
    per_core = 12_000                       # ~1e6 beam-cell updates per core per step (~1 s)
    sess = st.generate_session(n_agents=AGENTS_PER_GPU, n_packets=max(per_core * cores, 1), seed=42)
    for _ in range(min(args.warmup, 1)):
        cpu_baseline(sess, cores, per_core // 4)
    vals, secs = [], 0.0
    for _ in range(args.steps):
        r = cpu_baseline(sess, cores, per_core)
        vals.append(r['value'])
        secs += r['seconds']
    v = float(np.mean(vals))
    r['value'] = v
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': secs / max(args.steps, 1) * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64+int', 'data': 'synthetic',
        'config': workload_config(1), 'cpu_baseline': r,
        'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


def workload_config(n, grid_per_gpu=GRID_PER_GPU, agents_per_gpu=AGENTS_PER_GPU):
    side = grid_per_gpu * n
    if n == 1:
        what = 'BASELINE.json configs[1]'
    elif side == 65536 and agents_per_gpu * n == 1024:
        what = 'BASELINE.json configs[3]: 1024 agents, 65536^2 grid spatially tiled across 8 GPUs'
    else:
        what = f'the per-GPU band of BASELINE.json configs[3] ({grid_per_gpu} x {side} cells, {agents_per_gpu} agents per GPU) on {n} row bands'
    return {'workload': f'{agents_per_gpu * n} synthetic agents, {side}^2 grid at 5 cm, 1e7 beams/batch per GPU ({what})',
            'packets_per_batch_per_gpu': PACKETS_PER_BATCH, 'grid': f'{side}x{side} int8',
            'l2': f'{POOL} distinct 105 MB packet batches cycled (420 MB > 126 MB L2); grid/stamp hot set is '
                  'L2-resident by nature of the workload'}


DUMP_LIMIT_BYTES = 64_000_000


def dump_rows(height):
    """Fixed, seeded sample of grid rows for --dump-outputs: half of them, ascending.  The whole
    4096^2 grid in float32 (67 MB) would exceed DUMP_LIMIT_BYTES."""
    return np.sort(np.random.default_rng(0).choice(height, height // 2, replace=False))


def dump_outputs(out_dir, grid_sample, rows, counters):
    """Writes what the timed path handed its caller after the last timed step:
      grid.npy       float32 [len(rows), W]: those rows of the int8 occupancy grid (-1 / 0 / 100)
      grid_rows.npy  float64 [len(rows)]: the row indices of grid.npy (dump_rows())
      counters.npy   float64 [len(COUNTER_NAMES)]: the device counters of the last timed step (what
                     counters(reset=True) returns after it), in the order of _native.COUNTER_NAMES"""
    from occgrid_b200 import _native
    arrays = {'grid': np.asarray(grid_sample, np.float32), 'grid_rows': np.asarray(rows, np.float64),
              'counters': np.array([counters[k] for k in _native.COUNTER_NAMES], np.float64)}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f'--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit')
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f'{name}.npy'), a)


# ----------------------------------------------------------------------------------------------
#  GPU arm
# ----------------------------------------------------------------------------------------------

def multi_gpu_parity(torch, dist, dev, world, rank, exchange):
    """Before timing at N > 1: the same exchange path on a small seeded stream (1024 rows per GPU,
    16 agents per GPU, 3 batches of 40k packets per rank so both receive slots are reused), map
    all-gathered and compared on rank 0 with the C oracle over the canonical stream — the checker
    use of oracle/ (never timed).  -> {'map': 'bit-exact' | 'DIFFERS', ...} on every rank."""
    from occgrid_b200 import simulation_tools as st
    from occgrid_b200.distributed import TiledSwarmMap
    size = 1024 * world
    origin = (-size * 0.05 / 2,) * 2
    n_batches, per_rank = 3, 40_000
    sess = st.generate_session(n_agents=16 * world, n_packets=n_batches * per_rank * world, grid_size=size, origin=origin, seed=77)
    pk, idx, offs = sess['packets'], sess['agent_idx'], sess['agent_offsets']
    tmap = TiledSwarmMap(size, 0.05, origin[0], origin[1], device=dev, max_batch=per_rank, exchange=exchange)
    order = []
    for b in range(n_batches):
        base = b * per_rank * world
        sl = slice(base + rank * per_rank, base + (rank + 1) * per_rank)
        tmap.update_packets(pk[sl], agent_offsets=offs, agent_idx=idx[sl])
        order.append(np.arange(base, base + per_rank * world))          # canonical: rank 0's share, rank 1's, ...
    got = tmap.gather_grid()
    cn = tmap.counters()
    owned = torch.tensor([cn['owned_updates']], device=dev, dtype=torch.int64)
    dist.all_reduce(owned)
    flag = torch.zeros(1, device=dev, dtype=torch.int64)
    info = {}
    if rank == 0:
        from oracle import c_oracle
        o = np.concatenate(order)
        want = np.full((size, size), -1, np.int8)
        c = c_oracle.integrate_packets(pk[o], want, origin[0], origin[1], 0.05, agent_offsets=offs, agent_idx=idx[o])
        same = bool(np.array_equal(got, want)) and int(owned.item()) == c['updates']
        flag[0] = 1 if same else 0
        info = {'beams': int(c['beams']), 'known_cells': int((want != -1).sum()), 'grid': f'{size}x{size}',
                'checker': 'oracle/occgrid_oracle.c over the canonical stream'}
    dist.broadcast(flag, 0)
    del tmap
    torch.cuda.empty_cache()
    return dict(info, map='bit-exact' if int(flag.item()) == 1 else 'DIFFERS', exchange=exchange, ranks=world)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=500,
                    help='timed steps (default 500: ~0.17 s on one GPU, long enough for several clock samples)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--strategy', default='auto')
    ap.add_argument('--packets', type=int, default=PACKETS_PER_BATCH)
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-merge', action='store_true', help='skip the merged-grids/s leg (BASELINE configs[2])')
    ap.add_argument('--trace', action='store_true', help='print per-step wall times (debug)')
    ap.add_argument('--grid-per-gpu', type=int, default=0,
                    help='N>1: map side = this x N.  Default 8192 (with 128 agents per GPU: N=8 is BASELINE configs[3], '
                         '65536^2 / 1024 agents; N=2 and 4 keep the same per-GPU band)')
    ap.add_argument('--agents-per-gpu', type=int, default=0)
    ap.add_argument('--layout', default='bands', choices=['bands', 'lattice'],
                    help='N>1: rooms per band equal (bands, default) or one square lattice over the map (lattice: uneven bands)')
    ap.add_argument('--no-parity', action='store_true', help='N>1: skip the bit-exactness check against the oracle before timing')
    ap.add_argument('--raycast-ctas', type=int, default=0, help='cap persistent raycast CTAs per SM (0 = max)')
    ap.add_argument('--ingest', default='uniform', choices=['uniform', 'affine'],
                    help='N>1: which agents a rank receives (uniform = all agents, the worst case; affine = the agents of its band)')
    ap.add_argument('--exchange', default='p2p', choices=['p2p', 'nccl'],
                    help='N>1: routed records via peer-memory stores from the routing kernel (p2p) or NCCL all-to-all')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='single GPU: write the grid and counters of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    if args.impl == 'reference':
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from occgrid_b200 import _native, simulation_tools as st
    from occgrid_b200 import dual_bot_mapper as M

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback)')
    if args.dump_outputs and world > 1:
        raise SystemExit('--dump-outputs: single-GPU runs only')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        if os.environ.get('NCCL_DEBUG', '').upper() in ('', 'VERSION'):
            os.environ['NCCL_DEBUG'] = 'WARN'        # NCCL's version banner goes to stdout; this script prints ONE JSON line
        dist.init_process_group('nccl', device_id=dev)
    n = world
    if args.grid_per_gpu <= 0:
        args.grid_per_gpu = GRID_PER_GPU if n == 1 else 8192
    if args.agents_per_gpu <= 0:
        args.agents_per_gpu = AGENTS_PER_GPU if n == 1 else 128
    W = max(args.warmup, 3)
    K = args.steps
    npk = args.packets
    lib = _native.lib()
    lib.occgrid_set_raycast_ctas_per_sm(args.raycast_ctas)

    if n == 1:
        from occgrid_b200.dual_bot_mapper import OccupancyGrid
        sessions = [st.generate_session(n_agents=AGENTS_PER_GPU, n_packets=npk, seed=42 + i) for i in range(POOL)]
        s0 = sessions[0]
        grid = OccupancyGrid(strategy=args.strategy, max_batch=npk, device=dev, **s0['grid'])
        off = torch.from_numpy(s0['agent_offsets']).to(dev)
        dpk = [grid.stage_packets(s['packets'])[0] for s in sessions]
        stream = torch.cuda.current_stream().cuda_stream

        def step(i):
            pk = dpk[i % POOL]
            rc = lib.occgrid_integrate_packets(grid._geom, pk.data_ptr(), pk.shape[0], 42, 42, None, None,
                                               off.data_ptr(), AGENTS_PER_GPU, grid.grid_tensor.data_ptr(),
                                               grid._ws.data_ptr(), grid._ws.numel(), grid._counters.data_ptr(),
                                               grid._strategy, stream)
            if rc != 0:
                raise RuntimeError(_native.last_error())

    else:
        from occgrid_b200.distributed import TiledSwarmMap, make_rank_sessions
        parity = None
        if not args.no_parity:
            parity = multi_gpu_parity(torch, dist, dev, n, rank, args.exchange)
            if parity['map'] != 'bit-exact':
                if rank == 0:
                    print(json.dumps({'metric': METRIC, 'n_gpus': n, 'parity': parity, 'error': 'multi-GPU map differs from the oracle'}))
                dist.destroy_process_group()
                raise SystemExit(3)
        tmap, sessions, step = make_rank_sessions(n, rank, dev, npk, POOL, args.strategy,
                                                   grid_per_gpu=args.grid_per_gpu, agents_per_gpu=args.agents_per_gpu,
                                                   exchange=args.exchange, ingest=args.ingest, layout=args.layout)
        grid = tmap.local

    # warm-up (at least one pass over every batch of the pool, so that no allocation or
    # connection set-up is left for the timed region)
    for i in range(max(W, POOL)):
        step(i)
    if args.trace:
        for i in range(2 * POOL):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            step(i)
            torch.cuda.synchronize()
            if rank == 0:
                print(f'trace step {i}: {(time.perf_counter() - t0) * 1e3:.3f} ms', file=sys.stderr, flush=True)
    if n > 1:
        tmap.flush()
    torch.cuda.synchronize()
    grid._counters.zero_()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    if world > 1:
        dist.barrier()          # nobody enters the timed region before rank 0's sampler is up
    counters_before_last = torch.empty_like(grid._counters) if args.dump_outputs else None
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    ev0.record()
    t_host0 = time.perf_counter()
    for i in range(K):
        if counters_before_last is not None and i == K - 1:
            counters_before_last.copy_(grid._counters)     # on the stream: no host synchronisation
        step(W + i)
    host_ms_per_step = (time.perf_counter() - t_host0) * 1e3 / max(K, 1)      # enqueue cost: must stay well below ms_per_step
    if n > 1:
        tmap.flush()            # the last batch is integrated inside the timed region
    ev1.record()
    torch.cuda.synchronize()
    t_wall1 = time.time()
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    if args.dump_outputs:
        # taken before the profiling loop below integrates more batches into the same grid
        rows = dump_rows(grid.grid_tensor.shape[0])
        grid_sample = grid.grid_tensor[torch.from_numpy(rows).to(dev)].cpu().numpy()
        last_counters = dict(zip(_native.COUNTER_NAMES, (grid._counters - counters_before_last).cpu().tolist()))
    counters = grid.counters(reset=True)
    upd_key = 'updates' if n == 1 else 'owned_updates'
    updates = counters[upd_key]
    if world > 1:
        t = torch.tensor([updates], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        updates = int(t.item())
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    value = updates / (ms * 1e-3)

    # per-kernel device time (library hook: CUDA events around each launch, on its stream), from
    # a short extra loop outside the timed region; the dominant kernel feeds `roofline`
    P = 5
    if n > 1:
        tmap.flush()
    torch.cuda.synchronize()
    _native.profile_begin()
    for i in range(P):
        step(i)
    if n > 1:
        tmap.flush()
    torch.cuda.synchronize()
    prof = _native.profile_end()
    # prof[name] = (summed device ms, kernels launched); every scope runs once per step here
    kernels = {k: {'ms_per_launch': v[0] / P, 'launches_per_step': v[1] / P} for k, v in prof.items()}
    launches_per_step = sum(v[1] for v in prof.values()) / P
    dom = max(prof, key=lambda k: prof[k][0])
    dom_ms = prof[dom][0] / P
    dom_launches = 1.0
    hbm_peak, peak_src = measured_peaks()
    packets_total = npk * K * n
    upd_per_step_rank = updates / K / n
    # algorithmic bytes, charged to the kernel that moves them: the count pass reads the 42-byte wire
    # records; the raycast kernel reads one 48-byte pose record + one 4-byte bin index per packet and
    # produces one 1-byte cell value per beam-cell update (SURVEY §8d's per-unit figures)
    recs_per_step = float(counters.get('records', 0)) / max(K, 1) or float(npk)
    bytes_by_kernel = {'tile_count': 42.0 * npk, 'tile_raycast': 52.0 * recs_per_step + 1.0 * upd_per_step_rank,
                       'integrate_global': 42.0 * npk + 1.0 * upd_per_step_rank}
    alg_bytes = bytes_by_kernel.get(dom, 42.0 * npk + 1.0 * upd_per_step_rank) / dom_launches
    step_bytes = 42.0 * npk + 1.0 * upd_per_step_rank
    roof = {'bound': 'hbm', 'kernel': dom, 'achieved': alg_bytes / (dom_ms * 1e-3) / 1e9, 'peak': hbm_peak,
            'unit': 'GB/s', 'frac': alg_bytes / (dom_ms * 1e-3) / 1e9 / hbm_peak, 'traffic': ncu_traffic(),
            'ms_per_launch': dom_ms, 'share_of_step': prof[dom][0] / sum(v[0] for v in prof.values()),
            'peak_source': peak_src,
            'step': {'achieved': step_bytes / (ms / K * 1e-3) / 1e9, 'frac': step_bytes / (ms / K * 1e-3) / 1e9 / hbm_peak,
                     'bytes': '42 B/packet + 1 B/beam-cell update over the whole step (SURVEY §8d)'},
            'note': 'algorithmic bytes of the dominant kernel = 52 B per pose record (48-byte record + 4-byte bin index) + 1 B per '
                    'beam-cell update; by construction a small fraction of HBM: the binding resource is shared-memory '
                    'atomic throughput and instruction issue, see scatter_roofline_smem'}

    result = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': n, 'steps': K, 'warmup': W,
        'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f64+u32', 'data': 'synthetic',
        'config': workload_config(n, args.grid_per_gpu, args.agents_per_gpu) if n > 1 else workload_config(1),
        'beams_per_sec': 4.0 * packets_total / (ms * 1e-3),
        'strategy': args.strategy, 'host_enqueue_ms_per_step': host_ms_per_step,
    }
    if n > 1:
        result['exchange'] = tmap.exchange
        result['ingest'] = args.ingest
        result['layout'] = args.layout
        result['parity'] = parity

    # ---- single-GPU extras: scatter roofline, e2e, cpu baseline ------------------------------
    if n == 1:
        stream = torch.cuda.current_stream().cuda_stream
        cells = GRID_PER_GPU * GRID_PER_GPU
        plane = torch.zeros(cells, dtype=torch.int32, device=dev)
        nops = 1 << 28
        for _ in range(2):
            lib.occgrid_scatter_probe(0, plane.data_ptr(), cells, nops, 7, stream)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        for _ in range(5):
            lib.occgrid_scatter_probe(0, plane.data_ptr(), cells, nops, 9, stream)
        p1.record()
        torch.cuda.synchronize()
        probe_rate = 5 * nops / (p0.elapsed_time(p1) * 1e-3)
        del plane
        result['scatter_roofline'] = {'bound': 'l2-atomic', 'achieved': value, 'peak': probe_rate, 'unit': UNIT,
                                      'frac': value / probe_rate,
                                      'how': 'peak = same-run microkernel: 2^28 atomicMax(u32) per launch to uniformly '
                                             'random cells of a 4096^2 u32 plane (occgrid_scatter_probe kind 0): the ceiling '
                                             'of the GLOBAL_ATOMIC strategy; the default TILED strategy resolves the order '
                                             'stamps in shared memory and is bounded by scatter_roofline_smem instead'}
        # the ceiling of what the TILED strategy actually does: atomicMax on a window-sized tile in shared memory
        win_words = 116 * 117                       # (64 + 2R) x pitch words at 5 cm (occgrid_tiled.cu: tile_geom)
        probe_out = torch.zeros(1 << 16, dtype=torch.int32, device=dev)
        nops_s = 148 * 3 * 256 * 4096               # three 256-thread CTAs per SM, 4096 random atomics per thread
        for _ in range(2):
            lib.occgrid_scatter_probe(6, probe_out.data_ptr(), win_words, nops_s, 7, stream)
        p0.record()
        for _ in range(5):
            lib.occgrid_scatter_probe(6, probe_out.data_ptr(), win_words, nops_s, 9, stream)
        p1.record()
        torch.cuda.synchronize()
        smem_rate = 5 * nops_s / (p0.elapsed_time(p1) * 1e-3)
        atomics_per_update = 1.0                    # one shared-memory reduction per beam-cell update (minus skipped start cells)
        result['scatter_roofline_smem'] = {
            'bound': 'smem-atomic', 'achieved': value, 'peak': smem_rate, 'unit': UNIT, 'frac': value / smem_rate,
            'frac_raycast_kernel': (updates / K) / (kernels['tile_raycast']['ms_per_launch'] * 1e-3) / smem_rate,
            'how': 'peak = same-run microkernel: 444 CTAs x 256 threads x 4096 atomicMax(u32) to uniformly random words of a '
                   '116x117-word tile in shared memory (occgrid_scatter_probe kind 6; the stamp window of the TILED strategy), '
                   'nothing else in the loop; frac = whole step vs that rate, frac_raycast_kernel = the raycast kernel alone'}
        # e2e: the user's call — OccupancyGrid.update_packets(host buffer) + counters read-back
        host = [torch.from_numpy(s['packets']).pin_memory() for s in sessions]
        g2 = M.OccupancyGrid(strategy=args.strategy, max_batch=npk, device=dev, **s0['grid'])
        offs_np = s0['agent_offsets']
        for i in range(2):
            g2.update_packets(host[i % POOL], agent_offsets=offs_np)
            g2.counters()
        torch.cuda.synchronize()
        g2.counters(reset=True)
        Ke = max(3, min(K, 10))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e_upd = 0
        e0.record()
        for i in range(Ke):
            g2.update_packets(host[i % POOL], agent_offsets=offs_np)
            e_upd += g2.counters(reset=True)['updates']        # D2H of the step's result
        e1.record()
        torch.cuda.synchronize()
        e_ms = e0.elapsed_time(e1)
        # the same call with the consumers' read of `.grid` every step (the reference's renderer reads it every
        # frame, :512): 16 MiB more D2H per step
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r_upd = 0
        r0.record()
        for i in range(Ke):
            g2.update_packets(host[i % POOL], agent_offsets=offs_np)
            r_upd += g2.counters(reset=True)['updates']
            _ = g2.grid
        r1.record()
        torch.cuda.synchronize()
        r_ms = r0.elapsed_time(r1)
        result['e2e'] = {'value': e_upd / (e_ms * 1e-3), 'unit': UNIT,
                         'with_grid_readback': {'value': r_upd / (r_ms * 1e-3), 'unit': UNIT, 'ms_per_step': r_ms / Ke,
                                                'd2h_bytes_per_step': int(_native.N_COUNTERS * 8 + g2.grid_tensor.numel())},
                         'h2d_bytes_per_step': int(host[0].numel() + offs_np.nbytes),
                         'd2h_bytes_per_step': int(_native.N_COUNTERS * 8), 'steps': Ke,
                         'ms_per_step': e_ms / Ke,
                         'api': 'OccupancyGrid.update_packets(pinned host uint8[n,42]) + counters() read-back'}
        # extension: hit/miss count planes (occgrid_accumulate_packets) over the same resident batches
        counts = grid.counts_tensor
        grid._counters.zero_()

        def count_step(i):
            pk = dpk[i % POOL]
            rc = lib.occgrid_accumulate_packets(grid._geom, pk.data_ptr(), pk.shape[0], 42, 42, None, None,
                                                off.data_ptr(), AGENTS_PER_GPU, counts.data_ptr(), grid._ws.data_ptr(),
                                                grid._ws.numel(), grid._counters.data_ptr(), grid._strategy, stream)
            if rc != 0:
                raise RuntimeError(_native.last_error())

        for i in range(POOL):
            count_step(i)
        torch.cuda.synchronize()
        grid._counters.zero_()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for i in range(K):
            count_step(i)
        c1.record()
        torch.cuda.synchronize()
        c_ms = c0.elapsed_time(c1)
        result['count_mode'] = {'value': grid.counters(reset=True)['updates'] / (c_ms * 1e-3), 'unit': UNIT, 'ms_per_step': c_ms / K,
                                'what': 'extension: int32 hit/miss planes (atomic adds) instead of the last-writer-wins int8 grid'}
        if not args.no_cpu:
            result['cpu_baseline'] = cpu_baseline(s0, 1, 500_000)     # ~10 s of the reference's Python loop on one core
            result['cpu_baseline_c_port'] = c_port_rate(s0)
        # workload sensitivity: the same packets with every pose moved to a random place of the map (few
        # packets per tile, nothing re-scanned): both strategies, a short run each
        sens = {}
        dsess = [st.disperse_poses(s, seed=7 + i) for i, s in enumerate(sessions[:2])]
        dd = [grid.stage_packets(s['packets'])[0] for s in dsess]
        for sname in ('tiled', 'global_atomic'):
            gs_ = M.OccupancyGrid(strategy=sname, max_batch=npk, device=dev, **s0['grid'])

            def sstep(i):
                pk = dd[i % 2]
                rc = lib.occgrid_integrate_packets(gs_._geom, pk.data_ptr(), pk.shape[0], 42, 42, None, None, off.data_ptr(),
                                                   AGENTS_PER_GPU, gs_.grid_tensor.data_ptr(), gs_._ws.data_ptr(), gs_._ws.numel(),
                                                   gs_._counters.data_ptr(), gs_._strategy, stream)
                if rc != 0:
                    raise RuntimeError(_native.last_error())
            for i in range(3):
                sstep(i)
            torch.cuda.synchronize()
            gs_._counters.zero_()
            s0e, s1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0e.record()
            for i in range(6):
                sstep(i)
            s1e.record()
            torch.cuda.synchronize()
            s_ms = s0e.elapsed_time(s1e)
            sens[sname] = {'value': gs_.counters()['updates'] / (s_ms * 1e-3), 'unit': UNIT, 'ms_per_step': s_ms / 6}
            del gs_
        result['sensitivity'] = dict(sens, workload='dispersed poses: the configs[1] packets with every pose uniformly random over the '
                                                      '4096^2 map (no tile or cell locality); the headline workload re-scans 32 rooms')
        del dd
        if not args.no_merge:
            # second half of BASELINE.json's metric: merged grids/s on configs[2]
            del dpk, g2, host
            torch.cuda.empty_cache()
            import bench_merge
            result['merge'] = bench_merge.run_merge_bench(torch, dev, cpu_agents=0 if args.no_cpu else 8)
    if n > 1:
        # e2e at N GPUs: every rank hands ITS share to TiledSwarmMap.update_packets as a pinned host
        # buffer (H2D + route + exchange + integrate) and reads the step's counters back
        host = [s['packets'].cpu().pin_memory() for s in sessions]
        for i in range(2):
            s = sessions[i % POOL]
            tmap.update_packets(host[i % POOL], agent_offsets=s['agent_offsets'], agent_idx=s['agent_idx'])
        tmap.flush()
        torch.cuda.synchronize()
        grid.counters(reset=True)
        dist.barrier()
        Ke = max(3, min(K, 10))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(Ke):
            s = sessions[i % POOL]
            tmap.update_packets(host[i % POOL], agent_offsets=s['agent_offsets'], agent_idx=s['agent_idx'])
            grid.counters()                                   # D2H of the counters as they stand (the step itself is asynchronous)
        tmap.flush()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e_ms = float(t.item())
        u = torch.tensor([grid.counters(reset=True)['owned_updates']], device=dev, dtype=torch.int64)
        dist.all_reduce(u)
        result['e2e'] = {'value': int(u.item()) / (e_ms * 1e-3), 'unit': UNIT,
                         'h2d_bytes_per_step': int(host[0].numel()) * n, 'd2h_bytes_per_step': int(_native.N_COUNTERS * 8) * n,
                         'steps': Ke, 'ms_per_step': e_ms / Ke,
                         'api': 'TiledSwarmMap.update_packets(pinned host uint8[n,42] share per rank) + counters() read-back'}
    if n > 1 and not args.no_merge:
        # second half of BASELINE.json's metric at N GPUs (needs the integration buffers gone first)
        del tmap, sessions, host, step
        grid = None
        torch.cuda.empty_cache()
        import bench_merge
        result['merge'] = bench_merge.run_sharded_merge_bench(torch, dist, dev, n, rank)
    result['roofline'] = roof
    result['clocks'] = clocks
    result['kernels'] = kernels
    result['gpu_launches'] = int(round(launches_per_step * K))
    if rank == 0:
        print(json.dumps(result))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, grid_sample, rows, last_counters)     # after every timed leg: file I/O disturbs none
    if world > 1:
        dist.destroy_process_group()


def ncu_traffic():
    """dram bytes (read+write) per integrate launch from the committed ncu capture, if any."""
    p = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if os.path.exists(p):
        try:
            with open(p) as f:
                return json.load(f).get('dram_bytes_per_launch')
        except (ValueError, OSError):
            return None
    return None


if __name__ == '__main__':
    main()
