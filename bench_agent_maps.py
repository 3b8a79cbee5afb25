#!/usr/bin/env python
"""bench_agent_maps.py — per-agent maps: one packet batch into 64 agent grids on the device, then
MapMerger fuses them into the global map (packets -> agent maps -> global map on one GPU).

Workload = BASELINE configs[1]: generate_session(64 agents, 2.5e6 packets), every agent mapped in
its own odometry frame (zero offsets) onto 256^2 maps at 5 cm with origin (-4.0, -6.4): the room
(simulation_tools.ROOM_X / ROOM_Y) plus the 1.2 m sensor reach, so no beam is clipped.  As in
bench.py, a pool of 4 seeded batches (seeds 42..45) is cycled so that packet reads come from HBM.

    python bench_agent_maps.py [--steps 200] [--warmup 5] [--rounds 3]

Before timing, a 1e5-packet prefix is checked bit for bit against the oracle (per agent, the C
oracle's single-grid call over that agent's records); a mismatch exits with status 3.  Then:
  agent_maps     ms per occgrid_integrate_packets_agent_maps call (device events, --steps calls),
                 beam-cell updates/s from the device counters
  shared         the same batches into bench.py's shared 4096^2 map with the room offsets, timed in
                 the same process, alternated with agent_maps for --rounds rounds
  kernels        per-kernel device time of both (occgrid_profile_begin/end, a separate pass)
  merge          MapMerger.merge of the 64 maps; transforms = room offsets relative to agent 1's
                 frame (the first map is adopted as is, map_merger.py:40-43)
  end_to_end     packets -> published global map, from device-resident and from host packets
Prints ONE JSON line, with the GPU's name, power limit and SM clock read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import numpy as np

N_AGENTS = 64
N_PACKETS = 2_500_000
POOL = 4
MAP = dict(size=256, resolution=0.05, origin_x=-4.0, origin_y=-6.4)
ORACLE_SLOTS = ('packets', 'accepted', 'dropped', 'bad_pose', 'beams', 'hits', 'updates')


def gpu_details(torch, dev):
    out = {'name': torch.cuda.get_device_name(dev)}
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    try:
        r = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-i', str(dev.index)],
                           capture_output=True, text=True, timeout=20)
        f = [x.strip() for x in r.stdout.strip().split(',')]
        out.update(power_limit_w=float(f[1]), sm_mhz=int(f[2]), sm_max_mhz=int(f[3]))
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        out['nvidia_smi'] = 'unavailable'
    return out


def parity(M, sess, n_prefix):
    """Prefix of the first batch: the device stack vs the per-agent oracle, and the device counters
    vs the oracle's and the single-grid call's."""
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from agent_maps_util import integrate_packets_agent_maps
    pk = sess['packets'][:n_prefix]
    z = np.zeros((N_AGENTS + 1, 2))
    out = {}
    want = np.full((N_AGENTS, MAP['size'], MAP['size']), -1, np.int8)
    c = integrate_packets_agent_maps(pk, want, MAP['origin_x'], MAP['origin_y'], MAP['resolution'], agent_offsets=z)
    for strategy in ('tiled', 'global_atomic'):
        maps = M.AgentGrids(N_AGENTS, strategy=strategy, max_batch=n_prefix, **MAP)
        maps.update_packets(pk, agent_offsets=z)
        shared = M.OccupancyGrid(strategy=strategy, max_batch=n_prefix, **MAP)
        shared.update_packets(pk, agent_offsets=z)
        k = maps.counters()
        ok = np.array_equal(maps.grids, want) and k == shared.counters() and all(k[s] == c[s] for s in ORACLE_SLOTS)
        out[strategy] = 'bit-exact' if ok else 'MISMATCH'
    return out


def time_steps(torch, step, k):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(k):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k


def kernel_ms(torch, _native, step, k=5):
    torch.cuda.synchronize()
    _native.profile_begin()
    for i in range(k):
        step(i)
    torch.cuda.synchronize()
    return {name: round(v[0] / k, 4) for name, v in _native.profile_end().items()}


def wall_ms(torch, fn, repeat):
    ts = []
    for _ in range(repeat):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return sorted(ts)[len(ts) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--parity-packets', type=int, default=100_000)
    ap.add_argument('--repeat', type=int, default=3, help='merge / end-to-end repetitions (median)')
    args = ap.parse_args()
    if args.steps < 1 or args.rounds < 1:
        ap.error('--steps and --rounds must be at least 1')

    import torch
    from occgrid_b200 import _native, simulation_tools as st
    from occgrid_b200 import dual_bot_mapper as M
    from occgrid_b200.map_merger import MapMerger
    if not torch.cuda.is_available():
        raise SystemExit('bench_agent_maps.py needs a CUDA device (no CPU fallback)')
    dev = torch.device('cuda', torch.cuda.current_device())
    result = {'metric': 'agent_maps_step_ms', 'workload': f'{N_AGENTS} agents, {N_PACKETS} packets, own frames, '
              f'{MAP["size"]}^2 maps at {MAP["resolution"]} m', 'gpu': gpu_details(torch, dev)}

    sessions = [st.generate_session(n_agents=N_AGENTS, n_packets=N_PACKETS, seed=42 + i) for i in range(POOL)]
    s0 = sessions[0]
    result['parity'] = parity(M, s0, args.parity_packets)
    if any(v != 'bit-exact' for v in result['parity'].values()):
        result['error'] = 'agent maps differ from the oracle'
        print(json.dumps(result))
        raise SystemExit(3)
    result['parity_line'] = 'parity: bit-exact'

    lib = _native.lib()
    stream = torch.cuda.current_stream().cuda_stream
    maps = M.AgentGrids(N_AGENTS, max_batch=N_PACKETS, device=dev, **MAP)
    shared = M.OccupancyGrid(max_batch=N_PACKETS, device=dev, **s0['grid'])
    dpk = [maps.stage_packets(s['packets'])[0] for s in sessions]
    zoff = torch.zeros((N_AGENTS + 1, 2), dtype=torch.float64, device=dev)
    room_off = torch.from_numpy(s0['agent_offsets']).to(dev)

    def step_maps(i):
        pk = dpk[i % POOL]
        rc = lib.occgrid_integrate_packets_agent_maps(maps._geom, pk.data_ptr(), pk.shape[0], 42, 42, None, None,
                                                      zoff.data_ptr(), N_AGENTS, maps.grids_tensor.data_ptr(),
                                                      maps._ws.data_ptr(), maps._ws.numel(), maps._counters.data_ptr(),
                                                      maps._strategy, stream)
        if rc != 0:
            raise RuntimeError(_native.last_error())

    def step_shared(i):        # bench.py's single-GPU step
        pk = dpk[i % POOL]
        rc = lib.occgrid_integrate_packets(shared._geom, pk.data_ptr(), pk.shape[0], 42, 42, None, None,
                                           room_off.data_ptr(), N_AGENTS, shared.grid_tensor.data_ptr(),
                                           shared._ws.data_ptr(), shared._ws.numel(), shared._counters.data_ptr(),
                                           shared._strategy, stream)
        if rc != 0:
            raise RuntimeError(_native.last_error())

    for i in range(max(args.warmup, POOL)):
        step_maps(i)
        step_shared(i)
    rounds = {'agent_maps': [], 'shared': []}
    upd = {}
    for r in range(args.rounds):
        for name, step, grid in (('agent_maps', step_maps, maps), ('shared', step_shared, shared)):
            torch.cuda.synchronize()
            grid._counters.zero_()
            rounds[name].append(time_steps(torch, step, args.steps))
            upd[name] = grid.counters(reset=True)
    ms_maps, ms_shared = min(rounds['agent_maps']), min(rounds['shared'])
    result['agent_maps'] = {'ms_per_step': round(ms_maps, 4), 'ms_rounds': [round(x, 4) for x in rounds['agent_maps']],
                            'beam_cell_updates_per_s': upd['agent_maps']['updates'] / args.steps / (ms_maps * 1e-3),
                            'counters_per_step': {k: v // args.steps for k, v in upd['agent_maps'].items() if v}}
    result['shared'] = {'ms_per_step': round(ms_shared, 4), 'ms_rounds': [round(x, 4) for x in rounds['shared']],
                        'beam_cell_updates_per_s': upd['shared']['updates'] / args.steps / (ms_shared * 1e-3)}
    result['ratio_agent_maps_over_shared'] = round(ms_maps / ms_shared, 4)
    km, ks = kernel_ms(torch, _native, step_maps), kernel_ms(torch, _native, step_shared)
    result['kernels_ms'] = {'agent_maps': km, 'shared': ks}
    diff = {k: round(km.get(k, 0.0) - ks.get(k, 0.0), 4) for k in set(km) | set(ks)}
    result['kernel_ms_difference'] = dict(sorted(diff.items(), key=lambda kv: -kv[1]))

    # merge: the 64 device maps as they are (stack of contiguous [H, W] views, no copy)
    rel = s0['agent_offsets'][1:] - s0['agent_offsets'][1]
    tf = np.concatenate([rel, np.zeros((N_AGENTS, 1))], axis=1)                 # (tx, ty, theta)
    merged = {}

    def merge():
        merged['out'] = MapMerger(device=dev).merge(maps.grids_tensor, maps.origins, maps.res, tf)

    merge()                                                                         # warm-up
    result['merge'] = {'ms': round(wall_ms(torch, merge, args.repeat), 3), 'global_map_shape': list(merged['out'][0].shape),
                       'occupied_cells': int((merged['out'][0] == 100).sum())}

    def e2e_device():
        maps.clear()
        step_maps(0)
        merge()

    host_pk = s0['packets']

    def e2e_host():
        maps.clear()
        maps.update_packets(host_pk, agent_offsets=zoff)
        merge()

    e2e_device()
    e2e_host()
    result['end_to_end_ms'] = {'device_packets': round(wall_ms(torch, e2e_device, args.repeat), 3),
                               'host_packets': round(wall_ms(torch, e2e_host, args.repeat), 3)}
    result['gpu_after'] = gpu_details(torch, dev)
    print(result['parity_line'], file=sys.stderr)
    print(json.dumps(result))


if __name__ == '__main__':
    main()
