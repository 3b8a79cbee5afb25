#!/usr/bin/env python
"""bench_map_fuse.py — fused occupancy map: agent maps resampled into one global grid that keeps free
space (MapMerger.fuse_occupancy / mapmerge_warp_fuse), on the device.

Workloads:
  (a) swarm   BASELINE configs[1] (64 agents, 2.5e6 packets, seed 42) integrated by AgentGrids into
              64 maps of 256^2 at 5 cm in their own frames (bench_agent_maps.py), fused into the shared
              4096^2 map geometry with the room offsets as transforms.  Also timed: frontier_centroids
              on the fused map, and packets (device-resident) -> agent maps -> fused map -> centroids.
  (b) merge   BASELINE configs[2] as in bench_merge.py: 256 maps of 2048^2 from device_grids,
              theta ~ U(-pi, pi), t ~ U(-50, 50)^2, seed 0, fused at 5 cm into the square target that
              covers every transformed map corner.  The same maps are also fused at twice and half
              the resolution: the target cells (and so the cell evaluations) change by 4x while the
              stack is still read, which shows whether the kernel follows bytes or evaluations.

    python bench_map_fuse.py [--steps 50] [--warmup 3] [--repeat 5]

Before timing, all of (a) and 8 agents of (b) are compared with the NumPy reference
(tests/map_fuse_util.py) bit for bit; a mismatch exits with status 3.  Reported per workload:
ms per call from device events (warmed), the byte bound (stack read once + target written once over
the HBM peak the project uses: MEASURED_PEAKS.json, else 6650 GB/s), the achieved fraction of it, and
the kernel time from occgrid_profile_begin/end.  Prints ONE JSON line, with the GPU's name, power
limit and SM clock read in the same run.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np

SWARM_MAP = dict(size=256, resolution=0.05, origin_x=-4.0, origin_y=-6.4)
TILE = 64


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


def hbm_peak_gbs():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def event_ms(torch, fn, k):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(k):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k


def kernel_ms(torch, _native, fn, k):
    torch.cuda.synchronize()
    _native.profile_begin()
    for _ in range(k):
        fn()
    torch.cuda.synchronize()
    prof = _native.profile_end()
    return round(prof['merge_warp_fuse'][0] / k, 4), prof['merge_warp_fuse'][1] // k


def wall_ms(torch, fn, repeat):
    ts = []
    for _ in range(repeat):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return sorted(ts)[len(ts) // 2]


def agent_tile_pairs(T, origins, res, hw, gox, goy, g, n):
    """Agent-tile pairs the kernel walks (corner footprint + 2 cells, the host rule of map_fuse.cu):
    x 4096 = cell evaluations.  Arithmetic from the inputs, not a measurement."""
    h, w = hw
    pairs = 0
    for a in range(len(T)):
        x0, y0 = origins[a]
        cx = np.array([x0, x0 + w * res, x0, x0 + w * res])
        cy = np.array([y0, y0, y0 + h * res, y0 + h * res])
        gx = (T[a][0, 0] * cx + T[a][0, 1] * cy + T[a][0, 3] - gox) / g - 0.5
        gy = (T[a][1, 0] * cx + T[a][1, 1] * cy + T[a][1, 3] - goy) / g - 0.5
        j0, j1 = max(math.floor(gx.min()) - 2, 0), min(math.ceil(gx.max()) + 2, n - 1)
        i0, i1 = max(math.floor(gy.min()) - 2, 0), min(math.ceil(gy.max()) + 2, n - 1)
        if j0 <= j1 and i0 <= i1:
            pairs += (j1 // TILE - j0 // TILE + 1) * (i1 // TILE - i0 // TILE + 1)
    return pairs


def measure(torch, _native, fn, stack_bytes, target_cells, hbm, args, pairs=None):
    for _ in range(args.warmup):
        fn()
    ms = min(event_ms(torch, fn, args.steps) for _ in range(3))
    kms, launches = kernel_ms(torch, _native, fn, max(args.steps // 5, 3))
    nbytes = stack_bytes + target_cells
    bound_ms = nbytes / (hbm * 1e9) * 1e3
    out = {'ms_per_call': round(ms, 4), 'kernel_ms': kms, 'kernel_launches_per_call': launches,
           'bytes': nbytes, 'byte_bound_ms': round(bound_ms, 4), 'fraction_of_byte_bound': round(bound_ms / ms, 4),
           'kernel_fraction_of_byte_bound': round(bound_ms / kms, 4)}
    if pairs is not None:
        out['agent_tile_pairs'] = pairs
        out['cell_evaluations_per_s'] = pairs * TILE * TILE / (kms * 1e-3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--repeat', type=int, default=5, help='end-to-end and centroid repetitions (median)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')

    import torch
    from occgrid_b200 import _native, simulation_tools as st
    from occgrid_b200 import dual_bot_mapper as M
    from occgrid_b200.map_merger import MapMerger, se2_matrix
    from map_fuse_util import warp_fuse
    from bench_merge import device_grids
    if not torch.cuda.is_available():
        raise SystemExit('bench_map_fuse.py needs a CUDA device (no CPU fallback)')
    dev = torch.device('cuda', torch.cuda.current_device())
    hbm, hbm_src = hbm_peak_gbs()
    result = {'metric': 'map_fuse_ms', 'gpu': gpu_details(torch, dev), 'hbm_peak_gbs': hbm, 'hbm_peak_source': hbm_src,
              'parity': {}}
    merger = MapMerger(device=dev)
    lib = _native.lib()
    stream = torch.cuda.current_stream().cuda_stream

    # ---- (a) swarm: packets -> 64 agent maps -> shared 4096^2 map --------------------------------
    s = st.generate_session(n_agents=64, n_packets=2_500_000, seed=42)
    maps = M.AgentGrids(64, max_batch=2_500_000, device=dev, **SWARM_MAP)
    dpk = maps.stage_packets(s['packets'])[0]
    zoff = torch.zeros((65, 2), dtype=torch.float64, device=dev)
    maps.update_packets(dpk, agent_offsets=zoff)
    tf_a = np.stack([se2_matrix(x, y, 0.0) for x, y in s['agent_offsets'][1:]])
    G = s['grid']
    target = M.OccupancyGrid(G['size'], G['resolution'], G['origin_x'], G['origin_y'], device=dev)
    merger.fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, tf_a, target)
    want = warp_fuse(maps.grids, maps.origins, maps.res, tf_a, G['origin_x'], G['origin_y'], G['resolution'], G['size'], G['size'])
    result['parity']['swarm'] = 'bit-exact' if np.array_equal(target.grid, want) else 'MISMATCH'

    def fuse_a():
        merger.fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, tf_a, target)

    pairs_a = agent_tile_pairs(tf_a, maps.origins, maps.res, (256, 256), G['origin_x'], G['origin_y'], G['resolution'], G['size'])
    swarm = measure(torch, _native, fuse_a, maps.grids_tensor.numel(), G['size'] ** 2, hbm, args, pairs_a)
    swarm['workload'] = '64 maps of 256^2 (configs[1], own frames) -> 4096^2 at 0.05 m, room offsets'
    swarm['working_set_fits_l2'] = True
    cent = target.frontier_centroids()
    swarm['centroids'] = len(cent)
    swarm['frontier_centroids_ms'] = round(wall_ms(torch, target.frontier_centroids, args.repeat), 3)

    def e2e():
        maps.clear()
        rc = lib.occgrid_integrate_packets_agent_maps(maps._geom, dpk.data_ptr(), dpk.shape[0], 42, 42, None, None,
                                                      zoff.data_ptr(), 64, maps.grids_tensor.data_ptr(), maps._ws.data_ptr(),
                                                      maps._ws.numel(), maps._counters.data_ptr(), maps._strategy, stream)
        if rc != 0:
            raise RuntimeError(_native.last_error())
        fuse_a()
        target.frontier_centroids()

    e2e()
    swarm['end_to_end_ms'] = round(wall_ms(torch, e2e, args.repeat), 3)
    swarm['end_to_end'] = 'device packets -> agent maps -> fused map -> frontier centroids (host list)'
    result['swarm'] = swarm
    del target

    # ---- (b) merge: 256 x 2048^2, random SE(2) ----------------------------------------------------
    A, S, res = 256, 2048, 0.05
    stack = torch.stack(device_grids(torch, dev, A, S))
    torch.cuda.empty_cache()
    rng = np.random.default_rng(0)
    origins = np.tile(np.array([[-S * res / 2, -S * res / 2]]), (A, 1))
    tf_b = np.stack([se2_matrix(*rng.uniform(-50, 50, 2), rng.uniform(-math.pi, math.pi)) for _ in range(A)])
    c = np.array([[0, 0], [S, 0], [0, S], [S, S]], np.float64) * res + origins[0]
    px = tf_b[:, 0, 0, None] * c[:, 0] + tf_b[:, 0, 1, None] * c[:, 1] + tf_b[:, 0, 3, None]
    py = tf_b[:, 1, 0, None] * c[:, 0] + tf_b[:, 1, 1, None] * c[:, 1] + tf_b[:, 1, 3, None]
    gox, goy = float(px.min()), float(py.min())
    n_b = int(math.ceil(max(px.max() - gox, py.max() - goy) / res)) + 1

    sub = 8
    t8 = M.OccupancyGrid(n_b, res, gox, goy, device=dev, lazy_workspace=True)
    merger.fuse_occupancy(stack[:sub], origins[:sub], res, tf_b[:sub], t8)
    want = warp_fuse(stack[:sub].cpu().numpy(), origins[:sub], res, tf_b[:sub], gox, goy, res, n_b, n_b)
    result['parity']['merge_8_agents'] = 'bit-exact' if np.array_equal(t8.grid, want) else 'MISMATCH'
    del t8, want
    if any(v != 'bit-exact' for v in result['parity'].values()):
        result['error'] = 'fused map differs from the NumPy reference'
        print(json.dumps(result))
        raise SystemExit(3)

    merge = {}
    for name, g in (('res_0.05', res), ('res_0.10', 2 * res), ('res_0.025', res / 2)):
        n = int(math.ceil(max(px.max() - gox, py.max() - goy) / g)) + 1
        tb = M.OccupancyGrid(n, g, gox, goy, device=dev, lazy_workspace=True)

        def fuse_b():
            merger.fuse_occupancy(stack, origins, res, tf_b, tb)

        pairs = agent_tile_pairs(tf_b, origins, res, (S, S), gox, goy, g, n)
        merge[name] = measure(torch, _native, fuse_b, stack.numel(), n * n, hbm, args, pairs)
        merge[name]['target'] = f'{n}^2 at {g} m'
        merge[name]['fused_cells'] = {'unknown': int((tb.grid_tensor == -1).sum()), 'free': int((tb.grid_tensor == 0).sum()),
                                      'occupied': int((tb.grid_tensor == 100).sum())}
        del tb
        torch.cuda.empty_cache()
    merge['workload'] = '256 maps of 2048^2 (configs[2], device_grids, seed 0) -> square target covering every corner'
    merge['working_set_fits_l2'] = False
    result['merge'] = merge
    result['parity_line'] = 'parity: bit-exact'
    result['gpu_after'] = gpu_details(torch, dev)
    print(result['parity_line'], file=sys.stderr)
    print(json.dumps(result))


if __name__ == '__main__':
    main()
