#!/usr/bin/env python
"""bench_frontier_assign.py — frontier assignment by geodesic distance (OccupancyGrid.assign_frontiers /
occgrid_frontier_assign), on the device.

Workloads (64 robots each):
  (a) swarm       BASELINE configs[1] (64 agents, 2.5e6 packets, seed 42) integrated by AgentGrids into
                  64 maps of 256^2 in their own frames, fused into the shared 4096^2 map with the room
                  offsets; the robots stand at each agent's last pose mapped through its offset.  Each
                  robot reaches roughly its own room.
  (b) open        4096^2 at 5 cm: FREE with 10 % random obstacles, a 64-cell UNKNOWN border band; the
                  robots at random free cells.  Every robot reaches the whole map.
  (c) serpentine  4096^2: one 1-cell corridor of vertical runs 32 cells apart, joined alternately at the
                  top and the bottom, so the path crosses every tile row 128 times (the worst case for
                  worklist rounds); unknown pockets off the bottom joins; the robots on the corridor.

    python bench_frontier_assign.py [--steps 20] [--warmup 3] [--out profiles/r6_bench_frontier_assign.json]

Before timing, every workload is compared with the reference (tests/frontier_assign_util.py: the C
BFS per robot, the frontier oracle's clusters, the rule in NumPy) bit for bit; a mismatch exits with
status 3.  Reported per workload: ms per occgrid_frontier_assign call (device events, warmed, the
frontier list and clusters already on the device), the kernel time from occgrid_profile_begin/end,
assign_frontiers end to end (stencil + clustering + assignment + the one host read), worklist rounds,
(robot, tile) items, cells settled (reachable cells summed over the robots) per second, and the byte
floor: 4 B per settled cell written once, over the HBM peak, as a fraction of the call.  The CPU leg
is the C BFS over all robots on one core.  Writes the JSON to --out and prints it as one line, with
the GPU's name, power limit and SM clock read in the same run.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np

N_ROBOTS = 64


def open_map(rng, n=4096, band=64):
    grid = np.where(rng.random((n, n)) < 0.1, 100, 0).astype(np.int8)
    grid[:band] = -1
    grid[-band:] = -1
    grid[:, :band] = -1
    grid[:, -band:] = -1
    return grid


def serpentine_map(n=4096, pitch=32):
    grid = np.full((n, n), 100, np.int8)
    xs = list(range(1, n - 1, pitch))
    for i, x in enumerate(xs):
        grid[1:n - 1, x] = 0
        if i + 1 < len(xs):
            y = n - 2 if i % 2 == 0 else 1
            grid[y, x:xs[i + 1] + 1] = 0
            if i % 2 == 0:
                grid[n - 1, x + pitch // 2 - 2:x + pitch // 2 + 2] = -1   # unknown pocket below the join
    return grid


def reference(fa, grid, ox, oy, res, xy):
    """Fields by the C BFS on one core (timed), cells settled, and the reference assignment."""
    h, w = grid.shape
    fields, settled, t = {}, 0, 0.0
    for a in range(len(xy)):
        cell = fa.robot_cell(xy[a, 0], xy[a, 1], ox, oy, res, w, h)
        t0 = time.perf_counter()
        f = fa.oracle_geodesic(grid, *cell) if cell is not None else np.full((h, w), -1, np.int32)
        t += time.perf_counter() - t0
        settled += int((f >= 0).sum())
        fields[a] = f
    want = fa.assign_reference(grid, ox, oy, res, xy, fields=fields.__getitem__)
    return want, settled, t * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r6_bench_frontier_assign.json'))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')

    import torch
    import frontier_assign_util as fa
    from bench_map_fuse import event_ms, gpu_details, hbm_peak_gbs, wall_ms
    from occgrid_b200 import _native, simulation_tools as st
    from occgrid_b200 import dual_bot_mapper as M
    from occgrid_b200.map_merger import MapMerger, se2_matrix
    if not torch.cuda.is_available():
        raise SystemExit('bench_frontier_assign.py needs a CUDA device (no CPU fallback)')
    dev = torch.device('cuda', torch.cuda.current_device())
    hbm, hbm_src = hbm_peak_gbs()
    result = {'metric': 'frontier_assign_ms', 'gpu': gpu_details(torch, dev), 'hbm_peak_gbs': hbm, 'hbm_peak_source': hbm_src,
              'parity': {}}
    lib = _native.lib()
    rng = np.random.default_rng(0)

    def workload(name, grid_obj, xy, desc):
        grid = grid_obj.grid
        got = grid_obj.assign_frontiers(xy)                       # sizes the pool and the cluster columns
        want, settled, cpu_ms = reference(fa, grid, grid_obj.ox, grid_obj.oy, grid_obj.res, xy)
        try:
            fa.assert_same(got, want)
            result['parity'][name] = 'bit-exact'
        except AssertionError:
            result['parity'][name] = 'MISMATCH'
            return
        f, ws, kmax, pool = grid_obj._fr, grid_obj._ws_assign, grid_obj._fa_sizes['kmax'], got.stats['tile_pool']
        A = len(xy)
        d_xy = torch.from_numpy(np.ascontiguousarray(xy, np.float64)).to(dev)
        o = {k: torch.zeros(s, dtype=t, device=dev) for k, s, t in
             (('cl', (A,), torch.int32), ('co', (A,), torch.int32), ('go', (A, 2), torch.int32),
              ('ta', (A, 2), torch.float64), ('cs', (A, kmax), torch.int32), ('st', (1,), torch.int32), ('sx', (3,), torch.int64))}
        stream = torch.cuda.current_stream().cuda_stream

        def call():
            rc = lib.occgrid_frontier_assign(
                grid_obj.grid_tensor.data_ptr(), grid_obj.size, grid_obj.size, grid_obj.ox, grid_obj.oy, grid_obj.res,
                d_xy.data_ptr(), A, f['xy'].data_ptr(), f['count'].data_ptr(), f['label'].data_ptr(), f['root'].data_ptr(),
                f['cent'].data_ptr(), f['ncl'].data_ptr(), kmax, pool, o['cl'].data_ptr(), o['co'].data_ptr(),
                o['go'].data_ptr(), o['ta'].data_ptr(), o['cs'].data_ptr(), o['st'].data_ptr(), o['sx'].data_ptr(),
                ws.data_ptr(), ws.numel(), stream)
            if rc != 0:
                raise RuntimeError(_native.last_error())

        for _ in range(args.warmup):
            call()
        ms = min(event_ms(torch, call, args.steps) for _ in range(3))
        torch.cuda.synchronize()
        _native.profile_begin()
        for _ in range(args.steps):
            call()
        torch.cuda.synchronize()
        prof = _native.profile_end()['frontier_assign']
        rounds, items, slots = o['sx'].cpu().tolist()
        status = int(o['st'].item())
        if status != 0 or not np.array_equal(o['cl'].cpu().numpy(), want['cluster']):
            result['parity'][name] = f'MISMATCH (timed call, status {status})'
            return
        floor_ms = 4.0 * settled / (hbm * 1e9) * 1e3
        result[name] = {
            'workload': desc, 'robots': A, 'frontier_cells': got.stats['frontier_cells'], 'clusters': got.stats['clusters'],
            'assigned': int((got.cluster >= 0).sum()),
            'ms_per_call': round(ms, 4), 'kernel_ms': round(prof[0] / args.steps, 4), 'kernel_launches_per_call': prof[1] // args.steps,
            'assign_frontiers_ms': round(wall_ms(torch, lambda: grid_obj.assign_frontiers(xy), 5), 3),
            'rounds': rounds, 'items': items, 'tile_slots': slots, 'tile_pool': pool,
            'cells_settled': settled, 'cells_settled_per_s': round(settled / (ms * 1e-3), 1),
            'byte_floor_ms': round(floor_ms, 4), 'fraction_of_byte_floor': round(floor_ms / ms, 4),
            'cpu_oracle_ms_one_core': round(cpu_ms, 1)}

    # ---- (a) configs[1]: packets -> 64 agent maps -> fused 4096^2 map -------------------------------
    s = st.generate_session(n_agents=64, n_packets=2_500_000, seed=42)
    maps = M.AgentGrids(64, max_batch=2_500_000, device=dev, size=256, resolution=0.05, origin_x=-4.0, origin_y=-6.4)
    maps.update_packets(s['packets'], agent_offsets=np.zeros((65, 2)))
    G = s['grid']
    fused = M.OccupancyGrid(G['size'], G['resolution'], G['origin_x'], G['origin_y'], device=dev, lazy_workspace=True)
    tf = np.stack([se2_matrix(x, y, 0.0) for x, y in s['agent_offsets'][1:]])
    MapMerger(device=dev).fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, tf, fused)
    pk = s['packets']
    xy = np.full((64, 2), np.nan)
    for a in range(1, 65):
        r = pk[np.nonzero(s['agent_idx'] == a)[0][-1]]
        xy[a - 1] = (float(r[5:9].view('<f4')[0]) + s['agent_offsets'][a, 0], float(r[9:13].view('<f4')[0]) + s['agent_offsets'][a, 1])
    del maps
    workload('swarm', fused, xy, 'configs[1]: 64 agent maps fused into 4096^2 at 0.05 m, robots at their last poses')
    del fused
    torch.cuda.empty_cache()

    # ---- (b) open 4096^2 ------------------------------------------------------------------------------
    grid = open_map(rng)
    g = M.OccupancyGrid(4096, 0.05, 0.0, 0.0, device=dev, lazy_workspace=True)
    g.grid_tensor.copy_(torch.from_numpy(grid))
    ys, xs = np.nonzero(grid == 0)
    pick = rng.choice(len(xs), N_ROBOTS, replace=False)
    xy = np.stack([(xs[pick] + 0.5) * 0.05, (ys[pick] + 0.5) * 0.05], axis=1)
    workload('open', g, xy, 'open 4096^2: 10 % random obstacles, 64-cell unknown border band, 64 robots on random free cells')
    del g
    torch.cuda.empty_cache()

    # ---- (c) serpentine 4096^2 ----------------------------------------------------------------------
    grid = serpentine_map()
    g = M.OccupancyGrid(4096, 0.05, 0.0, 0.0, device=dev, lazy_workspace=True)
    g.grid_tensor.copy_(torch.from_numpy(grid))
    ys, xs = np.nonzero(grid == 0)
    pick = rng.choice(len(xs), N_ROBOTS, replace=False)
    xy = np.stack([(xs[pick] + 0.5) * 0.05, (ys[pick] + 0.5) * 0.05], axis=1)
    workload('serpentine', g, xy, 'serpentine 4096^2: vertical runs 32 cells apart, 128 crossings of every tile row, 64 robots on the path')
    del g

    result['gpu_after'] = gpu_details(torch, dev)
    if any(v != 'bit-exact' for v in result['parity'].values()):
        result['error'] = 'assignment differs from the reference'
        print(json.dumps(result))
        raise SystemExit(3)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(json.dumps(result) + '\n')
    print(json.dumps(result))


if __name__ == '__main__':
    main()
