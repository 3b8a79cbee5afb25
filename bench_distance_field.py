#!/usr/bin/env python
"""bench_distance_field.py — obstacle clearance on the device: the exact squared distance field
(occgrid_distance_field) and the navigation grid of a robot radius (occgrid_inflate).

Workloads:
  (a) swarm   BASELINE configs[1] (64 agents, 2.5e6 packets, seed 42) fused into the shared 4096^2 map
              as in bench_frontier_assign.py; its 64 robots at their last poses.
  (b) open    4096^2 at 5 cm with 10 % random obstacles and a 64-cell unknown border
              (bench_frontier_assign.open_map); 64 robots on random free cells.
  (c) merge   BASELINE configs[2]: 256 maps of 2048^2 (bench_merge.device_grids) fused into the 4803^2
              map at 5 cm as in bench_map_fuse.py; 64 robots on random free cells.
  (d) sparse  16384^2, FREE with 8 obstacles: the envelope of every row spans the whole row.

    python bench_distance_field.py [--steps 20] [--warmup 3] [--out profiles/r7_bench_distance_field.json]

Before timing, every workload is checked bit for bit: (a)-(c) against tests/distance_field_util.py
(scipy's feature transform for d2, the NumPy inflation and footprint rule), (d) against the closed form
min over the obstacles of dx^2 + dy^2 on the device; a mismatch exits with status 3.  Reported per
workload: ms per occgrid_distance_field and per occgrid_inflate call (64 robots, 0.15 m radius) from
device events, the kernel time from occgrid_profile_begin/end, and the byte floor, 1 B read + 4 B
written per cell over the HBM peak, as a fraction of the distance-field call; SciPy's
distance_transform_edt on one core on (a)-(c).  On (a), assign_frontiers with and without
robot_radius=0.15 end to end (median wall time), the robots with a target both ways, the robots
whose assignment changed, and the robots with a target at radii from 0 to 0.15 m.  Writes the JSON to
--out and prints it as one line, with the GPU's name, power limit and SM clock read in the same run.
"""
import argparse
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np

N_ROBOTS = 64
RADIUS = 0.15


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r7_bench_distance_field.json'))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')

    import torch
    from scipy.ndimage import distance_transform_edt
    import distance_field_util as du
    from bench_frontier_assign import open_map
    from bench_map_fuse import event_ms, gpu_details, hbm_peak_gbs, wall_ms
    from bench_merge import device_grids
    from occgrid_b200 import _native, simulation_tools as st
    from occgrid_b200 import dual_bot_mapper as M
    from occgrid_b200.map_merger import MapMerger, se2_matrix
    if not torch.cuda.is_available():
        raise SystemExit('bench_distance_field.py needs a CUDA device (no CPU fallback)')
    dev = torch.device('cuda', torch.cuda.current_device())
    hbm, hbm_src = hbm_peak_gbs()
    result = {'metric': 'distance_field_ms', 'gpu': gpu_details(torch, dev), 'hbm_peak_gbs': hbm, 'hbm_peak_source': hbm_src,
              'robot_radius_m': RADIUS, 'parity': {}}
    lib = _native.lib()
    stream = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(0)

    def free_robots(grid, res, ox, oy):
        ys, xs = np.nonzero(grid == 0)
        pick = rng.choice(len(xs), N_ROBOTS, replace=False)
        return np.stack([ox + (xs[pick] + 0.5) * res, oy + (ys[pick] + 0.5) * res], axis=1)

    def workload(name, g, xy, desc, check):
        """check(d2 device tensor, nav device tensor, max_d2) -> bool, before any timing."""
        n = g.size
        max_d2 = g._max_d2(RADIUS, 'bench')
        ws = g._edt_workspace()
        d2 = torch.empty((n, n), dtype=torch.int32, device=dev)
        nav = torch.empty((n, n), dtype=torch.int8, device=dev)
        A = 0 if xy is None else len(xy)
        d_xy = torch.from_numpy(np.ascontiguousarray(xy, np.float64)).to(dev) if A else None

        def edt():
            rc = lib.occgrid_distance_field(g.grid_tensor.data_ptr(), n, n, d2.data_ptr(), ws.data_ptr(), ws.numel(), stream)
            if rc != 0:
                raise RuntimeError(_native.last_error())

        def inflate():
            rc = lib.occgrid_inflate(g.grid_tensor.data_ptr(), n, n, g.ox, g.oy, g.res, max_d2, d_xy.data_ptr() if A else None, A,
                                     nav.data_ptr(), ws.data_ptr(), ws.numel(), stream)
            if rc != 0:
                raise RuntimeError(_native.last_error())

        edt()
        inflate()
        torch.cuda.synchronize()
        if not check(d2, nav, max_d2):
            result['parity'][name] = 'MISMATCH'
            return None
        result['parity'][name] = 'bit-exact'
        out = {'workload': desc, 'cells': n * n, 'robots': A, 'max_d2': max_d2,
               'obstacle_cells': int((g.grid_tensor > 50).sum()), 'free_cells': int((g.grid_tensor == 0).sum())}
        out['cells_inflated'] = int((nav != g.grid_tensor).sum())
        for label, fn in (('distance_field', edt), ('inflate', inflate)):
            for _ in range(args.warmup):
                fn()
            ms = min(event_ms(torch, fn, args.steps) for _ in range(3))
            torch.cuda.synchronize()
            _native.profile_begin()
            for _ in range(args.steps):
                fn()
            torch.cuda.synchronize()
            prof = _native.profile_end()['distance_field']
            out[f'{label}_ms'] = round(ms, 4)
            out[f'{label}_kernel_ms'] = round(prof[0] / args.steps, 4)
            out[f'{label}_launches_per_call'] = prof[1] // args.steps
        floor_ms = 5.0 * n * n / (hbm * 1e9) * 1e3
        out['byte_floor_ms'] = round(floor_ms, 4)
        out['fraction_of_byte_floor'] = round(floor_ms / out['distance_field_ms'], 4)
        result[name] = out
        return out

    def scipy_ms(grid):
        t0 = time.perf_counter()
        distance_transform_edt(grid <= 50)
        return round((time.perf_counter() - t0) * 1e3, 1)

    def reference_check(grid, xy, ox, oy, res):
        def check(d2, nav, max_d2):
            want = du.edt_reference(grid)
            return (np.array_equal(d2.cpu().numpy(), want) and
                    np.array_equal(nav.cpu().numpy(), du.inflate_reference(grid, max_d2, xy, ox, oy, res, d2=want)))
        return check

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
    grid = fused.grid
    out = workload('swarm', fused, xy, 'configs[1]: 64 agent maps fused into 4096^2 at 0.05 m, robots at their last poses',
                   reference_check(grid, xy, fused.ox, fused.oy, fused.res))
    if out is not None:
        out['scipy_edt_ms_one_core'] = scipy_ms(grid)
        point = fused.assign_frontiers(xy)
        wide = fused.assign_frontiers(xy, robot_radius=RADIUS)
        out['assign_frontiers_ms'] = round(wall_ms(torch, lambda: fused.assign_frontiers(xy), 5), 3)
        out['assign_frontiers_radius_ms'] = round(wall_ms(torch, lambda: fused.assign_frontiers(xy, robot_radius=RADIUS), 5), 3)
        out['robots_with_target'] = int((point.cluster >= 0).sum())
        out['robots_with_target_radius'] = int((wide.cluster >= 0).sum())
        out['assignments_changed'] = int((point.cluster != wide.cluster).sum())
        out['robots_with_target_by_radius'] = {str(r): int((fused.assign_frontiers(xy, robot_radius=r).cluster >= 0).sum())
                                               for r in (0.0, 0.025, 0.05, 0.075, 0.1, 0.125, 0.15)}
    del fused
    torch.cuda.empty_cache()

    # ---- (b) open 4096^2 ------------------------------------------------------------------------------
    grid = open_map(rng)
    g = M.OccupancyGrid(4096, 0.05, 0.0, 0.0, device=dev, lazy_workspace=True)
    g.grid_tensor.copy_(torch.from_numpy(grid))
    xy = free_robots(grid, 0.05, 0.0, 0.0)
    out = workload('open', g, xy, 'open 4096^2: 10 % random obstacles, 64-cell unknown border band, 64 robots on free cells',
                   reference_check(grid, xy, 0.0, 0.0, 0.05))
    if out is not None:
        out['scipy_edt_ms_one_core'] = scipy_ms(grid)
    del g
    torch.cuda.empty_cache()

    # ---- (c) configs[2]: 256 maps of 2048^2 fused into 4803^2 ---------------------------------------
    A, S, res = 256, 2048, 0.05
    stack = torch.stack(device_grids(torch, dev, A, S))
    torch.cuda.empty_cache()
    rng_b = np.random.default_rng(0)                 # the transforms of bench_map_fuse.py
    origins = np.tile(np.array([[-S * res / 2, -S * res / 2]]), (A, 1))
    tf_b = np.stack([se2_matrix(*rng_b.uniform(-50, 50, 2), rng_b.uniform(-math.pi, math.pi)) for _ in range(A)])
    c = np.array([[0, 0], [S, 0], [0, S], [S, S]], np.float64) * res + origins[0]
    px = tf_b[:, 0, 0, None] * c[:, 0] + tf_b[:, 0, 1, None] * c[:, 1] + tf_b[:, 0, 3, None]
    py = tf_b[:, 1, 0, None] * c[:, 0] + tf_b[:, 1, 1, None] * c[:, 1] + tf_b[:, 1, 3, None]
    gox, goy = float(px.min()), float(py.min())
    n_c = int(math.ceil(max(px.max() - gox, py.max() - goy) / res)) + 1
    g = M.OccupancyGrid(n_c, res, gox, goy, device=dev, lazy_workspace=True)
    MapMerger(device=dev).fuse_occupancy(stack, origins, res, tf_b, g)
    del stack
    torch.cuda.empty_cache()
    grid = g.grid
    xy = free_robots(grid, res, gox, goy)
    out = workload('merge', g, xy, f'configs[2]: 256 maps of 2048^2 fused into {n_c}^2 at 0.05 m, 64 robots on free cells',
                   reference_check(grid, xy, gox, goy, res))
    if out is not None:
        out['scipy_edt_ms_one_core'] = scipy_ms(grid)
    del g
    torch.cuda.empty_cache()

    # ---- (d) sparse 16384^2 -------------------------------------------------------------------------
    n = 16384
    g = M.OccupancyGrid(n, 0.05, 0.0, 0.0, device=dev, lazy_workspace=True)
    g.grid_tensor.zero_()
    obs = rng.integers(0, n, (8, 2))
    for x, y in obs:
        g.grid_tensor[int(y), int(x)] = 100

    def sparse_check(d2, nav, max_d2):
        xs = torch.arange(n, device=dev, dtype=torch.int64).view(1, -1)
        for y0 in range(0, n, 1024):
            ys = torch.arange(y0, y0 + 1024, device=dev, dtype=torch.int64).view(-1, 1)
            want = None
            for x, y in obs:
                d = (xs - int(x)) ** 2 + (ys - int(y)) ** 2
                want = d if want is None else torch.minimum(want, d)
            if not torch.equal(d2[y0:y0 + 1024].to(torch.int64), want):
                return False
            blocked = (g.grid_tensor[y0:y0 + 1024] == 0) & (want <= max_d2)
            if not torch.equal(nav[y0:y0 + 1024], torch.where(blocked, torch.full_like(nav[y0:y0 + 1024], 100),
                                                                 g.grid_tensor[y0:y0 + 1024])):
                return False
        return True

    out = workload('sparse', g, None, 'sparse 16384^2: FREE with 8 obstacles, no robots (closed-form check)', sparse_check)
    if out is not None:
        out['scipy_edt_ms_one_core'] = 'not measured (268 M cells)'
    del g
    torch.cuda.empty_cache()

    result['gpu_after'] = gpu_details(torch, dev)
    if any(v != 'bit-exact' for v in result['parity'].values()):
        result['error'] = 'distance field or navigation grid differs from the reference'
        print(json.dumps(result))
        raise SystemExit(3)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(json.dumps(result) + '\n')
    print(json.dumps(result))


if __name__ == '__main__':
    main()
