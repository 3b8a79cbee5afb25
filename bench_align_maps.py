#!/usr/bin/env python
"""bench_align_maps.py — correlative map alignment (MapMerger.align_maps / mapmerge_align): every agent
map searched over rotations x translations around its prior against one reference map, exactly, in one
device call.

Workloads:
  (a) swarm   BASELINE configs[1] (64 agents, 2.5e6 packets, seed 42) integrated by AgentGrids into 64
              maps of 256^2 at 5 cm, against their fusion into the shared 4096^2 map at the true room
              offsets.  Priors: truth perturbed by U(-1, 1) m and U(-20, 20) degrees about each map's
              centre (seed 1).  Search ±1.2 m and ±25 degrees at 0.5 degrees, clearance 0.1 m.
  (b) merge   configs[2] scale: 256 maps of 2048^2 from bench_merge.device_grids against their 4803^2
              fusion, as bench_register_maps.py (b).  Priors perturbed by U(-0.5, 0.5) m and U(-5, 5)
              degrees (seed 1).  Search ±0.6 m and ±6 degrees at 0.25 degrees, clearance 0.1 m.

    python bench_align_maps.py [--steps 5] [--warmup 1] [--out profiles/r9_bench_align_maps.json]

Before timing, every workload is checked: the winner's and the prior's score of a sample of agents
against the NumPy reference (tests/align_maps_util.py), and identical rows from the default block size
and s = 1 (no pruning); a mismatch exits with status 3.  Reported per workload: align_maps end to end
(host clock, including the distance field and both host reads), the mapmerge_align call alone (device
events), the distance field alone, the candidates searched and the share scored exactly, the gathers
per second of the call (gathers = bound lookups + exact lookups, counted here from the point counts:
n_angles * blocks * points per agent for the bounds, and candidates scored exactly * mean points per
agent for the exact pass), the call time for other block sizes, and for (a) how many agents end within
0.03 m and 0.01 degrees of the truth after align_maps -> register_maps and after register_maps alone.
Prints ONE JSON line (and writes it to --out), with the GPU's name, power limit and SM clock read in
the same run.
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

from bench_map_fuse import SWARM_MAP, event_ms, gpu_details


def about_centres(truth, centres, max_t, max_deg, seed=1):
    """truth[a] @ (rotation by U(-max_deg, max_deg) degrees about the map's centre, shift by U(-max_t, max_t) m)."""
    from occgrid_b200.map_merger import se2_matrix
    r = np.random.default_rng(seed)
    out = []
    for a in range(len(truth)):
        d = se2_matrix(*r.uniform(-max_t, max_t, 2), math.radians(r.uniform(-max_deg, max_deg)))
        c = centres[a]
        out.append(truth[a] @ se2_matrix(c[0], c[1], 0.0) @ d @ se2_matrix(-c[0], -c[1], 0.0))
    return np.stack(out)


def pose_error(T, T_true):
    d = np.linalg.inv(T_true) @ T
    return math.hypot(d[0, 3], d[1, 3]), abs(math.degrees(math.atan2(d[1, 0], d[0, 0])))


def run(torch, _native, merger, grids, origins, res, priors, reference, window, args, label):
    import align_maps_util as AU
    lib = _native.lib()
    st = torch.cuda.current_stream().cuda_stream
    A, h, w = (int(v) for v in grids.shape)
    max_offset, max_angle, step, clearance = window
    g = reference.res
    rc = round(max_offset / g)
    theta, rot = AU.rotation_table(max_angle, step)
    max_d2 = AU.max_d2_of(clearance, g)
    org = np.ascontiguousarray(origins, np.float64)
    pri = np.ascontiguousarray(priors, np.float64)
    d2 = reference.distance_field(to_host=False)
    n_pts = (grids > 50).sum(dim=(1, 2)).cpu().numpy().astype(np.int64)
    out = torch.empty((A, 6), dtype=torch.int64, device=grids.device)
    diag = torch.empty(2, dtype=torch.int64, device=grids.device)
    wss = {}

    def call(block=0):
        lib.mapmerge_align_set_block(block)
        ws = wss.get(block)
        if ws is None:
            nb = lib.mapmerge_align_workspace_bytes(A, w, h, reference.size, reference.size, max_d2, rc, len(rot), int(n_pts.sum()))
            ws = wss[block] = torch.empty(nb, dtype=torch.uint8, device=grids.device)
        _native.check(lib.mapmerge_align(grids.data_ptr(), A, w, h, res, org.ctypes.data, pri.ctypes.data, d2.data_ptr(),
                                         reference.size, reference.size, reference.ox, reference.oy, g, rot.ctypes.data, len(rot),
                                         rc, max_d2, out.data_ptr(), diag.data_ptr(), ws.data_ptr(), ws.numel(), st), 'mapmerge_align')
        lib.mapmerge_align_set_block(0)

    call(1)
    exhaustive = out.cpu().numpy()
    call(0)
    rows, dg = out.cpu().numpy(), diag.cpu().numpy()
    d2h = d2.cpu().numpy()
    ok = np.array_equal(rows, exhaustive)
    sample = sorted({0, A // 3, A // 2, A - 1} | set(np.flatnonzero(rows[:, 0] > rows[:, 4])[:2].tolist()))
    for a in sample:
        gh = grids[a].cpu().numpy()
        k, dx, dy = (int(v) for v in rows[a, 1:4])
        ok &= rows[a, 0] == AU.score_at(gh, org[a], res, pri[a], d2h, reference.ox, reference.oy, g, *rot[k], dx, dy, max_d2)
        ok &= rows[a, 4] == AU.score_at(gh, org[a], res, pri[a], d2h, reference.ox, reference.oy, g, 1.0, 0.0, 0, 0, max_d2)
        ok &= rows[a, 5] == n_pts[a]
    res_out = {'workload': label, 'parity': 'bit-exact' if ok else 'MISMATCH', 'agents': A, 'points': int(n_pts.sum()),
               'rotations': len(rot), 'max_offset_cells': rc, 'max_d2': max_d2, 'sampled_agents': sample}
    if not ok:
        return res_out
    for _ in range(args.warmup):
        call()
        reference.distance_field(to_host=False)
    res_out['align_call_ms'] = round(min(event_ms(torch, call, args.steps) for _ in range(3)), 4)
    res_out['distance_field_ms'] = round(min(event_ms(torch, lambda: reference.distance_field(to_host=False), args.steps)
                                             for _ in range(3)), 4)
    ts = []
    for _ in range(max(args.steps, 3)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        al = merger.align_maps(grids, origins, res, priors, reference, max_offset=max_offset, max_angle=max_angle,
                               angle_step=step, clearance=clearance)
        ts.append((time.perf_counter() - t0) * 1e3)
    res_out['align_maps_end_to_end_ms'] = round(sorted(ts)[len(ts) // 2], 3)
    live = n_pts > 0
    searched, scored = int(dg[0]), int(dg[1])
    nb = (-(-(2 * rc + 1) // 8)) ** 2
    bound_gathers = int((len(rot) * nb * n_pts[live]).sum())
    exact_gathers = int(round(scored * n_pts[live].mean()))
    res_out.update(candidates_searched=searched, candidates_scored_exactly=scored,
                   fraction_scored_exactly=round(scored / searched, 6), bound_gathers=bound_gathers,
                   exact_gathers_estimate=exact_gathers,
                   gathers_per_s=round((bound_gathers + exact_gathers) / (res_out['align_call_ms'] * 1e-3), 1),
                   exhaustive_gathers=int((len(rot) * (2 * rc + 1) ** 2 * n_pts[live]).sum()))
    sweep = {}
    for s in (2, 4, 16, 32):
        call(s)
        sweep[s] = round(min(event_ms(torch, lambda: call(s), max(args.steps // 2, 1)) for _ in range(2)), 4)
    res_out['align_call_ms_by_block'] = sweep
    torch.cuda.synchronize()
    _native.profile_begin()
    for _ in range(args.steps):
        call()
    torch.cuda.synchronize()
    prof = _native.profile_end()
    res_out['map_align_kernels_ms'] = round(prof['map_align'][0] / args.steps, 4)
    res_out['improved'] = int(al.improved.sum())
    return res_out, al


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=1)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r9_bench_align_maps.json'), help='also write the JSON line here')
    args = ap.parse_args()
    import torch
    from occgrid_b200 import _native, simulation_tools as st
    from occgrid_b200 import dual_bot_mapper as M
    from occgrid_b200.map_merger import MapMerger, se2_matrix
    from bench_merge import device_grids
    if not torch.cuda.is_available():
        raise SystemExit('bench_align_maps.py needs a CUDA device (no CPU fallback)')
    dev = torch.device('cuda', torch.cuda.current_device())
    result = {'metric': 'align_maps_ms', 'gpu': gpu_details(torch, dev)}
    merger = MapMerger(device=dev)
    failed = False

    # (a) configs[1]
    s = st.generate_session(n_agents=64, n_packets=2_500_000, seed=42)
    maps = M.AgentGrids(64, max_batch=2_500_000, device=dev, **SWARM_MAP)
    maps.update_packets(s['packets'], agent_offsets=np.zeros((65, 2)))
    truth = np.stack([se2_matrix(x, y, 0.0) for x, y in s['agent_offsets'][1:]])
    G = s['grid']
    ref_a = M.OccupancyGrid(G['size'], G['resolution'], G['origin_x'], G['origin_y'], device=dev, lazy_workspace=True)
    merger.fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, truth, ref_a)
    priors = about_centres(truth, maps.origins + 256 * 0.05 / 2, 1.0, 20.0)
    out = run(torch, _native, merger, maps.grids_tensor, maps.origins, maps.res, priors, ref_a,
              (1.2, math.radians(25), math.radians(0.5), 0.1), args,
              '64 maps of 256^2 (configs[1]) against their fused 4096^2 map; priors off by U(-1, 1) m, U(-20, 20) deg')
    if isinstance(out, dict):
        result['swarm'], failed = out, True
    else:
        result['swarm'], al = out
        reg = merger.register_maps(maps.grids_tensor, maps.origins, maps.res, al.transformation, reference=ref_a)
        alone = merger.register_maps(maps.grids_tensor, maps.origins, maps.res, priors, reference=ref_a)

        def recovered(r):
            return int(sum(1 for a in range(64) if r.accepted[a] and pose_error(r.transformation[a], truth[a])[0] <= 0.03
                           and pose_error(r.transformation[a], truth[a])[1] <= 0.01))
        result['swarm']['recovered_align_then_register'] = recovered(reg)
        result['swarm']['recovered_register_alone'] = recovered(alone)
    del maps, ref_a
    torch.cuda.empty_cache()

    # (b) configs[2] scale
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
    ref_b = M.OccupancyGrid(n_b, res, gox, goy, device=dev, lazy_workspace=True)
    merger.fuse_occupancy(stack, origins, res, tf_b, ref_b)
    priors_b = about_centres(tf_b, origins + S * res / 2, 0.5, 5.0)
    out = run(torch, _native, merger, stack, origins, res, priors_b, ref_b, (0.6, math.radians(6), math.radians(0.25), 0.1), args,
              f'256 maps of 2048^2 (configs[2] scale) against their fused {n_b}^2 map; priors off by U(-0.5, 0.5) m, U(-5, 5) deg')
    if isinstance(out, dict):
        result['merge'], failed = out, True
    else:
        result['merge'] = out[0]
    result['gpu_after'] = gpu_details(torch, dev)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')
    if failed:
        raise SystemExit(3)


if __name__ == '__main__':
    main()
