#!/usr/bin/env python
"""bench_register_maps.py — batched map registration (MapMerger.register_maps /
mapmerge_icp_register_batch): every agent map refined against one reference map in one device call.

Workloads (priors = true transform @ se2(dx, dy, dtheta) about the agent's frame, dx, dy ~
U(-0.15, 0.15) m, dtheta ~ U(-3, 3) degrees, seed 1):
  (a) swarm   BASELINE configs[1] (64 agents, 2.5e6 packets, seed 42) integrated by AgentGrids into
              64 maps of 256^2 at 5 cm; the reference is their fusion into the shared 4096^2 map
              with the true room offsets.
  (b) merge   configs[2] scale: 256 maps of 2048^2 from bench_merge.device_grids, true transforms
              theta ~ U(-pi, pi), t ~ U(-50, 50)^2 (seed 0), fused at 5 cm into the square map that
              covers every corner; that fused map is the reference.

    python bench_register_maps.py [--steps 5] [--warmup 1] [--out profiles/r7_bench_register_maps.json]

Before timing, every agent's batched result is compared bit for bit with a separate
mapmerge_icp_register call on the same inputs; a mismatch exits with status 3.  Reported per
workload: the batched call alone (device events), the same A registrations one by one through the C
ABI (device events, no host reads in between), register_maps end to end (host clock, two host
reads), the rounds (largest iteration count), the points x (iterations + 1) associations per second
of the batched call, and its kernel time.  Prints ONE JSON line (and writes it to --out), with the
GPU's name, power limit and SM clock read in the same run.
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


def perturbed(truth, seed=1):
    r = np.random.default_rng(seed)
    A = len(truth)
    d = np.stack([r.uniform(-0.15, 0.15, A), r.uniform(-0.15, 0.15, A), np.radians(r.uniform(-3, 3, A))], 1)
    out = []
    for a in range(A):
        c, s = math.cos(d[a, 2]), math.sin(d[a, 2])
        P = np.eye(4)
        P[0, 0], P[0, 1], P[0, 3], P[1, 0], P[1, 1], P[1, 3] = c, -s, d[a, 0], s, c, d[a, 1]
        out.append(truth[a] @ P)
    return np.stack(out)


def run(torch, _native, merger, grids, origins, res, priors, reference, args, label):
    lib = _native.lib()
    st = torch.cuda.current_stream().cuda_stream
    A = grids.shape[0]
    Tm = merger._as_matrices(priors, A)
    job = merger._registration_inputs(grids, np.ascontiguousarray(origins, np.float64), res, Tm, reference, 1.0)
    nbytes = lib.mapmerge_icp_register_batch_workspace_bytes(job.n_target, job.n_points, A, job.cells_w, job.cells_h)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=grids.device)
    out = torch.empty((A, 20), dtype=torch.float64, device=grids.device)

    def batched():
        _native.check(lib.mapmerge_icp_register_batch(job.sx.data_ptr(), job.sy.data_ptr(), job.offsets.data_ptr(), A,
                                                      job.tx.data_ptr(), job.ty.data_ptr(), job.n_target, job.min_x, job.min_y,
                                                      job.cell, job.cells_w, job.cells_h, 1.0, 30, 1e-6, 1e-6, out.data_ptr(),
                                                      ws.data_ptr(), ws.numel(), st), 'mapmerge_icp_register_batch')

    offs = job.offsets.cpu().numpy()
    big = int(np.diff(offs).max())
    sws = torch.empty(max(lib.mapmerge_icp_workspace_bytes(job.n_target, max(big, 1), job.cells_w, job.cells_h), 1),
                      dtype=torch.uint8, device=grids.device)
    one = torch.zeros((A, 20), dtype=torch.float64, device=grids.device)
    live = [a for a in range(A) if offs[a + 1] > offs[a]]

    def one_by_one():
        for a in live:
            n = int(offs[a + 1] - offs[a])
            _native.check(lib.mapmerge_icp_register(job.sx[offs[a]:].data_ptr(), job.sy[offs[a]:].data_ptr(), n, job.tx.data_ptr(),
                                                    job.ty.data_ptr(), job.n_target, job.min_x, job.min_y, job.cell, job.cells_w,
                                                    job.cells_h, 1.0, 30, 1e-6, 1e-6, one[a].data_ptr(), sws.data_ptr(), sws.numel(),
                                                    st), 'mapmerge_icp_register')

    batched()
    one_by_one()
    torch.cuda.synchronize()
    got, want = out.cpu().numpy(), one.cpu().numpy()
    for a in range(A):
        if a not in live:
            want[a, :16] = np.eye(4).ravel()
    parity = 'bit-exact' if np.array_equal(got.view(np.int64), want.view(np.int64)) else 'MISMATCH'
    res_out = {'parity_vs_single_calls': parity, 'agents': A, 'agents_with_points': len(live), 'source_points': job.n_points,
               'reference_points': job.n_target, 'cell_list': f'{job.cells_w} x {job.cells_h}'}
    if parity != 'bit-exact':
        return res_out
    for _ in range(args.warmup):
        batched()
        one_by_one()
    res_out['batched_ms'] = round(min(event_ms(torch, batched, args.steps) for _ in range(3)), 4)
    res_out['one_by_one_ms'] = round(min(event_ms(torch, one_by_one, max(args.steps // 2, 1)) for _ in range(2)), 4)
    res_out['speedup_vs_one_by_one'] = round(res_out['one_by_one_ms'] / res_out['batched_ms'], 2)
    torch.cuda.synchronize()
    _native.profile_begin()
    for _ in range(args.steps):
        batched()
    torch.cuda.synchronize()
    prof = _native.profile_end()
    res_out['batched_kernel_ms'] = round(prof['icp_batch'][0] / args.steps, 4)
    its = got[:, 18].astype(np.int64)
    n_a = np.diff(offs)
    res_out['rounds'] = int(its.max())
    res_out['iterations'] = {'min': int(its[live].min()), 'median': float(np.median(its[live])), 'max': int(its.max())}
    assoc = int((n_a * (its + 1) * (n_a > 0)).sum())
    res_out['point_associations'] = assoc
    res_out['point_iterations_per_s'] = round(assoc / (res_out['batched_ms'] * 1e-3), 1)
    res_out['accepted'] = int((got[:, 16] >= 0.6).sum())
    ts = []
    for _ in range(max(args.steps, 3)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        merger.register_maps(grids, origins, res, priors, reference=reference)
        ts.append((time.perf_counter() - t0) * 1e3)
    res_out['register_maps_end_to_end_ms'] = round(sorted(ts)[len(ts) // 2], 3)
    res_out['workload'] = label
    return res_out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=1)
    ap.add_argument('--out', default=None, help='also write the JSON line here')
    args = ap.parse_args()
    import torch
    from occgrid_b200 import _native, simulation_tools as st
    from occgrid_b200 import dual_bot_mapper as M
    from occgrid_b200.map_merger import MapMerger, se2_matrix
    from bench_merge import device_grids
    if not torch.cuda.is_available():
        raise SystemExit('bench_register_maps.py needs a CUDA device (no CPU fallback)')
    dev = torch.device('cuda', torch.cuda.current_device())
    result = {'metric': 'register_maps_ms', 'gpu': gpu_details(torch, dev)}
    merger = MapMerger(device=dev)

    # (a) configs[1]
    s = st.generate_session(n_agents=64, n_packets=2_500_000, seed=42)
    maps = M.AgentGrids(64, max_batch=2_500_000, device=dev, **SWARM_MAP)
    maps.update_packets(s['packets'], agent_offsets=np.zeros((65, 2)))
    truth = np.stack([se2_matrix(x, y, 0.0) for x, y in s['agent_offsets'][1:]])
    G = s['grid']
    ref_a = M.OccupancyGrid(G['size'], G['resolution'], G['origin_x'], G['origin_y'], device=dev, lazy_workspace=True)
    merger.fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, truth, ref_a)
    result['swarm'] = run(torch, _native, merger, maps.grids_tensor, maps.origins, maps.res, perturbed(truth), ref_a, args,
                          '64 maps of 256^2 (configs[1]) against their fused 4096^2 map, perturbed room offsets')
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
    result['merge'] = run(torch, _native, merger, stack, origins, res, perturbed(tf_b), ref_b, args,
                          f'256 maps of 2048^2 (configs[2] scale) against their fused {n_b}^2 map, perturbed transforms')
    result['gpu_after'] = gpu_details(torch, dev)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')
    if any(result[k].get('parity_vs_single_calls') != 'bit-exact' for k in ('swarm', 'merge')):
        raise SystemExit(3)


if __name__ == '__main__':
    main()
