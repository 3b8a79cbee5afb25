"""ctypes binding of the C ABI in ``include/occgrid_b200.h`` (liboccgrid_b200.so).

The shared library is built in-tree by :func:`build` (``nvcc -gencode
arch=compute_100a,code=sm_100a``); there is NO fallback: if it is missing or a CUDA device is
absent, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, 'csrc')
LIB_PATH = os.path.join(PKG_DIR, 'liboccgrid_b200.so')
SOURCES = ['occgrid_integrate.cu', 'occgrid_tiled.cu', 'occgrid_route.cu', 'occgrid_band.cu', 'mapmerge.cu', 'frontier.cu', 'icp.cu', 'icp_batch.cu', 'render.cu', 'map_fuse.cu', 'frontier_assign.cu', 'distance_field.cu', 'map_align.cu', 'slam_chain.cpp']
HEADERS = ['common.cuh', 'beam_expand.cuh', 'block_ops.cuh', 'icp_core.cuh', 'sincos_dd.cuh', os.path.join('..', '..', 'include', 'occgrid_b200.h')]

STRATEGY = {'auto': -1, 'global_atomic': 0, 'tiled': 1}
COUNTER_NAMES = ('packets', 'accepted', 'dropped', 'bad_pose', 'beams', 'hits', 'updates', 'slowpath',
                 'owned_updates', 'records')
N_COUNTERS = 16


class OccGridError(RuntimeError):
    pass


class Geom(C.Structure):
    """struct occgrid_geom"""
    _fields_ = [('ox', C.c_double), ('oy', C.c_double), ('res', C.c_double),
                ('size_x', C.c_int32), ('size_y', C.c_int32),
                ('win_x0', C.c_int32), ('win_y0', C.c_int32),
                ('win_w', C.c_int32), ('win_h', C.c_int32)]


class RouteJob(C.Structure):
    """struct occgrid_route_job"""
    _fields_ = [('d_packets', C.c_void_p), ('n', C.c_int64), ('stride', C.c_int32), ('rec_len', C.c_int32),
                ('d_agent_idx', C.c_void_p), ('d_drift', C.c_void_p), ('d_agent_off', C.c_void_p), ('n_agents', C.c_int32),
                ('ordinal_base', C.c_uint32), ('ox', C.c_double), ('oy', C.c_double), ('res', C.c_double),
                ('size_x', C.c_int32), ('n_bands', C.c_int32), ('src_rank', C.c_int32), ('band_y0', C.c_int32 * 33),
                ('d_peer_recs', C.c_void_p), ('d_peer_tiles', C.c_void_p), ('seg_capacity', C.c_int64), ('d_resv', C.c_void_p), ('d_status', C.c_void_p),
                ('d_counters', C.c_void_p)]


class BandCtx(C.Structure):
    """struct occgrid_band_ctx"""
    _fields_ = [('band_geom', Geom), ('n_bands', C.c_int32), ('rank', C.c_int32), ('seg_capacity', C.c_int64),
                ('d_recv', C.c_void_p * 2), ('d_recv_tiles', C.c_void_p * 2), ('d_seg_counts', C.c_void_p * 2),
                ('d_peer_recs', C.c_void_p * 2), ('d_peer_tiles', C.c_void_p * 2), ('d_peer_seg_counts', C.c_void_p * 2),
                ('d_peer_flags', C.c_void_p), ('d_my_flags', C.c_void_p), ('d_resv', C.c_void_p), ('d_status', C.c_void_p),
                ('d_grid', C.c_void_p), ('d_workspace', C.c_void_p), ('workspace_bytes', C.c_size_t), ('d_counters', C.c_void_p),
                ('ev_fused', C.c_void_p), ('ev_published', C.c_void_p), ('published_pending', C.c_int32)]


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA translation unit for sm_100a into liboccgrid_b200.so (in-tree)."""
    if not force and not _stale():
        return LIB_PATH
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    cmd = ['nvcc', '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
           '-Xcompiler', '-fPIC', '-Xcompiler', '-ffp-contract=off', '-shared', '-o', LIB_PATH] + srcs
    if verbose:
        cmd.insert(1, '-Xptxas=-v')
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise OccGridError('nvcc failed:\n' + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB_PATH


_lib = None


def lib():
    """Load the library (never builds implicitly on a GPU box: the .so travels with the repo)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OccGridError(f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                           '(needs nvcc).  There is no CPU fallback.')
    L = C.CDLL(LIB_PATH)
    vp, i64, i32, u32, sz = C.c_void_p, C.c_int64, C.c_int, C.c_uint32, C.c_size_t
    gp = C.POINTER(Geom)
    L.occgrid_abi_version.restype = i32
    L.occgrid_last_error.restype = C.c_char_p
    L.occgrid_workspace_bytes.restype = sz
    L.occgrid_workspace_bytes.argtypes = [gp, i64, i32]
    L.occgrid_workspace_reset.restype = i32
    L.occgrid_workspace_reset.argtypes = [vp, sz, vp]
    L.occgrid_integrate_packets.restype = i32
    L.occgrid_integrate_packets.argtypes = [gp, vp, i64, i32, i32, vp, vp, vp, i32, vp, vp, sz, vp, i32, vp]
    L.occgrid_agent_maps_workspace_bytes.restype = sz
    L.occgrid_agent_maps_workspace_bytes.argtypes = [gp, i32, i64, i32]
    L.occgrid_integrate_packets_agent_maps.restype = i32
    L.occgrid_integrate_packets_agent_maps.argtypes = [gp, vp, i64, i32, i32, vp, vp, vp, i32, vp, vp, sz, vp, i32, vp]
    L.occgrid_update_rays.restype = i32
    L.occgrid_update_rays.argtypes = [gp, vp, vp, i64, vp, vp, sz, vp, i32, vp]
    L.occgrid_scatter_probe.restype = i32
    L.occgrid_scatter_probe.argtypes = [i32, vp, i64, i64, u32, vp]
    L.occgrid_route_workspace_bytes.restype = sz
    L.occgrid_route_workspace_bytes.argtypes = [i64, i32]
    L.occgrid_route_packets.restype = i32
    L.occgrid_route_packets.argtypes = [gp, i32, vp, vp, i64, i32, i32, vp, vp, vp, i32, vp, i64, vp, vp, vp,
                                        vp, sz, vp]
    L.occgrid_integrate_poses.restype = i32
    L.occgrid_integrate_poses.argtypes = [gp, vp, i64, i32, vp, vp, sz, vp, i32, vp]
    L.occgrid_band_workspace_bytes.restype = sz
    L.occgrid_band_workspace_bytes.argtypes = [gp, i32, i64]
    L.occgrid_band_prepare.restype = i32
    L.occgrid_band_prepare.argtypes = [gp, vp, vp, i32, i64, vp, vp, sz, vp, vp]
    L.occgrid_band_raycast_route.restype = i32
    L.occgrid_band_raycast_route.argtypes = [gp, vp, i32, i64, i32, C.POINTER(RouteJob), vp, vp, sz, vp, vp]
    L.occgrid_band_step.restype = i32
    L.occgrid_band_step.argtypes = [C.POINTER(BandCtx), i64, i32, C.POINTER(RouteJob), i32, vp, vp]
    L.occgrid_band_join.restype = i32
    L.occgrid_band_join.argtypes = [C.POINTER(BandCtx), vp]
    L.occgrid_band_publish.restype = i32
    L.occgrid_band_publish.argtypes = [i32, i32, vp, i64, vp, vp, vp, u32, i32, vp, vp]
    L.occgrid_frontier_workspace_bytes.restype = sz
    L.occgrid_frontier_workspace_bytes.argtypes = [i64, i64]
    L.occgrid_frontiers.restype = i32
    L.occgrid_frontiers.argtypes = [vp, i32, i32, vp, i64, vp, vp, vp, sz, vp]
    L.occgrid_frontier_clusters.restype = i32
    L.occgrid_frontier_clusters.argtypes = [vp, vp, i64, i32, i32, C.c_double, C.c_double, C.c_double, vp, vp, vp, vp, vp,
                                            vp, sz, vp]
    L.occgrid_render_overlay.restype = i32
    L.occgrid_render_overlay.argtypes = [vp, i32, i32, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                         i32, i32, vp, vp, vp, vp]
    L.occgrid_set_raycast_ctas_per_sm.restype = i32
    L.occgrid_set_raycast_ctas_per_sm.argtypes = [i32]
    L.occgrid_profile_begin.restype = i32
    L.occgrid_profile_end.restype = i32
    L.occgrid_profile_end.argtypes = [vp, vp, i32]
    _bind_merge(L)
    _lib = L
    return L


def _bind_merge(L):
    """mapmerge_* entry points (include/occgrid_b200.h)."""
    vp, i64, i32, sz, dbl = C.c_void_p, C.c_int64, C.c_int32, C.c_size_t, C.c_double
    L.mapmerge_count_occupied.restype = C.c_int
    L.mapmerge_count_occupied.argtypes = [vp, i64, vp, vp]
    L.mapmerge_extract_workspace_bytes.restype = sz
    L.mapmerge_extract_workspace_bytes.argtypes = [i64]
    L.mapmerge_extract_transform.restype = C.c_int
    L.mapmerge_extract_transform.argtypes = [vp, i32, i32, dbl, dbl, dbl, vp, vp, vp, i64, vp, vp, vp, vp, sz, vp]
    L.mapmerge_extract_batch_workspace_bytes.restype = sz
    L.mapmerge_extract_batch_workspace_bytes.argtypes = [i64, i32]
    L.mapmerge_extract_batch_count.restype = C.c_int
    L.mapmerge_extract_batch_count.argtypes = [vp, i32, i32, i32, vp, vp, sz, i32, vp]
    L.mapmerge_extract_batch_write.restype = C.c_int
    L.mapmerge_extract_batch_write.argtypes = [vp, i32, i32, i32, dbl, vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, sz, vp]
    L.mapmerge_append_slice.restype = C.c_int
    L.mapmerge_append_slice.argtypes = [vp, vp, vp, i32, vp, vp, i64, vp, vp, vp, vp]
    L.mapmerge_bounds_workspace_bytes.restype = sz
    L.mapmerge_bounds.restype = C.c_int
    L.mapmerge_bounds.argtypes = [vp, vp, vp, vp, vp, sz, vp]
    L.mapmerge_voxel_workspace_bytes.restype = sz
    L.mapmerge_voxel_workspace_bytes.argtypes = [i64, i64]
    L.mapmerge_voxel_downsample.restype = C.c_int
    L.mapmerge_voxel_downsample.argtypes = [vp, vp, vp, i64, dbl, vp, vp, i64, vp, vp, vp, vp, vp, sz, vp]
    L.mapmerge_bounds_enc_reset.restype = C.c_int
    L.mapmerge_bounds_enc_reset.argtypes = [vp, vp]
    L.mapmerge_chain_workspace_bytes.restype = sz
    L.mapmerge_chain_workspace_bytes.argtypes = [vp, i32]
    L.mapmerge_chain_init.restype = C.c_int
    L.mapmerge_chain_init.argtypes = [vp, sz, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp]
    L.mapmerge_chain_run.restype = C.c_int
    L.mapmerge_chain_run.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, dbl, vp, vp, i64, vp, vp, vp]
    L.mapmerge_chain_poll.restype = C.c_int
    L.mapmerge_chain_poll.argtypes = [vp, vp, i32, vp, vp]
    L.mapmerge_chain_rebounds.restype = C.c_int
    L.mapmerge_chain_rebounds.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    L.mapmerge_chain_rebuild.restype = C.c_int
    L.mapmerge_chain_rebuild.argtypes = [vp, vp, i32, vp, vp, vp, i32, dbl, vp, vp, i64, vp, vp, vp, vp, vp, vp, sz, i64, vp]
    L.mapmerge_icp_workspace_bytes.restype = sz
    L.mapmerge_icp_workspace_bytes.argtypes = [i64, i64, i32, i32]
    L.mapmerge_icp_register.restype = C.c_int
    L.mapmerge_icp_register.argtypes = [vp, vp, i64, vp, vp, i64, dbl, dbl, dbl, i32, i32, dbl, i32, dbl, dbl, vp, vp, sz, vp]
    L.mapmerge_icp_register_batch_workspace_bytes.restype = sz
    L.mapmerge_icp_register_batch_workspace_bytes.argtypes = [i64, i64, C.c_int, i32, i32]
    L.mapmerge_icp_register_batch.restype = C.c_int
    L.mapmerge_icp_register_batch.argtypes = [vp, vp, vp, C.c_int, vp, vp, i64, dbl, dbl, dbl, i32, i32, dbl, i32, dbl, dbl,
                                              vp, vp, sz, vp]
    L.mapmerge_icp_batch_set_max_ctas.restype = C.c_int
    L.mapmerge_icp_batch_set_max_ctas.argtypes = [C.c_int]
    L.occgrid_slam_create.restype = vp
    L.occgrid_slam_create.argtypes = []
    L.occgrid_slam_destroy.restype = None
    L.occgrid_slam_destroy.argtypes = [vp]
    L.occgrid_slam_drift_table.restype = C.c_int
    L.occgrid_slam_drift_table.argtypes = [vp, vp, i64, i32, i32, vp, dbl, vp]
    L.occgrid_slam_counts.restype = C.c_int
    L.occgrid_slam_counts.argtypes = [vp, vp, vp, vp]
    L.occgrid_slam_closures.restype = C.c_int
    L.occgrid_slam_closures.argtypes = [vp, i64, vp, vp, vp, vp]
    L.occgrid_slam_correction_for_agent.restype = C.c_int
    L.occgrid_slam_correction_for_agent.argtypes = [vp, i32, vp]
    L.occgrid_accumulate_packets.restype = C.c_int
    L.occgrid_accumulate_packets.argtypes = [C.POINTER(Geom), vp, i64, i32, i32, vp, vp, vp, i32, vp, vp, sz, vp, i32, vp]
    L.occgrid_counts_to_logodds.restype = C.c_int
    L.occgrid_counts_to_logodds.argtypes = [vp, i64, dbl, dbl, dbl, dbl, vp, vp]
    L.mapmerge_rasterise.restype = C.c_int
    L.mapmerge_rasterise.argtypes = [vp, vp, vp, dbl, vp, i32, i32, vp, vp]
    L.mapmerge_fuse_max.restype = C.c_int
    L.mapmerge_fuse_max.argtypes = [vp, vp, i64, vp]
    L.mapmerge_warp_fuse_workspace_bytes.restype = sz
    L.mapmerge_warp_fuse_workspace_bytes.argtypes = [C.c_int, i32, i32]
    L.mapmerge_warp_fuse.restype = C.c_int
    L.mapmerge_warp_fuse.argtypes = [vp, C.c_int, i32, i32, dbl, vp, vp, dbl, dbl, dbl, i32, i32, vp, vp, sz, vp]
    L.occgrid_frontier_assign_workspace_bytes.restype = sz
    L.occgrid_frontier_assign_workspace_bytes.argtypes = [i32, i32, i32, i32, i64]
    L.occgrid_frontier_assign.restype = C.c_int
    L.occgrid_frontier_assign.argtypes = [vp, i32, i32, dbl, dbl, dbl, vp, i32, vp, vp, vp, vp, vp, vp, i32, i64,
                                          vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    L.occgrid_geodesic_field.restype = C.c_int
    L.occgrid_geodesic_field.argtypes = [vp, i32, i32, dbl, dbl, dbl, vp, i64, vp, vp, vp, vp, sz, vp]
    L.occgrid_distance_field_workspace_bytes.restype = sz
    L.occgrid_distance_field_workspace_bytes.argtypes = [i32, i32]
    L.occgrid_distance_field.restype = C.c_int
    L.occgrid_distance_field.argtypes = [vp, i32, i32, vp, vp, sz, vp]
    L.occgrid_inflate.restype = C.c_int
    L.occgrid_inflate.argtypes = [vp, i32, i32, dbl, dbl, dbl, i64, vp, i32, vp, vp, sz, vp]
    L.mapmerge_align_workspace_bytes.restype = sz
    L.mapmerge_align_workspace_bytes.argtypes = [C.c_int, i32, i32, i32, i32, i32, i32, i32, i64]
    L.mapmerge_align.restype = C.c_int
    L.mapmerge_align.argtypes = [vp, C.c_int, i32, i32, dbl, vp, vp, vp, i32, i32, dbl, dbl, dbl, vp, i32, i32, i32,
                                 vp, vp, vp, sz, vp]
    L.mapmerge_align_set_block.restype = C.c_int
    L.mapmerge_align_set_block.argtypes = [C.c_int]


KERNEL_NAMES = ('integrate_global', 'resolve', 'update_rays', 'tile_count', 'tile_scan', 'tile_scatter',
                'tile_raycast', 'tile_resolve', 'merge_extract', 'merge_bounds', 'merge_voxel', 'merge_raster',
                'merge_fuse', 'probe', 'route', 'frontier', 'frontier_cluster', 'chain_probe', 'chain_incremental',
                'chain_rebuild', 'icp', 'band_barrier', 'render', 'merge_scan', 'merge_warp_fuse', 'frontier_assign',
                'icp_batch', 'distance_field', 'map_align')


def profile_begin():
    check(lib().occgrid_profile_begin(), 'occgrid_profile_begin')


def profile_end():
    """-> {kernel name: (total ms, launches)} for kernels launched since profile_begin()."""
    n = len(KERNEL_NAMES)
    ms = (C.c_double * n)()
    cnt = (C.c_int64 * n)()
    check(lib().occgrid_profile_end(ms, cnt, n), 'occgrid_profile_end')
    return {KERNEL_NAMES[i]: (ms[i], cnt[i]) for i in range(n) if cnt[i]}


def check(rc, what):
    if rc != 0:
        msg = lib().occgrid_last_error().decode('utf-8', 'replace')
        raise OccGridError(f'{what} failed (rc={rc}): {msg}')


def last_error():
    return lib().occgrid_last_error().decode('utf-8', 'replace')
