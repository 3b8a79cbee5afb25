"""Drop-in surface of the reference's ``server_nodes/dual_bot_mapper.py`` hot path.

Same names, argument meaning and cell conventions as the reference (cited per item, paths
relative to the reference root), with the grid resident in B200 HBM and every update executed
by the hand-written sm_100a kernels behind ``include/occgrid_b200.h``:

* ``OccupancyGrid(size, resolution, origin_x, origin_y)``  — :110-179.  ``.grid`` reads back as
  ``np.int8 (size, size)`` indexed ``[gy, gx]`` with -1 / 0 / 100 (:92-94, :119, :150).
* ``update_ray(robot_x, robot_y, hit_x, hit_y, hit_valid)``    — :136-156 (a batch of one).
* ``update_packets(...)`` — NEW batched entry equal to running the per-packet loop body
  (:826-903) over the records in buffer order.
* ``PoseGraphSLAM`` — :244-338, host-side and sequential as in the reference; it only feeds the
  per-packet drift table (:855-857, :908-914) to the device path.

PyTorch owns the device buffers and streams; there is no CPU fallback — without the CUDA
library or a CUDA device the compute entry points raise.
"""
from __future__ import annotations

import ctypes
import dataclasses
import math
import struct

import numpy as np
import torch

from . import _native
from ._native import Geom, OccGridError

# -- protocol (:41-54) ---------------------------------------------------------
PACKET_FMT = '<4sBfffiIffffB'
PACKET_SIZE = struct.calcsize(PACKET_FMT)
PACKET_FMT_V1 = '<4sBfffiIffff'
PACKET_SIZE_V1 = struct.calcsize(PACKET_FMT_V1)
ZONE_FMT = '<4sffff'
ZONE_SIZE = struct.calcsize(ZONE_FMT)
TARGET_FMT = '<4sff'
TARGET_SIZE = struct.calcsize(TARGET_FMT)

# -- trust filter (:57-58) and sensor angles (:61-66) --------------------------
MAX_DIST_M = 1.20
MIN_DIST_M = 0.05
SENSOR_ANGLES_RAD = {'front': 0.0, 'left': math.pi / 2, 'back': math.pi, 'right': -math.pi / 2}

# -- landmark types (:69-74) ---------------------------------------------------
LM_NONE, LM_CORNER_L, LM_CORNER_R, LM_CORRIDOR, LM_DEAD_END, LM_OPEN = range(6)

# -- occupancy grid (:87-94) ---------------------------------------------------
GRID_RESOLUTION = 0.05
GRID_SIZE = 200
GRID_ORIGIN_X = -5.0
GRID_ORIGIN_Y = -5.0
CELL_UNKNOWN = -1
CELL_FREE = 0
CELL_OCCUPIED = 100

# -- frontier constants (:102-103) ---------------------------------------------
FRONTIER_MIN_CLUSTER = 3
FRONTIER_SEPARATION = 1.0

# -- dashboard colours (:346, :373) ---
BG_COLOR = (22, 33, 62)
CELL_COLOR_FREE = (30, 45, 70)

# -- SLAM constants (:97-99) ---------------------------------------------------
CLOSURE_RADIUS = 0.60
MIN_POSES_BETWEEN = 30
CLOSURE_CORRECTION = 0.5


def _require_cuda(device):
    if not torch.cuda.is_available():
        raise OccGridError('no CUDA device: the occupancy-grid engine has no CPU fallback')
    dev = torch.device(device)
    if dev.type != 'cuda':
        raise OccGridError(f'device must be a CUDA device, got {device!r}')
    return dev


def normalise_datagrams(datagrams):
    """Host batcher rule of the ingest loop (:828-838): 42-byte datagrams are v2, 41-byte ones
    v1 (landmark := LM_NONE), any other size is skipped.  Returns (uint8 [m, 42], kept indices)."""
    keep = [i for i, p in enumerate(datagrams) if len(p) in (PACKET_SIZE, PACKET_SIZE_V1)]
    arr = np.zeros((len(keep), PACKET_SIZE), np.uint8)
    for j, i in enumerate(keep):
        p = datagrams[i]
        arr[j, :len(p)] = np.frombuffer(bytes(p), np.uint8)
    return arr, np.asarray(keep, np.int64)


class OccupancyGrid:
    """2D occupancy grid for mapping (reference :110-179), resident on one B200.

    Extra keyword arguments (no reference counterpart):
      device        CUDA device (default current)
      window        (x0, y0, w, h): this object holds only that window of the global
                    ``size`` x ``size`` grid (one spatial tile of a multi-GPU map)
      strategy      'auto' | 'tiled' | 'global_atomic' — kernel family; results are identical
      max_batch     largest number of records a single ``update_packets`` call may carry
                    (sizes the device workspace once; grown on demand)
    """

    def __init__(self, size=GRID_SIZE, resolution=GRID_RESOLUTION,
                 origin_x=GRID_ORIGIN_X, origin_y=GRID_ORIGIN_Y, *,
                 device='cuda', window=None, strategy='auto', max_batch=1 << 16, lazy_workspace=False):
        self.size = int(size)
        self.res = float(resolution)
        self.ox = float(origin_x)
        self.oy = float(origin_y)
        self.device = _require_cuda(device)
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.window = tuple(int(v) for v in window) if window is not None else (0, 0, self.size, self.size)
        x0, y0, w, h = self.window
        self._geom = Geom(self.ox, self.oy, self.res, self.size, self.size, x0, y0, w, h)
        self._strategy = _native.STRATEGY[strategy]
        self._lib = _native.lib()
        with torch.cuda.device(self.device):
            self.grid_tensor = torch.full((h, w), CELL_UNKNOWN, dtype=torch.int8, device=self.device)
            self._counters = torch.zeros(_native.N_COUNTERS, dtype=torch.int64, device=self.device)
        self._ws = None
        self._ws_ray = None
        self._ws_capacity = 0
        self._host_cache = None
        self._pinned = None
        self._pinned_busy = None
        self._copy_stream = None
        self._tab_cache = None
        self._fr = None
        self._ws_assign = None
        self._ws_edt = None
        self._nav = None
        self._fa_sizes = {'pool': 4096, 'kmax': 1024}
        if not lazy_workspace:                  # (the multi-GPU band step brings its own workspace)
            self._ensure_workspace(int(max_batch))

    # ---- workspace -----------------------------------------------------------------------
    def _ensure_workspace(self, n_packets):
        if self._ws is not None and n_packets <= self._ws_capacity:
            return
        cap = max(n_packets, 1)
        nbytes = self._workspace_nbytes(cap)
        with torch.cuda.device(self.device):
            self._ws = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        self._ws_capacity = cap

    def _workspace_nbytes(self, cap):
        nbytes = self._lib.occgrid_workspace_bytes(self._geom, cap, self._strategy)
        if nbytes == 0:
            raise OccGridError('occgrid_workspace_bytes: ' + _native.last_error())
        return nbytes

    def _ray_workspace(self):
        if self._ws_ray is None:
            nbytes = self._lib.occgrid_workspace_bytes(self._geom, 0, _native.STRATEGY['global_atomic'])
            if self._strategy == _native.STRATEGY['global_atomic']:
                self._ws_ray = self._ws
            else:
                with torch.cuda.device(self.device):
                    self._ws_ray = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        return self._ws_ray

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    # ---- reference surface ---------------------------------------------------------------
    @property
    def grid(self):
        """Host view of the grid, ``np.int8 [gy, gx]`` (:119).  Synchronises and copies; the
        copy is cached until the next update.  Readers in the reference index it directly
        (renderer :512, frontiers :189-193)."""
        if self._host_cache is None:
            self._host_cache = self.grid_tensor.cpu().numpy()
        return self._host_cache

    def world_to_grid(self, wx, wy):
        """:121-125 — true division then int() truncation toward zero."""
        gx = int((wx - self.ox) / self.res)
        gy = int((wy - self.oy) / self.res)
        return gx, gy

    def grid_to_world(self, gx, gy):
        """:127-131 — cell centre."""
        wx = self.ox + (gx + 0.5) * self.res
        wy = self.oy + (gy + 0.5) * self.res
        return wx, wy

    def in_bounds(self, gx, gy):
        """:133-134"""
        return 0 <= gx < self.size and 0 <= gy < self.size

    def _bresenham(self, x0, y0, x1, y1):
        """:158-179 — host helper kept for API parity (the device walks the same line)."""
        cells = []
        dx, dy = abs(x1 - x0), abs(y1 - y0)
        sx = 1 if x0 < x1 else -1
        sy = 1 if y0 < y1 else -1
        err = dx - dy
        x, y = x0, y0
        while True:
            cells.append((x, y))
            if x == x1 and y == y1:
                return cells
            e2 = 2 * err
            if e2 > -dy:
                err -= dy
                x += sx
            if e2 < dx:
                err += dx
                y += sy

    def update_ray(self, robot_x, robot_y, hit_x, hit_y, hit_valid):
        """:136-156.  One ray = a batch of one through the same kernels."""
        rays = np.array([[robot_x, robot_y, hit_x, hit_y]], dtype=np.float64)
        self.update_rays(rays, np.array([1 if hit_valid else 0], dtype=np.uint8))

    # ---- batched entries -----------------------------------------------------------------
    def update_rays(self, rays, hit_valid):
        """Batched ``update_ray``: rays float64 [n, 4] = (robot_x, robot_y, hit_x, hit_y), applied
        in index order with the reference's last-writer-wins (:148-156)."""
        with torch.cuda.device(self.device):
            r = torch.as_tensor(rays, dtype=torch.float64).reshape(-1, 4)
            h = torch.as_tensor(hit_valid).to(torch.uint8).reshape(-1)
            if r.shape[0] != h.shape[0]:
                raise ValueError('rays and hit_valid differ in length')
            r = r.to(self.device, non_blocking=True).contiguous()
            h = h.to(self.device, non_blocking=True).contiguous()
            ws = self._ray_workspace()
            rc = self._lib.occgrid_update_rays(self._geom, r.data_ptr(), h.data_ptr(), r.shape[0],
                                               self.grid_tensor.data_ptr(), ws.data_ptr(), ws.numel(),
                                               self._counters.data_ptr(), self._strategy, self._stream())
            _native.check(rc, 'occgrid_update_rays')
        self._host_cache = None

    def _agent_table(self, separation, agent_offsets):
        if agent_offsets is None:
            # reference rule: ids {1, 2}; only agent 2 is shifted, along x (:842, :851-852)
            tab = np.array([[0.0, 0.0], [0.0, 0.0], [float(separation), 0.0]], np.float64)
        elif isinstance(agent_offsets, torch.Tensor):
            return agent_offsets.to(self.device, dtype=torch.float64).reshape(-1, 2).contiguous()
        else:
            tab = np.ascontiguousarray(agent_offsets, np.float64).reshape(-1, 2)
        cached = self._tab_cache
        if cached is not None and cached[0].shape == tab.shape and np.array_equal(cached[0], tab):
            return cached[1]                    # same table as last call: reuse the device copy
        dev_tab = torch.from_numpy(tab).to(self.device)
        self._tab_cache = (tab.copy(), dev_tab)
        return dev_tab

    def stage_packets(self, packets):
        """Host -> device staging of a record buffer.  Accepts bytes/bytearray/memoryview,
        numpy or torch uint8 ([n, stride] or flat, stride inferred as 42 for flat input), or a
        list of datagrams (normalised with the ingest rule, :828-838).  Returns
        (uint8 cuda tensor [n, stride], kept_indices or None)."""
        kept = None
        if isinstance(packets, (list, tuple)):
            packets, kept = normalise_datagrams(packets)
        if isinstance(packets, (bytes, bytearray, memoryview)):
            packets = np.frombuffer(packets, np.uint8)
        if isinstance(packets, np.ndarray):
            packets = torch.from_numpy(np.ascontiguousarray(packets, np.uint8))
        if not isinstance(packets, torch.Tensor) or packets.dtype != torch.uint8:
            raise TypeError('packets must be bytes, a uint8 array/tensor or a list of datagrams')
        if packets.dim() == 1:
            if packets.numel() % PACKET_SIZE:
                raise ValueError('flat packet buffer length is not a multiple of 42')
            packets = packets.reshape(-1, PACKET_SIZE)
        if packets.device.type != 'cuda':
            packets = packets.contiguous()
            if not packets.is_pinned():          # pageable input: one pass through a pinned staging buffer
                n = packets.numel()
                stage = self._pinned_staging(n)[:n].view(packets.shape)
                stage.copy_(packets)
                packets = stage.to(self.device, non_blocking=True)
                self._pinned_in_flight()
            else:
                packets = packets.to(self.device, non_blocking=True)
        return packets.contiguous(), kept

    def _pinned_staging(self, nbytes):
        """The reusable pinned staging buffer, safe to overwrite: the H2D copy that last read it
        (possibly still queued behind earlier kernels) has completed."""
        if self._pinned_busy is not None:
            self._pinned_busy.synchronize()
            self._pinned_busy = None
        if self._pinned is None or self._pinned.numel() < nbytes:
            self._pinned = torch.empty(max(nbytes, 1 << 16), dtype=torch.uint8).pin_memory()
        return self._pinned

    def _pinned_in_flight(self, stream=None):
        """Call right after enqueueing an async copy out of the staging buffer."""
        ev = torch.cuda.Event()
        ev.record(stream if stream is not None else torch.cuda.current_stream(self.device))
        self._pinned_busy = ev

    def update_packets(self, packets, separation=0.0, drift=None, agent_offsets=None,
                       agent_idx=None, rec_len=PACKET_SIZE):
        """Integrate a batch of QuasarPackets: equal to running the reference loop body
        (:826-903) over the records in buffer order.

        separation     ``--separation`` (:716): x offset of agent 2 (:851-852)
        drift          None or float64 [n, 2]: SLAM drift in force for each record (:855-857)
        agent_offsets  EXTENSION: float64 [A+1, 2] start offsets; ids 1..A accepted
        agent_idx      EXTENSION: int32 [n] agent index replacing the uint8 wire id
        """
        host = self._as_host_records(packets)
        if host is not None and host[0].shape[0] >= 2 * self.h2d_chunk:
            return self._update_packets_streamed(host[0], host[1], separation, drift, agent_offsets, agent_idx, rec_len)
        with torch.cuda.device(self.device):
            pk, kept = self.stage_packets(packets)
            self._integrate_device(pk, kept, separation, drift, agent_offsets, agent_idx, rec_len)

    h2d_chunk = 1 << 20          # records per H2D chunk of the streamed path (44 MB)

    def _as_host_records(self, packets):
        """(uint8 host tensor [n, stride], kept) when `packets` lives in host memory, else None."""
        kept = None
        if isinstance(packets, (list, tuple)):
            packets, kept = normalise_datagrams(packets)
        if isinstance(packets, (bytes, bytearray, memoryview)):
            packets = np.frombuffer(packets, np.uint8)
        if isinstance(packets, np.ndarray):
            packets = torch.from_numpy(np.ascontiguousarray(packets, np.uint8))
        if not isinstance(packets, torch.Tensor) or packets.dtype != torch.uint8 or packets.device.type != 'cpu':
            return None
        if packets.dim() == 1:
            if packets.numel() % PACKET_SIZE:
                raise ValueError('flat packet buffer length is not a multiple of 42')
            packets = packets.reshape(-1, PACKET_SIZE)
        return packets.contiguous(), kept

    def _update_packets_streamed(self, host, kept, separation, drift, agent_offsets, agent_idx, rec_len):
        """Large host batch: copy chunk c+1 over PCIe on a side stream while chunk c integrates.
        Chunks are applied in order, each resolving into the grid, so later records still win."""
        n, stride = host.shape
        with torch.cuda.device(self.device):
            main = torch.cuda.current_stream(self.device)
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(device=self.device)
                self._h2d = [torch.empty((self.h2d_chunk, 64), dtype=torch.uint8, device=self.device) for _ in range(2)]
                self._h2d_free = [None, None]
            if not host.is_pinned():
                self._pinned_staging(host.numel())
            d_all = torch.as_tensor(drift, dtype=torch.float64).reshape(-1, 2) if drift is not None else None
            if d_all is not None and kept is not None and d_all.shape[0] != n:
                d_all = d_all[torch.from_numpy(kept)]
            a_all = torch.as_tensor(agent_idx, dtype=torch.int32).reshape(-1) if agent_idx is not None else None
            for c, lo in enumerate(range(0, n, self.h2d_chunk)):
                hi = min(n, lo + self.h2d_chunk)
                slot = c & 1
                src = host[lo:hi]
                if not src.is_pinned():
                    stage = self._pinned[lo * stride:hi * stride].view(hi - lo, stride)
                    stage.copy_(src)
                    src = stage
                dst = self._h2d[slot].view(-1)[:(hi - lo) * stride].view(hi - lo, stride)
                with torch.cuda.stream(self._copy_stream):
                    if self._h2d_free[slot] is not None:
                        self._copy_stream.wait_event(self._h2d_free[slot])
                    dst.copy_(src, non_blocking=True)
                    ready = torch.cuda.Event()
                    ready.record(self._copy_stream)
                    if not host.is_pinned():
                        self._pinned_busy = ready         # the staging buffer is free once the last chunk has left it
                main.wait_event(ready)
                self._integrate_device(dst, None, separation, None if d_all is None else d_all[lo:hi], agent_offsets,
                                       None if a_all is None else a_all[lo:hi], rec_len)
                done = torch.cuda.Event()
                done.record(main)
                self._h2d_free[slot] = done

    def _integrate_device(self, pk, kept, separation, drift, agent_offsets, agent_idx, rec_len):
        with torch.cuda.device(self.device):
            n, stride = pk.shape
            if n == 0:
                return
            self._ensure_workspace(n)
            tab = self._agent_table(separation, agent_offsets)
            d_ptr = None
            if drift is not None:
                d = torch.as_tensor(drift, dtype=torch.float64)
                if kept is not None and d.shape[0] != n:
                    d = d[torch.from_numpy(kept)]
                d = d.reshape(n, 2).to(self.device, non_blocking=True).contiguous()
                d_ptr = d.data_ptr()
            a_ptr = None
            if agent_idx is not None:
                a = torch.as_tensor(agent_idx, dtype=torch.int32).reshape(n).to(self.device, non_blocking=True).contiguous()
                a_ptr = a.data_ptr()
            if self._accumulating:          # hit/miss count planes instead of the last-writer-wins grid
                rc = self._lib.occgrid_accumulate_packets(
                    self._geom, pk.data_ptr(), n, stride, rec_len, a_ptr, d_ptr, tab.data_ptr(), tab.shape[0] - 1,
                    self.counts_tensor.data_ptr(), self._ws.data_ptr(), self._ws.numel(),
                    self._counters.data_ptr(), self._strategy, self._stream())
                _native.check(rc, 'occgrid_accumulate_packets')
                return
            self._launch_packets(pk, rec_len, a_ptr, d_ptr, tab)
        self._host_cache = None

    def _launch_packets(self, pk, rec_len, a_ptr, d_ptr, tab):
        n, stride = pk.shape
        rc = self._lib.occgrid_integrate_packets(
            self._geom, pk.data_ptr(), n, stride, rec_len, a_ptr, d_ptr, tab.data_ptr(), tab.shape[0] - 1,
            self.grid_tensor.data_ptr(), self._ws.data_ptr(), self._ws.numel(),
            self._counters.data_ptr(), self._strategy, self._stream())
        _native.check(rc, 'occgrid_integrate_packets')

    # ---- extension: hit/miss counts and log-odds (no reference counterpart) -------------------
    _accumulating = False
    _counts = None

    @property
    def counts_tensor(self):
        """int32 [h, w, 2] device tensor, ``[..., 0]`` misses, ``[..., 1]`` hits (allocated on first use)."""
        if self._counts is None:
            h, w = self.grid_tensor.shape
            self._counts = torch.zeros((h, w, 2), dtype=torch.int32, device=self.device)
        return self._counts

    def accumulate_packets(self, packets, separation=0.0, drift=None, agent_offsets=None, agent_idx=None, rec_len=PACKET_SIZE):
        """EXTENSION (north-star wording; the reference keeps no counts): same decode, pose
        correction, beam expansion, ``_bresenham`` cells and per-cell clipping as
        ``update_packets``, but instead of storing FREE / OCCUPIED (:148-156) every FREE store
        counts one miss and every OCCUPIED store one hit.  Integer adds commute, so the planes
        equal ``np.add.at`` over the reference's cells; they accumulate across calls."""
        self._accumulating = True
        try:
            self.update_packets(packets, separation=separation, drift=drift, agent_offsets=agent_offsets,
                                agent_idx=agent_idx, rec_len=rec_len)
        finally:
            self._accumulating = False

    hit_counts = property(lambda self: self.counts_tensor[..., 1].cpu().numpy())
    miss_counts = property(lambda self: self.counts_tensor[..., 0].cpu().numpy())

    def reset_counts(self):
        if self._counts is not None:
            self._counts.zero_()

    def log_odds(self, l_occ=0.85, l_free=-0.4, l_min=-2.0, l_max=3.5, to_host=True):
        """float32 [h, w]: clamp(hits * l_occ + misses * l_free, l_min, l_max), evaluated from the
        integer planes (order-independent; equal to the float64 NumPy evaluation rounded to float32)."""
        with torch.cuda.device(self.device):
            h, w = self.grid_tensor.shape
            out = torch.empty((h, w), dtype=torch.float32, device=self.device)
            rc = self._lib.occgrid_counts_to_logodds(self.counts_tensor.data_ptr(), h * w, float(l_occ), float(l_free),
                                                     float(l_min), float(l_max), out.data_ptr(), self._stream())
            _native.check(rc, 'occgrid_counts_to_logodds')
        return out.cpu().numpy() if to_host else out

    def update_poses(self, pose_recs, ordinals_in_records=False):
        """Integrate decoded records (uint8 cuda tensor [n, 48] of ``occgrid_pose_rec``) — the
        receiving side of the multi-GPU routing.  Order = index (``occgrid_route_packets`` +
        all-to-all) or the ordinal carried in each record (``occgrid_route_packets_p2p``)."""
        with torch.cuda.device(self.device):
            if not (isinstance(pose_recs, torch.Tensor) and pose_recs.dtype == torch.uint8 and pose_recs.is_cuda
                    and pose_recs.dim() == 2 and pose_recs.shape[1] == 48):
                raise TypeError('pose_recs must be a uint8 CUDA tensor [n, 48]')
            pose_recs = pose_recs.contiguous()
            n = pose_recs.shape[0]
            if n == 0:
                return
            self._ensure_workspace(n)
            rc = self._lib.occgrid_integrate_poses(self._geom, pose_recs.data_ptr(), n, 1 if ordinals_in_records else 0,
                                                   self.grid_tensor.data_ptr(),
                                                   self._ws.data_ptr(), self._ws.numel(), self._counters.data_ptr(),
                                                   self._strategy, self._stream())
            _native.check(rc, 'occgrid_integrate_poses')
        self._host_cache = None

    # ---- frontiers (:181-237) — SURVEY §8 row f1 -------------------------------------------
    def _frontier_buffers(self, capacity):
        if self.window != (0, 0, self.size, self.size):
            raise OccGridError('frontier detection needs the whole grid (not a window of it)')
        if self._fr is None or self._fr['cap'] < capacity:
            n = self.size * self.size
            nb = self._lib.occgrid_frontier_workspace_bytes(n, capacity)
            with torch.cuda.device(self.device):
                self._fr = {
                    'cap': capacity,
                    'xy': torch.empty((capacity, 2), dtype=torch.int32, device=self.device),
                    'count': torch.zeros(1, dtype=torch.int64, device=self.device),
                    'status': torch.zeros(1, dtype=torch.int32, device=self.device),
                    'ws': torch.empty(nb, dtype=torch.uint8, device=self.device),
                    'label': torch.empty(capacity, dtype=torch.int32, device=self.device),
                    'root': torch.empty(capacity, dtype=torch.int32, device=self.device),
                    'size': torch.empty(capacity, dtype=torch.int32, device=self.device),
                    'cent': torch.empty((capacity, 2), dtype=torch.float64, device=self.device),
                    'ncl': torch.zeros(1, dtype=torch.int64, device=self.device),
                }
        return self._fr

    def _launch_frontiers(self, f):
        with torch.cuda.device(self.device):
            rc = self._lib.occgrid_frontiers(self.grid_tensor.data_ptr(), self.size, self.size, f['xy'].data_ptr(), f['cap'],
                                             f['count'].data_ptr(), f['status'].data_ptr(), f['ws'].data_ptr(), f['ws'].numel(),
                                             self._stream())
            _native.check(rc, 'occgrid_frontiers')

    def _detect_frontiers(self):
        """Runs the frontier stencil on the device; returns (buffers, count)."""
        cap = max(1 << 16, self.size * 8)
        while True:
            f = self._frontier_buffers(cap)
            self._launch_frontiers(f)
            with torch.cuda.device(self.device):
                host = torch.cat([f['count'], f['status'].to(torch.int64)]).cpu().tolist()
            if host[1] & 1:                       # more frontier cells than the buffer holds: grow and redo
                f['status'].zero_()
                cap *= 4
                continue
            return f, int(host[0])

    def get_frontiers(self):
        """:181-197 — FREE interior cells with an UNKNOWN 4-neighbour, as (gx, gy) tuples in the
        reference's row-major scan order."""
        f, n = self._detect_frontiers()
        xy = f['xy'][:n].cpu().numpy()
        return [(int(x), int(y)) for x, y in xy]

    def _launch_clusters(self, f, min_cluster):
        """Enqueues the stencil and the clustering into the buffers ``f``."""
        self._launch_frontiers(f)
        with torch.cuda.device(self.device):
            rc = self._lib.occgrid_frontier_clusters(
                f['xy'].data_ptr(), f['count'].data_ptr(), f['cap'], self.size, int(min_cluster), self.ox, self.oy, self.res,
                f['label'].data_ptr(), f['root'].data_ptr(), f['size'].data_ptr(), f['cent'].data_ptr(), f['ncl'].data_ptr(),
                f['ws'].data_ptr(), f['ws'].numel(), self._stream())
            _native.check(rc, 'occgrid_frontier_clusters')

    def _cluster(self, min_cluster=FRONTIER_MIN_CLUSTER):
        """Stencil + clustering enqueued back to back (the cluster kernels take the frontier count
        from device memory), then ONE host read of (count, status, clusters)."""
        cap = max(1 << 16, self.size * 8)
        if self._fr is not None:
            cap = max(cap, self._fr['cap'])
        while True:
            f = self._frontier_buffers(cap)
            self._launch_clusters(f, min_cluster)
            with torch.cuda.device(self.device):
                host = torch.cat([f['count'], f['status'].to(torch.int64), f['ncl']]).cpu().tolist()
            if host[1] & 1:                       # the list overflowed (count was forced to 0): grow and redo
                f['status'].zero_()
                cap *= 4
                continue
            return f, int(host[0]), int(host[2])

    def cluster_frontiers(self, frontier_cells=None):
        """:199-231 — 4-connected components of the current frontier set, in the reference's
        cluster order (by first cell), clusters below FRONTIER_MIN_CLUSTER dropped.  Cells inside a
        cluster are listed in scan order (the reference lists them in BFS order; only the centroid
        is consumed downstream, :953).  ``frontier_cells`` is accepted for signature parity and
        must be the list ``get_frontiers()`` returns for the current grid."""
        f, n, k = self._cluster()
        if frontier_cells is not None and len(frontier_cells) != n:
            raise ValueError('frontier_cells does not match the current grid (use get_frontiers())')
        if k == 0:
            return []
        xy = f['xy'][:n].cpu().numpy()
        label = f['label'][:n].cpu().numpy()
        roots = f['root'][:k].cpu().numpy()
        order = np.argsort(label, kind='stable')
        starts = np.searchsorted(label[order], roots, side='left')
        sizes = f['size'][:k].cpu().numpy()
        return [[(int(x), int(y)) for x, y in xy[order[s:s + c]]] for s, c in zip(starts, sizes)]

    def cluster_centroid_world(self, cluster):
        """:233-237"""
        avg_x = sum(c[0] for c in cluster) / len(cluster)
        avg_y = sum(c[1] for c in cluster) / len(cluster)
        return self.grid_to_world(avg_x, avg_y)

    def frontier_centroids(self):
        """The periodic step of main() (:950-954) in one device pass: get_frontiers ->
        cluster_frontiers -> [cluster_centroid_world(c) for c in clusters]."""
        f, n, k = self._cluster()
        return [(float(x), float(y)) for x, y in f['cent'][:k].cpu().numpy()]

    # ---- frontier assignment (EXTENSION; the reference's is commented out, :958-996) ---------------
    def _robot_positions(self, robot_xy, who):
        xy = np.ascontiguousarray(np.asarray(robot_xy, dtype=np.float64))
        if xy.ndim != 2 or xy.shape[1] != 2:
            raise ValueError(f'{who}: robot_xy must be [A, 2] world positions, got shape {xy.shape}')
        if not 1 <= xy.shape[0] <= MAX_ASSIGN_ROBOTS:
            raise ValueError(f'{who}: {xy.shape[0]} robots, need 1..{MAX_ASSIGN_ROBOTS}')
        if self.window != (0, 0, self.size, self.size):
            raise OccGridError(f'{who} needs the whole grid (not a window of it)')
        with torch.cuda.device(self.device):
            return torch.from_numpy(xy).to(self.device)

    def _assign_workspace(self, n_robots, max_clusters, tile_pool):
        nb = self._lib.occgrid_frontier_assign_workspace_bytes(self.size, self.size, n_robots, max_clusters, tile_pool)
        if nb == 0:
            raise OccGridError('occgrid_frontier_assign_workspace_bytes: ' + _native.last_error())
        if self._ws_assign is None or self._ws_assign.numel() < nb:
            self._ws_assign = None
            with torch.cuda.device(self.device):
                self._ws_assign = torch.empty(nb, dtype=torch.uint8, device=self.device)
        return self._ws_assign

    def assign_frontiers(self, robot_xy, min_cluster=FRONTIER_MIN_CLUSTER, robot_radius=None):
        """EXTENSION: one exploration target per robot by geodesic distance over the known free
        space (``occgrid_frontier_assign`` in include/occgrid_b200.h gives the exact rules).

        robot_xy  [A, 2] world positions, 1 <= A <= 65 535; a robot outside the grid or at a
                  non-finite position has no source and gets no target.
        Runs the frontier stencil, the clustering (``min_cluster`` as ``cluster_frontiers``) and the
        assignment back to back on the device and reads the result once.  Returns a
        ``FrontierAssignment``: robot a takes cluster ``cluster[a]`` (``frontier_centroids()``
        order, -1 for none) at path length ``cost[a]`` cells, reaching it first at cell ``goal[a]``;
        ``target_xy[a]`` is that cluster's centroid (NaN for none) and ``costs[a, k]`` robot a's
        path length to cluster k (-1 when unreachable).  The tile pool grows until it holds every
        field.

        robot_radius  None (a robot is a point) or metres >= 0: the stencil and the clustering still
                  run on ``grid_tensor``, and the paths run over ``navigation_grid(robot_radius,
                  robot_xy)``, so they keep that clearance from every obstacle except inside the
                  robots' own footprints."""
        max_d2 = None if robot_radius is None else self._max_d2(robot_radius, 'assign_frontiers')
        d_xy = self._robot_positions(robot_xy, 'assign_frontiers')
        A = d_xy.shape[0]
        n_tiles = ((self.size + 63) // 64) ** 2
        st = self._fa_sizes
        cap = max(1 << 16, self.size * 8, self._fr['cap'] if self._fr is not None else 0)
        dev = self.device
        while True:
            pool = min(max(st['pool'], 16 * A), A * n_tiles)       # A * n_tiles slots can never run out
            kmax = st['kmax']
            f = self._frontier_buffers(cap)
            ws = self._assign_workspace(A, kmax, pool)
            with torch.cuda.device(dev):
                out = {'cluster': torch.empty(A, dtype=torch.int32, device=dev),
                       'cost': torch.empty(A, dtype=torch.int32, device=dev),
                       'goal': torch.empty((A, 2), dtype=torch.int32, device=dev),
                       'target_xy': torch.empty((A, 2), dtype=torch.float64, device=dev),
                       'costs': torch.empty((A, kmax), dtype=torch.int32, device=dev)}
                hdr = torch.zeros(8, dtype=torch.int64, device=dev)     # count, frontier status, n_clusters, status, stats[3]
                status = torch.zeros(1, dtype=torch.int32, device=dev)
                self._launch_clusters(f, min_cluster)
                paths = self.grid_tensor if max_d2 is None else self._launch_inflate(max_d2, d_xy)
                rc = self._lib.occgrid_frontier_assign(
                    paths.data_ptr(), self.size, self.size, self.ox, self.oy, self.res, d_xy.data_ptr(), A,
                    f['xy'].data_ptr(), f['count'].data_ptr(), f['label'].data_ptr(), f['root'].data_ptr(), f['cent'].data_ptr(),
                    f['ncl'].data_ptr(), kmax, pool, out['cluster'].data_ptr(), out['cost'].data_ptr(), out['goal'].data_ptr(),
                    out['target_xy'].data_ptr(), out['costs'].data_ptr(), status.data_ptr(), hdr[4:7].data_ptr(),
                    ws.data_ptr(), ws.numel(), self._stream())
                _native.check(rc, 'occgrid_frontier_assign')
                hdr[0:1].copy_(f['count'])
                hdr[1:2].copy_(f['status'])
                hdr[2:3].copy_(f['ncl'])
                hdr[3:4].copy_(status)
                host = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in out.items()}
                host['hdr'] = torch.empty(8, dtype=torch.int64, pin_memory=True)
                host['hdr'].copy_(hdr, non_blocking=True)
                for k, v in out.items():
                    host[k].copy_(v, non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()          # the one host read
            count, fstatus, ncl, astatus, rounds, items, slots = host['hdr'][:7].tolist()
            if fstatus & 1:                       # the frontier list overflowed: grow and redo
                f['status'].zero_()
                cap *= 4
                continue
            if astatus & 2:
                raise OccGridError('occgrid_frontier_assign: a grid barrier of the worklist kernel timed out')
            if astatus & 1:                       # the tile pool ran out: grow and redo
                st['pool'] = pool * 4
                continue
            if astatus & 4:                       # more clusters than columns: widen and redo
                st['kmax'] = 1 << int(ncl - 1).bit_length()
                continue
            return FrontierAssignment(host['cluster'].numpy(), host['cost'].numpy(), host['goal'].numpy(),
                                      host['target_xy'].numpy(), host['costs'].numpy()[:, :ncl].copy(),
                                      {'frontier_cells': count, 'clusters': ncl, 'rounds': rounds, 'items': items,
                                       'tile_slots': slots, 'tile_pool': pool})

    def geodesic_distance(self, robot_xy, to_host=True, robot_radius=None):
        """EXTENSION: the geodesic field of one robot at world position ``robot_xy`` = (x, y):
        int32 [size, size] indexed [gy, gx], the 4-connected path length in cells over FREE cells
        from the robot's cell (0 there whatever its value), -1 where unreachable or when the robot
        is outside the grid.  For navigation: descend the field from a goal cell to the robot.
        With ``robot_radius`` (metres >= 0) the field runs over ``navigation_grid(robot_radius,
        robot_xy)``: a robot of that radius can follow it."""
        max_d2 = None if robot_radius is None else self._max_d2(robot_radius, 'geodesic_distance')
        xy = np.asarray(robot_xy, np.float64)
        if xy.size != 2:
            raise ValueError(f'geodesic_distance: robot_xy must be one (x, y) world position, got shape {xy.shape}')
        d_xy = self._robot_positions(xy.reshape(1, 2), 'geodesic_distance')
        pool = ((self.size + 63) // 64) ** 2                 # every tile: the pool cannot run out
        ws = self._assign_workspace(1, 1, pool)
        with torch.cuda.device(self.device):
            field = torch.empty((self.size, self.size), dtype=torch.int32, device=self.device)
            status = torch.zeros(1, dtype=torch.int32, device=self.device)
            paths = self.grid_tensor if max_d2 is None else self._launch_inflate(max_d2, d_xy)
            rc = self._lib.occgrid_geodesic_field(paths.data_ptr(), self.size, self.size, self.ox, self.oy, self.res,
                                                  d_xy.data_ptr(), pool, field.data_ptr(), status.data_ptr(), None,
                                                  ws.data_ptr(), ws.numel(), self._stream())
            _native.check(rc, 'occgrid_geodesic_field')
            if int(status.item()) != 0:
                raise OccGridError(f'occgrid_geodesic_field: status {int(status.item())} (worklist failed)')
        return field.cpu().numpy() if to_host else field

    # ---- obstacle clearance (EXTENSION) -------------------------------------------------------
    def _max_d2(self, robot_radius, who):
        """The one conversion of a robot radius: max_d2 = floor((robot_radius / res) ** 2) in fp64,
        so a cell is blocked when an obstacle's centre lies within robot_radius of its centre."""
        r = float(robot_radius)
        if not (math.isfinite(r) and r >= 0.0):
            raise ValueError(f'{who}: robot_radius must be finite and >= 0, got {robot_radius!r}')
        q = r / self.res
        q = q * q                                              # (r / res) ** 2, inf rather than OverflowError
        return (1 << 62) if q >= 2.0 ** 62 else math.floor(q)   # past 2 * 32767^2 every value blocks the same

    def _edt_workspace(self):
        if self.window != (0, 0, self.size, self.size):
            raise OccGridError('the distance field needs the whole grid (not a window of it)')
        nb = self._lib.occgrid_distance_field_workspace_bytes(self.size, self.size)
        if nb == 0:
            raise OccGridError('occgrid_distance_field_workspace_bytes: ' + _native.last_error())
        if self._ws_edt is None or self._ws_edt.numel() < nb:
            self._ws_edt = None
            with torch.cuda.device(self.device):
                self._ws_edt = torch.empty(nb, dtype=torch.uint8, device=self.device)
        return self._ws_edt

    def _launch_inflate(self, max_d2, d_xy, out=None):
        """Enqueues occgrid_inflate of grid_tensor with the robots d_xy ([A, 2] on the device or None)
        into ``out``, by default the cached navigation buffer; returns it."""
        ws = self._edt_workspace()
        with torch.cuda.device(self.device):
            if out is None:
                if self._nav is None:
                    self._nav = torch.empty((self.size, self.size), dtype=torch.int8, device=self.device)
                out = self._nav
            A = 0 if d_xy is None else int(d_xy.shape[0])
            rc = self._lib.occgrid_inflate(self.grid_tensor.data_ptr(), self.size, self.size, self.ox, self.oy, self.res,
                                           int(max_d2), d_xy.data_ptr() if A else None, A, out.data_ptr(),
                                           ws.data_ptr(), ws.numel(), self._stream())
            _native.check(rc, 'occgrid_inflate')
        return out

    def distance_field(self, to_host=True):
        """EXTENSION: the exact squared Euclidean distance from every cell to the nearest obstacle
        (a cell > 50), int32 [size, size] indexed [gy, gx], in cells between cell centres: 0 on
        obstacles, and -1 everywhere when the grid has no obstacle.  The clearance in metres is
        ``sqrt(d2) * res``."""
        ws = self._edt_workspace()
        with torch.cuda.device(self.device):
            d2 = torch.empty((self.size, self.size), dtype=torch.int32, device=self.device)
            rc = self._lib.occgrid_distance_field(self.grid_tensor.data_ptr(), self.size, self.size, d2.data_ptr(),
                                                  ws.data_ptr(), ws.numel(), self._stream())
            _native.check(rc, 'occgrid_distance_field')
        return d2.cpu().numpy() if to_host else d2

    def navigation_grid(self, robot_radius, robot_xy=None, to_host=True):
        """EXTENSION: the grid a robot of ``robot_radius`` metres can plan on, int8 [size, size]:
        every FREE cell whose centre lies within robot_radius of an obstacle's centre becomes
        OCCUPIED (max_d2 = floor((robot_radius / res) ** 2) cells^2), except in the footprints of the
        robots at ``robot_xy`` ([A, 2] world metres, 0 <= A <= 65 535, or None), so that a robot
        standing closer than its radius to a wall can still leave.  Other cells keep their value."""
        max_d2 = self._max_d2(robot_radius, 'navigation_grid')
        d_xy = None
        if robot_xy is not None:
            xy = np.ascontiguousarray(np.asarray(robot_xy, dtype=np.float64))
            if xy.ndim != 2 or xy.shape[1] != 2 or xy.shape[0] > MAX_ASSIGN_ROBOTS:
                raise ValueError(f'navigation_grid: robot_xy must be [A, 2] world positions with A <= {MAX_ASSIGN_ROBOTS}, '
                                 f'got shape {xy.shape}')
            if xy.shape[0]:
                with torch.cuda.device(self.device):
                    d_xy = torch.from_numpy(xy).to(self.device)
        with torch.cuda.device(self.device):
            out = torch.empty((self.size, self.size), dtype=torch.int8, device=self.device)
        self._launch_inflate(max_d2, d_xy, out)
        return out.cpu().numpy() if to_host else out

    # ---- overlay render (:492-527) — SURVEY §8 row f4 -----------------------------------------
    def render_overlay(self, width=1000, height=800, scale=100.0, offset_x=None, offset_y=None,
                       background=BG_COLOR, color=CELL_COLOR_FREE, to_host=True):
        """Headless ``MapRenderer._draw_occupancy``: an RGB image uint8 [height, width, 3] of the
        view the dashboard would show (``scale`` pixels per metre, ``offset_x/_y`` = screen position
        of the world origin, defaults = the renderer's start view :395-397): ``background`` with
        every visible cell that is neither UNKNOWN nor OCCUPIED painted ``color`` (:513-521)."""
        if self.window != (0, 0, self.size, self.size):
            raise OccGridError('render_overlay needs the whole grid (not a window of it)')
        offset_x = width / 2 if offset_x is None else offset_x
        offset_y = height / 2 if offset_y is None else offset_y
        bg = (ctypes.c_uint8 * 3)(*[int(c) for c in background])
        fg = (ctypes.c_uint8 * 3)(*[int(c) for c in color])
        with torch.cuda.device(self.device):
            out = torch.empty((int(height), int(width), 3), dtype=torch.uint8, device=self.device)
            rc = self._lib.occgrid_render_overlay(self.grid_tensor.data_ptr(), self.size, self.size, self.ox, self.oy, self.res,
                                                  float(scale), float(offset_x), float(offset_y), int(width), int(height),
                                                  bg, fg, out.data_ptr(), self._stream())
            _native.check(rc, 'occgrid_render_overlay')
        return out.cpu().numpy() if to_host else out

    # ---- bookkeeping ---------------------------------------------------------------------
    def counters(self, reset=False):
        """Device-side statistics (see the OCCGRID_C_* enum)."""
        vals = self._counters.cpu().tolist()
        if reset:
            self._counters.zero_()
        return {k: int(v) for k, v in zip(_native.COUNTER_NAMES, vals)}

    def clear(self):
        self.grid_tensor.fill_(CELL_UNKNOWN)
        self._host_cache = None


MAX_ASSIGN_ROBOTS = 65535


@dataclasses.dataclass(frozen=True)
class FrontierAssignment:
    """Result of ``OccupancyGrid.assign_frontiers`` for A robots and K clusters (NumPy arrays)."""
    cluster: np.ndarray      # int32 [A]: assigned cluster in frontier_centroids() order, -1 for none
    cost: np.ndarray         # int32 [A]: path length in cells to the cluster's nearest cell, -1 for none
    goal: np.ndarray         # int32 [A, 2]: (gx, gy) of that cell (lowest y * size + x on ties), -1 for none
    target_xy: np.ndarray    # float64 [A, 2]: the cluster's centroid in world metres, NaN for none
    costs: np.ndarray        # int32 [A, K]: path length from robot a to cluster k, -1 when unreachable
    stats: dict              # frontier cells, clusters, worklist rounds, (robot, tile) items, tile slots used, pool


def target_packets(result):
    """``TARGET_FMT`` datagrams (b'TARG', x, y as float32) for the robots of ``result`` that have a
    target, keyed by agent id: robot a of the ``assign_frontiers`` call is agent a + 1."""
    return {a + 1: struct.pack(TARGET_FMT, b'TARG', float(x), float(y))
            for a, (k, (x, y)) in enumerate(zip(result.cluster.tolist(), result.target_xy.tolist())) if k >= 0}


def _single_map_only(name):
    def method(self, *args, **kwargs):
        raise OccGridError(f'AgentGrids.{name}: single-map operation; run it on an OccupancyGrid built from grid(agent_id)')
    method.__name__ = name
    return method


class AgentGrids(OccupancyGrid):
    """EXTENSION: one occupancy grid per agent, integrated from ONE packet stream on the device.

    The reference's multi-agent architecture maps every robot in its own frame (``/agent_{id}/map``)
    and lets ``map_merger.py`` register and fuse the maps.  ``update_packets`` takes the same input
    as ``OccupancyGrid.update_packets`` (and streams large host batches the same way); grid a - 1 of
    the stack ends equal to ``OccupancyGrid.update_packets`` run over only the records of agent a.

      grids_tensor  int8 [n_agents, size, size] on the device, agent a at index a - 1
      origins       float64 [n_agents, 2], every row (origin_x, origin_y); ``res`` the resolution

    The stack is what ``MapMerger.merge(maps.grids_tensor, maps.origins, maps.res, transforms)``
    takes, without a copy.  All maps share one geometry.  ``agent_offsets`` must have n_agents + 1
    rows; the default is zero except row 2 = (separation, 0) (:851-852), so with separation = 0
    every agent maps in its own odometry frame.  Single-map operations (rays, pose records, counts,
    frontiers, rendering) raise ``OccGridError``.  For frontiers on the swarm's map,
    ``MapMerger().fuse_occupancy(maps.grids_tensor, maps.origins, maps.res, transforms, target)``
    fuses the stack into an ``OccupancyGrid`` that keeps free space; ``target.frontier_centroids()``
    and ``target.assign_frontiers(robot_xy)`` then run there.  Transforms that drift are refined
    first against the previous fused map, in one call for all agents: the loop is
    ``maps -> register_maps(grids_tensor, origins, res, priors, reference=last_fused) ->
    fuse_occupancy(..., result.transformation, target) -> assign_frontiers``.
    """

    def __init__(self, n_agents=2, size=GRID_SIZE, resolution=GRID_RESOLUTION,
                 origin_x=GRID_ORIGIN_X, origin_y=GRID_ORIGIN_Y, *,
                 device='cuda', strategy='auto', max_batch=1 << 16):
        self.n_agents = int(n_agents)
        if self.n_agents < 1:
            raise ValueError('n_agents must be >= 1')
        super().__init__(size, resolution, origin_x, origin_y, device=device, strategy=strategy, lazy_workspace=True)
        del self.grid_tensor
        with torch.cuda.device(self.device):
            self.grids_tensor = torch.full((self.n_agents, self.size, self.size), CELL_UNKNOWN, dtype=torch.int8,
                                           device=self.device)
        self.origins = np.tile(np.array([[self.ox, self.oy]], np.float64), (self.n_agents, 1))
        self._ensure_workspace(int(max_batch))

    def _workspace_nbytes(self, cap):
        nbytes = self._lib.occgrid_agent_maps_workspace_bytes(self._geom, self.n_agents, cap, self._strategy)
        if nbytes == 0:
            raise OccGridError('occgrid_agent_maps_workspace_bytes: ' + _native.last_error())
        return nbytes

    def _agent_table(self, separation, agent_offsets):
        if agent_offsets is None:
            agent_offsets = np.zeros((self.n_agents + 1, 2), np.float64)
            if self.n_agents >= 2:
                agent_offsets[2, 0] = float(separation)
        tab = super()._agent_table(separation, agent_offsets)
        if tab.shape[0] != self.n_agents + 1:
            raise ValueError(f'agent_offsets has {tab.shape[0]} rows, need n_agents + 1 = {self.n_agents + 1}')
        return tab

    def _launch_packets(self, pk, rec_len, a_ptr, d_ptr, tab):
        n, stride = pk.shape
        rc = self._lib.occgrid_integrate_packets_agent_maps(
            self._geom, pk.data_ptr(), n, stride, rec_len, a_ptr, d_ptr, tab.data_ptr(), self.n_agents,
            self.grids_tensor.data_ptr(), self._ws.data_ptr(), self._ws.numel(),
            self._counters.data_ptr(), self._strategy, self._stream())
        _native.check(rc, 'occgrid_integrate_packets_agent_maps')

    def grid(self, agent_id):
        """Host copy of agent ``agent_id``'s map, ``np.int8 [gy, gx]``, cached until the next update."""
        a = int(agent_id)
        if not 1 <= a <= self.n_agents:
            raise ValueError(f'agent_id {a} outside 1..{self.n_agents}')
        if self._host_cache is None:
            self._host_cache = {}
        if a not in self._host_cache:
            self._host_cache[a] = self.grids_tensor[a - 1].cpu().numpy()
        return self._host_cache[a]

    @property
    def grids(self):
        """Host copy of the stack, ``np.int8 [n_agents, size, size]``, cached until the next update."""
        if self._host_cache is None:
            self._host_cache = {}
        if 'all' not in self._host_cache:
            self._host_cache['all'] = self.grids_tensor.cpu().numpy()
        return self._host_cache['all']

    def clear(self):
        self.grids_tensor.fill_(CELL_UNKNOWN)
        self._host_cache = None

    update_ray = _single_map_only('update_ray')
    update_rays = _single_map_only('update_rays')
    update_poses = _single_map_only('update_poses')
    accumulate_packets = _single_map_only('accumulate_packets')
    log_odds = _single_map_only('log_odds')
    reset_counts = _single_map_only('reset_counts')
    counts_tensor = property(_single_map_only('counts_tensor'))
    hit_counts = property(_single_map_only('hit_counts'))
    miss_counts = property(_single_map_only('miss_counts'))
    get_frontiers = _single_map_only('get_frontiers')
    cluster_frontiers = _single_map_only('cluster_frontiers')
    frontier_centroids = _single_map_only('frontier_centroids')
    assign_frontiers = _single_map_only('assign_frontiers')
    geodesic_distance = _single_map_only('geodesic_distance')
    distance_field = _single_map_only('distance_field')
    navigation_grid = _single_map_only('navigation_grid')
    render_overlay = _single_map_only('render_overlay')


class PoseNode:
    """:244-258"""
    __slots__ = ('x', 'y', 'yaw', 'agent_id', 'landmark_type', 'timestamp', 'index',
                 'corrected_x', 'corrected_y')

    def __init__(self, x, y, yaw, agent_id, landmark_type, timestamp, index):
        self.x, self.y, self.yaw = x, y, yaw
        self.agent_id, self.landmark_type = agent_id, landmark_type
        self.timestamp, self.index = timestamp, index
        self.corrected_x, self.corrected_y = x, y


class PoseGraphSLAM:
    """Landmark loop closure (:261-338).  Sequential host logic, as in the reference: the hot
    path only consumes its output as the per-packet drift table."""

    def __init__(self, verbose=False):
        self.nodes = []
        self.landmarks = []
        self.closures = []
        self.last_closure_idx = {1: -MIN_POSES_BETWEEN, 2: -MIN_POSES_BETWEEN}
        self.verbose = verbose

    def add_pose(self, x, y, yaw, agent_id, landmark_type, timestamp):
        idx = len(self.nodes)
        node = PoseNode(x, y, yaw, agent_id, landmark_type, timestamp, idx)
        self.nodes.append(node)
        if landmark_type == LM_NONE:
            return False, 0.0, 0.0
        result = self._check_closure(node)
        self.landmarks.append((x, y, landmark_type, idx))
        return result

    def _check_closure(self, node):
        recent = node.index - self.last_closure_idx.get(node.agent_id, -999) < MIN_POSES_BETWEEN
        for lm_x, lm_y, lm_type, lm_idx in self.landmarks:
            if lm_type != node.landmark_type or node.index - lm_idx < MIN_POSES_BETWEEN or recent:
                continue
            dist = math.sqrt((node.x - lm_x) ** 2 + (node.y - lm_y) ** 2)
            if dist < CLOSURE_RADIUS:
                corr_dx = (lm_x - node.x) * CLOSURE_CORRECTION
                corr_dy = (lm_y - node.y) * CLOSURE_CORRECTION
                self.closures.append((lm_idx, node.index, corr_dx, corr_dy))
                self.last_closure_idx[node.agent_id] = node.index
                if self.verbose:
                    print(f'[SLAM] LOOP CLOSURE! Agent {node.agent_id} | Dist: {dist:.2f}m | '
                          f'Correction: ({corr_dx:.3f}, {corr_dy:.3f})')
                return True, corr_dx, corr_dy
        return False, 0.0, 0.0

    def get_correction_for_agent(self, agent_id):
        tx = ty = 0.0
        for _, node_idx, cdx, cdy in self.closures:
            if self.nodes[node_idx].agent_id == agent_id:
                tx += cdx
                ty += cdy
        return tx, ty


class NativePoseGraphSLAM:
    """``PoseGraphSLAM``'s loop-closure chain (:261-338) and the drift bookkeeping of the ingest
    loop (:850-857, :908-914) run by the C library over whole batches of datagrams
    (``occgrid_slam_*`` in the header; host code, no GPU).  State carries over from batch to
    batch like the reference's ``slam`` / ``drift_correction`` objects.  Same closures and the same
    fp64 corrections as ``PoseGraphSLAM``; the quadratic landmark scan is replaced by a spatial
    hash that returns the same first match."""

    def __init__(self):
        self._lib = _native.lib()
        self._h = self._lib.occgrid_slam_create()
        if not self._h:
            raise OccGridError('occgrid_slam_create failed')

    def __del__(self):
        h, self._h = getattr(self, '_h', None), None
        if h:
            self._lib.occgrid_slam_destroy(h)

    def drift_table(self, packets, separation=0.0, sizes=None):
        """``packets``: uint8 [n, stride >= 41] (42-byte v2 records, or v1 records padded to the
        stride with ``sizes`` giving each datagram's length).  Returns float64 [n, 2]."""
        pk = np.ascontiguousarray(packets, dtype=np.uint8)
        if pk.ndim != 2:
            raise ValueError('packets must be uint8 [n, record_bytes]')
        n, stride = pk.shape
        out = np.zeros((n, 2), np.float64)
        sz = None if sizes is None else np.ascontiguousarray(sizes, dtype=np.int32)
        if sz is not None and sz.shape != (n,):
            raise ValueError('sizes must have one entry per record')
        rc = self._lib.occgrid_slam_drift_table(self._h, pk.ctypes.data, n, stride, min(stride, PACKET_SIZE),
                                                sz.ctypes.data if sz is not None else None, float(separation), out.ctypes.data)
        _native.check(rc, 'occgrid_slam_drift_table')
        return out

    def _counts(self):
        c = (ctypes.c_int64 * 3)()
        _native.check(self._lib.occgrid_slam_counts(self._h, ctypes.byref(c, 0), ctypes.byref(c, 8), ctypes.byref(c, 16)),
                      'occgrid_slam_counts')
        return int(c[0]), int(c[1]), int(c[2])

    n_nodes = property(lambda self: self._counts()[0])
    n_landmarks = property(lambda self: self._counts()[1])

    @property
    def closures(self):
        """[(landmark node index, closing node index, corr_dx, corr_dy)] like ``PoseGraphSLAM.closures``."""
        n = self._counts()[2]
        lm, nd, xy = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros((n, 2), np.float64)
        _native.check(self._lib.occgrid_slam_closures(self._h, n, lm.ctypes.data, nd.ctypes.data, xy.ctypes.data, None),
                      'occgrid_slam_closures')
        return [(int(lm[i]), int(nd[i]), float(xy[i, 0]), float(xy[i, 1])) for i in range(n)]

    def get_correction_for_agent(self, agent_id):
        xy = (ctypes.c_double * 2)()
        _native.check(self._lib.occgrid_slam_correction_for_agent(self._h, int(agent_id), xy), 'occgrid_slam_correction_for_agent')
        return float(xy[0]), float(xy[1])


def _pack_datagrams(datagrams):
    """list of datagrams (any lengths) / bytes / uint8 [n, stride] -> (uint8 [n, 42], sizes or None)."""
    if isinstance(datagrams, np.ndarray):
        return datagrams, None
    if isinstance(datagrams, (bytes, bytearray, memoryview)):
        return np.frombuffer(bytes(datagrams), np.uint8).reshape(-1, PACKET_SIZE), None
    sizes = np.fromiter((len(d) for d in datagrams), np.int32, len(datagrams))
    if len(datagrams) and (sizes == PACKET_SIZE).all():
        return np.frombuffer(b''.join(datagrams), np.uint8).reshape(-1, PACKET_SIZE), None
    out = np.zeros((len(datagrams), PACKET_SIZE), np.uint8)
    for k, d in enumerate(datagrams):
        if len(d) in (PACKET_SIZE, PACKET_SIZE_V1):
            out[k, :len(d)] = np.frombuffer(d, np.uint8)
    return out, sizes


def slam_drift_table(datagrams, separation=0.0, slam=None, timestamps=None):
    """Run the sequential part of the ingest loop (:826-857, :908-914) on the host and return
    the drift (cdx, cdy) in force for every datagram, float64 [n, 2] — the input
    ``OccupancyGrid.update_packets(drift=...)`` needs to reproduce a SLAM-corrected session.
    Runs in the C library (``NativePoseGraphSLAM``) unless a Python ``PoseGraphSLAM`` is passed
    in (kept for callers that want its ``nodes`` list)."""
    if slam is None:
        slam = NativePoseGraphSLAM()
    if isinstance(slam, NativePoseGraphSLAM):
        pk, sizes = _pack_datagrams(datagrams)
        return slam.drift_table(pk, separation, sizes), slam
    drift = {1: (0.0, 0.0), 2: (0.0, 0.0)}
    out = np.zeros((len(datagrams), 2), np.float64)
    for k, data in enumerate(datagrams):
        lm = LM_NONE
        if len(data) == PACKET_SIZE:
            magic, agent_id, rx, ry, ryaw, _, _, _, _, _, _, lm = struct.unpack(PACKET_FMT, data)
        elif len(data) == PACKET_SIZE_V1:
            magic, agent_id, rx, ry, ryaw = struct.unpack(PACKET_FMT_V1, data)[:5]
        else:
            continue
        if magic != b'QSRL' or agent_id not in (1, 2):
            continue
        if agent_id == 2:
            rx += separation
        cdx, cdy = drift[agent_id]
        out[k] = (cdx, cdy)
        rx += cdx
        ry += cdy
        if not (math.isfinite(rx) and math.isfinite(ry) and math.isfinite(ryaw)):
            continue
        closure, ndx, ndy = slam.add_pose(rx, ry, ryaw, agent_id, lm,
                                          timestamps[k] if timestamps is not None else float(k))
        if closure:
            drift[agent_id] = (drift[agent_id][0] + ndx, drift[agent_id][1] + ndy)
    return out, slam


class IngestBatcher:
    """Host-side batcher for the server loop (:797-919): datagrams are pushed as they arrive
    (``data, addr = sock.recvfrom(...)``, :818), filtered by size exactly like :828-838, and a
    ``flush()`` — once per frame in the reference's loop (:816 caps a frame at 20 datagrams; any
    batch size works here) — runs the sequential SLAM chain over the pending records in the C
    library and integrates them on the device in ONE call.  Equal to the reference handling the
    same datagrams one by one: SLAM state and drift carry over between flushes, and a later batch
    overwrites an earlier one cell by cell (last writer wins, :148-156).

        batcher = IngestBatcher(occ_grid, separation=args.separation)
        ...
        batcher.push(data)                 # instead of unpack + 4x update_ray (:826-903)
        ...
        batcher.flush()                    # end of the frame's receive loop
    """

    def __init__(self, grid, separation=0.0, use_slam=True, capacity=4096):
        self.grid = grid
        self.separation = float(separation)
        self.slam = NativePoseGraphSLAM() if use_slam else None
        self.capacity = int(capacity)
        self._buf = torch.zeros((self.capacity, PACKET_SIZE), dtype=torch.uint8).pin_memory() \
            if torch.cuda.is_available() else torch.zeros((self.capacity, PACKET_SIZE), dtype=torch.uint8)
        self._np = self._buf.numpy()
        self._n = 0
        self.dropped = 0                    # datagrams of a foreign size (:836-838)
        self.total = 0                      # records handed to the device so far

    def push(self, data):
        n = len(data)
        if n == PACKET_SIZE:
            self._np[self._n] = np.frombuffer(data, np.uint8)
        elif n == PACKET_SIZE_V1:           # v1: no landmark byte -> LM_NONE (:832-835)
            row = self._np[self._n]
            row[:PACKET_SIZE_V1] = np.frombuffer(data, np.uint8)
            row[PACKET_SIZE_V1] = LM_NONE
        else:
            self.dropped += 1
            return
        self._n += 1
        if self._n == self.capacity:
            self.flush()

    def flush(self):
        """Integrate everything pushed since the last flush; returns the number of records."""
        n = self._n
        if n == 0:
            return 0
        pk = self._np[:n]
        drift = self.slam.drift_table(pk, self.separation) if self.slam is not None else None
        self.grid.update_packets(self._buf[:n], separation=self.separation, drift=drift)
        torch.cuda.current_stream(self.grid.device).synchronize()      # the staging rows are reused by the next push
        self._n = 0
        self.total += n
        return n


def replay_session(datagrams, grid=None, separation=0.0, use_slam=True, **grid_kwargs):
    """Headless restatement of ``main()``'s ingest loop for a recorded session: host SLAM
    chain -> drift table -> one batched device integration.  Returns (grid, slam)."""
    grid = grid if grid is not None else OccupancyGrid(**grid_kwargs)
    drift, slam = (slam_drift_table(datagrams, separation) if use_slam else (None, None))
    grid.update_packets(list(datagrams), separation=separation, drift=drift)
    return grid, slam
