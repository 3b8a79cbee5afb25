"""Drop-in surface of the reference's ``server_nodes/map_merger.py`` (ROS 2 node ``MapMerger``).

Same entry points and message shapes as the reference, without rclpy / Open3D: messages are
duck-typed (anything with ``.info.width/.height/.resolution/.origin.position.x/.y``,
``.data`` and ``.header.frame_id`` works — a real ``nav_msgs/OccupancyGrid`` included) and the
point cloud lives in B200 HBM as two fp64 arrays.  Per reference line:

* ``map_callback(msg, agent_id)``          :35-62   (+ ``transform=`` in place of the ICP call at
  :45-56 — ICP is outside this path, SURVEY §8 a13 — and ``fitness=`` for the gate at :54-56)
* ``grid_to_pcd(msg)``                     :64-85   occupied cells (> 50) -> cell-corner points
* ``publish_global_map(frame_id)``         :87-127  bbox -> int8 grid holding only -1 / 100
* ``merge(grids, origins, res, transforms)``  NEW batched entry: the same sequence of
  callbacks, publishing once at the end.

Everything numeric runs in the hand-written sm_100a kernels behind ``mapmerge_*``
(include/occgrid_b200.h); there is no CPU fallback.
"""
from __future__ import annotations

import ctypes
import math
from types import SimpleNamespace

import numpy as np
import torch

from . import _native
from ._native import OccGridError


def make_grid_msg(data, width, height, resolution, origin_x, origin_y, frame_id='map'):
    """A minimal stand-in for ``nav_msgs/OccupancyGrid`` (fields used at map_merger.py:65-71,
    :113-125)."""
    pos = SimpleNamespace(x=float(origin_x), y=float(origin_y), z=0.0)
    info = SimpleNamespace(width=int(width), height=int(height), resolution=float(resolution),
                           origin=SimpleNamespace(position=pos, orientation=SimpleNamespace(w=1.0)))
    return SimpleNamespace(header=SimpleNamespace(frame_id=frame_id, stamp=None), info=info, data=data)


def se2_matrix(tx, ty, theta):
    """4x4 homogeneous matrix of a planar rigid transform (what ICP returns at :58)."""
    c, s = math.cos(theta), math.sin(theta)
    T = np.eye(4)
    T[0, 0], T[0, 1], T[0, 3] = c, -s, tx
    T[1, 0], T[1, 1], T[1, 3] = s, c, ty
    return T


class _Cloud:
    """fp64 x[], y[] + device-resident count."""

    def __init__(self, capacity, device):
        self.capacity = int(capacity)
        self.x = torch.empty(self.capacity, dtype=torch.float64, device=device)
        self.y = torch.empty(self.capacity, dtype=torch.float64, device=device)
        self.count = torch.zeros(1, dtype=torch.int64, device=device)


class MapMerger:
    """Fuses per-agent occupancy grids into one global map (reference :9-127).

    agent_ids      kept for API parity (:12-15); subscriptions are the caller's business
    device         CUDA device
    registration   None: ``map_callback`` takes the rigid transform from its caller (what the
                   reference gets from Open3D); 'icp': a callback without a transform is
                   registered against the global cloud on the device first (:45-56)
    """

    def __init__(self, agent_ids=(1,), device='cuda', publisher=None, registration=None):
        if not torch.cuda.is_available():
            raise OccGridError('no CUDA device: the map-fusion engine has no CPU fallback')
        self.agent_ids = list(agent_ids) or [1]
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self._lib = _native.lib()
        self.map_resolution = 0.05          # :32
        self.map_origin = [0.0, 0.0]        # :33
        self.publisher = publisher          # optional callable(msg), stands in for :29
        self.published = None               # last published message
        if registration not in (None, 'icp'):
            raise ValueError("registration must be None (the caller supplies the transform) or 'icp'")
        self.registration = registration    # 'icp': callbacks without a transform run registration_icp (:45-52)
        self.last_registration = None
        self._local = None                  # scratch cloud of the callback being registered
        self._n_global = 0                  # host mirror of the global cloud size
        self._cloud = None                  # current global cloud
        self._spare = None                  # ping-pong partner for the voxel filter
        self._status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._bounds = torch.zeros(4, dtype=torch.float64, device=self.device)
        self._last = torch.zeros(1, dtype=torch.int64, device=self.device)
        self._ws = {}
        self._lattice_cap = 0
        self._voxel_points_cap = -1

    # ---- plumbing ------------------------------------------------------------------------
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _workspace(self, name, nbytes, zero=False):
        t = self._ws.get(name)
        if t is None or t.numel() < nbytes:
            alloc = torch.zeros if zero else torch.empty
            t = alloc(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=self.device)
            self._ws[name] = t
        return t

    def _ensure_capacity(self, need):
        if self._cloud is not None and self._cloud.capacity >= need:
            return
        cap = max(int(need * 1.5), 1 << 16)
        new, spare = _Cloud(cap, self.device), _Cloud(cap, self.device)
        if self._cloud is not None and self._n_global:
            n = self._n_global
            new.x[:n].copy_(self._cloud.x[:n])
            new.y[:n].copy_(self._cloud.y[:n])
            new.count.copy_(self._cloud.count)
        self._cloud, self._spare = new, spare

    def _check_status(self):
        st = int(self._status.item())
        if st:
            self._status.zero_()
            raise OccGridError('map merge overflow: ' + ', '.join(
                n for b, n in ((1, 'point capacity'), (2, 'voxel lattice capacity'),
                            (4, 'chain kernel aborted (a grid barrier timed out)')) if st & b))

    def _device_grid(self, msg, async_upload=False):
        data = msg.data
        h, w = int(msg.info.height), int(msg.info.width)
        if isinstance(data, torch.Tensor):
            # async_upload: pinned host grids upload without a sync per grid (only the batch path
            # asks for it: it reads the occupied counts back before returning, which orders every
            # upload before the caller can touch the source again)
            t = data.to(self.device, dtype=torch.int8,
                        non_blocking=bool(async_upload and not data.is_cuda and data.is_pinned())).reshape(h, w)
        else:
            t = torch.from_numpy(np.ascontiguousarray(np.asarray(data, dtype=np.int8).reshape(h, w))).to(self.device)
        return t.contiguous()

    def _extract(self, msg, T):
        """grid_to_pcd (+ transform) appended to the global cloud; returns points appended."""
        g = self._device_grid(msg)
        h, w = g.shape
        # worst case every cell is occupied; grow on demand instead of allocating H*W up front
        ws = self._workspace('extract', self._lib.mapmerge_extract_workspace_bytes(h * w))
        Tm = None
        if T is not None:
            Tm = np.ascontiguousarray(np.asarray(T, np.float64).reshape(4, 4))
        for attempt in range(2):
            rc = self._lib.mapmerge_extract_transform(
                g.data_ptr(), w, h, float(msg.info.resolution), float(msg.info.origin.position.x),
                float(msg.info.origin.position.y), Tm.ctypes.data if Tm is not None else None,
                self._cloud.x.data_ptr(), self._cloud.y.data_ptr(), self._cloud.capacity,
                self._cloud.count.data_ptr(), self._last.data_ptr(), self._status.data_ptr(),
                ws.data_ptr(), ws.numel(), self._stream())
            _native.check(rc, 'mapmerge_extract_transform')
            st = int(self._status.item())
            if st & 1 and attempt == 0:          # grow and retry once with room for every cell
                self._status.zero_()
                self._ensure_capacity(self._n_global + h * w)
                continue
            break
        self._check_status()
        return int(self._last.item())

    def _bounds_of(self, cloud):
        ws = self._workspace('bounds', self._lib.mapmerge_bounds_workspace_bytes())
        rc = self._lib.mapmerge_bounds(cloud.x.data_ptr(), cloud.y.data_ptr(), cloud.count.data_ptr(),
                                       self._bounds.data_ptr(), ws.data_ptr(), ws.numel(), self._stream())
        _native.check(rc, 'mapmerge_bounds')

    def _voxel_workspace(self, lattice_cells, points):
        """The lattice sits first in the workspace and must stay all-zero between calls, so the
        layout may only change together with a fresh (zeroed) allocation."""
        if lattice_cells > self._lattice_cap or points != self._voxel_points_cap:
            self._lattice_cap = max(int(lattice_cells * 1.5), self._lattice_cap)
            self._voxel_points_cap = points
            self._ws.pop('voxel', None)
        need = self._lib.mapmerge_voxel_workspace_bytes(self._lattice_cap, points)
        return self._workspace('voxel', need, zero=True)

    def _voxel_downsample(self, lattice_cells=None, sync=True, benc=None):
        """global_pcd = global_pcd.voxel_down_sample(map_resolution)  (:60).  `lattice_cells`: a
        conservative bound on the voxel lattice known to the caller (batched merge, no host round
        trip); otherwise the bounds are read back to size it."""
        if benc is None:
            self._bounds_of(self._cloud)
        v = self.map_resolution
        if lattice_cells is None:
            b = self._bounds.cpu().numpy()
            nx = int(math.floor((b[2] - (b[0] - v * 0.5)) / v)) + 1
            ny = int(math.floor((b[3] - (b[1] - v * 0.5)) / v)) + 1
            lattice_cells = nx * ny
        ws = self._voxel_workspace(lattice_cells, self._cloud.capacity)
        rc = self._lib.mapmerge_voxel_downsample(
            self._cloud.x.data_ptr(), self._cloud.y.data_ptr(), self._cloud.count.data_ptr(), self._cloud.capacity,
            v, self._bounds.data_ptr(), benc.data_ptr() if benc is not None else None, self._lattice_cap,
            self._spare.x.data_ptr(), self._spare.y.data_ptr(),
            self._spare.count.data_ptr(), self._status.data_ptr(), ws.data_ptr(), ws.numel(), self._stream())
        _native.check(rc, 'mapmerge_voxel_downsample')
        self._cloud, self._spare = self._spare, self._cloud
        if sync:
            self._n_global = int(self._cloud.count.item())
            self._check_status()

    # ---- reference surface ---------------------------------------------------------------
    @property
    def global_pcd(self):
        """Host copy of the global cloud as float64 [n, 3] (z = 0), like ``np.asarray(pcd.points)``."""
        n = self._n_global
        out = np.zeros((n, 3))
        if n:
            out[:, 0] = self._cloud.x[:n].cpu().numpy()
            out[:, 1] = self._cloud.y[:n].cpu().numpy()
        return out

    def grid_to_pcd(self, msg):
        """:64-85 — returns the points as float64 [k, 3] on the host (diagnostic twin of the fused
        device path used by map_callback)."""
        tmp = MapMerger(device=self.device)
        tmp._ensure_capacity(1 << 16)
        k = tmp._extract(msg, None)
        tmp._n_global = k
        return tmp.global_pcd

    def register(self, msg, threshold=1.0, max_iteration=30, relative_fitness=1e-6, relative_rmse=1e-6):
        """``o3d.pipelines.registration.registration_icp(local_pcd, global_pcd, threshold,
        identity, TransformationEstimationPointToPoint(), ICPConvergenceCriteria(max_iteration))``
        (:45-52) on the device.  Returns an object with ``transformation`` (4x4), ``fitness``,
        ``inlier_rmse`` and ``iterations``; None when the local cloud is empty."""
        if self._n_global == 0:
            raise OccGridError('register: the global cloud is empty')
        with torch.cuda.device(self.device):
            g = self._device_grid(msg)
            h, w = g.shape
            cnt = torch.zeros(1, dtype=torch.int64, device=self.device)
            _native.check(self._lib.mapmerge_count_occupied(g.data_ptr(), g.numel(), cnt.data_ptr(), self._stream()),
                          'mapmerge_count_occupied')
            k = int(cnt.item())
            if k == 0:
                return None
            if self._local is None or self._local.capacity < k:
                self._local = _Cloud(int(k * 1.25) + 16, self.device)
            loc = self._local
            loc.count.zero_()
            ws = self._workspace('extract', self._lib.mapmerge_extract_workspace_bytes(h * w))
            rc = self._lib.mapmerge_extract_transform(
                g.data_ptr(), w, h, float(msg.info.resolution), float(msg.info.origin.position.x),
                float(msg.info.origin.position.y), None, loc.x.data_ptr(), loc.y.data_ptr(), loc.capacity,
                loc.count.data_ptr(), self._last.data_ptr(), self._status.data_ptr(), ws.data_ptr(), ws.numel(), self._stream())
            _native.check(rc, 'mapmerge_extract_transform')
            self._bounds_of(self._cloud)
            bb = self._bounds.cpu().numpy().tolist()
            cell = float(threshold) / 4.0
            cw, ch = int((bb[2] - bb[0]) / cell) + 2, int((bb[3] - bb[1]) / cell) + 2
            nbytes = self._lib.mapmerge_icp_workspace_bytes(self._n_global, k, cw, ch)
            iws = self._workspace('icp', nbytes)
            res = torch.empty(20, dtype=torch.float64, device=self.device)
            rc = self._lib.mapmerge_icp_register(loc.x.data_ptr(), loc.y.data_ptr(), k, self._cloud.x.data_ptr(),
                                                 self._cloud.y.data_ptr(), self._n_global, bb[0], bb[1], cell, cw, ch,
                                                 float(threshold), int(max_iteration), float(relative_fitness),
                                                 float(relative_rmse), res.data_ptr(), iws.data_ptr(), iws.numel(), self._stream())
            _native.check(rc, 'mapmerge_icp_register')
            r = res.cpu().numpy()
            self._check_status()
            if r[18] < 0:                                   # a grid barrier of the loop kernel timed out
                raise OccGridError('register: the ICP loop kernel was aborted (grid barrier time-out)')
        self.last_registration = SimpleNamespace(transformation=r[:16].reshape(4, 4).copy(), fitness=float(r[16]),
                                                 inlier_rmse=float(r[17]), iterations=int(r[18]), correspondences=int(r[19]))
        return self.last_registration

    def _merge_one(self, msg, transform, fitness):
        """:36-60 without the publish.  Returns False where the reference returns early."""
        if transform is not None and np.asarray(transform).size == 3:
            transform = se2_matrix(*np.asarray(transform, np.float64).tolist())
        with torch.cuda.device(self.device):
            first = self._n_global == 0
            if not first and transform is None and self.registration == 'icp':
                reg = self.register(msg)                    # :45-52
                if reg is None:                             # empty local cloud (:37-38)
                    return False
                transform, fitness = reg.transformation, reg.fitness
            if not first and fitness < 0.6:                 # :54-56 — no state change, nothing published
                return False
            self._ensure_capacity(self._n_global + (1 << 16))
            k = self._extract(msg, None if first else transform)
            if k == 0:                                      # :37-38
                return False
            if first:                                       # :40-43
                self._n_global = k
                self.map_resolution = float(msg.info.resolution)
                self.map_origin = [float(msg.info.origin.position.x), float(msg.info.origin.position.y)]
            else:                                           # :58-60
                self._n_global += k
                self._voxel_downsample()
        return True

    def map_callback(self, msg, agent_id, transform=None, fitness=1.0):
        """:35-62.  ``transform`` (4x4 or (tx, ty, theta)) stands in for ``reg_p2p.transformation``;
        ``fitness`` for ``reg_p2p.fitness`` (rejected below 0.6, :54-56).  Returns the published
        message, or None where the reference returns early."""
        if not self._merge_one(msg, transform, fitness):
            return None
        return self.publish_global_map(getattr(getattr(msg, 'header', None), 'frame_id', 'map'))

    def publish_global_map(self, frame_id=None, to_host=True):
        """:87-127.  Returns (and hands to ``publisher``) a message whose ``data`` is the int8 grid
        as a NumPy array [height, width] (``.flatten().tolist()`` gives the reference's list)."""
        if self._n_global == 0:                             # :88-93
            return None
        with torch.cuda.device(self.device):
            self._bounds_of(self._cloud)
            min_x, min_y, max_x, max_y = self._bounds.cpu().numpy().tolist()
            res = self.map_resolution
            width = int(np.ceil((max_x - min_x) / res)) + 1     # :100
            height = int(np.ceil((max_y - min_y) / res)) + 1    # :101
            grid = torch.empty((height, width), dtype=torch.int8, device=self.device)
            rc = self._lib.mapmerge_rasterise(self._cloud.x.data_ptr(), self._cloud.y.data_ptr(),
                                              self._cloud.count.data_ptr(), res, self._bounds.data_ptr(),
                                              width, height, grid.data_ptr(), self._stream())
            _native.check(rc, 'mapmerge_rasterise')
            data = grid.cpu().numpy() if to_host else grid
        msg = make_grid_msg(data, width, height, res, min_x, min_y, frame_id='map_global')   # :113-123
        self.published = msg
        if self.publisher is not None:
            self.publisher(msg)
        return msg

    # ---- batched entry ---------------------------------------------------------------------
    def _as_device_grids(self, grids):
        """List of int8 [H, W] device tensors (no copies for tensors already in that form)."""
        out = []
        for g in grids:
            if isinstance(g, torch.Tensor) and g.is_cuda and g.dtype == torch.int8 and g.dim() == 2 and g.is_contiguous() \
                    and g.device == self.device:
                out.append(g)
            else:
                out.append(self._device_grid(make_grid_msg(g, g.shape[1], g.shape[0], 0.0, 0, 0), async_upload=True))
        return out

    @staticmethod
    def _as_matrices(transforms, A):
        """[A, 4, 4] float64 from None / [A, 4, 4] / [A, 3] (tx, ty, theta) / a list mixing both."""
        if transforms is None:
            return np.tile(np.eye(4), (A, 1, 1))
        try:
            t = np.asarray(transforms, np.float64)
        except ValueError:
            t = None
        if t is not None and t.shape == (A, 4, 4):
            return np.ascontiguousarray(t)
        out = np.tile(np.eye(4), (A, 1, 1))
        for a in range(A):
            T = transforms[a]
            if T is None:
                continue
            T = np.asarray(T, np.float64)
            out[a] = se2_matrix(*T.tolist()) if T.size == 3 else T.reshape(4, 4)
        return np.ascontiguousarray(out)

    def merge(self, grids, origins, res, transforms=None, fitness=None, to_host=True, publish=True, adopt_first=True):
        """Fuse A agent grids in order: ``grids`` int8 [A, H, W] (host or device), ``origins``
        float64 [A, 2], ``transforms`` [A, 4, 4] or [A, 3] (tx, ty, theta) or None (identity).
        Equal to A successive ``map_callback`` calls (same sequential voxel chain, :58-60);
        publishes once at the end.  Equal-shaped grids are extracted in one batched launch and
        fused by the incremental chain (``mapmerge_chain_*``: work per callback proportional to the
        slice, not to the accumulated cloud, while the voxel lattice stands still); the host reads
        the occupied-cell counts up front, the chain state every few callbacks and the final bounds.
        ``adopt_first=False`` (multi-GPU shards that do not hold the globally first cloud): the first
        local cloud is transformed like every other one.  ``publish=False``: fuse only.
        Returns (int8 grid [H', W'], (origin_x, origin_y))."""
        A = len(grids)
        with torch.cuda.device(self.device):
            dev = self._as_device_grids(grids)
            same_shape = all(d.shape == dev[0].shape for d in dev)
            counts, ptrs, bws = self._count_occupied(dev, same_shape)
            # host work that does not need the counts overlaps the counting pass
            org = np.ascontiguousarray(np.asarray(origins, np.float64).reshape(A, 2))
            Tm = self._as_matrices(transforms, A)
            fit = np.ones(A) if fitness is None else np.asarray(fitness, np.float64).reshape(A)
            hw = np.array([[d.shape[0], d.shape[1]] for d in dev], np.float64)
            n_occ = counts.cpu().numpy()                            # host sync 1
            plan = self._plan_merge(n_occ, fit, Tm, org, hw, res, adopt_first)
            if plan is None:
                return None, None
            use, order, first, bb, n_new = plan
            self._ensure_capacity(self._n_global + n_new + 1024)
            v = float(res) if first else self.map_resolution
            lat_w, lat_h = int((bb[2] - bb[0]) / v) + 4, int((bb[3] - bb[1]) / v) + 4
            stage = offs = None
            if same_shape:                       # all slices extracted + transformed in one launch
                stage, offs = self._write_slices(dev, ptrs, bws, counts, use, Tm, org, res, n_new)
            chain = None
            if first:                            # adopted as is (:40-43): no filter on this callback
                a = order.pop(0)
                if same_shape:
                    rc = self._lib.mapmerge_append_slice(stage.x.data_ptr(), stage.y.data_ptr(), offs.data_ptr(), a,
                                                         self._cloud.x.data_ptr(), self._cloud.y.data_ptr(), self._cloud.capacity,
                                                         self._cloud.count.data_ptr(), self._status.data_ptr(), None, self._stream())
                    _native.check(rc, 'mapmerge_append_slice')
                else:
                    self._extract_async(make_grid_msg(dev[a], dev[a].shape[1], dev[a].shape[0], res, org[a, 0], org[a, 1]),
                                        None if adopt_first else Tm[a])
                self.map_resolution = float(res)
                self.map_origin = [float(org[a, 0]), float(org[a, 1])]
            if same_shape:
                if order:
                    chain = self._run_chain(stage, offs, A, order, lat_w, lat_h, int(n_occ[use].max()))
            else:
                for a in order:
                    self._extract_async(make_grid_msg(dev[a], dev[a].shape[1], dev[a].shape[0], res, org[a, 0], org[a, 1]), Tm[a])
                    self._voxel_downsample(lattice_cells=lat_w * lat_h, sync=False)
            self.chain_stats = chain
            self._n_global = int(self._cloud.count.item())          # host sync (with the status word)
            self._check_status()
        if not publish:
            return None, None
        out = self.publish_global_map(to_host=to_host)
        if out is None:
            return None, None
        return out.data, (out.info.origin.position.x, out.info.origin.position.y)

    # ---- fused occupancy map (EXTENSION, no reference counterpart) ------------------------------
    def fuse_occupancy(self, grids, origins, res, transforms, target):
        """Resample every agent map into ``target`` under its agent->global transform and keep free
        space: each target cell becomes max(-1, max of the covering agents' cells at its centre), so
        occupied beats free beats unknown (``mapmerge_warp_fuse`` in include/occgrid_b200.h gives the
        exact arithmetic).  Unlike ``merge``, the result can be explored: ``target.get_frontiers()``,
        ``cluster_frontiers()`` and ``frontier_centroids()`` work on it.

        grids       int8 [A, H, W]; a contiguous CUDA tensor on this merger's device (such as
                    ``AgentGrids.grids_tensor``) is used without a copy, a host array is uploaded once
        origins     float64 [A, 2], agent a's (origin_x, origin_y); ``res`` the agents' resolution
        transforms  [A, 4, 4], [A, 3] (tx, ty, theta) or None (identity); every one applied as given
        target      an ``OccupancyGrid`` holding its whole grid, on this merger's device, with its own
                    size, resolution and origin; all of its cells are overwritten
        Returns ``target``.  The merger's cloud and state are left alone."""
        if target.window != (0, 0, target.size, target.size):
            raise OccGridError('fuse_occupancy: the target must hold its whole grid (not a window of it)')
        if target.device != self.device:
            raise OccGridError(f'fuse_occupancy: the target is on {target.device}, the merger on {self.device}')
        if isinstance(grids, torch.Tensor):
            if grids.is_cuda and grids.device != self.device:
                raise OccGridError(f'fuse_occupancy: the grids are on {grids.device}, the merger on {self.device}')
            if grids.dtype != torch.int8:
                raise ValueError('fuse_occupancy: grids must be int8')
        else:
            grids = np.ascontiguousarray(np.asarray(grids), dtype=np.int8)
        if grids.ndim != 3 or min(grids.shape) < 1:
            raise ValueError(f'fuse_occupancy: grids must be [A, H, W] with A, H, W >= 1, got {tuple(grids.shape)}')
        A, h, w = (int(v) for v in grids.shape)
        org = np.asarray(origins, np.float64)
        if org.size != 2 * A:
            raise ValueError(f'fuse_occupancy: origins must be [{A}, 2], got {org.shape}')
        org = np.ascontiguousarray(org.reshape(A, 2))
        if transforms is not None and len(transforms) != A:
            raise ValueError(f'fuse_occupancy: {len(transforms)} transforms for {A} grids')
        Tm = self._as_matrices(transforms, A)
        lib = self._lib
        with torch.cuda.device(self.device):
            if isinstance(grids, np.ndarray):
                grids = torch.from_numpy(grids).to(self.device)
            elif not (grids.is_cuda and grids.is_contiguous()):
                grids = grids.to(self.device).contiguous()
            nbytes = lib.mapmerge_warp_fuse_workspace_bytes(A, target.size, target.size)
            if nbytes == 0:
                raise OccGridError('mapmerge_warp_fuse_workspace_bytes: ' + _native.last_error())
            ws = self._workspace('fuse', nbytes)
            rc = lib.mapmerge_warp_fuse(grids.data_ptr(), A, w, h, float(res), org.ctypes.data, Tm.ctypes.data,
                                        target.ox, target.oy, target.res, target.size, target.size,
                                        target.grid_tensor.data_ptr(), ws.data_ptr(), ws.numel(), self._stream())
            _native.check(rc, 'mapmerge_warp_fuse')
        target._host_cache = None
        return target

    # ---- batched map registration (EXTENSION, no reference counterpart) -------------------------
    def register_maps(self, grids, origins, res, priors, reference=None, threshold=1.0, max_iteration=30,
                      relative_fitness=1e-6, relative_rmse=1e-6):
        """Refine every agent->global transform against ONE reference map in one device call: agent
        a's occupied cells (> 50) at cell corners, moved by ``priors[a]``, are registered with
        ``registration_icp(…, threshold, identity, point-to-point, max_iteration)`` (:45-52) against
        the reference cloud (``mapmerge_icp_register_batch`` in include/occgrid_b200.h).  Each
        agent's refinement equals a separate ``register``-style ICP call bit for bit; the cell list
        of the reference is built once and the loops of all agents run in one cooperative launch.

        grids       int8 [A, H, W] (``AgentGrids.grids_tensor`` is used without a copy); ``origins``
                    float64 [A, 2]; ``res`` the agents' resolution
        priors      [A, 4, 4], [A, 3] (tx, ty, theta) or None (identity): rigid agent->global
                    transforms (every entry finite, |RᵀR − I| <= 1e-9, as ``fuse_occupancy``)
        reference   None: the merger's global cloud (as ``register``); or an ``OccupancyGrid``
                    holding its whole grid on this device, whose occupied cells at cell corners are
                    the reference (typically the previous step's fused map)
        The host reads twice: the occupied counts with the reference bounds, then the results.
        Returns a namespace of NumPy arrays: ``refinement`` [A, 4, 4] (the ICP result U_a),
        ``transformation`` [A, 4, 4] (U_a @ prior_a in fp64 where accepted, else the prior; it goes
        straight into ``fuse_occupancy``), ``fitness``, ``inlier_rmse``, ``iterations``,
        ``correspondences`` and ``accepted`` (fitness >= 0.6, the gate at :54-56).  An agent with no
        occupied cells gets the identity refinement, fitness 0 and 0 iterations."""
        if isinstance(grids, torch.Tensor):
            if grids.is_cuda and grids.device != self.device:
                raise OccGridError(f'register_maps: the grids are on {grids.device}, the merger on {self.device}')
            if grids.dtype != torch.int8:
                raise ValueError('register_maps: grids must be int8')
        else:
            grids = np.ascontiguousarray(np.asarray(grids), dtype=np.int8)
        if grids.ndim != 3 or min(grids.shape) < 1:
            raise ValueError(f'register_maps: grids must be [A, H, W] with A, H, W >= 1, got {tuple(grids.shape)}')
        A = int(grids.shape[0])
        org = np.asarray(origins, np.float64)
        if org.size != 2 * A:
            raise ValueError(f'register_maps: origins must be [{A}, 2], got {org.shape}')
        org = np.ascontiguousarray(org.reshape(A, 2))
        if priors is not None:
            if len(priors) != A:
                raise ValueError(f'register_maps: {len(priors)} priors for {A} grids')
            for a in range(A):
                if priors[a] is not None and np.asarray(priors[a]).size not in (3, 16):
                    raise ValueError(f'register_maps: prior {a} must be 4x4 or (tx, ty, theta), got shape {np.asarray(priors[a]).shape}')
        Tm = self._as_matrices(priors, A)
        for a in range(A):                       # mapmerge_warp_fuse's rule, in the same fp64 arithmetic
            T = Tm[a]
            if not np.isfinite(T).all():
                raise OccGridError(f'register_maps: prior {a} has a non-finite entry')
            R = ((T[0, 0], T[0, 1]), (T[1, 0], T[1, 1]))
            for p in range(2):
                for q in range(2):
                    rtr = float(R[0][p]) * float(R[0][q]) + float(R[1][p]) * float(R[1][q])
                    if not abs(rtr - (1.0 if p == q else 0.0)) <= 1e-9:
                        raise OccGridError(f'register_maps: prior {a} is not rigid (|R^T R - I| > 1e-9)')
        if reference is not None:
            if reference.window != (0, 0, reference.size, reference.size):
                raise OccGridError('register_maps: the reference must hold its whole grid (not a window of it)')
            if reference.device != self.device:
                raise OccGridError(f'register_maps: the reference is on {reference.device}, the merger on {self.device}')
        elif self._n_global == 0:
            raise OccGridError('register_maps: the global cloud is empty')
        lib = self._lib
        with torch.cuda.device(self.device):
            job = self._registration_inputs(grids, org, res, Tm, reference, threshold)
            nbytes = lib.mapmerge_icp_register_batch_workspace_bytes(job.n_target, job.n_points, A, job.cells_w, job.cells_h)
            if nbytes == 0:
                raise OccGridError('mapmerge_icp_register_batch_workspace_bytes: ' + _native.last_error())
            iws = self._workspace('icp', nbytes)
            out = torch.empty((A, 20), dtype=torch.float64, device=self.device)
            rc = lib.mapmerge_icp_register_batch(job.sx.data_ptr(), job.sy.data_ptr(), job.offsets.data_ptr(), A, job.tx.data_ptr(),
                                                 job.ty.data_ptr(), job.n_target, job.min_x, job.min_y, job.cell, job.cells_w,
                                                 job.cells_h, float(threshold), int(max_iteration), float(relative_fitness),
                                                 float(relative_rmse), out.data_ptr(), iws.data_ptr(), iws.numel(), self._stream())
            _native.check(rc, 'mapmerge_icp_register_batch')
            r = out.cpu().numpy()                                               # host read 2
        if (r[:, 18] < 0).any():
            raise OccGridError('register_maps: the batched ICP loop kernel was aborted (grid barrier time-out)')
        U = np.ascontiguousarray(r[:, :16].reshape(A, 4, 4))
        fitness = r[:, 16].copy()
        accepted = fitness >= 0.6                                               # :54-56
        transformation = np.where(accepted[:, None, None], np.matmul(U, Tm), Tm)
        return SimpleNamespace(refinement=U, transformation=transformation, fitness=fitness, inlier_rmse=r[:, 17].copy(),
                               iterations=r[:, 18].astype(np.int64), correspondences=r[:, 19].astype(np.int64),
                               accepted=accepted)

    def _registration_inputs(self, grids, org, res, Tm, reference, threshold):
        """The device inputs of mapmerge_icp_register_batch: every agent's occupied cells moved by its
        prior (one batched extraction), the reference cloud and its cell list.  One host read: the
        occupied counts with the reference's bounds, size and the status word."""
        lib = self._lib
        A = int(grids.shape[0])
        if isinstance(grids, np.ndarray):
            grids = torch.from_numpy(grids).to(self.device)
        elif not (grids.is_cuda and grids.is_contiguous()):
            grids = grids.to(self.device).contiguous()
        dev = list(grids.unbind(0))
        counts, ptrs, bws = self._count_occupied(dev, True)
        if reference is None:
            ref, n_ref = self._cloud, torch.full((1,), self._n_global, dtype=torch.int64, device=self.device)
        else:                                    # the reference's occupied cells: at most one point per cell
            cells = reference.size * reference.size
            ref = self._reference_cloud(cells)
            ref.count.zero_()
            ws = self._workspace('extract', lib.mapmerge_extract_workspace_bytes(cells))
            g = reference.grid_tensor
            rc = lib.mapmerge_extract_transform(g.data_ptr(), reference.size, reference.size, reference.res, reference.ox,
                                                reference.oy, None, ref.x.data_ptr(), ref.y.data_ptr(), ref.capacity,
                                                ref.count.data_ptr(), self._last.data_ptr(), self._status.data_ptr(),
                                                ws.data_ptr(), ws.numel(), self._stream())
            _native.check(rc, 'mapmerge_extract_transform')
            n_ref = ref.count
        self._bounds_of(ref)
        head = torch.cat([counts.double(), self._bounds, n_ref.double(), self._status.double()]).cpu().numpy()   # host read 1
        n_occ = head[:A].astype(np.int64)
        bb = head[A:A + 4].tolist()
        n_target, status = int(head[A + 4]), int(head[A + 5])
        if status:
            self._check_status()
        if n_target == 0:
            raise OccGridError('register_maps: the reference has no occupied cells')
        cell = float(threshold) / 4.0
        cw, ch = int((bb[2] - bb[0]) / cell) + 2, int((bb[3] - bb[1]) / cell) + 2      # as register
        n_new = int(n_occ.sum())
        stage, offs = self._write_slices(dev, ptrs, bws, counts, np.ones(A, bool), Tm, org, res, n_new)
        return SimpleNamespace(sx=stage.x, sy=stage.y, offsets=offs, n_points=n_new, n_occupied=n_occ, tx=ref.x, ty=ref.y,
                               n_target=n_target, min_x=bb[0], min_y=bb[1], cell=cell, cells_w=cw, cells_h=ch)

    def _reference_cloud(self, capacity):
        """Scratch cloud for a reference map's points (grown, never shrunk)."""
        c = getattr(self, '_ref_cloud', None)
        if c is None or c.capacity < capacity:
            c = self._ref_cloud = _Cloud(capacity, self.device)
        return c

    # ---- pieces of the batched merge (also driven by distributed.ShardedMapMerger) ---------------
    def _count_occupied(self, dev, same_shape):
        """Pass 1 over the grids: occupied cells per grid (device int64 [A]).  Equal-shaped grids go
        through the batched scan (bulk-copy staged when every grid is 16-byte aligned)."""
        A = len(dev)
        counts = torch.zeros(A, dtype=torch.int64, device=self.device)
        ptrs = bws = None
        if same_shape:                           # one pass over all grids
            h, w = dev[0].shape
            ptrs = torch.from_numpy(np.array([d.data_ptr() for d in dev], np.int64)).to(self.device)
            bws = self._workspace('extract_batch', self._lib.mapmerge_extract_batch_workspace_bytes(h * w, A))
            bulk_ok = 1 if all(d.data_ptr() % 16 == 0 for d in dev) else 0       # cp.async.bulk needs 16-byte aligned sources
            rc = self._lib.mapmerge_extract_batch_count(ptrs.data_ptr(), A, w, h, counts.data_ptr(), bws.data_ptr(),
                                                        bws.numel(), bulk_ok, self._stream())
            _native.check(rc, 'mapmerge_extract_batch_count')
        else:
            for a in range(A):
                rc = self._lib.mapmerge_count_occupied(dev[a].data_ptr(), dev[a].numel(), counts[a:a + 1].data_ptr(), self._stream())
                _native.check(rc, 'mapmerge_count_occupied')
        return counts, ptrs, bws

    def _plan_merge(self, n_occ, fit, Tm, org, hw, res, adopt_first=True):
        """Host decisions of a batched merge: which agents take part (:37-38, :54-56), which cloud is
        adopted as is (:40-43; its transform becomes the identity in `Tm`), the callback order and a
        bound on every cloud of the chain.  -> (use, order, first, bb, n_new) or None."""
        have_cloud = self._n_global > 0
        use = (n_occ > 0) & (fit >= 0.6)                        # :37-38, :54-56
        if not have_cloud:
            nz = np.flatnonzero(n_occ > 0)
            if nz.size == 0:
                return None
            use[:nz[0]] = False
            use[nz[0]] = True                                   # the first cloud is adopted as is (:40-43):
            if adopt_first:
                Tm[nz[0]] = np.eye(4)                           # no ICP, no fitness test, no transform
        used = np.flatnonzero(use)
        if have_cloud:
            self._bounds_of(self._cloud)
            bb = self._bounds.cpu().numpy().tolist()
        else:
            bb = [math.inf, math.inf, -math.inf, -math.inf]
        if used.size:
            # transformed extents of the used grids bound every cloud of the chain
            x0, y0 = org[used, 0], org[used, 1]
            x1, y1 = x0 + hw[used, 1] * res, y0 + hw[used, 0] * res
            M = Tm[used]
            cx = np.stack([x0, x0, x1, x1], 1)
            cy = np.stack([y0, y1, y0, y1], 1)
            px = M[:, 0, 0, None] * cx + M[:, 0, 1, None] * cy + M[:, 0, 3, None]
            py = M[:, 1, 0, None] * cx + M[:, 1, 1, None] * cy + M[:, 1, 3, None]
            bb = [min(bb[0], float(px.min())), min(bb[1], float(py.min())), max(bb[2], float(px.max())), max(bb[3], float(py.max()))]
        n_new = int(n_occ[used].sum())
        if self._n_global + n_new == 0:
            return None
        return use, used.tolist(), not have_cloud, bb, n_new

    def _write_slices(self, dev, ptrs, bws, counts, use, Tm, org, res, n_new):
        """Pass 2: every used grid's occupied cells -> transformed points, agent after agent, in a
        staging cloud; offs[a] = start of agent a's slice."""
        A = len(dev)
        h, w = dev[0].shape
        stage = _Cloud(n_new + 16, self.device)
        offs = torch.zeros(A + 1, dtype=torch.int64, device=self.device)
        xf = torch.empty(A * 96, dtype=torch.uint8, device=self.device)
        org_d = torch.from_numpy(np.ascontiguousarray(org)).to(self.device)
        use_h = np.ascontiguousarray(use.astype(np.uint8))
        Tm = np.ascontiguousarray(Tm)
        rc = self._lib.mapmerge_extract_batch_write(
            ptrs.data_ptr(), A, w, h, float(res), org_d.data_ptr(), Tm.ctypes.data, use_h.ctypes.data, xf.data_ptr(),
            stage.x.data_ptr(), stage.y.data_ptr(), stage.capacity, counts.data_ptr(), offs.data_ptr(),
            self._status.data_ptr(), bws.data_ptr(), bws.numel(), self._stream())
        _native.check(rc, 'mapmerge_extract_batch_write')
        return stage, offs

    def _run_chain(self, stage, offs, n_agents, order, lat_w, lat_h, slice_cap):
        """The callbacks `global += slice; global = voxel_down_sample(global)` (:58-60) for the
        slices `order` of a batched extraction, through the incremental chain (mapmerge_chain_*
        in the header).  Callbacks are enqueued a few at a time without host round trips; the
        host only steps in for the ones that need the full filter."""
        lib = self._lib
        pcap = self._cloud.capacity
        dims = np.array([lat_w, lat_h, pcap, slice_cap], np.int64)
        nbytes = lib.mapmerge_chain_workspace_bytes(dims.ctypes.data, n_agents)
        if nbytes == 0:
            raise OccGridError('map merge: voxel lattice %d x %d too large' % (lat_w, lat_h))
        ws = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        vws = self._voxel_workspace(lat_w * lat_h, pcap)
        order_h = np.ascontiguousarray(np.asarray(order, np.int32))
        c = self._cloud
        rc = lib.mapmerge_chain_init(ws.data_ptr(), ws.numel(), dims.ctypes.data, n_agents, stage.x.data_ptr(), stage.y.data_ptr(),
                                     offs.data_ptr(), order_h.ctypes.data, len(order), c.x.data_ptr(), c.y.data_ptr(),
                                     c.count.data_ptr(), self._stream())
        _native.check(rc, 'mapmerge_chain_init')
        v = self.map_resolution
        state = (ctypes.c_int32 * 2)()
        stats = {'callbacks': len(order), 'rebuilds': 0, 'rebounds': 0, 'polls': 0}
        # a launch stops by itself at the first callback that needs the host, so a burst only bounds
        # how far the launch queue runs ahead: polls (a stream sync each) are what it costs
        cursor, burst = 0, 64
        while cursor < len(order):
            c = self._cloud
            k = min(burst, len(order) - cursor)
            rc = lib.mapmerge_chain_run(ws.data_ptr(), dims.ctypes.data, n_agents, len(order), k, stage.x.data_ptr(),
                                        stage.y.data_ptr(), offs.data_ptr(), v, c.x.data_ptr(), c.y.data_ptr(), c.capacity,
                                        c.count.data_ptr(), self._status.data_ptr(), self._stream())
            _native.check(rc, 'mapmerge_chain_run')
            _native.check(lib.mapmerge_chain_poll(ws.data_ptr(), dims.ctypes.data, n_agents, state, self._stream()), 'mapmerge_chain_poll')
            stats['polls'] += 1
            cursor, stalled = int(state[0]), int(state[1])
            if stalled == 0:                     # the burst ran through
                continue
            if stalled == 1:                   # the lattice moved: full filter + new voxel map
                sp = self._spare
                rc = lib.mapmerge_chain_rebuild(ws.data_ptr(), dims.ctypes.data, n_agents, stage.x.data_ptr(), stage.y.data_ptr(),
                                                offs.data_ptr(), order[cursor], v, c.x.data_ptr(), c.y.data_ptr(), c.capacity,
                                                c.count.data_ptr(), sp.x.data_ptr(), sp.y.data_ptr(), sp.count.data_ptr(),
                                                self._status.data_ptr(), vws.data_ptr(), vws.numel(), self._lattice_cap,
                                                self._stream())
                _native.check(rc, 'mapmerge_chain_rebuild')
                self._cloud, self._spare = self._spare, self._cloud
                stats['rebuilds'] += 1
                cursor += 1
            elif stalled == 3:                   # min corner may have moved inwards: exact bounds first
                rc = lib.mapmerge_chain_rebounds(ws.data_ptr(), dims.ctypes.data, n_agents, c.x.data_ptr(), c.y.data_ptr(),
                                                 c.count.data_ptr(), self._stream())
                _native.check(rc, 'mapmerge_chain_rebounds')
                stats['rebounds'] += 1
            else:
                self._check_status()
                raise OccGridError('map merge: voxel lattice does not fit the chain workspace')
        return stats

    def _extract_async(self, msg, T):
        """grid_to_pcd (+ transform) appended to the global cloud, no host read-back."""
        g = self._device_grid(msg)
        h, w = g.shape
        ws = self._workspace('extract', self._lib.mapmerge_extract_workspace_bytes(h * w))
        Tm = np.ascontiguousarray(np.asarray(T, np.float64).reshape(4, 4)) if T is not None else None
        rc = self._lib.mapmerge_extract_transform(
            g.data_ptr(), w, h, float(msg.info.resolution), float(msg.info.origin.position.x),
            float(msg.info.origin.position.y), Tm.ctypes.data if Tm is not None else None,
            self._cloud.x.data_ptr(), self._cloud.y.data_ptr(), self._cloud.capacity,
            self._cloud.count.data_ptr(), self._last.data_ptr(), self._status.data_ptr(),
            ws.data_ptr(), ws.numel(), self._stream())
        _native.check(rc, 'mapmerge_extract_transform')
