"""
ORACLE — TEST INFRASTRUCTURE ONLY.  ctypes front-end of oracle/occgrid_oracle.c.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

COUNTER_NAMES = ('packets', 'accepted', 'dropped', 'bad_pose', 'beams', 'hits', 'updates', 'spare')
_lib = None


def lib():
    global _lib
    if _lib is None:
        # build() compares modification times and returns at once when the library is current, so
        # a library left over from older sources is rebuilt rather than loaded without new symbols
        _lib = C.CDLL(_build.build(force=bool(os.environ.get('ORACLE_REBUILD'))))
        for fn in (_lib.oracle_integrate_packets, _lib.oracle_accumulate_packets):
            fn.restype = C.c_int
            fn.argtypes = [
                C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                C.c_double, C.c_double, C.c_double, C.c_int64, C.c_int64,
                C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
        _lib.oracle_update_rays.restype = C.c_int
        _lib.oracle_update_rays.argtypes = [
            C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_double, C.c_double,
            C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
        _lib.oracle_bresenham.restype = C.c_int64
        _lib.oracle_bresenham.argtypes = [C.c_int64] * 4 + [C.c_void_p, C.c_void_p, C.c_int64]
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _packets(fn, packets, plane, ox, oy, res, rec_len, stride, separation, drift, agent_offsets, agent_idx,
             window, size_x, size_y):
    pk = np.ascontiguousarray(packets, dtype=np.uint8)
    if stride is None:
        stride = pk.shape[1] if pk.ndim == 2 else rec_len
    n = pk.size // stride
    if agent_offsets is None:
        agent_offsets = np.array([[0.0, 0.0], [0.0, 0.0], [separation, 0.0]], np.float64)
    agent_offsets = np.ascontiguousarray(agent_offsets, np.float64)
    n_agents = agent_offsets.shape[0] - 1
    if drift is not None:
        drift = np.ascontiguousarray(drift, np.float64)
        assert drift.shape == (n, 2)
    if agent_idx is not None:
        agent_idx = np.ascontiguousarray(agent_idx, np.int32)
    assert plane.flags.c_contiguous
    h, w = plane.shape[:2]
    wx0, wy0 = window if window is not None else (0, 0)
    sx = size_x if size_x is not None else w
    sy = size_y if size_y is not None else h
    counters = np.zeros(8, np.uint64)
    rc = fn(_ptr(pk), n, stride, rec_len, _ptr(agent_idx), _ptr(drift), _ptr(agent_offsets), n_agents,
            ox, oy, res, sx, sy, wx0, wy0, w, h, _ptr(plane), _ptr(counters))
    if rc != 0:
        raise ValueError(f'{fn.__name__} rc={rc}')
    return dict(zip(COUNTER_NAMES, (int(c) for c in counters)))


def integrate_packets(packets, grid, ox, oy, res, rec_len=42, stride=None, separation=0.0,
                      drift=None, agent_offsets=None, agent_idx=None, window=None,
                      size_x=None, size_y=None):
    """packets: uint8 array [n, stride] (or flat).  grid: int8 [H, W], updated in place.
    window=(x0, y0) places `grid` as a tile of a (size_y, size_x) global grid."""
    assert grid.dtype == np.int8 and grid.ndim == 2
    return _packets(lib().oracle_integrate_packets, packets, grid, ox, oy, res, rec_len, stride, separation,
                    drift, agent_offsets, agent_idx, window, size_x, size_y)


def accumulate_packets(packets, counts, ox, oy, res, rec_len=42, stride=None, separation=0.0,
                       drift=None, agent_offsets=None, agent_idx=None, window=None,
                       size_x=None, size_y=None):
    """Count mode of integrate_packets: counts int32 [H, W, 2] = {miss, hit} per cell, added to in
    place.  Same records, keywords and counters; the cells integrate_packets would store FREE
    count one miss each, the OCCUPIED end cell of a valid hit one hit."""
    assert counts.dtype == np.int32 and counts.ndim == 3 and counts.shape[2] == 2
    return _packets(lib().oracle_accumulate_packets, packets, counts, ox, oy, res, rec_len, stride, separation,
                    drift, agent_offsets, agent_idx, window, size_x, size_y)


def update_rays(rays, hit, grid, ox, oy, res):
    rays = np.ascontiguousarray(rays, np.float64)
    hit = np.ascontiguousarray(hit, np.uint8)
    h, w = grid.shape
    counters = np.zeros(8, np.uint64)
    lib().oracle_update_rays(_ptr(rays), _ptr(hit), rays.shape[0], ox, oy, res, w, h,
                             _ptr(grid), _ptr(counters))
    return dict(zip(COUNTER_NAMES, (int(c) for c in counters)))


def bresenham(x0, y0, x1, y1):
    cap = max(abs(x1 - x0), abs(y1 - y0)) + 1
    xs = np.empty(cap, np.int32)
    ys = np.empty(cap, np.int32)
    n = lib().oracle_bresenham(x0, y0, x1, y1, _ptr(xs), _ptr(ys), cap)
    assert n == cap
    return list(zip(xs.tolist(), ys.tolist()))
