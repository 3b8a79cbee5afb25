"""Reference for per-agent maps (AgentGrids / occgrid_integrate_packets_agent_maps), built only from
the C oracle's single-grid call: per-agent maps are defined as the single-grid loop run over each
agent's records alone."""
import numpy as np

from oracle import c_oracle


def default_agent_offsets(n_agents, separation=0.0):
    """Zero offsets except row 2 = (separation, 0): the reference rule (dual_bot_mapper.py:851-852)."""
    tab = np.zeros((n_agents + 1, 2), np.float64)
    if n_agents >= 2:
        tab[2, 0] = separation
    return tab


def integrate_packets_agent_maps(packets, grids, ox, oy, res, rec_len=42, stride=None, separation=0.0,
                                 drift=None, agent_offsets=None, agent_idx=None):
    """For every agent a: c_oracle.integrate_packets over only the records whose agent (wire byte, or
    agent_idx[k]) is a, with their drift rows, onto grids[a - 1].  grids: int8 [A, H, W], updated in
    place; agent_offsets: A + 1 rows (default: default_agent_offsets).  Returns the counters of ONE
    integrate_packets over the whole batch on a scratch grid (the same records are decoded and
    walked, so the device's counters must equal them)."""
    assert grids.dtype == np.int8 and grids.ndim == 3 and grids.flags.c_contiguous
    A, h, w = grids.shape
    pk = np.ascontiguousarray(packets, dtype=np.uint8)
    if stride is None:
        stride = pk.shape[1] if pk.ndim == 2 else rec_len
    pk = pk.reshape(-1, stride)
    if agent_offsets is None:
        agent_offsets = default_agent_offsets(A, separation)
    agent_offsets = np.ascontiguousarray(agent_offsets, np.float64)
    assert agent_offsets.shape == (A + 1, 2)
    drift = None if drift is None else np.ascontiguousarray(drift, np.float64).reshape(-1, 2)
    agent_idx = None if agent_idx is None else np.ascontiguousarray(agent_idx, np.int32).reshape(-1)
    agent = pk[:, 4].astype(np.int64) if agent_idx is None else agent_idx.astype(np.int64)
    for a in range(1, A + 1):
        sel = np.flatnonzero(agent == a)
        if sel.size == 0:
            continue
        c_oracle.integrate_packets(pk[sel], grids[a - 1], ox, oy, res, rec_len=rec_len, stride=stride,
                                   drift=None if drift is None else drift[sel], agent_offsets=agent_offsets,
                                   agent_idx=None if agent_idx is None else agent_idx[sel])
    scratch = np.full((h, w), -1, np.int8)
    return c_oracle.integrate_packets(pk, scratch, ox, oy, res, rec_len=rec_len, stride=stride, drift=drift,
                                      agent_offsets=agent_offsets, agent_idx=agent_idx)
