"""B200-native occupancy-grid integration and map fusion for the swarm-SLAM server's hot path.

Import as ``occgrid_b200`` (the repository root carries an alias package, because this
directory's mandated name is not a Python identifier):

    from occgrid_b200.dual_bot_mapper import OccupancyGrid, AgentGrids
    from occgrid_b200.map_merger import MapMerger
"""
from . import _native  # noqa: F401
from ._native import OccGridError, build  # noqa: F401

__all__ = ['OccGridError', 'build']
