"""slam.net_b200 — B200-native CoreSLAM scan-to-map hot path (search + HoleMap integration).

Everything computational lives in csrc/ (sm_100a CUDA behind the C ABI of include/coreslam_b200.h);
this package is the loader plus the host-side mirror of the reference's public classes.
"""
from . import _native, parallel
from ._native import CoreSlamError, build, lib
from .coreslam import (Batch, CoreSLAMProcessor, gather_peak, HoleMap, LatticeHit, ObstacleMap, Processor, Ray, ScanCloud, ScanLog, ScanSegment, SearchResult,
                       host_map_checksum, host_obstacle_checksum, philox_offsets, scan_segments_to_cloud)

__all__ = ["Batch", "parallel", "CoreSLAMProcessor", "HoleMap", "LatticeHit", "Processor", "Ray", "ScanCloud", "ScanLog", "ScanSegment", "SearchResult",
           "CoreSlamError", "gather_peak", "build", "lib", "host_map_checksum", "host_obstacle_checksum", "philox_offsets", "scan_segments_to_cloud", "_native"]
