"""Host-side mirror of the reference's public surface for the CoreSLAM hot path, over the C ABI.

Same names, argument meaning and call order as the C# classes they stand in for
(paths relative to /root/reference):

  Ray, ScanSegment, ScanCloud   BaseSLAM/Ray.cs:10-32, ScanSegment.cs:13-29, ScanCloud.cs:10-21
  HoleMap                       CoreSLAM/HoleMap.cs:17-55
  ObstacleMap                   CoreSLAM/ObstacleMap.cs:11-44
  CoreSLAMProcessor             CoreSLAM/CoreSLAMProcessor.cs:18-775 (ctor :119, Reset :167, Update :717,
                                Dispose :757; properties :40-106)

The reference toolchain (.NET) is not available here, so this mirror is Python over ctypes; the C#
P/Invoke wrapper a SLAM.NET maintainer would add is in INTEGRATION.md / dotnet/.  All compute goes through
libcoreslam_b200.so (sm_100a kernels); nothing in this module computes distances or draws rays itself.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

from . import _native as N

_fp = C.POINTER(C.c_float)


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(_fp)


# ------------------------------------------------------------------------------------------------
# BaseSLAM data types
# ------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Ray:
    """BaseSLAM/Ray.cs:10-32 — polar point (radians, metres)."""
    Angle: float
    Radius: float


@dataclass
class ScanSegment:
    """BaseSLAM/ScanSegment.cs:13-29.  Rays may be a list of Ray or an (n,2) float32 array of
    (angle, radius) — the array form is what a lidar driver fills in place."""
    Rays: object = field(default_factory=list)
    Pose: Sequence[float] = (0.0, 0.0, 0.0)
    IsLast: bool = False

    def rays_array(self) -> np.ndarray:
        if isinstance(self.Rays, np.ndarray):
            return _f32(self.Rays).reshape(-1, 2)
        return _f32([(r.Angle, r.Radius) for r in self.Rays]).reshape(-1, 2)


@dataclass
class ScanCloud:
    """BaseSLAM/ScanCloud.cs:10-21 — Points is an (n,2) float32 array (List<Vector2>)."""
    Pose: Sequence[float] = (0.0, 0.0, 0.0)
    Points: np.ndarray = field(default_factory=lambda: np.zeros((0, 2), dtype=np.float32))


def pack_segments(segments: Sequence[ScanSegment]):
    """List<ScanSegment> -> the flat arrays cs_update_segments takes: rays (n,2) = (angle, radius) of all segments back
    to back, seg_first (n_segments+1) int32, seg_poses (n_segments,3)."""
    arrays = [seg.rays_array() for seg in segments]
    rays = np.concatenate(arrays, axis=0) if arrays else np.zeros((0, 2), dtype=np.float32)
    first = np.zeros(len(arrays) + 1, dtype=np.int32)
    if arrays:
        first[1:] = np.cumsum([a.shape[0] for a in arrays])
    poses = _f32([tuple(seg.Pose) for seg in segments]).reshape(-1, 3)
    return _f32(rays), first, poses


def scan_segments_to_cloud(segments: Sequence[ScanSegment], odometry_pose) -> ScanCloud:
    """ScanSegmentsToCloud, CoreSLAM/CoreSLAMProcessor.cs:187-207, on the host (the product path runs it on the
    device: Processor.update_segments / Processor.segments_to_cloud; this twin exists for comparisons).
    cosf/sinf come from the library's host build of its glibc-identical routine."""
    odo = _f32(odometry_pose)
    out = []
    L = N.lib()
    for seg in segments:
        pose = _f32(seg.Pose) - odo  # :194
        rays = seg.rays_array()
        ang = _f32(rays[:, 0] + pose[2])  # r.Angle + pose.Z
        c = np.empty_like(ang)
        s = np.empty_like(ang)
        if ang.size:
            L.cs_host_sincos(_ptr(ang), ang.size, _ptr(c), _ptr(s))
        pts = np.empty((ang.size, 2), dtype=np.float32)
        pts[:, 0] = pose[0] + rays[:, 1] * c  # :200
        pts[:, 1] = pose[1] + rays[:, 1] * s  # :201
        out.append(pts)
    points = np.concatenate(out, axis=0) if out else np.zeros((0, 2), dtype=np.float32)
    return ScanCloud(Pose=tuple(float(v) for v in odo), Points=points)


# ------------------------------------------------------------------------------------------------
# low-level handle wrapper
# ------------------------------------------------------------------------------------------------
@dataclass
class SearchResult:
    pose: np.ndarray
    distance: int
    index: int
    searched: bool
    visits: int


@dataclass
class LatticeHit:
    """One hypothesis of cs_relocalize: the lattice pose as evaluated (theta not normalised), its distance
    (CalculateDistanceSISD, CoreSLAMProcessor.cs:226-259) and its flat lattice index."""
    pose: np.ndarray
    distance: int
    index: int


def _result(r: N.Result) -> SearchResult:
    return SearchResult(np.array(list(r.pose), dtype=np.float32), int(r.distance), int(r.index), bool(r.searched),
                        int(r.visits))


class ScanLog:
    """Device-resident scan log (cs_scanlog_*): points, odometry and optional candidate offsets of a
    whole replay, uploaded once."""

    def __init__(self, n_scans: int, max_points: int, n_offsets: int = 0, device: int = 0):
        self._h = C.c_void_p()
        self.n_scans, self.max_points, self.n_offsets = n_scans, max_points, n_offsets
        N.check(N.lib().cs_scanlog_create(device, n_scans, max_points, n_offsets, C.byref(self._h)))

    def set(self, scan: int, points, odometry_pose, offsets=None):
        pts = _f32(points).reshape(-1, 2)
        odo = _f32(odometry_pose)
        off = None if offsets is None else _f32(offsets).reshape(-1, 3)
        if off is not None and off.shape[0] != self.n_offsets:
            raise ValueError("offsets must have n_offsets rows")
        N.check(N.lib().cs_scanlog_set(self._h, scan, _ptr(pts), pts.shape[0], _ptr(odo), _ptr(off)))

    def upload(self):
        N.check(N.lib().cs_scanlog_upload(self._h))

    def save(self, path: str):
        """Write the log as a CSLG file (cs_scanlog_save; format in include/coreslam_b200.h)."""
        N.check(N.lib().cs_scanlog_save(self._h, str(path).encode()))

    @classmethod
    def load(cls, path: str, device: int = 0) -> "ScanLog":
        """A device-resident log from a CSLG file (cs_scanlog_load): created, filled and uploaded."""
        n, mp, no = C.c_int32(), C.c_int32(), C.c_int32()
        N.check(N.lib().cs_scanlog_file_info(str(path).encode(), C.byref(n), C.byref(mp), C.byref(no)))
        self = cls.__new__(cls)
        self._h = C.c_void_p()
        self.n_scans, self.max_points, self.n_offsets = n.value, mp.value, no.value
        N.check(N.lib().cs_scanlog_load(device, str(path).encode(), C.byref(self._h)))
        return self

    def close(self):
        if self._h:
            N.lib().cs_scanlog_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Processor:
    """Thin object wrapper over a cs_processor handle (one per CoreSLAMProcessor)."""

    def __init__(self, physical_map_size: float, hole_map_size: int, start_pose, sigma_xy: float, sigma_theta: float,
                 iterations_per_thread: int, num_search_threads: int, *, device: int = 0, max_points: int = 0,
                 seed: int = 0, stream: int = 0, flags: int = 0, obstacle_map_size: int = 0):
        cfg = N.Config()
        cfg.physical_map_size = physical_map_size
        cfg.hole_map_size = hole_map_size
        cfg.obstacle_map_size = obstacle_map_size
        cfg.start_pose = (C.c_float * 3)(*[float(v) for v in start_pose])
        cfg.sigma_xy = sigma_xy
        cfg.sigma_theta = sigma_theta
        cfg.iterations_per_thread = iterations_per_thread
        cfg.num_search_threads = num_search_threads
        cfg.device = device
        cfg.max_points = max_points
        cfg.seed = seed
        cfg.stream = stream or None
        cfg.flags = flags
        self._h = C.c_void_p()
        N.check(N.lib().cs_create(C.byref(cfg), C.byref(self._h)))
        self.size = hole_map_size
        self.n_cand = max(num_search_threads, 1) * iterations_per_thread
        size = C.c_int32()
        scale = C.c_float()
        N.lib().cs_get_map_info(self._h, C.byref(size), C.byref(scale))
        self.scale = float(scale.value)
        self.seed = seed
        self.sigma_xy, self.sigma_theta = sigma_xy, sigma_theta
        self.obstacle_size = obstacle_map_size
        N.lib().cs_get_obstacle_map_info(self._h, C.byref(size), C.byref(scale))
        self.obstacle_scale = float(scale.value)

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            N.lib().cs_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, status):
        N.check(status, self._h)

    def reset(self):
        self._ck(N.lib().cs_reset(self._h))

    def sync(self):
        self._ck(N.lib().cs_sync(self._h))

    # -- properties -------------------------------------------------------------------------------
    def set_quality(self, q: int):
        self._ck(N.lib().cs_set_quality(self._h, int(q)))

    def set_hole_width(self, w: float):
        self._ck(N.lib().cs_set_hole_width(self._h, float(w)))

    def set_position_search_beginning(self, n: int):
        self._ck(N.lib().cs_set_position_search_beginning(self._h, int(n)))

    def get_pose(self) -> np.ndarray:
        p = np.zeros(3, dtype=np.float32)
        self._ck(N.lib().cs_get_pose(self._h, _ptr(p)))
        return p

    def set_pose(self, pose, last_odometry=(0, 0, 0), scan_count: int = 0):
        self._ck(N.lib().cs_set_pose(self._h, _ptr(_f32(pose)), _ptr(_f32(last_odometry)), int(scan_count)))

    # -- hot path ---------------------------------------------------------------------------------
    def search(self, points, search_pose, cand_poses=None, cand_cs=None, scan_index: int = 0, want_distances=True):
        pts = _f32(points).reshape(-1, 2)
        sp = _f32(search_pose)
        cp = None if cand_poses is None else _f32(cand_poses).reshape(-1, 3)
        n_cand = self.n_cand if cp is None else cp.shape[0]
        cs = None if cand_cs is None else _f32(cand_cs).reshape(-1, 2)
        if cs is not None and cs.shape[0] != n_cand + 1:
            raise ValueError("cand_cs needs n_cand+1 rows (row 0 = searchPose)")
        d = np.zeros(n_cand + 1, dtype=np.int32) if want_distances else None
        r = N.Result()
        self._ck(N.lib().cs_search(self._h, _ptr(pts), pts.shape[0], _ptr(sp), _ptr(cp), _ptr(cs), n_cand, scan_index,
                                   C.byref(r), None if d is None else d.ctypes.data_as(C.POINTER(C.c_int32))))
        return _result(r), d

    @staticmethod
    def _lattice(origin, step, count) -> N.Lattice:
        lat = N.Lattice()
        lat.origin = (C.c_float * 3)(*[float(v) for v in origin])
        lat.step = (C.c_float * 3)(*[float(v) for v in step])
        lat.count = (C.c_int32 * 3)(*[int(v) for v in count])
        return lat

    def relocalize(self, points, origin, step, count, window: int = 0, k: int = 1, want_distances=False):
        """cs_relocalize: the distance of the scan at every pose of the lattice origin + (ix, iy, it) * step, count =
        (nx, ny, ntheta) poses, and the k best poses that are strict local minima of (distance, flat index) within
        +-window lattice steps (include/coreslam_b200.h).  Returns (hits, volume): hits is a list of LatticeHit, best
        first; volume the (ntheta, ny, nx) int32 distances when want_distances, else None.  The handle's state is
        left as it was."""
        pts = _f32(points).reshape(-1, 2)
        lat = self._lattice(origin, step, count)
        hits = (N.LatticeHit * N.LATTICE_MAX_HITS)()
        n = C.c_int32(0)
        vol = None
        if want_distances and min(lat.count) >= 1 and lat.count[0] * lat.count[1] * lat.count[2] <= N.LATTICE_MAX_POSES:
            vol = np.empty((lat.count[2], lat.count[1], lat.count[0]), dtype=np.int32)  # (else the call fails)
        self._ck(N.lib().cs_relocalize(self._h, _ptr(pts), pts.shape[0], C.byref(lat), int(window), int(k), hits,
                                       C.byref(n), None if vol is None else vol.ctypes.data_as(C.POINTER(C.c_int32))))
        out = [LatticeHit(np.array(list(hits[i].pose), dtype=np.float32), int(hits[i].distance), int(hits[i].index))
               for i in range(n.value)]
        return out, vol

    def relocalize_bounded(self, points, origin, step, count, window: int = 0, k: int = 1):
        """cs_relocalize_bounded: the hits of relocalize for the same lattice, window and k, by branch and bound, on
        lattices of up to LATTICE_MAX_POSES_BOUNDED poses.  Returns (hits, stats): stats is a dict of
        cs_relocalize_stats (poses, evaluated, bounded, levels, passes, upper_bound).  The handle's state is left as it
        was."""
        pts = _f32(points).reshape(-1, 2)
        lat = self._lattice(origin, step, count)
        hits = (N.LatticeHit * N.LATTICE_MAX_HITS)()
        n = C.c_int32(0)
        st = N.RelocalizeStats()
        self._ck(N.lib().cs_relocalize_bounded(self._h, _ptr(pts), pts.shape[0], C.byref(lat), int(window), int(k), hits,
                                               C.byref(n), C.byref(st)))
        out = [LatticeHit(np.array(list(hits[i].pose), dtype=np.float32), int(hits[i].distance), int(hits[i].index))
               for i in range(n.value)]
        return out, {f: int(getattr(st, f)) for f, _ in N.RelocalizeStats._fields_ if f != "reserved"}

    @staticmethod
    def _sequence(scans, odometry):
        """scans (K arrays of (x, y) points) and odometry (K poses) -> the concatenated points, scan_first and odometry"""
        pts = [_f32(p).reshape(-1, 2) for p in scans]
        first = np.zeros(len(pts) + 1, dtype=np.int32)
        first[1:] = np.cumsum([p.shape[0] for p in pts])
        cat = np.ascontiguousarray(np.concatenate(pts) if pts else np.zeros((0, 2), np.float32))
        odo = _f32(odometry).reshape(-1, 3)
        if odo.shape[0] != len(pts):
            raise ValueError("odometry needs one pose per scan")
        return cat, first, odo

    def relocalize_sequence(self, scans, odometry, origin, step, count, window: int = 0, k: int = 1, want_distances=False):
        """cs_relocalize_sequence: relocalize with the last few scans.  scans: K <= SEQUENCE_MAX_SCANS arrays of points,
        each in its own lidar frame, oldest first; odometry: their K odometry poses.  The lattice pose is the pose of the
        last scan; every other scan is placed by its odometry relative to the last, and a pose's distance is the sum of
        the scans' distances (include/coreslam_b200.h).  Returns (hits, volume) as relocalize."""
        pts, first, odo = self._sequence(scans, odometry)
        lat = self._lattice(origin, step, count)
        hits = (N.LatticeHit * N.LATTICE_MAX_HITS)()
        n = C.c_int32(0)
        vol = None
        if want_distances and min(lat.count) >= 1 and lat.count[0] * lat.count[1] * lat.count[2] <= N.LATTICE_MAX_POSES:
            vol = np.empty((lat.count[2], lat.count[1], lat.count[0]), dtype=np.int32)  # (else the call fails)
        self._ck(N.lib().cs_relocalize_sequence(self._h, _ptr(pts), first.ctypes.data_as(C.POINTER(C.c_int32)), _ptr(odo),
                                                len(first) - 1, C.byref(lat), int(window), int(k), hits, C.byref(n),
                                                None if vol is None else vol.ctypes.data_as(C.POINTER(C.c_int32))))
        out = [LatticeHit(np.array(list(hits[i].pose), dtype=np.float32), int(hits[i].distance), int(hits[i].index))
               for i in range(n.value)]
        return out, vol

    def relocalize_sequence_bounded(self, scans, odometry, origin, step, count, window: int = 0, k: int = 1):
        """cs_relocalize_sequence_bounded: the hits of relocalize_sequence by branch and bound, on lattices of up to
        LATTICE_MAX_POSES_BOUNDED poses.  Returns (hits, stats) as relocalize_bounded."""
        pts, first, odo = self._sequence(scans, odometry)
        lat = self._lattice(origin, step, count)
        hits = (N.LatticeHit * N.LATTICE_MAX_HITS)()
        n = C.c_int32(0)
        st = N.RelocalizeStats()
        self._ck(N.lib().cs_relocalize_sequence_bounded(self._h, _ptr(pts), first.ctypes.data_as(C.POINTER(C.c_int32)),
                                                        _ptr(odo), len(first) - 1, C.byref(lat), int(window), int(k), hits,
                                                        C.byref(n), C.byref(st)))
        out = [LatticeHit(np.array(list(hits[i].pose), dtype=np.float32), int(hits[i].distance), int(hits[i].index))
               for i in range(n.value)]
        return out, {f: int(getattr(st, f)) for f, _ in N.RelocalizeStats._fields_ if f != "reserved"}

    def integrate(self, points, pose, pose_cs=None, wait=True) -> int:
        pts = _f32(points).reshape(-1, 2)
        v = C.c_int64(-1)
        cs = None if pose_cs is None else _f32(pose_cs)
        self._ck(N.lib().cs_integrate(self._h, _ptr(pts), pts.shape[0], _ptr(_f32(pose)), _ptr(cs),
                                      C.byref(v) if wait else None))
        return int(v.value)

    def update(self, points, odometry_pose, cand_offsets=None) -> SearchResult:
        pts = _f32(points).reshape(-1, 2)
        off = None if cand_offsets is None else _f32(cand_offsets).reshape(-1, 3)
        if off is not None and off.shape[0] != self.n_cand:
            raise ValueError("cand_offsets needs T*I = %d rows" % self.n_cand)
        r = N.Result()
        self._ck(N.lib().cs_update(self._h, _ptr(pts), pts.shape[0], _ptr(_f32(odometry_pose)), _ptr(off), C.byref(r)))
        return _result(r)

    def update_segments(self, segments: Sequence[ScanSegment], cand_offsets=None) -> SearchResult:
        """CoreSLAMProcessor.Update(List<ScanSegment>) whole, ScanSegmentsToCloud on the device (cs_update_segments)."""
        rays, first, poses = pack_segments(segments)
        off = None if cand_offsets is None else _f32(cand_offsets).reshape(-1, 3)
        if off is not None and off.shape[0] != self.n_cand:
            raise ValueError("cand_offsets needs T*I = %d rows" % self.n_cand)
        r = N.Result()
        self._ck(N.lib().cs_update_segments(self._h, _ptr(rays), first.ctypes.data_as(N._ip), _ptr(poses), rays.shape[0],
                                            poses.shape[0], _ptr(off), C.byref(r)))
        return _result(r)

    def segments_to_cloud(self, segments: Sequence[ScanSegment], odometry_pose) -> np.ndarray:
        """ScanSegmentsToCloud (:187-207) on the device for an explicit odometry pose; returns the (n,2) points."""
        rays, first, poses = pack_segments(segments)
        out = np.empty((rays.shape[0], 2), dtype=np.float32)
        self._ck(N.lib().cs_segments_to_cloud(self._h, _ptr(rays), first.ctypes.data_as(N._ip), _ptr(poses), rays.shape[0],
                                              poses.shape[0], _ptr(_f32(odometry_pose)), _ptr(out)))
        return out

    # -- multi-GPU candidate split (cs_update_begin / cs_update_finish) -----------------------------
    def update_begin(self, points, odometry_pose, cand_offsets, cand_first: int, cand_count: int) -> int:
        """Launches the search over flat candidate indices [cand_first, cand_first+cand_count) and returns
        the DEVICE address of the 8-byte packed arg-min to be min-reduced over the GPUs before
        update_finish()."""
        pts = _f32(points).reshape(-1, 2)
        off = None if cand_offsets is None else _f32(cand_offsets).reshape(-1, 3)
        if off is not None and off.shape[0] != self.n_cand:
            raise ValueError("cand_offsets needs T*I = %d rows (the full table on every GPU)" % self.n_cand)
        key = C.c_void_p()
        self._ck(N.lib().cs_update_begin(self._h, _ptr(pts), pts.shape[0], _ptr(_f32(odometry_pose)), _ptr(off),
                                         int(cand_first), int(cand_count), C.byref(key)))
        return int(key.value or 0)

    def update_finish(self) -> SearchResult:
        r = N.Result()
        self._ck(N.lib().cs_update_finish(self._h, C.byref(r)))
        return _result(r)

    # -- candidate-split group with the exchange inside the search kernel (cs_group_*) ---------------
    def group_export(self) -> bytes:
        """64-byte handle of this rank's exchange table (cs_group_export), to be passed to every other rank."""
        buf = (C.c_ubyte * 64)()
        self._ck(N.lib().cs_group_export(self._h, C.addressof(buf)))
        return bytes(buf)

    def group_attach(self, rank: int, world: int, handles: Sequence[bytes]):
        """One process per GPU: `handles[p]` = rank p's group_export() (entry `rank` is ignored)."""
        blob = (C.c_ubyte * (64 * world))()
        for p_, hd in enumerate(handles):
            for i, b in enumerate(bytes(hd)[:64]):
                blob[64 * p_ + i] = b
        self._ck(N.lib().cs_group_attach(self._h, int(rank), int(world), C.addressof(blob)))

    def group_attach_local(self, rank: int, world: int, peers: Sequence["Processor"]):
        """One process, several handles (one per device, or several on one device)."""
        arr = (C.c_void_p * world)(*[p_._h for p_ in peers])
        self._ck(N.lib().cs_group_attach_local(self._h, int(rank), int(world), arr))

    def group_detach(self):
        self._ck(N.lib().cs_group_detach(self._h))

    def replay(self, log: ScanLog, first: int = 0, count: Optional[int] = None, want_results=True):
        count = log.n_scans - first if count is None else count
        res = (N.Result * count)() if want_results else None
        self._ck(N.lib().cs_replay(self._h, log._h, first, count, res))
        return [_result(r) for r in res] if want_results else None

    # -- map --------------------------------------------------------------------------------------
    def map_download(self) -> np.ndarray:
        px = np.empty(self.size * self.size, dtype=np.uint16)
        self._ck(N.lib().cs_map_download(self._h, px.ctypes.data))
        return px

    def map_upload(self, pixels):
        px = np.ascontiguousarray(pixels, dtype=np.uint16).reshape(-1)
        if px.size != self.size * self.size:
            raise ValueError("pixels must have Size*Size entries")
        self._ck(N.lib().cs_map_upload(self._h, px.ctypes.data))

    def map_fill(self, value: int):
        self._ck(N.lib().cs_map_fill(self._h, int(value)))

    def map_export_begin(self, fmt: int, out: np.ndarray):
        """Asynchronous export (cs_map_export_begin): `out` must stay alive and untouched until map_export_wait()."""
        self._ck(N.lib().cs_map_export_begin(self._h, int(fmt), out.ctypes.data))

    def map_export_wait(self):
        self._ck(N.lib().cs_map_export_wait(self._h))

    def map_packed(self) -> np.ndarray:
        out = np.empty(self.size * self.size // 2, dtype=np.uint8)
        self._ck(N.lib().cs_map_packed(self._h, out.ctypes.data))
        return out

    def map_checksum(self) -> int:
        v = C.c_uint64()
        self._ck(N.lib().cs_map_checksum(self._h, C.byref(v)))
        return int(v.value)

    # -- ObstacleMap (needs obstacle_map_size > 0) -------------------------------------------------
    def set_unmapped_obstacle_hits(self, v: int):
        self._ck(N.lib().cs_set_unmapped_obstacle_hits(self._h, int(v)))

    def set_max_obstacle_hits(self, v: int):
        self._ck(N.lib().cs_set_max_obstacle_hits(self._h, int(v)))

    def obstacle_map_download(self) -> np.ndarray:
        px = np.empty((self.obstacle_size, self.obstacle_size), dtype=np.int8)
        self._ck(N.lib().cs_obstacle_map_download(self._h, px.ctypes.data))
        return px

    def obstacle_map_upload(self, pixels):
        px = np.ascontiguousarray(pixels, dtype=np.int8).reshape(-1)
        if px.size != self.obstacle_size * self.obstacle_size:
            raise ValueError("pixels must have Size*Size entries")
        self._ck(N.lib().cs_obstacle_map_upload(self._h, px.ctypes.data))

    def obstacle_map_fill(self, value: int):
        self._ck(N.lib().cs_obstacle_map_fill(self._h, int(value)))

    def obstacle_visits(self) -> int:
        v = C.c_int64()
        self._ck(N.lib().cs_get_obstacle_visits(self._h, C.byref(v)))
        return int(v.value)

    # -- diagnostics ------------------------------------------------------------------------------
    def set_flags(self, flags: int):
        self._ck(N.lib().cs_set_flags(self._h, int(flags)))

    def timing(self) -> N.Timing:
        t = N.Timing()
        self._ck(N.lib().cs_get_timing(self._h, C.byref(t)))
        return t

    def distances(self, count: Optional[int] = None) -> np.ndarray:
        count = self.n_cand + 1 if count is None else count
        d = np.zeros(count, dtype=np.int32)
        self._ck(N.lib().cs_get_distances(self._h, d.ctypes.data_as(C.POINTER(C.c_int32)), count))
        return d

    def rays(self, n_points: int) -> np.ndarray:
        r = np.zeros((n_points, 6), dtype=np.int32)
        self._ck(N.lib().cs_get_rays(self._h, r.ctypes.data_as(C.POINTER(C.c_int32)), n_points))
        return r

    def visits(self) -> int:
        v = C.c_int64()
        self._ck(N.lib().cs_get_visits(self._h, C.byref(v)))
        return int(v.value)

    def ring_cycles(self, count: Optional[int] = None) -> np.ndarray:
        """Diagnostics (first call enables recording): (count, 8) timeline records of the last step; record b < size
        is sub-task b of the draw kernel (cs_wedge_kernel), see cs_get_ring_cycles in include/coreslam_b200.h."""
        count = self.size if count is None else count
        out = np.zeros(count * 8, dtype=np.int64)
        self._ck(N.lib().cs_get_ring_cycles(self._h, out.ctypes.data_as(C.POINTER(C.c_int64)), count * 8))
        return out.reshape(count, 8)

    def search_plan(self, n_points: int, n_cand: Optional[int] = None) -> dict:
        """Which search kernel / launch shape a scan gets (cs_get_search_plan)."""
        plan = (C.c_int32 * 5)()
        self._ck(N.lib().cs_get_search_plan(self._h, int(n_points), int(self.n_cand if n_cand is None else n_cand), plan))
        return {"kernel": "cs_sort_kernel + cs_search2_kernel (heading-sorted slabs)" if plan[0] else "cs_search_kernel (warp per candidate)",
                "slab": bool(plan[0]), "grid": [int(plan[1]), int(plan[2])], "threads": int(plan[3]), "points_per_block": int(plan[4])}

    def launch_count(self) -> int:
        v = C.c_uint64()
        self._ck(N.lib().cs_get_launch_count(self._h, C.byref(v)))
        return int(v.value)


class Batch:
    """N independent sessions on one GPU (cs_batch_*): a parameter sweep / many replays advanced in
    lockstep, one kernel launch per stage for all of them.  obstacle_map_size > 0 gives every session its own
    ObstacleMap, updated by every step as in a Processor."""

    def __init__(self, n_sessions: int, physical_map_size: float, hole_map_size: int, start_poses, sigma_xy, sigma_theta,
                 iterations_per_thread: int, num_search_threads: int, *, device: int = 0, max_points: int = 0,
                 seeds=None, stream: int = 0, flags: int = 0, obstacle_map_size: int = 0):
        cfgs = (N.Config * n_sessions)()
        start_poses = np.broadcast_to(_f32(start_poses), (n_sessions, 3))
        sxy = np.broadcast_to(np.asarray(sigma_xy, dtype=np.float32), (n_sessions,))
        sth = np.broadcast_to(np.asarray(sigma_theta, dtype=np.float32), (n_sessions,))
        seeds = np.arange(n_sessions, dtype=np.uint64) if seeds is None else np.asarray(seeds, dtype=np.uint64)
        for j in range(n_sessions):
            c = cfgs[j]
            c.physical_map_size = physical_map_size
            c.hole_map_size = hole_map_size
            c.start_pose = (C.c_float * 3)(*[float(v) for v in start_poses[j]])
            c.sigma_xy = float(sxy[j])
            c.sigma_theta = float(sth[j])
            c.iterations_per_thread = iterations_per_thread
            c.num_search_threads = num_search_threads
            c.device = device
            c.max_points = max_points
            c.seed = int(seeds[j])
            c.stream = stream or None
            c.flags = flags
            c.obstacle_map_size = obstacle_map_size
        self._h = C.c_void_p()
        N.check(N.lib().cs_batch_create(cfgs, n_sessions, C.byref(self._h)))
        self.n = n_sessions
        self.size = hole_map_size
        self.obstacle_size = obstacle_map_size
        self.n_cand = max(num_search_threads, 1) * iterations_per_thread
        self.max_points = max_points if max_points > 0 else 16384  # stride of the points array = cfg.max_points, odd or even
        self.seeds, self.sigma_xy, self.sigma_theta = seeds, sxy, sth

    def _ck(self, status):
        N.check(status, batch=self._h)

    def close(self):
        if getattr(self, "_h", None):
            N.lib().cs_batch_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_params(self, session: int, quality: int, hole_width: float):
        self._ck(N.lib().cs_batch_set_params(self._h, int(session), int(quality), float(hole_width)))

    def update(self, points: Sequence[np.ndarray], odometry, cand_offsets=None, want_results=True):
        """points: one (P_j, 2) array per session; odometry (n, 3); cand_offsets (n, T*I, 3) or None."""
        buf = np.zeros((self.n, self.max_points, 2), dtype=np.float32)
        npts = np.zeros(self.n, dtype=np.int32)
        for j, p in enumerate(points):
            p = _f32(p).reshape(-1, 2)
            buf[j, :p.shape[0]] = p
            npts[j] = p.shape[0]
        odo = _f32(odometry).reshape(self.n, 3)
        off = None if cand_offsets is None else _f32(cand_offsets).reshape(self.n, self.n_cand, 3)
        res = (N.Result * self.n)() if want_results else None
        self._ck(N.lib().cs_batch_update(self._h, _ptr(buf), npts.ctypes.data_as(C.POINTER(C.c_int32)), _ptr(odo), _ptr(off), res))
        return [_result(r) for r in res] if want_results else None

    def submit(self, points: Sequence[np.ndarray], odometry, cand_offsets=None):
        """cs_batch_submit: stage and queue one Update of every session, return at once (at most two steps may wait for
        collect()).  Arguments as update()."""
        buf = np.zeros((self.n, self.max_points, 2), dtype=np.float32)
        npts = np.zeros(self.n, dtype=np.int32)
        for j, p in enumerate(points):
            p = _f32(p).reshape(-1, 2)
            buf[j, :p.shape[0]] = p
            npts[j] = p.shape[0]
        odo = _f32(odometry).reshape(self.n, 3)
        off = None if cand_offsets is None else _f32(cand_offsets).reshape(self.n, self.n_cand, 3)
        self._ck(N.lib().cs_batch_submit(self._h, _ptr(buf), npts.ctypes.data_as(C.POINTER(C.c_int32)), _ptr(odo), _ptr(off)))

    def collect(self, want_results=True):
        """cs_batch_collect: wait for the oldest submitted step; its result records."""
        res = (N.Result * self.n)() if want_results else None
        self._ck(N.lib().cs_batch_collect(self._h, res))
        return [_result(r) for r in res] if want_results else None

    def replay(self, log: ScanLog, first: int = 0, count: Optional[int] = None, want_results=True):
        count = log.n_scans - first if count is None else count
        res = (N.Result * self.n)() if want_results else None
        self._ck(N.lib().cs_batch_replay(self._h, log._h, first, count, res))
        return [_result(r) for r in res] if want_results else None

    def sync(self):
        self._ck(N.lib().cs_batch_sync(self._h))

    def poses(self) -> np.ndarray:
        out = np.zeros((self.n, 3), dtype=np.float32)
        self._ck(N.lib().cs_batch_get_poses(self._h, _ptr(out)))
        return out

    def map_download(self, session: int) -> np.ndarray:
        px = np.empty(self.size * self.size, dtype=np.uint16)
        self._ck(N.lib().cs_batch_map_download(self._h, int(session), px.ctypes.data))
        return px

    def map_checksums(self) -> np.ndarray:
        out = np.zeros(self.n, dtype=np.uint64)
        self._ck(N.lib().cs_batch_map_checksums(self._h, out.ctypes.data_as(C.POINTER(C.c_uint64))))
        return out

    def launch_count(self) -> int:
        v = C.c_uint64()
        self._ck(N.lib().cs_batch_get_launch_count(self._h, C.byref(v)))
        return int(v.value)

    def reset(self):
        """CoreSLAMProcessor.Reset of every session: maps refilled, poses back to the start poses, scan count 0."""
        self._ck(N.lib().cs_batch_reset(self._h))

    # -- ObstacleMaps (needs obstacle_map_size > 0) -------------------------------------------------
    def set_obstacle_params(self, session: int, unmapped_hits: int, max_hits: int):
        """session < 0: all.  max_hits applies from the next step, unmapped_hits from the next reset()."""
        self._ck(N.lib().cs_batch_set_obstacle_params(self._h, int(session), int(unmapped_hits), int(max_hits)))

    def obstacle_map_download(self, session: int) -> np.ndarray:
        px = np.empty((self.obstacle_size, self.obstacle_size), dtype=np.int8)
        self._ck(N.lib().cs_batch_obstacle_map_download(self._h, int(session), px.ctypes.data))
        return px

    def obstacle_checksums(self) -> np.ndarray:
        out = np.zeros(self.n, dtype=np.uint64)
        self._ck(N.lib().cs_batch_obstacle_checksums(self._h, out.ctypes.data_as(C.POINTER(C.c_uint64))))
        return out

    def obstacle_visits(self) -> np.ndarray:
        """Per session: ObstacleMap cells the rays touched since the last reset (measurement)."""
        out = np.zeros(self.n, dtype=np.int64)
        self._ck(N.lib().cs_batch_get_obstacle_visits(self._h, out.ctypes.data_as(C.POINTER(C.c_int64))))
        return out


def gather_peak(cells: int, per_thread: int = 256, repeats: int = 5, device: int = 0) -> float:
    """Measured random 2-byte gather rate (lookups/s) over a table of `cells` uint16."""
    v = C.c_double()
    N.check(N.lib().cs_gather_peak(device, int(cells), per_thread, repeats, C.byref(v)))
    return float(v.value)


def host_map_checksum(pixels, size: int) -> int:
    px = np.ascontiguousarray(pixels, dtype=np.uint16).reshape(-1)
    return int(N.lib().cs_host_map_checksum(px.ctypes.data, size))


def host_obstacle_checksum(pixels, size: int) -> int:
    """The hash of Batch.obstacle_checksums() for a host ObstacleMap (size * size sbyte, row-major)."""
    px = np.ascontiguousarray(pixels, dtype=np.int8).reshape(-1)
    if px.size != size * size:
        raise ValueError("expected %d pixels, got %d" % (size * size, px.size))
    return int(N.lib().cs_host_obstacle_checksum(px.ctypes.data, size))


def philox_offsets(seed: int, scan_index: int, n: int, sigma_xy: float, sigma_theta: float) -> np.ndarray:
    """Host twin of the on-device candidate generator (verification tables)."""
    out = np.zeros((n, 3), dtype=np.float32)
    if n:
        N.lib().cs_philox_offsets(seed, scan_index, n, sigma_xy, sigma_theta, _ptr(out))
    return out


# ------------------------------------------------------------------------------------------------
# reference-shaped classes
# ------------------------------------------------------------------------------------------------
class HoleMap:
    """CoreSLAM/HoleMap.cs:17-55.  Pixels is a *public field* in the reference and callers read it
    directly (Simulation/MainWindow.xaml.cs:227-229); here reading it pulls the device-resident map
    (after waiting for the pending integration)."""

    def __init__(self, proc: Processor, size_pixels: int, size_meters: float):
        self._proc = proc
        self.Size = size_pixels
        self.Scale = proc.scale

    @property
    def Pixels(self) -> np.ndarray:
        return self._proc.map_download()

    def GetPackedPixels(self) -> np.ndarray:
        return self._proc.map_packed()


class ObstacleMap:
    """CoreSLAM/ObstacleMap.cs:11-44.  Pixels is a public readonly sbyte[,] (first index Y); reading it pulls the
    device-resident map."""

    def __init__(self, proc: Processor, size_pixels: int, size_meters: float):
        self._proc = proc
        self.Size = size_pixels
        self.Scale = proc.obstacle_scale

    @property
    def Pixels(self) -> np.ndarray:
        return self._proc.obstacle_map_download()


class CoreSLAMProcessor:
    """Drop-in for CoreSLAM.CoreSLAMProcessor (CoreSLAM/CoreSLAMProcessor.cs): both halves of Update run on the
    device (HoleMap :496-534, ObstacleMap :540-593)."""

    def __init__(self, physicalMapSize: float, holeMapSize: int, obstacleMapSize: int, startPose, sigmaXY: float,
                 sigmaTheta: float, iterationsPerThread: int, numSearchThreads: int, *, device: int = 0,
                 seed: int = 0x5EED, max_points: int = 0, flags: int = 0):
        self.PhysicalMapSize = float(physicalMapSize)
        self.SigmaXY = float(sigmaXY)
        self.SigmaTheta = float(sigmaTheta)
        self.SearchIterationsPerThread = int(iterationsPerThread)
        self.NumSearchThreads = int(numSearchThreads)
        self._proc = Processor(physicalMapSize, holeMapSize, startPose, sigmaXY, sigmaTheta, iterationsPerThread,
                               numSearchThreads, device=device, seed=seed, max_points=max_points, flags=flags,
                               obstacle_map_size=obstacleMapSize)
        self.HoleMap = HoleMap(self._proc, holeMapSize, physicalMapSize)
        self.ObstacleMap = ObstacleMap(self._proc, obstacleMapSize, physicalMapSize) if obstacleMapSize > 0 else None
        self._quality, self._hole_width, self._psb = 50, 0.6, 5
        self._unmapped, self._max_hits = -5, 10
        self._pose = _f32(startPose)
        self.LastResult: Optional[SearchResult] = None

    # properties :40-106
    Pose = property(lambda s: s._pose.copy())
    Quality = property(lambda s: s._quality)
    HoleWidth = property(lambda s: s._hole_width)
    PositionSearchBeginning = property(lambda s: s._psb)
    UnmappedObstacleHits = property(lambda s: s._unmapped)
    MaxObstacleHits = property(lambda s: s._max_hits)

    @UnmappedObstacleHits.setter
    def UnmappedObstacleHits(self, v):
        """:98 — 'After changing this, Reset function has to be called!' """
        self._proc.set_unmapped_obstacle_hits(v)
        self._unmapped = int(v)

    @MaxObstacleHits.setter
    def MaxObstacleHits(self, v):
        self._proc.set_max_obstacle_hits(v)
        self._max_hits = int(v)

    @Quality.setter
    def Quality(self, v):
        self._proc.set_quality(v)
        self._quality = int(v)

    @HoleWidth.setter
    def HoleWidth(self, v):
        self._proc.set_hole_width(v)
        self._hole_width = float(v)

    @PositionSearchBeginning.setter
    def PositionSearchBeginning(self, v):
        self._proc.set_position_search_beginning(v)
        self._psb = int(v)

    def Reset(self):
        """:167-175"""
        self._proc.reset()
        self._pose = self._proc.get_pose()

    def Update(self, segments: List[ScanSegment], candidateOffsets=None):
        """:717-752.  candidateOffsets (T*I x 3) switches on verification mode for this scan."""
        if not segments:
            raise ValueError("Sequence contains no elements")  # segments.Last() on an empty list (:719)
        self.LastResult = self._proc.update_segments(segments, candidateOffsets)  # :719-752, cloud (:723) included
        self._pose = self.LastResult.pose

    def Relocalize(self, points, origin, step, count, window: int = 0, k: int = 1, want_distances=False):
        """No reference counterpart: where this scan cloud (ScanCloud.Points) lies on the current HoleMap, searched over
        a pose lattice (Processor.relocalize).  Changes nothing; adopt a hit with ResumeAt."""
        return self._proc.relocalize(points, origin, step, count, window, k, want_distances)

    def RelocalizeBounded(self, points, origin, step, count, window: int = 0, k: int = 1):
        """Relocalize's hits by branch and bound (Processor.relocalize_bounded), for fine lattices over a whole map.
        Returns (hits, stats).  Changes nothing; adopt a hit with ResumeAt."""
        return self._proc.relocalize_bounded(points, origin, step, count, window, k)

    def RelocalizeSequence(self, scans, odometry, origin, step, count, window: int = 0, k: int = 1, want_distances=False):
        """Relocalize with the last few scan clouds and the odometry poses they came with (Processor.relocalize_sequence),
        so that places that look alike to one scan are told apart.  A hit is the pose of the last scan: adopt it with
        ResumeAt(hit.pose, odometry[-1]).  Changes nothing."""
        return self._proc.relocalize_sequence(scans, odometry, origin, step, count, window, k, want_distances)

    def RelocalizeSequenceBounded(self, scans, odometry, origin, step, count, window: int = 0, k: int = 1):
        """RelocalizeSequence's hits by branch and bound (Processor.relocalize_sequence_bounded).  Returns (hits, stats)."""
        return self._proc.relocalize_sequence_bounded(scans, odometry, origin, step, count, window, k)

    def ResumeAt(self, pose, odometryPose):
        """Continue tracking from `pose` (e.g. a Relocalize hit): the next Update searches around
        pose + (odometry - odometryPose), as after PositionSearchBeginning scans."""
        self._proc.set_pose(pose, odometryPose, self._psb)
        self._pose = self._proc.get_pose()

    def Dispose(self):
        """:757-773"""
        self._proc.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.Dispose()
