"""Build + ctypes loading of the C-ABI library (include/coreslam_b200.h).

There is no Python/NumPy implementation of the hot path behind this: if the shared library cannot be
built or loaded, importing the compute entry points raises.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, "csrc")
BUILD_DIR = os.path.join(_HERE, "_build")
LIB_PATH = os.path.join(BUILD_DIR, "libcoreslam_b200.so")
HEADER = os.path.join(ROOT, "include", "coreslam_b200.h")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",                      # RyuJIT never contracts a*b+c; neither may we
    "-Xcompiler", "-fPIC,-ffp-contract=off",
    "-shared",
]


def _sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))] + [HEADER]


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(s) > t for s in _sources())


def build(force: bool = False, verbose: bool = False) -> str:
    """nvcc-compile the library in-tree for sm_100a (cross-compiles without a GPU).  CS_B200_LIB=<path> selects a library
    built elsewhere (A/B runs of kernel variants on the GPU box) instead."""
    override = os.environ.get("CS_B200_LIB")
    if override and not force:
        if not os.path.exists(override):
            raise RuntimeError("CS_B200_LIB=%s does not exist" % override)
        return override
    if not force and not _stale():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        if os.path.exists(LIB_PATH):
            return LIB_PATH  # prebuilt library shipped with the snapshot, no compiler on this box
        raise RuntimeError("nvcc not found and %s is missing" % LIB_PATH)
    os.makedirs(BUILD_DIR, exist_ok=True)
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH, os.path.join(CSRC, "cs_api.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


class Config(C.Structure):
    _fields_ = [
        ("physical_map_size", C.c_float),
        ("hole_map_size", C.c_int32),
        ("start_pose", C.c_float * 3),
        ("sigma_xy", C.c_float),
        ("sigma_theta", C.c_float),
        ("iterations_per_thread", C.c_int32),
        ("num_search_threads", C.c_int32),
        ("device", C.c_int32),
        ("max_points", C.c_int32),
        ("seed", C.c_uint64),
        ("stream", C.c_void_p),
        ("flags", C.c_uint32),
        ("obstacle_map_size", C.c_int32),
    ]


class Result(C.Structure):
    _fields_ = [
        ("pose", C.c_float * 3),
        ("distance", C.c_int32),
        ("index", C.c_int32),
        ("searched", C.c_int32),
        ("visits", C.c_int64),
    ]


class Timing(C.Structure):
    _fields_ = [
        ("search_ms", C.c_float),
        ("finalize_ms", C.c_float),
        ("integrate_ms", C.c_float),
        ("h2d_ms", C.c_float),
        ("total_device_ms", C.c_float),
        ("host_wait_ms", C.c_double),
        ("obstacle_ms", C.c_float),
        ("reserved", C.c_float),
    ]


class Lattice(C.Structure):
    _fields_ = [
        ("origin", C.c_float * 3),
        ("step", C.c_float * 3),
        ("count", C.c_int32 * 3),
    ]


class LatticeHit(C.Structure):
    _fields_ = [
        ("pose", C.c_float * 3),
        ("distance", C.c_int32),
        ("index", C.c_int32),
    ]


class RelocalizeStats(C.Structure):
    _fields_ = [
        ("poses", C.c_int64),
        ("evaluated", C.c_int64),
        ("bounded", C.c_int64),
        ("levels", C.c_int32),
        ("passes", C.c_int32),
        ("upper_bound", C.c_int32),
        ("reserved", C.c_int32),
    ]


LATTICE_MAX_POSES = 1 << 28
LATTICE_MAX_HITS = 64
LATTICE_MAX_POSES_BOUNDED = 2147483647
LATTICE_BOUNDED_MAX_NODES = 1 << 20
SEQUENCE_MAX_SCANS = 32

FLAG_ROW_MAJOR_MAP = 0x1
FLAG_TIMING = 0x2
FLAG_KEEP_DISTANCES = 0x4
FLAG_NO_HOST_SPIN = 0x8
FLAG_L2_PERSIST = 0x10
FLAG_DEBUG_RAYS = 0x20
FLAG_SEARCH_WARP = 0x40
FLAG_SEARCH_SLAB = 0x80
FLAG_DEBUG_BOUNDED_SPIN = 0x100  # device-side polls give up after 2 s (CS_TUNE_SPIN_MS) -> CS_ERR_CUDA instead of a hang
EXPORT_GRAY16, EXPORT_PACKED4, EXPORT_OBSTACLE_I8 = 0, 1, 2

STATUS_NAMES = {0: "CS_OK", 1: "CS_ERR_INVALID_ARGUMENT", 2: "CS_ERR_NO_DEVICE", 3: "CS_ERR_CUDA",
                4: "CS_ERR_OUT_OF_MEMORY", 5: "CS_ERR_CAPACITY", 6: "CS_ERR_STATE", 7: "CS_ERR_NCCL"}

_vp, _fp, _ip = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int32)

# name -> (restype, argtypes); also the export list checked by tests/test_abi.py
SIGNATURES = {
    "cs_abi_version": (C.c_int32, []),
    "cs_last_error": (C.c_char_p, [_vp]),
    "cs_device_count": (C.c_int32, []),
    "cs_create": (C.c_int, [C.POINTER(Config), C.POINTER(_vp)]),
    "cs_destroy": (C.c_int, [_vp]),
    "cs_reset": (C.c_int, [_vp]),
    "cs_set_quality": (C.c_int, [_vp, C.c_int32]),
    "cs_set_hole_width": (C.c_int, [_vp, C.c_float]),
    "cs_set_position_search_beginning": (C.c_int, [_vp, C.c_int32]),
    "cs_get_pose": (C.c_int, [_vp, _fp]),
    "cs_set_pose": (C.c_int, [_vp, _fp, _fp, C.c_int32]),
    "cs_get_map_info": (C.c_int, [_vp, _ip, _fp]),
    "cs_set_unmapped_obstacle_hits": (C.c_int, [_vp, C.c_int32]),
    "cs_set_max_obstacle_hits": (C.c_int, [_vp, C.c_int32]),
    "cs_get_obstacle_map_info": (C.c_int, [_vp, _ip, _fp]),
    "cs_obstacle_map_download": (C.c_int, [_vp, _vp]),
    "cs_obstacle_map_upload": (C.c_int, [_vp, _vp]),
    "cs_obstacle_map_fill": (C.c_int, [_vp, C.c_int32]),
    "cs_get_obstacle_visits": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
    "cs_search": (C.c_int, [_vp, _fp, C.c_int32, _fp, _fp, _fp, C.c_int32, C.c_uint32, C.POINTER(Result), _ip]),
    "cs_relocalize": (C.c_int, [_vp, _fp, C.c_int32, C.POINTER(Lattice), C.c_int32, C.c_int32, C.POINTER(LatticeHit), _ip,
                                _ip]),
    "cs_relocalize_bounded": (C.c_int, [_vp, _fp, C.c_int32, C.POINTER(Lattice), C.c_int32, C.c_int32, C.POINTER(LatticeHit),
                                        _ip, C.POINTER(RelocalizeStats)]),
    "cs_relocalize_sequence": (C.c_int, [_vp, _fp, _ip, _fp, C.c_int32, C.POINTER(Lattice), C.c_int32, C.c_int32,
                                         C.POINTER(LatticeHit), _ip, _ip]),
    "cs_relocalize_sequence_bounded": (C.c_int, [_vp, _fp, _ip, _fp, C.c_int32, C.POINTER(Lattice), C.c_int32, C.c_int32,
                                                 C.POINTER(LatticeHit), _ip, C.POINTER(RelocalizeStats)]),
    "cs_integrate": (C.c_int, [_vp, _fp, C.c_int32, _fp, _fp, C.POINTER(C.c_int64)]),
    "cs_update": (C.c_int, [_vp, _fp, C.c_int32, _fp, _fp, C.POINTER(Result)]),
    "cs_update_segments": (C.c_int, [_vp, _fp, _ip, _fp, C.c_int32, C.c_int32, _fp, C.POINTER(Result)]),
    "cs_segments_to_cloud": (C.c_int, [_vp, _fp, _ip, _fp, C.c_int32, C.c_int32, _fp, _fp]),
    "cs_group_export": (C.c_int, [_vp, C.c_void_p]),
    "cs_group_attach": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_void_p]),
    "cs_group_attach_local": (C.c_int, [_vp, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "cs_group_detach": (C.c_int, [_vp]),
    "cs_update_begin": (C.c_int, [_vp, _fp, C.c_int32, _fp, _fp, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "cs_update_finish": (C.c_int, [_vp, C.POINTER(Result)]),
    "cs_sync": (C.c_int, [_vp]),
    "cs_map_download": (C.c_int, [_vp, _vp]),
    "cs_map_upload": (C.c_int, [_vp, _vp]),
    "cs_map_fill": (C.c_int, [_vp, C.c_uint16]),
    "cs_map_packed": (C.c_int, [_vp, _vp]),
    "cs_map_export_begin": (C.c_int, [_vp, C.c_int32, _vp]),
    "cs_map_export_wait": (C.c_int, [_vp]),
    "cs_map_checksum": (C.c_int, [_vp, C.POINTER(C.c_uint64)]),
    "cs_host_map_checksum": (C.c_uint64, [_vp, C.c_int32]),
    "cs_set_flags": (C.c_int, [_vp, C.c_uint32]),
    "cs_get_timing": (C.c_int, [_vp, C.POINTER(Timing)]),
    "cs_get_distances": (C.c_int, [_vp, _ip, C.c_int32]),
    "cs_get_rays": (C.c_int, [_vp, _ip, C.c_int32]),
    "cs_get_visits": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
    "cs_get_ring_cycles": (C.c_int, [_vp, C.POINTER(C.c_int64), C.c_int32]),
    "cs_get_search_plan": (C.c_int, [_vp, C.c_int32, C.c_int32, _ip]),
    "cs_get_launch_count": (C.c_int, [_vp, C.POINTER(C.c_uint64)]),
    "cs_pinned_alloc": (C.c_int, [C.POINTER(_vp), C.c_uint64]),
    "cs_pinned_free": (C.c_int, [_vp]),
    "cs_scanlog_create": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_vp)]),
    "cs_scanlog_set": (C.c_int, [_vp, C.c_int32, _fp, C.c_int32, _fp, _fp]),
    "cs_scanlog_upload": (C.c_int, [_vp]),
    "cs_scanlog_destroy": (C.c_int, [_vp]),
    "cs_scanlog_save": (C.c_int, [_vp, C.c_char_p]),
    "cs_scanlog_load": (C.c_int, [C.c_int32, C.c_char_p, C.POINTER(_vp)]),
    "cs_scanlog_file_info": (C.c_int, [C.c_char_p, _ip, _ip, _ip]),
    "cs_scanlog_file_read": (C.c_int, [C.c_char_p, C.c_int32, _fp, _ip, _fp, _fp]),
    "cs_replay": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, C.POINTER(Result)]),
    "cs_batch_create": (C.c_int, [C.POINTER(Config), C.c_int32, C.POINTER(_vp)]),
    "cs_batch_destroy": (C.c_int, [_vp]),
    "cs_batch_last_error": (C.c_char_p, [_vp]),
    "cs_batch_size": (C.c_int32, [_vp]),
    "cs_batch_set_params": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_float]),
    "cs_batch_update": (C.c_int, [_vp, _fp, _ip, _fp, _fp, C.POINTER(Result)]),
    "cs_rings_hint": (C.c_int32, [C.c_int32, C.c_float, C.c_float, _fp, C.c_int32]),
    "cs_batch_submit": (C.c_int, [_vp, _fp, _ip, _fp, _fp]),
    "cs_batch_collect": (C.c_int, [_vp, C.POINTER(Result)]),
    "cs_batch_replay": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, C.POINTER(Result)]),
    "cs_batch_sync": (C.c_int, [_vp]),
    "cs_batch_get_poses": (C.c_int, [_vp, _fp]),
    "cs_batch_map_download": (C.c_int, [_vp, C.c_int32, _vp]),
    "cs_batch_map_checksums": (C.c_int, [_vp, C.POINTER(C.c_uint64)]),
    "cs_batch_get_launch_count": (C.c_int, [_vp, C.POINTER(C.c_uint64)]),
    "cs_batch_reset": (C.c_int, [_vp]),
    "cs_batch_set_obstacle_params": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int32]),
    "cs_batch_obstacle_map_download": (C.c_int, [_vp, C.c_int32, _vp]),
    "cs_batch_obstacle_checksums": (C.c_int, [_vp, C.POINTER(C.c_uint64)]),
    "cs_batch_get_obstacle_visits": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
    "cs_host_obstacle_checksum": (C.c_uint64, [_vp, C.c_int32]),
    "cs_philox_offsets": (None, [C.c_uint64, C.c_uint32, C.c_int32, C.c_float, C.c_float, _fp]),
    "cs_host_sincos": (None, [_fp, C.c_int32, _fp, _fp]),
    "cs_device_sincos": (C.c_int, [C.c_int32, _fp, C.c_int32, _fp, _fp]),
    "cs_host_normalize_angle": (C.c_float, [C.c_float]),
    "cs_gather_peak": (C.c_int, [C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_double)]),
}

_lib = None


def lib():
    """The loaded C-ABI library.  Raises if it is missing and cannot be built — no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    path = build()
    L = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    if L.cs_abi_version() != 1:
        raise RuntimeError("coreslam_b200 ABI mismatch")
    _lib = L
    return L


class CoreSlamError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__("%s: %s" % (STATUS_NAMES.get(status, status), message))
        self.status = status


def check(status: int, handle=None, batch=None):
    if status != 0:
        msg = lib().cs_batch_last_error(batch) if batch is not None else lib().cs_last_error(handle)
        raise CoreSlamError(status, msg.decode() if msg else "")
