"""Handle lifetimes: every create, successful or failed, and every destroy gives the device memory back.

A processor at the cfg2 shape (with an ObstacleMap and every lazily allocated buffer in use), a 256-session batch with
ObstacleMaps and a pipeline slot, and a batch create refused for its size after its HoleMaps and scratch are allocated
are cycled; the free device memory must come back to where it was.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import slam.net_b200 as sn
from slam.net_b200 import _native as N
from slam.net_b200 import synth

pytestmark = pytest.mark.gpu

CS_ERR_OUT_OF_MEMORY = 4
CYCLES = 10
# The GPU may be shared: far above what other work moves in a few seconds, far below one cycle's leak (the refused create
# alone allocates 8 GB of HoleMaps).
MARGIN = 1 << 30


def _processor_cycle(rp):
    p = sn.Processor(40.0, 2048, rp.odometry[0], 0.1, 0.17, 1024, 4, max_points=1024, obstacle_map_size=2048)
    p.update(rp.points[0], rp.odometry[0])
    p.map_packed()
    outs = {N.EXPORT_GRAY16: np.empty(2048 * 2048, np.uint16), N.EXPORT_PACKED4: np.empty(2048 * 2048 // 2, np.uint8),
            N.EXPORT_OBSTACLE_I8: np.empty(2048 * 2048, np.int8)}
    for fmt, out in outs.items():
        p.map_export_begin(fmt, out)
        p.map_export_wait()
    p.ring_cycles()
    p.close()


def _batch_cycle(rp):
    n = 256
    b = sn.Batch(n, 40.0, 1600, rp.odometry[0], 0.1, 0.17, 1000, 4, max_points=360, obstacle_map_size=400)
    b.submit([rp.points[0]] * n, np.tile(rp.odometry[0], (n, 1)))
    b.collect()
    b.close()


def _refused_batch_create():
    # 4096 sessions: 8 GB of 1024^2 HoleMaps, then 4096 ObstacleMaps of 16384^2 (1 TB) that cannot be allocated
    n = 4096
    cfgs = (N.Config * n)()
    for c in cfgs:
        c.physical_map_size, c.hole_map_size, c.obstacle_map_size = 40.0, 1024, 16384
        c.iterations_per_thread, c.num_search_threads, c.max_points = 4, 1, 360
    h = C.c_void_p()
    assert N.lib().cs_batch_create(cfgs, n, C.byref(h)) == CS_ERR_OUT_OF_MEMORY
    assert not h.value


def test_create_and_destroy_return_device_memory():
    rp = synth.make_replay(1, 1024, 40.0, seed=11)
    rp1 = synth.make_replay(1, 360, 40.0, seed=12)

    def cycle():
        _processor_cycle(rp)
        _batch_cycle(rp1)
        _refused_batch_create()

    cycle()  # first use: the context loads the kernels
    free_before, _ = torch.cuda.mem_get_info(0)
    for _ in range(CYCLES):
        cycle()
    free_after, _ = torch.cuda.mem_get_info(0)
    assert free_after >= free_before - MARGIN, (free_before, free_after)
