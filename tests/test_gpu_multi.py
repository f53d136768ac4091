"""Sharded paths on the GPU (SURVEY.md 8e): batches of independent sessions (cfg5) and the candidate split
with its 8-byte arg-min exchange (cfg4) — bit-exact against the CPU oracle / the single-handle path.

The candidate split is exercised on ONE device with two handles playing two ranks (same kernels, same
exchange code; the MIN runs through torch on the device keys), and, when the box has >= 2 GPUs, with two
real processes over NCCL.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import slam.net_b200 as sn
from slam.net_b200 import _native as N
from slam.net_b200 import parallel as par
from slam.net_b200 import synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_batch_update_matches_oracle_per_session():
    n_sess, n_scans, P, size, phys, iters, threads = 5, 12, 200, 256, 40.0, 48, 2
    rps = [synth.make_replay(n_scans, P, phys, seed=50 + j) for j in range(n_sess)]
    sxy = [0.05 + 0.02 * j for j in range(n_sess)]
    sth = [0.10 + 0.01 * j for j in range(n_sess)]
    b = sn.Batch(n_sess, phys, size, [rp.odometry[0] for rp in rps], sxy, sth, iters, threads, max_points=P)
    os_ = [orc.Processor(phys, size, rps[j].odometry[0], sxy[j], sth[j], iters, threads) for j in range(n_sess)]
    for j in range(n_sess):
        b.set_params(j, 40 + 30 * j, 0.4 + 0.3 * j)
        os_[j].quality = 40 + 30 * j
        os_[j].hole_width = 0.4 + 0.3 * j
    for k in range(n_scans):
        offs = np.stack([synth.candidate_offsets(70 + j, k, iters * threads, sxy[j], sth[j]) for j in range(n_sess)])
        res = b.update([rps[j].points[k] for j in range(n_sess)], np.stack([rps[j].odometry[k] for j in range(n_sess)]), offs)
        for j in range(n_sess):
            os_[j].update(rps[j].points[k], rps[j].odometry[k], offs[j])
            assert np.array_equal(res[j].pose, os_[j].pose), (k, j)
            assert res[j].searched == (k >= 5)
            if k >= 5:
                assert (res[j].distance, res[j].index) == (os_[j].last_distance, os_[j].last_index)
    assert np.array_equal(b.poses(), np.stack([o.pose for o in os_]))
    sums = b.map_checksums()
    for j in range(n_sess):
        assert int(sums[j]) == sn.host_map_checksum(np.array(os_[j].map.pixels), size)
    assert np.array_equal(b.map_download(3), np.array(os_[3].map.pixels))
    b.close()


def test_batch_replay_shared_log_philox_equals_single_handles():
    """Parameter sweep: every session replays the same log with its own seed / sigmas / HoleWidth (production
    mode, on-device Philox).  Must equal one cs_processor per session fed the same scans."""
    n_sess, n_scans, P, size, phys, iters, threads = 4, 14, 180, 200, 40.0, 32, 4
    rp = synth.make_replay(n_scans, P, phys, seed=9)
    seeds = [11, 22, 33, 44]
    sxy = [0.05, 0.1, 0.15, 0.2]
    sth = [0.05, 0.1, 0.17, 0.25]
    b = sn.Batch(n_sess, phys, size, rp.odometry[0], sxy, sth, iters, threads, max_points=P, seeds=seeds)
    log = sn.ScanLog(n_scans, P, n_offsets=0)
    for k in range(n_scans):
        log.set(k, rp.points[k], rp.odometry[k])
    log.upload()
    for j in range(n_sess):
        b.set_params(j, 50 + 10 * j, 0.6 + 0.2 * j)
    res = b.replay(log, 0, 6)
    res = b.replay(log, 6, n_scans - 6)
    for j in range(n_sess):
        p = sn.Processor(phys, size, rp.odometry[0], sxy[j], sth[j], iters, threads, max_points=P, seed=seeds[j])
        p.set_quality(50 + 10 * j)
        p.set_hole_width(0.6 + 0.2 * j)
        o = orc.Processor(phys, size, rp.odometry[0], sxy[j], sth[j], iters, threads)
        o.quality = 50 + 10 * j
        o.hole_width = 0.6 + 0.2 * j
        for k in range(n_scans):
            r = p.update(rp.points[k], rp.odometry[k], None)
            o.update(rp.points[k], rp.odometry[k], sn.philox_offsets(seeds[j], k, iters * threads, sxy[j], sth[j]))
        assert np.array_equal(r.pose, res[j].pose) and (r.distance, r.index) == (res[j].distance, res[j].index)
        assert np.array_equal(r.pose, o.pose)
        assert np.array_equal(b.map_download(j), p.map_download())
        assert np.array_equal(b.map_download(j), np.array(o.map.pixels))
        p.close()
    assert len(set(int(x) for x in b.map_checksums())) == n_sess  # the sweep really produced different maps
    log.close()
    b.close()


def test_batch_rejects_mismatched_configs():
    cfgs = (N.Config * 2)()
    for j, c in enumerate(cfgs):
        c.physical_map_size, c.hole_map_size = 10.0, 64 + 64 * j
        c.iterations_per_thread, c.num_search_threads = 4, 1
    h = N.C.c_void_p()
    assert N.lib().cs_batch_create(cfgs, 2, N.C.byref(h)) == 1  # CS_ERR_INVALID_ARGUMENT


@pytest.mark.parametrize("philox", [False, True])
def test_candidate_split_two_handles_one_device(philox):
    """Two 'ranks' on one GPU: each evaluates half of the flat candidate indices, the packed keys are
    min-reduced on the device, both finish with the pose and map of the unsplit reference run."""
    import torch
    n_scans, P, size, phys, iters, threads = 16, 300, 320, 40.0, 61, 4  # T*I + 1 = 245: odd split
    rp = synth.make_replay(n_scans, P, phys, seed=21)
    seed = 0xABCDEF
    ranks = [sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=P, seed=seed) for _ in range(2)]
    o = orc.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads)
    n_flat = iters * threads + 1
    for k in range(n_scans):
        off = (sn.philox_offsets(seed, k, iters * threads, 0.1, 0.17) if philox
               else synth.candidate_offsets(4, k, iters * threads, 0.1, 0.17))
        ptrs = []
        for g, p in enumerate(ranks):
            lo, cnt = par.candidate_slice(n_flat, 2, g)
            ptrs.append(p.update_begin(rp.points[k], rp.odometry[k], None if philox else off, lo, cnt))
        assert all(bool(x) == (k >= 5) for x in ptrs)
        if k >= 5:
            for p in ranks:
                p.sync()
            keys = [par.device_key_tensor(x, 0) for x in ptrs]
            m = torch.minimum(keys[0], keys[1])  # the 8-byte exchange, played by one device
            keys[0].copy_(m)
            keys[1].copy_(m)
            torch.cuda.synchronize()
        res = [p.update_finish() for p in ranks]
        o.update(rp.points[k], rp.odometry[k], off)
        for r in res:
            assert np.array_equal(r.pose, o.pose), k
            if k >= 5:
                assert (r.distance, r.index) == (o.last_distance, o.last_index)
    for p in ranks:
        assert np.array_equal(p.map_download(), np.array(o.map.pixels))
        p.close()


def test_split_phase_state_errors():
    p = sn.Processor(10.0, 64, (5, 5, 0), 0.1, 0.1, 8, 1, max_points=16)
    pts = np.array([[1.0, 0.0]], dtype=np.float32)
    with pytest.raises(sn.CoreSlamError):
        p.update_finish()                      # finish without begin
    with pytest.raises(sn.CoreSlamError):
        p.update_begin(pts, (5, 5, 0), None, 5, 100)   # slice outside [0, T*I+1)
    p.update_begin(pts, (5, 5, 0), None, 0, 9)
    with pytest.raises(sn.CoreSlamError):
        p.update(pts, (5, 5, 0), None)         # a split update is in flight
    p.update_finish()
    p.update(pts, (5, 5, 0), None)
    p.close()


def test_candidate_split_two_processes_nccl():
    """Real thing: 2 ranks, 2 GPUs, NCCL MIN all-reduce of the in-session key."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29517", os.path.join(ROOT, "tests", "mp_split_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "SPLIT_OK" in out.stdout


def test_batch_submit_collect_pipeline_equals_blocking_updates():
    """cs_batch_submit / cs_batch_collect (two steps in flight, host staging overlapped with the previous step) must give the
    records and maps of the blocking cs_batch_update, and refuse a third step in flight / a collect with nothing submitted."""
    n_sess, n_scans, P, size, phys, iters, threads = 4, 14, 300, 256, 40.0, 120, 2
    rps = [synth.make_replay(n_scans, P, phys, seed=250 + j) for j in range(n_sess)]
    sxy, sth = [0.05, 0.07, 0.09, 0.11], [0.10, 0.11, 0.12, 0.13]
    mk = lambda: sn.Batch(n_sess, phys, size, [rp.odometry[0] for rp in rps], sxy, sth, iters, threads, max_points=P, seeds=[9, 8, 7, 6])
    a, b = mk(), mk()
    args = []
    for k in range(n_scans):
        offs = None if k % 3 == 2 else np.stack([synth.candidate_offsets(270 + j, k, iters * threads, sxy[j], sth[j]) for j in range(n_sess)])
        pts = [rps[j].points[k][: P - 11 * j] for j in range(n_sess)]
        args.append((pts, np.stack([rps[j].odometry[k] for j in range(n_sess)]), offs))
    want = [a.update(*x) for x in args]
    with pytest.raises(Exception):
        b.collect()
    got = []
    b.submit(*args[0])
    for k in range(1, n_scans):
        b.submit(*args[k])
        if k == 1:
            with pytest.raises(Exception):
                b.submit(*args[k])  # a third step in flight is refused and changes nothing
        got.append(b.collect())
    got.append(b.collect())
    for k in range(n_scans):
        for j in range(n_sess):
            assert np.array_equal(got[k][j].pose, want[k][j].pose), (k, j)
            assert (got[k][j].distance, got[k][j].index) == (want[k][j].distance, want[k][j].index), (k, j)
    assert np.array_equal(a.map_checksums(), b.map_checksums())
    assert np.array_equal(a.poses(), b.poses())
    a.close()
    b.close()


def test_batch_odd_max_points_stride_is_the_callers():
    """ADVICE r1 (high): the stride of the caller's points array is cfg.max_points as passed — also when it is odd (a 361-ray
    lidar); only the internal staging stride is rounded up.  Every session j >= 1 must read its own points."""
    n_sess, n_scans, P, size, phys, iters, threads = 4, 9, 181, 256, 40.0, 40, 2
    rps = [synth.make_replay(n_scans, P, phys, seed=350 + j) for j in range(n_sess)]
    sxy, sth = [0.05, 0.07, 0.09, 0.11], [0.10, 0.11, 0.12, 0.13]
    b = sn.Batch(n_sess, phys, size, [rp.odometry[0] for rp in rps], sxy, sth, iters, threads, max_points=P)
    assert b.max_points == P and P % 2 == 1
    os_ = [orc.Processor(phys, size, rps[j].odometry[0], sxy[j], sth[j], iters, threads) for j in range(n_sess)]
    for k in range(n_scans):
        offs = np.stack([synth.candidate_offsets(370 + j, k, iters * threads, sxy[j], sth[j]) for j in range(n_sess)])
        assert all(rps[j].points[k].shape[0] == P for j in range(n_sess))  # full rows: a shifted stride would read a neighbour's points
        res = b.update([rps[j].points[k] for j in range(n_sess)], np.stack([rps[j].odometry[k] for j in range(n_sess)]), offs)
        for j in range(n_sess):
            os_[j].update(rps[j].points[k], rps[j].odometry[k], offs[j])
            assert np.array_equal(res[j].pose, os_[j].pose), (k, j)
    sums = b.map_checksums()
    for j in range(n_sess):
        assert int(sums[j]) == sn.host_map_checksum(np.array(os_[j].map.pixels), size), j
    b.close()


def test_batch_nan_point_in_one_session_does_not_truncate_the_others():
    """ADVICE r1 (medium): the rings a batch is launched with are the maximum over its sessions; a NaN point in one session
    (which the reference handles through cvttss2si) must neither hide an earlier, longer scan nor be forgotten itself."""
    n_sess, n_scans, P, size, phys, iters, threads = 3, 8, 120, 512, 40.0, 24, 1
    rp = synth.make_replay(n_scans, P, phys, seed=390)
    sxy, sth = [0.05] * n_sess, [0.1] * n_sess
    b = sn.Batch(n_sess, phys, size, rp.odometry[0], sxy, sth, iters, threads, max_points=P)
    os_ = [orc.Processor(phys, size, rp.odometry[0], sxy[j], sth[j], iters, threads) for j in range(n_sess)]
    for k in range(n_scans):
        long_pts = rp.points[k].copy()                    # session 0: the full-range scan
        nan_pts = (rp.points[k] * 0.3).astype(np.float32)  # session 1: short rays and one NaN point
        nan_pts[3, 0] = np.nan
        short_pts = (rp.points[k] * 0.1).astype(np.float32)  # session 2: very short rays (the last r the reduction sees)
        pts = [long_pts, nan_pts, short_pts]
        offs = np.stack([synth.candidate_offsets(395 + j, k, iters * threads, sxy[j], sth[j]) for j in range(n_sess)])
        res = b.update(pts, np.tile(rp.odometry[k], (n_sess, 1)), offs)
        for j in range(n_sess):
            os_[j].update(pts[j], rp.odometry[k], offs[j])
            assert np.array_equal(res[j].pose, os_[j].pose), (k, j)
    for j in range(n_sess):
        assert np.array_equal(b.map_download(j), np.array(os_[j].map.pixels)), j
    b.close()


@pytest.mark.parametrize("philox", [False, True])
def test_group_exchange_inside_the_search_kernel_two_handles_one_device(philox):
    """cs_group_attach_local: two handles on one GPU play two ranks; each evaluates its half of the candidates and the 8-byte
    arg-min is exchanged INSIDE the search kernels (peer-mapped tables, no host step between search and integration).  Both
    must end every scan on the unsplit oracle's pose, winner and map.  The two ranks' kernels wait for each other on the
    device, so the two Updates are issued from two host threads."""
    import threading
    n_scans, P, size, phys, iters, threads = 16, 300, 320, 40.0, 305, 4  # T*I + 1 = 1221: odd split, slab search
    rp = synth.make_replay(n_scans, P, phys, seed=23)
    seed = 0xBEEF
    ranks = [sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=P, seed=seed) for _ in range(2)]
    for g, p in enumerate(ranks):
        p.group_attach_local(g, 2, ranks)
    o = orc.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads)
    for k in range(n_scans):
        off = (sn.philox_offsets(seed, k, iters * threads, 0.1, 0.17) if philox
               else synth.candidate_offsets(6, k, iters * threads, 0.1, 0.17))
        res = [None, None]

        def run(g):
            res[g] = ranks[g].update(rp.points[k], rp.odometry[k], None if philox else off)

        ts = [threading.Thread(target=run, args=(g,)) for g in range(2)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        o.update(rp.points[k], rp.odometry[k], off)
        for r in res:
            assert np.array_equal(r.pose, o.pose), k
            if k >= 5:
                assert (r.distance, r.index) == (o.last_distance, o.last_index), k
    for p in ranks:
        assert np.array_equal(p.map_download(), np.array(o.map.pixels))
    ranks[0].group_detach()          # a detached handle searches every candidate again
    ranks[1].group_detach()
    off = synth.candidate_offsets(6, 99, iters * threads, 0.1, 0.17)
    r0 = ranks[0].update(rp.points[0], rp.odometry[-1], off)
    o.update(rp.points[0], rp.odometry[-1], off)
    assert np.array_equal(r0.pose, o.pose) and (r0.distance, r0.index) == (o.last_distance, o.last_index)
    for p in ranks:
        p.close()


def test_group_exchange_times_out_instead_of_hanging():
    """A rank whose partner never shows up must fail the call with CS_ERR_NCCL after the device-side timeout (2 s), not hang."""
    P, size, phys = 100, 128, 20.0
    rp = synth.make_replay(7, P, phys, seed=5)
    ranks = [sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, 64, 1, max_points=P) for _ in range(2)]
    for g, p in enumerate(ranks):
        p.group_attach_local(g, 2, ranks)
    for k in range(5):  # map-only scans: no search, no exchange
        ranks[0].update(rp.points[k], rp.odometry[k], None)
    with pytest.raises(sn.CoreSlamError) as e:
        ranks[0].update(rp.points[5], rp.odometry[5], None)  # rank 1 never calls
    assert "CS_ERR_NCCL" in str(e.value)
    for p in ranks:
        p.close()


def test_group_two_processes_peer_memory():
    """Real thing: 2 ranks, 2 GPUs, tables mapped with CUDA IPC, exchange over NVLink inside the search kernels."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29519", os.path.join(ROOT, "tests", "mp_split_worker.py"), "group"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "SPLIT_OK" in out.stdout


_BOUNDED_SPIN_CHILD = r"""
import sys
import numpy as np
sys.path.insert(0, %(root)r)
import slam.net_b200 as sn
from slam.net_b200 import _native as N, synth
P, size, phys = 200, 256, 20.0
rp = synth.make_replay(4, P, phys, seed=5)
p = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, 64, 1, max_points=P, flags=N.FLAG_DEBUG_BOUNDED_SPIN)
try:
    for k in range(4):
        p.update(rp.points[k], rp.odometry[k], None)
    p.sync()
    p.map_download()
    print("NO_ERROR")
except sn.CoreSlamError as e:
    print("ERROR:", e)
"""


def test_bounded_spin_turns_a_stuck_poll_into_an_error():
    """CS_FLAG_DEBUG_BOUNDED_SPIN: with the fault knob the draw kernel waits for a pose tag nobody publishes; its polls must
    give up (50 ms here), the grid must drain, and a later call on the handle must fail with CS_ERR_CUDA naming the poll —
    not hang.  Child process: the library reads its knobs once."""
    env = dict(os.environ, CS_TUNE_FAULT="1", CS_TUNE_SPIN_MS="50")
    out = subprocess.run([sys.executable, "-c", _BOUNDED_SPIN_CHILD % {"root": ROOT}], capture_output=True, text=True, timeout=300,
                         cwd=ROOT, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "ERROR:" in out.stdout and "CS_ERR_CUDA" in out.stdout and "bounded polls" in out.stdout, out.stdout


def test_bounded_spin_flag_changes_no_result():
    """The same replay with and without CS_FLAG_DEBUG_BOUNDED_SPIN: identical poses, distances and maps."""
    from slam.net_b200 import _native as N
    n_scans, P, size, phys, iters, threads = 12, 700, 512, 40.0, 256, 4
    rp = synth.make_replay(n_scans, P, phys, seed=31)
    a = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=P, seed=4)
    b = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=P, seed=4, flags=N.FLAG_DEBUG_BOUNDED_SPIN)
    for k in range(n_scans):
        ra = a.update(rp.points[k], rp.odometry[k], None)
        rb = b.update(rp.points[k], rp.odometry[k], None)
        assert np.array_equal(ra.pose, rb.pose) and (ra.distance, ra.index) == (rb.distance, rb.index)
    assert np.array_equal(a.map_download(), b.map_download())
    a.close()
    b.close()
