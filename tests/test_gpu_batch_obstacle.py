"""Session batches with an ObstacleMap per session (cs_batch_* with obstacle_map_size > 0): every batched Update is the
whole CoreSLAMProcessor.Update (:717-752), UpdateObstacleMap (:751) included, and cs_batch_reset is Reset (:167-175) of
every session.  Checked bit for bit against the CPU oracle and against one cs_processor per session.  The GPU tests are
marked gpu; the host checksum test runs anywhere."""
import ctypes as C

import numpy as np
import pytest

import slam.net_b200 as sn
from slam.net_b200 import _native as N
from slam.net_b200 import synth
from oracle import oracle as orc

gpu = pytest.mark.gpu
CS_ERR_INVALID_ARGUMENT, CS_ERR_STATE = 1, 6


def _oracle(phys, size, start, sxy, sth, iters, threads, obst, quality=50, hole_width=0.6, unmapped=-5, max_hits=10):
    o = orc.Processor(phys, size, start, sxy, sth, iters, threads, obstacle_map_size=obst)
    o.quality, o.hole_width = quality, np.float32(hole_width)
    o.unmapped_obstacle_hits, o.max_obstacle_hits = unmapped, max_hits
    o.reset()  # UnmappedObstacleHits takes effect here (:96-98, :170)
    return o


def _status(fn, *args):
    with pytest.raises(sn.CoreSlamError) as e:
        fn(*args)
    return e.value.status


def _obstacle_cell(pose_x, obst, phys):
    """ObstacleMap column of the robot (CoreSLAMProcessor.cs:545, :553: Convert.ToInt32 rounds half to even)."""
    return int(np.rint(np.float32(np.float32(pose_x) * np.float32(obst / np.float32(phys))) + np.float32(0.5)))


# -- 1 -----------------------------------------------------------------------------------------------------------------
@gpu
def test_batch_update_per_session_obstacle_maps_match_the_oracle():
    """Verification mode, cs_batch_update: five sessions with their own drives, Quality, HoleWidth, MaxObstacleHits and
    UnmappedObstacleHits.  Session 4 drives off its ObstacleMap (but stays on its HoleMap) from scan 6 on: its ObstacleMap
    must stay as it was (:557-560) while the other sessions' maps keep changing."""
    n_sess, n_scans, P, size, obst, phys, iters, threads = 5, 12, 200, 256, 64, 40.0, 48, 2
    rps = [synth.make_replay(n_scans, P, phys, seed=150 + j) for j in range(n_sess)]
    odo = [rp.odometry.copy() for rp in rps]
    # session 4: from scan 6 on, odometry moved into the band x in [39.375, 40) m: on the 256-px HoleMap, off the 64-px ObstacleMap
    odo[4][6:, 0] += np.float32(39.69 - float(odo[4][6:, 0].mean()))
    sxy = [0.05, 0.07, 0.09, 0.11, 0.02]
    sth = [0.10, 0.11, 0.12, 0.13, 0.03]
    quality = [40, 70, 100, 130, 50]
    hole_width = [0.4, 0.7, 1.0, 0.5, 0.6]
    max_hits = [1, 3, 10, 127, 10]
    unmapped = [-5, -1, 0, 7, -128]
    b = sn.Batch(n_sess, phys, size, [o[0] for o in odo], sxy, sth, iters, threads, max_points=P, obstacle_map_size=obst)
    os_ = []
    for j in range(n_sess):
        b.set_params(j, quality[j], hole_width[j])
        b.set_obstacle_params(j, unmapped[j], max_hits[j])
        os_.append(_oracle(phys, size, odo[j][0], sxy[j], sth[j], iters, threads, obst, quality[j], hole_width[j], unmapped[j],
                           max_hits[j]))
    assert (b.obstacle_map_download(1) == -5).all()  # UnmappedObstacleHits waits for the reset
    b.reset()
    for j in range(n_sess):
        assert (b.obstacle_map_download(j) == unmapped[j]).all(), j
    visits = np.zeros(n_sess, dtype=np.int64)
    snap = None
    for k in range(n_scans):
        offs = np.stack([synth.candidate_offsets(170 + j, k, iters * threads, sxy[j], sth[j]) for j in range(n_sess)])
        res = b.update([rps[j].points[k] for j in range(n_sess)], np.stack([odo[j][k] for j in range(n_sess)]), offs)
        for j in range(n_sess):
            os_[j].update(rps[j].points[k], odo[j][k], offs[j])
            visits[j] += os_[j].obstacle_visits
            assert np.array_equal(res[j].pose, os_[j].pose), (k, j)
            assert res[j].searched == (k >= 5), (k, j)
            if k >= 5:
                assert (res[j].distance, res[j].index) == (os_[j].last_distance, os_[j].last_index), (k, j)
        if k == 5:
            snap = [b.obstacle_map_download(j) for j in range(n_sess)]
        if k >= 6:  # the test's premise: session 4 is off its ObstacleMap and on its HoleMap
            assert _obstacle_cell(os_[4].pose[0], obst, phys) >= obst and os_[4].pose[0] < phys, k
    assert np.array_equal(b.poses(), np.stack([o.pose for o in os_]))
    sums = b.map_checksums()
    for j in range(n_sess):
        assert int(sums[j]) == sn.host_map_checksum(np.array(os_[j].map.pixels), size), j
        got = b.obstacle_map_download(j)
        assert np.array_equal(got, os_[j].obstacle_map.pixels), (j, int((got != os_[j].obstacle_map.pixels).sum()))
    assert np.array_equal(b.obstacle_visits(), visits)
    assert np.array_equal(b.obstacle_map_download(4), snap[4])  # off its map: untouched by scans 6..11
    for j in range(4):
        assert not np.array_equal(b.obstacle_map_download(j), snap[j]), j
    assert (b.obstacle_map_download(3) > 10).any()  # MaxObstacleHits = 127 lets hits count past the default 10
    assert b.obstacle_map_download(0).max() <= 1
    b.close()


# -- 2 -----------------------------------------------------------------------------------------------------------------
@gpu
def test_batch_replay_shared_log_equals_processors_and_oracle():
    """Production mode, cs_batch_replay of one shared log with per-session seeds, sigmas and obstacle parameters: the same
    pose and both maps as one cs_processor per session fed the same scans, and as the oracle."""
    n_sess, n_scans, P, size, obst, phys, iters, threads = 4, 14, 180, 200, 128, 40.0, 32, 4
    rp = synth.make_replay(n_scans, P, phys, seed=19)
    seeds = [101, 202, 303, 404]
    sxy = [0.05, 0.1, 0.15, 0.2]
    sth = [0.05, 0.1, 0.17, 0.25]
    max_hits = [2, 10, 5, 127]
    unmapped = [-5, -3, 0, -20]
    b = sn.Batch(n_sess, phys, size, rp.odometry[0], sxy, sth, iters, threads, max_points=P, seeds=seeds, obstacle_map_size=obst)
    for j in range(n_sess):
        b.set_obstacle_params(j, unmapped[j], max_hits[j])
    b.reset()
    log = sn.ScanLog(n_scans, P, n_offsets=0)
    for k in range(n_scans):
        log.set(k, rp.points[k], rp.odometry[k])
    log.upload()
    b.replay(log, 0, 6, want_results=False)
    res = b.replay(log, 6, n_scans - 6)
    sums = b.obstacle_checksums()
    for j in range(n_sess):
        p = sn.Processor(phys, size, rp.odometry[0], sxy[j], sth[j], iters, threads, max_points=P, seed=seeds[j], obstacle_map_size=obst)
        p.set_unmapped_obstacle_hits(unmapped[j])
        p.set_max_obstacle_hits(max_hits[j])
        p.reset()
        o = _oracle(phys, size, rp.odometry[0], sxy[j], sth[j], iters, threads, obst, unmapped=unmapped[j], max_hits=max_hits[j])
        for k in range(n_scans):
            r = p.update(rp.points[k], rp.odometry[k], None)
            o.update(rp.points[k], rp.odometry[k], sn.philox_offsets(seeds[j], k, iters * threads, sxy[j], sth[j]))
        assert np.array_equal(r.pose, res[j].pose) and (r.distance, r.index) == (res[j].distance, res[j].index), j
        assert np.array_equal(r.pose, o.pose), j
        assert np.array_equal(b.map_download(j), p.map_download()), j
        assert np.array_equal(b.map_download(j), np.array(o.map.pixels)), j
        got = b.obstacle_map_download(j)
        assert np.array_equal(got, p.obstacle_map_download()), j
        assert np.array_equal(got, o.obstacle_map.pixels), j
        assert int(sums[j]) == sn.host_obstacle_checksum(o.obstacle_map.pixels, obst), j
        assert b.obstacle_visits()[j] == p.obstacle_visits(), j
        p.close()
    assert len(set(int(x) for x in sums)) > 1
    log.close()
    b.close()


# -- 3 -----------------------------------------------------------------------------------------------------------------
@gpu
def test_batch_submit_collect_with_obstacle_maps_equals_blocking_updates():
    n_sess, n_scans, P, size, obst, phys, iters, threads = 4, 12, 300, 256, 100, 40.0, 120, 2
    rps = [synth.make_replay(n_scans, P, phys, seed=350 + j) for j in range(n_sess)]
    sxy, sth = [0.05, 0.07, 0.09, 0.11], [0.10, 0.11, 0.12, 0.13]

    def mk():
        b = sn.Batch(n_sess, phys, size, [rp.odometry[0] for rp in rps], sxy, sth, iters, threads, max_points=P, seeds=[9, 8, 7, 6],
                     obstacle_map_size=obst)
        for j in range(n_sess):
            b.set_obstacle_params(j, -5, [3, 10, 1, 50][j])
        return b

    a, b = mk(), mk()
    args = []
    for k in range(n_scans):
        offs = None if k % 3 == 2 else np.stack([synth.candidate_offsets(370 + j, k, iters * threads, sxy[j], sth[j]) for j in range(n_sess)])
        pts = [rps[j].points[k][: P - 13 * j] for j in range(n_sess)]
        args.append((pts, np.stack([rps[j].odometry[k] for j in range(n_sess)]), offs))
    want = [a.update(*x) for x in args]
    got = []
    b.submit(*args[0])
    for k in range(1, n_scans):
        b.submit(*args[k])
        got.append(b.collect())
    got.append(b.collect())
    for k in range(n_scans):
        for j in range(n_sess):
            assert np.array_equal(got[k][j].pose, want[k][j].pose), (k, j)
    assert np.array_equal(a.poses(), b.poses())
    assert np.array_equal(a.map_checksums(), b.map_checksums())
    assert np.array_equal(a.obstacle_checksums(), b.obstacle_checksums())
    assert np.array_equal(a.obstacle_visits(), b.obstacle_visits())
    for j in range(n_sess):
        assert np.array_equal(a.obstacle_map_download(j), b.obstacle_map_download(j)), j
    a.close()
    b.close()


# -- 4 -----------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("obst", [0, 96])
def test_batch_reset(obst):
    """UnmappedObstacleHits waits for reset(); reset() refills both maps of every session, puts the poses back to the start
    poses and restarts the scan count and the Philox stream, so a replay after it equals one of a fresh batch.  A batch
    without ObstacleMaps resets its HoleMaps and poses."""
    n_sess, n_scans, P, size, phys, iters, threads = 3, 10, 200, 192, 40.0, 40, 2
    rp = synth.make_replay(n_scans, P, phys, seed=23)
    starts = np.stack([rp.odometry[0] + np.float32([0.1 * j, -0.05 * j, 0.01 * j]) for j in range(n_sess)]).astype(np.float32)
    unmapped = [-9, 0, 4]
    log = sn.ScanLog(n_scans, P, n_offsets=0)
    for k in range(n_scans):
        log.set(k, rp.points[k], rp.odometry[k])
    log.upload()

    def mk():
        b = sn.Batch(n_sess, phys, size, starts, 0.08, 0.12, iters, threads, max_points=P, seeds=[5, 6, 7], obstacle_map_size=obst)
        for j in range(n_sess):
            b.set_params(j, 60 + 20 * j, 0.5 + 0.1 * j)
            if obst:
                b.set_obstacle_params(j, unmapped[j], 4 + j)
        return b

    b = mk()
    b.replay(log, 0, n_scans, want_results=False)
    first_poses, first_sums = b.poses(), b.map_checksums()
    if obst:
        before = [b.obstacle_map_download(j) for j in range(n_sess)]
        assert all((m != -5).any() for m in before)
        b.set_obstacle_params(-1, 11, 6)  # stored; the maps do not change until reset()
        for j in range(n_sess):
            assert np.array_equal(b.obstacle_map_download(j), before[j]), j
        for j in range(n_sess):
            b.set_obstacle_params(j, unmapped[j], 4 + j)
    b.reset()
    assert np.array_equal(b.poses(), starts)
    for j in range(n_sess):
        assert (b.map_download(j) == 32750).all(), j
        if obst:
            assert (b.obstacle_map_download(j) == unmapped[j]).all(), j
    if obst:
        assert (b.obstacle_visits() == 0).all()
    # the same replay again: the same poses and maps as the first time and as a fresh batch
    res = b.replay(log, 0, n_scans)
    fresh = mk()
    if obst:
        fresh.reset()  # (applies the UnmappedObstacleHits set after creation)
    res_f = fresh.replay(log, 0, n_scans)
    for j in range(n_sess):
        assert np.array_equal(res[j].pose, res_f[j].pose) and (res[j].distance, res[j].index) == (res_f[j].distance, res_f[j].index), j
    assert np.array_equal(b.poses(), fresh.poses()) and np.array_equal(b.poses(), first_poses)
    assert np.array_equal(b.map_checksums(), fresh.map_checksums()) and np.array_equal(b.map_checksums(), first_sums)
    if obst:
        assert np.array_equal(b.obstacle_checksums(), fresh.obstacle_checksums())
        assert np.array_equal(b.obstacle_visits(), fresh.obstacle_visits())
    # a reset while a submitted step waits for its collect is refused and changes nothing
    pts = [rp.points[0]] * n_sess
    odo = np.stack([rp.odometry[0]] * n_sess)
    b.submit(pts, odo)
    assert _status(b.reset) == CS_ERR_STATE
    b.collect()
    b.reset()
    assert np.array_equal(b.poses(), starts)
    log.close()
    b.close()
    fresh.close()


# -- 5 -----------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n_sess", [2, 64])
def test_batch_obstacle_launch_shape(n_sess):
    """One launch of each ObstacleMap kernel per step for all sessions (never a launch per session), and one checksum launch."""
    n_scans, P, size, obst, phys, iters, threads = 8, 160, 128, 64, 40.0, 20, 2
    rp = synth.make_replay(n_scans, P, phys, seed=31)
    plain = sn.Batch(n_sess, phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=P)
    withm = sn.Batch(n_sess, phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=P, obstacle_map_size=obst)
    for k in range(n_scans):
        pts = [rp.points[k]] * n_sess
        odo = np.stack([rp.odometry[k]] * n_sess)
        d = []
        for b in (plain, withm):
            c0 = b.launch_count()
            b.update(pts, odo, want_results=False)
            d.append(b.launch_count() - c0)
        assert d[1] == d[0] + 2, (k, d)
    c0 = withm.launch_count()
    withm.obstacle_checksums()
    assert withm.launch_count() - c0 == 1
    plain.close()
    withm.close()


# -- 6 -----------------------------------------------------------------------------------------------------------------
@gpu
def test_batch_obstacle_errors():
    cfgs = (N.Config * 2)()
    for c in cfgs:
        c.physical_map_size, c.hole_map_size = 10.0, 64
        c.iterations_per_thread, c.num_search_threads = 4, 1
    cfgs[0].obstacle_map_size, cfgs[1].obstacle_map_size = 32, 16
    h = C.c_void_p()
    assert N.lib().cs_batch_create(cfgs, 2, C.byref(h)) == CS_ERR_INVALID_ARGUMENT
    assert b"obstacle_map_size" in N.lib().cs_batch_last_error(None)
    for bad in (-1, 16385):
        cfgs[0].obstacle_map_size = cfgs[1].obstacle_map_size = bad
        assert N.lib().cs_batch_create(cfgs, 2, C.byref(h)) == CS_ERR_INVALID_ARGUMENT

    plain = sn.Batch(2, 10.0, 64, (5, 5, 0), 0.1, 0.1, 4, 1, max_points=16)
    assert _status(plain.set_obstacle_params, 0, -5, 10) == CS_ERR_STATE
    assert _status(plain.obstacle_checksums) == CS_ERR_STATE
    assert _status(plain.obstacle_visits) == CS_ERR_STATE
    assert _status(plain.obstacle_map_download, 0) == CS_ERR_STATE
    plain.close()

    b = sn.Batch(2, 10.0, 64, (5, 5, 0), 0.1, 0.1, 4, 1, max_points=16, obstacle_map_size=16)
    assert _status(b.set_obstacle_params, 2, -5, 10) == CS_ERR_INVALID_ARGUMENT
    for u, m in ((128, 10), (-129, 10), (-5, 128), (-5, -129)):
        assert _status(b.set_obstacle_params, 0, u, m) == CS_ERR_INVALID_ARGUMENT, (u, m)
    assert _status(b.obstacle_map_download, 2) == CS_ERR_INVALID_ARGUMENT
    assert _status(b.obstacle_map_download, -1) == CS_ERR_INVALID_ARGUMENT
    b.set_obstacle_params(-1, -128, 127)  # the sbyte limits themselves are accepted
    b.reset()
    assert (b.obstacle_map_download(1) == -128).all()
    b.close()


# -- 7 -----------------------------------------------------------------------------------------------------------------
@gpu
def test_cfg5_256_sessions_with_obstacle_maps_sampled_against_the_oracle():
    """The cfg5 geometry of tests/test_gpu_full_size.py (256 sessions, 360 points, 1000 candidates, 1600 x 1600 HoleMap,
    production mode) with a 400 x 400 ObstacleMap per session and a grid over MaxObstacleHits: 8 sampled sessions equal the
    oracle in pose, HoleMap checksum and ObstacleMap checksum."""
    n_sess, P, size, obst, phys, iters, threads, n_scans = 256, 360, 1600, 400, 40.0, 1000, 1, 9
    n_cand = iters * threads
    rp = synth.make_replay(n_scans, P, phys, seed=77)

    def params(s):
        return (np.float32(0.05 + 0.025 * (s % 5)), np.float32(0.0873 + 0.0436 * ((s // 5) % 4)), 30 + 20 * ((s // 20) % 6),
                np.float32(0.4 + 0.2 * ((s // 120) % 4)), 9000 + s, [1, 2, 5, 10, 40, 127][s % 6])

    prm = [params(s) for s in range(n_sess)]
    b = sn.Batch(n_sess, phys, size, rp.odometry[0], [q[0] for q in prm], [q[1] for q in prm], iters, threads, max_points=P,
                 seeds=[q[4] for q in prm], obstacle_map_size=obst)
    for j, q in enumerate(prm):
        b.set_params(j, q[2], float(q[3]))
        b.set_obstacle_params(j, -5, q[5])
    log = sn.ScanLog(n_scans, P, n_offsets=0)
    for k in range(n_scans):
        log.set(k, rp.points[k], rp.odometry[k])
    log.upload()
    b.replay(log, 0, n_scans, want_results=False)
    poses, sums, osums = b.poses(), b.map_checksums(), b.obstacle_checksums()
    for s in (0, 37, 64, 101, 128, 199, 230, 255):
        sxy, sth, q, hw, seed, mh = prm[s]
        o = _oracle(phys, size, rp.odometry[0], sxy, sth, iters, threads, obst, q, hw, max_hits=mh)
        for k in range(n_scans):
            o.update(rp.points[k], rp.odometry[k], sn.philox_offsets(seed, k, n_cand, sxy, sth) if k >= 5 else None)
        assert np.array_equal(poses[s], o.pose), s
        assert int(sums[s]) == sn.host_map_checksum(np.array(o.map.pixels), size), s
        assert int(osums[s]) == sn.host_obstacle_checksum(o.obstacle_map.pixels, obst), s
    assert len(set(int(x) for x in osums)) > n_sess // 2
    log.close()
    b.close()


# -- 8 -----------------------------------------------------------------------------------------------------------------
def _mix64(z):
    z = z + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


@pytest.mark.parametrize("size", [1, 5, 8, 13, 64, 101, 400])
def test_host_obstacle_checksum_matches_numpy(size):
    rng = np.random.default_rng(size)
    px = rng.integers(-128, 128, (size, size)).astype(np.int8)
    px.flat[0], px.flat[-1] = -128, 127
    with np.errstate(over="ignore"):
        i = np.arange(size * size, dtype=np.uint64)
        want = int(np.sum((px.reshape(-1).view(np.uint8).astype(np.uint64) + np.uint64(1)) * _mix64(i), dtype=np.uint64))
    assert sn.host_obstacle_checksum(px, size) == want
    # position-dependent: a swap of two different cells changes it
    q = px.copy().reshape(-1)
    q[0], q[-1] = q[-1], q[0]
    if size > 1:
        assert sn.host_obstacle_checksum(q, size) != want
