"""The heading-sorted slab search (cs_sort_kernel + cs_search2_kernel) vs the CPU oracle and vs the warp-per-candidate
kernel, through the C ABI.  CS_FLAG_SEARCH_SLAB forces the slab kernels for any candidate count, CS_FLAG_SEARCH_WARP
forces the other one; without either flag the library picks by candidate count (>= 1024 candidates: slabs).

Bit-exact: per-candidate distances, arg-min under the reference's tie-break order, poses, maps.
"""
import numpy as np
import pytest

import slam.net_b200 as sn
from slam.net_b200 import _native as N
from slam.net_b200 import parallel as par
from slam.net_b200 import synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

SLAB, WARP = N.FLAG_SEARCH_SLAB, N.FLAG_SEARCH_WARP


def _oracle_map(size, phys, pixels):
    m = orc.HoleMap(size, phys)
    m.pixels[:] = pixels
    return m


@pytest.mark.parametrize("layout", [0, N.FLAG_ROW_MAJOR_MAP])
@pytest.mark.parametrize("size,n_points,iters,threads", [(64, 1, 1, 1), (100, 37, 7, 3), (256, 360, 250, 4), (333, 2049, 33, 2),
                                                         (512, 5000, 16, 4), (300, 129, 1500, 3), (300, 70, 3011, 3)])
def test_slab_search_distances_bit_exact(layout, size, n_points, iters, threads):
    rng = np.random.default_rng(size * 7 + n_points)
    phys = 10.0
    px = synth.random_map(size, seed=size)
    p = sn.Processor(phys, size, (0, 0, 0), 0.1, 0.17, iters, threads, flags=layout | SLAB, max_points=max(n_points, 64), seed=1)
    p.map_upload(px)
    m = _oracle_map(size, phys, px)
    pts = rng.normal(0, 3.0, (n_points, 2)).astype(np.float32)
    for trial in range(3):
        sp = np.array([rng.uniform(0, phys), rng.uniform(0, phys), rng.uniform(-7, 7)], dtype=np.float32)
        if trial == 2:
            sp[:2] = [-3.0, phys + 2.0]  # mostly out of bounds
        off = rng.normal(0, [0.3, 0.3, 0.4], (iters * threads, 3)).astype(np.float32)
        cand = (sp[None, :] + off).astype(np.float32)
        best, bd, d, bi = orc.parallel_search(m, pts, sp, off, iters, threads)
        res, dist = p.search(pts, sp, cand)
        assert np.array_equal(dist, d)
        assert (res.distance, res.index) == (bd, bi)
        assert np.array_equal(res.pose, best)
    # fewer candidates than the handle's T*I in one call (the scratch is reused, sums must be back at zero)
    n_few = max(1, (iters * threads) // 3)
    best, bd, d, bi = orc.parallel_search(m, pts, sp, off[:n_few], n_few, 1)
    res, dist = p.search(pts, sp, cand[:n_few])
    assert np.array_equal(dist, d) and (res.distance, res.index) == (bd, bi)
    p.close()


def test_slab_search_edge_cases():
    size, phys = 128, 8.0
    p = sn.Processor(phys, size, (0, 0, 0), 0.1, 0.17, 8, 2, flags=SLAB, seed=1)
    px = synth.random_map(size, 3)
    p.map_upload(px)
    m = _oracle_map(size, phys, px)
    sp = np.array([4.0, 4.0, 0.5], dtype=np.float32)
    off = np.random.default_rng(0).normal(0, 0.2, (16, 3)).astype(np.float32)
    off[3, 2] = np.nan   # a NaN heading sorts into bin 0 and evaluates to int.MaxValue like in the reference
    off[5, 2] = 1e9      # far outside the binned range
    off[6, 2] = -1e9
    pts = np.array([[np.nan, 0.0], [np.inf, 1.0], [-np.inf, -1.0], [1e30, 1e30], [-1e30, 2.0], [0.3, -0.2],
                    [-4.0 - 0.5 / 16, -4.0 - 0.5 / 16], [3.99, 3.99], [1e-40, -1e-40]], dtype=np.float32)
    best, bd, d, bi = orc.parallel_search(m, pts, sp, off, 8, 2)
    res, dist = p.search(pts, sp, sp[None, :] + off)
    assert np.array_equal(dist, d) and (res.distance, res.index) == (bd, bi)
    far = np.array([1e6, -1e6, 0.0], dtype=np.float32)
    off[3, 2] = 0.1
    res, dist = p.search(pts[5:8], far, far[None, :] + off)
    assert (dist == 2147483647).all() and res.index == 0 and res.distance == 2147483647
    assert np.array_equal(res.pose, far)
    p.map_fill(1234)  # ties: every candidate in bounds -> flat index 0 wins
    small = np.array([[0.1, 0.1], [-0.1, 0.2]], dtype=np.float32)
    res, dist = p.search(small, sp, sp[None, :] + off * 0.01)
    assert res.index == 0 and (dist == 1234 * 1024).all()
    cand = (sp[None, :] + off).astype(np.float32)  # host-supplied cos/sin table is honoured
    ang = np.concatenate([[sp[2]], cand[:, 2]]).astype(np.float32)
    c, s = orc.libm_sincos(ang)
    p.map_upload(px)
    r1, d1 = p.search(pts, sp, cand)
    r2, d2 = p.search(pts, sp, cand, cand_cs=np.stack([c, s], axis=1))
    assert np.array_equal(d1, d2) and r1.index == r2.index
    p.close()


@pytest.mark.parametrize("iters", [300, 2500])  # 2500 x 4 + 1 candidates: the two-kernel sort
def test_slab_search_philox_mode_matches_host_twin(iters):
    size, phys, threads = 256, 10.0, 4
    p = sn.Processor(phys, size, (0, 0, 0), 0.1, 0.17, iters, threads, flags=SLAB, seed=0xC0FFEE)
    px = synth.random_map(size, 9)
    p.map_upload(px)
    m = _oracle_map(size, phys, px)
    pts = np.random.default_rng(4).normal(0, 2.0, (200, 2)).astype(np.float32)
    sp = np.array([5.0, 5.0, -1.0], dtype=np.float32)
    for scan in (0, 1, 77):
        off = sn.philox_offsets(0xC0FFEE, scan, iters * threads, 0.1, 0.17)
        best, bd, d, bi = orc.parallel_search(m, pts, sp, off, iters, threads)
        res, dist = p.search(pts, sp, None, scan_index=scan)
        assert np.array_equal(dist, d)
        assert (res.distance, res.index) == (bd, bi) and np.array_equal(res.pose, best)
    p.close()


@pytest.mark.parametrize("philox", [False, True])
@pytest.mark.parametrize("layout", [0, N.FLAG_ROW_MAJOR_MAP])
def test_slab_update_replay_bit_exact(philox, layout):
    n_scans, n_points, size, phys, iters, threads = 40, 360, 400, 40.0, 100, 4
    rp = synth.make_replay(n_scans, n_points, phys, seed=0x5EED0000)
    p = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, flags=layout | SLAB, max_points=n_points, seed=0x5EED0000)
    o = orc.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads)
    for k in range(n_scans):
        if philox:
            off = sn.philox_offsets(0x5EED0000, k, iters * threads, 0.1, 0.17)
            res = p.update(rp.points[k], rp.odometry[k], None)
        else:
            off = synth.candidate_offsets(0x5EED0000, k, iters * threads, 0.1, 0.17)
            res = p.update(rp.points[k], rp.odometry[k], off)
        o.update(rp.points[k], rp.odometry[k], off)
        assert np.array_equal(res.pose, o.pose), "scan %d" % k
        if res.searched:
            assert res.distance == o.last_distance and res.index == o.last_index
    assert np.array_equal(p.map_download(), np.array(o.map.pixels))
    p.close()


@pytest.mark.parametrize("philox", [False, True])
def test_slab_scanlog_replay_back_to_back(philox):
    """cs_replay queues every scan's sort / search / draw kernels back to back (programmatic dependent launches, no host
    round trip): the chain must give the oracle's poses and map, and the same as the warp-per-candidate kernel."""
    n_scans, n_points, size, phys, iters, threads = 60, 512, 640, 40.0, 320, 4
    rp = synth.make_replay(n_scans, n_points, phys, seed=77)
    log = sn.ScanLog(n_scans, n_points, n_offsets=0 if philox else iters * threads)
    offs = []
    for k in range(n_scans):
        off = (sn.philox_offsets(99, k, iters * threads, 0.1, 0.17) if philox else synth.candidate_offsets(5, k, iters * threads, 0.1, 0.17))
        offs.append(off)
        log.set(k, rp.points[k], rp.odometry[k], None if philox else off)
    log.upload()
    out = {}
    for name, flag in (("slab", SLAB), ("warp", WARP), ("auto", 0)):
        q = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, flags=flag, max_points=n_points, seed=99)
        res = q.replay(log, 0, 25)
        res += q.replay(log, 25, n_scans - 25)
        out[name] = (res, q.map_download(), q.get_pose())
        q.close()
    o = orc.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads)
    for k in range(n_scans):
        o.update(rp.points[k], rp.odometry[k], offs[k])
        for name in out:
            r = out[name][0][k]
            assert np.array_equal(r.pose, o.pose), (name, k)
            if k >= 5:
                assert (r.distance, r.index) == (o.last_distance, o.last_index), (name, k)
    for name in out:
        assert np.array_equal(out[name][1], np.array(o.map.pixels)), name
        assert np.array_equal(out[name][2], o.pose)
    log.close()


def test_slab_cfg2_slice_distances_equal_warp_kernel_and_oracle():
    """configs[1] at full size: 4096 candidates x 1024 points, 2048x2048 — the default choice here is the slab search."""
    n = 10
    rp = synth.make_replay(n, 1024, 40.0)
    ps = [sn.Processor(40.0, 2048, rp.odometry[0], 0.1, 0.17, 1024, 4, max_points=1024, flags=N.FLAG_KEEP_DISTANCES | f)
          for f in (0, WARP)]
    o = orc.Processor(40.0, 2048, rp.odometry[0], 0.1, 0.17, 1024, 4)
    for k in range(n):
        off = synth.candidate_offsets(12, k, 4096, 0.1, 0.17)
        rs = [p.update(rp.points[k], rp.odometry[k], off) for p in ps]
        sp = o.pose + (rp.odometry[k] - np.array(list(o._p.contents.last_odometry_pose), dtype=np.float32))
        if k >= 5:
            _, _, d, _ = orc.parallel_search(o.map, rp.points[k], sp.astype(np.float32), off, 1024, 4)
            for p in ps:
                assert np.array_equal(p.distances(), d)
        o.update(rp.points[k], rp.odometry[k], off)
        for r in rs:
            assert np.array_equal(r.pose, o.pose)
    assert ps[0].search_plan(1024)["slab"] and not ps[1].search_plan(1024)["slab"]  # the default really is the slab search
    for p in ps:
        assert np.array_equal(p.map_download(), np.array(o.map.pixels))
        p.close()


def test_slab_candidate_split_two_handles_one_device():
    """The multi-GPU candidate split with the slab kernels: each 'rank' sorts and evaluates its own slice of the flat indices."""
    import torch
    n_scans, P, size, phys, iters, threads = 14, 300, 320, 40.0, 61, 4
    rp = synth.make_replay(n_scans, P, phys, seed=21)
    ranks = [sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=P, seed=3, flags=SLAB) for _ in range(2)]
    o = orc.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads)
    n_flat = iters * threads + 1
    for k in range(n_scans):
        off = synth.candidate_offsets(4, k, iters * threads, 0.1, 0.17)
        ptrs = []
        for g, p in enumerate(ranks):
            lo, cnt = par.candidate_slice(n_flat, 2, g)
            ptrs.append(p.update_begin(rp.points[k], rp.odometry[k], off, lo, cnt))
        if k >= 5:
            for p in ranks:
                p.sync()
            keys = [par.device_key_tensor(x, 0) for x in ptrs]
            m = torch.minimum(keys[0], keys[1])
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


@pytest.mark.parametrize("flags", [SLAB, 0])
def test_slab_batch_update_matches_oracle_per_session(flags):
    """Session batches (grid.z = session): per-session sort + slab search, ragged point counts, verification tables.
    flags = 0: 300 candidates per session is above the batch threshold (256), so the default is the slab search too."""
    n_sess, n_scans, P, size, phys, iters, threads = 5, 12, 200, 256, 40.0, 150, 2
    rps = [synth.make_replay(n_scans, P, phys, seed=50 + j) for j in range(n_sess)]
    sxy = [0.05 + 0.02 * j for j in range(n_sess)]
    sth = [0.10 + 0.01 * j for j in range(n_sess)]
    b = sn.Batch(n_sess, phys, size, [rp.odometry[0] for rp in rps], sxy, sth, iters, threads, max_points=P, flags=flags)
    os_ = [orc.Processor(phys, size, rps[j].odometry[0], sxy[j], sth[j], iters, threads) for j in range(n_sess)]
    for k in range(n_scans):
        offs = np.stack([synth.candidate_offsets(70 + j, k, iters * threads, sxy[j], sth[j]) for j in range(n_sess)])
        pts = [rps[j].points[k][: P - 7 * j] for j in range(n_sess)]  # every session its own point count
        res = b.update(pts, np.stack([rps[j].odometry[k] for j in range(n_sess)]), offs)
        for j in range(n_sess):
            os_[j].update(pts[j], rps[j].odometry[k], offs[j])
            assert np.array_equal(res[j].pose, os_[j].pose), (k, j)
            if k >= 5:
                assert (res[j].distance, res[j].index) == (os_[j].last_distance, os_[j].last_index), (k, j)
    sums = b.map_checksums()
    for j in range(n_sess):
        assert int(sums[j]) == sn.host_map_checksum(np.array(os_[j].map.pixels), size)
    b.close()


def test_batch_with_scans_of_several_rounds():
    """A batch whose largest scan has more than 2048 rays, with ragged point counts (2600, 1500 and 700 rays in one launch
    sized for the largest): the draw kernel's big-scan path for a batch (grid.y = session, each session's task table built
    from its own counts, its tasks dealt over its blocks).  Every session must still equal the oracle (poses, winners, maps)."""
    n_sess, n_scans, P, size, phys, iters, threads = 3, 8, 2600, 512, 40.0, 40, 2
    rps = [synth.make_replay(n_scans, P, phys, seed=150 + j) for j in range(n_sess)]
    sxy, sth = [0.05, 0.07, 0.09], [0.10, 0.11, 0.12]
    b = sn.Batch(n_sess, phys, size, [rp.odometry[0] for rp in rps], sxy, sth, iters, threads, max_points=P)
    os_ = [orc.Processor(phys, size, rps[j].odometry[0], sxy[j], sth[j], iters, threads) for j in range(n_sess)]
    keep = [P, 1500, 700]  # three rounds, two rounds, one round
    for k in range(n_scans):
        offs = np.stack([synth.candidate_offsets(170 + j, k, iters * threads, sxy[j], sth[j]) for j in range(n_sess)])
        pts = [rps[j].points[k][: keep[j]] for j in range(n_sess)]
        res = b.update(pts, np.stack([rps[j].odometry[k] for j in range(n_sess)]), offs)
        for j in range(n_sess):
            os_[j].update(pts[j], rps[j].odometry[k], offs[j])
            assert np.array_equal(res[j].pose, os_[j].pose), (k, j)
            if k >= 5:
                assert (res[j].distance, res[j].index) == (os_[j].last_distance, os_[j].last_index), (k, j)
    for j in range(n_sess):
        assert np.array_equal(b.map_download(j), np.array(os_[j].map.pixels)), j
    b.close()


def test_slab_batch_replay_shared_log_philox():
    """Parameter sweep in production mode: one shared device-resident log, per-session seeds and sigmas, on-device Philox
    candidates sorted per session; equal to the oracle fed the host twin's deviates."""
    n_sess, n_scans, P, size, phys, iters, threads = 4, 14, 180, 200, 40.0, 80, 4
    rp = synth.make_replay(n_scans, P, phys, seed=9)
    seeds = [11, 22, 33, 44]
    sxy = [0.05, 0.1, 0.15, 0.2]
    sth = [0.05, 0.1, 0.17, 0.25]
    b = sn.Batch(n_sess, phys, size, rp.odometry[0], sxy, sth, iters, threads, max_points=P, seeds=seeds, flags=SLAB)
    log = sn.ScanLog(n_scans, P, n_offsets=0)
    for k in range(n_scans):
        log.set(k, rp.points[k], rp.odometry[k])
    log.upload()
    b.replay(log, 0, 6)
    res = b.replay(log, 6, n_scans - 6)
    for j in range(n_sess):
        o = orc.Processor(phys, size, rp.odometry[0], sxy[j], sth[j], iters, threads)
        for k in range(n_scans):
            o.update(rp.points[k], rp.odometry[k], sn.philox_offsets(seeds[j], k, iters * threads, sxy[j], sth[j]))
        assert np.array_equal(res[j].pose, o.pose) and (res[j].distance, res[j].index) == (o.last_distance, o.last_index)
        assert np.array_equal(b.map_download(j), np.array(o.map.pixels))
    log.close()
    b.close()


def test_slab_cfg2_back_to_back_equals_scan_by_scan():
    """cfg2 geometry: 150 scans queued back to back (programmatic dependent launches: the next scan's sort and search
    prologue run while the previous scan is still being integrated, map lines cached in L1 by one search are rewritten by
    the integration before the next search) must end exactly where the same scans end when every one is waited for."""
    n = 150
    rp = synth.make_replay(n, 1024, 40.0, seed=91)
    log = sn.ScanLog(n, 1024, n_offsets=4096)
    for k in range(n):
        log.set(k, rp.points[k], rp.odometry[k], synth.candidate_offsets(91, k, 4096, 0.1, 0.17))
    log.upload()
    out = []
    for chunk in (n, 1):
        p = sn.Processor(40.0, 2048, rp.odometry[0], 0.1, 0.17, 1024, 4, max_points=1024)
        assert p.search_plan(1024)["slab"]
        res = []
        for first in range(0, n, chunk):
            res += p.replay(log, first, chunk)  # want_results: waits for the chunk
        out.append((res, p.map_checksum(), p.get_pose()))
        p.close()
    (ra, ca, pa), (rb, cb, pb) = out
    assert ca == cb and np.array_equal(pa, pb)
    assert all(np.array_equal(x.pose, y.pose) and (x.distance, x.index) == (y.distance, y.index) for x, y in zip(ra, rb))
    log.close()


def test_glue_table_is_used_and_changes_nothing():
    """One session alone with the slab search: the publishing thread takes the winner's pose and (cos, sin) from the glue table
    the service warps filled (diagnostics record: word 4 of the publisher's record = 1) — for uploaded tables and for on-device
    Philox candidates — and every pose, distance, index and the final map equal the oracle's, as without the table."""
    n_scans, P, size, phys, iters, threads = 16, 500, 512, 40.0, 300, 4  # 1201 candidates: slab search
    rp = synth.make_replay(n_scans, P, phys, seed=77)
    p = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=P, seed=13)
    o = orc.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads)
    assert p.search_plan(P)["slab"]
    p.ring_cycles()  # enables the diagnostics records
    from_table = 0
    for k in range(n_scans):
        philox = k % 2 == 1
        off = sn.philox_offsets(13, k, iters * threads, 0.1, 0.17) if philox else synth.candidate_offsets(3, k, iters * threads, 0.1, 0.17)
        r = p.update(rp.points[k], rp.odometry[k], None if philox else off)
        o.update(rp.points[k], rp.odometry[k], off)
        assert np.array_equal(r.pose, o.pose), k
        if k >= 5:
            assert (r.distance, r.index) == (o.last_distance, o.last_index), k
            p.sync()
            rec = p.ring_cycles(size + 8192)[size + 8191]
            from_table += int(rec[4] == 1)
    assert from_table == n_scans - 5, from_table
    assert np.array_equal(p.map_download(), np.array(o.map.pixels))
    p.close()


def test_sort_queued_ahead_is_dropped_when_the_next_step_differs():
    """Slab search, one session: behind every searched scan the next scan's candidate sort is queued (production mode, and
    replays of a device-resident log with tables).  What was sorted ahead must only be used by the step it was sorted for:
    here the log is re-uploaded with another table for the next scan, the replay jumps to a non-consecutive scan, and a
    production-mode scan is followed by a table scan and back — every pose, distance and index must equal the oracle's."""
    n_scans, P, size, phys, iters, threads = 14, 400, 512, 40.0, 300, 4  # 1201 candidates: slab search
    n_cand = iters * threads
    rp = synth.make_replay(n_scans, P, phys, seed=91)
    offs = [synth.candidate_offsets(17, k, n_cand, 0.1, 0.17) for k in range(n_scans)]
    p = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=P, seed=21)
    o = orc.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads)
    assert p.search_plan(P)["slab"]
    log = sn.ScanLog(n_scans, P, n_offsets=n_cand)
    for k in range(n_scans):
        log.set(k, rp.points[k], rp.odometry[k], offs[k])
    log.upload()

    def check(r, k, off):
        o.update(rp.points[k], rp.odometry[k], off)
        assert np.array_equal(r.pose, o.pose), k
        if o.last_index >= 0:
            assert (r.distance, r.index) == (o.last_distance, o.last_index), k

    for k in range(7):                       # scans 0..6 one by one: scan k+1's sort is queued behind scan k
        check(p.replay(log, k, 1)[0], k, offs[k])
    new7 = synth.candidate_offsets(99, 7, n_cand, 0.1, 0.17)
    log.set(7, rp.points[7], rp.odometry[7], new7)   # another table for the scan whose sort is already queued
    log.upload()
    check(p.replay(log, 7, 1)[0], 7, new7)
    check(p.replay(log, 9, 1)[0], 9, offs[9])        # a jump: scan 8's sort was queued, scan 9 is asked for
    ph = sn.philox_offsets(21, 9, n_cand, 0.1, 0.17)  # (the Philox counter is the number of Updates so far: 0..7 and 9 = nine)
    r = p.update(rp.points[10], rp.odometry[10], None)  # production mode: sorted ahead of nothing, queues its own successor
    check(r, 10, ph)
    r = p.update(rp.points[11], rp.odometry[11], offs[11])  # a host table behind a production-mode scan
    check(r, 11, offs[11])
    ph = sn.philox_offsets(21, 11, n_cand, 0.1, 0.17)
    r = p.update(rp.points[12], rp.odometry[12], None)
    check(r, 12, ph)
    assert np.array_equal(p.map_download(), np.array(o.map.pixels))
    log.close()
    p.close()
