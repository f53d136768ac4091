"""CUDA path vs CPU oracle through the C ABI — bit-exact distances, arg-min, poses and map cells.

Everything here needs a B200 (pytest -m gpu).  The oracle (oracle/) is the checker only.
"""
import numpy as np
import pytest

import slam.net_b200 as sn
from slam.net_b200 import _native as N
from slam.net_b200 import synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

LAYOUTS = [0, N.FLAG_ROW_MAJOR_MAP]


def _mk(size, phys, iters, threads, flags=0, max_points=0, start=(0, 0, 0), seed=1):
    return sn.Processor(phys, size, start, 0.1, 0.17, iters, threads, flags=flags, max_points=max_points, seed=seed)


def _oracle_map(size, phys, pixels):
    m = orc.HoleMap(size, phys)
    m.pixels[:] = pixels
    return m


# ------------------------------------------------------------------------------------------------
# search
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flags", LAYOUTS)
@pytest.mark.parametrize("size,n_points,iters,threads", [(64, 1, 1, 1), (100, 37, 7, 3), (256, 360, 250, 4),
                                                         (333, 2049, 33, 2), (512, 5000, 16, 4)])
def test_search_distances_bit_exact(flags, size, n_points, iters, threads):
    rng = np.random.default_rng(size * 7 + n_points)
    phys = 10.0
    px = synth.random_map(size, seed=size)
    p = _mk(size, phys, iters, threads, flags=flags, max_points=max(n_points, 64))
    p.map_upload(px)
    assert np.array_equal(p.map_download(), px)
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
    p.close()


def test_search_edge_cases():
    size, phys = 128, 8.0
    p = _mk(size, phys, 8, 2)
    px = synth.random_map(size, 3)
    p.map_upload(px)
    m = _oracle_map(size, phys, px)
    sp = np.array([4.0, 4.0, 0.5], dtype=np.float32)
    off = np.random.default_rng(0).normal(0, 0.2, (16, 3)).astype(np.float32)
    # NaN / inf / huge points, points that land in (-1, 0) (truncate to cell 0, in bounds)
    pts = np.array([[np.nan, 0.0], [np.inf, 1.0], [-np.inf, -1.0], [1e30, 1e30], [-1e30, 2.0], [0.3, -0.2],
                    [-4.0 - 0.5 / 16, -4.0 - 0.5 / 16], [3.99, 3.99], [1e-40, -1e-40]], dtype=np.float32)
    best, bd, d, bi = orc.parallel_search(m, pts, sp, off, 8, 2)
    res, dist = p.search(pts, sp, sp[None, :] + off)
    assert np.array_equal(dist, d) and (res.distance, res.index) == (bd, bi)
    # nothing in bounds at all -> int.MaxValue everywhere, searchPose wins
    far = np.array([1e6, -1e6, 0.0], dtype=np.float32)
    res, dist = p.search(pts[5:8], far, far[None, :] + off)
    assert (dist == 2147483647).all() and res.index == 0 and res.distance == 2147483647
    assert np.array_equal(res.pose, far)
    # ties: constant map, every candidate in bounds -> flat index 0
    p.map_fill(1234)
    small = np.array([[0.1, 0.1], [-0.1, 0.2]], dtype=np.float32)
    res, dist = p.search(small, sp, sp[None, :] + off * 0.01)
    assert res.index == 0 and (dist == 1234 * 1024).all()
    # host-supplied cos/sin table is honoured
    cand = (sp[None, :] + off).astype(np.float32)
    ang = np.concatenate([[sp[2]], cand[:, 2]]).astype(np.float32)
    c, s = orc.libm_sincos(ang)
    p.map_upload(px)
    r1, d1 = p.search(pts, sp, cand)
    r2, d2 = p.search(pts, sp, cand, cand_cs=np.stack([c, s], axis=1))
    assert np.array_equal(d1, d2) and r1.index == r2.index
    p.close()


def test_search_kat_a_fresh_map():
    p = _mk(64, 8.0, 4, 1, start=(4, 4, 0))
    pts = np.array([[0.5, 0.0], [0.0, 0.5], [-0.5, 0.25]], dtype=np.float32)
    sp = np.array([4.0, 4.0, 0.3], dtype=np.float32)
    res, d = p.search(pts, sp, np.tile(sp, (4, 1)))
    assert (d == 33536000).all()
    far = np.array([[0.5, 0.0], [100.0, 0.0], [0.0, 200.0]], dtype=np.float32)
    res, d = p.search(far, [4.0, 4.0, 0.0], np.tile(np.array([4.0, 4.0, 0.0], dtype=np.float32), (4, 1)))
    assert (d == (32750 * 1024) // 3).all()
    p.close()


def test_search_philox_mode_matches_host_twin():
    size, phys, iters, threads = 256, 10.0, 100, 4
    p = _mk(size, phys, iters, threads, seed=0xC0FFEE)
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


# ------------------------------------------------------------------------------------------------
# integration
# ------------------------------------------------------------------------------------------------
def test_integrate_kat_c():
    p = _mk(32, 8.0, 1, 1, flags=N.FLAG_DEBUG_RAYS)
    pts = np.array([[2.0, 0.0]], dtype=np.float32)
    v = p.integrate(pts, [4.0, 4.0, 0.0])
    # default HoleWidth is 0.6; KAT-C uses 2.4
    p.map_fill(32750)
    p.set_hole_width(2.4)
    v = p.integrate(pts, [4.0, 4.0, 0.0])
    assert v == 14
    assert list(p.rays(1)[0]) == [16, 16, 29, 16, 24, 16]
    row = p.map_download().reshape(32, 32)[16]
    expect = {16: 39146, 17: 39146, 18: 39146, 19: 39146, 20: 36587, 21: 34029, 22: 31470, 23: 28912,
              24: 26353, 25: 28912, 26: 31470, 27: 34029, 28: 36587, 29: 39146}
    for x in range(32):
        assert row[x] == expect.get(x, 32750), x
    res, d = p.search(pts, [4.0, 4.0, 0.0], np.array([[4.0, 4.0, 0.0]], dtype=np.float32))
    assert d[0] == 26985472
    p.close()


@pytest.mark.parametrize("flags", LAYOUTS)
@pytest.mark.parametrize("size,n_rays,hw,q", [(64, 90, 0.6, 50), (200, 360, 0.6, 50), (256, 2048, 2.0, 200),
                                              (512, 4096, 0.3, 1), (96, 700, 5.0, 255)])
def test_integrate_map_bit_exact(flags, size, n_rays, hw, q):
    rng = np.random.default_rng(size + n_rays)
    phys = 8.0
    p = _mk(size, phys, 1, 1, flags=flags | N.FLAG_DEBUG_RAYS, max_points=n_rays)
    p.set_hole_width(hw)
    p.set_quality(q)
    m = orc.HoleMap(size, phys)
    m.fill(32750)
    for k in range(4):
        ang = np.linspace(0, 2 * np.pi, n_rays, endpoint=False) + rng.uniform(0, 0.01)
        if k == 2:  # unordered angles: ray order is the list order, not the angular order
            ang = rng.permutation(ang)
        rad = rng.uniform(0.02, 7.0, n_rays)
        if k == 3:  # walls hugging the robot: many rays per cell, short rays inside the hole width
            rad = rng.uniform(0.01, 0.5, n_rays)
        pts = np.stack([rad * np.cos(ang), rad * np.sin(ang)], axis=1).astype(np.float32)
        pose = np.array([rng.uniform(0.2, 7.8), rng.uniform(0.2, 7.8), rng.uniform(-4, 4)], dtype=np.float32)
        vo, rays_o = orc.update_hole_map(m, pts, pose, hw, q, rays=True)
        vg = p.integrate(pts, pose)
        assert np.array_equal(p.rays(n_rays), rays_o)
        assert vg == vo
        got = p.map_download()
        assert np.array_equal(got, np.array(m.pixels)), "scan %d: %d cells differ" % (k, np.count_nonzero(got != m.pixels))
    assert p.map_checksum() == sn.host_map_checksum(np.array(m.pixels), size)
    p.close()


def test_integrate_ray_order_kat_d():
    """Forward and reversed ray order give different maps; the GPU must match the forward order."""
    rng = np.random.default_rng(7)
    n = 2048
    ang = np.linspace(0, 2 * np.pi, n, endpoint=False)
    rad = 1.0 + 0.5 * rng.random(n)
    pts = np.stack([rad * np.cos(ang), rad * np.sin(ang)], axis=1).astype(np.float32)
    pose = [4.0, 4.0, 0.1]
    a = orc.HoleMap(256, 8.0)
    b = orc.HoleMap(256, 8.0)
    a.fill(32750)
    b.fill(32750)
    orc.update_hole_map(a, pts, pose, 0.6, 50)
    orc.update_hole_map(b, pts[::-1].copy(), pose, 0.6, 50)
    p = _mk(256, 8.0, 1, 1, max_points=n)
    p.integrate(pts, pose)
    got = p.map_download()
    assert np.array_equal(got, np.array(a.pixels))
    assert not np.array_equal(got, np.array(b.pixels))
    p.map_fill(32750)
    p.integrate(pts[::-1].copy(), pose)
    assert np.array_equal(p.map_download(), np.array(b.pixels))
    p.close()


def test_integrate_edge_cases():
    size, phys = 64, 8.0
    p = _mk(size, phys, 1, 1)
    m = orc.HoleMap(size, phys)
    m.fill(32750)
    pts = np.array([[30.0, 0.1], [-30.0, 5.0], [0.2, 40.0], [3.0, -45.0], [25.0, 25.0], [-25.0, 24.0],  # clipped
                    [0.05, 0.0], [0.0, -0.05], [1.0, 1.0], [1.0, 1.0], [-2.0, 2.0],                     # short, duplicate, diagonal
                    [2.0, 0.0], [0.0, 2.0], [-2.0, 0.0], [0.0, -2.0]], dtype=np.float32)               # axis aligned
    for pose in ([4.0, 4.0, 0.0], [0.01, 0.01, 0.7], [7.99, 7.99, -2.0], [0.0, 7.9, 3.0]):
        vo = orc.update_hole_map(m, pts, pose, 0.6, 50)
        vg = p.integrate(pts, pose)
        assert vg == vo
        assert np.array_equal(p.map_download(), np.array(m.pixels))
    # robot outside the map: nothing is drawn (:509-512)
    before = p.map_download()
    assert p.integrate(pts, [-1.0, 4.0, 0.0]) == 0
    assert p.integrate(pts, [4.0, 9.0, 0.0]) == 0
    assert np.array_equal(p.map_download(), before)
    p.close()


# ------------------------------------------------------------------------------------------------
# Update: state machine + search + integration
# ------------------------------------------------------------------------------------------------
def _replay_pair(n_scans, n_points, size, phys, iters, threads, philox, flags=0, seed=0x5EED0000):
    rp = synth.make_replay(n_scans, n_points, phys, seed=seed)
    start = rp.odometry[0]
    p = sn.Processor(phys, size, start, 0.1, 0.17, iters, threads, flags=flags, max_points=n_points, seed=seed)
    o = orc.Processor(phys, size, start, 0.1, 0.17, iters, threads)
    return rp, p, o


@pytest.mark.parametrize("philox", [False, True])
@pytest.mark.parametrize("flags", LAYOUTS)
def test_update_replay_bit_exact(philox, flags):
    n_scans, n_points, size, phys, iters, threads = 40, 360, 400, 40.0, 100, 4
    rp, p, o = _replay_pair(n_scans, n_points, size, phys, iters, threads, philox, flags)
    for k in range(n_scans):
        if philox:
            off = sn.philox_offsets(0x5EED0000, k, iters * threads, 0.1, 0.17)
            res = p.update(rp.points[k], rp.odometry[k], None)
        else:
            off = synth.candidate_offsets(0x5EED0000, k, iters * threads, 0.1, 0.17)
            res = p.update(rp.points[k], rp.odometry[k], off)
        o.update(rp.points[k], rp.odometry[k], off)
        assert np.array_equal(res.pose, o.pose), "scan %d" % k
        assert res.searched == (k >= 5)
        if res.searched:
            assert res.distance == o.last_distance and res.index == o.last_index
    assert np.array_equal(p.get_pose(), o.pose)
    assert np.array_equal(p.map_download(), np.array(o.map.pixels))
    # the search actually follows the truth trajectory (sanity of the workload, not parity)
    err = np.hypot(*(p.get_pose()[:2] - rp.truth[-1][:2]))
    assert err < 0.5
    p.close()


def test_update_reset_and_properties():
    rp, p, o = _replay_pair(12, 200, 256, 40.0, 50, 2, False)
    p.set_position_search_beginning(2)
    o.position_search_beginning = 2
    p.set_quality(120)
    o.quality = 120
    p.set_hole_width(1.5)
    o.hole_width = 1.5
    for rnd in range(2):
        for k in range(12):
            off = synth.candidate_offsets(1, k, 100, 0.1, 0.17)
            res = p.update(rp.points[k], rp.odometry[k], off)
            o.update(rp.points[k], rp.odometry[k], off)
            assert np.array_equal(res.pose, o.pose)
            assert res.searched == (k >= 2)
        assert np.array_equal(p.map_download(), np.array(o.map.pixels))
        p.reset()
        o.reset()
        assert (p.map_download() == 32750).all()
        assert np.array_equal(p.get_pose(), o.pose)
    p.close()


def test_replay_api_equals_update_sequence():
    n_scans, n_points, size, phys, iters, threads = 30, 300, 320, 40.0, 64, 2
    rp, p, o = _replay_pair(n_scans, n_points, size, phys, iters, threads, False)
    log = sn.ScanLog(n_scans, n_points, n_offsets=iters * threads)
    offs = [synth.candidate_offsets(5, k, iters * threads, 0.1, 0.17) for k in range(n_scans)]
    for k in range(n_scans):
        log.set(k, rp.points[k], rp.odometry[k], offs[k])
        o.update(rp.points[k], rp.odometry[k], offs[k])
    log.upload()
    res = p.replay(log, 0, 10) + p.replay(log, 10, 20)
    assert np.array_equal(res[-1].pose, o.pose)
    assert np.array_equal(p.map_download(), np.array(o.map.pixels))
    # same through cs_update on a second handle
    q = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=n_points)
    for k in range(n_scans):
        r = q.update(rp.points[k], rp.odometry[k], offs[k])
        assert np.array_equal(r.pose, res[k].pose) and r.distance == res[k].distance and r.index == res[k].index
    assert q.map_checksum() == p.map_checksum()
    assert sum(r.visits for r in res) > 0
    log.close()
    p.close()
    q.close()


def test_mirror_class_update():
    """The reference-shaped class: CoreSLAMProcessor(...).Update(List<ScanSegment>)."""
    rp = synth.make_replay(8, 180, 40.0)
    T, I = 2, 40
    with sn.CoreSLAMProcessor(40.0, 256, 64, rp.odometry[0], 0.1, 0.17, I, T, max_points=180) as slam:
        o = orc.Processor(40.0, 256, rp.odometry[0], 0.1, 0.17, I, T)
        assert slam.HoleMap.Size == 256 and slam.HoleMap.Scale == np.float32(256 / 40.0)
        slam.HoleWidth = 2.0
        o.hole_width = 2.0
        ang = (np.arange(180) * (2 * np.pi / 180)).astype(np.float32)
        for k in range(8):
            rad = np.hypot(rp.points[k][:, 0], rp.points[k][:, 1]).astype(np.float32)
            seg = sn.ScanSegment(Rays=np.stack([ang, rad], axis=1), Pose=rp.odometry[k], IsLast=True)
            off = synth.candidate_offsets(9, k, T * I, 0.1, 0.17)
            slam.Update([seg], candidateOffsets=off)
            cloud = orc.segment_to_cloud(np.stack([ang, rad], axis=1), rp.odometry[k], rp.odometry[k])
            o.update(cloud, rp.odometry[k], off)
            assert np.array_equal(slam.Pose, o.pose)
        assert np.array_equal(slam.HoleMap.Pixels, np.array(o.map.pixels))
        assert np.array_equal(slam.HoleMap.GetPackedPixels(), o.map.packed())


# ------------------------------------------------------------------------------------------------
# BASELINE.json configurations at full size
# ------------------------------------------------------------------------------------------------
def test_cfg1_single_scan_1000_iterations():
    """configs[0]: 360-point scan, 1000 iterations, 1600x1600 @2.5 cm."""
    rp = synth.make_replay(8, 360, 40.0)
    for threads in (1, 4):
        p = sn.Processor(40.0, 1600, rp.odometry[0], 0.1, 0.17, 1000, threads, max_points=360)
        o = orc.Processor(40.0, 1600, rp.odometry[0], 0.1, 0.17, 1000, threads)
        for k in range(8):
            off = synth.candidate_offsets(11, k, 1000 * threads, 0.1, 0.17)
            r = p.update(rp.points[k], rp.odometry[k], off)
            o.update(rp.points[k], rp.odometry[k], off)
            assert np.array_equal(r.pose, o.pose)
        assert p.map_checksum() == sn.host_map_checksum(np.array(o.map.pixels), 1600)
        p.close()


def test_cfg2_replay_slice_4096x1024():
    """configs[1] at full size for a slice of the replay: 4096 candidates x 1024 points, 2048x2048."""
    n = 12
    rp = synth.make_replay(n, 1024, 40.0)
    p = sn.Processor(40.0, 2048, rp.odometry[0], 0.1, 0.17, 1024, 4, max_points=1024, flags=N.FLAG_KEEP_DISTANCES)
    o = orc.Processor(40.0, 2048, rp.odometry[0], 0.1, 0.17, 1024, 4)
    for k in range(n):
        off = synth.candidate_offsets(12, k, 4096, 0.1, 0.17)
        r = p.update(rp.points[k], rp.odometry[k], off)
        sp = o.pose + (rp.odometry[k] - np.array(list(o._p.contents.last_odometry_pose), dtype=np.float32))
        if k >= 5:
            _, _, d, _ = orc.parallel_search(o.map, rp.points[k], sp.astype(np.float32), off, 1024, 4)
            assert np.array_equal(p.distances(), d)
        o.update(rp.points[k], rp.odometry[k], off)
        assert np.array_equal(r.pose, o.pose)
    assert np.array_equal(p.map_download(), np.array(o.map.pixels))
    p.close()


def test_cfg3_integration_stress_8192_rays_4096_map():
    """configs[2]: 8192-ray scans at 1 cm into a 4096x4096 map, bit-exact map diff."""
    rp = synth.make_replay(6, 8192, 40.96)
    p = sn.Processor(40.96, 4096, rp.odometry[0], 0.1, 0.17, 1, 1, max_points=8192)
    m = orc.HoleMap(4096, 40.96)
    m.fill(32750)
    for k in range(6):
        pose = rp.truth[k].astype(np.float32)
        vo = orc.update_hole_map(m, rp.points[k], pose, 0.6, 50)
        vg = p.integrate(rp.points[k], pose)
        assert vg == vo
    got = p.map_download()
    assert np.array_equal(got, np.array(m.pixels)), "%d cells differ" % np.count_nonzero(got != m.pixels)
    p.close()


@pytest.mark.parametrize("n_rays", [2500, 4096])
def test_integrate_large_map_several_rounds_sorted_and_unsorted(n_rays):
    """Big scans (more than 2048 rays) on a 4096 x 4096 map, rays up to 3000 cells long: the draw kernel's big-scan path
    (the 64-register instance, the task table built from the scan's own counts).  A permuted scan puts candidates of every
    wedge into every batch of 32 rays, and short rays among the long ones crowd the inner levels.  Sorted, permuted,
    reversed and border-clipped scans, all bit-exact against the cell-by-cell oracle."""
    size, phys = 4096, 40.96
    rng = np.random.default_rng(n_rays)
    p = _mk(size, phys, 1, 1, max_points=n_rays)
    m = orc.HoleMap(size, phys)
    m.fill(32750)
    for k in range(5):
        ang = np.linspace(0, 2 * np.pi, n_rays, endpoint=False) + rng.uniform(0, 0.01)
        rad = rng.uniform(8.0, 19.0, n_rays)
        if k == 1:
            ang = rng.permutation(ang)       # unordered: rays of one round lie all around the ring
        if k == 2:
            ang = ang[::-1].copy()
        if k == 3:
            ang = rng.permutation(ang)
            rad = np.where(rng.random(n_rays) < 0.5, rng.uniform(0.05, 2.0, n_rays), rad)  # contested inner cells too
        if k == 4:
            rad = rng.uniform(11.0, 30.0, n_rays)  # far ends clipped at the map border
        pts = np.stack([rad * np.cos(ang), rad * np.sin(ang)], axis=1).astype(np.float32)
        pose = np.array([20.0 + rng.uniform(-1, 1), 20.0 + rng.uniform(-1, 1), rng.uniform(-3, 3)], dtype=np.float32)
        vo = orc.update_hole_map(m, pts, pose, 0.6, 50)
        vg = p.integrate(pts, pose)
        assert vg == vo, k
        got = p.map_download()
        assert np.array_equal(got, np.array(m.pixels)), "scan %d: %d cells differ" % (k, np.count_nonzero(got != m.pixels))
    p.close()


def test_cfg4_large_map_search_8192():
    """configs[3] single-GPU part: 8192x8192 map (128 MB), large candidate set, distances bit-exact."""
    size, phys = 8192, 81.92
    rp = synth.make_replay(3, 1024, phys)
    p = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, 2048, 4, max_points=1024)
    m = orc.HoleMap(size, phys)
    m.fill(32750)
    for k in range(3):
        pose = rp.truth[k].astype(np.float32)
        orc.update_hole_map(m, rp.points[k], pose, 0.6, 50)
        p.integrate(rp.points[k], pose)
    sp = rp.truth[2].astype(np.float32)
    off = synth.candidate_offsets(13, 0, 8192, 0.1, 0.17)
    best, bd, d, bi = orc.parallel_search(m, rp.points[2], sp, off, 2048, 4)
    res, dist = p.search(rp.points[2], sp, sp[None, :] + off)
    assert np.array_equal(dist, d) and (res.distance, res.index) == (bd, bi)
    assert p.map_checksum() == sn.host_map_checksum(np.array(m.pixels), size)
    p.close()
