"""cs_relocalize on the device against the CPU oracle: every distance of the lattice, the window-minima selection, the
hits against cs_search, relocalising a scan on a map built by another processor and resuming there, and no effect on
the Update sequence of the handle.

Everything here needs a B200 (pytest -m gpu).  The oracle (oracle/) is the checker only."""
import ctypes as C

import numpy as np
import pytest

import slam.net_b200 as sn
from slam.net_b200 import _native as N
from slam.net_b200 import synth
from oracle import oracle as orc
from relocalize_ref import INT_MAX, lattice_pose, oracle_volume, reference_hits

pytestmark = pytest.mark.gpu

LAYOUTS = [0, N.FLAG_ROW_MAJOR_MAP]


def _oracle_map(size, phys, pixels):
    m = orc.HoleMap(size, phys)
    m.pixels[:] = pixels
    return m


def _driven_map(size, phys, n_scans, n_points, flags=0):
    """The HoleMap after a synthetic drive (synth.make_replay) through the room."""
    rp = synth.make_replay(n_scans, n_points, phys)
    p = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, 64, 4, max_points=n_points, flags=flags, seed=3)
    for k in range(n_scans):
        p.update(rp.points[k], rp.odometry[k])
    px = p.map_download()
    p.close()
    return px, rp


def _hits(hits):
    return [(h.distance, h.index) for h in hits]


# ------------------------------------------------------------------------------------------------
# every distance of small lattices
# ------------------------------------------------------------------------------------------------
# (map, size, phys, points): an odd map size, a single point, an odd count, more than one chunk of points, a driven map
CASES = [("random", 333, 10.0, 1), ("random", 256, 10.0, 37), ("random", 512, 10.0, 5000), ("replay", 400, 40.0, 360)]


def _case(kind, size, phys, n_points, flags):
    rng = np.random.default_rng(size + n_points)
    if kind == "random":
        px = synth.random_map(size, seed=size)
        pts = rng.normal(0, 3.0, (n_points, 2)).astype(np.float32)
        # x from -1 m to 23 m: the last columns lie wholly off the map; headings from -4 to +4 rad
        lattice = ([-1.0, -0.6, -4.0], [2.0, 1.1, 0.5], [13, 11, 17])
    else:
        px, rp = _driven_map(size, phys, 20, n_points, flags)
        pts = rp.points[7]
        # x from -2 m to 94 m: the poses beyond about 80 m throw every point off the 40 m map
        lattice = ([-2.0, 3.0, -3.5], [8.0, 3.1, 0.45], [13, 11, 17])
    p = sn.Processor(phys, size, [0, 0, 0], 0.1, 0.17, 8, 1, flags=flags, max_points=max(n_points, 64))
    p.map_upload(px)
    return p, _oracle_map(size, phys, px), pts, lattice


@pytest.mark.parametrize("flags", LAYOUTS)
@pytest.mark.parametrize("kind,size,phys,n_points", CASES)
def test_lattice_distances_match_the_oracle(flags, kind, size, phys, n_points):
    p, m, pts, (origin, step, count) = _case(kind, size, phys, n_points, flags)
    hits, vol = p.relocalize(pts, origin, step, count, window=1, k=64, want_distances=True)
    ref = oracle_volume(m, pts, origin, step, count)
    assert vol.shape == (count[2], count[1], count[0])
    assert np.array_equal(vol, ref)
    assert (ref == INT_MAX).any() and (ref < INT_MAX).any()  # wholly off the map, and in reach
    assert _hits(hits) == reference_hits(ref, 1, 64)
    # a hit is a lattice pose as evaluated, and cs_search returns the same distance for it as an absolute candidate
    for h in hits[:8]:
        assert np.array_equal(h.pose, lattice_pose(origin, step, count, h.index))
        res, d = p.search(pts, h.pose, h.pose[None, :])
        assert d[1] == h.distance == d[0]
    p.close()


# ------------------------------------------------------------------------------------------------
# selection: window minima + top-k over a volume of several select blocks and merge rounds
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big_case():
    size, phys = 256, 10.0
    px = synth.random_map(size, seed=21)
    pts = np.random.default_rng(21).normal(0, 2.5, (24, 2)).astype(np.float32)
    # 80 x 50 x 50 = 200000 poses: 49 blocks of the select kernel, two merge rounds
    lattice = ([-0.5, 0.25, -3.3], [0.14, 0.21, 0.13], [80, 50, 50])
    p = sn.Processor(phys, size, [0, 0, 0], 0.1, 0.17, 8, 1, max_points=64)
    p.map_upload(px)
    ref = oracle_volume(_oracle_map(size, phys, px), pts, *lattice)
    yield p, pts, lattice, ref
    p.close()


@pytest.mark.parametrize("window", [0, 1, 2])
@pytest.mark.parametrize("k", [1, 8, 64])
def test_hits_match_the_reference_selection(big_case, window, k):
    p, pts, (origin, step, count), ref = big_case
    hits, vol = p.relocalize(pts, origin, step, count, window=window, k=k, want_distances=(k == 8))
    if vol is not None:
        assert np.array_equal(vol, ref)
    assert _hits(hits) == reference_hits(ref, window, k)
    assert len(hits) == k


def test_fewer_minima_than_k_and_nothing_in_reach():
    size, phys = 128, 8.0
    p = sn.Processor(phys, size, [0, 0, 0], 0.1, 0.17, 8, 1, max_points=64)
    px = synth.random_map(size, seed=5)
    p.map_upload(px)
    pts = np.random.default_rng(5).normal(0, 1.0, (9, 2)).astype(np.float32)
    lattice = ([1.0, 1.5, 0.2], [0.9, 0.8, 0.6], [6, 5, 4])
    ref = oracle_volume(_oracle_map(size, phys, px), pts, *lattice)
    hits, _ = p.relocalize(pts, *lattice, window=2, k=64)
    assert 0 < len(hits) < 64 and _hits(hits) == reference_hits(ref, 2, 64)
    # a window wider than the lattice: the global minimum alone
    hits, _ = p.relocalize(pts, *lattice, window=2**31 - 1, k=64)
    assert _hits(hits) == reference_hits(ref, 6, 64) and len(hits) == 1
    # a constant map: a plateau where the lower flat index wins every tie
    p.map_fill(1000)
    ref = oracle_volume(_oracle_map(size, phys, np.full(size * size, 1000, np.uint16)), pts, *lattice)
    hits, _ = p.relocalize(pts, *lattice, window=1, k=64)
    assert _hits(hits) == reference_hits(ref, 1, 64)
    # every pose off the map
    hits, vol = p.relocalize(pts, [100.0, -50.0, 0.0], [0.5, 0.5, 0.3], [7, 6, 5], window=0, k=8, want_distances=True)
    assert hits == [] and (vol == INT_MAX).all()
    p.close()


# ------------------------------------------------------------------------------------------------
# relocalise a scan on another processor's map and resume tracking there
# ------------------------------------------------------------------------------------------------
def _angle_diff(a, b):
    return float((a - b + np.pi) % (2 * np.pi) - np.pi)


def test_relocalize_and_resume_on_a_downloaded_map():
    size, phys, n_points, iters, threads = 800, 40.0, 360, 250, 4  # 5 cm cells
    j, n_more = 40, 12
    rp = synth.make_replay(j + 1 + n_more, n_points, phys)
    a = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=n_points, seed=11)
    for k in range(j + 1):
        ra = a.update(rp.points[k], rp.odometry[k])
    pose_a = ra.pose
    b = sn.Processor(phys, size, [30.0, 8.0, 2.5], 0.1, 0.17, iters, threads, max_points=n_points, seed=12)
    b.map_upload(a.map_download())

    coarse = (0.1, 0.1, np.float32(np.pi / 90))  # 10 cm x 2 degrees over the whole room (5 m .. 35 m)
    hits, _ = b.relocalize(rp.points[j], [5.0, 5.0, -np.pi], coarse, [301, 301, 180], window=2, k=8)
    assert len(hits) == 8
    best = None
    for h in hits:  # 1 cm x 0.25 degrees over +-1 coarse step around every coarse hypothesis
        fine_step = (0.01, 0.01, np.float32(np.pi / 720))
        origin = h.pose - np.float32([0.1, 0.1, 8 * fine_step[2]])
        fh, _ = b.relocalize(rp.points[j], origin, fine_step, [21, 21, 17], window=0, k=1)
        if fh and (best is None or fh[0].distance < best.distance):
            best = fh[0]
    assert abs(best.pose[0] - pose_a[0]) <= coarse[0] and abs(best.pose[1] - pose_a[1]) <= coarse[1]
    assert abs(_angle_diff(best.pose[2], pose_a[2])) <= coarse[2]

    b.set_pose(best.pose, rp.odometry[j], scan_count=5)  # PositionSearchBeginning: the next Update searches
    cell = phys / size
    for k in range(j + 1, j + 1 + n_more):
        ra = a.update(rp.points[k], rp.odometry[k])
        rb = b.update(rp.points[k], rp.odometry[k])
        assert rb.searched
        assert np.hypot(*(rb.pose[:2] - ra.pose[:2])) <= 2 * cell, k
        assert abs(_angle_diff(rb.pose[2], ra.pose[2])) <= np.radians(1.0), k
    a.close()
    b.close()


def test_drop_in_resume_at():
    size, phys, n_points = 400, 40.0, 360
    rp = synth.make_replay(12, n_points, phys)
    a = sn.CoreSLAMProcessor(phys, size, 0, rp.odometry[0], 0.1, 0.17, 100, 4, max_points=n_points)
    for k in range(10):
        a.Update([sn.ScanSegment(Rays=_rays(rp.points[k]), Pose=tuple(rp.odometry[k]), IsLast=True)])
    b = sn.CoreSLAMProcessor(phys, size, 0, [20, 20, 0], 0.1, 0.17, 100, 4, max_points=n_points)
    b._proc.map_upload(a.HoleMap.Pixels)
    # a lattice of +-0.5 m and +-10 degrees around the truth: this test is about the drop-in's calls, the whole-room search
    # is test_relocalize_and_resume_on_a_downloaded_map's
    origin = np.float32(rp.truth[9]) - np.float32([0.5, 0.5, np.radians(10)])
    hits, _ = b.Relocalize(rp.points[9], origin, [0.05, 0.05, np.radians(1)], [21, 21, 21], 2, 4)
    assert hits and np.hypot(*(hits[0].pose[:2] - a.Pose[:2])) <= 0.15
    b.ResumeAt(hits[0].pose, rp.odometry[9])
    assert np.array_equal(b.Pose, hits[0].pose)
    seg = [sn.ScanSegment(Rays=_rays(rp.points[10]), Pose=tuple(rp.odometry[10]), IsLast=True)]
    b.Update(seg)
    assert b.LastResult.searched
    a.Dispose()
    b.Dispose()


def _rays(points):
    """(angle, radius) rays whose ScanSegmentsToCloud with segment pose = odometry gives back `points` (up to rounding)."""
    pts = np.asarray(points, dtype=np.float64)
    return np.stack([np.arctan2(pts[:, 1], pts[:, 0]), np.hypot(pts[:, 0], pts[:, 1])], axis=1).astype(np.float32)


# ------------------------------------------------------------------------------------------------
# no interference with the Update sequence
# ------------------------------------------------------------------------------------------------
def _drive(verification, interleave):
    n_scans, n_points, size, phys, iters, threads = 12, 360, 512, 40.0, 512, 4  # 2048 candidates: slab search, sort ahead
    flags = N.FLAG_KEEP_DISTANCES if verification else 0
    rp = synth.make_replay(n_scans, n_points, phys)
    p = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=n_points, flags=flags, seed=0xBEEF)
    out, upd_launches, rel_launches = [], [], []
    for k in range(n_scans):
        if interleave and k > 0:
            pose = p.get_pose()
            dist = p.distances() if verification else None
            n0 = p.launch_count()
            lattice = ([5.0, 5.0, -np.pi], [0.25, 0.25, np.pi / 45], [121, 121, 90])
            p.relocalize(rp.points[k - 1], *lattice, window=1, k=8, want_distances=(k % 2 == 0))
            rel_launches.append(p.launch_count() - n0)
            assert np.array_equal(p.get_pose(), pose)
            if verification:
                assert np.array_equal(p.distances(), dist)
        off = synth.candidate_offsets(1, k, iters * threads, 0.1, 0.17) if verification else None
        n0 = p.launch_count()
        r = p.update(rp.points[k], rp.odometry[k], off)
        upd_launches.append(p.launch_count() - n0)
        out.append((r.pose.tobytes(), r.distance, r.index, r.searched, p.map_checksum()))
    if verification:
        out.append(p.distances().tobytes())
    p.close()
    return out, upd_launches, rel_launches


@pytest.mark.parametrize("verification", [False, True], ids=["production", "verification"])
def test_relocalize_between_updates_changes_nothing(verification):
    plain, plain_launches, _ = _drive(verification, False)
    mixed, mixed_launches, rel = _drive(verification, True)
    assert mixed == plain
    assert mixed_launches == plain_launches  # no sort or other kernel added to any Update
    assert len(set(rel)) == 1 and rel[0] >= 2  # a relocalize call launches its own kernels and nothing else


# ------------------------------------------------------------------------------------------------
# bad arguments
# ------------------------------------------------------------------------------------------------
def test_bad_arguments_leave_the_handle_usable():
    size, phys = 128, 8.0
    p = sn.Processor(phys, size, [4, 4, 0], 0.1, 0.17, 8, 2, max_points=64)
    p.map_upload(synth.random_map(size, seed=2))
    pts = np.random.default_rng(2).normal(0, 1.0, (16, 2)).astype(np.float32)
    good = ([1.0, 1.0, -1.0], [0.5, 0.5, 0.2], [8, 8, 8])

    def status(points=pts, n=None, lattice=good, window=0, k=4, hits=True, n_hits=True):
        lat = N.Lattice()
        lat.origin = (C.c_float * 3)(*lattice[0])
        lat.step = (C.c_float * 3)(*lattice[1])
        lat.count = (C.c_int32 * 3)(*lattice[2])
        out = (N.LatticeHit * 64)()
        nh = C.c_int32()
        pp = None if points is None else np.ascontiguousarray(points, np.float32).ctypes.data_as(C.POINTER(C.c_float))
        return N.lib().cs_relocalize(p._h, pp, len(pts) if n is None else n, C.byref(lat), window, k, out if hits else None,
                                     C.byref(nh) if n_hits else None, None)

    bad_arg, capacity = 1, 5
    assert status() == 0
    assert status(points=None) == bad_arg
    assert status(hits=False) == bad_arg and status(n_hits=False) == bad_arg
    assert status(n=0) == bad_arg and status(n=-3) == bad_arg
    assert status(window=-1) == bad_arg
    assert status(k=0) == bad_arg and status(k=65) == bad_arg
    assert status(lattice=(good[0], good[1], [8, 0, 8])) == bad_arg
    assert status(lattice=([np.nan, 1.0, 0.0], good[1], good[2])) == bad_arg
    assert status(lattice=([1.0, np.inf, 0.0], good[1], good[2])) == bad_arg
    for s in (0.0, -0.5, np.nan, np.inf):
        assert status(lattice=(good[0], [0.5, s, 0.2], good[2])) == bad_arg
    assert status(lattice=(good[0], [0.5, np.nan, 0.2], [8, 1, 8])) == 0  # (the step of a single-point axis is unused)
    assert status(n=65) == capacity
    assert status(lattice=(good[0], good[1], [1 << 10, 1 << 10, 1 << 9])) == capacity
    # still usable: the same call, and an Update
    hits, _ = p.relocalize(pts, *good, window=0, k=4)
    assert len(hits) == 4
    with pytest.raises(sn.CoreSlamError):
        p.relocalize(pts, *good, window=0, k=65)
    r = p.update(pts, [4.0, 4.0, 0.0])
    assert r.pose.shape == (3,)
    p.close()


# ------------------------------------------------------------------------------------------------
# full size: cfg2's geometry, a whole-room lattice of about 1e8 poses
# ------------------------------------------------------------------------------------------------
def test_full_size_room_lattice():
    size, phys, n_points = 2048, 40.0, 1024
    px, rp = _driven_map(size, phys, 30, n_points)
    p = sn.Processor(phys, size, [0, 0, 0], 0.1, 0.17, 64, 4, max_points=n_points)
    p.map_upload(px)
    pts = rp.points[17]
    # 5 cm x 1.25 degrees over the room: 600 x 600 x 288 = 1.04e8 poses
    origin, step, count = [5.0, 5.0, -np.pi], [0.05, 0.05, 2 * np.pi / 288], [600, 600, 288]
    hits, vol = p.relocalize(pts, origin, step, count, window=2, k=64, want_distances=True)
    m = _oracle_map(size, phys, px)
    rng = np.random.default_rng(17)
    for idx in rng.integers(0, vol.size, 1000):
        assert vol.ravel()[idx] == orc.distance(m, pts, lattice_pose(origin, step, count, int(idx))), idx
    assert _hits(hits) == reference_hits(vol, 2, 64)
    top, _ = p.relocalize(pts, origin, step, count, window=0, k=8)
    assert _hits(top) == reference_hits(vol, 0, 8)
    p.close()
