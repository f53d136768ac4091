"""cs_relocalize_bounded on the device: its hits are those of cs_relocalize on the same handle (poses, distances, indices,
order) in both map layouts, on random and driven maps, with 1, 37 and 5000 points, windows 0..2 and k of 1, 8 and 64,
odd counts, single-point axes and poses wholly off the map; a pass that has to raise its upper bound; the capacity
error; no effect on an Update sequence; and one lattice of more than 2^28 poses against the reference selection.

Everything here needs a B200 (pytest -m gpu)."""
import ctypes as C

import numpy as np
import pytest

import slam.net_b200 as sn
from slam.net_b200 import _native as N
from slam.net_b200 import synth
from relocalize_ref import INT_MAX, reference_hits

pytestmark = pytest.mark.gpu

LAYOUTS = [0, N.FLAG_ROW_MAJOR_MAP]


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
    return [(h.distance, h.index, h.pose.tobytes()) for h in hits]


def _same(p, pts, lattice, window, k):
    """The bounded call's hits against cs_relocalize's on the same handle; returns the stats."""
    ref, _ = p.relocalize(pts, *lattice, window=window, k=k)
    got, stats = p.relocalize_bounded(pts, *lattice, window=window, k=k)
    assert _hits(got) == _hits(ref), (lattice, window, k, stats)
    c = lattice[2]
    assert stats["poses"] == c[0] * c[1] * c[2]
    assert stats["passes"] >= 1 and stats["levels"] >= 1
    assert 0 <= stats["evaluated"] <= stats["passes"] * stats["poses"]
    return stats


# (map, size, phys, points): a single point, more than one chunk of points, driven maps
CASES = [("random", 333, 10.0, 1), ("random", 256, 10.0, 37), ("random", 512, 10.0, 5000), ("replay", 400, 40.0, 360),
         ("replay", 1024, 30.0, 37)]


def _case(kind, size, phys, n_points, flags):
    rng = np.random.default_rng(size + n_points)
    if kind == "random":
        px = synth.random_map(size, seed=size)
        pts = rng.normal(0, 0.2 * phys, (n_points, 2)).astype(np.float32)
    else:
        px, rp = _driven_map(size, phys, 20, n_points, flags)
        pts = rp.points[7]
    p = sn.Processor(phys, size, [0, 0, 0], 0.1, 0.17, 8, 1, flags=flags, max_points=max(n_points, 64))
    p.map_upload(px)
    # odd counts; x from -10 % to 125 % of the map (poses partly off it); headings -4 .. +3.5 rad
    coarse = ([-0.1 * phys, -0.05 * phys, -4.0], [1.35 * phys / 212, 1.1 * phys / 177, 0.75], [213, 177, 11])
    # a fine lattice (about a quarter of a cell per step) over part of the room: the deep levels of the descent prune
    cell = phys / size
    fine = ([0.3 * phys, 0.35 * phys, -3.3], [0.27 * cell, 0.23 * cell, 0.11], [301, 259, 7])
    return p, pts, [coarse, fine]


@pytest.fixture(scope="module", params=[(c, f) for c in CASES for f in LAYOUTS],
                ids=["%s-%d-%dpts-%s" % (c[0], c[1], c[3], "rowmajor" if f else "tiled") for c in CASES for f in LAYOUTS])
def case(request):
    (kind, size, phys, n_points), flags = request.param
    p, pts, lattices = _case(kind, size, phys, n_points, flags)
    yield p, pts, lattices
    p.close()


@pytest.mark.parametrize("window", [0, 1, 2])
@pytest.mark.parametrize("k", [1, 8, 64])
def test_hits_match_relocalize(case, window, k):
    p, pts, lattices = case
    for lattice in lattices:
        _same(p, pts, lattice, window, k)


def test_single_point_axes_and_off_map_poses():
    size, phys = 400, 40.0
    px, rp = _driven_map(size, phys, 20, 360)
    p = sn.Processor(phys, size, [0, 0, 0], 0.1, 0.17, 8, 1, max_points=360)
    p.map_upload(px)
    pts = rp.points[9]
    lattices = [
        ([20.0, -5.0, -1.0], [0.3, 0.21, 0.2], [1, 255, 9]),   # one x
        ([-5.0, 20.0, 2.5], [0.21, 0.3, 0.2], [255, 1, 9]),    # one y
        ([-3.0, 4.0, 0.7], [0.13, 0.17, 0.2], [333, 290, 1]),  # one heading
        ([17.0, 23.0, -7.0], [0.1, 0.1, 0.05], [1, 1, 501]),   # headings only, beyond -2 pi
        ([-60.0, -60.0, 0.0], [0.5, 0.5, 0.3], [64, 64, 5]),   # wholly off the map: no hit at all
        ([-60.0, 10.0, 0.0], [0.55, 0.5, 0.3], [161, 37, 5]),  # the first columns wholly off the map
    ]
    for lattice in lattices:
        for window, k in [(0, 8), (1, 64), (2, 1)]:
            _same(p, pts, lattice, window, k)
    got, _ = p.relocalize_bounded(pts, *lattices[4], window=1, k=8)
    assert got == []
    p.close()


def test_raised_upper_bound_is_still_exact():
    """A uniform map: every pose of the lattice has the same distance, so with window 1 there is one window minimum
    (flat index 0) and the first U (the k-th seed distance) finds fewer than k: the second pass runs with
    U = INT32_MAX - 1 and evaluates everything."""
    size, phys = 256, 10.0
    p = sn.Processor(phys, size, [0, 0, 0], 0.1, 0.17, 8, 1, max_points=64)
    p.map_upload(np.full((size, size), 31000, dtype=np.uint16))
    pts = np.random.default_rng(4).normal(0, 0.5, (40, 2)).astype(np.float32)
    # 3 x 3 top-level nodes per heading: 54 seeds, all at the same distance, so the first U is that distance
    lattice = ([3.0, 3.0, -0.5], [0.01, 0.01, 0.1], [301, 283, 6])
    stats = _same(p, pts, lattice, 1, 8)
    assert stats["passes"] >= 2
    assert stats["upper_bound"] == INT_MAX - 1
    # a plateau in a driven room: a window of equal distances ahead of the better poses
    px, rp = _driven_map(size, phys, 20, 64)
    px = px.reshape(size, size)
    px[60:200, 60:200] = 20000
    p.map_upload(px)
    stats = _same(p, pts, ([4.0, 4.0, -0.5], [0.02, 0.02, 0.1], [120, 120, 6]), 2, 64)
    p.close()


def test_capacity_on_a_uniform_map_leaves_the_handle_usable():
    """(Also the handle's first relocalisation call: the bounded call allocates its scratch itself.)"""
    size, phys = 2048, 20.0
    p = sn.Processor(phys, size, [0, 0, 0], 0.1, 0.17, 8, 1, max_points=64)
    p.map_upload(np.full((size, size), 30000, dtype=np.uint16))
    pts = np.random.default_rng(6).normal(0, 0.3, (16, 2)).astype(np.float32)
    # 2048 x 2048 x 300 poses on the map, 1.2e6 tiles of 32 x 32: none can be pruned, more than 2^20 survive
    big = ([1.0, 1.0, -1.0], [0.008, 0.008, 0.01], [2048, 2048, 300])
    with pytest.raises(sn.CoreSlamError) as e:
        p.relocalize_bounded(pts, *big, window=0, k=8)
    assert e.value.status == 5  # CS_ERR_CAPACITY
    # a lattice the budget allows, the same call as cs_relocalize; and an Update
    _same(p, pts, ([1.0, 1.0, -1.0], [0.008, 0.008, 0.01], [300, 300, 40]), 1, 8)
    with pytest.raises(sn.CoreSlamError):
        p.relocalize_bounded(pts, *big, window=0, k=65)
    r = p.update(pts, [4.0, 4.0, 0.0])
    assert r.pose.shape == (3,)
    p.close()


def test_bad_arguments():
    size, phys = 128, 8.0
    p = sn.Processor(phys, size, [4, 4, 0], 0.1, 0.17, 8, 2, max_points=64)
    p.map_upload(synth.random_map(size, seed=2))
    pts = np.random.default_rng(2).normal(0, 1.0, (16, 2)).astype(np.float32)

    def status(lattice, n=16, k=4, window=0, stats=True):
        lat = N.Lattice()
        lat.origin = (C.c_float * 3)(*lattice[0])
        lat.step = (C.c_float * 3)(*lattice[1])
        lat.count = (C.c_int32 * 3)(*lattice[2])
        out = (N.LatticeHit * 64)()
        nh = C.c_int32()
        st = N.RelocalizeStats()
        return N.lib().cs_relocalize_bounded(p._h, pts.ctypes.data_as(C.POINTER(C.c_float)), n, C.byref(lat), window, k, out,
                                             C.byref(nh), C.byref(st) if stats else None)

    good = ([1.0, 1.0, -1.0], [0.5, 0.5, 0.2], [8, 8, 8])
    assert status(good) == 0 and status(good, stats=False) == 0
    assert status(good, n=0) == 1 and status(good, k=0) == 1 and status(good, window=-1) == 1
    assert status((good[0], [0.5, 0.0, 0.2], good[2])) == 1
    assert status(good, n=65) == 5
    # 2^31 poses: over CS_LATTICE_MAX_POSES_BOUNDED; and more than 2^28 tiles
    assert status((good[0], good[1], [1 << 16, 1 << 15, 1])) == 5
    assert status((good[0], good[1], [1, 1, (1 << 28) + 1])) == 5
    p.close()


# ------------------------------------------------------------------------------------------------
# no effect on the handle's Update sequence
# ------------------------------------------------------------------------------------------------
def _drive(interleave):
    n_scans, n_points, size, phys, iters, threads = 10, 360, 512, 40.0, 128, 4
    rp = synth.make_replay(n_scans, n_points, phys)
    p = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=n_points, seed=0xBEEF)
    out = []
    for k in range(n_scans):
        if interleave and k > 0:
            pose = p.get_pose()
            lattice = ([5.0, 5.0, -np.pi], [0.05, 0.05, np.pi / 45], [601, 601, 90])
            p.relocalize_bounded(rp.points[k - 1], *lattice, window=1, k=8)
            assert np.array_equal(p.get_pose(), pose)
        r = p.update(rp.points[k], rp.odometry[k])
        out.append((r.pose.tobytes(), r.distance, r.index, r.searched, p.map_checksum()))
    p.close()
    return out


def test_bounded_calls_between_updates_change_nothing():
    assert _drive(True) == _drive(False)


# ------------------------------------------------------------------------------------------------
# more than 2^28 poses (one cs_relocalize call takes at most 2^28): against the reference selection on the full volume
# ------------------------------------------------------------------------------------------------
def test_lattice_over_the_exhaustive_limit():
    size, phys, n_points = 2048, 40.0, 360
    px, rp = _driven_map(size, phys, 40, n_points)
    p = sn.Processor(phys, size, [0, 0, 0], 0.1, 0.17, 64, 4, max_points=n_points)
    p.map_upload(px)
    pts = rp.points[23]
    # 4 cm x 2/3 degree over the room: 751 x 751 x 540 = 3.05e8 poses, assembled from one cs_relocalize call per heading
    origin, step, count = [5.0, 5.0, -np.pi], [0.04, 0.04, float(np.float32(2 * np.pi / 540))], [751, 751, 540]
    total = count[0] * count[1] * count[2]
    assert total > N.LATTICE_MAX_POSES
    vol = np.empty((count[2], count[1], count[0]), dtype=np.int32)
    for it in range(count[2]):
        # heading `it` of the lattice is origin + (float)it * step in f32, the origin of a lattice with one heading
        th = np.float32(origin[2]) + np.float32(it) * np.float32(step[2])
        _, part = p.relocalize(pts, [origin[0], origin[1], float(th)], step, [count[0], count[1], 1], window=0, k=1,
                               want_distances=True)
        vol[it] = part[0]
    for window, k in [(1, 8), (0, 64)]:
        got, stats = p.relocalize_bounded(pts, origin, step, count, window=window, k=k)
        ref = reference_hits(vol, window, k)
        assert [(h.distance, h.index) for h in got] == ref, stats
        assert stats["poses"] == total
        assert stats["evaluated"] < total
    p.close()

