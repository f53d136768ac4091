"""The four device implementations of the reference's distance (CalculateDistanceSISD, CoreSLAMProcessor.cs:226-259) at
the limits of their contract, against independent references (the CPU oracle, and numpy_volume / reference_hits of
relocalize_ref):

- capacity: 65536-point scans on maps of 65535, where the unsigned sums and the slab search's 17-bit in-bounds count
  are exactly full, through cs_search (warp and slab kernels), cs_relocalize, cs_relocalize_bounded and cs_update;
- non-finite, huge and denormal points, and headings of +-1e3 and +-1e5 rad, through both relocalisation calls;
- lattice shapes on either side of the 32 x 32 tiles, the 16 x 8 warp patches and the 32 / 64 / 128 top levels of the
  branch and bound, windows from 0 to wider than the lattice, and fine lattices whose wide windows reach pruned tiles;
- plateaus of equal distances from lattice steps below the float resolution of the origin;
- one handle's scratch grown and reused by calls of different shapes.

Everything here needs a B200 (pytest -m gpu)."""
import numpy as np
import pytest

import slam.net_b200 as sn
from slam.net_b200 import _native as N
from slam.net_b200 import synth
from oracle import oracle as orc
from relocalize_ref import INT_MAX, lattice_axes, numpy_volume, reference_hits

pytestmark = pytest.mark.gpu

LAYOUTS = [0, N.FLAG_ROW_MAJOR_MAP]
LAYOUT_IDS = ["tiled", "rowmajor"]
SLAB, WARP = N.FLAG_SEARCH_SLAB, N.FLAG_SEARCH_WARP
f32 = np.float32

# the point set of the search edge-case tests (test_search_edge_cases): NaN, +-inf, +-1e30, (-1, 0) landings, denormals
EDGE_POINTS = np.array([[np.nan, 0.0], [np.inf, 1.0], [-np.inf, -1.0], [1e30, 1e30], [-1e30, 2.0], [0.3, -0.2],
                        [-4.0 - 0.5 / 16, -4.0 - 0.5 / 16], [3.99, 3.99], [1e-40, -1e-40], [0.0, np.nan],
                        [np.nan, np.nan], [-1e-45, 1e-45]], dtype=np.float32)


def _proc(size, phys, flags=0, max_points=64, iters=8, threads=1, start=(0, 0, 0)):
    return sn.Processor(phys, size, start, 0.1, 0.17, iters, threads, flags=flags, max_points=max_points, seed=1)


def _driven_map(size, phys, n_scans=20, n_points=360):
    rp = synth.make_replay(n_scans, n_points, phys)
    p = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, 64, 4, max_points=n_points, seed=3)
    for k in range(n_scans):
        p.update(rp.points[k], rp.odometry[k])
    px = p.map_download()
    p.close()
    return px, rp


def _keys(hits):
    return [(h.distance, h.index) for h in hits]


def _full(hits):
    return [(h.distance, h.index, h.pose.tobytes()) for h in hits]


def _relocalize_both(p, px, pts, lattice, cases, volume=None):
    """The exhaustive volume against numpy_volume, then for every (window, k) the hits of cs_relocalize and of
    cs_relocalize_bounded against reference_hits.  Returns the bounded calls' stats."""
    origin, step, count = lattice
    if volume is None:
        volume = numpy_volume(px, p.size, p.scale, pts, origin, step, count)
    _, vol = p.relocalize(pts, origin, step, count, window=0, k=1, want_distances=True)
    bad = np.argwhere(vol != volume)
    assert bad.size == 0, ("volume", lattice, len(bad), bad[:4], vol[tuple(bad[0])], volume[tuple(bad[0])])
    out = []
    total = count[0] * count[1] * count[2]
    for window, k in cases:
        ref = reference_hits(volume, window, k)
        got, _ = p.relocalize(pts, origin, step, count, window=window, k=k)
        assert _keys(got) == ref, ("relocalize", lattice, window, k)
        bnd, st = p.relocalize_bounded(pts, origin, step, count, window=window, k=k)
        assert _full(bnd) == _full(got), ("bounded", lattice, window, k, st)
        assert st["poses"] == total and st["passes"] >= 1 and 0 <= st["evaluated"] <= st["passes"] * total
        out.append(st)
    return out


# ------------------------------------------------------------------------------------------------
# 1. capacity: 65536 points on maps of 65535
# ------------------------------------------------------------------------------------------------
CAP_SIZE, CAP_PHYS = 256, 10.0
CAP_ITERS, CAP_THREADS = 2100, 4  # 8400 candidates: more than 8192, so the slab search sorts with two kernels


def _cap_map(kind):
    px = np.full(CAP_SIZE * CAP_SIZE, 65535, dtype=np.uint16)
    if kind == "dips":  # a few lower cells, so that the arg-min is not decided by the flat index alone
        rng = np.random.default_rng(17)
        cells = rng.choice(px.size, px.size // 50, replace=False)
        px[cells] = rng.integers(30000, 65535, cells.size)
    return px


def _cap_scans():
    """65536 points all in bounds at every tested pose; the same with one point off the map; 65535 points."""
    rng = np.random.default_rng(23)
    full = rng.uniform(-3.0, 3.0, (65536, 2)).astype(np.float32)
    one_off = full.copy()
    one_off[40000] = [1e4, -1e4]
    return {"65536": full, "65536-one-off": one_off, "65535": full[:65535].copy()}


_CAP_ORACLE = {}


def _cap_oracle(kind, scan):
    """orc.parallel_search of one (map, scan) pair, computed once for every layout and kernel."""
    if (kind, scan) not in _CAP_ORACLE:
        m = orc.HoleMap(CAP_SIZE, CAP_PHYS)
        m.pixels[:] = _cap_map(kind)
        sp = np.array([5.0, 5.0, 0.3], dtype=np.float32)
        off = np.random.default_rng(5).normal(0, [0.3, 0.3, 0.4], (CAP_ITERS * CAP_THREADS, 3)).astype(np.float32)
        _CAP_ORACLE[(kind, scan)] = (sp, off, orc.parallel_search(m, _cap_scans()[scan], sp, off, CAP_ITERS, CAP_THREADS))
    return _CAP_ORACLE[(kind, scan)]


@pytest.mark.parametrize("kernel", [SLAB, WARP], ids=["slab", "warp"])
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
@pytest.mark.parametrize("kind", ["flat", "dips"])
def test_capacity_search(kind, layout, kernel):
    p = _proc(CAP_SIZE, CAP_PHYS, layout | kernel, 65536, CAP_ITERS, CAP_THREADS)
    p.map_upload(_cap_map(kind))
    for scan, pts in _cap_scans().items():
        sp, off, (best, bd, d, bi) = _cap_oracle(kind, scan)
        if scan == "65536":
            assert d[0] == 65535 * 1024 if kind == "flat" else d[0] < 65535 * 1024
        res, dist = p.search(pts, sp, sp[None, :] + off)
        assert np.array_equal(dist, d), (scan, np.count_nonzero(dist != d))
        assert (res.distance, res.index) == (bd, bi), scan
        assert np.array_equal(res.pose, best), scan
    p.close()


# every pose keeps the scan on the map: x, y in [4.6, 5.4]
CAP_LATTICE = ([4.6, 4.65, -0.5], [0.08, 0.07, 0.3], [11, 9, 3])
_CAP_VOLUME = {}


def _cap_volume(kind, scan):
    if (kind, scan) not in _CAP_VOLUME:
        _CAP_VOLUME[(kind, scan)] = numpy_volume(_cap_map(kind), CAP_SIZE, f32(CAP_SIZE) / f32(CAP_PHYS), _cap_scans()[scan], *CAP_LATTICE)
    return _CAP_VOLUME[(kind, scan)]


@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
@pytest.mark.parametrize("kind", ["flat", "dips"])
def test_capacity_relocalize(kind, layout):
    px = _cap_map(kind)
    p = _proc(CAP_SIZE, CAP_PHYS, layout, 65536)
    p.map_upload(px)
    for scan, pts in _cap_scans().items():
        stats = _relocalize_both(p, px, pts, CAP_LATTICE, [(0, 1), (0, 64), (1, 8), (3, 64)], volume=_cap_volume(kind, scan))
        if kind == "flat" and scan == "65536":
            assert stats[0]["upper_bound"] == 65535 * 1024
    p.close()


@pytest.mark.parametrize("kernel", [SLAB, WARP], ids=["slab", "warp"])
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
def test_capacity_update(layout, kernel):
    """Two whole Updates (search and HoleMap integration) of 65536 points on a map of 65535, with the candidates given
    (the verification mode), against orc.Processor: pose, distance, index and every cell of the HoleMap."""
    iters, threads = 64, 4
    start = [5.0, 5.0, 0.2]
    p = _proc(CAP_SIZE, CAP_PHYS, layout | kernel, 65536, iters, threads, start=start)
    o = orc.Processor(CAP_PHYS, CAP_SIZE, start, 0.1, 0.17, iters, threads)
    px = _cap_map("dips")
    p.map_upload(px)
    o.map.pixels[:] = px
    p.set_position_search_beginning(0)
    o.position_search_beginning = 0
    pts = _cap_scans()["65536"]
    for k, odo in enumerate([[0.0, 0.0, 0.0], [0.05, -0.03, 0.02]]):
        off = synth.candidate_offsets(0xCA9, k, iters * threads, 0.1, 0.17)
        r = p.update(pts, odo, off)
        o.update(pts, odo, off)
        assert r.searched
        assert np.array_equal(r.pose, o.pose), k
        assert (r.distance, r.index) == (o.last_distance, o.last_index), k
        got = p.map_download()
        assert np.array_equal(got, np.array(o.map.pixels)), (k, np.count_nonzero(got != o.map.pixels))
    p.close()


# ------------------------------------------------------------------------------------------------
# 2. non-finite and extreme points, large headings
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
def test_relocalize_non_finite_points_and_large_headings(layout):
    size, phys = 128, 8.0
    px = synth.random_map(size, seed=3)
    p = _proc(size, phys, layout, 512)
    p.map_upload(px)
    scan = np.random.default_rng(8).normal(0, 1.5, (300, 2)).astype(np.float32)
    pts = scan.copy()
    pts[::25][:len(EDGE_POINTS)] = EDGE_POINTS  # spread through the scan, so every chunk of points has some
    cases = [(0, 8), (1, 8), (1, 64), (3, 64)]
    lattices = [
        ([-0.4, -0.3, 0.0], [0.29, 0.31, 0.21], [33, 31, 5]),      # from the map's corner, heading 0 first
        ([1.0, 1.5, 1e3], [0.2, 0.2, 0.13], [30, 27, 6]),
        ([1.0, 1.5, -1e3], [0.2, 0.2, 0.13], [30, 27, 6]),
        ([2.0, 1.0, 1e5], [0.15, 0.17, 0.05], [33, 17, 5]),       # ulp(1e5) is 0.0078: five distinct headings
        ([2.0, 1.0, -1e5], [0.15, 0.17, 0.05], [33, 17, 5]),
    ]
    for lattice in lattices:
        _relocalize_both(p, px, pts, lattice, cases)
    # only the non-finite and huge points: nothing is ever in bounds, no hit
    far = EDGE_POINTS[[0, 1, 2, 3, 4, 9, 10]]
    lattice = lattices[0]
    _, vol = p.relocalize(far, *lattice, want_distances=True)
    assert (vol == INT_MAX).all()
    assert p.relocalize_bounded(far, *lattice, window=1, k=8)[0] == []
    p.close()


# ------------------------------------------------------------------------------------------------
# 3. lattice shapes and windows
# ------------------------------------------------------------------------------------------------
SIDES = [1, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 257]
# every side on both axes: side i along x with side i + 6 along y
SHAPES = [(SIDES[i], SIDES[(i + 6) % len(SIDES)]) for i in range(len(SIDES))]
SWEEP_CASES = [(0, 1), (0, 64), (1, 64), (3, 1), (8, 64), (16, 64), (17, 64), (33, 1), (33, 64), (300, 64)]


@pytest.fixture(scope="module")
def sweep_map():
    size, phys = 256, 20.0
    px, rp = _driven_map(size, phys, 20, 200)
    return size, phys, px, rp.points[11]


@pytest.fixture(scope="module", params=LAYOUTS, ids=LAYOUT_IDS)
def sweep_proc(request, sweep_map):
    size, phys, px, pts = sweep_map
    p = _proc(size, phys, request.param, 256)
    p.map_upload(px)
    yield p, request.param
    p.close()


@pytest.mark.parametrize("c0,c1", SHAPES, ids=["%dx%d" % s for s in SHAPES])
def test_shape_sweep(sweep_map, sweep_proc, c0, c1):
    size, phys, px, pts = sweep_map
    p, layout = sweep_proc
    if layout and (c0, c1) not in SHAPES[::3]:
        pytest.skip("the row-major layout runs every third shape")
    cell = phys / size
    # about 1.3 cells per step along x and y, over the middle of the room; three headings
    origin = [0.5 * phys - 0.65 * cell * c0, 0.5 * phys - 0.6 * cell * c1, -0.2]
    lattice = (origin, [1.3 * cell, 1.2 * cell, 0.07], [c0, c1, 3])
    _relocalize_both(p, px, pts, lattice, SWEEP_CASES)


# the top level of the descent is 32, 64 or 128 poses a side (max(c0, c1) <= 32, <= 64, else); the step sets the cell
# span of the top level's children and with it the number of min-window grids
FINE = [(32, 29, 0.25), (33, 20, 0.25), (64, 64, 0.25), (65, 47, 0.25), (128, 120, 0.25), (129, 129, 0.25),
        (257, 200, 0.25), (129, 100, 0.6), (129, 100, 1.5), (65, 70, 3.0)]


@pytest.mark.parametrize("c0,c1,per_cell", FINE, ids=["%dx%d-%g" % f for f in FINE])
def test_fine_lattices_prune_and_stay_exact(sweep_map, sweep_proc, c0, c1, per_cell):
    size, phys, px, pts = sweep_map
    p, layout = sweep_proc
    if layout and per_cell != 0.25:
        pytest.skip("the row-major layout runs the quarter-cell lattices")
    cell = phys / size
    step = per_cell * cell
    lattice = ([0.5 * phys - 0.5 * step * c0, 0.45 * phys - 0.5 * step * c1, 0.3], [step, step * 0.9, 0.04], [c0, c1, 4])
    cases = [(0, 1), (0, 64), (1, 64), (8, 64), (17, 64), (33, 64), (max(c0, c1), 8)]
    st = _relocalize_both(p, px, pts, lattice, cases)[0]
    if c0 * c1 >= 128 * 120 and per_cell < 1:
        # window 0, k 1: the best seed is a U the best pose meets in one pass, and some quarter-cell patches are bounded
        # out.  (With k 64 there are fewer seeds than k, so U starts at INT32_MAX - 1 and nothing is pruned.)
        assert st["passes"] == 1 and st["evaluated"] < st["poses"], st


# A scan of a few points: the bound of a node is then close to the distance of its poses, so a grid window narrower
# than the cell span of a point (a bound above some pose's distance) prunes a pose that is a hit.  A random map has no
# two neighbouring cells alike; 8 headings give the fine lattices enough top-level seeds for a finite first U at k 8.
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
@pytest.mark.parametrize("n_points", [1, 3, 17])
def test_few_point_scans_on_fine_lattices(layout, n_points):
    size, phys = 333, 10.0
    px = synth.random_map(size, seed=size)
    p = _proc(size, phys, layout, 64)
    p.map_upload(px)
    pts = np.random.default_rng(n_points).normal(0, 1.5, (n_points, 2)).astype(np.float32)
    cell = phys / size
    for c0, c1, per_cell in [(32, 29, 0.25), (64, 64, 0.25), (65, 47, 0.6), (129, 129, 0.25), (257, 200, 0.25),
                             (129, 100, 1.5)]:
        step = per_cell * cell
        lattice = ([0.5 * phys - 0.5 * step * c0, 0.5 * phys - 0.5 * step * c1, -0.7], [step, step, 0.09], [c0, c1, 8])
        _relocalize_both(p, px, pts, lattice, [(0, 1), (0, 8), (1, 8), (2, 64)])
    p.close()


# ------------------------------------------------------------------------------------------------
# 4. plateaus: lattice steps below the float resolution of the origin
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
def test_plateaus_from_float_resolution(layout):
    size, phys = 1024, 40.0
    px, rp = _driven_map(size, phys, 20, 180)
    p = _proc(size, phys, layout, 256)
    p.map_upload(px)
    pts = rp.points[13]
    ulp = float(np.spacing(f32(30.0)))  # 1.9e-6 m: runs of lattice x (and y) coordinates round to one value
    lattices = [([30.0, 29.0, -0.4], [0.4 * ulp, 0.7 * ulp, 0.02], [150, 140, 12]),
                ([29.9, 30.1, 1.1], [1.3 * ulp, 0.35 * ulp, 0.015], [90, 200, 8])]
    seen_second_pass = False
    for lattice in lattices:
        xs, ys, _ = lattice_axes(*lattice)
        assert len(np.unique(xs)) < len(xs) or len(np.unique(ys)) < len(ys)  # genuine runs of equal coordinates
        volume = numpy_volume(px, size, p.scale, pts, *lattice)
        cases = [(0, 64), (1, 8), (1, 64), (3, 64), (max(lattice[2]), 8)]
        c0, c1, c2 = lattice[2]
        top = next(t for t in (5, 6, 7) if max(c0, c1) <= 1 << t or t == 7)  # the descent's top level (nodes a side)
        n_top = -(-c0 >> top) * -(-c1 >> top) * c2
        for (window, k), st in zip(cases, _relocalize_both(p, px, pts, lattice, cases, volume=volume)):
            if len(reference_hits(volume, window, k)) < k and n_top >= k:
                # the first U (the k-th seed distance) is finite and fewer than k candidates exist at all
                assert st["passes"] >= 2, (lattice, window, k, st)
                seen_second_pass = True
    assert seen_second_pass
    p.close()


# ------------------------------------------------------------------------------------------------
# 5. scratch reuse on one handle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
def test_scratch_reuse_matches_fresh_handles(layout, sweep_map):
    size, phys, px, pts = sweep_map
    cell = phys / size
    mid = 0.5 * phys

    def lat(c0, c1, c2, per_cell):
        s = per_cell * cell
        return ([mid - 0.5 * s * c0, mid - 0.5 * s * c1, -0.3], [s, s, 0.05], [c0, c1, c2])

    # (bounded?, lattice, window, k, number of points): large, small, larger, small again
    calls = [(False, lat(200, 180, 6, 1.0), 2, 64, 200), (True, lat(400, 380, 8, 0.25), 1, 64, 200),
             (False, lat(9, 7, 3, 2.0), 0, 1, 37), (True, lat(33, 17, 2, 0.5), 5, 8, 37),
             (True, lat(700, 650, 10, 0.25), 3, 64, 200), (False, lat(300, 310, 9, 0.5), 1, 8, 150),
             (True, lat(16, 16, 1, 1.0), 0, 64, 1), (False, lat(64, 64, 4, 0.7), 17, 64, 200),
             (True, lat(129, 65, 5, 0.25), 33, 64, 120)]

    def run(p, call):
        bounded, lattice, window, k, n = call
        if bounded:
            return _full(p.relocalize_bounded(pts[:n], *lattice, window=window, k=k)[0]), None
        hits, vol = p.relocalize(pts[:n], *lattice, window=window, k=k, want_distances=True)
        return _full(hits), vol

    shared = _proc(size, phys, layout, 256)
    shared.map_upload(px)
    for call in calls:
        got, got_vol = run(shared, call)
        fresh = _proc(size, phys, layout, 256)
        fresh.map_upload(px)
        ref, ref_vol = run(fresh, call)
        fresh.close()
        assert got == ref, call
        assert got_vol is None or np.array_equal(got_vol, ref_vol), call
        assert got, call
    shared.close()
