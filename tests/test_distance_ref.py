"""relocalize_ref.numpy_volume, the vectorised reference of the lattice distance, against the CPU oracle pose by pose
(oracle_volume, one CalculateDistanceSISD call per pose): random and driven maps, lattices that straddle and leave the
map, headings at 0, +-pi/2, +-pi and at +-1e3 and +-1e5 rad, non-finite, huge, denormal and (-1, 0) points, and a
full-capacity scan of 65536 points on a map of 65535.  The GPU tests of the distance kernels check against
numpy_volume, so it has to be the oracle's function exactly.  No GPU needed."""
import numpy as np
import pytest

from oracle import oracle as orc
from relocalize_ref import INT_MAX, lattice_axes, numpy_volume, oracle_volume

f32 = np.float32
# the point set of the search edge-case tests: NaN, +-inf, +-1e30, (-1, 0) landings and denormals
EDGE_POINTS = np.array([[np.nan, 0.0], [np.inf, 1.0], [-np.inf, -1.0], [1e30, 1e30], [-1e30, 2.0], [0.3, -0.2],
                        [-4.0 - 0.5 / 16, -4.0 - 0.5 / 16], [3.99, 3.99], [1e-40, -1e-40], [0.0, np.nan],
                        [-1e-45, 1e-45]], dtype=np.float32)


def _oracle_map(pixels, size, phys):
    m = orc.HoleMap(size, phys)
    m.pixels[:] = np.asarray(pixels, dtype=np.uint16).ravel()
    return m


def _driven(size, phys):
    from slam.net_b200 import synth
    rp = synth.make_replay(12, 180, phys)
    m = orc.HoleMap(size, phys)
    m.fill(32750)
    for k in range(12):
        orc.update_hole_map(m, rp.points[k], rp.odometry[k], 0.6, 50)
    return m, rp.points[5]


def _check(m, pts, lattice):
    ref = oracle_volume(m, pts, *lattice)
    got = numpy_volume(m.pixels, m.size, m.scale, pts, *lattice)
    assert got.shape == ref.shape and got.dtype == np.int32
    bad = np.argwhere(got != ref)
    assert bad.size == 0, (lattice, bad[:5], got[tuple(bad[0])], ref[tuple(bad[0])])
    return ref


@pytest.mark.parametrize("kind", ["random", "driven"])
def test_matches_oracle_on_maps_and_lattices(kind):
    from slam.net_b200 import synth
    size, phys = 96, 8.0
    if kind == "random":
        m = _oracle_map(synth.random_map(size, seed=11), size, phys)
        pts = np.random.default_rng(3).normal(0, 2.0, (57, 2)).astype(np.float32)
    else:
        m, pts = _driven(size, 40.0)
        size, phys = m.size, 40.0
    lattices = [
        ([-0.3 * phys, -0.2 * phys, -3.5], [1.6 * phys / 23, 1.5 * phys / 19, 0.9], [24, 20, 8]),  # straddles the map
        ([1.5 * phys, -2.0 * phys, 0.3], [0.1, 0.1, 0.2], [6, 5, 3]),                              # wholly off it
        ([0.45 * phys, 0.4 * phys, 0.0], [0.3 * phys / size, 0.27 * phys / size, 0.01], [17, 13, 4]),  # fine
    ]
    vols = [_check(m, pts, lat) for lat in lattices]
    assert (vols[0] == INT_MAX).any() and (vols[0] < INT_MAX).any()
    assert (vols[1] == INT_MAX).all()


@pytest.mark.parametrize("center", [0.0, np.pi / 2, -np.pi / 2, np.pi, -np.pi, 1e3, -1e3, 1e5, -1e5])
def test_matches_oracle_at_special_and_large_headings(center):
    """Headings one ulp-scale step around 0, +-pi/2, +-pi (exact zeros of cos or sin in f32 nearby), and far out where
    the range reduction of cosf/sinf is the large-argument one."""
    from slam.net_b200 import synth
    size, phys = 80, 8.0
    m = _oracle_map(synth.random_map(size, seed=5), size, phys)
    pts = np.random.default_rng(9).normal(0, 2.5, (41, 2)).astype(np.float32)
    c = f32(center)
    step = max(float(np.spacing(c)) * 3, 1e-7)
    lattice = ([1.0, 1.5, float(c - f32(5 * step))], [0.6, 0.55, step], [11, 9, 11])
    _check(m, pts, lattice)
    # a coarse heading sweep around the same centre
    _check(m, pts, ([2.0, 2.0, float(c) - 3.0], [0.9, 0.8, 0.7], [6, 6, 9]))


def test_matches_oracle_on_non_finite_extreme_and_boundary_points():
    from slam.net_b200 import synth
    size, phys = 128, 8.0
    px = synth.random_map(size, seed=3)
    m = _oracle_map(px, size, phys)
    scale = f32(m.scale)
    rng = np.random.default_rng(1)
    # points that land in (-1, 0) at pose (0, 0, 0) (cell 0, in bounds) and just below -1 (off the map), and just below
    # size (the last cell)
    cell = 1.0 / float(scale)
    edge = np.array([[-0.9 * cell, 0.1], [0.1, -0.9 * cell], [-1.6 * cell, 0.2], [0.2, -1.6 * cell],
                     [phys - 0.6 * cell, 0.3], [0.3, phys - 0.6 * cell], [-0.5 * cell, -0.5 * cell]], dtype=np.float32)
    pts = np.concatenate([EDGE_POINTS, edge, rng.normal(0, 2.0, (30, 2)).astype(np.float32)])
    lattices = [
        ([0.0, 0.0, 0.0], [0.25 * cell, 0.25 * cell, 0.01], [9, 9, 3]),          # heading 0 at the map's corner
        ([-0.5, -0.5, -3.2], [0.45, 0.45, 0.8], [21, 21, 9]),                    # straddles the map
        ([3.0, 4.0, 1e5], [0.5, 0.5, 0.37], [5, 4, 6]),                          # a large heading
    ]
    for lat in lattices:
        _check(m, pts, lat)
    # only non-finite and huge points: no point is ever in bounds
    vol = _check(m, EDGE_POINTS[[0, 1, 2, 3, 4, 9]], lattices[1])
    assert (vol == INT_MAX).all()
    # (-1, 0) landings are cell 0: at pose (0, 0, 0) these three points all read cell (0, 0)
    corner = np.array([[-0.9 * cell, 0.0], [0.0, -0.9 * cell], [-0.5 * cell, -0.5 * cell]], dtype=np.float32)
    vol = _check(m, corner, ([0.0, 0.0, 0.0], [1.0, 1.0, 1.0], [1, 1, 1]))
    assert vol[0, 0, 0] == int(px[0]) * 1024


def test_full_capacity_scan_on_a_saturated_map():
    """65536 points on a map of 65535: the sum 65535 * 65536 needs all 32 bits of an unsigned accumulator.  Checked
    against the value computed by hand, against the oracle, and with one point off the map (65535 in bounds)."""
    size, phys = 64, 8.0
    m = orc.HoleMap(size, phys)
    m.fill(65535)
    rng = np.random.default_rng(2)
    pts = rng.uniform(-1.5, 1.5, (65536, 2)).astype(np.float32)
    lattice = ([3.5, 3.6, -0.4], [0.1, 0.12, 0.5], [3, 2, 2])
    vol = _check(m, pts, lattice)
    assert (vol == 65535 * 1024).all()
    one_off = pts.copy()
    one_off[777] = [1e3, 0.0]
    vol = _check(m, one_off, lattice)
    assert (vol == (65535 * 65535 * 1024) // 65536).all()
    # a few lower cells: the poses differ
    m.pixels.reshape(size, size)[28:36, 30:34] = 1000
    vol = _check(m, pts, lattice)
    assert len(np.unique(vol)) > 1 and (vol < 65535 * 1024).all()


def test_lattice_axes_single_points():
    xs, ys, ts = lattice_axes([1.0, 2.0, 3.0], [0.5, 0.25, 7.0], [1, 3, 1])
    assert list(xs) == [1.0] and list(ys) == [2.0, 2.25, 2.5] and list(ts) == [3.0]
