"""cs_relocalize_sequence and cs_relocalize_sequence_bounded on the device: K = 1 is cs_relocalize / cs_relocalize_bounded
bit for bit whatever the odometry; every volume entry is the sum of cs_search distances of the scans at their composed
poses (and sequence_ref's volume); hits against the reference selection; bounded equals exhaustive for K up to 32 with
1-point and > 1024-point scans; the INT32_MAX rule; saturated maps at full capacity; the aliasing corridor the feature
exists for; no state change; errors and scratch reuse.

Everything here needs a B200 (pytest -m gpu)."""
import numpy as np
import pytest

import slam.net_b200 as sn
from slam.net_b200 import _native as N
from slam.net_b200 import synth
from relocalize_ref import INT_MAX, lattice_axes, lattice_pose, reference_hits
import sequence_ref as sr

pytestmark = pytest.mark.gpu

LAYOUTS = [0, N.FLAG_ROW_MAJOR_MAP]
LAYOUT_IDS = ["tiled", "rowmajor"]


def _hits(hits):
    return [(h.distance, h.index, h.pose.tobytes()) for h in hits]


def _frame(odo, rot=1.2, shift=(7.5, -3.25)):
    """poses (n, 3) expressed in an odometry frame rotated by rot and shifted"""
    odo = np.asarray(odo, dtype=np.float64)
    c, s = np.cos(rot), np.sin(rot)
    return np.stack([c * odo[:, 0] - s * odo[:, 1] + shift[0], s * odo[:, 0] + c * odo[:, 1] + shift[1], odo[:, 2] + rot],
                    axis=1).astype(np.float32)


_DRIVEN = {}


def _driven(size=400, phys=40.0, n_scans=20, n_points=360):
    """A HoleMap after a synthetic drive, and the drive (computed once per module)"""
    key = (size, phys, n_scans, n_points)
    if key not in _DRIVEN:
        rp = synth.make_replay(n_scans, n_points, phys)
        p = sn.Processor(phys, size, rp.odometry[0], 0.1, 0.17, 64, 4, max_points=n_points, seed=3)
        for k in range(n_scans):
            p.update(rp.points[k], rp.odometry[k])
        _DRIVEN[key] = (p.map_download(), rp)
        p.close()
    return _DRIVEN[key]


def _handle(px, phys, flags, max_points=2048):
    p = sn.Processor(phys, px.shape[0] if px.ndim == 2 else int(np.sqrt(px.size)), [0, 0, 0], 0.1, 0.17, 8, 1, flags=flags,
                     max_points=max_points)
    p.map_upload(px)
    return p


# the lattice shapes of the single-scan tests: odd counts, poses off the map, headings beyond +-pi
def _lattices(phys, size):
    cell = phys / size
    return [([-0.1 * phys, -0.05 * phys, -4.0], [1.35 * phys / 60, 1.1 * phys / 47, 0.75], [61, 47, 11]),
            ([0.3 * phys, 0.35 * phys, -3.3], [0.27 * cell, 0.23 * cell, 0.11], [101, 77, 5]),
            ([-60.0, 10.0, 0.0], [0.55, 0.5, 0.3], [161, 37, 3])]


@pytest.mark.parametrize("flags", LAYOUTS, ids=LAYOUT_IDS)
def test_one_scan_is_relocalize(flags):
    px, rp = _driven()
    p = _handle(px, 40.0, flags)
    pts = rp.points[9]
    for odo in ([0, 0, 0], [12.5, -7.25, 2.0], [-1e3, 3e3, -40.0]):
        for lattice in _lattices(40.0, 400):
            for window, k in [(0, 8), (1, 64), (2, 1)]:
                ref, vref = p.relocalize(pts, *lattice, window=window, k=k, want_distances=True)
                got, vol = p.relocalize_sequence([pts], [odo], *lattice, window=window, k=k, want_distances=True)
                assert np.array_equal(vol, vref) and _hits(got) == _hits(ref), (odo, lattice, window, k)
                bref, sref = p.relocalize_bounded(pts, *lattice, window=window, k=k)
                bgot, sgot = p.relocalize_sequence_bounded([pts], [odo], *lattice, window=window, k=k)
                assert _hits(bgot) == _hits(bref) == _hits(ref) and sgot == sref
    p.close()


def _drive_sequence(rp, last, n, rot=1.2):
    idx = list(range(last - n + 1, last + 1))
    return [rp.points[i] for i in idx], _frame(rp.odometry[idx], rot)


@pytest.mark.parametrize("flags", LAYOUTS, ids=LAYOUT_IDS)
@pytest.mark.parametrize("K", [2, 5])
def test_every_term_is_a_search_distance(flags, K):
    px, rp = _driven()
    phys, size = 40.0, 400
    p = _handle(px, phys, flags)
    scans, odo = _drive_sequence(rp, 17, K)
    cell = phys / size
    t0 = rp.truth[17]
    lattice = ([t0[0] - 10 * cell, t0[1] - 8 * cell, t0[2] - 0.3], [0.7 * cell, 0.9 * cell, 0.1], [29, 19, 7])
    _, vol = p.relocalize_sequence(scans, odo, *lattice, k=4, want_distances=True)
    ref = sr.sequence_volume(p.map_download(), size, p.scale, scans, odo, *lattice)
    assert np.array_equal(vol, ref)
    # a sample of poses through cs_search, each scan at its composed pose as an absolute candidate
    xs, ys, ts = lattice_axes(*lattice)
    rng = np.random.default_rng(K + flags)
    for n in rng.choice(vol.size, 40, replace=False):
        it, iy, ix = np.unravel_index(n, vol.shape)
        pose = [xs[ix], ys[iy], ts[it]]
        ds = []
        for i in range(K):
            q = sr.scan_pose(pose, odo, i)
            _, d = p.search(scans[i], q, cand_poses=q.reshape(1, 3))
            ds.append(int(d[1]))
        assert vol[it, iy, ix] == (INT_MAX if INT_MAX in ds else sum(ds)), (n, ds)
    p.close()


def test_hits_against_reference_selection():
    px, rp = _driven()
    p = _handle(px, 40.0, 0)
    scans, odo = _drive_sequence(rp, 15, 4)
    lattice = _lattices(40.0, 400)[0]
    for window in (0, 1, 2):
        for k in (1, 8, 64):
            hits, vol = p.relocalize_sequence(scans, odo, *lattice, window=window, k=k, want_distances=True)
            assert [(h.distance, h.index) for h in hits] == reference_hits(vol, window, k)
            for h in hits:
                assert h.pose.tobytes() == lattice_pose(*lattice, h.index).tobytes()
    p.close()


def _bounded_same(p, scans, odo, lattice, window, k):
    ref, vol = p.relocalize_sequence(scans, odo, *lattice, window=window, k=k, want_distances=True)
    got, st = p.relocalize_sequence_bounded(scans, odo, *lattice, window=window, k=k)
    assert _hits(got) == _hits(ref), (lattice, window, k, st)
    c = lattice[2]
    assert st["poses"] == c[0] * c[1] * c[2] and 0 <= st["evaluated"] <= st["passes"] * st["poses"]
    return vol, st


@pytest.mark.parametrize("flags", LAYOUTS, ids=LAYOUT_IDS)
@pytest.mark.parametrize("kind", ["random", "driven"])
@pytest.mark.parametrize("K", [1, 2, 5, 32])
def test_bounded_equals_exhaustive(flags, kind, K):
    rng = np.random.default_rng(K * 7 + flags + (kind == "driven"))
    if kind == "random":
        size, phys = 256, 10.0
        px = synth.random_map(size, seed=size + K).reshape(size, size)
        # unequal scans: 1 point, more than one 1024-point chunk, and sizes between
        sizes = {1: [1], 2: [1, 1500], 5: [1, 1500, 37, 5, 300]}.get(K) or list(rng.integers(1, 120, K))
        scans = [rng.normal(0, 0.2 * phys, (int(n), 2)).astype(np.float32) for n in sizes]
        odo = np.cumsum(rng.normal(0, 0.03 * phys, (K, 3)) * [1, 1, 0.3], axis=0).astype(np.float32)
        odo = _frame(odo, rot=-2.0)
    else:
        size, phys = 400, 40.0
        px, rp = _driven()
        idx = [i % 20 for i in range(20 - K, 20)] if K <= 20 else [i % 20 for i in range(K)]
        scans, odo = [rp.points[i] for i in idx], _frame(rp.odometry[idx])
        if K > 1:  # a scan of more than one 1024-point chunk
            scans[0] = np.concatenate([rp.points[j] for j in range(4)])[:1100]
    p = _handle(px, phys, flags, max_points=2048)
    cell = phys / size
    # partly off the map, and a fine patch that prunes
    lattices = [([-0.2 * phys, 0.1 * phys, -1.0], [1.3 * phys / 47, 0.9 * phys / 41, 0.45], [47, 41, 5]),
                ([0.3 * phys, 0.3 * phys, -0.4], [0.4 * cell, 0.35 * cell, 0.07], [97, 83, 3])]
    for lattice in lattices:
        for window, k in [(0, 8), (1, 1), (2, 64)]:
            _bounded_same(p, scans, odo, lattice, window, k)
    p.close()


def test_scan_off_the_map_is_int_max():
    """The oldest scan's odometry lies 30 m behind the anchor: over part of the lattice it lands off the 40 m map while
    the anchor stays on it.  Those poses are INT32_MAX in the volume, and neither call reports them."""
    px, rp = _driven()
    p = _handle(px, 40.0, 0)
    old = rp.points[3][np.hypot(rp.points[3][:, 0], rp.points[3][:, 1]) < 3.0]  # the oldest scan's points within 3 m
    scans = [old, rp.points[10]]
    odo = np.array([[-30.0, 0.0, 0.0], [0.0, 0.0, 0.0]], dtype=np.float32)
    lattice = ([2.0, 15.0, -0.2], [0.5, 0.5, 0.2], [70, 20, 3])  # x from 2 to 36.5 m: the oldest scan near x - 30
    hits, vol = p.relocalize_sequence(scans, odo, *lattice, k=64, want_distances=True)
    _, one = p.relocalize(scans[1], *lattice, want_distances=True)
    xs = lattice_axes(*lattice)[0]
    off = xs < 20.0  # the oldest scan lies at x - 29.4 or less, wholly off the map
    assert len(old) > 10 and np.all(vol[:, :, off] == INT_MAX) and np.all(one[:, :, off] < INT_MAX)
    assert np.any(vol[:, :, xs > 33.0] < INT_MAX)
    bh, _ = p.relocalize_sequence_bounded(scans, odo, *lattice, k=64)
    for h in hits + bh:
        assert not off[h.index % lattice[2][0]] and h.distance < INT_MAX
    assert _hits(bh) == _hits(hits)
    p.close()


@pytest.mark.parametrize("flags", LAYOUTS, ids=LAYOUT_IDS)
def test_saturated_map_at_full_capacity(flags):
    size, phys, n = 256, 10.0, 65536
    p = sn.Processor(phys, size, [0, 0, 0], 0.1, 0.17, 8, 1, flags=flags, max_points=n)
    p.map_fill(65535)
    rng = np.random.default_rng(1)
    scans = [rng.uniform(-1.0, 1.0, (n, 2)).astype(np.float32) for _ in range(32)]
    odo = np.cumsum(rng.normal(0, 0.05, (32, 3)), axis=0).astype(np.float32)
    lattice = ([4.5, 4.5, -0.2], [0.05, 0.05, 0.2], [3, 2, 3])
    hits, vol = p.relocalize_sequence(scans, odo, *lattice, k=64, want_distances=True)
    assert np.all(vol == 32 * 1024 * 65535) and 32 * 1024 * 65535 == 2147450880
    bh, _ = p.relocalize_sequence_bounded(scans, odo, *lattice, k=64)
    assert _hits(bh) == _hits(hits) and len(hits) == 18 and all(h.distance == 2147450880 for h in hits)
    p.close()


# ------------------------------------------------------------------------------------------------
# the aliasing corridor
# ------------------------------------------------------------------------------------------------
class NicheCorridor(synth.Room):
    """A corridor along x, closed at its left end, with identical niches in its upper wall every PERIOD metres from
    NICHE0 on.  The lidar sees RANGE metres, less than the niche period: in the periodic part one scan looks the same at
    every niche."""
    Y0, Y1, X0, X1 = 9.0, 11.0, 2.0, 19.0
    NICHE0, PERIOD, WIDTH, DEPTH, N = 8.0, 3.0, 1.0, 0.4, 4
    RANGE = 1.6

    def __init__(self, physical_size=20.0):
        self.physical_size = float(physical_size)
        segs = [((self.X0, self.Y0), (self.X1, self.Y0)), ((self.X0, self.Y0), (self.X0, self.Y1))]
        x = self.X0
        for i in range(self.N):
            a = self.NICHE0 + i * self.PERIOD
            b = a + self.WIDTH
            segs += [((x, self.Y1), (a, self.Y1)), ((a, self.Y1), (a, self.Y1 + self.DEPTH)),
                     ((a, self.Y1 + self.DEPTH), (b, self.Y1 + self.DEPTH)), ((b, self.Y1 + self.DEPTH), (b, self.Y1))]
            x = b
        segs.append(((x, self.Y1), (self.X1, self.Y1)))
        self.a = np.array([s[0] for s in segs], dtype=np.float64)
        self.b = np.array([s[1] for s in segs], dtype=np.float64)

    def cast(self, pose, angles, max_range=40.0):
        return super().cast(pose, angles, min(max_range, self.RANGE))


def corridor_drive(room, x0, step, seed, n_points=360):
    """(truth poses, scans) of a drive along the middle of the corridor from x0 towards its far end"""
    rng = np.random.default_rng(seed)
    xs = np.arange(x0, room.X1 - 1.0, step)
    truth = np.stack([xs, np.full_like(xs, 10.0), np.zeros_like(xs)], axis=1)
    return truth, [synth.lidar_scan(room, t, n_points, rng) for t in truth]


# the map: one drive at 5 cm steps; the scans to relocalise: another drive (other range noise) at 25 cm steps whose last
# scan lies just past the first niche, SEQ_K scans long, so that its oldest scans saw the plain wall before the niches
SEQ_K, SEQ_ANCHOR_X = 16, 9.6


def corridor_case():
    room = NicheCorridor()
    map_truth, map_scans = corridor_drive(room, 2.5, 0.05, 11)
    truth, scans = corridor_drive(room, SEQ_ANCHOR_X - 0.25 * (SEQ_K - 1), 0.25, 12)
    truth, scans = truth[:SEQ_K], scans[:SEQ_K]
    odo = _frame(truth, rot=1.2, shift=(-4.0, 6.5))
    cell = 20.0 / 400
    lattice = ([3.0, 9.5, -0.1], [cell, cell, np.radians(1.0)], [281, 21, 13])
    return room, map_truth, map_scans, truth, scans, odo, lattice


def test_sequence_tells_niches_apart():
    size, phys = 400, 20.0
    room, map_truth, map_scans, truth, scans, odo, lattice = corridor_case()
    p = sn.Processor(phys, size, [0, 0, 0], 0.1, 0.17, 8, 1, max_points=512)
    for t, pts in zip(map_truth, map_scans):
        p.integrate(pts, t.astype(np.float32))
    cell = phys / size
    xs = lattice_axes(*lattice)[0]
    tx = truth[-1]
    single, _ = p.relocalize(scans[-1], *lattice, window=10, k=8)
    near = lambda h, x: abs(float(h.pose[0]) - x) <= 2 * cell + 1e-6 and abs(float(h.pose[1]) - tx[1]) <= 2 * cell + 1e-6
    niches = [[h for h in single if near(h, tx[0] + i * NicheCorridor.PERIOD)] for i in range(3)]
    assert sum(1 for n in niches if n) >= 2, [(h.pose, h.distance) for h in single]
    d = sorted(n[0].distance for n in niches if n)
    assert d[1] <= 1.05 * d[0], d  # two niches within 5 %: one scan cannot tell them apart

    hits, vol = p.relocalize_sequence(scans, odo, *lattice, window=10, k=8, want_distances=True)
    best = hits[0]
    assert near(best, tx[0]) and abs(float(best.pose[2]) - tx[2]) <= 2 * np.radians(1.0) + 1e-6, (best.pose, tx)
    # the best sequence distance around the next niche's hypothesis
    other = int(vol[:, :, np.abs(xs - (tx[0] + NicheCorridor.PERIOD)) <= 3 * cell].min())
    assert other > 1.25 * best.distance, (best.distance, other)
    bh, _ = p.relocalize_sequence_bounded(scans, odo, *lattice, window=10, k=8)
    assert _hits(bh) == _hits(hits)
    p.close()


@pytest.mark.parametrize("production", [False, True])
def test_no_state_change(production):
    px, rp = _driven(400, 40.0, 20, 360)
    iters, threads = 64, 4

    def run(with_calls):
        p = sn.Processor(40.0, 400, rp.odometry[0], 0.1, 0.17, iters, threads, max_points=360, seed=5)
        poses, dists = [], []
        for k in range(12):
            off = None if production else synth.candidate_offsets(1, k, iters * threads, 0.1, 0.17)
            r = p.update(rp.points[k], rp.odometry[k], off)
            poses.append(r.pose.tobytes())
            dists.append(r.distance)
            if with_calls and k >= 2:
                scans, odo = [rp.points[i] for i in range(k - 2, k + 1)], rp.odometry[k - 2:k + 1]
                lat = ([r.pose[0] - 0.5, r.pose[1] - 0.5, r.pose[2] - 0.1], [0.05, 0.05, 0.02], [21, 21, 11])
                p.relocalize_sequence(scans, odo, *lat, window=1, k=4, want_distances=True)
                p.relocalize_sequence_bounded(scans, odo, *lat, window=1, k=4)
        m = p.map_download()
        p.close()
        return poses, dists, m

    a, b = run(False), run(True)
    assert a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2], b[2])


def test_errors_and_scratch_reuse():
    px, rp = _driven()
    p = _handle(px, 40.0, 0, max_points=400)
    scans, odo = _drive_sequence(rp, 12, 3)
    lat = _lattices(40.0, 400)[0]
    pts = np.concatenate(scans)
    first = np.array([0, len(scans[0]), len(scans[0]) + len(scans[1]), len(pts)], dtype=np.int32)
    L = N.lib()
    hits = (N.LatticeHit * N.LATTICE_MAX_HITS)()
    n = N.C.c_int32()
    latc = p._lattice(*lat)
    ip = lambda a: None if a is None else a.ctypes.data_as(N.C.POINTER(N.C.c_int32))
    fp = lambda a: None if a is None else a.ctypes.data_as(N.C.POINTER(N.C.c_float))
    bad_odo = odo.copy()
    bad_odo[1, 2] = np.nan
    first_bad = first.copy()
    first_bad[0] = 1
    first_empty = first.copy()
    first_empty[2] = first_empty[1]
    big = [np.zeros((401, 2), np.float32)]
    cases = [  # (points, first, odometry, n_scans, k, expected)
        (pts, None, odo, 3, 4, 1), (pts, first, None, 3, 4, 1), (pts, first, odo, 0, 4, 1), (pts, first, odo, 33, 4, 1),
        (pts, first_bad, odo, 3, 4, 1), (pts, first_empty, odo, 3, 4, 1), (pts, first, bad_odo, 3, 4, 1),
        (pts, first, odo, 3, 0, 1), (big[0], np.array([0, 401], np.int32), odo[:1], 1, 4, 5)]
    for q, f, o, ns, k, want in cases:
        for fn in (L.cs_relocalize_sequence, L.cs_relocalize_sequence_bounded):
            st = fn(p._h, fp(q), ip(f), fp(o), ns, N.C.byref(latc), 0, k, hits, N.C.byref(n), None)
            assert st == want, (ns, k, st)
    too_many = p._lattice([0, 0, 0], [0.1, 0.1, 0.1], [1 << 10, 1 << 10, 1 << 9])
    assert L.cs_relocalize_sequence(p._h, fp(pts), ip(first), fp(odo), 3, N.C.byref(too_many), 0, 4, hits, N.C.byref(n), None) == 5
    # the handle stays usable, and interleaved calls with different K and lattices match fresh handles
    runs = [(scans, odo, lat), (scans[:1], odo[:1], _lattices(40.0, 400)[1]), (scans[1:], odo[1:], _lattices(40.0, 400)[2])]
    got = []
    for s, o, lt in runs * 2:
        got.append((_hits(p.relocalize_sequence(s, o, *lt, window=1, k=8)[0]), _hits(p.relocalize_sequence_bounded(s, o, *lt, window=1, k=8)[0])))
    p.close()
    for i, (s, o, lt) in enumerate(runs):
        q = _handle(px, 40.0, 0, max_points=400)
        want = (_hits(q.relocalize_sequence(s, o, *lt, window=1, k=8)[0]), _hits(q.relocalize_sequence_bounded(s, o, *lt, window=1, k=8)[0]))
        q.close()
        assert got[i] == want and got[i + len(runs)] == want
