"""cs_relocalize_sequence without a GPU: the exports in the header, ctypes and C#, CS_SEQUENCE_MAX_SCANS in all three, the
odometry composition of sequence_ref against a scalar restatement, sequence_volume against the oracle pose by pose, and
the bound lemma the bounded call rests on, for sequences: the sum of the scans' node bounds is <= the sequence distance
of every pose of the node."""
import os
import re

import numpy as np
import pytest

from slam.net_b200 import _native as N
from relocalize_ref import INT_MAX, lattice_axes
import sequence_ref as sr
from test_relocalize_bounded_abi import _grids, _maps

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32


def _read(*parts):
    return open(os.path.join(ROOT, *parts)).read()


def test_exports_and_constant_agree_between_header_python_and_csharp():
    hdr = _read("include", "coreslam_b200.h")
    cs = _read("dotnet", "CoreSlamNative.cs")
    for name in ("cs_relocalize_sequence", "cs_relocalize_sequence_bounded"):
        assert re.search(r"cs_status %s\(" % name, hdr)
        assert name in N.SIGNATURES
        assert re.search(r"\[DllImport\(Lib\)\] public static extern CsStatus %s\(" % name, cs)
    assert int(re.search(r"#define CS_SEQUENCE_MAX_SCANS (\d+)", hdr).group(1)) == N.SEQUENCE_MAX_SCANS == 32
    assert int(re.search(r"SequenceMaxScans = (\d+);", cs).group(1)) == 32
    assert int(re.search(r"#define CS_LAT_SEQ_MAX (\d+)", _read("slam.net_b200", "csrc", "cs_lattice.cuh")).group(1)) == 32
    b200 = _read("dotnet", "CoreSLAMProcessor.B200.cs")
    assert "RelocalizeSequence(Vector2[][] scans, Vector3[] odometry" in b200 and "RelocalizeSequenceBounded(" in b200
    py = _read("slam.net_b200", "coreslam.py")
    for name in ("def relocalize_sequence(", "def relocalize_sequence_bounded(", "def RelocalizeSequence(",
                 "def RelocalizeSequenceBounded("):
        assert name in py


def _scalar_offsets(odometry):
    """sequence_ref.offsets one np.float32 operation at a time"""
    o = [[f32(v) for v in row] for row in np.asarray(odometry, dtype=np.float32)]
    a = o[-1]
    ca, sa = (f32(v[0]) for v in sr._sincos(a[2]))
    out = []
    for x, y, t in o:
        ex = f32(x - a[0])
        ey = f32(y - a[1])
        p = f32(ca * ex)
        q = f32(sa * ey)
        dx = f32(p + q)
        p = f32(ca * ey)
        q = f32(sa * ex)
        dy = f32(p - q)
        out.append((dx, dy, f32(t - a[2])))
    return out


def _scalar_pose(pose, d):
    x, y, t = (f32(v) for v in pose)
    c, s = (f32(v[0]) for v in sr._sincos(t))
    dx, dy, dth = d
    ox = f32(f32(c * dx) - f32(s * dy))
    oy = f32(f32(s * dx) + f32(c * dy))
    return f32(x + ox), f32(y + oy), f32(t + dth)


@pytest.mark.parametrize("rot", [np.pi, -np.pi, np.pi / 2, -np.pi / 2, 1e3, 0.0, 1.2])
@pytest.mark.parametrize("shift", [0.0, 1e3, -3e4])
def test_composition_matches_a_scalar_restatement(rot, shift):
    rng = np.random.default_rng(int(abs(rot) * 100 + abs(shift)))
    k = 7
    # a drive in the map frame, then expressed in an odometry frame rotated by rot and shifted by shift
    steps = rng.normal(0, 0.3, (k, 3)) * [1, 1, 0.3]
    path = np.cumsum(steps, axis=0)
    c, s = np.cos(rot), np.sin(rot)
    odo = np.stack([c * path[:, 0] - s * path[:, 1] + shift, s * path[:, 0] + c * path[:, 1] - 0.5 * shift, path[:, 2] + rot], axis=1)
    odo = odo.astype(np.float32)
    dx, dy, dth = sr.offsets(odo)
    ref = _scalar_offsets(odo)
    for i in range(k):
        for got, want in zip((dx[i], dy[i], dth[i]), ref[i]):
            assert np.float32(got).tobytes() == np.float32(want).tobytes()
    # the anchor: ex = ey = dtheta = +0, so its dx and dy are zeros (of either sign)
    assert dth[-1].tobytes() == np.float32(0).tobytes() and dx[-1] == 0 and dy[-1] == 0
    for pose in ([3.25, -1.5, 0.7], [1e3, 2e3, -1e3], [0.0, 0.0, np.pi]):
        for i in range(k):
            got = sr.scan_pose(pose, odo, i)
            want = _scalar_pose(pose, ref[i])
            assert got.tobytes() == np.array(want, dtype=np.float32).tobytes()
        # the anchor sits at the lattice pose (up to the sign of a zero)
        assert np.array_equal(sr.scan_pose(pose, odo, k - 1), np.asarray(pose, dtype=np.float32))


def _sequence(kind, size, phys, k, seed):
    """k scans and odometry poses near the middle of the map (odometry in a rotated, shifted frame)"""
    from slam.net_b200 import synth
    rng = np.random.default_rng(seed)
    if kind == "driven":
        rp = synth.make_replay(12, 180, phys)
        scans = [rp.points[i] for i in range(12 - k, 12)]
        odo = np.asarray(rp.odometry[12 - k:12], dtype=np.float32)
    else:
        scans = [rng.normal(0, 0.15 * phys, (int(rng.integers(1, 30)), 2)).astype(np.float32) for _ in range(k)]
        odo = np.cumsum(rng.normal(0, 0.05 * phys, (k, 3)) * [1, 1, 0.5], axis=0).astype(np.float32)
    rot, sh = 1.2, np.float32(7.5)
    c, s = np.cos(rot), np.sin(rot)
    odo = np.stack([c * odo[:, 0] - s * odo[:, 1] + sh, s * odo[:, 0] + c * odo[:, 1] - sh, odo[:, 2] + rot], axis=1).astype(np.float32)
    return scans, odo


@pytest.mark.parametrize("kind,size,phys", [("random", 96, 6.0), ("driven", 160, 40.0)])
@pytest.mark.parametrize("k", [1, 3])
def test_sequence_volume_is_the_sum_of_oracle_distances(kind, size, phys, k):
    from oracle import oracle as orc
    px = _maps(kind, size, phys)
    m = orc.HoleMap(size, phys)
    m.pixels[:] = px.ravel()
    scans, odo = _sequence(kind, size, phys, k, size + k)
    cell = phys / size
    for origin, step, count in [([0.3 * phys, 0.35 * phys, -4.0], [2.5 * cell, 2.0 * cell, 1.7], [5, 4, 5]),
                                ([-0.3 * phys, 0.6 * phys, 1.0], [0.3 * phys, 0.25 * phys, 0.9], [6, 5, 3])]:
        vol = sr.sequence_volume(px, size, m.scale, scans, odo, origin, step, count)
        xs, ys, ts = lattice_axes(origin, step, count)
        for it, t in enumerate(ts):
            for iy, y in enumerate(ys):
                for ix, x in enumerate(xs):
                    ds = [orc.distance(m, scans[i], sr.scan_pose([x, y, t], odo, i)) for i in range(k)]
                    want = INT_MAX if INT_MAX in ds else sum(ds)
                    assert vol[it, iy, ix] == want, (it, iy, ix, ds)
        if k == 1:
            from relocalize_ref import numpy_volume
            assert np.array_equal(vol, numpy_volume(px, size, m.scale, scans[0], origin, step, count))


def _seq_node_bound(grids, size, scans, odo, scale, origin, step, it, x0, x1, y0, y1):
    """sum over the scans of _node_bound's term, each scan's cells at its own offset and heading; INT_MAX when some scan
    lies wholly off the map at every pose of the node"""
    theta = f32(f32(origin[2]) + f32(f32(it) * f32(step[2])))
    dx, dy, dth = sr.offsets(odo)
    ox, oy = sr.scan_offsets_at(theta, dx, dy)
    scale = f32(scale)
    total = 0
    for k, pts in enumerate(scans):
        tk = f32(theta + dth[k])
        ck, sk = (f32(v[0]) for v in sr._sincos(tk))
        c, s = f32(ck * scale), f32(sk * scale)
        X, Y = pts[:, 0], pts[:, 1]
        cx, sy, sx, cy = (c * X).astype(f32), (s * Y).astype(f32), (s * X).astype(f32), (c * Y).astype(f32)

        def cells(axis, i, first, second, sign):
            coord = f32(f32(origin[axis]) + f32(f32(i) * f32(step[axis])))
            pp = f32(f32(f32(coord + (ox[k] if axis == 0 else oy[k])) * scale) + f32(0.5))
            v = (pp + first).astype(f32)
            v = (v - second if sign < 0 else v + second).astype(f32)
            return np.trunc(np.maximum(v, f32(-2.0))).astype(np.int64)

        xl, xh = cells(0, x0, cx, sy, -1), cells(0, x1, cx, sy, -1)
        yl, yh = cells(1, y0, sx, cy, +1), cells(1, y1, sx, cy, +1)
        off = (xh < 0) | (xl >= size) | (yh < 0) | (yl >= size)
        if off.all():
            return INT_MAX
        inside = (xl >= 0) & (xh < size) & (yl >= 0) & (yh < size)
        span = np.maximum(xh - xl, yh - yl)
        j = np.where(span > 0, np.ceil(np.log2(span + 1.0)).astype(np.int64), 0)
        t = 0
        for i in np.flatnonzero(inside & (j < len(grids))):
            t += int(grids[j[i]][yl[i], xl[i]])
        total += t * 1024 // len(pts)
    return total


@pytest.mark.parametrize("kind,size,phys", [("random", 96, 6.0), ("driven", 160, 40.0)])
@pytest.mark.parametrize("block", [3, 8])
def test_sequence_node_bound_is_below_every_pose_of_the_node(kind, size, phys, block):
    from oracle import oracle as orc
    px = _maps(kind, size, phys)
    m = orc.HoleMap(size, phys)
    m.pixels[:] = px.ravel()
    scans, odo = _sequence(kind, size, phys, 3, size * 7 + block)
    # one scan's odometry far from the anchor: at some poses it lies off the map while the anchor stays on it
    odo = odo.copy()
    odo[0, :2] += np.float32(0.45 * phys)
    cell = phys / size
    grids = _grids(px, 6)
    seen_off, seen_bound = False, False
    for origin, step, count in [([-0.5 * phys, -0.5 * phys, -5.0], [2.0 * phys / 19, 2.0 * phys / 17, 2.5], [19, 17, 5]),
                                ([0.4 * phys, 0.45 * phys, 3.0], [0.35 * cell, 0.3 * cell, 0.4], [19, 17, 3])]:
        vol = sr.sequence_volume(px, size, m.scale, scans, odo, origin, step, count)
        for it in range(count[2]):
            for y0 in range(0, count[1], block):
                for x0 in range(0, count[0], block):
                    x1, y1 = min(x0 + block, count[0]) - 1, min(y0 + block, count[1]) - 1
                    b = _seq_node_bound(grids, size, scans, odo, m.scale, origin, step, it, x0, x1, y0, y1)
                    low = int(vol[it, y0:y1 + 1, x0:x1 + 1].min())
                    assert b <= low, (origin, it, x0, y0, b, low)
                    seen_off |= b == INT_MAX
                    seen_bound |= 0 < b < INT_MAX
    assert seen_off and seen_bound
