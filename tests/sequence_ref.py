"""Reference side of the cs_relocalize_sequence tests: the odometry composition of include/coreslam_b200.h in float32 numpy
(one rounding per operation, cos/sin from the oracle's libm) and the distance volume of a scan sequence, the sum of the
scans' CalculateDistanceSISD terms with the INT32_MAX rule.  Host-side only."""
import numpy as np

from relocalize_ref import INT_MAX, lattice_axes

f32 = np.float32


def _sincos(theta):
    from oracle import oracle as orc
    c, s = orc.libm_sincos(np.asarray(theta, dtype=np.float32).reshape(-1))
    return np.asarray(c, dtype=np.float32), np.asarray(s, dtype=np.float32)


def offsets(odometry):
    """(K, 3) odometry -> (dx, dy, dtheta) of every scan relative to the last (the anchor), each (K,) float32:
    e = o - a, dx = ca*ex + sa*ey, dy = ca*ey - sa*ex, dtheta = o.theta - a.theta."""
    o = np.asarray(odometry, dtype=np.float32).reshape(-1, 3)
    a = o[-1]
    ca, sa = (v[0] for v in _sincos(a[2]))
    ex, ey = o[:, 0] - a[0], o[:, 1] - a[1]
    dx = (ca * ex) + (sa * ey)
    dy = (ca * ey) - (sa * ex)
    return dx.astype(f32), dy.astype(f32), (o[:, 2] - a[2]).astype(f32)


def scan_offsets_at(theta, dx, dy):
    """the offsets (ox, oy) the scans add to the lattice x, y at heading theta (c, s = cosf, sinf(theta), unscaled):
    ox = c*dx - s*dy, oy = s*dx + c*dy"""
    c, s = (v[0] for v in _sincos(theta))
    return ((c * dx) - (s * dy)).astype(f32), ((s * dx) + (c * dy)).astype(f32)


def scan_pose(pose, odometry, k):
    """the absolute pose of scan k when the last scan is at `pose`, one float32 rounding per operation"""
    dx, dy, dth = offsets(odometry)
    x, y, t = (f32(v) for v in pose)
    ox, oy = scan_offsets_at(t, dx[k:k + 1], dy[k:k + 1])
    return np.array([x + ox[0], y + oy[0], t + dth[k]], dtype=np.float32)


def axes_volume(pixels, size, scale, points, xs, ys, t, chunk=1 << 23):
    """The reference's distance (CalculateDistanceSISD) of one scan at every pose (xs[ix], ys[iy], t) -> (len(ys), len(xs))
    int32; relocalize_ref.numpy_volume's arithmetic on explicit axes."""
    pix = np.append(np.asarray(pixels, dtype=np.int64).ravel(), 0)
    off_map = size * size
    scale = f32(scale)
    pts = np.asarray(points, dtype=np.float32).reshape(-1, 2)
    n = pts.shape[0]
    X, Y = pts[:, 0], pts[:, 1]
    cth, sth = _sincos(t)
    px = (np.asarray(xs, np.float32) * scale + f32(0.5)).astype(np.float32)
    py = (np.asarray(ys, np.float32) * scale + f32(0.5)).astype(np.float32)
    out = np.empty((len(py), len(px)), dtype=np.int32)
    rows = max(1, chunk // max(1, len(px) * n))
    with np.errstate(invalid="ignore", over="ignore"):
        c, s = f32(cth[0] * scale), f32(sth[0] * scale)
        cx, sy, sx, cy = c * X, s * Y, s * X, c * Y
        vx = (px[:, None] + cx[None, :]) - sy[None, :]
        vy = (py[:, None] + sx[None, :]) + cy[None, :]
        inx = (vx > -1) & (vx < size)
        iny = (vy > -1) & (vy < size)
        cellx = np.where(inx, np.trunc(np.where(inx, vx, 0)), 0).astype(np.int64)
        rowy = np.where(iny, np.trunc(np.where(iny, vy, 0)), 0).astype(np.int64) * size
        for y0 in range(0, len(py), rows):
            y1 = min(y0 + rows, len(py))
            ok = iny[y0:y1, None, :] & inx[None, :, :]
            idx = np.where(ok, rowy[y0:y1, None, :] + cellx[None, :, :], off_map)
            d = (pix[idx].sum(axis=2) * 1024) // n
            out[y0:y1] = np.where(ok.any(axis=2), d, INT_MAX)
    return out


def sequence_volume(pixels, size, scale, scans, odometry, origin, step, count):
    """The distance volume of a scan sequence -> (count[2], count[1], count[0]) int32: at every lattice pose the sum over
    the scans of each scan's distance at its composed pose, INT_MAX when any scan's is INT_MAX."""
    xs, ys, ts = lattice_axes(origin, step, count)
    dx, dy, dth = offsets(odometry)
    vol = np.empty((len(ts), len(ys), len(xs)), dtype=np.int64)
    for it, t in enumerate(ts):
        ox, oy = scan_offsets_at(t, dx, dy)
        total = np.zeros((len(ys), len(xs)), dtype=np.int64)
        off = np.zeros((len(ys), len(xs)), dtype=bool)
        for k, pts in enumerate(scans):
            d = axes_volume(pixels, size, scale, pts, (xs + ox[k]).astype(f32), (ys + oy[k]).astype(f32), f32(t + dth[k]))
            off |= d == INT_MAX
            total += d
        vol[it] = np.where(off, INT_MAX, total)
    assert vol.max() <= INT_MAX
    return vol.astype(np.int32)
