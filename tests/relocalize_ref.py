"""Reference side of the cs_relocalize tests: lattice poses and distance volumes from the CPU oracle (one call per pose,
or numpy_volume, the same function vectorised for large lattices and scans), and the selection (window minima of
(distance, flat index), best first) in numpy.  Host-side only; the oracle is imported lazily so the selection can be
tested without building it."""
import numpy as np

INT_MAX = 2147483647


def lattice_axes(origin, step, count):
    """The coordinates of the lattice along x, y, theta: origin + (float)i * step in float32, one rounding per
    operation (an axis with one point is its origin)."""
    axes = []
    for o, s, c in zip(origin, step, count):
        i = np.arange(int(c), dtype=np.float32)
        s = np.float32(s) if int(c) > 1 else np.float32(0.0)
        axes.append((np.float32(o) + i * s).astype(np.float32))
    return axes


def lattice_pose(origin, step, count, index):
    xs, ys, ts = lattice_axes(origin, step, count)
    c0, c1 = int(count[0]), int(count[1])
    return np.array([xs[index % c0], ys[index // c0 % c1], ts[index // (c0 * c1)]], dtype=np.float32)


def oracle_volume(hole_map, points, origin, step, count):
    """oracle.distance (CalculateDistanceSISD) at every lattice pose -> (count[2], count[1], count[0]) int32."""
    from oracle import oracle as orc
    xs, ys, ts = lattice_axes(origin, step, count)
    vol = np.empty((len(ts), len(ys), len(xs)), dtype=np.int32)
    for it, t in enumerate(ts):
        for iy, y in enumerate(ys):
            for ix, x in enumerate(xs):
                vol[it, iy, ix] = orc.distance(hole_map, points, np.array([x, y, t], dtype=np.float32))
    return vol


def numpy_volume(pixels, size, scale, points, origin, step, count, chunk=1 << 23):
    """oracle_volume in vectorised float32 numpy: the reference's distance (CalculateDistanceSISD) at every lattice pose
    -> (count[2], count[1], count[0]) int32.  Every operation is one f32 rounding in the reference's order (numpy does
    not contract a*b + c); cos/sin come from the oracle's libm.  The cell test is the (int) cast of cvttss2si: in bounds
    exactly when -1 < v < size (NaN fails both comparisons; (-1, 0) truncates to cell 0).  Poses are taken a block of
    rows at a time, about `chunk` lookups per block."""
    from oracle import oracle as orc
    f32 = np.float32
    pix = np.append(np.asarray(pixels, dtype=np.int64).ravel(), 0)  # one zero cell past the map for the off-map points
    off_map = size * size
    scale = f32(scale)
    pts = np.asarray(points, dtype=np.float32).reshape(-1, 2)
    n = pts.shape[0]
    X, Y = pts[:, 0], pts[:, 1]
    xs, ys, ts = lattice_axes(origin, step, count)
    cth, sth = orc.libm_sincos(ts)
    px = (xs * scale + f32(0.5)).astype(np.float32)  # :232, two roundings
    py = (ys * scale + f32(0.5)).astype(np.float32)  # :233
    vol = np.empty((len(ts), len(ys), len(xs)), dtype=np.int32)
    rows = max(1, chunk // max(1, len(xs) * n))
    with np.errstate(invalid="ignore", over="ignore"):
        for it in range(len(ts)):
            c, s = f32(cth[it] * scale), f32(sth[it] * scale)  # :234-235
            cx, sy, sx, cy = c * X, s * Y, s * X, c * Y
            vx = (px[:, None] + cx[None, :]) - sy[None, :]  # :240, (nx, n)
            vy = (py[:, None] + sx[None, :]) + cy[None, :]  # :241, (ny, n)
            inx = (vx > -1) & (vx < size)
            iny = (vy > -1) & (vy < size)
            cellx = np.where(inx, np.trunc(np.where(inx, vx, 0)), 0).astype(np.int64)
            rowy = np.where(iny, np.trunc(np.where(iny, vy, 0)), 0).astype(np.int64) * size
            for y0 in range(0, len(ys), rows):
                y1 = min(y0 + rows, len(ys))
                ok = iny[y0:y1, None, :] & inx[None, :, :]  # (rows, nx, n)
                idx = np.where(ok, rowy[y0:y1, None, :] + cellx[None, :, :], off_map)
                total = pix[idx].sum(axis=2)
                d = (total * 1024) // n  # :253, divided by every point
                vol[it, y0:y1] = np.where(ok.any(axis=2), d, INT_MAX)
    return vol


def reference_hits(vol, window, k):
    """[(distance, flat index)] of at most k poses whose distance is < INT_MAX and whose key (distance, flat index) is
    below the key of every other pose within +-window steps on each axis (box clipped at the edges), ascending.
    Exact integer work throughout: the box minimum of the int32 distances first, then the ties at a lower flat index."""
    vol = np.ascontiguousarray(vol, dtype=np.int32)
    ok = vol < INT_MAX
    if window > 0:
        from scipy import ndimage
        ok &= vol == ndimage.minimum_filter(vol, size=2 * window + 1, mode="constant", cval=INT_MAX)
    if window > 2:
        # the offset loop below takes (2 window + 1)^3 passes: for wide boxes take the box minimum of the keys instead.
        # ndimage filters in double, so the key is (rank of the distance, flat index), kept below 2^53 to stay exact
        values, rank = np.unique(vol, return_inverse=True)
        n = vol.size
        assert len(values) * n < 1 << 53
        key = rank.reshape(vol.shape).astype(np.int64) * n + np.arange(n, dtype=np.int64).reshape(vol.shape)
        ok &= key == ndimage.minimum_filter(key, size=2 * window + 1, mode="constant", cval=len(values) * n)
        window = 0
    cand = np.flatnonzero(ok)
    d = vol.ravel()[cand]
    if window > 0 and cand.size:
        # an equal distance in the box at a lower flat index, i.e. at an offset (dt, dy, dx) below (0, 0, 0)
        c2, c1, c0 = vol.shape
        it, iy, ix = np.unravel_index(cand, vol.shape)
        tied = np.zeros(cand.size, dtype=bool)
        r = range(-window, window + 1)
        for dt in r:
            for dy in r:
                for dx in r:
                    if (dt, dy, dx) >= (0, 0, 0):
                        continue
                    t, y, x = it + dt, iy + dy, ix + dx
                    inb = (t >= 0) & (t < c2) & (y >= 0) & (y < c1) & (x >= 0) & (x < c0)
                    tied[inb] |= vol[t[inb], y[inb], x[inb]] == d[inb]
        cand, d = cand[~tied], d[~tied]
    key = (d.astype(np.int64) << 32) | cand.astype(np.int64)
    if key.size > k:
        key = np.partition(key, k - 1)[:k]
    return [(int(v >> 32), int(v & 0xFFFFFFFF)) for v in np.sort(key)]


def brute_force_hits(vol, window, k):
    """reference_hits by the definition, pose by pose (small volumes only)."""
    vol = np.asarray(vol)
    c2, c1, c0 = vol.shape
    out = []
    for it in range(c2):
        for iy in range(c1):
            for ix in range(c0):
                d = int(vol[it, iy, ix])
                if d == INT_MAX:
                    continue
                idx = (it * c1 + iy) * c0 + ix
                best = True
                for t in range(max(it - window, 0), min(it + window, c2 - 1) + 1):
                    for y in range(max(iy - window, 0), min(iy + window, c1 - 1) + 1):
                        for x in range(max(ix - window, 0), min(ix + window, c0 - 1) + 1):
                            n = (t * c1 + y) * c0 + x
                            if n != idx and (int(vol[t, y, x]), n) < (d, idx):
                                best = False
                if best:
                    out.append((d, idx))
    return sorted(out)[:k]
