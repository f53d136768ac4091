"""cs_relocalize_bounded without a GPU: the layout of cs_relocalize_stats in the header, ctypes and C#, the new constants,
and the lemma the branch and bound rests on, in numpy against the CPU oracle: the bound of a block of poses of one
heading (DESIGN section 4) is <= the oracle's distance (CalculateDistanceSISD) of every pose of the block."""
import ctypes
import os
import re

import numpy as np
import pytest

from slam.net_b200 import _native as N
from relocalize_ref import INT_MAX, lattice_axes, oracle_volume

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _read(*parts):
    return open(os.path.join(ROOT, *parts)).read()


def test_stats_layout_and_constants():
    assert ctypes.sizeof(N.RelocalizeStats) == 40
    offsets = {name: getattr(N.RelocalizeStats, name).offset for name, _ in N.RelocalizeStats._fields_}
    assert offsets == {"poses": 0, "evaluated": 8, "bounded": 16, "levels": 24, "passes": 28, "upper_bound": 32, "reserved": 36}
    hdr = _read("include", "coreslam_b200.h")
    assert int(re.search(r"#define CS_LATTICE_MAX_POSES_BOUNDED (\d+)", hdr).group(1)) == N.LATTICE_MAX_POSES_BOUNDED == 2 ** 31 - 1
    assert eval(re.search(r"#define CS_LATTICE_BOUNDED_MAX_NODES (\(1 << \d+\))", hdr).group(1)) == N.LATTICE_BOUNDED_MAX_NODES
    cs = _read("dotnet", "CoreSlamNative.cs")
    assert re.search(r"LatticeMaxPosesBounded = 2147483647;", cs)
    assert re.search(r"LatticeBoundedMaxNodes = 1 << 20;", cs)


def test_stats_field_lists_agree_between_header_python_and_csharp():
    hdr = _read("include", "coreslam_b200.h")
    body = re.search(r"typedef struct cs_relocalize_stats \{(.*?)\} cs_relocalize_stats;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    c = [(m.group(1), m.group(2)) for m in re.finditer(r"(int64_t|int32_t)\s+(\w+)\s*;", body)]
    types = {"int64_t": ctypes.c_int64, "int32_t": ctypes.c_int32}
    assert [(n, types[t]) for t, n in c] == list(N.RelocalizeStats._fields_)
    cs = _read("dotnet", "CoreSlamNative.cs")
    body = cs[cs.index("public struct CsRelocalizeStats "):]
    body = re.sub(r"//[^\n]*", "", body[body.index("{") + 1:body.index("}")])
    fields = [(m.group(1), m.group(2)) for m in re.finditer(r"public\s+(long|int)\s+(\w+)\s*;", body)]
    kinds = {"int64_t": "long", "int32_t": "int"}
    assert [(kinds[t], n.replace("_", "")) for t, n in c] == [(t, n.lower()) for t, n in fields]


def test_csharp_stub_and_wrapper_present():
    cs = _read("dotnet", "CoreSlamNative.cs")
    assert re.search(r"\[DllImport\(Lib\)\] public static extern CsStatus cs_relocalize_bounded\(", cs)
    assert "RelocalizeBounded(" in _read("dotnet", "CoreSLAMProcessor.B200.cs")
    assert "def relocalize_bounded(" in _read("slam.net_b200", "coreslam.py")
    assert "def RelocalizeBounded(" in _read("slam.net_b200", "coreslam.py")


# ------------------------------------------------------------------------------------------------
# the bound lemma, in numpy with the oracle's f32 arithmetic
# ------------------------------------------------------------------------------------------------
def _grids(px, n):
    """G_j[y][x] = min of the map over [x, x+2^j) x [y, y+2^j) clipped to the map, j = 0..n."""
    g = [px.astype(np.int64)]
    size = px.shape[0]
    for j in range(1, n + 1):
        h = 1 << (j - 1)
        a = g[-1].copy()
        a[:, :size - h] = np.minimum(a[:, :size - h], g[-1][:, h:])
        b = a.copy()
        b[:size - h, :] = np.minimum(a[:size - h, :], a[h:, :])
        g.append(b)
    return g


def _cells(p, origin, step, i, scale, first, second, sign):
    """x (or y) of every point at lattice index i: (int)((p + first) -/+ second), the device's rounding order."""
    f32 = np.float32
    coord = f32(f32(origin) + f32(f32(i) * f32(step)))
    pp = f32(f32(coord * scale) + f32(0.5))
    v = (pp + first).astype(np.float32)
    v = (v - second if sign < 0 else v + second).astype(np.float32)
    return np.trunc(np.maximum(v, f32(-2.0))).astype(np.int64)


def _node_bound(grids, size, pts, scale, origin, step, it, x0, x1, y0, y1):
    from oracle import oracle as orc
    f32 = np.float32
    theta = f32(f32(origin[2]) + f32(f32(it) * f32(step[2])))
    cth, sth = orc.libm_sincos(np.array([theta], dtype=np.float32))
    c, s = f32(cth[0] * scale), f32(sth[0] * scale)
    X, Y = pts[:, 0], pts[:, 1]
    cx, sy, sx, cy = (c * X).astype(f32), (s * Y).astype(f32), (s * X).astype(f32), (c * Y).astype(f32)
    xl, xh = (_cells(pts, origin[0], step[0], i, scale, cx, sy, -1) for i in (x0, x1))
    yl, yh = (_cells(pts, origin[1], step[1], i, scale, sx, cy, +1) for i in (y0, y1))
    off = (xh < 0) | (xl >= size) | (yh < 0) | (yl >= size)
    inside = (xl >= 0) & (xh < size) & (yl >= 0) & (yh < size)
    if off.all():
        return INT_MAX
    span = np.maximum(xh - xl, yh - yl)
    j = np.where(span > 0, np.ceil(np.log2(span + 1.0)).astype(np.int64), 0)
    total = 0
    for i in np.flatnonzero(inside & (j < len(grids))):
        total += int(grids[j[i]][yl[i], xl[i]])
    return total * 1024 // len(pts)


def _maps(kind, size, phys):
    from oracle import oracle as orc
    from slam.net_b200 import synth
    if kind == "random":
        return synth.random_map(size, seed=size).reshape(size, size)
    rp = synth.make_replay(12, 180, phys)
    m = orc.HoleMap(size, phys)
    m.fill(32750)
    for k in range(12):
        orc.update_hole_map(m, rp.points[k], rp.odometry[k], 0.6, 50)
    return np.array(m.pixels, dtype=np.uint16).reshape(size, size)


@pytest.mark.parametrize("kind,size,phys,n_points", [("random", 96, 6.0, 23), ("driven", 160, 40.0, 180)])
@pytest.mark.parametrize("block", [3, 4, 7, 8, 16])
def test_node_bound_is_below_every_pose_of_the_node(kind, size, phys, n_points, block):
    from oracle import oracle as orc
    px = _maps(kind, size, phys)
    m = orc.HoleMap(size, phys)
    m.pixels[:] = px.ravel()
    scale = np.float32(m.scale)
    rng = np.random.default_rng(size * 31 + block)
    pts = rng.normal(0, 0.15 * phys, (n_points, 2)).astype(np.float32)
    cell = phys / size
    lattices = [
        # x and y from -70 % to 170 % of the map (nodes partly and wholly off it), headings from -5 to +5 rad
        ([-0.7 * phys, -0.7 * phys, -5.0], [2.4 * phys / 37, 2.4 * phys / 33, 2.5], [37, 33, 5]),
        # about a third of a cell per step in the middle of the map: bounds that prune
        ([0.4 * phys, 0.45 * phys, 3.0], [0.35 * cell, 0.3 * cell, 0.4], [37, 33, 3]),
    ]
    grids = _grids(px, 6)
    seen_off, seen_bound = False, False
    for origin, step, count in lattices:
        vol = oracle_volume(m, pts, origin, step, count)
        assert len(lattice_axes(origin, step, count)[2]) == count[2]
        for it in range(count[2]):
            for y0 in range(0, count[1], block):
                for x0 in range(0, count[0], block):
                    x1, y1 = min(x0 + block, count[0]) - 1, min(y0 + block, count[1]) - 1
                    b = _node_bound(grids, size, pts, scale, origin, step, it, x0, x1, y0, y1)
                    low = int(vol[it, y0:y1 + 1, x0:x1 + 1].min())
                    assert b <= low, (origin, it, x0, y0, b, low)
                    seen_off |= b == INT_MAX
                    seen_bound |= 0 < b < INT_MAX
    assert seen_off and seen_bound  # nodes wholly off the map, and nodes with a bound that prunes something
