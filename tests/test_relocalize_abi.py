"""cs_relocalize without a GPU: the struct layouts of the ctypes and C# mirrors, the C# stubs, and the reference
selection the GPU tests compare against (tests/relocalize_ref.py) on hand-made volumes."""
import ctypes
import os
import re

import numpy as np
import pytest

from slam.net_b200 import _native as N
from relocalize_ref import INT_MAX, brute_force_hits, lattice_axes, lattice_pose, reference_hits

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _read(*parts):
    return open(os.path.join(ROOT, *parts)).read()


def _c_struct_fields(text, name):
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return [(m.group(1), m.group(2), int(m.group(3) or 1))
            for m in re.finditer(r"(float|int32_t)\s+(\w+)(?:\[(\d+)\])?\s*;", body)]


def _cs_struct_fields(text, name):
    body = text[text.index("public unsafe struct %s " % name):]
    body = body[body.index("{") + 1:body.index("}")]
    body = re.sub(r"//[^\n]*", "", body)
    return [(m.group(2), m.group(3), int(m.group(4) or 1))
            for m in re.finditer(r"public\s+(fixed\s+)?(float|int)\s+(\w+)(?:\[(\d+)\])?\s*;", body)]


def test_struct_sizes():
    assert ctypes.sizeof(N.Lattice) == 36
    assert ctypes.sizeof(N.LatticeHit) == 20
    hdr = _read("include", "coreslam_b200.h")
    assert int(re.search(r"#define CS_LATTICE_MAX_HITS (\d+)", hdr).group(1)) == N.LATTICE_MAX_HITS
    assert eval(re.search(r"#define CS_LATTICE_MAX_POSES (\(1 << \d+\))", hdr).group(1)) == N.LATTICE_MAX_POSES


@pytest.mark.parametrize("c_name,cs_name,ct", [("cs_lattice", "CsLattice", N.Lattice), ("cs_lattice_hit", "CsLatticeHit", N.LatticeHit)])
def test_field_lists_agree_between_header_python_and_csharp(c_name, cs_name, ct):
    """Same fields, same order, same types and lengths in include/coreslam_b200.h, the ctypes loader and the C# stubs."""
    c = _c_struct_fields(_read("include", "coreslam_b200.h"), c_name)
    assert [f[1] for f in c] == [f[0] for f in ct._fields_]
    kinds = {"float": "float", "int32_t": "int"}
    cs = _cs_struct_fields(_read("dotnet", "CoreSlamNative.cs"), cs_name)
    assert [(kinds[t], n.lower(), k) for t, n, k in c] == [(t, n.lower(), k) for t, n, k in cs]
    for (t, n, k), (fname, ftype) in zip(c, ct._fields_):
        base = ctypes.c_float if t == "float" else ctypes.c_int32
        assert ftype == (base * k if k > 1 else base), n


def test_csharp_stubs_present():
    cs = _read("dotnet", "CoreSlamNative.cs")
    for name in ("cs_set_pose", "cs_relocalize"):
        assert re.search(r"\[DllImport\(Lib\)\] public static extern CsStatus %s\(" % name, cs), name
    wrapper = _read("dotnet", "CoreSLAMProcessor.B200.cs")
    assert "public CsLatticeHit[] Relocalize(" in wrapper
    assert re.search(r"public void ResumeAt\(Vector3 pose, Vector3 odometryPose\)", wrapper)
    assert "cs_set_pose(handle, p, o, positionSearchBeginning)" in wrapper


def test_lattice_coordinates_round_once_per_operation():
    xs, ys, ts = lattice_axes([-1.5, 0.1, -3.5], [0.1, 0.07, 0.3], [7, 5, 30])
    for i in range(7):
        assert xs[i] == np.float32(np.float32(-1.5) + np.float32(np.float32(i) * np.float32(0.1)))
    assert ts[-1] > np.pi  # headings beyond +-pi are kept as they are
    # one point on an axis: the origin, whatever the step
    assert lattice_axes([1.0, 2.0, 3.0], [np.nan, -1.0, 0.0], [1, 1, 1])[0][0] == np.float32(1.0)
    assert np.array_equal(lattice_pose([0, 0, 0], [1, 2, 3], [4, 5, 6], (2 * 5 + 3) * 4 + 1), np.float32([1, 6, 6]))


def _check(vol, window, k, expect=None):
    got = reference_hits(vol, window, k)
    assert got == brute_force_hits(vol, window, k)
    if expect is not None:
        assert got == expect
    return got


def test_selection_plateau_and_ties():
    vol = np.full((3, 4, 5), 7, dtype=np.int32)
    # a plateau: every pose has the same distance, so the lower flat index wins; every pose but the first has a
    # neighbour one step below it on some axis
    assert _check(vol, 0, 3) == [(7, 0), (7, 1), (7, 2)]
    assert _check(vol, 1, 64) == [(7, 0)]
    # a second minimum with the same distance two steps away survives window 1, not window 2
    vol[1, 1, 1] = 3
    vol[1, 1, 3] = 3
    assert _check(vol, 1, 2) == [(3, 26), (3, 28)]
    assert _check(vol, 2, 2) == [(3, 26)]  # every other pose has one of the two 3s in its box


def test_selection_edges_and_unreachable_poses():
    rng = np.random.default_rng(3)
    vol = rng.integers(0, 50, (4, 6, 7)).astype(np.int32)
    vol[0, 0, 0] = -0  # a corner minimum: the box is clipped at the lattice edges
    vol[:, :, 6] = INT_MAX  # off the map: never reported, and never blocks a neighbour
    for window in (0, 1, 2, 3):
        for k in (1, 8, 64):
            hits = _check(vol, window, k)
            assert hits[0] == (0, 0) or window == 0
            assert all(d < INT_MAX for d, _ in hits)
    assert _check(np.full((2, 2, 2), INT_MAX, dtype=np.int32), 1, 8) == []


def test_selection_window_larger_than_the_lattice_and_fewer_than_k():
    rng = np.random.default_rng(5)
    vol = rng.integers(0, 1000, (3, 5, 4)).astype(np.int32)
    best = np.unravel_index(np.argmin(vol), vol.shape)
    flat = int(np.ravel_multi_index(best, vol.shape))
    assert _check(vol, 50, 64) == [(int(vol[best]), flat)]  # one window covers all: only the global minimum
    few = _check(vol, 2, 64)
    assert 1 <= len(few) < 64
    assert _check(vol, 0, 64) == sorted((int(d), i) for i, d in enumerate(vol.ravel()))[:60]


def test_selection_random_volumes_against_the_definition():
    rng = np.random.default_rng(11)
    for trial in range(9):
        shape = tuple(int(v) for v in rng.integers(1, 7 if trial < 6 else 13, 3))
        # many ties, at the magnitudes real distances have (sum * 1024 / P of 16-bit cells: up to 2^26)
        vol = (rng.integers(0, 6, shape) * (1 << 24) + rng.integers(0, 2, shape)).astype(np.int32)
        vol[rng.random(shape) < 0.2] = INT_MAX
        for window in (0, 1, 2, 3, 5):  # (from 3 on the reference takes the box minimum of the keys)
            for k in (1, 8, 64):
                _check(vol, window, k)
