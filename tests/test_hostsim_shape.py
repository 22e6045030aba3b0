"""CPU: the host build of the shape-descriptor core (deepemia_b200/csrc/core/emia_shape.cuh) against oracle/shape.py, bit for bit in
every column, on contours from cv2.findContours; the convex hull it builds on (emia_convex_hull) against cv2.convexHull; known answers;
and the argument checks of emia_contour_shape_list and the shape variants of the measurement CSV entry points."""
import ctypes
import math
import os
import subprocess

import cv2
import numpy as np
import pytest

from oracle import shape as oshape

HERE = os.path.dirname(os.path.abspath(__file__))
HS_DIR = os.path.join(HERE, "hostsim")
HS = os.path.join(HS_DIR, "libemia_hostsim_shape.so")
CORE = os.path.join(HERE, "..", "deepemia_b200", "csrc", "core")
GATE = 5.0                                           # the smallest area gate of the measurement loop


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """build() compiles tests/hostsim/hostsim_shape.cpp; a missing or stale build is compiled into a temporary directory."""
    srcs = [os.path.join(HS_DIR, "hostsim_shape.cpp")] + [os.path.join(CORE, f) for f in os.listdir(CORE)]
    path = HS
    if not os.path.exists(HS) or any(os.path.getmtime(s) > os.path.getmtime(HS) for s in srcs):
        path = str(tmp_path_factory.mktemp("hostsim_shape") / "libemia_hostsim_shape.so")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++", "hostsim_shape.cpp", "-o", path],
                              cwd=HS_DIR)
    lib = ctypes.CDLL(path)
    vp, ll = ctypes.c_void_p, ctypes.c_longlong
    lib.sim_shape.argtypes = [vp, vp, ll, ctypes.c_double, vp]
    lib.sim_hulls.argtypes = [vp, vp, ll, vp, vp]
    return lib


def pack(contours):
    off = np.zeros(len(contours) + 1, np.int64)
    off[1:] = np.cumsum([len(c) for c in contours])
    flat = np.concatenate([np.asarray(c).reshape(-1, 2) for c in contours]).astype(np.int64)
    return (flat[:, 0] | (flat[:, 1] << 16)).astype(np.uint32), off


def core_shape(L, contours, um_pix=1.0):
    pts, off = pack(contours)
    out = np.zeros((len(contours), 10), np.float64)
    L.sim_shape(pts.ctypes.data, off.ctypes.data, len(contours), um_pix, out.ctypes.data)
    return out


def core_hulls(L, contours):
    pts, off = pack(contours)
    hull = np.zeros(max(int(off[-1]), 1), np.int32)
    hoff = np.zeros(len(contours) + 1, np.int64)
    L.sim_hulls(pts.ctypes.data, off.ctypes.data, len(contours), hull.ctypes.data, hoff.ctypes.data)
    return [hull[hoff[k]:hoff[k + 1]] for k in range(len(contours))]


def contours_of(mask, offset=(0, 0)):
    cs, _ = cv2.findContours(mask, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE, offset=offset)
    return [c.reshape(-1, 2) for c in cs]


def corpus(seed=0):
    """Contours from cv2.findContours: random polygons and discs, axis-aligned rectangles (collinear vertices), rotated squares (Feret
    ties), 1-px lines and spurs (self-touching contours), and the same shapes moved next to coordinate 8191."""
    rng = np.random.default_rng(seed)
    out = []
    S = 160
    for f in range(2700):
        m = np.zeros((S, S), np.uint8)
        kind = f % 6
        for _ in range(int(rng.integers(4, 12))):
            cx, cy = (int(v) for v in rng.integers(10, S - 10, 2))
            if kind == 0:
                k = int(rng.integers(3, 9))
                poly = np.stack([cx + rng.integers(-30, 31, k), cy + rng.integers(-30, 31, k)], 1).astype(np.int32)
                cv2.fillPoly(m, [poly], 1)
            elif kind == 1:
                cv2.circle(m, (cx, cy), int(rng.integers(1, 40)), 1, -1)
            elif kind == 2:
                w, h = (int(v) for v in rng.integers(1, 50, 2))
                m[cy:cy + h, cx:cx + w] = 1
            elif kind == 3:
                a, b = (int(v) for v in rng.integers(-20, 21, 2))
                sq = np.array([[cx + a, cy + b], [cx - b, cy + a], [cx - a, cy - b], [cx + b, cy - a]], np.int32)
                cv2.fillPoly(m, [sq], 1)
            elif kind == 4:
                p0 = (cx, cy)
                p1 = tuple(int(v) for v in rng.integers(0, S, 2))
                if rng.random() < 0.6:
                    cv2.circle(m, p0, int(rng.integers(3, 15)), 1, -1)
                cv2.line(m, p0, p1, 1, 1)
            else:
                m |= (rng.random((S, S)) < 0.004).astype(np.uint8)
                cv2.circle(m, (cx, cy), int(rng.integers(2, 25)), 1, -1)
        off = (8191 - S + 1, 8191 - S + 1) if f % 5 == 4 else (0, 0)
        out += contours_of(m, off)
    return out


@pytest.fixture(scope="module")
def contours():
    cs = corpus()
    assert len(cs) >= 10000
    return cs


def test_hull_matches_opencv(L, contours):
    """emia_convex_hull, rotated to its smallest (y, x) vertex, gives cv2.convexHull's vertices, rotated likewise."""
    for c, h in zip(contours, core_hulls(L, contours)):
        got = c[h].astype(np.int64)
        if len(got):
            s = int(np.lexsort((got[:, 0], got[:, 1]))[0])
            got = np.roll(got, -s, axis=0)
        np.testing.assert_array_equal(got, oshape.canonical_hull(c))


def test_core_matches_oracle_bit_for_bit(L, contours):
    gated = [c for c in contours if cv2.contourArea(c.reshape(-1, 1, 2).astype(np.int32)) >= GATE]
    assert len(gated) >= 10000
    near = [c for c in gated if c.max() >= 8100]
    assert len(near) > 500
    for u in (1.0, 0.37, 3e-7):
        got = core_shape(L, gated, u)
        want = np.array([oshape.shape_descriptors(c, u) for c in gated])
        bad = np.nonzero(~(got == want).all(1))[0]
        assert len(bad) == 0, (u, len(bad), gated[bad[0]].tolist(), got[bad[0]].tolist(), want[bad[0]].tolist())
    # the corpus reaches the cases the definitions single out
    h = [oshape.canonical_hull(c) for c in gated]
    ties = sum(1 for hh in h if len(hh) > 2 and np.count_nonzero(np.triu(((hh[:, None] - hh[None]) ** 2).sum(-1) ==
                                                                        ((hh[:, None] - hh[None]) ** 2).sum(-1).max(), 1)) > 1)
    assert ties > 100
    assert sum(1 for c, hh in zip(gated, h) if len(hh) < len(c)) > 1000                   # collinear or concave vertices dropped
    assert sum(1 for c in gated if len({tuple(p) for p in c.tolist()}) < len(c)) > 50      # self-touching contours


def test_known_answers(L):
    # an axis-aligned k x k square: diagonals tie, the angle is 45
    for k, (x0, y0) in ((10, (3, 4)), (2, (0, 0)), (300, (7890, 7890))):
        m = np.zeros((y0 + k + 2, x0 + k + 2), np.uint8)
        m[y0:y0 + k, x0:x0 + k] = 1
        c = contours_of(m)[0]
        v = core_shape(L, [c], 0.5)[0]
        s = k - 1
        assert v[:8].tolist() == [s * s * 0.25, s * s * 0.25, 1.0, 2.0 * s, 1.0, math.sqrt(2.0 * s * s) * 0.5, s * 0.5, 45.0]
        assert v[8:].tolist() == [x0 + s / 2, y0 + s / 2]
    # a 1 x k strip: a 2-vertex contour, no area; its Feret diameters are its length and 0
    for k, vertical in ((7, False), (12, True)):
        m = np.zeros((20, 20), np.uint8)
        if vertical:
            m[2:2 + k, 5] = 1
        else:
            m[5, 2:2 + k] = 1
        c = contours_of(m)[0]
        v = core_shape(L, [c])[0]
        assert len(c) == 2 and v[[0, 1, 3, 5, 6, 7]].tolist() == [0.0, 0.0, 2.0 * (k - 1), k - 1.0, 0.0, 90.0 if vertical else 0.0]
    # a right triangle with legs 30 and 40 (hypotenuse 50): min width = 30 * 40 / 50, max-Feret direction (30, 40)
    tri = np.array([[10, 20], [10, 60], [40, 20]])
    v = core_shape(L, [tri])[0]
    assert v[:8].tolist() == [600.0, 600.0, 1.0, 120.0, 1.0, 50.0, 24.0, math.atan2(40.0, 30.0) * (180.0 / math.pi)]
    assert abs(v[8] - 20.0) < 1e-12 and abs(v[9] - 100.0 / 3) < 1e-12
    assert v.tolist() == oshape.shape_descriptors(tri)


def test_entry_point_arguments():
    import __graft_entry__ as ge
    ge.build()
    from deepemia_b200 import _lib
    lib = _lib.load()
    d = ctypes.c_void_p(16)                                       # never dereferenced: every call below fails its checks first
    ok = [d] * 6                                                  # item_inst, rec_off, scr_off, cont_off, pt_off, cstart
    assert lib.emia_contour_shape_list(-1, *ok, 0, 1.0, d, d, d, None, d, None) == -1
    assert lib.emia_contour_shape_list(4, *ok, -1, 1.0, d, d, d, None, d, None) == -1
    assert lib.emia_contour_shape_list(4, d, d, d, None, d, d, 0, 1.0, d, d, d, None, d, None) == -1     # packed layout: cont_off needed
    assert lib.emia_contour_shape_list(4, *ok, 9, 1.0, d, None, d, None, d, None) == -1
    assert lib.emia_contour_shape_list(4, *ok, 9, 1.0, d, d, d, None, None, None) == -1
    assert b"emia_contour_shape_list" in lib.emia_last_error()
    assert lib.emia_contour_shape_list(0, *([None] * 6), 0, 1.0, None, None, None, None, None, None) == 0
    assert lib.emia_csv_measure_shape_count(d, d, -1, d, None, d, d, d, 3, d, None) == -1
    assert lib.emia_csv_measure_shape_count(d, d, 5, d, None, d, d, d, 2, d, None) == -1
    assert lib.emia_csv_measure_shape_count(d, d, 5, d, None, d, d, d, 3, None, None) == -1
    assert b"emia_csv_measure_shape_count" in lib.emia_last_error()
    assert lib.emia_csv_measure_shape_write(d, d, 5, d, None, d, d, d, 3, None, d, None) == -1
    assert lib.emia_csv_measure_shape_write(d, d, 5, d, None, d, d, d, 3, d, None, None) == -1
    assert lib.emia_csv_measure_shape_write(d, None, 5, d, None, None, d, d, 3, d, d, None) == -1
    assert b"emia_csv_measure_shape_write" in lib.emia_last_error()
    assert lib.emia_csv_measure_shape_write(None, None, 0, None, None, None, None, None, 3, None, None, None) == 0
