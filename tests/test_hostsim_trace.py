"""CPU: the seeded border trace of k_contour_trace_slab (the first contour followed without mark planes, from the first
foreground pixel; a restart with marks unless every border-start candidate was accounted for) against the classic
RETR_EXTERNAL driver emia_find_external_contours, on every small mask and on 10^6 random ones.  Vertex lists, cstart,
contour count, point count and running arcLength must be identical, and the seeded contour may only be taken as the
only one when the classic trace finds exactly one contour."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
HS_DIR = os.path.join(HERE, "hostsim")
HS = os.path.join(HS_DIR, "libemia_hostsim_trace.so")


@pytest.fixture(scope="module")
def L():
    core = os.path.join(HERE, "..", "deepemia_b200", "csrc", "core")
    srcs = [os.path.join(HS_DIR, "hostsim_trace.cpp")] + [os.path.join(core, f) for f in os.listdir(core)]
    if not os.path.exists(HS) or any(os.path.getmtime(s) > os.path.getmtime(HS) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++", "hostsim_trace.cpp", "-o", HS],
                              cwd=HS_DIR)
    lib = ctypes.CDLL(HS)
    lib.sim_trace_seeded_check.restype = ctypes.c_longlong
    lib.sim_trace_seeded_check.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_void_p]
    return lib


def _check(L, masks, H, W, stats, cap_pts=None, cap_c=None):
    """Index of the first mask where the seeded trace differs from the classic one, or -1."""
    cap_pts = 4 * H * W + 8 if cap_pts is None else cap_pts
    cap_c = H * W + 2 if cap_c is None else cap_c
    if masks is None:
        return L.sim_trace_seeded_check(None, 0, H, W, cap_pts, cap_c, stats.ctypes.data)
    masks = np.ascontiguousarray(masks, dtype=np.uint8)
    return L.sim_trace_seeded_check(masks.ctypes.data, len(masks), H, W, cap_pts, cap_c, stats.ctypes.data)


@pytest.mark.parametrize("H", [1, 2, 3, 4, 5])
def test_seeded_trace_every_mask_up_to_5x5(L, H):
    for W in range(1, 6):
        stats = np.zeros(3, np.int64)
        assert _check(L, None, H, W, stats) == -1, (H, W)
        assert stats[2] == 0


def _lines(rng, B, H, W, k):
    """1-pixel-wide digital lines (k per mask, 8-connected) through random points at random angles."""
    yy, xx = np.mgrid[0:H, 0:W]
    out = np.zeros((B, H, W), bool)
    for _ in range(k):
        t = rng.uniform(0, np.pi, (B, 1, 1))
        a, b = np.cos(t), np.sin(t)
        px, py = rng.uniform(0, W, (B, 1, 1)), rng.uniform(0, H, (B, 1, 1))
        d = a * (xx - px) + b * (yy - py)
        out |= np.abs(d) <= 0.5 * np.maximum(np.abs(a), np.abs(b))
    return out


def _discs(rng, B, H, W, k, rmax):
    yy, xx = np.mgrid[0:H, 0:W]
    out = np.zeros((B, H, W), bool)
    for _ in range(k):
        cx, cy = rng.uniform(-2, W + 2, (B, 1, 1)), rng.uniform(-2, H + 2, (B, 1, 1))
        rx, ry = rng.uniform(0.4, rmax, (B, 1, 1)), rng.uniform(0.4, rmax, (B, 1, 1))
        out |= ((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2 <= 1.0
    return out


def _rings(rng, B, H, W):
    yy, xx = np.mgrid[0:H, 0:W]
    cx, cy = rng.uniform(0, W, (B, 1, 1)), rng.uniform(0, H, (B, 1, 1))
    r0 = rng.uniform(0.0, 0.4 * max(H, W), (B, 1, 1))
    r1 = r0 + rng.uniform(0.5, 3.0, (B, 1, 1))
    d = np.sqrt((xx - cx) ** 2 + ((yy - cy) * rng.uniform(0.5, 2.0, (B, 1, 1))) ** 2)
    return (d >= r0) & (d <= r1)


def _batch(rng, kind, B, H, W):
    if kind == "noise":
        return rng.random((B, H, W)) < rng.uniform(0.05, 0.95, (B, 1, 1))
    if kind == "rings":
        return _rings(rng, B, H, W)
    if kind == "lines":
        return _lines(rng, B, H, W, int(rng.integers(1, 4)))
    if kind == "necks":      # blobs joined (or not) by 1-pixel lines
        return _discs(rng, B, H, W, 2, max(2.0, 0.3 * min(H, W) + 1)) | _lines(rng, B, H, W, 1)
    if kind == "components":
        return _discs(rng, B, H, W, int(rng.integers(2, 6)), 3.0)
    # blobs with pinholes and bites: holes, stray candidates inside the border
    return _discs(rng, B, H, W, 1, 0.7 * max(H, W)) & (rng.random((B, H, W)) < rng.uniform(0.8, 1.0, (B, 1, 1)))


KINDS = ["noise", "rings", "lines", "necks", "components", "holes"]


def test_seeded_trace_random_masks(L):
    rng = np.random.default_rng(20261021)
    total = 0
    stats = np.zeros(3, np.int64)
    per_kind = {k: 0 for k in KINDS}
    while total < 1_000_000:
        kind = KINDS[int(rng.integers(len(KINDS)))]
        if rng.random() < 0.1:    # crops wider than 4 words take the word-by-word scan
            H, W = int(rng.integers(1, 13)), int(rng.integers(129, 260))
            B = 400
        else:
            H, W = int(rng.integers(1, 13)), int(rng.integers(1, 71))
            B = 2000
        m = _batch(rng, kind, B, H, W)
        r = _check(L, m, H, W, stats)
        assert r == -1, (kind, H, W, m[r].astype(np.uint8))
        total += B
        per_kind[kind] += B
    assert stats[2] == 0
    assert min(per_kind.values()) > 50_000, per_kind
    assert stats[0] > 50_000 and stats[1] > stats[0], stats


def test_seeded_trace_overflow_matches(L):
    """Capacities too small for the vertices or the contours: the seeded trace overflows exactly when the classic one does."""
    rng = np.random.default_rng(7)
    stats = np.zeros(3, np.int64)
    for kind in KINDS:
        for cap_pts, cap_c in ((6, 64), (64, 1), (12, 2)):
            m = _batch(rng, kind, 2000, 10, 40)
            assert _check(L, m, 10, 40, stats, cap_pts=cap_pts, cap_c=cap_c) == -1, (kind, cap_pts, cap_c)
