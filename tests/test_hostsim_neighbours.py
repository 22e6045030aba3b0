"""CPU: the host build of the neighbour core (deepemia_b200/csrc/core/emia_neighbour.cuh) against oracle/neighbours.py: the exact
mask-to-mask squared distance against the Euclidean distance transform and an integer brute force on random and constructed pairs,
the ring-search stop rule on lattices of exact ties, and the whole grid search (centroid nearest neighbour, closest mask, touching,
agglomerates) on constructed frames."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import neighbours as onb

HERE = os.path.dirname(os.path.abspath(__file__))
HS_DIR = os.path.join(HERE, "hostsim")
HS = os.path.join(HS_DIR, "libemia_hostsim_neighbour.so")
CORE = os.path.join(HERE, "..", "deepemia_b200", "csrc", "core")


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """build() compiles tests/hostsim/hostsim_neighbour.cpp; a missing or stale build is compiled into a temporary directory."""
    srcs = [os.path.join(HS_DIR, "hostsim_neighbour.cpp")] + [os.path.join(CORE, f) for f in os.listdir(CORE)]
    path = HS
    if not os.path.exists(HS) or any(os.path.getmtime(s) > os.path.getmtime(HS) for s in srcs):
        path = str(tmp_path_factory.mktemp("hostsim_neighbour") / "libemia_hostsim_neighbour.so")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++", "hostsim_neighbour.cpp", "-o", path],
                              cwd=HS_DIR)
    lib = ctypes.CDLL(path)
    vp, i, ll, d = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_double
    lib.sim_pair_d2.argtypes = [vp, i, i, i, i, vp, i, i, i, i, ll]
    lib.sim_pair_d2.restype = ll
    lib.sim_ring_done.argtypes = [i, i, d]
    lib.sim_neighbours.argtypes = [vp, vp, vp, vp, vp, vp, vp, i, i, i, i, i, d, vp, vp]
    return lib


def crop(piece, pad_words=0, pad_rows=0):
    """A piece as a bit-packed crop (words, ry0, wc0, ch, cw), grown by pad_words word columns on the left and pad_rows rows on
    both sides (other word alignments of the same mask)."""
    y0, x0, m = piece
    wc0 = max(x0 // 32 - pad_words, 0)
    cw = (x0 + m.shape[1] + 31) // 32 - wc0
    ry0 = max(y0 - pad_rows, 0)
    ch = y0 + m.shape[0] + pad_rows - ry0
    full = np.zeros((ch, cw * 32), np.uint8)
    full[y0 - ry0:y0 - ry0 + m.shape[0], x0 - wc0 * 32:x0 - wc0 * 32 + m.shape[1]] = m
    words = np.packbits(full, axis=1, bitorder="little").view(np.uint32).copy()
    return words, ry0, wc0, ch, cw


def sim_d2(L, a, b, limit=2 ** 62, pads=(0, 0, 0, 0)):
    wa, *ga = crop(a, pads[0], pads[1])
    wb, *gb = crop(b, pads[2], pads[3])
    return L.sim_pair_d2(wa.ctypes.data, *ga, wb.ctypes.data, *gb, limit)


def brute_d2(a, b):
    ya, xa = np.nonzero(a[2])
    yb, xb = np.nonzero(b[2])
    dy = (ya[:, None] + a[0]) - (yb[None, :] + b[0])
    dx = (xa[:, None] + a[1]) - (xb[None, :] + b[1])
    return int((dy.astype(np.int64) ** 2 + dx.astype(np.int64) ** 2).min())


def blob(rng, h, w, p=0.5):
    m = rng.random((h, w)) < p
    if not m.any():
        m[rng.integers(h), rng.integers(w)] = True
    return m


def constructed_pairs():
    sq = np.ones((5, 5), bool)
    ring = np.ones((21, 21), bool); ring[3:18, 3:18] = False
    line_h, line_v = np.ones((1, 40), bool), np.ones((40, 1), bool)
    spur = np.zeros((15, 15), bool); spur[7, :] = True; spur[:, 7] = True; spur[0:3, 0:3] = True
    return [
        ((10, 10, sq), (12, 12, sq), 0),                    # overlap
        ((10, 10, sq), (10, 15, sq), 1),                    # 4-adjacent
        ((10, 10, sq), (15, 15, sq), 2),                    # 8-adjacent (corners)
        ((10, 10, sq), (10, 16, sq), 4),                    # one-pixel gap
        ((10, 10, sq), (16, 16, sq), 8),
        ((0, 0, ring), (8, 8, sq), 36),                     # inside the ring's hole, 6 pixels from every side
        ((0, 0, ring), (5, 5, np.ones((11, 11), bool)), 9),
        ((3, 30, line_h), (2, 31, line_v), 0),              # crossing lines
        ((3, 30, line_h), (5, 31, line_v), 4),
        ((3, 30, line_h), (4, 70, line_v), 2),
        ((20, 20, spur), (20, 36, sq), 13),                 # the spur end 2 px left and 3 px below
        ((8180, 8150, np.ones((12, 30), bool)), (8160, 8185, np.ones((7, 7), bool)), 232),   # near coordinate 8191
        ((8185, 8185, np.ones((7, 7), bool)), (8185, 8170, np.ones((7, 12), bool)), 16),
    ]


def test_pair_d2_constructed(L):
    for a, b, want in constructed_pairs():
        assert onb.pair_d2(a, b) == want == brute_d2(a, b), (a[:2], b[:2])
        for pads in [(0, 0, 0, 0), (1, 2, 0, 1), (0, 3, 2, 0)]:
            assert sim_d2(L, a, b, pads=pads) == want
            assert sim_d2(L, b, a, pads=pads) == want
        assert sim_d2(L, a, b, limit=want + 1) == want          # exact below the limit
        assert sim_d2(L, a, b, limit=max(want, 1)) >= max(want, 1) or want == 0


def test_pair_d2_random(L):
    rng = np.random.default_rng(11)
    n_checked = 0
    for t in range(3000):
        h1, w1, h2, w2 = rng.integers(1, 40, 4)
        p1, p2 = rng.choice([0.05, 0.3, 0.9]), rng.choice([0.05, 0.3, 0.9])
        base = 8100 if t % 7 == 0 else 0
        a = (base + int(rng.integers(0, 50)), base + int(rng.integers(0, 50)), blob(rng, h1, w1, p1))
        b = (base + int(rng.integers(0, 50)), base + int(rng.integers(0, 50)), blob(rng, h2, w2, p2))
        want = brute_d2(a, b)
        pads = tuple(int(v) for v in rng.integers(0, 3, 4))
        assert sim_d2(L, a, b, pads=pads) == want, (t, a[:2], b[:2])
        if t % 5 == 0:
            assert onb.pair_d2(a, b) == want
        lim = int(rng.integers(0, 300))                          # below the limit: exact; otherwise at least the limit
        got = sim_d2(L, a, b, limit=lim)
        assert got == want if want < lim else got >= lim
        n_checked += 1
    assert n_checked == 3000


def test_pair_d2_against_edt_on_lines_and_spurs(L):
    rng = np.random.default_rng(12)
    for t in range(1000):
        a = np.zeros((30, 30), bool)
        b = np.zeros((30, 30), bool)
        for m in (a, b):
            for _ in range(int(rng.integers(1, 4))):                # 1-px lines and spurs
                if rng.random() < 0.5:
                    m[int(rng.integers(30)), int(rng.integers(0, 10)):int(rng.integers(10, 30))] = True
                else:
                    m[int(rng.integers(0, 10)):int(rng.integers(10, 30)), int(rng.integers(30))] = True
        pa = (int(rng.integers(0, 100)), int(rng.integers(0, 100)), a)
        pb = (int(rng.integers(0, 100)), int(rng.integers(0, 100)), b)
        ta, tb = onb.tight(pa), onb.tight(pb)
        assert sim_d2(L, ta, tb) == onb.pair_d2(ta, tb) == brute_d2(ta, tb)


def test_ring_stop_rule(L):
    # the bound (r * cs)^2 must be exceeded, not reached: a tie at exactly that distance may lie one ring further
    assert not L.sim_ring_done(1, 10, 100.0)
    assert L.sim_ring_done(1, 10, 99.999999)
    assert not L.sim_ring_done(0, 10, 0.0)
    assert L.sim_ring_done(3, 7, 440.0) and not L.sim_ring_done(3, 7, 441.0)


def pack_set(pieces):
    crops, meta, off, bbox = [], [], [0], []
    for p in pieces:
        p = onb.tight(p)
        w, ry0, wc0, ch, cw = crop(p)
        crops.append(w.reshape(-1))
        meta.append([ry0, wc0, ch, cw, wc0 * 32, (wc0 + cw) * 32, 1, 0])
        off.append(off[-1] + w.size)
        bbox.append([p[0], p[1], p[0] + p[2].shape[0] - 1, p[1] + p[2].shape[1] - 1])
    return (np.concatenate(crops).astype(np.uint32), np.asarray(meta, np.int32), np.asarray(off, np.int64), np.asarray(bbox, np.int32))


def sim_neighbours(L, pieces, listed, class_idx, H, W, cs, um_pix):
    n = len(pieces)
    crops, meta, off, bbox = pack_set(pieces)
    cent = np.array([onb.centroid(onb.tight(p)) for p in pieces], np.float64)
    lst = np.asarray(listed, np.uint8)
    cls = np.asarray(class_idx, np.int32)
    nbf = np.zeros((n, 4)); nbi = np.zeros((n, 6), np.int32)
    L.sim_neighbours(crops.ctypes.data, meta.ctypes.data, off.ctypes.data, bbox.ctypes.data, cls.ctypes.data, lst.ctypes.data,
                     cent.ctypes.data, n, int(cls.max()) + 1, H, W, cs, um_pix, nbf.ctypes.data, nbi.ctypes.data)
    return nbf, nbi


def check(L, pieces, listed, class_idx, H, W, um_pix=0.5, cell_sizes=(3, 16, 64, 1000)):
    want_f, want_i = onb.neighbours(pieces, listed, class_idx, um_pix)
    for cs in cell_sizes:
        got_f, got_i = sim_neighbours(L, pieces, listed, class_idx, H, W, cs, um_pix)
        assert np.array_equal(got_i, want_i), (cs, np.nonzero((got_i != want_i).any(1))[0][:5])
        assert np.array_equal(got_f.view(np.int64), want_f.view(np.int64)), cs
    return want_f, want_i


def sq(y, x, s):
    return (y, x, np.ones((s, s), bool))


def test_lattice_of_ties(L):
    """A square lattice: every instance has four centroid neighbours at the same d2 and four closest masks at the same D2; the
    searches must pick the lowest index whatever cell size puts the tie on a ring boundary."""
    for pitch, s in ((10, 4), (12, 12), (8, 7)):
        pieces = [sq(3 + pitch * r, 5 + pitch * c, s) for r in range(9) for c in range(9)]
        order = np.random.default_rng(pitch).permutation(len(pieces))     # indices not in raster order
        pieces = [pieces[k] for k in order]
        f, i = check(L, pieces, [True] * len(pieces), [0] * len(pieces), 128, 128, cell_sizes=(3, 5, pitch, 2 * pitch, 31, 200))
        if pitch == s:
            assert (i[:, 5] == len(pieces)).all() and (i[:, 4] == 0).all()   # edge to edge: D2 = 1, one agglomerate
        else:
            assert (i[:, 5] == 1).all()


def test_constructed_frame(L):
    H, W = 300, 400
    pieces, cls, listed = [], [], []
    for k in range(12):                                          # a chain across many cells: one agglomerate
        pieces.append(sq(20, 10 + 6 * k, 6)); cls.append(0); listed.append(True)
    ring = np.ones((40, 40), bool); ring[6:34, 6:34] = False
    pieces.append((100, 100, ring)); cls.append(0); listed.append(True)
    pieces.append(sq(115, 115, 8)); cls.append(0); listed.append(True)   # inside the ring's hole
    for k in range(10):                                          # two classes interleaved: never neighbours
        pieces.append(sq(200, 10 + 8 * k, 7)); cls.append(1 + k % 2); listed.append(True)
    pieces.append(sq(290, 390, 5)); cls.append(0); listed.append(True)   # isolated, far from its class
    pieces.append(sq(150, 300, 5)); cls.append(3); listed.append(True)   # alone in its class: empty fields
    pieces.append(sq(21, 12, 3)); cls.append(0); listed.append(False)    # not listed: nobody's neighbour
    f, i = check(L, pieces, listed, cls, H, W)
    assert (i[:12, 4] == 0).all() and (i[:12, 5] == 12).all()
    assert i[13, 2] == 12 and i[12, 2] == 13
    assert i[-2, 1] == -1 and np.isnan(f[-2, 2:]).all() and i[-2, 5] == 1
    assert i[-1, 0] == 0
    for k in range(14, 24):
        assert cls[i[k, 1]] == cls[k] and i[k, 3] == 0


def test_random_frames(L):
    rng = np.random.default_rng(13)
    for t in range(6):
        H, W = int(rng.integers(100, 400)), int(rng.integers(100, 400))
        n = int(rng.integers(20, 120))
        pieces = []
        for _ in range(n):
            h, w = int(rng.integers(1, 25)), int(rng.integers(1, 25))
            pieces.append((int(rng.integers(0, H - h)), int(rng.integers(0, W - w)), blob(rng, h, w, rng.choice([0.3, 0.8, 1.0]))))
        cls = rng.integers(0, 3, n)
        listed = rng.random(n) < 0.9
        check(L, pieces, listed, cls, H, W, um_pix=float(rng.choice([1.0, 0.37])), cell_sizes=(4, 23, 97))
