"""CPU: the host build of the RLE read-back core (deepemia_b200/csrc/core/emia_rle.cuh: number parser, per-run checks, run extent and
the canonical bbox geometry shared with emia_mask_bbox) against a numpy decoder, and the argument checks of the read-back entry points
of libemia.so."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
HS_DIR = os.path.join(HERE, "hostsim")
HS = os.path.join(HS_DIR, "libemia_hostsim_rle.so")
CORE = os.path.join(HERE, "..", "deepemia_b200", "csrc", "core")

OK, NO_SEP, BAD_CHAR, ODD, LONG, BAD_RUN, PAST_END, UNSORTED, AREA = range(9)


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """build() compiles tests/hostsim/hostsim_rle.cpp; a missing or stale build is compiled into a temporary directory."""
    srcs = [os.path.join(HS_DIR, "hostsim_rle.cpp"), os.path.join(HERE, "..", "include", "emia.h")] + \
        [os.path.join(CORE, f) for f in os.listdir(CORE)]
    path = HS
    if not os.path.exists(HS) or any(os.path.getmtime(s) > os.path.getmtime(HS) for s in srcs):
        path = str(tmp_path_factory.mktemp("hostsim_rle") / "libemia_hostsim_rle.so")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++", "hostsim_rle.cpp", "-o", path],
                              cwd=HS_DIR)
    lib = ctypes.CDLL(path)
    vp, ll = ctypes.c_void_p, ctypes.c_longlong
    lib.sim_rle_parse_uint.argtypes = [vp, ll, vp]
    lib.sim_rle_plan.argtypes = [vp, ll, ctypes.c_int, ctypes.c_int, vp, vp, vp]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def np_decode(vals, H, W):
    """Reference decoder: column-major, 1-indexed (start, length) pairs -> H x W 0/1 mask."""
    flat = np.zeros(H * W, np.uint8)
    v = np.asarray(vals, np.int64).reshape(-1, 2)
    for s, n in v:
        flat[s - 1:s - 1 + n] = 1
    return flat.reshape(W, H).T


def np_encode(m):
    flat = np.concatenate([[0], m.T.reshape(-1).astype(np.int8), [0]])
    d = np.diff(flat)
    starts, ends = np.nonzero(d == 1)[0], np.nonzero(d == -1)[0]
    return np.stack([starts + 1, ends - starts], 1).reshape(-1).tolist()


def canonical(m):
    """(meta[8], bbox[4], area) of from_masks / emia_mask_bbox for a 0/1 mask."""
    ys, xs = np.nonzero(m)
    if len(ys) == 0:
        return [0, 0, 0, 0, 0, 0, 1, 0], [-1] * 4, 0
    y0, y1, x0, x1 = int(ys.min()), int(ys.max()), int(xs.min()), int(xs.max())
    wc0 = x0 >> 5
    return [y0, wc0, y1 - y0 + 1, (x1 >> 5) - wc0 + 1, x0, x1 + 1, 1, 0], [y0, x0, y1, x1], int(len(ys))


def plan(L, vals, H, W):
    runs = np.ascontiguousarray(np.asarray(vals, np.int64).reshape(-1))
    meta, bbox, area = np.zeros(8, np.int32), np.zeros(4, np.int32), ctypes.c_longlong()
    code = L.sim_rle_plan(_p(runs) if runs.size else None, runs.size // 2, H, W, _p(meta), _p(bbox), ctypes.byref(area))
    return code, meta.tolist(), bbox.tolist(), area.value


def test_number_parser(L):
    def parse(s, avail=None):
        b = np.frombuffer(s, np.uint8).copy()
        v = ctypes.c_longlong()
        k = L.sim_rle_parse_uint(_p(b), len(b) if avail is None else avail, ctypes.byref(v))
        return k, v.value
    assert parse(b"123 45") == (3, 123)
    assert parse(b"7\r\n") == (1, 7)
    assert parse(b"000000000000000001") == (18, 1)
    assert parse(b"999999999999999999") == (18, 999999999999999999)
    assert parse(b"1000000000000000000")[0] == -1                 # 19 digits
    assert parse(b"12345", avail=2) == (2, 12)                    # stops at the end of the line
    assert parse(b"9", avail=1) == (1, 9)


@pytest.mark.parametrize("H,W", [(37, 45), (64, 33), (1, 70), (50, 1), (32, 32)])
def test_plan_matches_numpy_decoder(L, H, W):
    rng = np.random.default_rng(H * 1000 + W)
    cases = []
    full = np.ones((H, W), np.uint8)
    cases.append(full)                                            # the full frame: one run of H * W
    cases.append(np.zeros((H, W), np.uint8))                      # empty
    m = np.zeros((H, W), np.uint8); m[H - 1, 0] = 1; m[0, min(1, W - 1)] = 1
    cases.append(m)                                               # wraps from row H-1 into row 0 of the next column
    m = np.zeros((H, W), np.uint8); m[:, W // 3:W // 3 + 3] = 1; m[: H // 2, W // 3 + 3:W // 3 + 4] = 1
    cases.append(m)                                               # whole columns: a run over several columns
    m = np.zeros((H, W), np.uint8); m[H // 2, W - 1] = 1
    cases.append(m)                                               # single pixel in the last (partial) word
    m = np.zeros((H, W), np.uint8); m[0, :] = 1; m[H - 1, :] = 1
    cases.append(m)                                               # rows 0 and H-1
    for _ in range(6):
        cases.append((rng.random((H, W)) < rng.uniform(0.05, 0.95)).astype(np.uint8))
    for m in cases:
        vals = np_encode(m)
        assert np.array_equal(np_decode(vals, H, W), m)
        code, meta, bbox, area = plan(L, vals, H, W)
        want = canonical(m)
        assert code == OK and (meta, bbox, area) == want, (H, W, vals[:8])


def test_plan_accepts_adjacent_runs(L):
    H, W = 10, 7
    vals = [3, 4, 7, 2, 60, 1]                                    # run 2 starts right after run 1 ends
    code, meta, bbox, area = plan(L, vals, H, W)
    assert code == OK and (meta, bbox, area) == canonical(np_decode(vals, H, W))


@pytest.mark.parametrize("vals,code", [
    ([0, 3], BAD_RUN), ([5, 0], BAD_RUN), ([-4, 2], BAD_RUN),
    ([69, 3], PAST_END), ([71, 1], PAST_END), ([1, 71], PAST_END), ([68, 3], OK),
    ([10, 5, 3, 2], UNSORTED), ([10, 5, 14, 2], UNSORTED), ([10, 5, 10, 1], UNSORTED),
    ([10, 5, 15, 1], OK),
    ([1, 2, 5, 0, 0, 1], BAD_RUN),                                # the first bad run names the code
])
def test_plan_rejections(L, vals, code):
    got, meta, bbox, area = plan(L, vals, 10, 7)
    assert got == code
    if code != OK:
        assert meta == [0, 0, 0, 0, 0, 0, 1, 0] and bbox == [-1] * 4 and area == 0


def test_plan_area_limit(L):
    H = W = 65535
    code, meta, bbox, area = plan(L, [1, 2 ** 31 - 1], H, W)
    assert code == OK and area == 2 ** 31 - 1 and meta[:4] == [0, 0, H, (((2 ** 31 - 2) // H) >> 5) + 1]
    assert plan(L, [1, 2 ** 31], H, W)[0] == AREA
    assert plan(L, [1, 2 ** 30, 2 ** 30 + 2, 2 ** 30], H, W)[0] == AREA


def test_read_back_entry_points_check_arguments():
    import __graft_entry__ as ge
    ge.build()
    from deepemia_b200 import _lib
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)                                   # never dereferenced: every call below fails its checks first
    assert lib.emia_rle_line_count(None, 10, dummy, None) == -1
    assert lib.emia_rle_line_count(dummy, -1, dummy, None) == -1
    assert lib.emia_rle_line_index(dummy, 10, None, dummy, None) == -1
    assert lib.emia_rle_parse_count(dummy, None, 3, dummy, dummy, None) == -1
    assert lib.emia_rle_parse_count(dummy, dummy, -1, dummy, dummy, None) == -1
    assert lib.emia_rle_parse_fill(dummy, dummy, 3, dummy, dummy, dummy, None, dummy, dummy, dummy, None) == -1
    ok = [dummy] * 6
    assert lib.emia_rle_decode_plan(dummy, dummy, None, 1, 10, 10, *ok[:4], None, None) == -1
    assert b"emia_rle_decode_plan" in lib.emia_last_error()
    for H, W in ((0, 10), (10, 0), (65536, 10), (10, 65536), (-1, 5)):
        assert lib.emia_rle_decode_plan(dummy, dummy, None, 1, H, W, *ok[:5], None) == -1
    assert lib.emia_rle_decode(None, dummy, None, 1, 10, dummy, dummy, dummy, None) == -1
    assert lib.emia_rle_decode(dummy, dummy, None, 1, 65536, dummy, dummy, dummy, None) == -1
    assert lib.emia_rle_decode(dummy, dummy, None, 1, 0, dummy, dummy, dummy, None) == -1
    assert lib.emia_rle_decode(dummy, dummy, None, -1, 10, dummy, dummy, dummy, None) == -1
