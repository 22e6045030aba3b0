"""CPU: the host build of the COCO counts-string core (deepemia_b200/csrc/core/emia_coco.cuh: delta lengths in characters and JSON
bytes, the writer, the value decoder) against oracle/coco.py, the restatement of pycocotools' rleToString / rleFrString."""
import ctypes
import itertools
import json
import os
import subprocess

import numpy as np
import pytest

from oracle import coco

HERE = os.path.dirname(os.path.abspath(__file__))
HS_DIR = os.path.join(HERE, "hostsim")
HS = os.path.join(HS_DIR, "libemia_hostsim_coco.so")
CORE = os.path.join(HERE, "..", "deepemia_b200", "csrc", "core")
ALPHABET = "".join(chr(c) for c in range(48, 112))


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """build() compiles tests/hostsim/hostsim_coco.cpp; a missing or stale build is compiled into a temporary directory."""
    srcs = [os.path.join(HS_DIR, "hostsim_coco.cpp"), os.path.join(HERE, "..", "include", "emia.h")] + \
        [os.path.join(CORE, f) for f in os.listdir(CORE)]
    path = HS
    if not os.path.exists(HS) or any(os.path.getmtime(s) > os.path.getmtime(HS) for s in srcs):
        path = str(tmp_path_factory.mktemp("hostsim_coco") / "libemia_hostsim_coco.so")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++", "hostsim_coco.cpp", "-o", path],
                              cwd=HS_DIR)
    lib = ctypes.CDLL(path)
    vp, ll = ctypes.c_void_p, ctypes.c_longlong
    lib.sim_coco_delta_len.argtypes = [ll, vp]
    lib.sim_coco_put_delta.argtypes = [ll, vp]
    lib.sim_coco_value.argtypes = [vp, ctypes.c_int]
    lib.sim_coco_value.restype = ll
    lib.sim_coco_encode.argtypes = [vp, ll, vp]
    lib.sim_coco_encode.restype = ll
    lib.sim_coco_decode.argtypes = [vp, ll, ll, vp, vp]
    lib.sim_coco_put_many.argtypes = [vp, ll, vp, vp]
    lib.sim_coco_encode_many.argtypes = [vp, vp, ll, vp, vp]
    lib.sim_coco_decode_many.argtypes = [vp, vp, ll, vp, vp, vp, vp]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def json_text(s):
    """The bytes json.dumps writes for the string s, without its quotes."""
    return json.dumps(s).encode()[1:-1]


def np_delta_chars(xs):
    """Vectorised rleToString of single values: the characters of each delta, row-major, and how many each has."""
    x = np.asarray(xs, np.int64).copy()
    chars = np.zeros((len(x), 8), np.int64)
    alive = np.ones(len(x), bool)
    for k in range(8):
        g = x & 0x1f
        x = x >> 5
        more = np.where(g & 0x10, x != -1, x != 0) & alive
        chars[:, k] = np.where(alive, np.where(more, g | 0x20, g) + 48, 0)
        alive = more
    return chars[chars > 0].astype(np.uint8), (chars > 0).sum(1)


def json_escape(raw):
    raw = np.asarray(raw, np.uint8)
    return np.repeat(raw, np.where(raw == 92, 2, 1)).tobytes()


def put_many(L, xs):
    xs = np.ascontiguousarray(xs, np.int64)
    out = np.zeros(14 * len(xs) + 1, np.uint8)
    off = np.zeros(len(xs) + 1, np.int64)
    L.sim_coco_put_many(_p(xs), len(xs), _p(out), _p(off))
    return out[:off[-1]].tobytes(), off


def test_every_delta_up_to_2_pow_20(L):
    xs = np.arange(-2 ** 20, 2 ** 20 + 1, dtype=np.int64)
    got, off = put_many(L, xs)
    raw, nchars = np_delta_chars(xs)
    assert got == json_escape(raw)
    jl = np.array([L.sim_coco_delta_len(int(x), None) for x in xs[::997]])
    assert np.array_equal(jl, np.diff(off)[::997])
    sample = xs[::4099]
    assert raw.tobytes().count(b"\\") > 1000
    for x in sample.tolist():
        s = coco.rle_to_string([x])
        assert json_text(s) == put_many(L, [x])[0]
        ch = ctypes.c_int()
        assert L.sim_coco_delta_len(x, ctypes.byref(ch)) == len(json_text(s)) and ch.value == len(s)
        assert L.sim_coco_value(s.encode(), len(s)) == x == coco.rle_fr_string(s)[0]
    # the decoder over every delta: each value is its own characters
    ends = np.cumsum(nchars)
    starts = ends - nchars
    buf = raw.tobytes()
    for k in range(0, len(xs), 1013):
        assert L.sim_coco_value(buf[starts[k]:ends[k]], int(nchars[k])) == xs[k]


def test_group_boundaries_up_to_2_pow_31(L):
    vals = set()
    for g in range(1, 8):
        for b in (5 * g - 1, 5 * g):
            for v in (2 ** b - 1, 2 ** b, 2 ** b + 1):
                vals |= {v, -v}
    vals |= {2 ** 31 - 1, -(2 ** 31 - 1), 2 ** 31, -(2 ** 31)}
    for x in sorted(v for v in vals if abs(v) <= 2 ** 31):
        s = coco.rle_to_string([x])
        assert put_many(L, [x])[0] == json_text(s), x
        ch = ctypes.c_int()
        assert L.sim_coco_delta_len(x, ctypes.byref(ch)) == len(json_text(s)) and ch.value == len(s) <= 7
        assert L.sim_coco_value(s.encode(), len(s)) == x == coco.rle_fr_string(s)[0]


def _decode(L, s, H, W):
    b = s.encode() if isinstance(s, str) else s
    cnts = np.zeros(max(len(b), 1), np.int64)
    m = ctypes.c_longlong()
    st = L.sim_coco_decode(b, len(b), H * W, _p(cnts), ctypes.byref(m))
    return st, cnts[:m.value].tolist()


def test_random_count_sequences_both_ways(L):
    rng = np.random.default_rng(11)
    nseq = 10 ** 6
    lens = rng.integers(1, 9, nseq)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    total = int(off[-1])
    bits = rng.integers(0, 32, total)
    cnts = (rng.integers(0, 2 ** 31, total) >> bits).astype(np.int64)         # log-uniform-ish in [0, 2^31 - 1]
    out_off = np.zeros(nseq + 1, np.int64)
    L.sim_coco_encode_many(_p(cnts), _p(off), nseq, None, _p(out_off))
    out = np.zeros(int(out_off[-1]) + 1, np.uint8)
    L.sim_coco_encode_many(_p(cnts), _p(off), nseq, _p(out), _p(out_off))
    # against the vectorised oracle: count i > 2 coded as its difference to count i - 2 of the same sequence
    idx = np.arange(total) - np.repeat(off[:-1], lens)
    prev = np.concatenate([[0, 0], cnts[:-2]])
    deltas = np.where(idx > 2, cnts - prev, cnts)
    raw, nchars = np_delta_chars(deltas)
    assert out[:out_off[-1]].tobytes() == json_escape(raw)
    # and back: the plain strings (no JSON escape) of every sequence decode to its counts
    char_off = np.concatenate([[0], np.cumsum(np.add.reduceat(nchars, off[:-1]))]).astype(np.int64)
    hw = np.add.reduceat(cnts, off[:-1]).astype(np.int64)
    got = np.zeros(len(raw) + 1, np.int64)
    m = np.zeros(nseq, np.int64)
    st = np.zeros(nseq, np.int32)
    L.sim_coco_decode_many(_p(np.ascontiguousarray(raw)), _p(char_off), nseq, _p(hw), _p(got), _p(m), _p(st))
    assert not st.any() and np.array_equal(m, lens)
    flat = got[np.concatenate([np.arange(char_off[q], char_off[q] + lens[q]) for q in range(0, nseq, 997)])]
    assert np.array_equal(flat, cnts[np.concatenate([np.arange(off[q], off[q + 1]) for q in range(0, nseq, 997)])])
    # the Python restatement on a sample, both directions
    for q in range(0, nseq, 9973):
        c = cnts[off[q]:off[q + 1]].tolist()
        s = coco.rle_to_string(c)
        assert json_text(s) == out[out_off[q]:out_off[q + 1]].tobytes()
        assert coco.rle_fr_string(s) == c
        assert _decode(L, s, 1, int(sum(c))) == (coco.OK, c)


def test_every_short_string(L):
    """Every string of 1-3 characters of the alphabet: status and counts as the oracle gives them (frame of the counts' sum)."""
    n = 0
    for k in (1, 2, 3):
        for t in itertools.product(ALPHABET, repeat=k):
            s = "".join(t)
            if (ord(s[-1]) - 48) & 0x20:
                assert _decode(L, s, 1, 1)[0] == coco.counts_status(s, 1, 1) in (coco.OPEN_VALUE, coco.RANGE)
                continue
            want = coco.rle_fr_string(s)
            hw = max(sum(want), 1)
            st = coco.counts_status(s, 1, hw)
            got_st, got = _decode(L, s, 1, hw)
            assert got_st == st, s
            if st == coco.OK:
                assert got == want, s
                n += 1
    assert n > 1000


@pytest.mark.parametrize("counts,s", [([0, 4], "04"), ([9], "9"), ([16], "`0"), ([32], "P1"), ([44], "\\1")])
def test_known_answers(L, counts, s):
    assert coco.rle_to_string(counts) == s
    assert coco.rle_fr_string(s) == counts
    want = json_text(s)
    out = np.zeros(32, np.uint8)
    c = np.asarray(counts, np.int64)
    assert L.sim_coco_encode(_p(c), len(c), _p(out)) == len(want)
    assert out[:len(want)].tobytes() == want
    assert _decode(L, s, 1, sum(counts)) == (coco.OK, counts)


def test_a_mask_round_trip():
    m = np.zeros((5, 4), np.uint8)
    m[4, 0] = m[0, 1] = m[2:, 3] = 1
    counts = coco.rle_encode(m)
    assert counts == [4, 2, 11, 3] and sum(counts) == 20
    assert counts == coco.counts_from_runs([(5, 2), (18, 3)], 5, 4)
    assert coco.rle_encode(np.zeros((3, 3))) == [9] and coco.rle_encode(np.ones((3, 3))) == [0, 9]
    assert coco.runs_from_counts(coco.rle_fr_string(coco.rle_to_string(counts))) == [(5, 2), (18, 3)]


@pytest.mark.parametrize("s,H,W,status", [
    ("04", 1, 4, coco.OK), ("0 4", 1, 4, coco.BAD_CHAR), ("0p", 1, 4, coco.BAD_CHAR), ("0/", 1, 4, coco.BAD_CHAR),
    ("0P", 1, 4, coco.OPEN_VALUE), ("", 1, 4, coco.SUM), ("05", 1, 4, coco.SUM), ("0O", 2, 2, coco.RANGE),
    ("PPPPPPP0", 1, 1, coco.RANGE), ("ooooooO", 1, 1, coco.RANGE), ("PPPPPP2", 1, 1, coco.RANGE),
    ("04O", 1, 8, coco.RANGE), ("0x4", 1, 4, coco.BAD_CHAR), ("0Ox", 1, 4, coco.RANGE)])
def test_malformed_statuses(L, s, H, W, status):
    assert coco.counts_status(s, H, W) == status
    assert _decode(L, s, H, W)[0] == status
