"""CPU: the host build of the number formatting core of the result CSV writers (deepemia_b200/csrc/core/emia_text.cuh): shortest digits
against std::to_chars, layouts against Python repr / str(np.float64) / str(np.float32), integers against str(); and the argument
checks of the CSV text entry points of libemia.so."""
import ctypes
import os
import struct
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
HS_DIR = os.path.join(HERE, "hostsim")
HS = os.path.join(HS_DIR, "libemia_hostsim_text.so")
CORE = os.path.join(HERE, "..", "deepemia_b200", "csrc", "core")
THREADS = max(1, os.cpu_count() or 1)
NUM_MAX = 32
F64, F32, INT = 0, 1, 2


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """build() compiles tests/hostsim/hostsim_text.cpp; a missing or stale build is compiled into a temporary directory."""
    srcs = [os.path.join(HS_DIR, "hostsim_text.cpp")] + [os.path.join(CORE, f) for f in os.listdir(CORE)]
    path = HS
    if not os.path.exists(HS) or any(os.path.getmtime(s) > os.path.getmtime(HS) for s in srcs):
        path = str(tmp_path_factory.mktemp("hostsim_text") / "libemia_hostsim_text.so")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-x", "c++", "hostsim_text.cpp", "-o",
                               path], cwd=HS_DIR)
    lib = ctypes.CDLL(path)
    vp, ll, ull = ctypes.c_void_p, ctypes.c_longlong, ctypes.c_ulonglong
    lib.sim_check_f32.argtypes = [ull, ull, ull, ctypes.c_int, vp, vp]
    lib.sim_check_f32.restype = ll
    lib.sim_check_f64_random.argtypes = [ull, ll, ctypes.c_int, vp, vp]
    lib.sim_check_f64_random.restype = ll
    lib.sim_check_f64_list.argtypes = [vp, ll]
    lib.sim_check_f64_list.restype = ll
    lib.sim_format.argtypes = [vp, vp, ll, ctypes.c_int, vp, vp]
    lib.sim_i64_len.argtypes = [ll]
    return lib


def check_f32(L, lo, hi, step=1):
    bad, first = ctypes.c_longlong(), ctypes.c_ulonglong()
    n = L.sim_check_f32(lo, hi, step, THREADS, ctypes.byref(bad), ctypes.byref(first))
    assert bad.value == 0, f"{bad.value} of {n} float32 patterns differ from std::to_chars, first 0x{first.value:08x}"
    return n


def fmt(L, values, kind):
    """Texts of the core's formatter for `values` (kind F64: repr(float), F32: str(np.float32), INT: str(int))."""
    n = len(values)
    v = np.asarray(values if kind != INT else np.zeros(n), np.float64)
    iv = np.asarray(values if kind == INT else np.zeros(n), np.int64)
    out = np.zeros(n * NUM_MAX, np.uint8)
    ln = np.zeros(n, np.int32)
    L.sim_format(v.ctypes.data, iv.ctypes.data, n, kind, out.ctypes.data, ln.ctypes.data)
    raw = out.tobytes()
    return [raw[k * NUM_MAX:k * NUM_MAX + ln[k]].decode() for k in range(n)]


def f64_edges():
    """Subnormals, powers of 2 and 10 at +-1 ulp, the neighbourhoods of 1e-4 and 1e16, DBL_MAX."""
    v = [5e-324, 1e-323, 1.5e-323, 2.225073858507201e-308, 2.2250738585072014e-308, np.finfo(np.float64).max, 1e-4, 1e16, 1e-5,
         9.999999999999999e15, 1e15, 0.1, 0.2, 0.3, 1 / 3]
    v += [struct.unpack("<d", struct.pack("<Q", b))[0] for b in list(range(1, 64)) + [(1 << 52) - k for k in range(1, 16)]]
    v += [2.0 ** e for e in range(-1074, 1024)] + [float(f"1e{e}") for e in range(-323, 309)]
    v += [np.nextafter(np.float64(c), d) for c in (1e-4, 1e16, 1e-5, 1e15) for d in (0.0, np.inf)]
    v += [np.nextafter(np.float64(x), d) for x in [2.0 ** e for e in range(-1022, 1023)] + [float(f"1e{e}") for e in range(-307, 308)]
          for d in (0.0, np.inf)]
    return np.array(v, np.float64)


def layout_values(seed, n):
    """About n values from the generators of the digit checks: random bit patterns, log-uniform magnitudes, the layout thresholds of
    both formats at a few ulps, small integers, special values."""
    rng = np.random.default_rng(seed)
    bits = rng.integers(0, 2 ** 63, n // 4, dtype=np.int64).view(np.float64)
    bits = bits[np.isfinite(bits)] * rng.choice([-1.0, 1.0], len(bits[np.isfinite(bits)]))
    logu = 10.0 ** rng.uniform(-8, 20, n // 4) * rng.choice([-1.0, 1.0], n // 4)
    near = []
    for c in (1e-4, 1e-5, 1e16, 1e15, 1e6, 1e5, 1.0, 0.5):
        x32 = np.float32(c)
        near += [np.nextafter(np.float64(c), np.inf * s) for s in (-1, 1)] + [c]
        near += [float(np.frombuffer(np.array([x32.view(np.int32) + d], np.int32).tobytes(), np.float32)[0]) for d in range(-40, 41)]
    ints = np.arange(-2000, 2000, dtype=np.float64).tolist() + [2.0 ** 53, 1e15, 123456789.0, 1e16, 1e22]
    special = [np.nan, -np.nan, np.inf, -np.inf, 0.0, -0.0]
    return np.concatenate([bits, logu, rng.uniform(-1e4, 1e4, n // 4), np.array(near + ints + special, np.float64),
                           np.float32(logu).astype(np.float64)])


def test_f32_digits_every_exponent(L):
    """A dense sample of every float32 exponent (every 97th pattern) and the first and last 64 mantissas of each binade."""
    n = check_f32(L, 0, 2 ** 31, 97)
    assert n > 2 ** 31 // 97 - 2 ** 23
    for e in range(256):
        check_f32(L, e << 23, (e << 23) + 64)
        check_f32(L, ((e + 1) << 23) - 64, (e + 1) << 23)


def test_f64_digits_random_and_edges(L):
    bad, first = ctypes.c_longlong(), ctypes.c_ulonglong()
    n = L.sim_check_f64_random(20261020, 10 ** 7, THREADS, ctypes.byref(bad), ctypes.byref(first))
    assert n > 9 * 10 ** 6
    assert bad.value == 0, f"{bad.value} of {n} binary64 patterns differ from std::to_chars, first 0x{first.value:016x}"
    v = f64_edges()
    k = L.sim_check_f64_list(v.ctypes.data, len(v))
    assert k == -1, repr(v[k])


def test_f64_layout_is_python_repr(L):
    v = np.concatenate([layout_values(1, 100000), f64_edges()])
    got = fmt(L, v, F64)
    want = [repr(float(x)) for x in v]
    assert want == [str(np.float64(x)) for x in v]                 # csv.writer writes both the same way
    bad = [(w, g) for w, g in zip(want, got) if w != g]
    assert not bad, bad[:10]


def test_f32_layout_is_numpy_str(L):
    v = layout_values(2, 100000)
    with np.errstate(over="ignore"):
        v32 = v.astype(np.float32)
    got = fmt(L, v32.astype(np.float64), F32)
    want = [str(x) for x in v32]
    bad = [(w, g) for w, g in zip(want, got) if w != g]
    assert not bad, bad[:10]
    assert fmt(L, [np.float32(1e-4), np.nextafter(np.float32(1e-4), np.float32(1)), 999999.94, 1e6, 123456789.0], F32) == \
        ["1e-04", "0.000100000005", "999999.94", "1e+06", "1.2345679e+08"]


def test_specials_and_integral_values(L):
    assert fmt(L, [np.nan, np.inf, -np.inf, -0.0, 0.0, 3.0, 1e16, 1e-5, 0.0001, -1e22], F64) == \
        ["nan", "inf", "-inf", "-0.0", "0.0", "3.0", "1e+16", "1e-05", "0.0001", "-1e+22"]
    assert fmt(L, [np.nan, -np.inf, -0.0, 3.0], F32) == ["nan", "-inf", "-0.0", "3.0"]


def test_integers(L):
    v = [0, 1, -1, 9, 10, 99, 100, -100, 2 ** 31 - 1, -2 ** 31, 2 ** 32, 10 ** 18, 10 ** 18 - 1, 2 ** 63 - 1, -2 ** 63]
    assert fmt(L, v, INT) == [str(x) for x in v]
    assert [L.sim_i64_len(x) for x in v] == [len(str(x)) for x in v]


def test_csv_text_entry_points_check_arguments():
    import __graft_entry__ as ge
    ge.build()
    from deepemia_b200 import _lib
    lib = _lib.load()
    d = ctypes.c_void_p(16)                                       # never dereferenced: every call below fails its checks first
    assert lib.emia_csv_rle_count(d, d, -1, 4, d, None) == -1
    assert lib.emia_csv_rle_count(d, d, 3, -1, d, None) == -1
    assert lib.emia_csv_rle_count(None, d, 3, 4, d, None) == -1
    assert lib.emia_csv_rle_count(d, d, 3, 4, None, None) == -1
    assert b"emia_csv_rle_count" in lib.emia_last_error()
    assert lib.emia_csv_rle_write(d, d, 3, None, 4, d, d, None) == -1
    assert lib.emia_csv_rle_write(d, d, 3, d, 4, None, d, None) == -1
    assert lib.emia_csv_rle_write(d, d, 3, d, 4, d, None, None) == -1
    assert lib.emia_csv_rle_write(d, d, 3, d, 2 ** 31, d, d, None) == -1
    ok = [d] * 7
    assert lib.emia_csv_measure_count(d, d, -1, d, None, d, d, 3, d, None) == -1
    assert lib.emia_csv_measure_count(d, d, 5, d, None, d, d, 2, d, None) == -1
    assert lib.emia_csv_measure_count(d, None, 5, d, None, d, d, 3, d, None) == -1
    assert lib.emia_csv_measure_count(d, d, 5, d, None, d, None, 3, d, None) == -1
    assert b"emia_csv_measure_count" in lib.emia_last_error()
    assert lib.emia_csv_measure_write(d, d, 5, d, None, d, d, 3, None, d, None) == -1
    assert lib.emia_csv_measure_write(d, d, 5, d, None, d, d, 3, d, None, None) == -1
    assert lib.emia_csv_measure_write(d, d, 5, None, None, d, d, 3, d, d, None) == -1
    assert b"emia_csv_measure_write" in lib.emia_last_error()
    assert lib.emia_csv_rle_count(None, None, 0, 0, None, None) == 0                 # nothing to do: no pointer needed
    assert lib.emia_csv_measure_write(None, None, 0, None, None, None, None, 3, None, None, None) == 0
    del ok
