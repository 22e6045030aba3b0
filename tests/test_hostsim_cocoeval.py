"""CPU: the host build of the COCO segm evaluation core (deepemia_b200/csrc/core/emia_cocoeval.cuh: the match step, the IoU, the
precision / recall lookup), driven as the kernels drive it, against the dense evaluateImg / accumulate loops of oracle/cocoeval.py
on derandomized random cases.  Precision must be exactly equal (np.array_equal on float64)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import cocoeval as ce

HERE = os.path.dirname(os.path.abspath(__file__))
HS_DIR = os.path.join(HERE, "hostsim")
HS = os.path.join(HS_DIR, "libemia_hostsim_cocoeval.so")
CORE = os.path.join(HERE, "..", "deepemia_b200", "csrc", "core")
THR = np.array([min([t, 1 - 1e-10]) for t in ce.IOU_THRS], np.float64)


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """build() compiles tests/hostsim/hostsim_cocoeval.cpp; a missing or stale build is compiled into a temporary directory."""
    srcs = [os.path.join(HS_DIR, "hostsim_cocoeval.cpp")] + [os.path.join(CORE, f) for f in os.listdir(CORE)]
    path = HS
    if not os.path.exists(HS) or any(os.path.getmtime(s) > os.path.getmtime(HS) for s in srcs):
        path = str(tmp_path_factory.mktemp("hostsim_cocoeval") / "libemia_hostsim_cocoeval.so")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++", "hostsim_cocoeval.cpp", "-o", path],
                              cwd=HS_DIR)
    lib = ctypes.CDLL(path)
    vp = ctypes.c_void_p
    lib.sim_ce_iou.argtypes = [ctypes.c_longlong, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_int]
    lib.sim_ce_iou.restype = ctypes.c_double
    lib.sim_ce_match.argtypes = [ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, ctypes.c_int, vp]
    lib.sim_ce_accumulate.argtypes = [ctypes.c_int, vp, vp, ctypes.c_int, vp, ctypes.c_int, ctypes.c_double, vp, vp]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def test_iou(L):
    rng = np.random.default_rng(11)
    for _ in range(20000):
        ad, ag = (int(v) for v in rng.integers(0, 1 << 31, 2))
        inter = int(rng.integers(0, min(ad, ag) + 1))
        for crowd in (0, 1):
            want = ce.rle_iou(inter, ad, ag, crowd)
            assert L.sim_ce_iou(inter, ad, ag, crowd) == want
    assert L.sim_ce_iou(0, 0, 0, 0) == 0.0 and L.sim_ce_iou(0, 5, 0, 1) == 0.0


def _sim_eval(L, ious, gt_area, crowd, ids, dt_area, rng_a, order_rng):
    """evaluateImg through the core: the candidates of each detection in a random order."""
    D, G = ious.shape
    ig = np.array([bool(c) or a < rng_a[0] or a > rng_a[1] for a, c in zip(gt_area, crowd)], np.int32)
    cand = np.stack([order_rng.permutation(G) for _ in range(D)]).astype(np.int32) if D and G else np.zeros((D, G), np.int32)
    m = np.full((len(THR), D), -1, np.int32)
    L.sim_ce_match(D, G, _p(np.ascontiguousarray(ious, np.float64)), _p(cand), _p(ig), _p(np.asarray(crowd, np.int32)), _p(THR), len(THR),
                   _p(m))
    idv = np.asarray(ids, np.float64)
    dtm = np.where(m >= 0, idv[np.maximum(m, 0)] if G else 0.0, 0.0)
    dtIg = np.where(m >= 0, ig[np.maximum(m, 0)] if G else 0, 0).astype(bool)
    out = np.array([a < rng_a[0] or a > rng_a[1] for a in dt_area], bool).reshape(1, D)
    return dtm, dtIg | ((dtm == 0) & out)


def test_match_against_dense_loop(L):
    rng = np.random.default_rng(2024)
    levels = np.concatenate([ce.IOU_THRS, [1 - 1e-10, 1.0, 0.0, 0.3]])
    for case in range(3000):
        D, G = int(rng.integers(0, 9)), int(rng.integers(0, 9))
        if case % 3 == 0:                          # ties: IoUs on the threshold grid
            ious = rng.choice(levels, (D, G))
        else:
            ious = np.where(rng.random((D, G)) < 0.6, rng.random((D, G)), 0.0)
        gt_area = rng.choice([0.0, 500.0, 1024.0, 1024.5, 5000.0, 9216.0, 20000.0], G)
        crowd = rng.random(G) < 0.25
        ids = rng.integers(0, 4, G)               # id 0 included: dtm == 0 counts as no match
        dt_area = rng.choice([10.0, 1024.0, 5000.0, 20000.0], D)
        a_rng = ce.AREA_RNG[case % 4]
        want_dtm, want_ig, _ = ce.evaluate_img_dense(ious.reshape(D, G), gt_area, crowd, list(ids), dt_area, a_rng)
        dtm, ig = _sim_eval(L, ious, gt_area, crowd, ids, dt_area, a_rng, rng)
        assert np.array_equal(dtm, want_dtm) and np.array_equal(ig, want_ig), case


def test_accumulate_against_reference(L):
    rng = np.random.default_rng(77)
    eps = float(np.spacing(1))
    for case in range(2000):
        n = int(rng.integers(0, 60)) if case % 10 else int(rng.integers(500, 3000))
        kind = rng.choice(3, n, p=rng.dirichlet([1, 1, 1]))       # 0 tp, 1 fp, 2 ignored
        tp = (kind == 0).astype(np.int32)
        fp = (kind == 1).astype(np.int32)
        npig = int(tp.sum()) + int(rng.integers(0 if tp.sum() else 1, 5))
        # one image: scores strictly decreasing keep the sequence; dtm 1 for a tp, 0 otherwise; dtIg for the ignored ones
        T = 1
        E = [(np.linspace(1, 0, n, endpoint=False), tp.reshape(T, n).astype(np.float64), (kind == 2).reshape(T, n),
              np.array([0] * npig, int))]
        q_want, r_want = ce.accumulate_one(E, n, iou_thrs=[.5])
        q = np.zeros(101)
        rec = np.zeros(1)
        L.sim_ce_accumulate(n, _p(tp), _p(fp), npig, _p(ce.REC_THRS), 101, eps, _p(q), _p(rec))
        assert np.array_equal(q, q_want[0]) and rec[0] == r_want[0], case
