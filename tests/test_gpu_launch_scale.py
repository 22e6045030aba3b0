"""Per-instance results do not depend on the launch size.

Above a size threshold the hot-path kernels hand a CTA, warp or lane more than one instance: K1 CTAs loop over instances with a
double-buffered prefetch, K5a lanes take their next instance from a shared counter, K2 warps reuse a global scratch plane, the
byte-mask and histogram kernels cap their grid at 65 535 CTAs, and K5b/c work through the slots in a length-sorted order.
The other parity tests run at sizes where every worker gets one item.  Here a seeded pool of diverse instances, small enough
for one item per worker and pinned against the CPU reference, is gathered by a seeded random permutation into a set past each
threshold (engine.select keeps an instance's geometry), and copy j must give exactly pool member perm[j]'s result.  All
comparisons are bitwise and run on the device; float64 results are compared through their int64 views.  Every threshold is
computed from the device's SM count and asserted to be crossed."""
import cv2
import numpy as np
import pytest
import torch
from scipy import ndimage as ndi

from deepemia_b200 import _lib, engine, synthetic as syn
from oracle import d2_paste, dedup, measure, morphology

pytestmark = pytest.mark.gpu

H, W = 240, 300                    # the right frame edge is not on a word boundary
P1_CTAS_PER_SM = {0: 8, 1: 4, 2: 32}   # default resident CTAs per SM of k_paste / k_paste_bulk / k_paste_v2
P1_MAX_CTAS_PER_SM = 255           # largest ctas_per_sm the K1 entry point takes
TRACE_THREADS = 128                # EMIA_TRACE_THREADS: lanes of a k_contour_trace_slab CTA
TRACE_CTAS_PER_SM = 8
TRACE_CHUNK = 1024                 # EMIA_TRACE_CHUNK
MORPH_MAX_CTAS = 148 * 4           # EMIA_MORPH_MAX_CTAS (a constant of the kernel, not the device's SM count)
MORPH_WARPS = 6                    # EMIA_MORPH_WARPS
GRID_CAP = 65535                   # grid cap of k_mask_bbox / k_mask_pack / k_mask_unpack / k_gray_hist
ORDER_BINS = 64                    # EMIA_ORDER_BINS
PRESORT_MAX = 256                  # EMIA_PRESORT_MAX: longer contours take the serial hull
ORDER_CLAMP = (ORDER_BINS - 2) * 8  # vertex count from which every slot falls into the longest order class


def _sms(dev):
    return torch.cuda.get_device_properties(dev).multi_processor_count


def _trace_chunk(n, sms):
    """Instances per CTA of k_contour_trace_slab (emia_contour_trace_slab)."""
    per = TRACE_CTAS_PER_SM * sms
    chunk = -(-((n + per - 1) // per) // TRACE_THREADS) * TRACE_THREADS
    return min(max(chunk, TRACE_THREADS), TRACE_CHUNK)


def _check(got, want, what, perm=None):
    """Bitwise equality of per-copy arrays (first dimension = copy); on a mismatch, name the first differing copy and its
    pool member."""
    assert got.shape == want.shape, f"{what}: shape {tuple(got.shape)} vs {tuple(want.shape)}"
    if torch.equal(got, want):
        return
    bad = (got != want).reshape(got.shape[0], -1).any(1).nonzero()[:, 0]
    j = int(bad[0])
    member = f", pool member {int(perm[j])}" if perm is not None else ""
    raise AssertionError(f"{what}: {len(bad)} copies differ, first copy {j}{member}: "
                         f"{got[j].reshape(-1)[:16].tolist()} vs {want[j].reshape(-1)[:16].tolist()}")


def _segments(starts, counts):
    """Flat int64 indices of the ranges [starts[i], starts[i] + counts[i]) one after the other."""
    counts = counts.to(torch.int64)
    total = int(counts.sum())
    first = torch.cumsum(counts, 0) - counts
    rep = torch.repeat_interleave(torch.arange(len(counts), device=counts.device), counts, output_size=total)
    return starts.to(torch.int64)[rep] + torch.arange(total, device=counts.device) - first[rep]


# ---- the pool --------------------------------------------------------------------------------------------------------------

def _comb(rng, m, x0, y0, w, h):
    """One component whose top and bottom edges jump at every column: about 4 vertices per column."""
    mid = y0 + h // 2
    top = rng.integers(y0, mid, w)
    bot = rng.integers(mid + 1, y0 + h, w)
    for c in range(w):
        m[top[c]:bot[c], x0 + c] = 1


def _mask_pool():
    """(masks uint8 [P, H, W], kinds): every kind of instance the kernels branch on; the noise masks come last."""
    rng = np.random.default_rng(20261020)
    out, kinds = [], []

    def add(m, kind):
        out.append(m); kinds.append(kind)

    def blank():
        return np.zeros((H, W), np.uint8)

    for m in syn.masks_from_polys(syn.particle_field(rng, 1900, H, W, rmin=3, rmax=40, margin=42), H, W):
        add(m, "particle")
    for y, x in [(0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1), (5, 31), (5, 32), (100, 63), (100, 64)] + \
            [(int(rng.integers(0, H)), int(rng.integers(0, W))) for _ in range(40)]:
        m = blank(); m[y, x] = 1; add(m, "speck")
    for _ in range(60):
        m = blank()
        y, x = int(rng.integers(0, H)), int(rng.integers(0, W - 60))
        k = int(rng.integers(0, 4))
        if k == 0:
            m[y, x:x + int(rng.integers(2, 60))] = 1
        elif k == 1:
            m[max(0, y - 50):y, x] = 1
        else:
            cv2.line(m, (x, y), (x + int(rng.integers(5, 60)), y + (1 if k == 2 else -1) * int(rng.integers(5, 60))), 1, 1)
        add(m, "line")
    for _ in range(60):
        m = blank()
        r = int(rng.integers(4, 41))
        cv2.circle(m, (int(rng.integers(r + 2, W - r - 2)), int(rng.integers(r + 2, H - r - 2))), r, 1, int(rng.integers(1, 4)))
        add(m, "ring")
    for _ in range(60):
        m = blank()
        r1, r2 = int(rng.integers(2, 20)), int(rng.integers(2, 20))
        cx, cy = int(rng.integers(25, W - 90)), int(rng.integers(25, H - 25))
        cv2.circle(m, (cx, cy), r1, 1, -1); cv2.circle(m, (cx + r1 + r2 + int(rng.integers(3, 30)), cy), r2, 1, -1)
        add(m, "two")
    for k in range(80):
        m = blank()
        r = int(rng.integers(3, 31))
        side = k % 4
        c = int(rng.integers(r, (W if side < 2 else H) - r))
        centre = [(c, 0), (c, H - 1), (0, c), (W - 1, c)][side]
        if k % 8 < 4:
            cv2.circle(m, centre, r, 1, -1)
        else:
            x, y = centre
            m[max(0, y - r):y + r + 1, max(0, x - r):x + r + 1] = 1
        add(m, "edge")
    for k in range(40):
        m = blank()
        b = 32 * int(rng.integers(1, W // 32))
        y = int(rng.integers(0, H - 30))
        if k % 4 == 0:
            m[y:y + 25, b - 1] = 1                      # the last column of a word
        elif k % 4 == 1:
            m[y:y + 25, b] = 1                          # the first column of a word
        else:
            m[y:y + int(rng.integers(1, 30)), b - int(rng.integers(1, 5)):b + int(rng.integers(1, 5))] = 1
        add(m, "word")
    for _ in range(30):
        add(blank(), "empty")
    for k in range(12):                                 # padded K2 plane > 1024 words: the global-workspace path
        m = blank()
        if k % 3 == 0:
            cv2.circle(m, (W // 2 + k, H // 2), 100, 1, -1)
        elif k % 3 == 1:
            m[20:220, 40 + k:240 + k] = 1; m[60:90, 90:100] = 0          # with a hole to fill
        else:
            cv2.circle(m, (W // 2, H // 2), 100, 1, 4)                 # a 200 x 200 ring
        add(m, "huge")
    for w in (40, 70, 100, 130, 160, 200, 240, 280) * 2:                # > 256 (serial hull) and > 496 vertices (clamped class)
        m = blank()
        _comb(rng, m, int(rng.integers(0, W - w + 1)), int(rng.integers(0, 60)), w, int(rng.integers(60, 180)))
        add(m, "comb")
    for _ in range(12):                                 # trace tests only: more contours than the single-pass slab holds
        m = blank()
        y, x = int(rng.integers(0, H - 60)), int(rng.integers(0, W - 60))
        m[y:y + 60, x:x + 60] = rng.random((60, 60)) < 0.45
        add(m, "noise")
    return np.stack(out), np.array(kinds)


def _contours(iset):
    """Per instance: (n_contours, index of cstart entry 0, index of the first vertex, vertex count), for either layout."""
    n = iset.n
    nc = iset.extra["n_contours"][:n]
    ar = torch.arange(n, device=iset.device, dtype=torch.int64)
    base = ar * iset.cstart_stride if iset.cstart_stride else iset.cont_off[:n] + ar
    cs = iset.cstart.to(torch.int64)
    cs0 = cs[base]
    return nc, base, iset.pt_off[:n] + cs0, cs[base + nc] - cs0


def _check_contours(big, pool, perm, keep=None):
    """Vertex lists, contour starts, n_contours, perim0 and scratch_bytes of every kept copy = those of its pool member."""
    ids = torch.arange(big.n, device=big.device) if keep is None else keep.nonzero()[:, 0]
    src = perm[ids]
    nb, bb, vb, cb = (t[ids] for t in _contours(big))
    np_, bp, vp, cp = (t[src] for t in _contours(pool))
    _check(nb, np_, "n_contours", src)
    _check(cb, cp, "vertex count", src)
    _check(big.extra["scratch_bytes"][ids], pool.extra["scratch_bytes"][src], "scratch_bytes", src)
    _check(big.perim0[ids].view(torch.int64), pool.perim0[src].view(torch.int64), "perim0", src)
    assert torch.equal(big.cstart.to(torch.int64)[_segments(bb, nb + 1)], pool.cstart.to(torch.int64)[_segments(bp, np_ + 1)]), "contour starts"
    assert torch.equal(big.pts[_segments(vb, cb)], pool.pts[_segments(vp, cp)]), "vertices"


@pytest.fixture(scope="module")
def pool(cuda_device):
    """The mask pool as an InstanceSet, traced on the exact path and measured, pinned against numpy / OpenCV / the oracle."""
    masks, kinds = _mask_pool()
    P = len(masks)
    assert P <= MORPH_MAX_CTAS * MORPH_WARPS            # one instance per K2 warp, and per CTA / lane elsewhere
    iset = engine.from_masks(torch.as_tensor(masks, device=cuda_device))
    ar = masks.reshape(P, -1).sum(1)
    assert np.array_equal(iset.area.cpu().numpy(), ar)
    bb = iset.bbox.cpu().numpy()
    for i in range(P):
        ref = dedup.get_mask_bbox(masks[i])
        assert tuple(bb[i]) == (tuple(int(v) for v in ref) if ref is not None else (-1, -1, -1, -1)), f"bbox of member {i}"
    engine.trace(iset, single_pass=False)
    got = engine.contours_to_host(iset)
    nv = np.zeros(P, np.int64)
    perim0 = iset.perim0.cpu().numpy()
    for i in range(P):
        ref = cv2.findContours(masks[i] * 255, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)[0]
        assert len(got[i]) == len(ref), f"member {i} ({kinds[i]}): {len(got[i])} contours vs {len(ref)}"
        for a, b in zip(got[i], ref):
            assert np.array_equal(a, b[:, 0, :]), f"member {i} ({kinds[i]})"
        nv[i] = sum(len(c) for c in ref)
        if ref:
            assert perim0[i] == cv2.arcLength(ref[0], True), f"perim0 of member {i}"
    assert (nv > PRESORT_MAX).sum() >= 8 and (nv > ORDER_CLAMP).sum() >= 4, "the pool must reach the serial hull and the clamped class"
    ident = engine.groups_from_offsets([0, P], cuda_device)
    meas = engine.measure_list(iset, ident, um_pix=0.5)
    # records against the oracle's measurement loop, on a seeded sample
    rec = meas.records.cpu().numpy(); off = meas.rec_off.cpu().numpy()
    for i in np.random.default_rng(3).choice(np.nonzero(kinds != "noise")[0], 300, replace=False):
        rows = measure.measure_masks([masks[i]], [0], (H, W), 0.5)
        mine = rec[off[i]:off[i + 1]]
        mine = mine[mine[:, engine.REC_MEASURED] == 1.0]
        assert len(mine) == len(rows), f"member {i}"
        for g, r in zip(mine, rows):
            np.testing.assert_allclose(g[:12], np.array([float(v) for v in r[3:15]]), rtol=1e-5, atol=0, err_msg=f"member {i}")
    # single pass on the pool itself (one instance per lane): the slab overflows exactly for the members that exceed it
    meta = iset.meta.cpu().numpy()
    ch, cw = meta[:, 2].astype(np.int64), meta[:, 3].astype(np.int64)
    cap = np.where((ch > 0) & (cw > 0), 4 * (ch + 32 * cw) + 32, 0)      # vertex slab of k_trace_caps
    nc = iset.extra["n_contours"][:P].cpu().numpy()
    over = (nc > engine.CAP_CONTOURS) | (nv > cap)
    assert np.array_equal(np.nonzero(over)[0], np.nonzero(kinds == "noise")[0]), "only the noise members overflow the slab"
    sp = engine.trace(engine.select(iset, np.arange(P)), single_pass=True)
    assert int(sp.extra["overflow"][0]) == int(over.sum())
    ident_perm = torch.arange(P, device=cuda_device)
    _check_contours(sp, iset, ident_perm, torch.as_tensor(~over, device=cuda_device))
    return {"iset": iset, "masks": masks, "kinds": kinds, "P": P, "meas": meas, "over": torch.as_tensor(over, device=cuda_device),
            "clean": np.nonzero(~over)[0]}


def _perm(seed, n, members, dev):
    return torch.as_tensor(np.random.default_rng(seed).choice(members, n), dtype=torch.int64, device=dev)


# ---- K1: multi-instance CTAs -------------------------------------------------------------------------------------------------

def _heads_pool():
    """Heads of particles of radius 3-40 plus boxes that are dead (outside the frame, degenerate), cover the whole frame,
    are tiny or hang over an edge.  Returns probs, boxes, the index of the first special box, and the pool indices of the
    whole-frame and tiny boxes."""
    probs, boxes, _, _ = syn.synthetic_heads(41, 2400, H, W, rmin=3, rmax=40, margin=20)
    rng = np.random.default_rng(42)
    dead = [[-50, -50, -10, -10], [W + 5, 3, W + 40, 30], [5, 5, 5, 40], [7, 9, 30, 9], [10, H + 2, 40, H + 30], [30, 20, 12, 40]]
    whole = [[0, 0, W, H], [-5, -7, W + 6, H + 3], [0.5, 0.25, W - 0.5, H - 0.75], [-30, 0, W + 30, H]]
    tiny = [[50.25, 60.5, 51.0, 61.25], [0, 0, 1, 1], [W - 1.5, H - 1.25, W, H], [100.1, 7.3, 100.9, 9.9]]
    over = [[-10, -10, 30, 25], [W - 20, H - 15, W + 30, H + 9], [W - 0.5, 3, W + 5, 30], [-3, H - 40, 25, H + 12]]
    extra = np.array(dead * 4 + whole * 4 + tiny * 4 + over * 4, np.float32)
    eprobs = rng.random((len(extra), 28, 28)).astype(np.float16).astype(np.float32)
    n0 = len(probs)
    off = [n0, n0 + 4 * len(dead), n0 + 4 * (len(dead) + len(whole)), n0 + 4 * (len(dead) + len(whole) + len(tiny))]
    return np.concatenate([probs, eprobs]), np.concatenate([boxes, extra]), n0, np.arange(off[1], off[2]), np.arange(off[2], off[3])


def _k1_order(rng, n, P, dead, whole, tiny, grids):
    """Pool index per copy: random, except that for every grid G one CTA's sequence goes live -> dead -> dead -> live and
    another's alternates whole-frame and tiny boxes (its rows_per_band changes at every instance)."""
    live = np.setdiff1d(np.arange(P), dead)
    order = rng.choice(live, n)
    for r, G in enumerate(grids):
        pos = np.arange(5 + 2 * r, n, G)
        k = np.arange(len(pos))
        sel = (k % 4 == 1) | (k % 4 == 2)
        order[pos[sel]] = rng.choice(dead, int(sel.sum()))
        pos = np.arange(6 + 2 * r, n, G)
        k = np.arange(len(pos))
        order[pos] = np.where(k % 2 == 0, rng.choice(whole, len(pos)), rng.choice(tiny, len(pos)))
    return order


def _k1_outputs(s):
    return s.meta, s.crop_off, s.crops[:s.total_crop_words], s.bbox, s.area, s.frames


@pytest.mark.parametrize("scale", [(1.0, 1.0), (1.28, 0.77)], ids=["unscaled", "scaled"])
@pytest.mark.parametrize("frames", [False, True], ids=["crops", "frames"])
@pytest.mark.parametrize("variant,dtype", [(0, torch.float32), (1, torch.float32), (2, torch.float32), (2, torch.float16)],
                         ids=["v0", "v1", "v2", "v2-fp16"])
def test_k1_multi_instance_ctas(cuda_device, variant, dtype, frames, scale):
    sx, sy = scale
    sms = _sms(cuda_device)
    probs, boxes, n0, whole, tiny = _heads_pool()
    P = len(probs)
    assert P <= P1_MAX_CTAS_PER_SM * sms
    tp = torch.as_tensor(probs, device=cuda_device).to(dtype).contiguous()
    tb = torch.as_tensor(boxes, device=cuda_device)
    fr = True if frames else None
    pool = engine.paste(tp, tb, H, W, scale_x=sx, scale_y=sy, frames=fr, variant=variant, ctas_per_sm=P1_MAX_CTAS_PER_SM)
    # the pool against the Detectron2 restatement, on a seeded sample that holds every special box
    rng = np.random.default_rng(variant * 10 + frames)
    sample = np.unique(np.concatenate([rng.choice(P, 120, replace=False), np.arange(n0, P)]))
    ref_masks, _, _, _ = d2_paste.predictor_instances(probs[sample], boxes[sample], np.ones(len(sample), np.float32),
                                                      np.zeros(len(sample), np.int32), sx, sy, H, W)
    _, keep = d2_paste.detector_postprocess_boxes(boxes[sample], sx, sy, H, W)
    assert np.array_equal(pool.valid.cpu().numpy()[sample], keep)
    got = engine.unpack_masks(pool, sample).cpu().numpy().astype(bool)
    assert np.array_equal(got[keep], ref_masks)
    assert not got[~keep].any()
    assert keep.sum() < len(sample)
    dead = np.nonzero(~d2_paste.detector_postprocess_boxes(boxes, sx, sy, H, W)[1])[0]      # dead at this scale
    assert len(dead) >= 8

    grid_default = P1_CTAS_PER_SM[variant if (variant != 1 or frames) else 0] * sms
    n = 3 * P1_CTAS_PER_SM[2] * sms + 101
    assert n > grid_default and n <= P1_MAX_CTAS_PER_SM * sms     # several instances per default CTA; one in the reference
    order = _k1_order(rng, n, P, dead, whole, tiny, [sms, grid_default])
    perm = torch.as_tensor(order, device=cuda_device)
    bp, bbx = tp[perm].contiguous(), tb[perm].contiguous()
    ref = engine.paste(bp, bbx, H, W, scale_x=sx, scale_y=sy, frames=fr, variant=variant, ctas_per_sm=P1_MAX_CTAS_PER_SM)
    # the one-instance-per-CTA reference is the pool, copy for copy
    sel = engine.select(pool, perm)
    names = ("meta", "crop_off", "crops", "bbox", "area", "frames")
    for name, a, b in zip(names, _k1_outputs(ref), (sel.meta, sel.crop_off, sel.crops[:sel.total_crop_words], sel.bbox, sel.area,
                                                    pool.frames[perm] if frames else None)):
        if a is not None:
            _check(a, b, f"reference {name}", perm if a.shape[0] == n else None)
    for ctas in (0, 1):          # default grid (n > grid), and one CTA per SM (about 100 instances each)
        out = engine.paste(bp, bbx, H, W, scale_x=sx, scale_y=sy, frames=fr, variant=variant, ctas_per_sm=ctas)
        for name, a, b in zip(names, _k1_outputs(out), _k1_outputs(ref)):
            if a is not None:
                _check(a, b, f"ctas_per_sm={ctas} {name}", perm if a.shape[0] == n else None)
        assert torch.equal(out.valid, ref.valid)


# ---- K5a: persistent lanes ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("per_chunk", [128, 896], ids=["two-per-lane", "capped-chunk"])
def test_k5a_persistent_lanes(cuda_device, pool, per_chunk):
    sms = _sms(cuda_device)
    n = TRACE_CTAS_PER_SM * sms * per_chunk + 317
    chunk = _trace_chunk(n, sms)
    assert chunk > TRACE_THREADS                                   # lanes take more than one instance
    if per_chunk == 896:
        assert chunk == TRACE_CHUNK                                # the production regime
    perm = _perm(per_chunk, n, np.arange(pool["P"]), cuda_device)
    big = engine.trace(engine.select(pool["iset"], perm), single_pass=True)
    over = pool["over"][perm]
    assert int(over.sum()) > 0 and int(big.extra["overflow"][0]) == int(over.sum())
    assert not big.extra["n_contours"][:n][over].any()
    _check_contours(big, pool["iset"], perm, ~over)
    del big
    exact = engine.trace(engine.select(pool["iset"], perm), single_pass=False)
    _check_contours(exact, pool["iset"], perm)


# ---- K5b/c work order --------------------------------------------------------------------------------------------------------

def _order_key(item_inst, rec_off, cstart, stride, cont_off):
    """numpy restatement of emia_order_key: 62 - min(vertices >> 3, 62); dead or contour-less slots 63."""
    nc = np.diff(rec_off)
    key = np.full(len(item_inst), ORDER_BINS - 1, np.int64)
    live = (item_inst >= 0) & (nc >= 1)
    i = item_inst[live].astype(np.int64)
    base = i * stride if stride else cont_off[i] + i
    v = cstart[base + nc[live]].astype(np.int64) - cstart[base]
    key[live] = (ORDER_BINS - 2) - np.minimum(np.maximum(v, 0) >> 3, ORDER_BINS - 2)
    return key


def _order_case(rng, L, case, stride):
    n_inst = max(1, min(L, 20000))
    nc = rng.integers(0, 4, n_inst)
    if case == "one-class":
        nc = np.maximum(nc, 1)
    v_tot = {"mixed": rng.integers(0, 1001, n_inst), "one-class": rng.integers(80, 88, n_inst),
             "dead": rng.integers(0, 1001, n_inst), "clamp": rng.integers(ORDER_CLAMP - 24, ORDER_CLAMP + 24, n_inst)}[case]
    cap = engine.CAP_CONTOURS + 1
    nc = np.minimum(nc, cap - 1)
    cont_off = np.concatenate([[0], np.cumsum(nc)]).astype(np.int64)
    cstart = np.zeros(n_inst * cap if stride else int(cont_off[-1]) + n_inst + 1, np.int32)
    for i in np.nonzero(nc)[0]:
        base = i * cap if stride else cont_off[i] + i
        cs0 = int(rng.integers(0, 1000))                  # the key uses the difference, not the entries
        inner = np.sort(rng.integers(0, v_tot[i] + 1, nc[i] - 1)) if nc[i] > 1 else np.zeros(0, np.int64)
        cstart[base:base + nc[i] + 1] = cs0 + np.concatenate([[0], inner, [v_tot[i]]])
    item_inst = rng.integers(0, n_inst, L).astype(np.int32)
    if case == "dead":
        item_inst[:] = -1
    elif case == "mixed":
        item_inst[rng.random(L) < 0.1] = -1
    cnt = np.where(item_inst >= 0, nc[np.maximum(item_inst, 0)], 0)
    rec_off = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    return item_inst, rec_off, cont_off, cstart


@pytest.mark.parametrize("stride", [engine.CAP_CONTOURS + 1, 0], ids=["slab", "packed"])
@pytest.mark.parametrize("L", [1, 255, 256, 257, 65536, 65536 + 123, (1 << 20) + 77])
def test_k5_work_order_abi(cuda_device, L, stride):
    lib = _lib.load()
    rng = np.random.default_rng(L + stride)
    for case in ("mixed", "dead", "one-class", "clamp"):
        item_inst, rec_off, cont_off, cstart = _order_case(rng, L, case, stride)
        t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=cuda_device)   # noqa: E731
        d_inst, d_off, d_cont, d_cs = t(item_inst), t(rec_off), t(cont_off), t(cstart)
        order = torch.full((L,), -1, dtype=torch.int32, device=cuda_device)
        bins = torch.empty(2 * ORDER_BINS, dtype=torch.int32, device=cuda_device)
        _lib.check(lib.emia_list_measure_order(L, d_inst.data_ptr(), d_off.data_ptr(), d_cont.data_ptr() if not stride else 0,
                                               d_cs.data_ptr(), stride, order.data_ptr(), bins.data_ptr(),
                                               torch.cuda.current_stream().cuda_stream), "emia_list_measure_order")
        got = order.cpu().numpy().astype(np.int64)
        assert np.array_equal(np.sort(got), np.arange(L)), f"{case}: not a permutation of the slots"
        key = _order_key(item_inst, rec_off, cstart, stride, cont_off)
        assert (np.diff(key[got]) >= 0).all(), f"{case}: keys out of order"
        if case == "dead":
            assert (key == ORDER_BINS - 1).all()
        if case == "one-class":
            assert len(np.unique(key[item_inst >= 0])) == 1
        if case == "clamp" and L >= 256:              # the case spans the clamped class and the classes below it
            assert ((key == 0) & (item_inst >= 0)).any() and ((key > 0) & (key < ORDER_BINS - 1)).any()


def _groups(rng, n_inst, L_min, dev):
    """Lists built directly: shorter than their capacity (the tail slots hold garbage ids), empty, and with an id listed twice."""
    caps = []
    while sum(caps) < L_min:
        caps.append(int(rng.choice([0, 1, 6, 37, 300, 2048, 5000])))
    off = np.concatenate([[0], np.cumsum(caps)]).astype(np.int32)
    length = np.zeros(len(caps), np.int32)
    idx = np.full(int(off[-1]), -77777, np.int32)
    for g, c in enumerate(caps):
        k = c if g % 3 == 0 else (0 if g % 5 == 1 else int(rng.integers(0, c + 1)))
        length[g] = k
        idx[off[g]:off[g] + k] = rng.integers(0, n_inst, k)
        if k >= 2:
            idx[off[g] + k - 1] = idx[off[g]]
    t = lambda a: torch.as_tensor(a, device=dev)   # noqa: E731
    return engine.Groups(cap_off_host=off, cap_off=t(off), length=t(length), idx=t(idx))


def _check_records(m, groups, big_perm, pool_meas):
    """Rows of every list slot = the rows of the pool member behind its instance; dead slots have none."""
    L = groups.total_cap
    cap_off = groups.cap_off_host
    g_of = np.repeat(np.arange(groups.G), np.diff(cap_off))
    ln = groups.length.cpu().numpy()
    live = np.arange(L) - cap_off[g_of] < ln[g_of]
    dev = m.records.device
    live_t = torch.as_tensor(live, device=dev)
    inst = groups.idx.to(torch.int64)[:L][live_t]
    member = big_perm[inst]
    cnt = m.rec_off[1:] - m.rec_off[:-1]
    assert not cnt[~live_t].any(), "a dead slot has records"
    pcnt = (pool_meas.rec_off[1:] - pool_meas.rec_off[:-1])[member]
    _check(cnt[live_t], pcnt, "records per slot", member)
    assert m.n_records == int(cnt.sum())
    rows = _segments(m.rec_off[:-1][live_t], pcnt)
    prow = _segments(pool_meas.rec_off[:-1][member], pcnt)
    _check(m.records[rows].view(torch.int64), pool_meas.records[prow].view(torch.int64), "records")
    assert torch.equal(m.rec_inst[rows].to(torch.int64), torch.repeat_interleave(inst, pcnt)), "rec_inst"


@pytest.fixture(scope="module")
def big_clean(cuda_device, pool):
    """The pool without the overflowing members, past the two-per-lane trace threshold, single-pass traced (slab layout)."""
    sms = _sms(cuda_device)
    n = TRACE_CTAS_PER_SM * sms * TRACE_THREADS + 317
    perm = _perm(7, n, pool["clean"], cuda_device)
    big = engine.trace(engine.select(pool["iset"], perm), single_pass=True)
    assert int(big.extra["overflow"][0]) == 0
    return big, perm


def test_k5_work_order_measure_list(cuda_device, pool, big_clean, monkeypatch):
    big, perm = big_clean
    rng = np.random.default_rng(11)
    groups = _groups(rng, big.n, engine.MEASURE_ORDER_MIN_SLOTS + 4321, cuda_device)
    assert groups.total_cap >= engine.MEASURE_ORDER_MIN_SLOTS
    runs = {}
    for on in (True, False):
        monkeypatch.setattr(engine, "MEASURE_ORDER", on)
        c0 = engine.LAUNCHES["count"]
        m = engine.measure_list(big, groups, um_pix=0.5)
        runs[on] = (m, engine.LAUNCHES["count"] - c0)
    (a, la), (b, lb) = runs[True], runs[False]
    assert la - lb == 2, "the ordered run must launch the two order kernels"
    assert torch.equal(a.rec_off, b.rec_off) and torch.equal(a.rec_inst, b.rec_inst)
    _check(a.records.view(torch.int64), b.records.view(torch.int64), "records ordered vs list order")
    _check_records(a, groups, perm, pool["meas"])
    # the sync-free variant, ordered
    monkeypatch.setattr(engine, "MEASURE_ORDER", True)
    arena = engine.Arena(cuda_device)
    for _ in range(3):             # the first run may outgrow the default capacities: the guard trips and the run repeats
        arena.begin()
        c = engine.measure_list(big, groups, um_pix=0.5, arena=arena)
        done = arena.finish()
        if done:
            break
    assert done
    c.finalize()
    assert torch.equal(c.rec_off, a.rec_off) and torch.equal(c.rec_inst, a.rec_inst)
    _check(c.records.view(torch.int64), a.records.view(torch.int64), "records with an arena")
    # the ordered path forced on short lists, around the hull's packing of 8 items x 4 warps
    monkeypatch.setattr(engine, "MEASURE_ORDER_MIN_SLOTS", 0)
    for L in (1, 7, 8, 9, 31, 32, 33):
        g = engine.groups_from_lists([rng.integers(0, big.n, L).tolist()], cuda_device)
        c0 = engine.LAUNCHES["count"]
        o = engine.measure_list(big, g, um_pix=0.5)
        ordered_launches = engine.LAUNCHES["count"] - c0
        monkeypatch.setattr(engine, "MEASURE_ORDER", False)
        c0 = engine.LAUNCHES["count"]
        u = engine.measure_list(big, g, um_pix=0.5)
        assert ordered_launches - (engine.LAUNCHES["count"] - c0) == 2
        monkeypatch.setattr(engine, "MEASURE_ORDER", True)
        assert torch.equal(o.rec_off, u.rec_off) and torch.equal(o.rec_inst, u.rec_inst)
        _check(o.records.view(torch.int64), u.records.view(torch.int64), f"records at L={L}")
        _check_records(o, g, perm, pool["meas"])


# ---- K2: persistent warps ----------------------------------------------------------------------------------------------------

F, E, D = engine.MORPH_FILL, engine.MORPH_ERODE, engine.MORPH_DILATE


def _scipy_chain(m, ops):
    for op in ops:
        m = (ndi.binary_fill_holes(m).astype(np.uint8) if op == F else morphology.erosion(m) if op == E else morphology.dilation(m))
    return m


def _k2_outputs(s):
    return s.meta, s.crop_off, s.crops[:s.total_crop_words], s.bbox, s.area


@pytest.mark.parametrize("case", ["open", "close", "mixed"])
def test_k2_persistent_warps(cuda_device, pool, case):
    P = pool["P"]
    n = 4 * MORPH_MAX_CTAS * MORPH_WARPS + 17
    assert P <= MORPH_MAX_CTAS * MORPH_WARPS < n
    perm = _perm({"open": 21, "close": 22, "mixed": 23}[case], n, np.arange(P), cuda_device)
    src = pool["iset"]
    kinds = pool["kinds"]
    assert (kinds == "huge").any() and (kinds == "ring").any()     # the global-workspace path and the flood plane
    ops, ops_b = {"open": ([F, E, D], None), "close": ([F, D, E], None), "mixed": ([F, E, D], [F, D, E])}[case]
    big_in = engine.select(src, perm)
    if case == "mixed":
        sel_np = np.random.default_rng(5).integers(0, 3, n).astype(np.int32)
        apply = torch.as_tensor(sel_np, device=cuda_device)
        got = engine.morph(big_in, ops, apply=apply, ops_b=ops_b)
        per = [engine.morph(src, ops, apply=torch.full((P,), a, dtype=torch.int32, device=cuda_device), ops_b=ops_b) for a in range(3)]
        want = engine.select(engine.concat(per), apply.to(torch.int64) * P + perm)
    else:
        got = engine.morph(big_in, ops)
        per = [engine.morph(src, ops)]
        want = engine.select(per[0], perm)
    for name, a, b in zip(("meta", "crop_off", "crops", "bbox", "area"), _k2_outputs(got), _k2_outputs(want)):
        _check(a, b, name, perm if a.shape[0] == n else None)
    # the pool results against scipy, on a seeded sample that holds every huge mask and ring
    rng = np.random.default_rng(6)
    sample = np.unique(np.concatenate([rng.choice(P, 150, replace=False), np.nonzero(np.isin(kinds, ["huge", "ring", "comb"]))[0]]))
    for a, res in enumerate(per):
        chain = [] if case == "mixed" and a == 0 else (ops_b if case == "mixed" and a == 2 else ops)
        bits = engine.unpack_masks(res, sample).cpu().numpy()
        areas = res.area.cpu().numpy()
        for k, i in enumerate(sample):
            ref = _scipy_chain(pool["masks"][i], chain)
            assert np.array_equal(bits[k], ref), f"{case} chain {a}: member {i} ({kinds[i]})"
            assert areas[i] == int(ref.sum())


# ---- grids capped at 65 535 CTAs ---------------------------------------------------------------------------------------------

def test_byte_masks_past_grid_cap(cuda_device):
    h, w = 20, 40
    n = GRID_CAP + 1000
    rng = np.random.default_rng(12)
    dens = rng.choice([0.0, 0.02, 0.3, 1.0], n)
    masks = (rng.random((n, h, w)) < dens[:, None, None]).astype(np.uint8)
    masks[::97] = 0
    masks[5::101, 3:9, 30:35] = 1                         # across the word boundary
    t = torch.as_tensor(masks, device=cuda_device)
    iset = engine.from_masks(t)
    assert iset.n > GRID_CAP
    any_y, any_x = masks.any(2), masks.any(1)
    area = masks.reshape(n, -1).sum(1)
    bbox = np.full((n, 4), -1, np.int64)
    nz = area > 0
    bbox[nz, 0] = any_y[nz].argmax(1); bbox[nz, 2] = h - 1 - any_y[nz][:, ::-1].argmax(1)
    bbox[nz, 1] = any_x[nz].argmax(1); bbox[nz, 3] = w - 1 - any_x[nz][:, ::-1].argmax(1)
    assert np.array_equal(iset.area.cpu().numpy(), area)
    assert np.array_equal(iset.bbox.cpu().numpy(), bbox)
    assert torch.equal(engine.unpack_masks(iset), t)
    idx = rng.permutation(n)
    idx = np.concatenate([idx, idx[:777]]).astype(np.int32)      # every instance, some twice
    assert torch.equal(engine.unpack_masks(iset, idx), t[torch.as_tensor(idx, dtype=torch.int64, device=cuda_device)])


def test_gray_hist_past_grid_cap(cuda_device, pool):
    P = pool["P"]
    rng = np.random.default_rng(13)
    image = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    gray = cv2.cvtColor(image, cv2.COLOR_BGR2GRAY)
    ph = engine.gray_hist(pool["iset"], image)
    hh = ph.cpu().numpy()
    for i in rng.choice(P, 200, replace=False):
        assert np.array_equal(hh[i], np.bincount(gray[pool["masks"][i] > 0], minlength=256)), f"member {i}"
    n = GRID_CAP + 777
    perm = _perm(14, n, np.arange(P), cuda_device)
    got = engine.gray_hist(engine.select(pool["iset"], perm), image)
    assert got.shape[0] > GRID_CAP
    _check(got, ph[perm], "histogram", perm)
