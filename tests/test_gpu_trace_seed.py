"""K5a seeded trace: emia_contour_trace_slab (k_trace_seed + k_contour_trace_slab, which follows the first contour of a crop
without mark planes and re-traces with marks only when that contour was not the only one) against the classic two-pass
path emia_contour_count + emia_contour_store, bitwise: vertices, contour starts, n_contours, scratch bytes, perim0.  On one
full bench shard (the flagship workload's instances) and on adversarial masks imported with emia_mask_pack, gathered past
the persistent-lane threshold."""
import ctypes
import os

import numpy as np
import pytest
import torch

import bench
from deepemia_b200 import engine

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _contours(iset):
    """Per instance: (n_contours, index of cstart entry 0, index of the first vertex, vertex count), for either layout."""
    n = iset.n
    nc = iset.extra["n_contours"][:n]
    ar = torch.arange(n, device=iset.device, dtype=torch.int64)
    base = ar * iset.cstart_stride if iset.cstart_stride else iset.cont_off[:n] + ar
    cs = iset.cstart.to(torch.int64)
    cs0 = cs[base]
    return nc, base, iset.pt_off[:n] + cs0, cs[base + nc] - cs0


def _segments(starts, counts):
    counts = counts.to(torch.int64)
    total = int(counts.sum())
    first = torch.cumsum(counts, 0) - counts
    rep = torch.repeat_interleave(torch.arange(len(counts), device=counts.device), counts, output_size=total)
    return starts.to(torch.int64)[rep] + torch.arange(total, device=counts.device) - first[rep]


def _equal(got, want, what):
    assert got.shape == want.shape, f"{what}: shape {tuple(got.shape)} vs {tuple(want.shape)}"
    if not torch.equal(got, want):
        bad = (got != want).reshape(got.shape[0], -1).any(1).nonzero()[:, 0]
        raise AssertionError(f"{what}: {len(bad)} instances differ, first {int(bad[0])}")


def _compare(seeded, exact):
    """Every instance that did not overflow the slabs: seeded results == exact results."""
    keep = (seeded.extra["n_contours"][:seeded.n] > 0) | (exact.extra["n_contours"][:exact.n] == 0)
    over = int(seeded.extra["overflow"][0])
    assert int((~keep).sum()) <= over
    ids = keep.nonzero()[:, 0]
    ns, bs, vs, cs = (t[ids] for t in _contours(seeded))
    ne, be, ve, ce = (t[ids] for t in _contours(exact))
    _equal(ns, ne, "n_contours")
    _equal(cs, ce, "vertex count")
    _equal(seeded.extra["scratch_bytes"][ids], exact.extra["scratch_bytes"][ids], "scratch_bytes")
    _equal(seeded.perim0[ids].view(torch.int64), exact.perim0[ids].view(torch.int64), "perim0")
    assert torch.equal(seeded.cstart.to(torch.int64)[_segments(bs, ns + 1)], exact.cstart.to(torch.int64)[_segments(be, ne + 1)]), \
        "contour starts"
    assert torch.equal(seeded.pts[_segments(vs, cs)], exact.pts[_segments(ve, ce)]), "vertices"
    return len(ids)


def _hostsim():
    lib = ctypes.CDLL(os.path.join(HERE, "hostsim", "libemia_hostsim_trace.so"))
    lib.sim_trace_seeded_check.restype = ctypes.c_longlong
    lib.sim_trace_seeded_check.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_void_p]
    return lib


def _fast_fraction(iset, sample):
    """Share of the sampled instances whose seeded contour is their only one (no re-trace), from the host build of the same
    trace on the unpacked crops, each zero-padded into one frame."""
    meta = iset.meta.cpu().numpy()[sample]
    off = iset.crop_off.cpu().numpy()
    crops = iset.crops.cpu().numpy().view(np.uint32)
    ch, cw = meta[:, 2].astype(np.int64), meta[:, 3].astype(np.int64)
    Hp, Wp = int(ch.max()), int(32 * cw.max())
    masks = np.zeros((len(sample), Hp, Wp), np.uint8)
    for k, i in enumerate(sample):
        words = crops[off[i]:off[i] + ch[k] * cw[k]].reshape(ch[k], cw[k])
        bits = np.unpackbits(words.view(np.uint8), bitorder="little").reshape(ch[k], 32 * cw[k])
        masks[k, :ch[k], :32 * cw[k]] = bits
    stats = np.zeros(3, np.int64)
    assert _hostsim().sim_trace_seeded_check(masks.ctypes.data, len(masks), Hp, Wp, 4 * Hp * Wp + 8, Hp * Wp + 2,
                                             stats.ctypes.data) == -1
    return stats[0] / len(sample)


def test_seeded_trace_bench_shard(cuda_device):
    """One full bench shard: all 2048 tiles of the flagship step (about 10^6 instances) pasted as crops."""
    protos = torch.as_tensor(bench._prototypes(), device=cuda_device)
    _, _, (proto, boxes, _, _) = bench.shard(0, 1, bench.N_TILES)
    probs = protos[torch.as_tensor(proto, device=cuda_device)].contiguous()
    iset = engine.paste(probs, torch.as_tensor(boxes, device=cuda_device), bench.H, bench.W)
    del probs
    n = iset.n
    assert n > 900_000
    seeded = engine.trace(engine.select(iset, np.arange(n)), single_pass=True)
    exact = engine.trace(engine.select(iset, np.arange(n)), single_pass=False)
    assert int(seeded.extra["overflow"][0]) == 0
    assert _compare(seeded, exact) == n
    frac = _fast_fraction(iset, np.random.default_rng(5).choice(n, 20000, replace=False))
    print(f"bench shard: {n} instances, seeded contour was the only one for {100 * frac:.2f} % of a 20000-instance sample")
    assert frac >= 0.99


def _adversarial(rng, P, H, W):
    """Byte masks [P, H, W]: rings, blobs with pinholes, several components, 1-pixel lines and necks, noise, specks, blobs
    on the crop edges and on word boundaries."""
    yy, xx = np.mgrid[0:H, 0:W]
    out = np.zeros((P, H, W), bool)
    kind = rng.integers(0, 8, P)

    def discs(n, k, rmax):
        m = np.zeros((n, H, W), bool)
        for _ in range(k):
            cx, cy = rng.uniform(-2, W + 2, (n, 1, 1)), rng.uniform(-2, H + 2, (n, 1, 1))
            rx, ry = rng.uniform(0.4, rmax, (n, 1, 1)), rng.uniform(0.4, rmax, (n, 1, 1))
            m |= ((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2 <= 1.0
        return m

    def lines(n, k):
        m = np.zeros((n, H, W), bool)
        for _ in range(k):
            t = rng.uniform(0, np.pi, (n, 1, 1))
            a, b = np.cos(t), np.sin(t)
            d = a * (xx - rng.uniform(0, W, (n, 1, 1))) + b * (yy - rng.uniform(0, H, (n, 1, 1)))
            m |= np.abs(d) <= 0.5 * np.maximum(np.abs(a), np.abs(b))
        return m

    for k in range(8):
        sel = np.nonzero(kind == k)[0]
        n = len(sel)
        if k == 0:      # rings
            cx, cy = rng.uniform(10, W - 10, (n, 1, 1)), rng.uniform(10, H - 10, (n, 1, 1))
            r0 = rng.uniform(0, 25, (n, 1, 1))
            d = np.hypot(xx - cx, yy - cy)
            m = (d >= r0) & (d <= r0 + rng.uniform(0.5, 3, (n, 1, 1)))
        elif k == 1:    # blobs with pinholes
            m = discs(n, 1, 30) & (rng.random((n, H, W)) < rng.uniform(0.85, 1.0, (n, 1, 1)))
        elif k == 2:    # several components
            m = discs(n, int(rng.integers(2, 7)), 8)
        elif k == 3:    # 1-pixel lines
            m = lines(n, int(rng.integers(1, 4)))
        elif k == 4:    # blobs joined by 1-pixel necks
            m = discs(n, 2, 12) | lines(n, 1)
        elif k == 5:    # noise
            m = rng.random((n, H, W)) < rng.uniform(0.05, 0.6, (n, 1, 1))
            m &= discs(n, 1, 20)
        elif k == 6:    # specks
            m = rng.random((n, H, W)) < 0.002
        else:           # plain blobs, many on the frame edge or across a word boundary
            m = discs(n, 1, 35)
        out[sel] = m
    return out.astype(np.uint8)


def test_seeded_trace_adversarial_masks(cuda_device):
    H, W = 72, 150           # crops up to 5 words wide, the right edge off a word boundary
    masks = _adversarial(np.random.default_rng(20261021), 6000, H, W)
    pool = engine.from_masks(torch.as_tensor(masks, device=cuda_device))
    sms = torch.cuda.get_device_properties(cuda_device).multi_processor_count
    n = 8 * sms * 896 + 317                     # chunks of 1024 instances: every lane takes several
    perm = np.random.default_rng(1).integers(0, len(masks), n)
    seeded = engine.trace(engine.select(pool, perm), single_pass=True)
    exact = engine.trace(engine.select(pool, perm), single_pass=False)
    kept = _compare(seeded, exact)
    assert kept >= n - int(seeded.extra["overflow"][0])
    nc = exact.extra["n_contours"][:n]
    assert int((nc > 1).sum()) > n // 10 and int((nc == 0).sum()) > 0
    frac = _fast_fraction(pool, np.arange(len(masks)))
    print(f"adversarial masks: seeded contour was the only one for {100 * frac:.2f} % of {len(masks)} masks")
    assert 0.05 < frac < 0.95                    # both the seeded path and the re-trace are exercised
