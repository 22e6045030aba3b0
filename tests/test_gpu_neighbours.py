"""GPU: neighbours_results.csv — engine.neighbours (kernels k_nb_*) exactly against oracle/neighbours.py on constructed frames (lattice
ties, chains and rings across many grid cells, an isolated particle, interleaved classes, a class with one listed instance, specks
below the area gate, two um_pix values), random particle fields, permuted sets and production sizes; the CSV bytes against csv.writer
over inference.neighbour_rows; and the option of run_inference / remeasure_results."""
import csv
import io
import os

import numpy as np
import pytest
import torch

from deepemia_b200 import adapters, engine, synthetic as syn
from deepemia_b200.functions import inference as inf
from deepemia_b200.utils import measurements as um
from oracle import neighbours as onb

pytestmark = pytest.mark.gpu


def writer_text(rows):
    buf = io.StringIO()
    csv.writer(buf).writerows(rows)
    return buf.getvalue().encode("utf-8")


def pieces(iset):
    """(y0, x0, bool mask) per instance from its crop, unpacked on the host (None for an empty mask)."""
    meta = iset.meta.cpu().numpy()
    off = iset.crop_off.cpu().numpy()
    words = iset.crops.cpu().numpy().view(np.uint32)
    out = []
    for i in range(iset.n):
        ry0, wc0, ch, cw = (int(v) for v in meta[i, :4])
        w = np.ascontiguousarray(words[off[i]:off[i] + ch * cw].reshape(ch, cw))
        m = np.unpackbits(w.view(np.uint8), axis=1, bitorder="little").astype(bool)
        out.append((ry0, wc0 * 32, m) if m.any() else None)
    return out


def listed_of(iset):
    listed = np.zeros(iset.n, bool)
    rec = iset.records.cpu().numpy()
    listed[iset.rec_inst.cpu().numpy()[rec[:, engine.REC_MEASURED] == 1.0]] = True
    return listed


def run(iset, class_idx, um_pix):
    engine.measure(iset, um_pix=um_pix, min_area=engine.default_min_area(iset.H, iset.W))
    nb = engine.neighbours(iset, class_idx, um_pix)
    assert nb.values.dtype == torch.float64 and nb.ints.dtype == torch.int32
    return nb, nb.values.cpu().numpy(), nb.ints.cpu().numpy()


def check_exact(iset, class_idx, um_pix):
    nb, f, i = run(iset, class_idx, um_pix)
    listed = listed_of(iset)
    assert np.array_equal(i[:, 0].astype(bool), listed)
    want_f, want_i = onb.neighbours(pieces(iset), listed, class_idx, um_pix)
    bad = np.nonzero((i != want_i).any(1))[0]
    assert len(bad) == 0, (bad[:5], i[bad[:3]].tolist(), want_i[bad[:3]].tolist())
    assert np.array_equal(f.view(np.int64), want_f.view(np.int64))
    return nb, f, i


def frame_from(parts, H, W):
    ms = []
    for y, x, m in parts:
        full = np.zeros((H, W), np.uint8)
        full[y:y + m.shape[0], x:x + m.shape[1]] = m
        ms.append(full)
    return engine.from_masks(torch.as_tensor(np.stack(ms), device="cuda"))


def sq(y, x, s):
    return (y, x, np.ones((s, s), bool))


@pytest.mark.parametrize("pitch,s", [(10, 4), (12, 12), (9, 8)])
def test_lattice_ties_go_to_the_lowest_index(cuda_device, pitch, s):
    parts = [sq(3 + pitch * r, 5 + pitch * c, s) for r in range(12) for c in range(12)]
    parts = [parts[k] for k in np.random.default_rng(pitch).permutation(len(parts))]
    iset = frame_from(parts, 160, 160)
    _, f, i = check_exact(iset, [0] * len(parts), 0.5)
    if pitch == s:
        assert (i[:, 4] == 0).all() and (i[:, 5] == len(parts)).all()
    else:
        assert (i[:, 5] == 1).all() and (i[:, 3] == 0).all()


@pytest.mark.parametrize("um_pix", [1.0, 0.37])
def test_constructed_frame(cuda_device, um_pix):
    H, W = 700, 900
    parts, cls = [], []
    for k in range(60):                                                    # a chain across many grid cells: one agglomerate
        parts.append(sq(20 + (k % 2), 10 + 7 * k, 7)); cls.append(0)
    t = np.linspace(0, 2 * np.pi, 40, endpoint=False)                      # a ring of discs that touch their neighbours
    for a in t:
        y, x = int(300 + 120 * np.sin(a)), int(450 + 120 * np.cos(a))
        parts.append(sq(y, x, 20)); cls.append(0)
    ring = np.ones((80, 80), bool); ring[10:70, 10:70] = False
    parts.append((520, 100, ring)); cls.append(0)
    parts.append(sq(550, 130, 20)); cls.append(0)                          # inside the ring's hole
    for k in range(20):                                                     # two classes interleaved: never neighbours
        parts.append(sq(640, 300 + 9 * k, 8)); cls.append(1 + k % 2)
    parts.append(sq(690, 890, 6)); cls.append(0)                           # isolated: the search grows to the frame size
    parts.append(sq(400, 800, 9)); cls.append(3)                           # the only listed instance of its class
    parts.append(sq(300, 450, 1)); cls.append(3)                           # specks below the area gate: not listed
    parts.append((100, 600, np.ones((1, 2), bool))); cls.append(0)
    iset = frame_from(parts, H, W)
    _, f, i = check_exact(iset, cls, um_pix)
    assert (i[:60, 5] == 60).all() and (i[:60, 4] == 0).all()
    assert (i[60:100, 5] == 40).all() and (i[60:100, 4] == 60).all()
    assert i[-4, 1] >= 0 and i[-3, 1] == -1 and np.isnan(f[-3, 2:]).all() and i[-3, 5] == 1
    assert not i[-2, 0] and not i[-1, 0]
    assert all(cls[i[k, 1]] == cls[k] for k in range(102, 122))


@pytest.mark.parametrize("seed,n,H,W", [(1, 150, 400, 500), (2, 600, 1024, 1024)])
def test_random_fields(cuda_device, seed, n, H, W):
    rng = np.random.default_rng(seed)
    ms = syn.masks_from_polys(syn.particle_field(rng, n, H, W, rmin=3, rmax=25, margin=0), H, W)
    iset = engine.from_masks(torch.as_tensor(np.stack(ms), device=cuda_device))
    check_exact(iset, rng.integers(0, 2, iset.n).tolist(), 0.5)


def test_permuted_set_gives_permuted_relations(cuda_device):
    rng = np.random.default_rng(5)
    H = W = 800
    ms = syn.masks_from_polys(syn.particle_field(rng, 400, H, W, rmin=4, rmax=20, margin=0), H, W)
    a = engine.from_masks(torch.as_tensor(np.stack(ms), device=cuda_device))
    cls = rng.integers(0, 2, a.n)
    perm = rng.permutation(a.n)
    b = engine.select(a, perm.tolist())
    _, fa, ia = run(a, cls.tolist(), 0.5)
    _, fb, ib = run(b, cls[perm].tolist(), 0.5)
    assert np.array_equal(fb.view(np.int64), fa[perm].view(np.int64))
    ok = ib[:, 1] >= 0
    assert np.array_equal(perm[ib[ok, 1]], ia[perm][ok, 1])               # centroid nearest neighbours (no exact ties here)
    assert np.array_equal(ib[:, 3], ia[perm, 3]) and np.array_equal(ib[:, 5], ia[perm, 5])
    lst = ib[:, 0] == 1
    assert np.array_equal(lst, ia[perm, 0] == 1) and lst.sum() > 300
    root_a = ia[:, 4]
    assert np.array_equal(root_a[perm[ib[lst, 4]]], root_a[perm][lst])     # the same components


def production(iset, class_idx, um_pix, sample, rng):
    nb, f, i = run(iset, class_idx, um_pix)
    listed = listed_of(iset)
    o = onb.Neighbours(pieces(iset), listed, class_idx)
    idx = np.nonzero(listed)[0]
    nn, d2 = o.nearest(idx, chunk=256)                                      # centroid NN of every instance, brute force
    assert np.array_equal(i[idx, 1], nn)
    has = nn >= 0
    assert np.array_equal(f[idx[has], 2].view(np.int64), (np.sqrt(d2[has]) * um_pix).view(np.int64))
    pick = rng.choice(idx, min(sample, len(idx)), replace=False)
    want_f, want_i = o.rows(um_pix, pick)
    assert np.array_equal(i[pick], want_i[pick])
    assert np.array_equal(f[pick].view(np.int64), want_f[pick].view(np.int64))
    return i


def test_production_micrograph(cuda_device):
    H = W = 8192
    probs, boxes, _, classes = syn.synthetic_heads(11, 20000, H, W, rmin=4, rmax=30, margin=0)
    iset = engine.paste(torch.as_tensor(probs, device=cuda_device), torch.as_tensor(boxes, device=cuda_device), H, W, frames=None)
    i = production(iset, [int(c) % 3 for c in classes[:iset.n]], 0.5, 400, np.random.default_rng(1))
    assert i[:, 0].sum() > 15000 and (i[:, 3] > 0).sum() > 100


def test_production_batch(cuda_device):
    H = W = 1024
    rng = np.random.default_rng(2)
    for f in range(64):
        probs, boxes, _, classes = syn.synthetic_heads(100 + f, 500, H, W, rmin=4, rmax=30, margin=0)
        iset = engine.paste(torch.as_tensor(probs, device=cuda_device), torch.as_tensor(boxes, device=cuda_device), H, W, frames=None)
        production(iset, [int(c) % 3 for c in classes[:iset.n]], 0.5, 5, rng)


def test_csv_bytes_match_csv_writer(cuda_device):
    rng = np.random.default_rng(7)
    H, W = 300, 400
    ms = syn.masks_from_polys(syn.particle_field(rng, 120, H, W, rmin=3, rmax=20, margin=0), H, W)
    ms.append(np.zeros((H, W), np.uint8)); ms[-1][5, 5] = 1                     # a speck: no row
    iset = engine.from_masks(torch.as_tensor(np.stack(ms), device=cuda_device))
    classes = [k % 4 for k in range(iset.n)]
    for name, psum, names in (("a.png", "500", ["pore", "throat", "x"]), ('we,ird "x".tif', 'a,"b', None)):
        fields, cidx = inf._class_table(classes, names)
        nb, _, i = run(iset, cidx, 0.25)
        got = engine.neighbours_csv_text(iset, nb, name, psum, cidx, fields)
        rows = inf.neighbour_rows(iset, nb, name, psum, cidx, fields)
        assert got == writer_text(rows)
        assert len(rows) == i[:, 0].sum() < iset.n and all(len(r) == len(um.NEIGHBOUR_HEADER) for r in rows)
    assert um.NEIGHBOUR_HEADER == onb.NEIGHBOUR_HEADER
    with pytest.raises(ValueError, match="nb must"):
        engine.neighbours_csv_text(iset, engine.NeighbourResult(nb.values[1:], nb.ints[1:]), "a", "1", cidx, fields)


def test_run_inference_and_remeasure_with_neighbours(cuda_device, tmp_path):
    imgs = [("a,1.png", np.random.default_rng(7).integers(0, 255, (160, 200, 3), dtype=np.uint8)),
            ("b.tif", np.random.default_rng(8).integers(0, 255, (150, 180, 3), dtype=np.uint8))]
    pred = syn.FakeHeadPredictor(base_seed=9, n=24)
    small = adapters.determine_small_classes(adapters.calculate_average_mask_sizes([pred], [im for _, im in imgs]))
    css = {"class_0": {"confidence_threshold": 0.3}, "class_1": {"confidence_threshold": 0.2}}
    kw = dict(tile_size=96, overlap_ratio=0.25, confidence_mode="manual", class_specific_settings=css, spatial_rules=syn.POLYHIPES_RULES)
    bar = lambda im: ('5"0,0', 0.5)                                   # noqa: E731
    common = dict(visualize=False, images=imgs, predictors=[pred], thing_classes=["pore", "throat"], small_classes=small,
                  scale_bar_fn=bar, **kw)
    inf.run_inference("polyhipes_tommy", str(tmp_path / "plain"), **common)
    inf.run_inference("polyhipes_tommy", str(tmp_path / "nb"), neighbours=True, **common)
    assert "neighbours_results.csv" not in os.listdir(tmp_path / "plain")
    assert sorted(os.listdir(tmp_path / "nb")) == sorted(os.listdir(tmp_path / "plain") + ["neighbours_results.csv"])
    for f in os.listdir(tmp_path / "plain"):
        assert (tmp_path / "plain" / f).read_bytes() == (tmp_path / "nb" / f).read_bytes()
    text = (tmp_path / "nb" / "neighbours_results.csv").read_bytes()
    rows = list(csv.reader(io.StringIO(text.decode())))
    meas = list(csv.reader(io.StringIO((tmp_path / "plain" / "measurements_results.csv").read_text())))
    assert rows[0] == um.NEIGHBOUR_HEADER
    ids = [r[0] for r in rows[1:]]
    assert len(ids) > 10 and ids == list(dict.fromkeys(r[0] for r in meas[1:]))    # one row per instance with measurement rows
    for src in ("plain", "nb"):
        out = tmp_path / (src + "_again")
        inf.remeasure_results("polyhipes_tommy", str(tmp_path / src), str(out), images=imgs, scale_bar_fn=bar, neighbours=True)
        assert (out / "neighbours_results.csv").read_bytes() == text
    inf.remeasure_results("polyhipes_tommy", str(tmp_path / "nb"), str(tmp_path / "back"), images=imgs, scale_bar_fn=bar)
    assert "neighbours_results.csv" not in os.listdir(tmp_path / "back")
