"""GPU: COCO instance JSON with compressed RLE — engine.coco_annotations_text against json.dumps of oracle/coco.py, the device decode of
counts strings (engine._coco_decode / coco_decode) against rle_decode, and the flows: run_inference(coco_json=True),
load_coco_results and measure_coco."""
import json

import numpy as np
import pytest
import torch

from deepemia_b200 import _lib, adapters, engine, synthetic as syn
from deepemia_b200.functions import inference as inf
from oracle import coco

pytestmark = pytest.mark.gpu


def edge_masks(H, W, seed):
    rng = np.random.default_rng(seed)
    ms = [np.zeros((H, W), np.uint8), np.ones((H, W), np.uint8)]                                # empty, full frame
    for y, x in ((0, 0), (H - 1, W - 1), (H - 1, 0), (0, W - 1)):                                # single corner pixels
        m = np.zeros((H, W), np.uint8); m[y, x] = 1; ms.append(m)
    if H > 2 and W > 2:
        m = np.zeros((H, W), np.uint8); m[H - 1, 1] = 1; m[0, 2] = 1; m[H - 2:, 0] = 1; ms.append(m)   # runs wrapping columns
        m = np.zeros((H, W), np.uint8); m[:, 1:] = 1; ms.append(m)                                 # pixel 0 unset, last set
    for f in (44, 44 + 32 * 44, 12 * 32 + 44, 1388):                                               # counts whose strings hold '\'
        if f < H * W:
            m = np.zeros(H * W, np.uint8); m[f:f + min(44, H * W - f)] = 1; ms.append(m.reshape(W, H).T.copy())
    m = np.zeros(H * W, np.uint8)
    for a in range(0, H * W - 100, 100):
        m[a + 44:a + 88] = 1                                                                       # many deltas of 0 and 44
    ms.append(m.reshape(W, H).T.copy())
    for p in (0.05, 0.5, 0.95):
        ms.append((rng.random((H, W)) < p).astype(np.uint8))                                        # random fields
    if H > 40 and W > 40:
        ms += syn.masks_from_polys(syn.particle_field(rng, 12, H, W, rmin=3, rmax=20, margin=0), H, W)
    return ms


def oracle_text(masks, image_id, cats, scores, first_id):
    return ", ".join(json.dumps(coco.annotation(first_id + i, image_id, cats[i], m, scores[i]))
                     for i, m in enumerate(masks)).encode()


def oracle_text_from_runs(run_off, runs, H, W, image_id, cats, scores, first_id):
    """The same entries computed from the K6 runs alone (area, tight bbox and counts), for frames too large to unpack."""
    ro, rn = run_off.cpu().numpy(), runs.cpu().numpy()
    out = []
    for i in range(len(ro) - 1):
        r = rn[ro[i]:ro[i + 1]]
        area = int(r[:, 1].sum()) if len(r) else 0
        if area:
            f0, f1 = r[:, 0] - 1, r[:, 0] + r[:, 1] - 2
            x0, x1 = f0 // H, f1 // H
            y0 = np.where(x0 == x1, f0 - x0 * H, 0)
            y1 = np.where(x0 == x1, f1 - x1 * H, H - 1)
            bbox = [float(x0.min()), float(y0.min()), float(x1.max() - x0.min() + 1), float(y1.max() - y0.min() + 1)]
        else:
            bbox = [0.0, 0.0, 0.0, 0.0]
        out.append(json.dumps({"id": first_id + i, "image_id": image_id, "category_id": int(cats[i]),
                               "segmentation": {"size": [H, W], "counts": coco.rle_to_string(coco.counts_from_runs(r, H, W))},
                               "area": area, "bbox": bbox, "iscrowd": 0, "score": float(scores[i])}))
    return ", ".join(out).encode()


def strings_of(text):
    return [a["segmentation"]["counts"] for a in json.loads(b"[" + text + b"]")] if text else []


def assert_same_tables(dec, ref):
    assert dec.n == ref.n and dec.total_crop_words == ref.total_crop_words
    for f in ("meta", "crop_off", "bbox", "area"):
        assert torch.equal(getattr(dec, f), getattr(ref, f)), f
    t = ref.total_crop_words
    assert torch.equal(dec.crops[:t], ref.crops[:t])


def decode_strings(strings, H, W):
    raw = [s.encode() for s in strings]
    off = np.concatenate([[0], np.cumsum([len(b) for b in raw])]).astype(np.int64)
    return engine._coco_decode(b"".join(raw), off, H, W)


@pytest.mark.parametrize("H,W", [(97, 101), (50, 45), (1, 1), (64, 1), (1, 77), (33, 2)])
def test_annotations_text_and_round_trip(cuda_device, H, W):
    masks = edge_masks(H, W, H * W)
    rng = np.random.default_rng(H + W)
    n = len(masks)
    cats = rng.integers(0, 7, n).tolist()
    scores = [np.float32(v) for v in rng.random(n)]
    scores[0], scores[-1] = np.float32(1.0), np.float32(1e-7)
    src = engine.from_masks(torch.as_tensor(np.stack(masks), device=cuda_device))
    run_off, runs = engine.rle_encode(src)
    text = engine.coco_annotations_text(src, run_off, runs, 3, cats, scores, 5)
    assert text == oracle_text(masks, 3, cats, scores, 5)
    assert text == oracle_text_from_runs(run_off, runs, H, W, 3, cats, scores, 5)
    if H * W > 100:
        assert b"\\\\" in text
    dec, status = decode_strings(strings_of(text), H, W)
    assert not status.any()
    assert_same_tables(dec, engine.rle_decode(run_off, runs, H, W))
    assert np.array_equal(engine.unpack_masks(dec).cpu().numpy(), np.stack(masks))


def test_random_fields_and_ids(cuda_device):
    H, W = 300, 250
    probs, boxes, scores, _ = syn.synthetic_heads(4, 150, H, W, duplicate_frac=0.3, rmin=3, rmax=60, margin=0)
    src = engine.paste(torch.as_tensor(probs, device=cuda_device), torch.as_tensor(boxes, device=cuda_device), H, W, frames=None)
    run_off, runs = engine.rle_encode(src)
    cats = [int(v) for v in np.random.default_rng(1).integers(0, 2 ** 31 - 1, src.n)]
    sc = [np.float32(s) for s in scores]
    sc[3], sc[4] = np.float32(np.inf), np.float32(-0.0)
    text = engine.coco_annotations_text(src, run_off, runs, 2 ** 40, cats, sc, 2 ** 33)
    assert text == oracle_text(engine.unpack_masks(src).cpu().numpy(), 2 ** 40, cats, sc, 2 ** 33)
    dec, status = decode_strings(strings_of(text), H, W)
    assert not status.any()
    assert_same_tables(dec, engine.rle_decode(run_off, runs, H, W))


def test_adjacent_runs_and_zero_counts(cuda_device):
    """Strings pycocotools does not write but reads: zero counts inside, several values that leave adjacent runs."""
    H, W = 4, 3
    for counts, runs in (([0, 2, 0, 3, 7], [(1, 2), (3, 3)]), ([2, 0, 0, 4, 6], [(3, 4)]), ([12], []), ([0, 12], [(1, 12)]),
                         ([3, 0, 9], [])):
        dec, status = decode_strings([coco.rle_to_string(counts)], H, W)
        assert status.tolist() == [0]
        ro = torch.tensor([0, len(runs)], dtype=torch.int64, device=cuda_device)
        rn = torch.tensor(np.asarray(runs, np.int64).reshape(-1, 2), device=cuda_device)
        want = engine.from_masks(engine.unpack_masks(engine.rle_decode(ro, rn, H, W)))
        assert_same_tables(dec, want)


def test_malformed_strings_name_their_annotation(cuda_device, tmp_path):
    H, W = 6, 5
    good = coco.rle_to_string([3, 4, 23])
    cases = [("3 4", 1), ("3p", 1), ("3P", 2), ("", 4), ("34", 4), ("3O", 3), ("PPPPPPP0", 3)]
    strings = [good] + [s for s, _ in cases] + [good]
    _, status = decode_strings(strings, H, W)
    assert status.tolist() == [0] + [c for _, c in cases] + [0]
    assert all(status[1 + k] == coco.counts_status(s, H, W) for k, (s, _) in enumerate(cases))
    with pytest.raises(_lib.EmiaError, match="string 1: .*outside '0'..'o'"):
        engine.coco_decode(strings, H, W)
    assert engine.coco_decode([good] * 70, H, W).area.tolist() == [4] * 70
    # in a file: the annotation's id
    im = np.zeros((H, W, 3), np.uint8)
    d = {"images": [{"id": 7, "file_name": "a.png", "height": H, "width": W}],
         "annotations": [{"id": 10 + k, "image_id": 7, "category_id": 0, "segmentation": {"size": [H, W], "counts": s}}
                         for k, s in enumerate([good, good, "3P", "", good])], "categories": []}
    path = tmp_path / "c.json"
    path.write_text(json.dumps(d))
    with pytest.raises(_lib.EmiaError, match="annotation 12: counts end inside a value"):
        inf.load_coco_results(str(path), [("a.png", im)])
    for k, (field, value, why) in enumerate([("segmentation", [[1, 2, 3, 4, 5, 6]], "polygons"),
                                             ("segmentation", {"size": [H, W], "counts": [30]}, "uncompressed"),
                                             ("segmentation", {"size": [W, H], "counts": good}, "size"),
                                             ("image_id", 8, "no images entry"), ("category_id", -1, "non-negative"),
                                             ("category_id", 1.5, "non-negative")]):
        bad = json.loads(json.dumps(d))
        bad["annotations"][2] = dict(bad["annotations"][2], **{field: value, "id": 99})
        path.write_text(json.dumps(bad))
        with pytest.raises(ValueError, match=f"annotation 99: .*{why}"):
            inf.load_coco_results(str(path), [("a.png", im)])
    d["annotations"] = d["annotations"][:2]
    path.write_text(json.dumps(d))
    with pytest.raises(ValueError, match="matches no image"):
        inf.load_coco_results(str(path), [("b.png", im)])
    with pytest.raises(ValueError, match="twice"):
        inf.load_coco_results(str(path), [("a.png", im), ("a.png", im)])
    sets = inf.load_coco_results(str(path), [("a.png", im), ("b.png", np.zeros((3, 3, 3), np.uint8))])
    assert sets["a.png"].n == 2 and sets["a.png"].scores is None and sets["a.png"].classes.tolist() == [0, 0]
    assert sets["b.png"].n == 0


def test_production_size_micrograph(cuda_device):
    """A 20 k-instance 8192 x 8192 micrograph: many CTAs, long strings; the text and the round trip."""
    H = W = 8192
    probs, boxes, scores, _ = syn.synthetic_heads(100, 20000, H, W, rmin=4, rmax=30, margin=0)
    iset = engine.paste(torch.as_tensor(probs, device=cuda_device), torch.as_tensor(boxes, device=cuda_device), H, W, frames=None)
    run_off, runs = engine.rle_encode(iset)
    cats = [k % 3 for k in range(iset.n)]
    sc = [np.float32(s) for s in scores[:iset.n]]
    text = engine.coco_annotations_text(iset, run_off, runs, 1, cats, sc, 1)
    assert text == oracle_text_from_runs(run_off, runs, H, W, 1, cats, sc, 1)
    dec, status = decode_strings(strings_of(text), H, W)
    assert not status.any()
    assert_same_tables(dec, engine.rle_decode(run_off, runs, H, W))


# ---- flows ----------------------------------------------------------------------------------------------------------------------
def _flow_setup():
    imgs = [("a.png", np.random.default_rng(7).integers(0, 255, (160, 200, 3), dtype=np.uint8)),
            ("empty.png", np.zeros((40, 50, 3), np.uint8)),
            ("b.tif", np.random.default_rng(8).integers(0, 255, (150, 180, 3), dtype=np.uint8))]
    pred = syn.FakeHeadPredictor(base_seed=9, n=24)
    css = {"class_0": {"confidence_threshold": 0.3}, "class_1": {"confidence_threshold": 0.2}}
    small = adapters.determine_small_classes(adapters.calculate_average_mask_sizes([pred], [im for _, im in imgs]))
    kw = dict(visualize=False, images=imgs, predictors=[pred], thing_classes=["pore", "throat"], small_classes=small,
              spatial_rules=syn.POLYHIPES_RULES, tile_size=96, overlap_ratio=0.25, confidence_mode="manual", class_specific_settings=css)
    return imgs, kw


@pytest.mark.parametrize("options", [{}, {"shape_columns": True, "neighbours": True}])
def test_run_inference_load_and_measure(cuda_device, tmp_path, monkeypatch, options):
    imgs, kw = _flow_setup()
    captured = []
    real = engine.coco_annotations_text

    def spy(iset, run_off, runs, image_id, category_ids, scores, first_id):
        captured.append((image_id, engine.unpack_masks(iset).cpu().numpy(), list(category_ids), list(scores)))
        return real(iset, run_off, runs, image_id, category_ids, scores, first_id)
    monkeypatch.setattr(engine, "coco_annotations_text", spy)
    bar = lambda im: ("500", 0.5)                                                   # noqa: E731
    plain, with_coco = tmp_path / "plain", tmp_path / "coco"
    inf.run_inference("polyhipes_tommy", str(plain), scale_bar_fn=bar, **kw, **options)
    assert not (plain / "coco_instances.json").exists() and not captured
    inf.run_inference("polyhipes_tommy", str(with_coco), scale_bar_fn=bar, coco_json=True, **kw, **options)
    for f in ("R50_flip_results.csv", "measurements_results.csv"):
        assert (plain / f).read_bytes() == (with_coco / f).read_bytes()
    # the file is json.dumps of the oracle dict
    by_id = {c[0]: c for c in captured}
    oimgs = []
    for j, (name, im) in enumerate(imgs):
        c = by_id.get(j + 1)
        oimgs.append((name, im.shape[0], im.shape[1], list(zip(c[1], c[2], c[3])) if c else []))
    data = (with_coco / "coco_instances.json").read_bytes()
    assert data == coco.coco_file(oimgs, kw["thing_classes"])
    d = json.loads(data)
    assert len(d["annotations"]) > 10 and {c["id"] for c in d["categories"]} >= {0, 1}
    # read back: the sets of the RLE file, plus classes and scores
    sets = inf.load_coco_results(str(with_coco / "coco_instances.json"), imgs)
    rle = inf.load_rle_results(str(with_coco / "R50_flip_results.csv"), imgs)
    for j, (name, _) in enumerate(imgs):
        assert_same_tables(sets[name], rle[name])
        c = by_id.get(j + 1)
        assert sets[name].classes.tolist() == ([int(v) for v in c[2]] if c else [])
        if c:
            assert np.array_equal(sets[name].scores.cpu().numpy(), np.asarray(c[3], np.float32))
    # and measured again: the bytes run_inference wrote
    again = tmp_path / "again"
    inf.measure_coco(str(with_coco / "coco_instances.json"), str(again), images=imgs, scale_bar_fn=bar, **options)
    assert (again / "measurements_results.csv").read_bytes() == (with_coco / "measurements_results.csv").read_bytes()
    if options.get("neighbours"):
        assert (again / "neighbours_results.csv").read_bytes() == (with_coco / "neighbours_results.csv").read_bytes()
    assert len((again / "measurements_results.csv").read_bytes().splitlines()) > 3


def test_malformed_strings_past_the_first_window(cuda_device):
    """Errors after character 32, where the carries across windows (last value end, parity sums, pixels so far) decide."""
    H = W = 64
    counts = [30, 20] * 40
    counts.append(H * W - sum(counts))
    s = coco.rle_to_string(counts)
    assert len(s) > 64
    strings = [s]
    for p in range(33, len(s)):
        strings += [s[:p] + c + s[p + 1:] for c in " O0oP"] + [s[:p]]
    _, status = decode_strings(strings, H, W)
    want = [coco.counts_status(t, H, W) for t in strings]
    assert status.tolist() == want
    assert set(want) == {coco.OK, coco.BAD_CHAR, coco.OPEN_VALUE, coco.RANGE, coco.SUM}


def test_same_size_images_and_foreign_categories(cuda_device, tmp_path):
    """Several images of one frame size (decoded together, then split), one without annotations, one of another size; a category
    id with no name, a large one, and scores missing from one image."""
    H, W = 48, 40
    rng = np.random.default_rng(3)
    def disc(h, w, cy, cx, r):
        yy, xx = np.mgrid[:h, :w]
        return ((yy - cy) ** 2 + (xx - cx) ** 2 <= r * r).astype(np.uint8)
    masks = {name: [disc(h, w, *rng.integers(6, 14, 2), 5) | disc(h, w, h - 9, w - 9 - 3 * k, 4 + k) for k in range(3)]
             for name, h, w in (("a.png", H, W), ("c.png", H, W), ("d.png", 20, 30))}
    masks["b.png"] = []
    shapes = {"a.png": (H, W), "b.png": (H, W), "c.png": (H, W), "d.png": (20, 30)}
    cats = {"a.png": [0, 5, 2 ** 31 - 1], "c.png": [1, 0, 5], "d.png": [5, 5, 0]}
    d = {"images": [{"id": 10 + j, "file_name": n, "height": shapes[n][0], "width": shapes[n][1]}
                    for j, n in enumerate(("a.png", "b.png", "c.png", "d.png"))], "annotations": [],
         "categories": [{"id": 0, "name": "pore"}, {"id": 5, "name": "grain"}]}
    for j, n in enumerate(("a.png", "b.png", "c.png", "d.png")):
        for k, m in enumerate(masks[n]):
            a = coco.annotation(len(d["annotations"]) + 1, 10 + j, cats[n][k], m, np.float32(0.25 * k + 0.1))
            if n == "c.png" and k == 1:
                del a["score"]
            d["annotations"].append(a)
    path = tmp_path / "c.json"
    path.write_text(json.dumps(d))
    images = [(n, np.zeros(shapes[n] + (3,), np.uint8)) for n in ("a.png", "b.png", "c.png", "d.png")]
    sets = inf.load_coco_results(str(path), images)
    for n, _ in images:
        if masks[n]:
            assert_same_tables(sets[n], engine.from_masks(torch.as_tensor(np.stack(masks[n]), device=cuda_device)))
            assert sets[n].classes.tolist() == cats[n]
        else:
            assert sets[n].n == 0 and sets[n].classes.tolist() == []
    assert sets["a.png"].scores.tolist() == [np.float32(0.1), np.float32(0.35), np.float32(0.6)]
    assert sets["c.png"].scores is None
    out = tmp_path / "m"
    inf.measure_coco(str(path), str(out), images=images, scale_bar_fn=lambda im: ("500", 0.5))
    text = (out / "measurements_results.csv").read_bytes()
    assert b"a.png_3,2147483647,class_2147483647," in text and b",5,grain," in text and b",0,pore," in text
    bad = json.loads(json.dumps(d))
    bad["images"][1]["id"] = 10
    path.write_text(json.dumps(bad))
    with pytest.raises(ValueError, match="image id 10 appears twice"):
        inf.load_coco_results(str(path), images)
