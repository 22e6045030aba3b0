"""GPU: reading the RLE wire format back — R50_flip_results.csv text -> runs (engine.rle_parse_csv) -> instances (engine.rle_decode),
bit for bit the tables of from_masks; mask_utils.rle_decoding; load_rle_results / remeasure_results against a second run_inference."""
import csv
import io

import numpy as np
import pytest
import torch

from deepemia_b200 import _lib, adapters, engine, synthetic as syn
from deepemia_b200.functions import inference as inf
from deepemia_b200.utils import mask_utils

pytestmark = pytest.mark.gpu


def np_decode(vals, H, W):
    """Reference decoder: column-major, 1-indexed (start, length) pairs -> H x W 0/1 mask."""
    flat = np.zeros(H * W, np.uint8)
    for s, n in np.asarray(vals, np.int64).reshape(-1, 2):
        flat[s - 1:s - 1 + n] = 1
    return flat.reshape(W, H).T


def edge_masks(H, W, seed):
    rng = np.random.default_rng(seed)
    ms = []
    m = np.zeros((H, W), np.uint8); m[0, 3:9] = 1; m[H - 1, 5:40] = 1; ms.append(m)            # rows 0 and H-1
    m = np.zeros((H, W), np.uint8); m[:, 30:35] = 1; ms.append(m)                               # whole columns (one run)
    m = np.zeros((H, W), np.uint8); m[:, W - 3:] = 1; m[:H // 2, W - 4] = 1; ms.append(m)       # columns up to the last partial word
    m = np.zeros((H, W), np.uint8); m[H - 1, 10] = 1; m[0, 11] = 1; ms.append(m)                # a run wrapping into the next column
    for y, x in ((0, 0), (H - 1, W - 1), (H // 2, 31), (7, 32), (H - 1, 0), (0, W - 1)):      # single pixels
        m = np.zeros((H, W), np.uint8); m[y, x] = 1; ms.append(m)
    ms.append(np.ones((H, W), np.uint8))                                                        # the full frame
    ms.append(np.zeros((H, W), np.uint8))                                                       # empty
    ms.append((rng.random((H, W)) < 0.5).astype(np.uint8))                                     # many short runs
    ms += syn.masks_from_polys(syn.particle_field(rng, 30, H, W, rmin=3, rmax=30, margin=0), H, W)
    ms.append(np.zeros((H, W), np.uint8))
    return ms


def assert_canonical(dec, src):
    """dec has exactly the tables of from_masks(unpack_masks(src))."""
    ref = engine.from_masks(engine.unpack_masks(src))
    assert dec.n == ref.n and dec.total_crop_words == ref.total_crop_words
    for f in ("meta", "crop_off", "bbox", "area"):
        assert torch.equal(getattr(dec, f), getattr(ref, f)), f
    t = ref.total_crop_words
    assert torch.equal(dec.crops[:t], ref.crops[:t])


@pytest.mark.parametrize("H,W", [(97, 101), (64, 45), (1, 77), (83, 1)])
def test_round_trip_bit_exact(cuda_device, H, W):
    masks = edge_masks(H, W, H * W) if H > 8 and W > 40 else \
        [(np.random.default_rng(k).random((H, W)) < 0.4).astype(np.uint8) for k in range(6)] + [np.ones((H, W), np.uint8),
                                                                                               np.zeros((H, W), np.uint8)]
    src = engine.from_masks(torch.as_tensor(np.stack(masks), device=cuda_device))
    run_off, runs = engine.rle_encode(src)
    dec = engine.rle_decode(run_off, runs, H, W)
    assert_canonical(dec, src)
    got = engine.unpack_masks(dec).cpu().numpy()
    ro, rn = run_off.cpu().numpy(), runs.cpu().numpy()
    for i, m in enumerate(masks):
        assert np.array_equal(got[i], np_decode(rn[ro[i]:ro[i + 1]], H, W)), i
        assert np.array_equal(got[i], m), i


@pytest.mark.parametrize("seed,n,H,W", [(1, 60, 256, 256), (2, 200, 720, 1000), (3, 40, 300, 250)])
def test_decode_of_k1_pasted_sets(cuda_device, seed, n, H, W):
    probs, boxes, _, _ = syn.synthetic_heads(seed, n, H, W, duplicate_frac=0.3, rmin=6, rmax=40, margin=0)
    src = engine.paste(torch.as_tensor(probs, device=cuda_device), torch.as_tensor(boxes, device=cuda_device), H, W, frames=None)
    run_off, runs = engine.rle_encode(src)
    assert_canonical(engine.rle_decode(run_off, runs, H, W), src)


def test_decode_rejects_bad_runs_and_frames(cuda_device):
    def dec(vals_list, H=10, W=7):
        ro = torch.tensor(np.cumsum([0] + [len(v) // 2 for v in vals_list]), dtype=torch.int64, device=cuda_device)
        rn = torch.tensor(np.asarray(sum(vals_list, []), np.int64).reshape(-1, 2), device=cuda_device)
        return engine.rle_decode(ro, rn, H, W)
    assert dec([[3, 4, 7, 2], []]).area.tolist() == [6, 0]                   # adjacent runs are fine; an empty mask
    for vals, why in (([0, 3], "start < 1"), ([4, 0], "length < 1"), ([69, 3], "past pixel"),
                      ([10, 5, 3, 2], "unsorted"), ([10, 5, 12, 2], "overlapping")):
        with pytest.raises(_lib.EmiaError, match=f"instance 1: .*{why}"):
            dec([[1, 2], vals])
    for H, W in ((0, 5), (5, 65536)):
        with pytest.raises(_lib.EmiaError, match="65535"):
            dec([[1, 2]], H, W)


def _csv_text(ids, ro, rn):
    """The rows exactly as run_inference writes them (csv.writer, \\r\\n line ends)."""
    buf = io.StringIO()
    w = csv.writer(buf)
    w.writerow(["ImageId", "EncodedPixels"])
    w.writerows((ids[i], " ".join(str(int(v)) for v in rn[ro[i]:ro[i + 1]].reshape(-1))) for i in range(len(ids)))
    return buf.getvalue().encode()


def test_text_parses_to_the_k6_runs(cuda_device):
    H, W = 97, 101
    masks = edge_masks(H, W, 5)
    src = engine.from_masks(torch.as_tensor(np.stack(masks), device=cuda_device))
    run_off, runs = engine.rle_encode(src)
    ro, rn = run_off.cpu().numpy(), runs.cpu().numpy()
    ids = [("img,a,b" if i % 3 == 0 else 'q"uote' if i % 3 == 1 else "plain") for i in range(len(masks))]
    text = _csv_text(ids, ro, rn)
    assert b'"img,a,b",' in text and b'"q""uote",' in text and b"\r\n" in text and b"plain,\r\n" in text      # quoted ids, empty masks
    for variant in (text, text.replace(b"\r\n", b"\n"), text.rstrip(b"\r\n"),
                    text.replace(b" ", b"  ").replace(b"\r\n", b"  \r\n\r\n \r\n")):      # repeated / trailing blanks, blank lines
        got_ids, got_off, got_runs = engine.rle_parse_csv(variant, cuda_device)
        assert got_ids == ids
        assert torch.equal(got_off, run_off) and torch.equal(got_runs, runs)
    assert_canonical(engine.rle_decode(*engine.rle_parse_csv(text, cuda_device)[1:], H, W), src)
    big = _csv_text(["x"] * 3000, np.arange(3001) * 40, np.arange(1, 240001, dtype=np.int64) * 3)   # many text chunks
    ids2, off2, runs2 = engine.rle_parse_csv(big, cuda_device)
    assert len(ids2) == 3000 and off2.tolist() == (np.arange(3001) * 20).tolist()
    assert torch.equal(runs2.reshape(-1).cpu(), torch.arange(1, 240001, dtype=torch.int64)[:runs2.numel()] * 3)
    assert engine.rle_parse_csv(b"ImageId,EncodedPixels\r\n", cuda_device)[0] == []


@pytest.mark.parametrize("line,why", [("a,1 2 x3 4", "character other than a digit"), ("a,1 2 3", "odd number"),
                                      ("a,1 " + "1" * 19, "more than 18 digits"), ("a 1 2", "no comma"), ("a,1 2;", "character")])
def test_malformed_text_names_its_line(cuda_device, line, why):
    text = f"ImageId,EncodedPixels\r\na,1 2 5 1\r\n\r\n{line}\r\na,3 1\r\n".encode()
    with pytest.raises(_lib.EmiaError, match=f"line 4: .*{why}"):
        engine.rle_parse_csv(text, cuda_device)
    with pytest.raises(_lib.EmiaError, match="line 1: header"):
        engine.rle_parse_csv(b"Id,Pixels\r\na,1 2\r\n", cuda_device)


@pytest.mark.parametrize("enc,why", [("0 2", "start < 1"), ("5 0", "length < 1"), ("60 2", "past pixel"), ("60 1", None),
                                     ("9 2 3 1", "unsorted"), ("9 2 10 4", "overlapping"), ("9 2 11 4", None)])
def test_bad_runs_name_their_line(cuda_device, tmp_path, enc, why):
    path = tmp_path / "R50_flip_results.csv"
    path.write_bytes(f"ImageId,EncodedPixels\r\na,1 2 5 1\r\nb,4 4\r\n\r\na,{enc}\r\n".encode())
    images = [("a.png", np.zeros((6, 10, 3), np.uint8)), ("b.png", np.zeros((8, 9, 3), np.uint8))]
    if why is None:
        sets = inf.load_rle_results(str(path), images)
        assert sets["a.png"].n == 2 and sets["b.png"].n == 1 and sets["b.png"].area.tolist() == [4]
    else:
        with pytest.raises(_lib.EmiaError, match=f"line 5: .*{why}"):
            inf.load_rle_results(str(path), images)


def test_rle_decoding_inverts_rle_encoding(cuda_device):
    H, W = 97, 101
    for m in edge_masks(H, W, 9):
        enc = mask_utils.rle_encoding(m)
        assert np.array_equal(mask_utils.rle_decoding(enc, m.shape), m)
        assert np.array_equal(mask_utils.rle_decoding(" ".join(map(str, enc)), (H, W)), m)


def test_load_rle_results_errors(cuda_device, tmp_path):
    path = tmp_path / "R50_flip_results.csv"
    path.write_bytes(b"ImageId,EncodedPixels\r\na,1 2\r\nc,1 1\r\n")
    im = np.zeros((5, 5, 3), np.uint8)
    with pytest.raises(_lib.EmiaError, match="line 3: ImageId 'c' matches no image"):
        inf.load_rle_results(str(path), [("a.png", im)])
    with pytest.raises(ValueError, match="share the ImageId 'a'"):
        inf.load_rle_results(str(path), [("a.png", im), ("a.tif", im), ("c.png", im)])
    sets = inf.load_rle_results(str(path), [("a.png", im), ("c.tif", im), ("d.png", np.zeros((7, 3, 3), np.uint8))])
    assert [sets[k].n for k in ("a.png", "c.tif", "d.png")] == [1, 1, 0]


@pytest.mark.parametrize("contrast", [False, True])
def test_remeasure_equals_a_run_with_the_new_scale(cuda_device, tmp_path, contrast):
    """run_inference without a scale (psum "0", um_pix 1.0), then remeasure_results with the scale bar: the same bytes as a run
    made with that scale bar in the first place."""
    imgs = [("a.png", np.random.default_rng(7).integers(0, 255, (160, 200, 3), dtype=np.uint8)),
            ("b.tif", np.random.default_rng(8).integers(0, 255, (150, 180, 3), dtype=np.uint8))]
    pred = syn.FakeHeadPredictor(base_seed=9, n=24)
    cfg = {"inference_settings": {"confidence_mode": "manual", "tile_settings": {"tile_size": 96, "overlap_ratio": 0.25},
                                  "class_specific_settings": {"class_0": {"confidence_threshold": 0.3}, "class_1": {"confidence_threshold": 0.2}}}}
    small = adapters.determine_small_classes(adapters.calculate_average_mask_sizes([pred], [im for _, im in imgs]))
    kw = dict(visualize=False, images=imgs, predictors=[pred], thing_classes=["pore", "throat"], small_classes=small,
              spatial_rules=syn.POLYHIPES_RULES, tile_size=96, overlap_ratio=0.25, confidence_mode="manual",
              class_specific_settings=cfg["inference_settings"]["class_specific_settings"])
    unscaled, scaled, again = tmp_path / "unscaled", tmp_path / "scaled", tmp_path / "again"
    inf.run_inference("polyhipes_tommy", str(unscaled), scale_bar_fn=lambda im: ("0", 1.0), **kw)
    old = inf.measure_contrast_distribution
    inf.measure_contrast_distribution = contrast
    try:
        inf.run_inference("polyhipes_tommy", str(scaled), scale_bar_fn=lambda im: ("500", 0.5), **kw)
        with pytest.raises(ValueError):
            inf.remeasure_results("polyhipes_tommy", str(unscaled), str(unscaled), images=imgs, scale_bar_fn=lambda im: ("500", 0.5))
        inf.remeasure_results("polyhipes_tommy", str(unscaled), str(again), images=imgs, scale_bar_fn=lambda im: ("500", 0.5))
    finally:
        inf.measure_contrast_distribution = old
    want = (scaled / "measurements_results.csv").read_bytes()
    assert (again / "measurements_results.csv").read_bytes() == want
    assert want != (unscaled / "measurements_results.csv").read_bytes() and len(want.splitlines()) > 3
    # the decoded instances are the ones whose rows were written: same count per image as the RLE file
    rle = list(csv.reader(open(unscaled / "R50_flip_results.csv")))
    sets = inf.load_rle_results(str(unscaled / "R50_flip_results.csv"), imgs)
    assert sum(s.n for s in sets.values()) == len(rle) - 1
    for name, im in imgs:
        rows = [r[1] for r in rle[1:] if r[0] == name.rsplit(".", 1)[0]]
        got = engine.unpack_masks(sets[name]).cpu().numpy()
        for k, enc in enumerate(rows):
            assert np.array_equal(got[k], np_decode([int(v) for v in enc.split()], *im.shape[:2]))
