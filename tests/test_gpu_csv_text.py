"""GPU: the result CSV files formatted on the device (engine.rle_csv_text, engine.measurements_csv_text) are byte for byte what
csv.writer writes for the rows of the host path — the " ".join of the K6 runs and the rows of inference.measure_masks — and
run_inference / remeasure_results write the files that path composes."""
import csv
import io
import re
import types

import numpy as np
import pytest
import torch

from deepemia_b200 import adapters, engine, synthetic as syn
from deepemia_b200.functions import inference as inf
from deepemia_b200.utils.measurements import record_to_dict, KEY_ORDER

pytestmark = pytest.mark.gpu

IDS = ["plain", "img,a,b", 'q"uote', "naïve µm 試料", "", " lead and trail "]


def writer_text(rows):
    buf = io.StringIO()
    csv.writer(buf).writerows(rows)
    return buf.getvalue().encode("utf-8")


def host_rle_text(run_off, runs, image_id):
    ro, rn = run_off.cpu().numpy(), runs.cpu().numpy()
    return writer_text((image_id, " ".join(str(int(v)) for v in rn[ro[i]:ro[i + 1]].reshape(-1))) for i in range(len(ro) - 1))


def shaped_masks(H, W, seed):
    """Empty, full frame, single pixels, multi-contour instances, contours of fewer than 5 vertices, specks below the area gate,
    random particles."""
    rng = np.random.default_rng(seed)
    ms = [np.zeros((H, W), np.uint8), np.ones((H, W), np.uint8)]
    for y, x in ((0, 0), (H - 1, W - 1), (H // 2, min(31, W - 1))):
        m = np.zeros((H, W), np.uint8); m[y, x] = 1; ms.append(m)
    if H >= 40 and W >= 40:
        m = np.zeros((H, W), np.uint8); m[2:12, 3:15] = 1; m[20:31, 22:36] = 1; m[35, 5] = 1; ms.append(m)   # 3 contours
        m = np.zeros((H, W), np.uint8); m[5:9, 5:9] = 1; ms.append(m)                                       # 4 vertices, area 9
        m = np.zeros((H, W), np.uint8); m[5:8, 30:32] = 1; m[15:25, 10:30] = 1; ms.append(m)                # a speck and a body
        ms += syn.masks_from_polys(syn.particle_field(rng, 12, H, W, rmin=3, rmax=min(H, W) / 4, margin=0), H, W)
    ms.append((rng.random((H, W)) < 0.3).astype(np.uint8))
    return ms


@pytest.mark.parametrize("H,W", [(97, 101), (64, 1), (1, 77), (1, 1)])
def test_rle_text_of_edge_masks(cuda_device, H, W):
    src = engine.from_masks(torch.as_tensor(np.stack(shaped_masks(H, W, H + W)), device=cuda_device))
    run_off, runs = engine.rle_encode(src)
    for image_id in IDS:
        got = engine.rle_csv_text(run_off, runs, image_id)
        assert got == host_rle_text(run_off, runs, image_id), image_id
        ids, ro, rn = engine.rle_parse_csv(b"ImageId,EncodedPixels\r\n" + got, cuda_device)
        assert ids == [image_id] * src.n and torch.equal(ro, run_off) and torch.equal(rn, runs)
    assert engine.rle_csv_text(run_off[:1], runs[:0], "x") == b""


@pytest.mark.parametrize("seed,n,H,W", [(1, 60, 256, 256), (2, 300, 720, 1000)])
def test_rle_text_of_k1_pasted_sets(cuda_device, seed, n, H, W):
    probs, boxes, _, _ = syn.synthetic_heads(seed, n, H, W, duplicate_frac=0.3, rmin=6, rmax=40, margin=0)
    src = engine.paste(torch.as_tensor(probs, device=cuda_device), torch.as_tensor(boxes, device=cuda_device), H, W, frames=None)
    run_off, runs = engine.rle_encode(src)
    assert engine.rle_csv_text(run_off, runs, IDS[seed]) == host_rle_text(run_off, runs, IDS[seed])


def host_measure_text(iset, classes, shape, um_pix, name, psum, class_names, image, contrast):
    old = inf.measure_contrast_distribution
    inf.measure_contrast_distribution = contrast
    try:
        return writer_text(inf.measure_masks(iset, classes, shape, um_pix, name, psum, class_names=class_names, original_image=image))
    finally:
        inf.measure_contrast_distribution = old


def device_measure_text(iset, classes, shape, um_pix, name, psum, class_names, image, contrast):
    old = inf.measure_contrast_distribution
    inf.measure_contrast_distribution = contrast
    try:
        return inf._measure_text(iset, classes, shape, um_pix, name, psum, class_names=class_names, original_image=image)
    finally:
        inf.measure_contrast_distribution = old


@pytest.mark.parametrize("contrast", [False, True])
@pytest.mark.parametrize("um_pix", [0.5, 1.0, 3e-7, 7.5e8])
def test_measure_text_matches_measure_masks_rows(cuda_device, contrast, um_pix):
    H, W = 97, 101
    masks = shaped_masks(H, W, 3)
    image = np.random.default_rng(4).integers(0, 255, (H, W, 3), dtype=np.uint8)
    classes = [k % 4 for k in range(len(masks))]                      # 2 and 3 lie outside class_names
    for name, psum, names in (("a.png", "500", ["pore", "throat"]), ('we,ird "x".tif', 'a,"b', ["c,1", 'q"2']),
                              ("µ.png", 0.25, None)):
        iset = engine.from_masks(torch.as_tensor(np.stack(masks), device=cuda_device))
        want = host_measure_text(iset, classes, image.shape, um_pix, name, psum, names, image, contrast)
        got = device_measure_text(iset, classes, image.shape, um_pix, name, psum, names, image, contrast)
        assert got == want
    assert b"e-" in want or b"e+" in want or um_pix in (0.5, 1.0)
    rows = list(csv.reader(io.StringIO(want.decode())))
    assert any(r[3] == "0" for r in rows) and len({r[0] for r in rows}) < len(rows)     # < 5 vertices; multi-contour instances


def test_every_layout_branch_on_the_device(cuda_device):
    """A hand-made records tensor through the kernels: NaN, +-inf, -0.0, subnormals, both sides of 1e-4 / 1e16 / 1e6, integral values,
    fewer than 5 vertices, unmeasured records."""
    f32_1e4 = float(np.float32(1e-4))
    vals = [np.nan, np.inf, -np.inf, -0.0, 0.0, 5e-324, 2.2250738585072014e-308, 1e-45, 1e-4, np.nextafter(1e-4, 0), f32_1e4,
            float(np.nextafter(np.float32(1e-4), np.float32(1))), 1e16, np.nextafter(1e16, 0), 999999.94, 1e6, 123456789.0, 3.0,
            -1.5, 1e300, 1e39, 0.1, 2.0 ** 60, 1 / 3]
    rng = np.random.default_rng(5)
    R = 64
    rec = rng.choice(np.array(vals), (R, 16))
    rec[:, engine.REC_NVERT] = rng.choice([3.0, 4.0, 5.0, 100.0], R)
    rec[:, engine.REC_MEASURED] = rng.choice([1.0, 1.0, 1.0, 0.0], R)
    n = 20
    rec_inst = np.sort(rng.integers(0, n, R)).astype(np.int32)
    contrast = rng.choice(np.array(vals[:12] + [np.nan] * 4), (n, 3))
    contrast[3] = np.nan
    iset = types.SimpleNamespace(records=torch.as_tensor(rec, device=cuda_device), rec_inst=torch.as_tensor(rec_inst, device=cuda_device),
                                 n_records=R, n=n, device=cuda_device)
    fields = [(0, "pore"), ("7", "x,y")]
    cidx = rng.integers(0, 2, n)
    for con in (None, contrast):
        with np.errstate(over="ignore"):
            rows = []
            for r in range(R):
                if rec[r, engine.REC_MEASURED] != 1.0:
                    continue
                m = record_to_dict(rec[r])
                k = int(rec_inst[r])
                if con is not None:
                    m["contrast_d10"], m["contrast_d50"], m["contrast_d90"] = (None if np.isnan(v) else np.float64(v) for v in con[k])
                rows.append([f"im_{k + 1}", *fields[cidx[k]]] + [m[key] for key in KEY_ORDER] + ["p", "im"])
        assert engine.measurements_csv_text(iset, "im", "p", cidx, fields, con) == writer_text(rows)
    with pytest.raises(ValueError, match="class_idx"):
        engine.measurements_csv_text(iset, "im", "p", np.full(n, 2), fields)


@pytest.mark.parametrize("contrast", [False, True])
def test_run_inference_and_remeasure_files_match_the_host_path(cuda_device, tmp_path, monkeypatch, contrast):
    imgs = [("a,1.png", np.random.default_rng(7).integers(0, 255, (160, 200, 3), dtype=np.uint8)),
            ("b.tif", np.random.default_rng(8).integers(0, 255, (150, 180, 3), dtype=np.uint8))]
    pred = syn.FakeHeadPredictor(base_seed=9, n=24)
    small = adapters.determine_small_classes(adapters.calculate_average_mask_sizes([pred], [im for _, im in imgs]))
    css = {"class_0": {"confidence_threshold": 0.3}, "class_1": {"confidence_threshold": 0.2}}
    kw = dict(tile_size=96, overlap_ratio=0.25, confidence_mode="manual", class_specific_settings=css, spatial_rules=syn.POLYHIPES_RULES)
    bar = lambda im: ('5"0,0', 0.5)                                   # noqa: E731
    # the host path composes its rows from the same per-image inputs: the runs K6 gives, and measure_masks over the final set
    host_rle, host_rows = [], []
    dev_rle_text, dev_measure_text = engine.rle_csv_text, inf._measure_text

    def rle_text(run_off, runs, image_id):
        ro, rn = run_off.cpu().numpy(), runs.cpu().numpy()
        host_rle.extend((image_id, " ".join(str(int(v)) for v in rn[ro[i]:ro[i + 1]].reshape(-1))) for i in range(len(ro) - 1))
        return dev_rle_text(run_off, runs, image_id)

    def measure_text(iset, classes, shape, um_pix, name, psum, class_names=None, original_image=None):
        host_rows.extend(inf.measure_masks(iset, classes, shape, um_pix, name, psum, class_names=class_names,
                                           original_image=original_image))
        return dev_measure_text(iset, classes, shape, um_pix, name, psum, class_names=class_names, original_image=original_image)

    monkeypatch.setattr(engine, "rle_csv_text", rle_text)
    monkeypatch.setattr(inf, "_measure_text", measure_text)
    old = inf.measure_contrast_distribution
    inf.measure_contrast_distribution = contrast
    try:
        inf.run_inference("polyhipes_tommy", str(tmp_path / "run"), visualize=False, images=imgs, predictors=[pred],
                          thing_classes=["pore", "throat"], small_classes=small, scale_bar_fn=bar, **kw)
        monkeypatch.undo()
        rle_want = writer_text([["ImageId", "EncodedPixels"]] + host_rle)
        meas_want = writer_text([inf.CSV_HEADER] + host_rows)
        assert (tmp_path / "run" / "R50_flip_results.csv").read_bytes() == rle_want
        assert (tmp_path / "run" / "measurements_results.csv").read_bytes() == meas_want
        assert len(meas_want.splitlines()) > 10
        bar2 = lambda im: (0.125, 3e-7)                               # noqa: E731
        inf.remeasure_results("polyhipes_tommy", str(tmp_path / "run"), str(tmp_path / "again"), images=imgs, scale_bar_fn=bar2)
        old_rows = list(csv.reader(io.StringIO(meas_want.decode())))
        class_of = {r[0]: (r[1], r[2]) for r in old_rows[1:]}
        sets = inf.load_rle_results(str(tmp_path / "run" / "R50_flip_results.csv"), imgs)
        rows = []
        for name, image in imgs:
            got = inf.measure_masks(sets[name], [0] * sets[name].n, image.shape, 3e-7, name, 0.125, original_image=image)
            for r in got:
                r[1], r[2] = class_of[r[0]]
            rows += got
        assert (tmp_path / "again" / "measurements_results.csv").read_bytes() == writer_text([inf.CSV_HEADER] + rows)
        # an instance with a measured contour but no row in the old file: the same error as before
        (tmp_path / "cut").mkdir()
        (tmp_path / "cut" / "R50_flip_results.csv").write_bytes((tmp_path / "run" / "R50_flip_results.csv").read_bytes())
        first = old_rows[1][0]
        (tmp_path / "cut" / "measurements_results.csv").write_bytes(writer_text([inf.CSV_HEADER] + [r for r in old_rows[1:] if r[0] != first]))
        with pytest.raises(ValueError, match=f"remeasure_results: {re.escape(first)} has a measured contour but no row"):
            inf.remeasure_results("polyhipes_tommy", str(tmp_path / "cut"), str(tmp_path / "x"), images=imgs, scale_bar_fn=bar2)
    finally:
        inf.measure_contrast_distribution = old


def test_production_size_micrograph(cuda_device):
    """A 20 k-instance 8192 x 8192 micrograph: many CTAs, long lines and several contours per instance."""
    H = W = 8192
    probs, boxes, _, _ = syn.synthetic_heads(100, 20000, H, W, rmin=4, rmax=30, margin=0)
    iset = engine.paste(torch.as_tensor(probs, device=cuda_device), torch.as_tensor(boxes, device=cuda_device), H, W, frames=None)
    run_off, runs = engine.rle_encode(iset)
    assert engine.rle_csv_text(run_off, runs, "micrograph") == host_rle_text(run_off, runs, "micrograph")
    classes = [k % 3 for k in range(iset.n)]
    want = host_measure_text(iset, classes, (H, W), 0.5, "micrograph.tif", "500", ["pore", "throat"], None, False)
    got = device_measure_text(iset, classes, (H, W), 0.5, "micrograph.tif", "500", ["pore", "throat"], None, False)
    assert got == want and len(want.splitlines()) > 15000
