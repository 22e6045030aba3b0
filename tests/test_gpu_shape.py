"""GPU: the shape descriptors (engine.shape_descriptors / shape_list, kernel k_contour_shape) against oracle/shape.py, the K5 work
order, and the opt-in shape columns of measurements_results.csv through measurements_csv_text, run_inference and remeasure_results."""
import csv
import io

import numpy as np
import pytest
import torch

from deepemia_b200 import adapters, engine, synthetic as syn
from deepemia_b200.functions import inference as inf
from deepemia_b200.utils import measurements as um
from oracle import shape as oshape

pytestmark = pytest.mark.gpu

ANGLE = 7                                             # Feret angle: CUDA's atan2 is not glibc's; within 1e-12 degrees


def writer_text(rows):
    buf = io.StringIO()
    csv.writer(buf).writerows(rows)
    return buf.getvalue().encode("utf-8")


def masks(H, W, seed):
    """Multi-contour instances, specks below the area gate, a full frame, squares (Feret ties) and random particles."""
    rng = np.random.default_rng(seed)
    ms = [np.ones((H, W), np.uint8)]
    m = np.zeros((H, W), np.uint8); m[2:12, 3:15] = 1; m[20:31, 22:36] = 1; m[35, 5] = 1; m[40:42, 50:52] = 1; ms.append(m)
    m = np.zeros((H, W), np.uint8); m[5:8, 30:32] = 1; m[15:25, 10:30] = 1; m[60:61, 10:70] = 1; ms.append(m)
    m = np.zeros((H, W), np.uint8); m[50:80, 50:80] = 1; ms.append(m)
    ms += syn.masks_from_polys(syn.particle_field(rng, 40, H, W, rmin=3, rmax=min(H, W) / 4, margin=0), H, W)
    ms.append((rng.random((H, W)) < 0.3).astype(np.uint8))
    return ms


def check_against_oracle(iset, um_pix):
    shape = engine.shape_descriptors(iset)
    assert shape.shape == (iset.n_records, engine.SHAPE_FIELDS) and shape.dtype == torch.float64
    got = shape.cpu().numpy()
    rec = iset.records.cpu().numpy()
    contours = [c for cl in engine.contours_to_host(iset) for c in cl]
    assert len(contours) == len(got)
    measured = rec[:, engine.REC_MEASURED] == 1.0
    assert np.isnan(got[~measured]).all()
    want = np.array([oshape.shape_descriptors(c, um_pix) for c, m in zip(contours, measured) if m])
    exact = [f for f in range(engine.SHAPE_FIELDS) if f != ANGLE]
    bad = np.nonzero(~(got[measured][:, exact] == want[:, exact]).all(1))[0]
    assert len(bad) == 0, (len(bad), got[measured][bad[0]].tolist(), want[bad[0]].tolist())
    assert np.abs(got[measured][:, ANGLE] - want[:, ANGLE]).max() <= 1e-12
    return measured


@pytest.mark.parametrize("um_pix", [1.0, 0.37])
def test_from_masks_matches_oracle(cuda_device, um_pix):
    H, W = 150, 170
    iset = engine.from_masks(torch.as_tensor(np.stack(masks(H, W, 3)), device=cuda_device))
    engine.measure(iset, um_pix=um_pix, min_area=engine.default_min_area(H, W))
    measured = check_against_oracle(iset, um_pix)
    cnt = np.diff(iset.cont_off.cpu().numpy())
    assert (~measured).any() and (cnt > 1).sum() >= 3                          # NaN rows; multi-contour instances


@pytest.mark.parametrize("seed,n,H,W", [(1, 300, 720, 1000), (2, 3000, 2048, 2048)])
def test_k1_pasted_sets_match_oracle(cuda_device, seed, n, H, W):
    probs, boxes, _, _ = syn.synthetic_heads(seed, n, H, W, duplicate_frac=0.3, rmin=3, rmax=40, margin=0)
    iset = engine.paste(torch.as_tensor(probs, device=cuda_device), torch.as_tensor(boxes, device=cuda_device), H, W, frames=None)
    engine.measure(iset, um_pix=0.5, min_area=engine.default_min_area(H, W))
    check_against_oracle(iset, 0.5)


def test_work_order_gives_the_same_values(cuda_device, monkeypatch):
    """The same contours gathered into a list past MEASURE_ORDER_MIN_SLOTS (the K5 work order) give the same values per record."""
    H = W = 2048
    probs, boxes, _, _ = syn.synthetic_heads(5, 2000, H, W, rmin=3, rmax=40, margin=0)
    iset = engine.paste(torch.as_tensor(probs, device=cuda_device), torch.as_tensor(boxes, device=cuda_device), H, W, frames=None)
    engine.measure(iset, um_pix=0.5)
    small = engine.shape_descriptors(iset).cpu().numpy().view(np.int64)
    rng = np.random.default_rng(6)
    L = engine.MEASURE_ORDER_MIN_SLOTS + 777
    idx = rng.integers(0, iset.n, L)
    groups = engine.groups_from_lists([idx[:L // 2].tolist(), idx[L // 2:].tolist()], cuda_device)
    assert groups.total_cap >= engine.MEASURE_ORDER_MIN_SLOTS and engine.MEASURE_ORDER
    meas = engine.measure_list(iset, groups, um_pix=0.5)
    launches = []
    for on in (True, False):
        monkeypatch.setattr(engine, "MEASURE_ORDER", on)
        c0 = engine.LAUNCHES["count"]
        vals = engine.shape_list(iset, meas, 0.5).cpu().numpy().view(np.int64)
        launches.append(engine.LAUNCHES["count"] - c0)
        big = vals if on else big
        assert np.array_equal(vals, big)
    assert launches[0] - launches[1] == 2                                     # the ordered run launches the two order kernels
    cont_off = iset.cont_off.cpu().numpy()
    want = np.concatenate([small[cont_off[i]:cont_off[i + 1]] for i in idx])
    assert big.shape == want.shape and np.array_equal(big, want)


def test_explicit_contour_mirror(cuda_device):
    c = np.array([[10, 20], [10, 60], [40, 20]], np.int32).reshape(-1, 1, 2)
    got = um.shape_descriptors(c, um_pix=2.0)
    assert list(got) == um.SHAPE_HEADER == oshape.SHAPE_HEADER
    want = oshape.shape_descriptors(c, 2.0)
    assert [got[k] for k in um.SHAPE_HEADER if k != "Feret angle"] == [v for k, v in zip(um.SHAPE_HEADER, want) if k != "Feret angle"]
    assert abs(got["Feret angle"] - want[ANGLE]) <= 1e-12


def measure_text(iset, classes, shape, um_pix, name, psum, class_names, image, contrast, device):
    old = inf.measure_contrast_distribution
    inf.measure_contrast_distribution = contrast
    try:
        if device:
            return inf._measure_text(iset, classes, shape, um_pix, name, psum, class_names=class_names, original_image=image,
                                     shape_columns=True)
        return writer_text(inf.measure_masks(iset, classes, shape, um_pix, name, psum, class_names=class_names, original_image=image,
                                             shape_columns=True))
    finally:
        inf.measure_contrast_distribution = old


@pytest.mark.parametrize("contrast", [False, True])
@pytest.mark.parametrize("um_pix", [0.5, 3e-7])
def test_csv_text_with_shape_matches_measure_masks_rows(cuda_device, contrast, um_pix):
    H, W = 150, 170
    ms = masks(H, W, 4)
    image = np.random.default_rng(4).integers(0, 255, (H, W, 3), dtype=np.uint8)
    classes = [k % 3 for k in range(len(ms))]
    for name, psum, names in (("a.png", "500", ["pore", "throat"]), ('we,ird "x".tif', 'a,"b', None)):
        iset = engine.from_masks(torch.as_tensor(np.stack(ms), device=cuda_device))
        want = measure_text(iset, classes, image.shape, um_pix, name, psum, names, image, contrast, False)
        got = measure_text(iset, classes, image.shape, um_pix, name, psum, names, image, contrast, True)
        assert got == want
    rows = list(csv.reader(io.StringIO(want.decode())))
    assert len(rows) > 20 and all(len(r) == 30 for r in rows)
    iset = engine.from_masks(torch.as_tensor(np.stack(ms), device=cuda_device))
    engine.measure(iset)
    with pytest.raises(ValueError, match="shape"):
        engine.measurements_csv_text(iset, "a", "1", [0] * iset.n, [(0, "x")], shape=engine.shape_descriptors(iset)[1:])


def test_run_inference_and_remeasure_with_shape_columns(cuda_device, tmp_path):
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
    inf.run_inference("polyhipes_tommy", str(tmp_path / "shape"), shape_columns=True, **common)
    plain = (tmp_path / "plain" / "measurements_results.csv").read_bytes()
    shaped = (tmp_path / "shape" / "measurements_results.csv").read_bytes()
    assert (tmp_path / "plain" / "R50_flip_results.csv").read_bytes() == (tmp_path / "shape" / "R50_flip_results.csv").read_bytes()
    pl, sl = plain.split(b"\r\n"), shaped.split(b"\r\n")
    assert len(pl) == len(sl) > 10
    for a, b in zip(pl, sl):
        if a:
            assert b.startswith(a + b",") and len(next(csv.reader([b.decode()]))) == 30
    assert next(csv.reader([sl[0].decode()])) == inf.CSV_HEADER + um.SHAPE_HEADER
    # re-measuring the default run, and the run that already has the shape columns, with the same scale bar
    for src in ("plain", "shape"):
        inf.remeasure_results("polyhipes_tommy", str(tmp_path / src), str(tmp_path / (src + "_again")), images=imgs, scale_bar_fn=bar,
                              shape_columns=True)
        assert (tmp_path / (src + "_again") / "measurements_results.csv").read_bytes() == shaped
    inf.remeasure_results("polyhipes_tommy", str(tmp_path / "shape"), str(tmp_path / "back"), images=imgs, scale_bar_fn=bar)
    assert (tmp_path / "back" / "measurements_results.csv").read_bytes() == plain
