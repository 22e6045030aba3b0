"""GPU: COCO segm evaluation on the device (engine.coco_evaluate, functions.inference.evaluate_coco) against oracle/cocoeval.py,
the numpy restatement of pycocotools' COCOeval: precision, recall and stats exactly equal, the CSV byte for byte, the flows and
the error paths."""
import json

import numpy as np
import pytest

from deepemia_b200 import _lib, synthetic as syn
from deepemia_b200.functions import inference as inf
from oracle import cocoeval as ce

pytestmark = pytest.mark.gpu


def write(tmp_path, name, d):
    p = tmp_path / name
    p.write_text(json.dumps(d))
    return str(p)


def check(tmp_path, gt, dt, **kw):
    want = ce.evaluate(gt, dt, **kw)
    got = inf.evaluate_coco(write(tmp_path, "gt.json", gt), write(tmp_path, "dt.json", dt), str(tmp_path / "out"), **kw)
    assert np.array_equal(got["precision"], want["precision"])
    assert np.array_equal(got["recall"], want["recall"])
    assert got["stats"] == want["stats"] and got["per_category"] == want["per_category"]
    assert (tmp_path / "out" / "coco_eval_results.csv").read_bytes() == want["csv"]
    return got


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_synthetic_against_oracle(cuda_device, tmp_path, seed):
    """Shifted / dilated / eroded masks, dropped, duplicate and spurious particles, tied scores, three categories, crowd GTs,
    `area` fields unlike the popcount, an image without GT, one without detections, two frame sizes."""
    gt, dt = ce.synthetic_case(seed, [(256, 256), (256, 256), (200, 300), (256, 256), (200, 300)], [60, 0, 40, 50, 30], n_cats=3,
                                crowd_frac=0.1, score_levels=8)
    dt["annotations"] = [a for a in dt["annotations"] if a["image_id"] != gt["images"][0]["id"]]     # the last image: no detections
    for a in gt["annotations"][5:60:9]:                          # GTs without `area`: the popcount
        del a["area"]
    # a GT of id 0 with two exact copies among the detections: dtm == 0 counts as no match.  Its `area` field puts it in the
    # medium range while the detections' popcount areas are small: at "small" it is an ignored GT matched by in-range detections
    g0 = gt["annotations"][3]
    g0.update(id=0, area=5000.0, iscrowd=0)
    img0 = next(e for e in dt["images"] if e["id"] == g0["image_id"])
    assert img0 and g0["segmentation"]["size"] == [img0["height"], img0["width"]]
    for sc in (0.99, 0.05):
        dt["annotations"].append({"id": len(dt["annotations"]) + 1, "image_id": g0["image_id"], "category_id": g0["category_id"],
                                  "segmentation": dict(g0["segmentation"]), "score": sc})
    got = check(tmp_path, gt, dt)
    assert (got["precision"] > 0).any()
    check(tmp_path, gt, dt, max_dets=(1, 3, 5))                 # truncation inside images


def test_bbox_area_and_categories_by_name(cuda_device, tmp_path):
    gt, dt = ce.synthetic_case(4, [(128, 128), (96, 160)], [30, 25], n_cats=2)
    for a in dt["annotations"]:                                 # loadRes' bbox branch: area = w * h
        a["bbox"] = [0.0, 0.0, float(a["id"] % 40), 33.0]
    check(tmp_path, gt, dt)
    dt["categories"] = [{"id": c["id"] - 1, "name": c["name"]} for c in dt["categories"]]
    for a in dt["annotations"]:
        a["category_id"] -= 1
    check(tmp_path, gt, dt, match_categories="name")


@pytest.mark.parametrize("max_dets", [(1, 10, 100), (100, 1000, 30000)])
def test_micrograph_scale(cuda_device, tmp_path, max_dets):
    """The 8192 x 8192 micrograph with ~20 k instances."""
    gt, dt = ce.synthetic_case(10, [(8192, 8192)], 20000, n_cats=1, rmin=4, rmax=30, crowd_frac=0.01)
    got = check(tmp_path, gt, dt, max_dets=max_dets)
    assert got["stats"][0] > 0


def test_run_inference_file_against_itself(cuda_device, tmp_path):
    imgs, kw = _flow_setup()
    inf.run_inference("polyhipes_tommy", str(tmp_path / "run"), scale_bar_fn=lambda im: ("500", 0.5), coco_json=True, **kw)
    path = str(tmp_path / "run" / "coco_instances.json")
    d = json.loads(open(path).read())
    got = inf.evaluate_coco(path, path)
    want = ce.evaluate(d, d)
    assert got["stats"] == want["stats"] and np.array_equal(got["precision"], want["precision"])
    assert got["stats"][0] == pytest.approx(1.0, abs=1e-15) and got["stats"][8] == pytest.approx(1.0, abs=1e-15)
    # a ground truth with 1-based category ids and the same names
    g1 = dict(d, categories=[{"id": c["id"] + 1, "name": c["name"]} for c in d["categories"]],
              annotations=[dict(a, category_id=a["category_id"] + 1) for a in d["annotations"]])
    p1 = write(tmp_path, "gt1.json", g1)
    by_name = inf.evaluate_coco(p1, path, match_categories="name")
    assert by_name["stats"] == got["stats"]
    by_id = inf.evaluate_coco(p1, path)
    assert by_id["stats"] == ce.evaluate(g1, d)["stats"] and by_id["stats"] != got["stats"]


def _flow_setup():
    from deepemia_b200 import adapters
    imgs = [("a.png", np.random.default_rng(7).integers(0, 255, (160, 200, 3), dtype=np.uint8)),
            ("b.tif", np.random.default_rng(8).integers(0, 255, (150, 180, 3), dtype=np.uint8))]
    pred = syn.FakeHeadPredictor(base_seed=9, n=24)
    css = {"class_0": {"confidence_threshold": 0.3}, "class_1": {"confidence_threshold": 0.2}}
    small = adapters.determine_small_classes(adapters.calculate_average_mask_sizes([pred], [im for _, im in imgs]))
    kw = dict(visualize=False, images=imgs, predictors=[pred], thing_classes=["pore", "throat"], small_classes=small,
              spatial_rules=syn.POLYHIPES_RULES, tile_size=96, overlap_ratio=0.25, confidence_mode="manual", class_specific_settings=css)
    return imgs, kw


def test_errors(cuda_device, tmp_path):
    gt, dt = ce.synthetic_case(5, [(64, 64)], 5, n_cats=2)
    g, d = write(tmp_path, "gt.json", gt), write(tmp_path, "dt.json", dt)
    for bad in [(1, 10), (10, 10, 100), (0, 1, 2), (1, 2, 3.0), (1, True, 3), "abc"]:
        with pytest.raises(ValueError, match="max_dets"):
            inf.evaluate_coco(g, d, max_dets=bad)
    d2 = json.loads(json.dumps(dt))
    del d2["annotations"][2]["score"]
    with pytest.raises(ValueError, match=f"annotation {d2['annotations'][2]['id']}: score"):
        inf.evaluate_coco(g, write(tmp_path, "d2.json", d2))
    d3 = json.loads(json.dumps(dt))
    d3["images"][0]["file_name"] = "nowhere.png"
    with pytest.raises(ValueError, match="nowhere.png"):
        inf.evaluate_coco(g, write(tmp_path, "d3.json", d3))
    g4 = json.loads(json.dumps(gt))
    g4["categories"][1]["name"] = g4["categories"][0]["name"]
    with pytest.raises(ValueError, match="given twice"):
        inf.evaluate_coco(write(tmp_path, "g4.json", g4), d, match_categories="name")
    d5 = json.loads(json.dumps(dt))
    d5["annotations"][1]["segmentation"] = [[0, 0, 5, 0, 5, 5]]
    with pytest.raises(ValueError, match="compressed-RLE"):
        inf.evaluate_coco(g, write(tmp_path, "d5.json", d5))
    g6 = json.loads(json.dumps(gt))
    g6["annotations"][0]["segmentation"]["size"] = [32, 64]
    with pytest.raises(ValueError, match="size"):
        inf.evaluate_coco(write(tmp_path, "g6.json", g6), d)
    d7 = json.loads(json.dumps(dt))
    d7["annotations"][0]["segmentation"]["counts"] = "0" * 3
    with pytest.raises(_lib.EmiaError):
        inf.evaluate_coco(g, write(tmp_path, "d7.json", d7))
    with pytest.raises(ValueError, match="match_categories"):
        inf.evaluate_coco(g, d, match_categories="nope")
