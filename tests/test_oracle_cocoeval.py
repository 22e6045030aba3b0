"""CPU: hand-derived known answers for oracle/cocoeval.py, the numpy restatement of pycocotools' COCOeval (segm) that the device
evaluation (engine.coco_evaluate, functions.inference.evaluate_coco) is checked against."""
import numpy as np
import pytest

from oracle import coco, cocoeval as ce

EPS1 = float(1 / (1 + np.spacing(1)))          # the precision of one true positive: tp / (fp + tp + np.spacing(1))


def box(H, W, y0, y1, x0, x1):
    m = np.zeros((H, W), np.uint8)
    m[y0:y1, x0:x1] = 1
    return m


def seg(m):
    return {"size": list(m.shape), "counts": coco.rle_to_string(coco.rle_encode(m))}


def files(images, gts, dts, cats=((1, "pore"),), dt_cats=None):
    """images [(id, name, H, W)]; gts [(image id, cat, mask, extra)]; dts [(image id, cat, mask, score, extra)]."""
    imgs = [{"id": i, "file_name": n, "height": H, "width": W} for i, n, H, W in images]
    gt = {"images": imgs, "categories": [{"id": c, "name": n} for c, n in cats],
          "annotations": [dict({"id": k + 1, "image_id": i, "category_id": c, "segmentation": seg(m), "area": int(m.sum()),
                                "iscrowd": 0}, **e) for k, (i, c, m, e) in enumerate(gts)]}
    dt = {"images": [dict(e) for e in imgs], "categories": [{"id": c, "name": n} for c, n in (dt_cats or cats)],
          "annotations": [dict({"id": k + 1, "image_id": i, "category_id": c, "segmentation": seg(m), "score": s}, **e)
                          for k, (i, c, m, s, e) in enumerate(dts)]}
    return gt, dt


def test_perfect_predictions():
    H, W = 64, 64
    small, medium = box(H, W, 0, 10, 0, 10), box(H, W, 20, 60, 20, 60)
    gt, dt = files([(1, "a.png", H, W)], [(1, 1, small, {}), (1, 1, medium, {})], [(1, 1, small, .9, {}), (1, 1, medium, .8, {})])
    r = ce.evaluate(gt, dt)
    p = r["precision"]
    assert np.all(p[:, :, 0, 0, 1:] == 1.0)                    # all: two true positives, the second has precision exactly 1
    assert p[0, :, 0, 0, 0].tolist() == [EPS1] * 51 + [0.0] * 50    # maxDets 1: one of the two
    assert np.all(p[:, :, 0, 1, :] == EPS1) and np.all(p[:, :, 0, 2, 1:] == EPS1)  # one TP each in small / medium (2nd of the image)
    assert np.all(p[:, :, 0, 3, :] == -1) and np.all(r["recall"][:, 0, 3, :] == -1)  # no large GT
    assert np.all(r["recall"][:, 0, 0, 0] == 0.5)               # maxDets 1 of 2
    assert r["stats"][0] == 1.0 and r["stats"][5] == -1.0 and r["stats"][6] == 0.5 and r["stats"][8] == 1.0
    assert r["per_category"] == {"pore": 1.0}


def test_two_gt_three_dt():
    H, W = 10, 100
    A, B = box(H, W, 0, H, 0, 10), box(H, W, 0, H, 50, 60)
    d1, d2, d3 = A, box(H, W, 0, H, 20, 30), box(H, W, 0, H, 52, 62)      # IoU 1, 0, 80 / 120
    gt, dt = files([(1, "a.png", H, W)], [(1, 1, A, {}), (1, 1, B, {})], [(1, 1, d1, .9, {}), (1, 1, d2, .8, {}), (1, 1, d3, .7, {})])
    r = ce.evaluate(gt, dt)
    p, rc = r["precision"][:, :, 0, 0, 2], r["recall"][:, 0, 0, 2]
    lo = [EPS1] * 51
    for t in range(4):                                          # .50 .. .65: d3 matches B
        assert p[t].tolist() == lo + [2 / 3] * 50 and rc[t] == 1.0
    for t in range(4, 10):
        assert p[t].tolist() == lo + [0.0] * 50 and rc[t] == 0.5


def test_crowd_matched_twice():
    H, W = 10, 100
    crowd, B = box(H, W, 0, H, 0, 20), box(H, W, 0, H, 50, 60)
    gt, dt = files([(1, "a.png", H, W)], [(1, 1, crowd, {"iscrowd": 1}), (1, 1, B, {})],
                   [(1, 1, box(H, W, 0, H, 0, 10), .9, {}), (1, 1, box(H, W, 0, H, 10, 20), .8, {}), (1, 1, B, .7, {})])
    _, _, gts, dts, _ = ce.prepare(gt, dt)
    g, d = gts[1, 1], dts[1, 1]
    cands = ce.sparse_ious(d, g, H, W)
    assert cands[0] == [(0, 1.0)] and cands[1] == [(0, 1.0)]    # inter / area_d for a crowd GT
    dtm, dtIg, gtIg = ce.evaluate_img(cands, [x["area"] for x in g], [x["iscrowd"] for x in g], [1, 2], [x["area"] for x in d],
                                      ce.AREA_RNG[0])
    assert (dtm[:, 0] == 1).all() and (dtm[:, 1] == 1).all() and dtIg[:, :2].all() and (dtm[:, 2] == 2).all()
    r = ce.evaluate(gt, dt)
    assert np.all(r["precision"][:, :, 0, 0, 2] == EPS1)        # the crowd matches are ignored: one TP, no FP


def _both(ious, gt_area, crowd, ids, dt_area, rng):
    """evaluate_img over the dense matrix, and the dense reference loop: must agree."""
    cands = [[(g, v) for g, v in enumerate(row) if v > 0] for row in ious]
    sp = ce.evaluate_img(cands, gt_area, crowd, ids, dt_area, rng)
    de = ce.evaluate_img_dense(np.asarray(ious, np.float64).reshape(len(dt_area), len(gt_area)), gt_area, crowd, ids, dt_area, rng)
    assert np.array_equal(sp[0], de[0]) and np.array_equal(sp[1], de[1]) and np.array_equal(sp[2], de[2])
    return sp


def test_area_ignored_gt_only_as_fallback():
    dtm, dtIg, _ = _both([[0.9, 0.6]], [2000.0, 100.0], [0, 0], [10, 11], [100.0], ce.AREA_RNG[1])   # GT 10 ignored at "small"
    assert dtm[:3, 0].tolist() == [11, 11, 11] and not dtIg[:3, 0].any()      # t <= .60: the non-ignored GT, despite its IoU
    assert dtm[3:, 0].tolist() == [10] * 6 + [0] and dtIg[3:9, 0].all()       # then the ignored one, up to IoU .9


def test_iou_ties_go_to_the_later_gt():
    dtm, _, _ = _both([[0.7, 0.7, 0.3]], [100.0] * 3, [0] * 3, [10, 11, 12], [100.0], ce.AREA_RNG[0])
    assert dtm[:5, 0].tolist() == [11] * 5


def test_gt_id_zero_counts_as_no_match():
    H, W = 10, 100
    A = box(H, W, 0, H, 0, 10)
    gt, dt = files([(1, "a.png", H, W)], [(1, 1, A, {"id": 0})], [(1, 1, A, .9, {}), (1, 1, A, .8, {})])
    dtm, dtIg, _ = _both([[1.0], [1.0]], [100.0], [0], [0], [100.0, 100.0], ce.AREA_RNG[0])
    assert not dtm.any() and not dtIg.any()
    r = ce.evaluate(gt, dt)
    assert np.all(r["precision"][:, :, 0, 0, 2] == 0.0) and np.all(r["recall"][:, 0, 0, 2] == 0.0)


def test_loadres_area():
    H, W = 64, 64
    m = box(H, W, 0, 10, 0, 10)
    gt, dt = files([(1, "a.png", H, W)], [(1, 1, m, {})], [(1, 1, m, .9, {"bbox": [0.0, 0.0, 40.0, 40.0]}), (1, 1, m, .8, {"bbox": [0, 0, 3, 5]})])
    assert [x["area"] for x in ce.prepare(gt, dt)[3][1, 1]] == [1600.0, 15.0]     # bbox branch: w * h of each bbox
    dt["annotations"][0].pop("bbox")
    assert [x["area"] for x in ce.prepare(gt, dt)[3][1, 1]] == [100.0, 100.0]     # first annotation without bbox: popcount
    gt["annotations"][0]["area"] = 2500.5                                         # the GT area is the file's field
    assert ce.prepare(gt, dt)[2][1, 1][0]["area"] == 2500.5


def test_truncation_at_max_dets():
    H, W = 10, 100
    ms = [box(H, W, 0, H, 20 * k, 20 * k + 10) for k in range(4)]
    gt, dt = files([(1, "a.png", H, W)], [(1, 1, m, {}) for m in ms[:3]], [(1, 1, m, .9 - .1 * k, {}) for k, m in enumerate(ms)])
    r = ce.evaluate(gt, dt, max_dets=(1, 2, 3))
    assert r["recall"][:, 0, 0, :].tolist() == [[1 / 3, 2 / 3, 1.0]] * 10
    assert np.all(r["precision"][:, :, 0, 0, 2] == 1.0)         # the 4th (a false positive) is past maxDets[-1]
    with pytest.raises(ValueError):
        ce.evaluate(gt, dt, max_dets=(1, 10, 10))


def test_equal_scores_across_images():
    H, W = 10, 100
    A, B = box(H, W, 0, H, 0, 10), box(H, W, 0, H, 50, 60)
    gt, dt = files([(2, "b.png", H, W), (1, "a.png", H, W)], [(1, 1, A, {}), (2, 1, A, {})], [(2, 1, A, .5, {}), (1, 1, B, .5, {})])
    r = ce.evaluate(gt, dt)                                     # image 1's false positive comes first: rc [0, .5], pr [0, .5]
    assert np.all(r["precision"][:, :51, 0, 0, 2] == 0.5) and np.all(r["precision"][:, 51:, 0, 0, 2] == 0.0)


def test_category_without_gt():
    H, W = 10, 100
    A = box(H, W, 0, H, 0, 10)
    gt, dt = files([(1, "a.png", H, W)], [(1, 1, A, {})], [(1, 2, A, .9, {})], cats=((1, "pore"), (2, "throat")))
    r = ce.evaluate(gt, dt)
    assert np.all(r["precision"][:, :, 1] == -1) and r["per_category"]["throat"] == -1.0
    assert np.all(r["precision"][:, :, 0, 0, :] == 0.0)         # pore: a GT and no detection


def test_image_without_gt_all_false_positives():
    H, W = 10, 100
    A = box(H, W, 0, H, 0, 10)
    gt, dt = files([(1, "a.png", H, W), (2, "b.png", H, W)], [(1, 1, A, {})],
                   [(2, 1, A, .9, {}), (2, 1, A, .8, {}), (1, 1, A, .7, {})])
    r = ce.evaluate(gt, dt)
    assert np.all(r["precision"][:, :, 0, 0, 2] == 1 / 3) and r["stats"][0] == pytest.approx(1 / 3)


def test_match_categories_by_name():
    H, W = 10, 100
    A = box(H, W, 0, H, 0, 10)
    gt, dt = files([(1, "a.png", H, W)], [(1, 1, A, {})], [(1, 0, A, .9, {}), (1, 1, box(H, W, 0, H, 50, 60), .8, {})],
                   cats=((1, "pore"), (2, "throat")), dt_cats=((0, "pore"), (1, "throat")))
    assert ce.evaluate(gt, dt, match_categories="name")["per_category"] == {"pore": EPS1, "throat": -1.0}
    assert ce.evaluate(gt, dt)["per_category"] == {"pore": 0.0, "throat": -1.0}
    gt["categories"][1]["name"] = "pore"
    with pytest.raises(ValueError):
        ce.evaluate(gt, dt, match_categories="name")


def test_csv_and_errors():
    H, W = 10, 100
    A = box(H, W, 0, H, 0, 10)
    gt, dt = files([(1, "a.png", H, W)], [(1, 1, A, {})], [(1, 1, A, .9, {})])
    text = ce.evaluate(gt, dt)["csv"].decode()
    lines = text.split("\r\n")
    assert lines[0] == "Metric,Category,IoU,Area,MaxDets,Value" and lines[1].startswith("AP,all,0.50:0.95,all,100,")
    assert lines[13] == f"AP,pore,0.50:0.95,all,100,{EPS1!r}" and len(lines) == 15
    del dt["annotations"][0]["score"]
    with pytest.raises(ValueError):
        ce.evaluate(gt, dt)
    dt["annotations"][0]["score"] = 0.5
    dt["images"][0]["file_name"] = "other.png"
    with pytest.raises(ValueError):
        ce.evaluate(gt, dt)


def test_sparse_equals_dense_random():
    rng = np.random.default_rng(5)
    for _ in range(200):
        D, G = int(rng.integers(0, 7)), int(rng.integers(0, 7))
        ious = np.where(rng.random((D, G)) < 0.5, rng.choice([0.5, 0.55, 0.7, 0.95, 1.0, rng.random()], (D, G)), 0.0)
        area = rng.choice([10.0, 1024.0, 2000.0, 9216.0, 20000.0], G)
        _both(ious, area, rng.random(G) < 0.3, list(rng.integers(0, 3, G)), rng.choice([10.0, 5000.0, 20000.0], D),
              ce.AREA_RNG[int(rng.integers(0, 4))])
