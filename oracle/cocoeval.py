"""Oracle: COCO `segm` evaluation, a numpy restatement of pycocotools 2.0 `COCO.loadRes` + `COCOeval` (`evaluate`,
`evaluateImg`, `accumulate`, `summarize`) for iouType="segm", useCats=1 (test infrastructure only).

pycocotools is not a dependency of the project and is not installed here: nothing in this file has been checked against the
real library.  It restates the library from its published source, with these rules:

  images       the GT file's `images`, ascending id.  A DT `images` entry is matched to a GT image by file_name and its
               annotations are re-keyed to that id; a DT image without GT counterpart is an error (loadRes' assertion).  The
               frame size is the GT entry's height / width; every segmentation's size must equal it.
  categories   the GT file's category ids, ascending.  DT annotations of another category are dropped.  With
               match_categories="name" a DT category id is first mapped, through the DT file's categories, to the GT category
               of the same name (duplicate GT names are an error).
  GT           per (image, category) in file order; area = the file's `area` (the popcount when the field is absent: a
               deviation, pycocotools raises there); ignore = bool(iscrowd) (the file's own `ignore` is overwritten, as
               _prepare does); the annotation id is kept.
  DT           loadRes: ids 1, 2, ... in file order, iscrowd 0; area = bbox[2] * bbox[3] when the file's first annotation has
               a non-empty bbox (loadRes' bbox branch), else the popcount; score = the JSON number as a float64 (a detection
               without a numeric score is an error).
  IoU          maskApi.c rleIou: inter / (area_d + area_g - inter) as double, inter / area_d for a crowd GT, 0 when
               inter == 0; computed exactly only for pairs whose rleToBbox boxes overlap (bbIou's prefilter).
  evaluateImg  per (image, category, area range), maxDet = maxDets[-1]: detections stably sorted by -score and truncated,
               GTs stably sorted by _ignore = ignore or area outside the range; at each IoU threshold t a detection takes,
               among GTs not yet matched at t (crowd GTs can be matched again) with iou >= min(t, 1 - 1e-10), the one with the
               largest IoU among non-ignored GTs (ties to the later GT position), and only when there is none the same choice
               among ignored GTs: what the reference's dense loop with its `break` computes (evaluate_img_dense), for a
               sparse candidate list in any order (evaluate_img).  dtIg = the matched GT's _ignore, or for an unmatched
               detection whether its area is outside the range; dtm = the matched GT's id, and dtm == 0 counts as no match
               (a GT with id 0 is matched, but its detection is a false positive unless ignored).
  accumulate   per (category, area, maxDet): the first maxDet detections of every image, in image order, stably sorted by
               -score; npig non-ignored GTs (entry skipped, -1, when 0); tp / fp cumulative sums; rc = tp / npig,
               pr = tp / (fp + tp + np.spacing(1)), pr replaced by its reverse running maximum; q[r] = pr[searchsorted(rc,
               recThrs[r], 'left')], 0 past the end; recall = rc[-1] (0 without detections).
  summarize    the 12 segm stats, each the numpy mean of the selected entries > -1 (-1 when none).  pycocotools' first stat
               uses a literal maxDets=100; here every AP stat uses maxDets[2], which is the same for the default (1, 10, 100).
"""
import csv
import io
import math
from collections import defaultdict

import cv2
import numpy as np

from deepemia_b200 import synthetic as syn
from oracle import coco

IOU_THRS = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
REC_THRS = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
AREA_RNG = [[0 ** 2, 1e5 ** 2], [0 ** 2, 32 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]]
AREA_LBL = ["all", "small", "medium", "large"]
CSV_HEADER = ["Metric", "Category", "IoU", "Area", "MaxDets", "Value"]


def _is_number(v):
    return isinstance(v, (int, float)) and not isinstance(v, bool)


def check_max_dets(max_dets):
    md = tuple(max_dets)
    if len(md) != 3 or not all(isinstance(m, (int, np.integer)) and not isinstance(m, bool) and m > 0 for m in md) or \
            not md[0] < md[1] < md[2]:
        raise ValueError(f"max_dets must be three strictly increasing positive ints, not {max_dets!r}")
    return tuple(int(m) for m in md)


def category_map(gt, dt, match_categories="id"):
    """{DT category id: GT category id} for the DT categories that are evaluated (all GT ids under "id")."""
    gt_ids = sorted(c["id"] for c in gt.get("categories", []))
    if match_categories == "id":
        return {c: c for c in gt_ids}
    if match_categories != "name":
        raise ValueError(f"match_categories must be 'id' or 'name', not {match_categories!r}")
    by_name = {}
    for c in gt.get("categories", []):
        if c.get("name") in by_name:
            raise ValueError(f"GT category name {c.get('name')!r} is given twice")
        by_name[c.get("name")] = c["id"]
    return {c["id"]: by_name[c.get("name")] for c in dt.get("categories", []) if c.get("name") in by_name}


# ---- masks: counts, rleToBbox, exact intersections ------------------------------------------------------------------------
def rle_to_bbox(cnts, H):
    """maskApi.c rleToBbox (x, y, w, h), including the full-height widening when a run wraps columns."""
    m = (len(cnts) // 2) * 2
    if m == 0:
        return (0, 0, 0, 0)
    xs, ys, xe, ye, cc, xp = 1 << 62, 1 << 62, 0, 0, 0, 0
    for j in range(m):
        cc += cnts[j]
        t = cc - j % 2
        y = t % H
        x = (t - y) // H
        if j % 2 == 0:
            xp = x
        elif xp < x:
            ys, ye = 0, H - 1
        xs, xe, ys, ye = min(xs, x), max(xe, x), min(ys, y), max(ye, y)
    return (xs, ys, xe - xs + 1, ye - ys + 1)


class Mask:
    """One compressed-RLE segmentation: its foreground intervals [s, e) on the column-major axis, popcount and rleToBbox."""
    __slots__ = ("s", "e", "area", "box")

    def __init__(self, counts, H):
        cnts = coco.rle_fr_string(counts)
        pos = np.concatenate([[0], np.cumsum(np.asarray(cnts, np.int64))])
        self.s, self.e = pos[1:-1:2], pos[2::2]
        self.area = int((self.e - self.s).sum())
        self.box = rle_to_bbox(cnts, H)


def _boxes_overlap(a, b):
    w = min(a[0] + a[2], b[0] + b[2]) - max(a[0], b[0])
    h = min(a[1] + a[3], b[1] + b[3]) - max(a[1], b[1])
    return w > 0 and h > 0


def intersection(a, b):
    if not len(a.s) or not len(b.s):
        return 0
    return int(np.maximum(0, np.minimum(a.e[:, None], b.e[None, :]) - np.maximum(a.s[:, None], b.s[None, :])).sum())


def rle_iou(inter, area_d, area_g, crowd):
    """maskApi.c rleIou for one pair."""
    if inter == 0:
        return 0.0
    return float(inter) / float(area_d if crowd else area_d + area_g - inter)


def sparse_ious(dts, gts, H, W):
    """[(g, iou), ...] per detection for the GTs whose boxes overlap its box (a grid of the GT boxes keeps it sparse)."""
    cs = max(16, int(math.ceil(math.sqrt(H * W / max(len(gts), 1)))))
    grid = defaultdict(list)
    for g, gm in enumerate(gts):
        x, y, w, h = gm["mask"].box
        if w and h:
            for cy in range(y // cs, (y + h - 1) // cs + 1):
                for cx in range(x // cs, (x + w - 1) // cs + 1):
                    grid[cy, cx].append(g)
    out = []
    for dm in dts:
        x, y, w, h = dm["mask"].box
        cand = set()
        if w and h:
            for cy in range(y // cs, (y + h - 1) // cs + 1):
                for cx in range(x // cs, (x + w - 1) // cs + 1):
                    cand.update(grid.get((cy, cx), ()))
        lst = []
        for g in sorted(cand):
            gm = gts[g]
            if _boxes_overlap(dm["mask"].box, gm["mask"].box):
                inter = intersection(dm["mask"], gm["mask"])
                lst.append((g, rle_iou(inter, dm["mask"].area, gm["mask"].area, gm["iscrowd"])))
        out.append(lst)
    return out


# ---- loadRes + _prepare ----------------------------------------------------------------------------------------------------
def prepare(gt, dt, match_categories="id"):
    """(image ids ascending, category ids ascending, {(img, cat): [GT dict]}, {(img, cat): [DT dict]}, {img: (H, W)})."""
    imgs = {}
    names = {}
    for e in gt.get("images", []):
        imgs[e["id"]] = (int(e["height"]), int(e["width"]))
        names[e.get("file_name")] = e["id"]
    img_ids = sorted(imgs)
    cmap = category_map(gt, dt, match_categories)
    cat_ids = sorted(c["id"] for c in gt.get("categories", []))
    cats = set(cat_ids)

    def seg_mask(ann, img):
        seg = ann.get("segmentation")
        if not isinstance(seg, dict) or not isinstance(seg.get("counts"), str):
            raise ValueError(f"annotation {ann.get('id')!r}: only compressed-RLE segmentations are read")
        if list(seg.get("size", [])) != list(imgs[img]):
            raise ValueError(f"annotation {ann.get('id')!r}: size {seg.get('size')!r} is not the image's")
        return Mask(seg["counts"], imgs[img][0])

    gts, dts = defaultdict(list), defaultdict(list)
    for ann in gt.get("annotations", []):
        if ann.get("image_id") not in imgs:
            raise ValueError(f"GT annotation {ann.get('id')!r}: image_id {ann.get('image_id')!r} has no images entry")
        m = seg_mask(ann, ann["image_id"])
        if ann.get("category_id") not in cats:
            continue
        area = ann["area"] if "area" in ann else m.area
        gts[ann["image_id"], ann["category_id"]].append({"id": ann["id"], "area": float(area), "iscrowd": bool(ann.get("iscrowd", 0)),
                                                        "mask": m})
    dt_img = {}
    for e in dt.get("images", []):
        if e.get("file_name") not in names:
            raise ValueError(f"DT image {e.get('id')!r}: file_name {e.get('file_name')!r} has no GT image")
        dt_img[e.get("id")] = names[e.get("file_name")]
    anns = dt.get("annotations", [])
    bbox_area = bool(anns) and bool(anns[0].get("bbox"))
    for k, ann in enumerate(anns):
        if not _is_number(ann.get("score")) or math.isnan(ann["score"]):
            raise ValueError(f"DT annotation {ann.get('id')!r}: no numeric score")
        if ann.get("image_id") not in dt_img:
            raise ValueError(f"DT annotation {ann.get('id')!r}: image_id {ann.get('image_id')!r} has no images entry")
        img = dt_img[ann["image_id"]]
        m = seg_mask(ann, img)
        cat = cmap.get(ann.get("category_id"))
        if cat is None:
            continue
        if bbox_area:
            bb = ann["bbox"]
            area = float(bb[2] * bb[3])
        else:
            area = float(m.area)
        dts[img, cat].append({"id": k + 1, "area": area, "score": float(ann["score"]), "mask": m})
    return img_ids, cat_ids, gts, dts, imgs


# ---- evaluateImg -----------------------------------------------------------------------------------------------------------
def evaluate_img_dense(ious, gt_area, gt_crowd, gt_ids, dt_area, a_rng, iou_thrs=IOU_THRS):
    """The reference's loop.  ious [D, G] with detections in score order (already truncated) and GTs in file order.
    Returns (dtm [T, D] float, dtIg [T, D] bool, gtIg [G] int in sorted-GT order)."""
    G, D, T = len(gt_area), len(dt_area), len(iou_thrs)
    ig0 = [int(bool(c) or a < a_rng[0] or a > a_rng[1]) for a, c in zip(gt_area, gt_crowd)]
    gtind = np.argsort(ig0, kind="mergesort")
    gtIg = np.array([ig0[i] for i in gtind])
    iscrowd = [int(gt_crowd[i]) for i in gtind]
    ids = [gt_ids[i] for i in gtind]
    ious = ious[:, gtind] if G and D else ious
    gtm = np.zeros((T, G))
    dtm = np.zeros((T, D))
    dtIg = np.zeros((T, D))
    if G and D:
        for tind, t in enumerate(iou_thrs):
            for dind in range(D):
                iou = min([t, 1 - 1e-10])
                m = -1
                for gind in range(G):
                    if gtm[tind, gind] > 0 and not iscrowd[gind]:
                        continue
                    if m > -1 and gtIg[m] == 0 and gtIg[gind] == 1:
                        break
                    if ious[dind, gind] < iou:
                        continue
                    iou = ious[dind, gind]
                    m = gind
                if m == -1:
                    continue
                dtIg[tind, dind] = gtIg[m]
                dtm[tind, dind] = ids[m]
                gtm[tind, m] = dind + 1
    a = np.array([d < a_rng[0] or d > a_rng[1] for d in dt_area]).reshape((1, D))
    dtIg = np.logical_or(dtIg, np.logical_and(dtm == 0, np.repeat(a, T, 0)))
    return dtm, dtIg, gtIg


def evaluate_img(cands, gt_area, gt_crowd, gt_ids, dt_area, a_rng, iou_thrs=IOU_THRS):
    """The same over sparse candidates: cands[d] = [(g, iou), ...] in any order, g the GT's file-order index."""
    G, D, T = len(gt_area), len(cands), len(iou_thrs)
    gt_area = np.asarray(gt_area, np.float64).reshape(-1)
    crowd = np.asarray(gt_crowd, bool).reshape(-1)
    ig = crowd | (gt_area < a_rng[0]) | (gt_area > a_rng[1])
    gtm = np.zeros((T, G), bool)
    dtm = np.zeros((T, D))
    dtIg = np.zeros((T, D), bool)
    for t, thr in enumerate(iou_thrs):
        thr = min(thr, 1 - 1e-10)
        for d in range(D):
            best = None
            for g, iou in cands[d]:
                if iou < thr or (gtm[t, g] and not crowd[g]):
                    continue
                key = (not ig[g], iou, g)
                if best is None or key > best:
                    best = key
            if best is None:
                continue
            g = best[2]
            dtIg[t, d] = ig[g]
            dtm[t, d] = gt_ids[g]
            gtm[t, g] = True
    out = np.array([d < a_rng[0] or d > a_rng[1] for d in dt_area], bool).reshape(1, D)
    dtIg = dtIg | ((dtm == 0) & out)
    return dtm, dtIg, np.sort(ig.astype(int), kind="mergesort")


# ---- accumulate ------------------------------------------------------------------------------------------------------------
def accumulate_one(E, max_det, iou_thrs=IOU_THRS, rec_thrs=REC_THRS):
    """One (category, area, maxDet): E = [(dtScores [D], dtm [T, D], dtIg [T, D], gtIg [G]) per image in image order].
    Returns (q [T, R], recall [T]) or None when the entry stays -1."""
    if not E:
        return None
    dtScores = np.concatenate([e[0][0:max_det] for e in E])
    inds = np.argsort(-dtScores, kind="mergesort")
    dtm = np.concatenate([e[1][:, 0:max_det] for e in E], axis=1)[:, inds]
    dtIg = np.concatenate([e[2][:, 0:max_det] for e in E], axis=1)[:, inds]
    gtIg = np.concatenate([e[3] for e in E])
    npig = np.count_nonzero(gtIg == 0)
    if npig == 0:
        return None
    tps = np.logical_and(dtm, np.logical_not(dtIg))
    fps = np.logical_and(np.logical_not(dtm), np.logical_not(dtIg))
    tp_sum = np.cumsum(tps, axis=1).astype(dtype=np.float64)
    fp_sum = np.cumsum(fps, axis=1).astype(dtype=np.float64)
    T, R = len(iou_thrs), len(rec_thrs)
    q_all, rec = np.zeros((T, R)), np.zeros(T)
    for t, (tp, fp) in enumerate(zip(tp_sum, fp_sum)):
        nd = len(tp)
        rc = tp / npig
        pr = tp / (fp + tp + np.spacing(1))
        rec[t] = rc[-1] if nd else 0
        if nd:
            pr = np.maximum.accumulate(pr[::-1])[::-1]     # the reference's backward `if pr[i] > pr[i-1]` loop
        inds = np.searchsorted(rc, rec_thrs, side="left")
        q = np.zeros(R)
        ok = inds < nd                                     # the reference's try / except: 0 from the first index past the end
        q[ok] = pr[inds[ok]]
        q_all[t] = q
    return q_all, rec


def accumulate(evals, img_ids, cat_ids, max_dets):
    """evals[(img, cat, a)] = evaluate_img output + dtScores -> (precision [T, R, K, A, M], recall [T, K, A, M])."""
    T, R, K, A, M = len(IOU_THRS), len(REC_THRS), len(cat_ids), len(AREA_RNG), len(max_dets)
    precision = -np.ones((T, R, K, A, M))
    recall = -np.ones((T, K, A, M))
    for k, c in enumerate(cat_ids):
        for a in range(A):
            E = [evals[i, c, a] for i in img_ids if (i, c, a) in evals]
            for m, md in enumerate(max_dets):
                r = accumulate_one(E, md)
                if r is not None:
                    precision[:, :, k, a, m], recall[:, k, a, m] = r
    return precision, recall


# ---- summarize and the CSV -------------------------------------------------------------------------------------------------
def _mean(s):
    return float(np.mean(s[s > -1])) if len(s[s > -1]) else -1.0


def _summarize(precision, recall, max_dets, ap, iou_thr=None, area="all", max_det=None):
    aind = [i for i, lbl in enumerate(AREA_LBL) if lbl == area]
    mind = [i for i, m in enumerate(max_dets) if m == max_det]
    s = precision if ap else recall
    if iou_thr is not None:
        s = s[np.where(iou_thr == IOU_THRS)[0]]
    s = s[:, :, :, aind, mind] if ap else s[:, :, aind, mind]
    return _mean(s)


STAT_ROWS = [(1, None, "all", 2), (1, .5, "all", 2), (1, .75, "all", 2), (1, None, "small", 2), (1, None, "medium", 2),
             (1, None, "large", 2), (0, None, "all", 0), (0, None, "all", 1), (0, None, "all", 2), (0, None, "small", 2),
             (0, None, "medium", 2), (0, None, "large", 2)]


def summarize(precision, recall, max_dets):
    """The 12 stats and the per-category AP (IoU .50:.95, area all, maxDets[2])."""
    stats = [_summarize(precision, recall, max_dets, ap, t, a, max_dets[m]) for ap, t, a, m in STAT_ROWS]
    per_cat = [_mean(precision[:, :, k, 0, 2]) for k in range(precision.shape[2])]
    return stats, per_cat


def _iou_label(t):
    return "0.50:0.95" if t is None else f"{t:.2f}"


def csv_text(stats, per_cat, cat_names, max_dets):
    """coco_eval_results.csv as csv.writer writes it."""
    buf = io.StringIO()
    w = csv.writer(buf)
    w.writerow(CSV_HEADER)
    for (ap, t, a, m), v in zip(STAT_ROWS, stats):
        w.writerow(["AP" if ap else "AR", "all", _iou_label(t), a, max_dets[m], repr(float(v))])
    for name, v in zip(cat_names, per_cat):
        w.writerow(["AP", name, _iou_label(None), "all", max_dets[2], repr(float(v))])
    return buf.getvalue().encode("utf-8")


def evaluate(gt, dt, max_dets=(1, 10, 100), match_categories="id"):
    """The json-loaded GT and DT dicts -> {"stats", "per_category" {name: AP}, "precision", "recall", "csv"}."""
    max_dets = check_max_dets(max_dets)
    img_ids, cat_ids, gts, dts, imgs = prepare(gt, dt, match_categories)
    evals = {}
    for (i, c) in set(gts) | set(dts):
        g, d = gts.get((i, c), []), dts.get((i, c), [])
        order = np.argsort([-x["score"] for x in d], kind="mergesort")[:max_dets[-1]]
        d = [d[j] for j in order]
        H, W = imgs[i]
        cands = sparse_ious(d, g, H, W)
        for a, rng in enumerate(AREA_RNG):
            dtm, dtIg, gtIg = evaluate_img(cands, [x["area"] for x in g], [x["iscrowd"] for x in g], [x["id"] for x in g],
                                           [x["area"] for x in d], rng)
            evals[i, c, a] = (np.array([x["score"] for x in d]), dtm, dtIg, gtIg)
    precision, recall = accumulate(evals, img_ids, cat_ids, max_dets)
    stats, per_cat = summarize(precision, recall, max_dets)
    names = {c["id"]: c.get("name") for c in gt.get("categories", [])}
    cat_names = [names[c] for c in cat_ids]
    return {"stats": stats, "per_category": dict(zip(cat_names, per_cat)), "precision": precision, "recall": recall,
            "csv": csv_text(stats, per_cat, cat_names, max_dets)}


# ---- synthetic test inputs -------------------------------------------------------------------------------------------------

def _poly_pixels(poly, H, W):
    """(ys, xs) of a filled polygon, rasterized in its own bounding box (no full-frame mask) and clipped to the frame."""
    p = np.round(poly).astype(np.int32)
    x0, y0 = p.min(0)
    x1, y1 = p.max(0)
    crop = np.zeros((y1 - y0 + 1, x1 - x0 + 1), np.uint8)
    cv2.fillPoly(crop, [p - [x0, y0]], 1)
    ys, xs = np.nonzero(crop)
    ys, xs = ys + y0, xs + x0
    ok = (ys >= 0) & (ys < H) & (xs >= 0) & (xs < W)
    return ys[ok], xs[ok]


def _morph_pixels(ys, xs, H, W, op, r):
    """dilate (op > 0) or erode (op < 0) the pixel set with a (2r + 1)^2 square, in a padded local crop."""
    if not len(ys):
        return ys, xs
    y0, x0 = ys.min() - r, xs.min() - r
    crop = np.zeros((ys.max() - y0 + r + 1, xs.max() - x0 + r + 1), np.uint8)
    crop[ys - y0, xs - x0] = 1
    k = np.ones((2 * r + 1, 2 * r + 1), np.uint8)
    crop = cv2.dilate(crop, k) if op > 0 else cv2.erode(crop, k)
    ys, xs = np.nonzero(crop)
    ys, xs = ys + y0, xs + x0
    ok = (ys >= 0) & (ys < H) & (xs >= 0) & (xs < W)
    return ys[ok], xs[ok]


def coco_counts(ys, xs, H, W):
    """The compressed RLE counts string (coco.rle_to_string) of the pixel set (ys, xs) of an H x W frame, from its column-major
    runs, without a full-frame mask."""
    p = np.unique(xs.astype(np.int64) * H + ys)
    if not len(p):
        return coco.rle_to_string(coco.counts_from_runs(np.zeros((0, 2), np.int64), H, W))
    brk = np.nonzero(np.diff(p) != 1)[0]
    st = np.concatenate([[p[0]], p[brk + 1]])
    en = np.concatenate([p[brk], [p[-1]]]) + 1
    return coco.rle_to_string(coco.counts_from_runs(np.stack([st + 1, en - st], 1), H, W))


def synthetic_case(seed, frames, n_per_image, n_cats=2, rmin=4.0, rmax=30.0, crowd_frac=0.05, drop_frac=0.1, dup_frac=0.05,
                   spurious_frac=0.05, other_cat_frac=0.05, score_levels=50):
    """Test input: a ground-truth COCO dict of star-polygon particles (synthetic.particle_field) and a predictions dict derived from it: shifted,
    dilated or eroded masks, dropped particles, duplicates, spurious particles, another category now and then, scores on a
    coarse grid (ties), crowd GTs and GT `area` fields unlike the popcount.  frames: [(H, W)] per image; n_per_image: GT
    particles per image (an int, or a list; 0 gives an image without GT).  Returns (gt, dt) as json-ready dicts."""
    rng = np.random.default_rng(seed)
    images, gts, dts = [], [], []
    counts = n_per_image if isinstance(n_per_image, (list, tuple)) else [n_per_image] * len(frames)
    for j, ((H, W), n) in enumerate(zip(frames, counts)):
        iid = 2 * j + 7                               # ids unlike positions; listed in reverse order below
        images.append({"id": iid, "file_name": f"img_{j:03d}.png", "height": H, "width": W})
        for poly in syn.particle_field(rng, n, H, W, rmin=rmin, rmax=rmax, margin=0):
            ys, xs = _poly_pixels(poly, H, W)
            if not len(ys):
                continue
            cat = int(rng.integers(1, n_cats + 1))
            crowd = int(rng.random() < crowd_frac)
            area = float(len(ys)) if rng.random() < 0.8 else float(len(ys)) * float(rng.uniform(0.5, 40.0))
            gts.append({"id": len(gts) + 1, "image_id": iid, "category_id": cat, "segmentation": {"size": [H, W],
                        "counts": coco_counts(ys, xs, H, W)}, "area": area, "iscrowd": crowd})
            if rng.random() < drop_frac:
                continue
            for _ in range(2 if rng.random() < dup_frac else 1):
                u = rng.random()
                if u < 0.4:
                    dy, dx = (int(v) for v in rng.integers(-3, 4, 2))
                    py, px = ys + dy, xs + dx
                    ok = (py >= 0) & (py < H) & (px >= 0) & (px < W)
                    py, px = py[ok], px[ok]
                elif u < 0.6:
                    py, px = _morph_pixels(ys, xs, H, W, 1, int(rng.integers(1, 3)))
                elif u < 0.8:
                    py, px = _morph_pixels(ys, xs, H, W, -1, 1)
                else:
                    py, px = ys, xs
                dcat = cat if rng.random() >= other_cat_frac else int(rng.integers(1, n_cats + 1))
                dts.append((iid, H, W, dcat, py, px))
        for poly in syn.particle_field(rng, int(n * spurious_frac) + (1 if n == 0 else 0), H, W, rmin=rmin, rmax=rmax, margin=0):
            ys, xs = _poly_pixels(poly, H, W)
            dts.append((iid, H, W, int(rng.integers(1, n_cats + 1)), ys, xs))
    order = rng.permutation(len(dts))
    dt_anns = []
    for k in order:
        iid, H, W, cat, ys, xs = dts[k]
        dt_anns.append({"id": len(dt_anns) + 1, "image_id": iid, "category_id": cat, "segmentation": {"size": [H, W],
                        "counts": coco_counts(ys, xs, H, W)}, "score": float(rng.integers(1, score_levels + 1)) / score_levels})
    cats = [{"id": c, "name": f"class_{c}"} for c in range(1, n_cats + 1)]
    gt = {"images": images[::-1], "annotations": gts, "categories": cats}
    dt = {"images": [dict(e) for e in images], "annotations": dt_anns, "categories": cats}
    return gt, dt
