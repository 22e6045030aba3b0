"""Mirror of the hot-path functions of the reference's src/functions/inference.py — same names, argument meaning, return
conventions (lists of H x W numpy masks, numpy scalar scores, int classes) and quirks (SURVEY.md Appendix A) — with every mask
operation executed by libemia.so on the GPU.  Between the steps of one function the instances stay bit-packed on the device;
numpy masks are only materialised for what a function returns.

Pre-paste hook (SURVEY §8b): a `predictor` here is any object with

    heads(image) -> HeadOutputs(probs [N,28,28] f32, boxes [N,4] f32 xyxy in model-input coordinates, scores [N] f32,
                                classes [N] int, input_size (in_h, in_w))          # CUDA tensors

i.e. what Detectron2's GeneralizedRCNN.inference(batched_inputs, do_postprocess=False) yields (INTEGRATION.md shows the
adapter).  detector_postprocess + paste_masks_in_image then happen in K1.  A list of such predictors is an ensemble.

Module-level settings mirror the reference's module globals (inference.py:55-93) and can be overridden by the host application.
"""
import csv
import json
import os
from dataclasses import dataclass

import cv2
import numpy as np
import torch

from .. import engine
from ..utils import _bridge
from ..utils.mask_utils import rle_encoding  # noqa: F401  (re-exported like the reference's import)
from ..utils import spatial_constraints as _sc
from ..utils.measurements import record_to_dict, KEY_ORDER, SHAPE_HEADER, NEIGHBOUR_HEADER

# ---- module-level settings (reference: config.yaml via inference.py:55-93) ---------------------------------------------------
PARALLEL_MASK_PROCESSING = True            # l4_performance_optimizations.enable_parallel_mask_processing
TILE_BATCH_SIZE = 4                        # inference_settings.tile_settings.tile_batch_size (no effect on results)
ENSEMBLE_WEIGHTS = {"R50": 0.6, "R101": 0.4}
MIN_TOTAL_MASKS = 10
MIN_RELATIVE_INCREASE = 0.25
MAX_CONSECUTIVE_ZERO = 2
MIN_ITERATIONS = 2
measure_contrast_distribution = False

CSV_HEADER = ["Instance_ID", "Class", "Class_Name", "Major axis length", "Minor axis length", "Eccentricity", "C. Length",
              "C. Width", "Circular eq. diameter", "Aspect ratio", "Circularity", "Chord length", "Ferret diameter", "Roundness",
              "Sphericity", "Contrast d10", "Contrast d50", "Contrast d90", "Detected scale bar", "File name"]


@dataclass
class HeadOutputs:
    probs: torch.Tensor
    boxes: torch.Tensor
    scores: torch.Tensor
    classes: torch.Tensor
    input_size: tuple


# =================================================================================================================
# small helpers with the reference's names
# =================================================================================================================
def iou(mask1, mask2):
    """inference.py:422-435: sum(and) / sum(or), 0 when the union is empty."""
    iset = _bridge.upload([mask1, mask2])
    inter, a, b = (int(v) for v in engine.pair_counts(iset, [0], [1])[0].tolist())
    union = a + b - inter
    return inter / union if union > 0 else 0


def get_mask_bbox(mask):
    """inference.py:2722-2733 -> (y_min, x_min, y_max, x_max) or None."""
    return _sc.get_mask_bbox(mask)


def bboxes_overlap(bbox1, bbox2):
    """inference.py:2680-2694.  The tuples are unpacked as (y_min, x_min, y_max, x_max) whatever the caller stored (Q1)."""
    return _sc.bboxes_overlap(bbox1, bbox2)


def calculate_iou(mask1, mask2, bbox1=None, bbox2=None):
    """inference.py:2697-2719: bbox pre-test (with the tuples as given), then intersection / union."""
    if bbox1 is not None and bbox2 is not None and not bboxes_overlap(bbox1, bbox2):
        return 0.0
    return _sc.calculate_iou(mask1, mask2)


def is_edge_mask(mask, tile_size, overlap_ratio):
    """inference.py:2522-2549."""
    edge_width = int(tile_size * overlap_ratio / 2)
    b = get_mask_bbox(mask)
    if b is None:
        return True
    y_min, x_min, y_max, x_max = b
    return bool(y_min < edge_width or y_max > tile_size - edge_width or x_min < edge_width or x_max > tile_size - edge_width)


def generate_tiles_with_overlap(image, tile_size, overlap_ratio):
    """inference.py:2488-2519 -> [(tile_image zero-padded to tile_size, x_offset, y_offset), ...] (input preparation for the model)."""
    h, w = image.shape[:2]
    stride = int(tile_size * (1 - overlap_ratio))
    tiles = []
    for y in range(0, h, stride):
        for x in range(0, w, stride):
            tile = image[y:min(y + tile_size, h), x:min(x + tile_size, w)]
            if tile.shape[0] < tile_size or tile.shape[1] < tile_size:
                padded = np.zeros((tile_size, tile_size, 3), dtype=image.dtype)
                padded[:tile.shape[0], :tile.shape[1]] = tile
                tile = padded
            tiles.append((tile, x, y))
    return tiles


def calculate_image_quality_score(image):
    """inference.py:256-283: 0.4 * mean(gray) / 255 + 0.6 * std(gray) / 128, clipped to [0, 1].  The grey histogram comes from
    the GPU; mean and (population) standard deviation follow exactly from its integer counts."""
    from fractions import Fraction
    counts = [int(v) for v in engine.image_gray_hist(image).cpu().numpy()]
    n = sum(counts)
    s1 = sum(k * c for k, c in enumerate(counts))
    s2 = sum(k * k * c for k, c in enumerate(counts))
    brightness = (s1 / n) / 255.0
    var = Fraction(s2, n) - Fraction(s1, n) ** 2
    contrast = float(np.sqrt(np.float64(float(var)))) / 128.0
    return np.clip((0.4 * brightness) + (0.6 * contrast), 0.0, 1.0)


def adaptive_confidence_threshold(base_threshold, image, target_class, small_classes, confidence_mode='auto'):
    """inference.py:286-336 (the reference reads confidence_mode from its config; here it is an argument)."""
    if confidence_mode == "manual":
        return base_threshold
    quality_score = calculate_image_quality_score(image)
    if quality_score < 0.3:
        return base_threshold * 0.7
    if quality_score < 0.5:
        return base_threshold * 0.85
    return base_threshold


def get_confidence_threshold(image, target_class, small_classes, class_specific_settings=None, confidence_mode='auto'):
    """inference.py:339-362."""
    class_config = (class_specific_settings or {}).get(f"class_{target_class}", {})
    is_small = target_class in small_classes
    base_threshold = class_config.get("confidence_threshold", 0.3 if is_small else 0.5)
    return adaptive_confidence_threshold(base_threshold, image, target_class, small_classes, confidence_mode)


def process_masks_parallel(masks):
    """inference.py:170-213: fill holes -> erosion(disk 1) -> dilation(disk 1) for every mask (uint8 out)."""
    if len(masks) == 0:
        return []
    out = engine.process_masks_parallel(_bridge.upload(masks))
    return _bridge.download(out, None, np.uint8)


def _universal_min_size(image_shape, is_small_class, min_crys_size):
    if min_crys_size is not None:
        return min_crys_size
    area = image_shape[0] * image_shape[1]
    return max(3, int(area * 0.000005)) if is_small_class else max(25, int(area * 0.0001))


def postprocess_masks_universal(ori_mask, ori_score, image, target_class, is_small_class, min_crys_size=None):
    """inference.py:1739-1813: fill holes; small class: erosion, large class: opening; keep masks with sum >= min size (bool out)."""
    if len(ori_mask) == 0:
        return []
    iset = _bridge.upload(ori_mask)
    out, kept = engine.postprocess_masks_universal(iset, _bridge.one_group(iset.n, iset.device), is_small_class,
                                                   _universal_min_size(image.shape, is_small_class, min_crys_size))
    return _bridge.download(out, kept.to_lists()[0], bool)


def deduplicate_masks_smart(masks, scores, classes, iou_threshold=0.4, max_aspect_ratio=None, edge_filter_margin=0.3):
    """inference.py:2552-2677 (quirks Q1, Q2, Q10).  Returns the caller's own mask / score / class objects in keep order."""
    if len(masks) == 0:
        return [], [], []
    iset = _bridge.upload(masks, scores, classes)
    keep = _dedup_smart_ids(iset, iou_threshold, max_aspect_ratio)
    return [masks[i] for i in keep], [scores[i] for i in keep], [classes[i] for i in keep]


def _dedup_smart_ids(iset, iou_threshold, max_aspect_ratio=None):
    g = _bridge.one_group(iset.n, iset.device)
    engine.trace(iset)
    kept = engine.dedup_smart(iset, g, iou_threshold, max_aspect_ratio)
    flag = iset.extra.get("overflow")
    if flag is not None and int(flag.item()):
        engine.trace(iset, single_pass=False)
        kept = engine.dedup_smart(iset, g, iou_threshold, max_aspect_ratio)
    return kept.to_lists()[0]


# =================================================================================================================
# device-resident building blocks
# =================================================================================================================
@dataclass
class _Dev:
    """Instances of one image on the device + the host-side lists that go with them."""
    iset: object            # engine.InstanceSet or None when empty
    scores: list            # numpy scalars, one per instance
    classes: list
    dtypes: list            # numpy dtype each mask has when handed back to the caller (uint8 / bool)

    def __len__(self):
        return 0 if self.iset is None else self.iset.n


_EMPTY = _Dev(None, [], [], [])


def _materialise(d):
    if len(d) == 0:
        return []
    raw = engine.unpack_masks(d.iset).cpu().numpy()
    return [raw[i].astype(bool) if d.dtypes[i] is bool else raw[i] for i in range(len(d))]


def _concat(parts):
    parts = [p for p in parts if len(p)]
    if not parts:
        return _EMPTY
    if len(parts) == 1:
        return parts[0]
    iset = engine.concat([p.iset for p in parts])
    return _Dev(iset, sum((p.scores for p in parts), []), sum((p.classes for p in parts), []), sum((p.dtypes for p in parts), []))


def _select(d, idx):
    idx = list(idx)
    if not idx:
        return _EMPTY
    return _Dev(engine.select(d.iset, idx), [d.scores[i] for i in idx], [d.classes[i] for i in idx], [d.dtypes[i] for i in idx])


def _with_scores(d):
    dev = d.iset.device
    d.iset.scores = torch.as_tensor(np.asarray([float(s) for s in d.scores], np.float32), device=dev)
    d.iset.classes = torch.as_tensor(np.asarray([int(c) for c in d.classes], np.int32), device=dev)
    return d


def _predict(predictor, image):
    """predictor(image)['instances'] of the reference: K1 on the head outputs; instances dropped by Boxes.nonempty() excluded.
    Returns (InstanceSet over ALL heads, ids of the valid ones, host scores float32, host classes int64)."""
    ho = predictor.heads(image)
    H, W = image.shape[:2]
    in_h, in_w = ho.input_size
    probs = ho.probs.reshape(-1, engine.MASK_SIDE, engine.MASK_SIDE)
    if probs.dtype not in (torch.float16, torch.float32):
        probs = probs.to(torch.float32)
    probs = probs.contiguous()                  # fp16 (AMP heads) is widened exactly inside K1
    iset = engine.paste(probs, ho.boxes.to(torch.float32).contiguous(), H, W, scale_x=float(W) / float(in_w),
                        scale_y=float(H) / float(in_h))
    valid = iset.valid.cpu().numpy()
    ids = np.nonzero(valid)[0]
    scores = ho.scores.detach().cpu().numpy().astype(np.float32)[ids]
    classes = ho.classes.detach().cpu().numpy().astype(np.int64)[ids]
    return iset, ids, scores, classes


def _inorder_dedup_ids(iset, ids, thr):
    if not len(ids):
        return []
    return engine.dedup_inorder(iset, _bridge.list_group(ids, iset.device), thr).to_lists()[0]


def _dev_run_class_specific_inference(predictor, image, target_class, small_classes, confidence_threshold=0.3, iou_threshold=0.7,
                                      class_specific_settings=None, confidence_mode='auto'):
    if isinstance(predictor, list):
        return _dev_run_ensemble_inference(predictor, image, target_class, small_classes, confidence_threshold, iou_threshold,
                                           class_specific_settings=class_specific_settings, confidence_mode=confidence_mode)
    iset, ids, pred_scores, pred_classes = _predict(predictor, image)
    class_mask = pred_classes == target_class
    ids_c, scores_c = ids[class_mask], pred_scores[class_mask]
    confidence_mask = scores_c >= confidence_threshold
    filtered_ids, filtered_scores = ids_c[confidence_mask], scores_c[confidence_mask]
    if len(filtered_ids) == 0:
        return _EMPTY
    is_small_class = target_class in small_classes
    if class_specific_settings is None:
        class_specific_settings = {}
    min_size = class_specific_settings.get(f"class_{target_class}", {}).get("min_size", 5 if is_small_class else 25)
    # postprocess_masks (mask_utils.py:38-84) incl. its early exits
    if filtered_scores.all() < 0.5:
        return _EMPTY
    dev = iset.device
    post, gated = engine.postprocess_masks(iset, _bridge.list_group(filtered_ids, dev), min_size)
    proc_ids = gated.to_lists()[0]
    if len(proc_ids) > 2 and PARALLEL_MASK_PROCESSING:
        post = engine.process_masks_parallel(post)
    if not proc_ids:
        return _EMPTY
    thr = 0.5 if is_small_class else iou_threshold
    kept = _inorder_dedup_ids(post, proc_ids, thr)
    pos = {inst: k for k, inst in enumerate(proc_ids)}
    out = engine.select(post, kept)
    return _Dev(out, [filtered_scores[pos[i]] for i in kept], [target_class] * len(kept), [np.uint8] * len(kept))


def _dev_universal(iset, ids, image_shape, is_small_class, min_crys_size):
    """postprocess_masks_universal on the list `ids`: (post InstanceSet, surviving ids in order)."""
    post, kept = engine.postprocess_masks_universal(iset, _bridge.list_group(ids, iset.device), is_small_class,
                                                    _universal_min_size(image_shape, is_small_class, min_crys_size))
    return post, kept.to_lists()[0]


def _dev_run_ensemble_inference(predictors, image, target_class, small_classes, conf_threshold, iou_threshold,
                                class_specific_settings=None, confidence_mode='auto'):
    parts = []
    weights = list(ENSEMBLE_WEIGHTS.values())[:len(predictors)]
    for predictor, weight in zip(predictors, weights):
        iset, ids, pred_scores, pred_classes = _predict(predictor, image)
        if len(ids) == 0:
            continue
        class_mask = (pred_classes == target_class) & (pred_scores >= conf_threshold)
        m_ids, scores = ids[class_mask], pred_scores[class_mask]
        if len(m_ids) == 0:
            continue
        is_small_class = target_class in small_classes
        post, surv = _dev_universal(iset, m_ids, image.shape, is_small_class, None)
        pos = {inst: k for k, inst in enumerate(m_ids)}
        if surv:
            parts.append(_Dev(engine.select(post, surv), [scores[pos[i]] * weight for i in surv], [target_class] * len(surv),
                              [bool] * len(surv)))
    allp = _concat(parts)
    if len(allp) == 0:
        return _EMPTY
    _with_scores(allp)
    keep = _dedup_smart_ids(allp.iset, iou_threshold)
    return _select(allp, keep)


def _dev_run_iterative_class_inference(predictor, image, target_class, small_classes, confidence_threshold=0.3, min_crys_size=None):
    is_small_class = target_class in small_classes
    iou_threshold = 0.5 if is_small_class else 0.7
    allp = _EMPTY
    unique = _EMPTY
    prev_count = 0
    no_new_mask_iters = 0
    iteration = 0
    while True:
        iteration += 1
        iset, ids, pred_scores, pred_classes = _predict(predictor, image)
        class_mask = (pred_classes == target_class) & (pred_scores >= confidence_threshold)
        f_ids, filtered_scores = ids[class_mask], pred_scores[class_mask]
        if len(f_ids) > 0:
            post, surv = _dev_universal(iset, f_ids, image.shape, is_small_class, min_crys_size)
            if surv:
                # Q7: the i-th SURVIVOR takes the score of the i-th FILTERED detection (inference.py:2230-2234)
                new = _Dev(engine.select(post, surv), [filtered_scores[i] for i in range(len(surv))], [target_class] * len(surv),
                           [bool] * len(surv))
                allp = _concat([allp, new])
        kept = _inorder_dedup_ids(allp.iset, list(range(len(allp))), iou_threshold) if len(allp) else []
        unique = _select(allp, kept)
        new_count = len(unique)
        added = new_count - prev_count
        if added == 0:
            no_new_mask_iters += 1
        else:
            no_new_mask_iters = 0
        if no_new_mask_iters >= MAX_CONSECUTIVE_ZERO:
            break
        if new_count >= MIN_TOTAL_MASKS and iteration >= MIN_ITERATIONS:
            required_increase = max(1, int(prev_count * MIN_RELATIVE_INCREASE))
            if added < required_increase:
                break
        prev_count = new_count
        allp = unique
    return unique


def _dev_process_single_scale(predictor, image, target_class, small_classes, confidence_threshold, scale):
    if scale != 1.0:
        h, w = image.shape[:2]
        new_h, new_w = int(h * scale), int(w * scale)
        scaled_image = cv2.resize(image, (new_w, new_h), interpolation=cv2.INTER_LINEAR)     # model input preparation
    else:
        scaled_image = image
    original_image_area = image.shape[0] * image.shape[1]
    is_small_class = target_class in small_classes
    base_min_size = max(3, int(original_image_area * 0.000005)) if is_small_class else max(25, int(original_image_area * 0.0001))
    scaled_min_size = int(base_min_size * (scale ** 2))
    d = _dev_run_iterative_class_inference(predictor, scaled_image, target_class, small_classes, confidence_threshold,
                                           min_crys_size=scaled_min_size)
    if scale != 1.0 and len(d):
        back, _ = engine.resize_place(d.iset, image.shape[0], image.shape[1], image.shape[0], image.shape[1])
        d = _Dev(back, d.scores, d.classes, [bool] * len(d))
    return d


def _dev_run_adaptive_multiscale_inference(predictor, image, target_class, confidence_threshold=0.3, small_classes=set()):
    parts = []
    scale_performance = {}

    def one(scale):
        d = _dev_process_single_scale(predictor, image, target_class, small_classes, confidence_threshold, scale)
        return d

    for scale in [0.7, 1.0, 1.5]:
        d = one(scale)
        scale_performance[scale] = len(d)
        parts.append(d)
    baseline_1x = scale_performance.get(1.0, 0)
    upscale_benefit = scale_performance.get(1.5, 0) > baseline_1x * 0.1
    downscale_benefit = scale_performance.get(0.7, 0) > baseline_1x * 0.1
    for cond, scales in ((upscale_benefit, [2.0, 2.5]), (downscale_benefit, [0.5, 0.6])):
        if cond:
            for scale in scales:
                d = one(scale)
                if len(d) < baseline_1x * 0.05:
                    break
                parts.append(d)
    allp = _concat(parts)
    if len(allp) == 0:
        return _EMPTY
    _with_scores(allp)
    keep = engine.dedup_sorted(allp.iset, _bridge.one_group(len(allp), allp.iset.device), 0.4).to_lists()[0]
    return _select(allp, keep)


def _dev_tile_based_inference_pipeline(predictor, image, target_class, small_classes, confidence_threshold, tile_size=512,
                                       overlap_ratio=0.1, upscale_factor=2.0, scale_bar_info=None, iou_threshold=0.7,
                                       edge_filter_enabled=True, class_specific_settings=None, confidence_mode='auto'):
    h, w = image.shape[:2]
    full = _dev_run_class_specific_inference(predictor, image, target_class, small_classes, confidence_threshold,
                                             iou_threshold=iou_threshold, class_specific_settings=class_specific_settings,
                                             confidence_mode=confidence_mode)
    parts = [full]
    for tile_img, x_offset, y_offset in generate_tiles_with_overlap(image, tile_size, overlap_ratio):
        tile_h, tile_w = tile_img.shape[:2]
        upscaled_h, upscaled_w = int(tile_h * upscale_factor), int(tile_w * upscale_factor)
        upscaled_tile = cv2.resize(tile_img, (upscaled_w, upscaled_h), interpolation=cv2.INTER_LINEAR)     # model input preparation
        t = _dev_run_class_specific_inference(predictor, upscaled_tile, target_class, small_classes, confidence_threshold,
                                              iou_threshold=iou_threshold, class_specific_settings=class_specific_settings,
                                              confidence_mode=confidence_mode)
        if not len(t):
            continue
        off = np.tile(np.array([[x_offset, y_offset]], np.int32), (len(t), 1))
        placed, edge = engine.resize_place(t.iset, tile_h, tile_w, h, w, off_xy=off, tile_size=tile_size, overlap_ratio=overlap_ratio)
        d = _Dev(placed, t.scores, t.classes, [bool] * len(t))
        if edge_filter_enabled:
            keep = np.nonzero(edge.cpu().numpy()[:len(t)] == 0)[0].tolist()
            d = _select(d, keep)
        parts.append(d)
    allp = _concat(parts)
    if len(allp) == 0:
        return _EMPTY
    _with_scores(allp)
    keep = _dedup_smart_ids(allp.iset, 0.4)
    return _select(allp, keep)


# =================================================================================================================
# the reference's entry points (lists of numpy masks in / out)
# =================================================================================================================
def _lists(d, empty_as_arrays=False):
    if len(d) == 0:
        return (np.array([]), np.array([]), np.array([])) if empty_as_arrays else ([], [], [])
    return _materialise(d), list(d.scores), list(d.classes)


def run_class_specific_inference(predictor, image, target_class, small_classes, confidence_threshold=0.3, iou_threshold=0.7,
                                 class_specific_settings=None, confidence_mode='auto'):
    """inference.py:1353-1461."""
    d = _dev_run_class_specific_inference(predictor, image, target_class, small_classes, confidence_threshold, iou_threshold,
                                          class_specific_settings, confidence_mode)
    return _lists(d, empty_as_arrays=isinstance(predictor, list))


def run_ensemble_inference(predictors, image, target_class, small_classes, conf_threshold, iou_threshold,
                           class_specific_settings=None, confidence_mode='auto'):
    """inference.py:1464-1600: per model class/confidence filter -> postprocess_masks_universal -> score * weight ->
    deduplicate_masks_smart.  Empty result: three empty numpy arrays (:1586)."""
    d = _dev_run_ensemble_inference(predictors, image, target_class, small_classes, conf_threshold, iou_threshold,
                                    class_specific_settings, confidence_mode)
    return _lists(d, empty_as_arrays=True)


def run_iterative_class_inference(predictor, image, target_class, small_classes, confidence_threshold=0.3, min_crys_size=None):
    """inference.py:2069-2297 (Q7 reproduced)."""
    return _lists(_dev_run_iterative_class_inference(predictor, image, target_class, small_classes, confidence_threshold, min_crys_size))


def process_single_scale(predictor, image, target_class, small_classes, confidence_threshold, scale):
    """inference.py:1987-2066."""
    return _lists(_dev_process_single_scale(predictor, image, target_class, small_classes, confidence_threshold, scale))


def run_adaptive_multiscale_inference(predictor, image, target_class, confidence_threshold=0.3, small_classes=set()):
    """inference.py:1833-1984."""
    return _lists(_dev_run_adaptive_multiscale_inference(predictor, image, target_class, confidence_threshold, small_classes))


def run_multiscale_class_inference(predictor, image, target_class, confidence_threshold=0.3, small_classes=set()):
    """inference.py:1816-1830."""
    return run_adaptive_multiscale_inference(predictor, image, target_class, confidence_threshold, small_classes)


def tile_based_inference_pipeline(predictor, image, target_class, small_classes, confidence_threshold, tile_size=512,
                                  overlap_ratio=0.1, upscale_factor=2.0, scale_bar_info=None, iou_threshold=0.7,
                                  edge_filter_enabled=True, class_specific_settings=None, confidence_mode='auto'):
    """inference.py:2299-2485: full-image pass + upscaled tiles, NEAREST back-projection, edge filter, global
    deduplicate_masks_smart at 0.4 (Q8)."""
    d = _dev_tile_based_inference_pipeline(predictor, image, target_class, small_classes, confidence_threshold, tile_size,
                                           overlap_ratio, upscale_factor, scale_bar_info, iou_threshold, edge_filter_enabled,
                                           class_specific_settings, confidence_mode)
    return _lists(d)


# =================================================================================================================
# measurement loop + CSV (inference.py:987-1010, :1148-1253) and the per-image part of run_inference (:776-905)
# =================================================================================================================
def measure_masks(masks, classes, image_shape, um_pix, test_img, psum, class_names=None, original_image=None, shape_columns=False):
    """Rows of measurements_results.csv for one image: one row per external contour whose contourArea reaches the gate (Q12).
    shape_columns: the row continues after "File name" with the ten SHAPE_HEADER values (engine.shape_descriptors) as Python
    floats."""
    if (masks.n if isinstance(masks, engine.InstanceSet) else len(masks)) == 0:
        return []
    iset = masks if isinstance(masks, engine.InstanceSet) else _bridge.upload(masks)
    engine.measure(iset, um_pix=um_pix, min_area=engine.default_min_area(image_shape[0], image_shape[1]))
    rec = iset.records.cpu().numpy()
    cont_off = iset.cont_off.cpu().numpy()
    shape = engine.shape_descriptors(iset).cpu().numpy() if shape_columns else None
    hist = None
    if measure_contrast_distribution and original_image is not None:
        from ..utils.contrast import percentiles_from_counts
        hist = engine.gray_hist(iset, original_image).cpu().numpy()
    rows = []
    for k, cls in enumerate(classes):
        cls = int(cls)
        name = class_names[cls] if class_names is not None and cls < len(class_names) else f"class_{cls}"
        for j in range(cont_off[k], cont_off[k + 1]):
            if rec[j, engine.REC_MEASURED] != 1.0:
                continue
            m = record_to_dict(rec[j])
            if hist is not None:
                m["contrast_d10"], m["contrast_d50"], m["contrast_d90"] = percentiles_from_counts(hist[k])
            rows.append([f"{test_img}_{k + 1}", cls, name] + [m[key] for key in KEY_ORDER] + [psum, test_img] +
                        ([float(v) for v in shape[j]] if shape is not None else []))
    return rows


def _measure_text(iset, classes, image_shape, um_pix, test_img, psum, class_names=None, original_image=None, shape_columns=False):
    """measure_masks' rows as the text csv.writer writes for them, formatted on the device (engine.measurements_csv_text)."""
    if iset.n == 0:
        return b""
    engine.measure(iset, um_pix=um_pix, min_area=engine.default_min_area(image_shape[0], image_shape[1]))
    fields, class_idx = _class_table(classes, class_names)
    return engine.measurements_csv_text(iset, test_img, psum, class_idx, fields, _contrast(iset, original_image),
                                        engine.shape_descriptors(iset) if shape_columns else None)


def neighbour_rows(iset, nb, file_name, psum, class_idx, class_fields):
    """Rows of neighbours_results.csv for one image from the device values of nb = engine.neighbours(iset, class_idx, ...): one per
    listed instance, in instance order, as Python values (None for an empty field).  The reference for the device text of
    engine.neighbours_csv_text, as measure_masks is for the measurement rows."""
    vals = nb.values.cpu().numpy()
    ints = nb.ints.cpu().numpy()
    ident = lambda k: f"{file_name}_{int(k) + 1}"                                   # noqa: E731
    rows = []
    for k in range(iset.n):
        listed, nn, closest, touching, agg, size = (int(v) for v in ints[k])
        if not listed:
            continue
        cls, name = class_fields[int(class_idx[k])]
        has = nn >= 0
        rows.append([ident(k), cls, name, float(vals[k, 0]), float(vals[k, 1]), ident(nn) if has else None,
                     float(vals[k, 2]) if has else None, ident(closest) if has else None, float(vals[k, 3]) if has else None, touching,
                     ident(agg), size, psum, file_name])
    return rows


def _class_table(classes, class_names):
    """(Class, Class_Name) pairs of the distinct classes as measure_masks names them, and each instance's index among them.
    class_names: a list indexed by class, or a dict {class: name}; a class it does not name is class_<class>."""
    fields, index, class_idx = [], {}, []
    for cls in classes:
        cls = int(cls)
        if cls not in index:
            index[cls] = len(fields)
            if isinstance(class_names, dict):
                name = class_names.get(cls, f"class_{cls}")
            else:
                name = class_names[cls] if class_names is not None and cls < len(class_names) else f"class_{cls}"
            fields.append((cls, name))
        class_idx.append(index[cls])
    return fields, class_idx


def _contrast(iset, original_image):
    """float64 [n, 3] contrast d10 / d50 / d90 per instance (NaN where measure_masks writes None), or None when not measured."""
    if not (measure_contrast_distribution and original_image is not None):
        return None
    from ..utils.contrast import percentiles_from_counts
    hist = engine.gray_hist(iset, original_image).cpu().numpy()
    return np.array([[np.nan if v is None else v for v in percentiles_from_counts(h)] for h in hist], np.float64).reshape(-1, 3)


def _infer_image_dev(predictors, image, num_classes, small_classes, class_specific_settings=None, confidence_mode='manual',
                     confidence_fn=None, tile_size=512, overlap_ratio=0.1, upscale_factor=2.0, edge_filter_enabled=True,
                     ensemble_enabled=True, ensemble_small_only=True, classes_to_infer=None, spatial_rules=None, dataset_name=None):
    """The per-image body of run_inference (inference.py:776-905) with the result left on the device (_Dev)."""
    class_specific_settings = class_specific_settings or {}
    parts = []
    target_classes = range(num_classes) if classes_to_infer is None else [c for c in classes_to_infer if c < num_classes]
    for target_class in target_classes:
        is_small_class = target_class in small_classes
        class_cfg = class_specific_settings.get(f"class_{target_class}", {})
        if confidence_mode == 'manual':
            confidence_thresh = class_cfg.get("confidence_threshold", 0.3 if is_small_class else 0.5)
        elif confidence_fn is not None:
            confidence_thresh = confidence_fn(image, target_class, small_classes)
        else:
            confidence_thresh = get_confidence_threshold(image, target_class, small_classes, class_specific_settings, confidence_mode)
        iou_thresh = class_cfg.get("iou_threshold", 0.5 if is_small_class else 0.7)
        use_ensemble = ensemble_enabled and (not ensemble_small_only or is_small_class)
        active = predictors if (use_ensemble and len(predictors) > 1) else [predictors[0]]
        parts.append(_dev_tile_based_inference_pipeline(active[0] if len(active) == 1 else active, image, target_class, small_classes,
                                                        confidence_thresh, tile_size=tile_size, overlap_ratio=overlap_ratio,
                                                        upscale_factor=upscale_factor, iou_threshold=iou_thresh,
                                                        edge_filter_enabled=edge_filter_enabled,
                                                        class_specific_settings=class_specific_settings, confidence_mode=confidence_mode))
    allp = _concat(parts)
    if len(allp) == 0:
        return _EMPTY
    _with_scores(allp)
    keep = _dedup_smart_ids(allp.iset, 0.7)
    final = _select(allp, keep)
    if len(final):
        rules = spatial_rules
        if rules is None and _sc._constraint_loader is not None:
            rules = _sc._constraint_loader(dataset_name)
        if rules and rules.get('enabled', False):
            _with_scores(final)
            k2 = engine.apply_spatial_constraints(final.iset, _bridge.one_group(len(final), final.iset.device), rules).to_lists()[0]
            final = _select(final, k2)
    return final


def infer_image(predictors, image, num_classes, small_classes, **kwargs):
    """The per-image body of run_inference (inference.py:776-905): per class tile_based_inference_pipeline, cross-class
    deduplicate_masks_smart at 0.7, apply_spatial_constraints.  Returns (masks, scores, classes) as the reference's lists."""
    return _lists(_infer_image_dev(predictors, image, num_classes, small_classes, **kwargs))


# class colours of the overlay / legend, BGR (src/functions/inference.py:972-981)
CLASS_COLORS_BGR = [(0, 255, 0), (255, 0, 0), (0, 0, 255), (255, 255, 0), (255, 0, 255), (0, 255, 255), (128, 0, 128), (255, 165, 0)]


def write_class_color_legend(output_dir, thing_classes):
    """class_color_legend.txt as run_inference writes it (src/functions/inference.py:1302-1314): one line per class with the
    overlay colour converted from BGR to RGB."""
    path = os.path.join(output_dir, "class_color_legend.txt")
    with open(path, "w") as f:
        f.write("Class Color Legend:\n")
        f.write("==================\n")
        for i, class_name in enumerate(thing_classes):
            b, g, r = CLASS_COLORS_BGR[i % len(CLASS_COLORS_BGR)]
            f.write(f"Class {i} ({class_name}): RGB{(r, g, b)}\n")
    return path


# ---- providers: what the reference's run_inference pulls from its own subsystems (config, dataset registry, model zoo, image
# folder, scale-bar OCR).  A host application registers them once; run_inference is then callable exactly as main.py:480-488 does.
_PROVIDERS = {"config": None, "thing_classes": None, "predictors": None, "images": None, "scale_bar": None}


def set_providers(config=None, thing_classes=None, predictors=None, images=None, scale_bar=None):
    """config(dataset_name) -> dict (the reference's get_config(dataset_name=...): `inference_settings` / `inference_overrides`,
    `scale_bar_rois`); thing_classes(dataset_name) -> [names] (MetadataCatalog ...thing_classes); predictors(dataset_name,
    threshold, thing_classes) -> [head adapters] (R50, R101 order; deepemia_b200.adapters); images(dataset_name) -> iterable of
    (file name, BGR uint8 image); scale_bar(image, roi_config, dataset_name) -> (psum, um_pix) (detect_scale_bar).
    Passing None leaves a provider unchanged; spatial rules come from utils.spatial_constraints.set_constraint_loader."""
    for k, v in (("config", config), ("thing_classes", thing_classes), ("predictors", predictors), ("images", images),
                 ("scale_bar", scale_bar)):
        if v is not None:
            _PROVIDERS[k] = v


def clear_providers():
    for k in _PROVIDERS:
        _PROVIDERS[k] = None


def _resolve_images(dataset_name, images):
    """The (file name, image) pairs of a run: the given ones, else the images provider's, else None."""
    return images if images is not None else (_PROVIDERS["images"](dataset_name) if _PROVIDERS["images"] else None)


def _dataset_config(dataset_name):
    cfg_fn = _PROVIDERS["config"]
    return cfg_fn(dataset_name) if cfg_fn else {}


def _stem(name):
    """The ImageId of an image's rows in R50_flip_results.csv: its file name without the extension."""
    return name.rsplit(".", 1)[0]


def _scale_bars(images, dataset_name, dataset_config, output_dir, scale_bar_fn=None, draw_scalebar=False):
    """(psum, um_pix) of every image, in order, as run_inference resolves them (inference.py:744-773): scale_bar_fn, else the
    scale_bar provider, else the package's own detector (batched over all images when there is more than one), else ("0", 1.0).
    An iterator: an image's own detection (and, with draw_scalebar, its debug overlay) happens when its value is taken."""
    cfg_fn = _PROVIDERS["config"]
    rois = dataset_config.get("scale_bar_rois", {})
    roi_config = rois.get(dataset_name, rois.get("default", {"x_start_factor": 0.667, "y_start_factor": 0.866, "width_factor": 1.0,
                                                            "height_factor": 0.067}))
    user_fn = scale_bar_fn or ((lambda im: _PROVIDERS["scale_bar"](im, roi_config, dataset_name)) if _PROVIDERS["scale_bar"] else None)
    from ..utils import scalebar_ocr as _sb
    if cfg_fn and _sb._state["config"] is None:
        _sb.set_config_provider(cfg_fn)
    own_detector = user_fn is None and (_sb._state["ocr"] is not None or _sb.easyocr_available())

    def scale_bar(im, name):
        if user_fn is not None:
            return user_fn(im)
        if not own_detector:
            return "0", 1.0
        # the reference's own call (inference.py:751-762): on a copy; with draw_scalebar the debug overlay is saved next to the results
        work = im.copy()
        r = _sb.detect_scale_bar(work, roi_config=roi_config, dataset_name=dataset_name, draw_debug=bool(draw_scalebar))
        if draw_scalebar:
            cv2.imwrite(os.path.join(output_dir, f"{name}_scalebar_debug.png"), work)
        return r
    # the scale bars of ALL images in one launch per stage (and frame size) when the package's own detector is in use; a failure
    # of the batch falls back to the reference's per-image call with its per-image try / except (inference.py:750-773)
    batch_bars = None
    if own_detector and not draw_scalebar and len(images) > 1:
        try:
            batch_bars = _sb.detect_scale_bars([im for _, im in images], roi_config=roi_config, dataset_name=dataset_name)
        except Exception:
            batch_bars = None

    def each():
        for k, (name, image) in enumerate(images):
            try:
                bar = batch_bars[k] if batch_bars is not None else scale_bar(image, name)
            except Exception:
                bar = "0", 1.0                                          # inference.py:767-773
            yield bar
    return each()


def _write_csv(path, header, texts):
    """A result file: csv.writer's header line, then the device-formatted rows."""
    with open(path, "wb") as f:
        f.write((",".join(engine.csv_field(h) for h in header) + "\r\n").encode("utf-8"))
        for t in texts:
            f.write(t)


def _write_coco(path, images, ann_texts, thing_classes, classes):
    """coco_instances.json: json.dumps of {"images", "annotations", "categories"}, the annotations being the device texts."""
    cats = [{"id": k, "name": n} for k, n in enumerate(thing_classes)]
    cats += [{"id": c, "name": f"class_{c}"} for c in sorted(classes) if c >= len(thing_classes)]
    with open(path, "wb") as f:
        f.write((json.dumps({"images": images})[:-1] + ', "annotations": [').encode())
        f.write(b", ".join(t for t in ann_texts if t))
        f.write(('], "categories": ' + json.dumps(cats) + "}").encode())


def run_inference(dataset_name, output_dir, visualize=True, threshold=0.65, draw_id=False, dataset_format="json", draw_scalebar=False,
                  *, images=None, predictors=None, thing_classes=None, small_classes=None, scale_bar_fn=None, shape_columns=False,
                  neighbours=False, coco_json=False, **infer_kwargs):
    """run_inference (src/functions/inference.py:499-1351), same signature and call shape as main.py:480-488:

        run_inference(dataset_name, output_dir, visualize=..., threshold=..., draw_id=..., dataset_format=..., draw_scalebar=...)

    with the reference's own subsystems behind registered providers (set_providers) or the keyword-only overrides.  Settings are
    read from the dataset config exactly as :517-556 does (confidence mode, class-specific settings, tile / ensemble settings,
    classes_to_infer); small classes come from the mask-size heuristic (:719-723) unless given.  Per image: scale bar ->
    per-class tile pipeline -> cross-class de-dup -> spatial constraints (:776-905), all on the device; the RLE rows of
    R50_flip_results.csv and the rows of measurements_results.csv are produced from the SAME device-resident instance set (one
    K6 and one K5 pass per image, no mask round trip).  Writes R50_flip_results.csv, measurements_results.csv,
    class_color_legend.txt and, with visualize, <name>_predictions.png (overlay kernel + labels).  shape_columns: each row of
    measurements_results.csv continues after "File name" with the ten SHAPE_HEADER columns (area, convex hull, Feret diameters,
    centroid: engine.shape_descriptors).  neighbours: also writes neighbours_results.csv (NEIGHBOUR_HEADER: nearest neighbour, edge
    distance, touching neighbours and agglomerate of every instance with rows in measurements_results.csv; engine.neighbours).
    coco_json: also writes coco_instances.json, COCO instance JSON with compressed RLE (oracle/coco.py defines it): every image, one
    annotation per line of R50_flip_results.csv (category_id = Class, the score of the final set), formatted on the device
    (engine.coco_annotations_text) from the same K6 runs."""
    images = _resolve_images(dataset_name, images)
    if thing_classes is None and _PROVIDERS["thing_classes"]:
        thing_classes = _PROVIDERS["thing_classes"](dataset_name)
    thing_classes = list(thing_classes or [])
    if predictors is None and _PROVIDERS["predictors"]:
        predictors = _PROVIDERS["predictors"](dataset_name, threshold, thing_classes)
    if images is None or not predictors:
        raise FileNotFoundError(f"No trained models / images registered for dataset '{dataset_name}': call "
                                "deepemia_b200.functions.inference.set_providers(...) (or pass images= and predictors=)")
    images = list(images)
    dataset_config = _dataset_config(dataset_name)
    inf_settings = dataset_config.get("inference_overrides", {}) or dataset_config.get("inference_settings", {})
    tile_cfg = inf_settings.get("tile_settings", {})
    ens_cfg = inf_settings.get("ensemble_settings", {})
    kw = dict(class_specific_settings=inf_settings.get("class_specific_settings", {}),
              confidence_mode=inf_settings.get("confidence_mode", "auto"),
              tile_size=tile_cfg.get("tile_size", 512), overlap_ratio=tile_cfg.get("overlap_ratio", 0.1),
              upscale_factor=tile_cfg.get("upscale_factor", 2.0), edge_filter_enabled=tile_cfg.get("edge_filter_enabled", True),
              ensemble_enabled=ens_cfg.get("enabled", True), ensemble_small_only=ens_cfg.get("small_classes_only", True),
              classes_to_infer=inf_settings.get("inference_settings", {}).get("classes_to_infer", None))
    kw.update(infer_kwargs)
    num_classes = len(thing_classes) if thing_classes else int(kw.pop("num_classes", 1))
    kw.pop("num_classes", None)
    if small_classes is None:
        from ..adapters import calculate_average_mask_sizes, determine_small_classes
        small_classes = determine_small_classes(calculate_average_mask_sizes(predictors, [im for _, im in images[:5]]), 50)
    small_classes = set(small_classes)
    os.makedirs(output_dir, exist_ok=True)
    bars = _scale_bars(images, dataset_name, dataset_config, output_dir, scale_bar_fn, draw_scalebar)
    rle_text, meas_text, nb_text = [], [], []
    coco_images, coco_ann, coco_classes, n_ann = [], [], set(), 0
    shape_kw = {"shape_columns": True} if shape_columns else {}      # without the option, _measure_text is called as it always was
    for (name, image), (psum, um_pix) in zip(images, bars):
        d = _infer_image_dev(predictors, image, num_classes, small_classes, dataset_name=dataset_name, **kw)
        if coco_json:
            coco_images.append({"id": len(coco_images) + 1, "file_name": name, "height": int(image.shape[0]),
                                "width": int(image.shape[1])})
        if len(d) == 0:
            continue
        run_off, runs = engine.rle_encode(d.iset)                       # K6 over the final set, once
        rle_text.append(engine.rle_csv_text(run_off, runs, _stem(name)))
        if coco_json:
            coco_ann.append(engine.coco_annotations_text(d.iset, run_off, runs, len(coco_images), d.classes, d.scores, n_ann + 1))
            coco_classes.update(int(c) for c in d.classes)
            n_ann += len(d)
        meas_text.append(_measure_text(d.iset, d.classes, image.shape, um_pix, name, psum, class_names=thing_classes,
                                       original_image=image, **shape_kw))
        if neighbours:
            fields, class_idx = _class_table(d.classes, thing_classes)
            nb = engine.neighbours(d.iset, class_idx, um_pix)
            nb_text.append(engine.neighbours_csv_text(d.iset, nb, name, psum, class_idx, fields))
        if visualize:
            from ..utils.visualize import render_predictions
            cv2.imwrite(os.path.join(output_dir, f"{name}_predictions.png"), render_predictions(image, d.iset, d.classes, thing_classes))
    _write_csv(os.path.join(output_dir, "R50_flip_results.csv"), ["ImageId", "EncodedPixels"], rle_text)
    _write_csv(os.path.join(output_dir, "measurements_results.csv"), CSV_HEADER + (SHAPE_HEADER if shape_columns else []), meas_text)
    if neighbours:
        _write_csv(os.path.join(output_dir, "neighbours_results.csv"), NEIGHBOUR_HEADER, nb_text)
    if coco_json:
        _write_coco(os.path.join(output_dir, "coco_instances.json"), coco_images, coco_ann, thing_classes, coco_classes)
    write_class_color_legend(output_dir, thing_classes)
    return None


# =================================================================================================================
# reading saved results back: R50_flip_results.csv -> instances (RLE decode on the device) -> a new measurements_results.csv
# =================================================================================================================
def load_rle_results(path, images):
    """R50_flip_results.csv -> {file name: engine.InstanceSet} for the (file name, image) pairs `images` that run_inference takes.
    Rows match an image by stem, as run_inference writes them; instance k of an image is the k-th row with its ImageId, in file
    order; an image without rows maps to an empty set.  The file is parsed once and decoded once per distinct frame size, on the
    device.  Raises ValueError when two names share a stem, EmiaError naming the line of a malformed row or of an ImageId that
    matches no image."""
    images = list(images)
    by_stem = {}
    for k, (name, _) in enumerate(images):
        stem = _stem(name)
        if stem in by_stem:
            raise ValueError(f"load_rle_results: {images[by_stem[stem]][0]!r} and {name!r} share the ImageId {stem!r}")
        by_stem[stem] = k
    with open(path, "rb") as f:
        data = f.read()
    try:
        ids, run_off, runs, line_no = engine._rle_parse(data)
    except engine._lib.EmiaError as e:
        raise engine._lib.EmiaError(f"{path}: {e}") from None
    rows_of = [[] for _ in images]
    for r, stem in enumerate(ids):
        k = by_stem.get(stem)
        if k is None:
            raise engine._lib.EmiaError(f"{path}: line {line_no[r]}: ImageId {stem!r} matches no image")
        rows_of[k].append(r)
    by_size = {}
    for k, (_, image) in enumerate(images):
        by_size.setdefault(tuple(int(s) for s in image.shape[:2]), []).append(k)
    out, bad = {}, []
    for (H, W), ks in by_size.items():
        rows = [r for k in ks for r in rows_of[k]]
        iset, status = engine._rle_decode(run_off, runs, H, W, rows)
        bad += [(int(line_no[rows[j]]), int(status[j])) for j in np.nonzero(status)[0][:1]]
        a = 0
        for k in ks:
            m = len(rows_of[k])
            out[images[k][0]] = iset if len(ks) == 1 else engine.select(iset, list(range(a, a + m)))
            a += m
    if bad:
        line, code = min(bad)
        raise engine._lib.EmiaError(f"{path}: line {line}: {engine.RLE_STATUS[code]}")
    return out


def remeasure_results(dataset_name, results_dir, output_dir, *, images=None, scale_bar_fn=None, shape_columns=False, neighbours=False):
    """Measure the masks a run_inference call saved in results_dir again, without the models: writes output_dir/
    measurements_results.csv as run_inference would with the scale bars (and settings such as measure_contrast_distribution) of
    now.  Images and scale bars resolve exactly as in run_inference (images= / the images provider; scale_bar_fn / the scale_bar
    provider / the package's detector).  Class and Class_Name of an instance are those of its rows in results_dir's
    measurements_results.csv; an instance without rows there has no contour above the area gate (which depends only on the frame
    size) and gets none here either.  shape_columns: as in run_inference, whether or not the old file has them.  neighbours: also
    writes output_dir/neighbours_results.csv as run_inference does, with the classes of the old rows."""
    if os.path.realpath(output_dir) == os.path.realpath(results_dir):
        raise ValueError("remeasure_results: output_dir must differ from results_dir (its measurements_results.csv is an input)")
    images = _resolve_images(dataset_name, images)
    if images is None:
        raise FileNotFoundError(f"No images registered for dataset '{dataset_name}': call "
                                "deepemia_b200.functions.inference.set_providers(...) (or pass images=)")
    images = list(images)
    sets = load_rle_results(os.path.join(results_dir, "R50_flip_results.csv"), images)
    with open(os.path.join(results_dir, "measurements_results.csv"), newline="") as f:
        old = list(csv.reader(f))
    if not old or old[0] not in (CSV_HEADER, CSV_HEADER + SHAPE_HEADER):
        raise ValueError(f"remeasure_results: {results_dir}/measurements_results.csv does not start with the measurements header")
    class_of = {r[0]: (r[1], r[2]) for r in old[1:]}
    os.makedirs(output_dir, exist_ok=True)
    texts, nb_text = [], []
    for (name, image), (psum, um_pix) in zip(images, _scale_bars(images, dataset_name, _dataset_config(dataset_name), output_dir,
                                                                  scale_bar_fn)):
        iset = sets[name]
        measured = _measure_saved(iset, image, um_pix)
        if len(measured) == 0:
            continue
        index, class_idx = {}, [0] * iset.n         # (Class, Class_Name) of the old rows -> index; unmeasured instances: unused
        for k in measured.tolist():
            key = f"{name}_{k + 1}"
            if key not in class_of:
                raise ValueError(f"remeasure_results: {key} has a measured contour but no row in {results_dir}/measurements_results.csv")
            class_idx[k] = index.setdefault(class_of[key], len(index))
        _saved_texts(texts, nb_text, iset, name, image, psum, um_pix, class_idx, list(index), shape_columns, neighbours)
    _write_results(output_dir, texts, nb_text, shape_columns, neighbours)


def _measure_saved(iset, image, um_pix):
    """engine.measure of an image's saved instances -> the ids (ascending) of those with a measured contour."""
    if iset.n == 0:
        return np.zeros(0, np.int64)
    engine.measure(iset, um_pix=um_pix, min_area=engine.default_min_area(image.shape[0], image.shape[1]))
    return np.unique(iset.rec_inst[iset.records[:, engine.REC_MEASURED] == 1.0].cpu().numpy())


def _saved_texts(texts, nb_text, iset, name, image, psum, um_pix, class_idx, class_fields, shape_columns, neighbours):
    """The measurements_results.csv rows (and neighbours_results.csv rows) of one image's measured saved instances."""
    texts.append(engine.measurements_csv_text(iset, name, psum, class_idx, class_fields, _contrast(iset, image),
                                              engine.shape_descriptors(iset) if shape_columns else None))
    if neighbours:
        nb = engine.neighbours(iset, class_idx, um_pix)
        nb_text.append(engine.neighbours_csv_text(iset, nb, name, psum, class_idx, class_fields))


def _write_results(output_dir, texts, nb_text, shape_columns, neighbours):
    _write_csv(os.path.join(output_dir, "measurements_results.csv"), CSV_HEADER + (SHAPE_HEADER if shape_columns else []), texts)
    if neighbours:
        _write_csv(os.path.join(output_dir, "neighbours_results.csv"), NEIGHBOUR_HEADER, nb_text)


# =================================================================================================================
# COCO instance JSON (coco_instances.json, or any COCO file with compressed-RLE masks) -> instances -> measurements_results.csv
# =================================================================================================================
def _coco_error(path, ann, why):
    return ValueError(f"{path}: annotation {ann.get('id')!r}: {why}")


def _decode_coco(path, names, sizes, d=None):
    """(file dict, per-image [(counts bytes, category, score or None, annotation)] in file order, [((H, W), image positions,
    InstanceSet of their annotations in that order)] with one decode per distinct frame size) of a COCO instance file, for the
    images `names` of frame sizes `sizes`.  d: the file, already parsed."""
    by_name = {}
    for k, name in enumerate(names):
        if name in by_name:
            raise ValueError(f"load_coco_results: the file name {name!r} is given twice")
        by_name[name] = k
    if d is None:
        with open(path, "rb") as f:
            d = json.loads(f.read())
    img_of, matched = {}, set()
    for e in d.get("images", []):
        name = e.get("file_name")
        k = by_name.get(name)
        if k is None:
            raise ValueError(f"{path}: image {e.get('id')!r}: file_name {name!r} matches no image")
        if k in matched:
            raise ValueError(f"{path}: image {e.get('id')!r}: file_name {name!r} appears twice")
        if e.get("id") in img_of:
            raise ValueError(f"{path}: image id {e.get('id')!r} appears twice")
        img_of[e.get("id")] = k
        matched.add(k)
    per = [[] for _ in names]                      # (counts bytes, category, score or None, annotation) per image, file order
    for ann in d.get("annotations", []):
        seg = ann.get("segmentation")
        if not isinstance(seg, dict) or not isinstance(seg.get("counts"), str):
            raise _coco_error(path, ann, "only compressed-RLE segmentations are read (not polygons or uncompressed counts lists)")
        if ann.get("image_id") not in img_of:
            raise _coco_error(path, ann, f"image_id {ann.get('image_id')!r} has no images entry")
        k = img_of[ann["image_id"]]
        H, W = sizes[k]
        if list(seg.get("size", [])) != [H, W]:
            raise _coco_error(path, ann, f"size {seg.get('size')!r} is not the image's [{H}, {W}]")
        cat = ann.get("category_id")
        if isinstance(cat, bool) or not isinstance(cat, int) or not 0 <= cat <= 2 ** 31 - 1:
            raise _coco_error(path, ann, f"category_id {cat!r} is not a non-negative integer")
        per[k].append((seg["counts"].encode("utf-8"), cat, ann.get("score"), ann))
    by_size = {}
    for k, hw in enumerate(sizes):
        by_size.setdefault(tuple(hw), []).append(k)
    groups, bad = [], []
    for (H, W), ks in by_size.items():
        items = [it for k in ks for it in per[k]]
        raw = [it[0] for it in items]
        off = np.concatenate([[0], np.cumsum([len(b) for b in raw])]).astype(np.int64)
        iset, status = engine._coco_decode(b"".join(raw), off, H, W)
        bad += [(items[j][3], int(status[j])) for j in np.nonzero(status)[0][:1]]
        groups.append(((H, W), ks, iset))
    if bad:
        ann, code = min(bad, key=lambda b: d["annotations"].index(b[0]))
        raise engine._lib.EmiaError(f"{path}: annotation {ann.get('id')!r}: {engine.COCO_STATUS[code]}")
    return d, per, groups


def _load_coco(path, images):
    """(file dict, {file name: InstanceSet with classes / scores}) of a COCO instance file for the (file name, image) pairs."""
    images = list(images)
    d, per, groups = _decode_coco(path, [name for name, _ in images], [tuple(int(v) for v in im.shape[:2]) for _, im in images])
    out = {}
    for _, ks, iset in groups:
        a = 0
        for k in ks:
            m = len(per[k])
            s = iset if len(ks) == 1 else engine.select(iset, list(range(a, a + m)))
            dev = s.device
            s.classes = torch.as_tensor(np.asarray([it[1] for it in per[k]], np.int32), device=dev)
            scores = [it[2] for it in per[k]]
            s.scores = torch.as_tensor(np.asarray(scores, np.float32), device=dev) if all(
                isinstance(v, (int, float)) and not isinstance(v, bool) for v in scores) else None
            out[images[k][0]] = s
            a += m
    return d, out


def load_coco_results(path, images):
    """A COCO instance JSON file with compressed-RLE masks (coco_instances.json of run_inference, an annotation tool's export, a
    dataset's ground truth) -> {file name: engine.InstanceSet} for the (file name, image) pairs `images` that run_inference takes.
    Images are matched by file_name; instance k of an image is its k-th annotation in file order; an image without annotations maps
    to an empty set.  iset.classes (int32) holds the category_id values and iset.scores (float32) the scores when every annotation
    of the image has one.  The file is parsed with json.loads; the counts strings are decoded on the device, once per distinct frame
    size, into the tight bbox crops rle_decode gives.  Raises ValueError for a polygon or uncompressed segmentation, a size that is
    not the image's, an image_id without images entry, a category_id that is not a non-negative integer (each naming the
    annotation's id), an images entry that matches no image or a file name given twice; EmiaError naming the annotation of a
    malformed counts string."""
    return _load_coco(path, images)[1]


def measure_coco(path, output_dir, *, images=None, dataset_name=None, scale_bar_fn=None, shape_columns=False, neighbours=False):
    """Measure the masks of a COCO instance JSON file (load_coco_results): writes output_dir/measurements_results.csv (and, with
    neighbours, neighbours_results.csv) as run_inference writes them for the same masks.  Class is the category_id; Class_Name its
    name in the file's categories (class_<id> when it has none).  Images and scale bars resolve as in remeasure_results (images= /
    the images provider; scale_bar_fn / the scale_bar provider / the package's detector); shape_columns as in run_inference."""
    images = _resolve_images(dataset_name, images)
    if images is None:
        raise FileNotFoundError(f"No images registered for dataset '{dataset_name}': call "
                                "deepemia_b200.functions.inference.set_providers(...) (or pass images=)")
    images = list(images)
    d, sets = _load_coco(path, images)
    names = {c.get("id"): c.get("name") for c in d.get("categories", [])}
    os.makedirs(output_dir, exist_ok=True)
    texts, nb_text = [], []
    for (name, image), (psum, um_pix) in zip(images, _scale_bars(images, dataset_name, _dataset_config(dataset_name), output_dir,
                                                                  scale_bar_fn)):
        iset = sets[name]
        if len(_measure_saved(iset, image, um_pix)) == 0:
            continue
        fields, class_idx = _class_table(iset.classes.cpu().numpy().tolist(), names)
        _saved_texts(texts, nb_text, iset, name, image, psum, um_pix, class_idx, fields, shape_columns, neighbours)
    _write_results(output_dir, texts, nb_text, shape_columns, neighbours)


# =================================================================================================================
# COCO segm evaluation of a detections file against a ground-truth file (definition: oracle/cocoeval.py)
# =================================================================================================================
COCO_EVAL_HEADER = ["Metric", "Category", "IoU", "Area", "MaxDets", "Value"]
# (AP or AR, IoU threshold or None for .50:.95, area range, index into max_dets) of COCOeval.summarize's 12 segm stats
COCO_STAT_ROWS = [(1, None, "all", 2), (1, .5, "all", 2), (1, .75, "all", 2), (1, None, "small", 2), (1, None, "medium", 2),
                  (1, None, "large", 2), (0, None, "all", 0), (0, None, "all", 1), (0, None, "all", 2), (0, None, "small", 2),
                  (0, None, "medium", 2), (0, None, "large", 2)]


def _coco_mean(s):
    return float(np.mean(s[s > -1])) if len(s[s > -1]) else -1.0


def _coco_summarize(precision, recall, max_dets):
    """COCOeval.summarize on the host arrays: the 12 stats and the per-category AP (IoU .50:.95, area all, maxDets[2])."""
    stats = []
    for ap, thr, area, m in COCO_STAT_ROWS:
        aind = [i for i, lbl in enumerate(engine.COCO_AREA_LBL) if lbl == area]
        s = precision if ap else recall
        if thr is not None:
            s = s[np.where(thr == engine.COCO_IOU_THRS)[0]]
        s = s[:, :, :, aind, [m]] if ap else s[:, :, aind, [m]]
        stats.append(_coco_mean(s))
    return stats, [_coco_mean(precision[:, :, k, 0, 2]) for k in range(precision.shape[2])]


def _coco_number(v):
    return isinstance(v, (int, float)) and not isinstance(v, bool) and not (isinstance(v, float) and v != v)


def evaluate_coco(gt_path, dt_path, output_dir=None, *, max_dets=(1, 10, 100), match_categories="id"):
    """COCO `segm` evaluation of the detections file dt_path (coco_instances.json of run_inference, or any COCO instance JSON with
    compressed-RLE masks and scores) against the ground truth gt_path: pycocotools' COCOeval (iouType "segm") with maxDets
    max_dets, on the device.  Returns {"stats": the 12 numbers of COCOeval.summarize, "per_category": {name: AP}, "precision"
    [10, 101, K, 4, 3], "recall" [10, K, 4, 3]} (numpy float64, -1 where COCOeval leaves -1); with output_dir also writes
    coco_eval_results.csv.  The default max_dets are pycocotools' and keep only the 100 best detections of an image: a dense
    micrograph needs larger values, e.g. (100, 1000, 30000).  The frame sizes come from the GT file's images; no pixel data is read.

    Images are matched by file_name; categories are the GT file's, and match_categories="name" maps a DT category_id to the GT
    category of the same name (run_inference writes 0-based thing_classes ids, annotation tools usually start at 1).  Raises
    ValueError, naming the file and the annotation or image, for max_dets that are not three strictly increasing positive ints, a
    detection without a numeric score, a DT image whose file_name has no GT image, a GT category name given twice under "name",
    and the load_coco_results errors."""
    md = tuple(int(m) for m in engine.check_max_dets(max_dets))
    if match_categories not in ("id", "name"):
        raise ValueError(f"evaluate_coco: match_categories must be 'id' or 'name', not {match_categories!r}")
    with open(gt_path, "rb") as f:
        gt = json.loads(f.read())
    with open(dt_path, "rb") as f:
        dt = json.loads(f.read())
    gimgs = sorted(gt.get("images", []), key=lambda e: e.get("id"))
    names = [e.get("file_name") for e in gimgs]
    seen = set()
    for e in gimgs:
        if e.get("file_name") in seen:
            raise ValueError(f"{gt_path}: image {e.get('id')!r}: file_name {e.get('file_name')!r} appears twice")
        seen.add(e.get("file_name"))
    sizes = [(int(e["height"]), int(e["width"])) for e in gimgs]
    cat_ids = sorted(c["id"] for c in gt.get("categories", []))
    kidx = {c: k for k, c in enumerate(cat_ids)}
    if match_categories == "name":
        by_name = {}
        for c in gt.get("categories", []):
            if c.get("name") in by_name:
                raise ValueError(f"{gt_path}: category {c.get('id')!r}: name {c.get('name')!r} is given twice")
            by_name[c.get("name")] = c["id"]
        dmap = {c.get("id"): kidx[by_name[c.get("name")]] for c in dt.get("categories", []) if c.get("name") in by_name}
    else:
        dmap = kidx
    dt_anns = dt.get("annotations", [])
    for ann in dt_anns:
        if not _coco_number(ann.get("score")):
            raise _coco_error(dt_path, ann, f"score {ann.get('score')!r} is not a number")
    for e in dt.get("images", []):
        if e.get("file_name") not in seen:
            raise ValueError(f"{dt_path}: image {e.get('id')!r}: file_name {e.get('file_name')!r} has no GT image")
    bbox_area = bool(dt_anns) and bool(dt_anns[0].get("bbox"))      # loadRes' bbox branch: area = w * h of each bbox
    _, gper, ggroups = _decode_coco(gt_path, names, sizes, d=gt)
    _, dper, dgroups = _decode_coco(dt_path, names, sizes, d=dt)
    gt_sets, dt_sets = [], []
    for (_, ks, gi), (_, _, di) in zip(ggroups, dgroups):
        g_items = [(k, it) for k in ks for it in gper[k]]
        d_items = [(k, it) for k in ks for it in dper[k]]
        g_pop = gi.area.cpu().numpy() if g_items else np.zeros(0)
        d_pop = di.area.cpu().numpy() if d_items else np.zeros(0)
        gt_sets.append({"iset": gi, "image": np.array([k for k, _ in g_items], np.int64),
                        "category": np.array([kidx.get(it[1], -1) for _, it in g_items], np.int64),
                        "area": np.array([float(it[3]["area"]) if "area" in it[3] else float(g_pop[j])
                                          for j, (_, it) in enumerate(g_items)], np.float64),
                        "iscrowd": np.array([bool(it[3].get("iscrowd", 0)) for _, it in g_items], bool),
                        "id": np.array([int(it[3].get("id", -1)) for _, it in g_items], np.int64)})
        dt_sets.append({"iset": di, "image": np.array([k for k, _ in d_items], np.int64),
                        "category": np.array([dmap.get(it[1], -1) for _, it in d_items], np.int64),
                        "score": np.array([float(it[2]) for _, it in d_items], np.float64),
                        "area": np.array([float(it[3]["bbox"][2] * it[3]["bbox"][3]) if bbox_area else float(d_pop[j])
                                          for j, (_, it) in enumerate(d_items)], np.float64)})
    precision, recall = engine.coco_evaluate(gt_sets, dt_sets, len(names), len(cat_ids), md)
    precision, recall = precision.cpu().numpy(), recall.cpu().numpy()
    stats, per_cat = _coco_summarize(precision, recall, md)
    cnames = {c["id"]: c.get("name") for c in gt.get("categories", [])}
    cat_names = [cnames[c] for c in cat_ids]
    if output_dir is not None:
        os.makedirs(output_dir, exist_ok=True)
        with open(os.path.join(output_dir, "coco_eval_results.csv"), "w", newline="", encoding="utf-8") as f:
            w = csv.writer(f)
            w.writerow(COCO_EVAL_HEADER)
            iou = lambda t: "0.50:0.95" if t is None else f"{t:.2f}"      # noqa: E731
            for (ap, t, area, m), v in zip(COCO_STAT_ROWS, stats):
                w.writerow(["AP" if ap else "AR", "all", iou(t), area, md[m], repr(float(v))])
            for name, v in zip(cat_names, per_cat):
                w.writerow(["AP", name, iou(None), "all", md[2], repr(float(v))])
    return {"stats": stats, "per_category": dict(zip(cat_names, per_cat)), "precision": precision, "recall": recall}
