"""Batched, device-resident forms of the reference's inference flows.

The reference (src/functions/inference.py) walks its flows one predictor call at a time, in Python, and converts every mask to
a full-frame numpy array between the steps.  Here the head outputs of ALL predictor calls of a batch — every tile of a
micrograph plus the full-image pass, every image, every scale, every model — sit in flat device arrays (`HeadBatch`), each
step of a flow is ONE launch (per frame size) over all of them, lists are (length, index) arrays that never leave the device,
and nothing is read back until the flow is finished (`engine.Arena`: capacities + device-side guards).

    class_specific(...)        run_class_specific_inference  :1353-1461  for every unit and every target class
    tile_pipeline(...)         tile_based_inference_pipeline :2299-2485  + the per-image tail of run_inference :859-868
                               (cross-class deduplicate_masks_smart at 0.7, apply_spatial_constraints) + morphometry :1148-1253
    ensemble_multiscale(...)   run_ensemble_inference :1464-1598 merged with the multi-scale pass :1833-1984 (BASELINE config 4)

A `HeadBatch` holds what Detectron2's GeneralizedRCNN.inference(do_postprocess=False) yields for U calls on frames of one size.
"""
from dataclasses import dataclass, field
from typing import Optional

import numpy as np
import torch

from . import engine

PARALLEL_MASK_PROCESSING = True       # l4_performance_optimizations.enable_parallel_mask_processing (inference.py:1443)


@dataclass
class HeadBatch:
    probs: torch.Tensor        # [n, 28, 28] float32 / float16
    boxes: torch.Tensor        # [n, 4] float32 xyxy, model-input coordinates
    scores: torch.Tensor       # [n] float32
    classes: torch.Tensor      # [n] int32
    unit_off: np.ndarray       # host int64 [U + 1]: unit u owns instances [unit_off[u], unit_off[u + 1])
    H: int                     # frame the predictor saw (the image / upscaled tile / rescaled image handed to it)
    W: int
    scale_x: float = 1.0       # output / model-input size (detector_postprocess)
    scale_y: float = 1.0

    @property
    def n(self):
        return int(self.unit_off[-1])

    @property
    def U(self):
        return len(self.unit_off) - 1


@dataclass
class ClassParams:
    """What run_inference derives per target class (src/functions/inference.py:790-826)."""
    target_class: int
    is_small: bool
    confidence_threshold: float
    iou_threshold: float = 0.7
    min_size: Optional[float] = None      # postprocess_masks' min_crys_size (default 5 small / 25 large, :1431)

    @property
    def gate_size(self):
        return self.min_size if self.min_size is not None else (5 if self.is_small else 25)

    @property
    def inorder_iou(self):
        return 0.5 if self.is_small else self.iou_threshold          # :1453


class _Layouts:
    """Host-side tables of a batch shape (unit sizes), cached: nothing in here depends on device data."""

    def __init__(self):
        self.cache = {}

    def get(self, key, make):
        v = self.cache.get(key)
        if v is None:
            if len(self.cache) > 64:
                self.cache.clear()
            v = make()
            self.cache[key] = v
        return v


_layouts = _Layouts()


def paste_units(hb, arena, tag):
    """K1 over every unit of the batch (crops only), sync-free."""
    n = hb.n
    meta, crop_off = engine.paste_plan(hb.boxes, hb.H, hb.W, hb.scale_x, hb.scale_y)
    cap = engine.buffer_len(crop_off[n:], n, arena, tag + ".crops", n * 1024 + 65536, meta)
    crops = torch.empty(cap, dtype=torch.int32, device=hb.boxes.device)
    return engine.paste(hb.probs, hb.boxes, hb.H, hb.W, scores=hb.scores, classes=hb.classes, scale_x=hb.scale_x, scale_y=hb.scale_y,
                        plan=(meta, crop_off, cap), crops_out=crops, abort=arena.abort)


def _class_space(hb, n_classes, device):
    """GroupSpace with one section per target class; every section has one list per unit with the unit's size as capacity,
    initialised to the identity lists (every head of the unit)."""
    sizes = np.diff(hb.unit_off).astype(np.int64)
    key = ("class_space", sizes.tobytes(), n_classes, str(device))

    def make():
        sp = engine.GroupSpace([sizes] * n_classes, device)
        ident = torch.arange(hb.n, dtype=torch.int32, device=device).repeat(n_classes)
        lens = torch.as_tensor(np.tile(sizes, n_classes).astype(np.int32), device=device)
        return sp, ident, lens

    sp, ident, lens = _layouts.get(key, make)
    cur = sp.fresh()
    if hb.n:
        cur.idx[:ident.numel()].copy_(ident)
    if lens.numel():
        cur.length[:lens.numel()].copy_(lens)
    return cur


def _whole(space):
    """All groups of a space as one Groups object."""
    return engine.Groups(cap_off_host=space.cap_abs, cap_off=space.cap_off, length=space.length, idx=space.idx)


def class_specific(hb, params, arena, tag="cs", iset=None, out_space=None):
    """run_class_specific_inference (single predictor, src/functions/inference.py:1353-1461) for every unit of `hb` and every
    target class of `params`, all at once.  Returns (post-processed InstanceSet, GroupSpace whose section c holds the kept
    lists of params[c]: one list per unit, in the reference's order).  Instances keep their head scores / classes."""
    dev = hb.boxes.device
    C = len(params)
    if iset is None:
        iset = paste_units(hb, arena, tag)
    s0 = _class_space(hb, C, dev)
    s1 = s0.fresh()
    for c, p in enumerate(params):
        # class + confidence filter (:1411-1420) and postprocess_masks' zero-score early exit (mask_utils.py:59)
        engine.filter_heads(iset, s0.section(c), p.target_class, p.confidence_threshold, zero_score_empties=True, out=s1.section(c))
    # postprocess_masks (mask_utils.py:38-84): column gate per class (min_crys_size differs), then closing / first-come
    # overlap removal over the lists of all classes in one launch each
    s2 = s1.fresh()
    for c, p in enumerate(params):
        g = engine.column_gate(iset, s1.section(c), p.gate_size)
        s2.section(c).length.copy_(g.length)
        s2.section(c).idx.copy_(g.idx)
    gated = _whole(s2)
    members = engine.mark_members(iset, gated, -1)
    closed = engine.morph(iset, [engine.MORPH_FILL, engine.MORPH_DILATE, engine.MORPH_ERODE], apply=members, arena=arena, tag=tag + ".close")
    post = engine.overlap_first_come(closed, gated, arena=arena, tag=tag + ".ofc")
    if PARALLEL_MASK_PROCESSING:
        # process_masks_parallel only runs on lists of more than two masks (:1443)
        big = engine.mark_members(post, gated, 2)
        post = engine.process_masks_parallel(post, apply=big, arena=arena, tag=tag)
    s3 = out_space if out_space is not None else s2.fresh()
    for c, p in enumerate(params):
        engine.dedup_inorder(post, s2.section(c), p.inorder_iou, out=s3.section(c))
    return post, s3


@dataclass
class FlowResult:
    iset: engine.InstanceSet            # the combined destination set (original-image frame)
    per_class: Optional[engine.Groups]  # lists after the per-class stage (one per class and image)
    kept: engine.Groups                 # final lists, one per image
    meas: Optional[engine.Measurements]
    extra: dict = field(default_factory=dict)


def _tile_layout(full_hb, tile_hb, B, T, C, dev):
    """Group-list tables of the tile pipeline: for class c and image b, `full_image_masks + all_tile_masks` (:2452)."""
    fs, ts = np.diff(full_hb.unit_off).astype(np.int64), np.diff(tile_hb.unit_off).astype(np.int64)
    key = ("tile_layout", fs.tobytes(), ts.tobytes(), B, T, C, str(dev))

    def make():
        # final space: sections [full c0 .. full c(C-1), tile c0 .. tile c(C-1)]
        sp = engine.GroupSpace([fs] * C + [ts] * C, dev)
        lists, add = [], np.zeros(len(sp.cap_abs) - 1, np.int32)
        for c in range(C):
            for b in range(B):
                lists.append([sp.group_index(c, b)] + [sp.group_index(C + c, b * T + t) for t in range(T)])
            a0, a1 = sp.group_index(C + c, 0), sp.group_index(C + c, B * T - 1) + 1
            add[a0:a1] = full_hb.n                       # tile instances follow the full-image instances in the combined set
        cross = [[c * B + b for c in range(C)] for b in range(B)]
        return sp, lists, add, cross, {}

    return _layouts.get(key, make)


def tile_pipeline(full_hb, tile_hb, tile_xy, image_hw, tile_size, overlap_ratio, params, arena, edge_filter_enabled=True,
                  cross_class_iou=0.7, rules=None, um_pix=1.0, measure=True, min_area=None):
    """The per-image body of run_inference for B images of one size (src/functions/inference.py:776-905), batched:

      per class (tile_based_inference_pipeline :2299-2485): run_class_specific_inference on the full image and on every
      upscaled tile -> NEAREST back-projection (:2399-2403) -> edge filter (:2405-2407) -> placement (:2410-2416) ->
      `full + tiles` -> deduplicate_masks_smart(0.4) (:2472, Q8)
      then: all classes -> deduplicate_masks_smart(0.7) (:859) -> apply_spatial_constraints (:868) -> measurement loop (:1148-1253).

    full_hb: one unit per image (frame h x w).  tile_hb: B * T units, image-major, frame (tile_size * upscale)^2.
    tile_xy: host int array [T, 2] of (x_offset, y_offset) (generate_tiles_with_overlap order).  params: list of ClassParams.
    Everything is enqueued without a host synchronisation; the caller finishes with arena.finish()."""
    dev = full_hb.boxes.device
    h, w = image_hw
    B, T, C = full_hb.U, len(tile_xy), len(params)
    assert tile_hb.U == B * T
    sp_proto, lists, id_add, cross, tabs = _tile_layout(full_hb, tile_hb, B, T, C, dev)
    final = sp_proto.fresh()
    # ---- full-image pass and tile pass: K1 -> class filter -> K2 -> in-order de-dup, each over all its units and classes
    post_f, kept_f = class_specific(full_hb, params, arena, tag="full")
    post_t, kept_t = class_specific(tile_hb, params, arena, tag="tile")
    # ---- K3: everything into the image frame, one combined instance set [full | tiles]
    comb = engine.Combined([post_f.n, post_t.n], h, w, dev)
    key = ("tile_xy", np.asarray(tile_xy, np.int32).tobytes(), np.asarray(tile_hb.unit_off).tobytes(), B, str(dev))

    def make_xy():
        xy = np.tile(np.asarray(tile_xy, np.int32).reshape(T, 2), (B, 1))
        return (torch.as_tensor(np.ascontiguousarray(xy), device=dev),
                torch.as_tensor(np.asarray(tile_hb.unit_off, np.int32), device=dev))

    xy_t, uoff_t = _layouts.get(key, make_xy)
    off_xy = engine.unit_broadcast(uoff_t, tile_hb.U, tile_hb.n, xy_t, 2)
    # only instances that are still in a list are back-projected (and later traced)
    comb.plan(0, post_f, h, w, alive=engine.mark_members(post_f, _whole(kept_f), -1))
    comb.plan(1, post_t, tile_size, tile_size, off_xy, alive=engine.mark_members(post_t, _whole(kept_t), -1))
    iset = comb.place(arena, tag="k3", edge={1: (tile_size, overlap_ratio)} if edge_filter_enabled else None)
    # ---- lists into the final space: full lists as they are, tile lists through the edge filter
    for c in range(C):
        final.section(c).length.copy_(kept_f.section(c).length)
        final.section(c).idx.copy_(kept_f.section(c).idx)
    kt = _whole(kept_t)
    tile_out = engine.Groups(cap_off_host=kt.cap_off_host, cap_off=kt.cap_off,
                             length=final.length[int(final.g0[C]):], idx=final.idx[int(final.cap_abs[int(final.g0[C])]):])
    if edge_filter_enabled:
        engine.filter_flag(kt, comb.edge[int(comb.start[1]):], 0, out=tile_out)
    else:
        tile_out.length[:kt.length.numel()].copy_(kt.length)
        tile_out.idx[:kt.idx.numel()].copy_(kt.idx)
    per_class_in = engine.flatten(final, lists, id_add, cache=tabs.setdefault("f1", {}))
    # ---- per class and image: deduplicate_masks_smart at 0.4 (needs the contour perimeters of the compactness pre-filter)
    engine.trace(iset, arena=arena)
    sp2 = _space_like(tabs, "sp2", per_class_in, dev)
    engine.dedup_smart(iset, per_class_in, 0.4, out=sp2.section(0))
    # ---- all classes of an image: deduplicate_masks_smart at 0.7, spatial constraints, morphometry
    allc = engine.flatten(sp2, cross, cache=tabs.setdefault("f2", {}))
    kept = engine.dedup_smart(iset, allc, cross_class_iou)
    kept = engine.apply_spatial_constraints(iset, kept, rules)
    meas = engine.measure_list(iset, kept, um_pix=um_pix, min_area=min_area, arena=arena) if measure else None
    return FlowResult(iset=iset, per_class=sp2.section(0), kept=kept, meas=meas, extra={"combined": comb})


def _space_like(tabs, name, groups, dev):
    """A one-section GroupSpace with the capacities of `groups` (cached layout, fresh arrays)."""
    proto = tabs.get(name)
    if proto is None:
        proto = engine.GroupSpace([np.diff(groups.cap_off_host).astype(np.int64)], dev)
        tabs[name] = proto
    return proto.fresh()


def ensemble_multiscale(heads, weights, image_hw, params, arena, sorted_iou=0.4, rules=None, um_pix=1.0, measure=True,
                        min_area=None):
    """BASELINE config 4 (SURVEY.md section 8d): R50 + R101 ensemble merged with multi-scale inference on a batch of B images.

    heads[s][m]: HeadBatch of model m on every image rescaled by scale s (one unit per image; frame int(h * s) x int(w * s)).
    Per (scale, model): class + confidence filter (:1519-1523) -> postprocess_masks_universal with the scaled minimum size
    (:1739-1813, :2026-2031) -> NEAREST back-projection to h x w (:2044-2054) -> score * weight (:1553);
    per image and class: score-sorted greedy iou() de-dup at 0.4 across scales and models (:1964-1978) ->
    deduplicate_masks_smart at the class IoU threshold (:1590); then all classes: deduplicate_masks_smart(0.7) (:859) ->
    spatial constraints (:868) -> morphometry.  heads: {scale: [HeadBatch per model]}."""
    scales = list(heads.keys())
    M = len(weights)
    dev = heads[scales[0]][0].boxes.device
    h, w = image_hw
    B, C = heads[scales[0]][0].U, len(params)
    parts = [(s, m) for s in scales for m in range(M)]
    sizes = [np.diff(heads[s][m].unit_off).astype(np.int64) for s, m in parts]
    key = ("ems", tuple(z.tobytes() for z in sizes), B, C, str(dev))

    def make():
        # final space: sections [(part 0, class 0), (part 0, class 1), ..., (part P-1, class C-1)], B groups each
        sp = engine.GroupSpace([z for z in sizes for _ in range(C)], dev)
        starts = np.concatenate([[0], np.cumsum([int(z.sum()) for z in sizes])])
        lists, add = [], np.zeros(len(sp.cap_abs) - 1, np.int32)
        for c in range(C):
            for b in range(B):
                lists.append([sp.group_index(pi * C + c, b) for pi in range(len(parts))])
        for pi in range(len(parts)):
            for c in range(C):
                a0 = sp.group_index(pi * C + c, 0)
                add[a0:a0 + B] = starts[pi]
        cross = [[c * B + b for c in range(C)] for b in range(B)]
        return sp, lists, add, cross, {}

    sp_proto, lists, id_add, cross, tabs = _layouts.get(key, make)
    final = sp_proto.fresh()
    comb = engine.Combined([int(z.sum()) for z in sizes], h, w, dev)
    area0 = h * w
    posts = []
    for pi, (s, m) in enumerate(parts):
        hb = heads[s][m]
        iset = paste_units(hb, arena, f"ems{pi}")
        s0 = _class_space(hb, C, dev)
        s1 = s0.fresh()
        for c, p in enumerate(params):
            engine.filter_heads(iset, s0.section(c), p.target_class, p.confidence_threshold, out=s1.section(c))
        # postprocess_masks_universal: the operator chain depends on the class (erosion only for small classes), the minimum
        # size on class and scale (process_single_scale :2026-2031: int(base * scale^2) of the ORIGINAL image area)
        # one launch for both kinds of class: selector 1 = opening (large classes), 2 = erosion only (small classes)
        sel = None
        for c, p in enumerate(params):
            sel = engine.mark_members(iset, s1.section(c), -1, value=2 if p.is_small else 1, into=sel)
        post = engine.morph(iset, [engine.MORPH_FILL, engine.MORPH_ERODE, engine.MORPH_DILATE], apply=sel, arena=arena, tag=f"ems{pi}.univ",
                            ops_b=[engine.MORPH_FILL, engine.MORPH_ERODE])
        for c, p in enumerate(params):
            base_min = max(3, int(area0 * 0.000005)) if p.is_small else max(25, int(area0 * 0.0001))
            engine.filter_area(post, s1.section(c), int(base_min * (s ** 2)), out=final.section(pi * C + c))
        post.scores = engine.scale_scores(iset.scores, weights[m])
        posts.append(post)
        alive = engine.mark_members(post, final.range(pi * C, (pi + 1) * C), -1)      # survivors of the size filter, any class
        comb.plan(pi, post, h, w, alive=alive)
    iset = comb.place(arena, tag="k3")
    per_class_in = engine.flatten(final, lists, id_add, cache=tabs.setdefault("f1", {}))
    sp2 = _space_like(tabs, "sp2", per_class_in, dev)
    s_sorted = engine.dedup_sorted(iset, per_class_in, sorted_iou)
    engine.trace(iset, arena=arena)
    # one deduplicate_masks_smart call per class threshold (lists of the other classes pass through empty)
    thr = sorted(set(p.iou_threshold for p in params))
    if len(thr) == 1:
        engine.dedup_smart(iset, s_sorted, thr[0], out=sp2.section(0))
    else:
        for c, p in enumerate(params):
            sub = engine.Groups(cap_off_host=(per_class_in.cap_off_host[c * B:(c + 1) * B + 1] - per_class_in.cap_off_host[c * B]).astype(np.int32),
                                cap_off=None, length=s_sorted.length[c * B:(c + 1) * B], idx=s_sorted.idx[int(per_class_in.cap_off_host[c * B]):])
            sub.cap_off = torch.as_tensor(sub.cap_off_host, device=dev)
            o = engine.Groups(cap_off_host=sub.cap_off_host, cap_off=sub.cap_off, length=sp2.length[c * B:(c + 1) * B],
                              idx=sp2.idx[int(per_class_in.cap_off_host[c * B]):])
            engine.dedup_smart(iset, sub, p.iou_threshold, out=o)
    allc = engine.flatten(sp2, cross, cache=tabs.setdefault("f2", {}))
    kept = engine.dedup_smart(iset, allc, 0.7)
    kept = engine.apply_spatial_constraints(iset, kept, rules)
    meas = engine.measure_list(iset, kept, um_pix=um_pix, min_area=min_area, arena=arena) if measure else None
    return FlowResult(iset=iset, per_class=sp2.section(0), kept=kept, meas=meas, extra={"combined": comb, "posts": posts})


# =================================================================================================================
# static layouts + CUDA graphs: a flow over units padded to a fixed capacity is a FIXED sequence of launches — captured once,
# replayed per batch (no Python, no launch gaps).  Padding heads carry a degenerate box: detector_postprocess' Boxes.nonempty()
# drops them (meta.valid = 0), so they never enter a list.
# =================================================================================================================
def pad_units(probs, boxes, scores, classes, unit_off, cap):
    """Host arrays of U units -> arrays of U * cap heads (unit u at [u * cap, u * cap + n_u), the rest padding)."""
    unit_off = np.asarray(unit_off, np.int64)
    U = len(unit_off) - 1
    sizes = np.diff(unit_off)
    assert sizes.max(initial=0) <= cap
    dst = (np.repeat(np.arange(U, dtype=np.int64) * cap, sizes) + (np.arange(unit_off[-1]) - np.repeat(unit_off[:-1], sizes)))
    P = np.zeros((U * cap,) + probs.shape[1:], probs.dtype); P[dst] = probs
    Bx = np.zeros((U * cap, 4), np.float32); Bx[dst] = boxes
    S = np.zeros(U * cap, np.float32); S[dst] = scores
    C = np.full(U * cap, -1, np.int32); C[dst] = classes
    return P, Bx, S, C, (np.arange(U + 1, dtype=np.int64) * cap), dst


class GraphedFlow:
    """fn(arena) -> FlowResult over STATIC input tensors, captured into a CUDA graph after the eager runs have filled the
    layout caches and settled the arena's capacities.  replay() enqueues the whole flow as one graph launch; finish() checks
    the captured run (abort flag and totals, rewritten by every replay) exactly as after an eager run."""

    def __init__(self, fn, arena, pool=None):
        self.fn, self.arena, self.pool = fn, arena, pool
        self.graph = None
        self.res = None
        self._run = None
        self.launches = 0

    def settle(self, max_runs=12):
        """Eager runs until no capacity guard trips (reads the totals back: set-up, not steady state)."""
        for _ in range(max_runs):
            self.arena.begin()
            self.res = self.fn(self.arena)
            if self.arena.finish():
                return self.res
        raise engine._lib.EmiaError("the arena did not converge")

    def capture(self):
        torch.cuda.synchronize()
        l0 = engine.LAUNCHES["count"]
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, pool=self.pool):
            self._run = self.arena.begin()
            self.res = self.fn(self.arena)
        self.graph = g
        self.launches = engine.LAUNCHES["count"] - l0
        return self

    @property
    def abort(self):
        """Abort flag of the captured run (device int32, rewritten by every replay)."""
        return self._run[0]

    def replay(self):
        self.graph.replay()
        return self.res

    def finish(self):
        return self.arena.finish(self._run)
