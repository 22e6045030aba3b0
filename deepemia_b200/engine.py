"""Device-resident engine over libemia.so: instances stay bit-packed in HBM from the mask head to the CSV row.

Every computation on the path is a kernel of libemia.so called through the C ABI (include/emia.h) with raw tensor pointers.
PyTorch provides device memory (torch.empty / zeros), streams, events and CUDA graphs, memcpy-type plumbing (copy_, clone, cat of
already-computed arrays, the identity index lists of a layout) and — in bench.py / distributed.py — torch.distributed.
"""
import csv
import io
import math
from dataclasses import dataclass, field
from typing import Optional

import numpy as np
import torch

from . import _lib

MASK_SIDE = 28
REC_FIELDS = 16
(REC_MAJOR, REC_MINOR, REC_ECC, REC_LENGTH, REC_WIDTH, REC_CED, REC_ASPECT, REC_CIRC, REC_CHORDS, REC_FERET, REC_ROUND,
 REC_SPHER, REC_AREA, REC_PERIM, REC_NVERT, REC_MEASURED) = range(16)

FUSED_K4 = True
MEASURE_ORDER = bool(int(__import__("os").environ.get("EMIA_MEASURE_ORDER", "1")))   # length-sorted work order of K5b/c (0: list order)
MEASURE_ORDER_MIN_SLOTS = 65536
LAUNCHES = {"count": 0}   # kernels launched through the ABI (bench.py reports it as gpu_launches)
STAGE_TIMING = {"enabled": False, "events": []}   # (name, start, end) CUDA events when enabled (bench.py --breakdown)


NVTX = {"enabled": bool(int(__import__("os").environ.get("EMIA_NVTX", "0")))}   # EMIA_NVTX=1: one NVTX range per stage (nsys / ncu --nvtx)


class _stage:
    """A named stage of the path: an NVTX range when EMIA_NVTX=1, CUDA events when STAGE_TIMING is enabled (bench.py --breakdown)."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if NVTX["enabled"]:
            torch.cuda.nvtx.range_push("emia:" + self.name)
        if STAGE_TIMING["enabled"]:
            self.a = torch.cuda.Event(enable_timing=True); self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if STAGE_TIMING["enabled"]:
            self.b.record()
            STAGE_TIMING["events"].append((self.name, self.a, self.b))
        if NVTX["enabled"]:
            torch.cuda.nvtx.range_pop()
        return False


def stage_summary():
    torch.cuda.synchronize()
    out = {}
    for name, a, b in STAGE_TIMING["events"]:
        out.setdefault(name, []).append(a.elapsed_time(b))
    STAGE_TIMING["events"].clear()
    return {k: float(np.mean(v)) for k, v in out.items()}


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(dev):
    if not torch.cuda.is_available():
        raise _lib.EmiaError("deepemia_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device(dev if dev is not None else "cuda")


def pitch_words_for(W):
    """256-bit aligned bit rows (the paste kernel writes frames with 256-bit stores): pitch = 32 * ceil(W / 256) bytes.
    The ABI accepts any pitch that is a multiple of 4 words; pitches that are not multiples of 8 fall back to 128-bit stores."""
    return 8 * ((W + 255) // 256)


def exclusive_scan_(t):
    """In-place exclusive scan of t[0:n] with the total in t[n] (int64, n+1 entries)."""
    lib = _lib.load()
    n = t.numel() - 1
    nb = int(lib.emia_scan_workspace_bytes(n))
    ws = torch.empty(nb, dtype=torch.uint8, device=t.device)
    _lib.check(lib.emia_exclusive_scan_i64(_ptr(t), n, _ptr(ws), nb, _stream()), "emia_exclusive_scan_i64")
    LAUNCHES["count"] += 3
    return t


class Arena:
    """Capacities of the variable-size device buffers of a flow (crop words, contour vertices, records, ...): the one place
    that decides how such a buffer is sized when its size is known only after a device-side scan (see buffer_len()).

    A run is enqueued WITHOUT reading any size back: begin() makes a fresh abort flag, every variable-size output goes into a
    buffer of the arena's current capacity, and a device-side guard (emia_capacity_guard) compares the real total with it.
    On overflow the guard raises the abort flag and empties the geometry of the affected instance set, so that no later
    kernel touches memory outside the buffers.  finish() is the one host synchronisation of a run: it reads the flag and the
    recorded totals, grows the capacities that were too small (fit()) and tells the caller to run again.

    Capacities only grow, to total * margin + 64, so that shards of similar size keep running sync-free whatever their exact
    instance counts are.  The batched flows use margin 1.25.  TilePipeline uses its hint_margin, 1.05: it fits its capacities
    to the totals of an exact-size run, and an overflow there makes the next run exact again."""

    def __init__(self, device, margin=1.25):
        self.dev = torch.device(device)
        self.margin = margin
        self.caps = {}
        self.abort = None
        self._totals = []
        self.runs = 0
        self.aborts = 0

    def begin(self):
        """Start a run: a fresh abort flag and no recorded totals.  Returns the run (abort flag, recorded totals), which
        finish(run) can check after later runs have begun (a run captured in a CUDA graph and replayed)."""
        self.abort = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self._totals = []
        self.runs += 1
        return self.abort, self._totals

    def cap(self, name, default):
        c = self.caps.get(name)
        if c is None or c < 1:
            c = max(int(default), 1)
            self.caps[name] = c
        return c

    def fit(self, name, total):
        """Raise the capacity of `name` to total * margin + 64 when that is larger."""
        self.caps[name] = max(self.caps.get(name, 0), int(total * self.margin) + 64)

    def guard(self, name, total, poison_meta=None, poison_n=0):
        """total: int64 device tensor view of ONE element (e.g. crop_off[n:]).  Enqueues the device-side check."""
        lib = _lib.load()
        cap = self.caps[name]
        _lib.check(lib.emia_capacity_guard(_ptr(total), cap, _ptr(self.abort), _ptr(poison_meta), int(poison_n), _stream()),
                   "emia_capacity_guard")
        LAUNCHES["count"] += 1
        self._totals.append((name, total))

    def finish(self, run=None):
        """One host synchronisation: True when the run (default: the last one begun) is valid; False when a guard tripped
        (capacities grown: run again)."""
        abort, totals = run if run is not None else (self.abort, self._totals)
        vals = torch.cat([abort.to(torch.int64)] + [t.reshape(-1)[:1] for _, t in totals]).tolist()
        if not vals[0]:
            return True
        self.aborts += 1
        grown = False
        for (name, _), v in zip(totals, vals[1:]):
            if v > self.caps[name]:
                self.fit(name, v)
                grown = True
        if not grown:       # the flag came from a kernel-side overflow (contour slab): give everything more room
            for k in self.caps:
                self.caps[k] = int(self.caps[k] * 2)
        return False


def buffer_len(total, n, arena=None, name=None, default=0, poison_meta=None):
    """Elements to allocate for a variable-length buffer of n instances whose size is the device scalar `total` (an int64 view
    of one element, e.g. crop_off[n:], after the scan).  Without an arena: the total read back (one host synchronisation; 0,
    without one, when n == 0).  With an arena: its capacity for `name` (`default` on first use), checked on the device by a
    guard that, on overflow, also empties the geometry poison_meta [n, 8] of the instances."""
    if arena is None:
        return int(total.item()) if n else 0
    c = arena.cap(name, default)
    arena.guard(name, total, poison_meta, n if poison_meta is not None else 0)
    return c


@dataclass
class InstanceSet:
    """n bit-packed instances of one frame size (see "Instance layout" in include/emia.h)."""
    n: int
    H: int
    W: int
    meta: torch.Tensor            # int32 [n, 8]
    crop_off: torch.Tensor        # int64 [n+1]
    crops: torch.Tensor           # int32 words
    bbox: torch.Tensor            # int32 [n, 4]  (y_min, x_min, y_max, x_max) or -1
    area: torch.Tensor            # int32 [n]
    scores: Optional[torch.Tensor] = None   # float32 [n]
    classes: Optional[torch.Tensor] = None  # int32 [n]
    frames: Optional[torch.Tensor] = None   # int32 [slots, H, pitch_words]
    total_crop_words: int = 0
    # contours / morphometry (filled by measure())
    cont_off: Optional[torch.Tensor] = None
    pt_off: Optional[torch.Tensor] = None
    pts: Optional[torch.Tensor] = None
    cstart: Optional[torch.Tensor] = None
    records: Optional[torch.Tensor] = None
    rec_inst: Optional[torch.Tensor] = None
    perim0: Optional[torch.Tensor] = None
    n_records: int = 0
    cstart_stride: int = 0        # 0: packed cstart (cont_off[i] + i); else ints per instance slab
    extra: dict = field(default_factory=dict)

    @property
    def device(self):
        return self.meta.device

    @property
    def valid(self):
        return self.meta[:, 6] != 0


def paste_plan(boxes, H, W, scale_x=1.0, scale_y=1.0):
    """Geometry of K1 for n boxes: meta [n,8] and crop_off [n+1] (exclusive scan of the crop sizes, total in [n]).  No sync."""
    lib = _lib.load()
    n = int(boxes.shape[0])
    assert boxes.dtype == torch.float32 and boxes.is_contiguous()
    meta = torch.empty((n, 8), dtype=torch.int32, device=boxes.device)
    crop_off = torch.empty(n + 1, dtype=torch.int64, device=boxes.device)
    with _stage("paste_plan+scan"):
        _lib.check(lib.emia_paste_plan(_ptr(boxes), n, scale_x, scale_y, H, W, _ptr(meta), _ptr(crop_off), _stream()), "emia_paste_plan")
        exclusive_scan_(crop_off)
    LAUNCHES["count"] += 1
    return meta, crop_off


def paste(probs, boxes, H, W, scores=None, classes=None, scale_x=1.0, scale_y=1.0, frames=None, frame_slots=0,
          variant=2, crops_out=None, plan=None, ctas_per_sm=0, abort=None):
    """K1.  probs [n,28,28] f32 (or f16, as an AMP mask head emits them), boxes [n,4] f32 xyxy (device tensors) -> InstanceSet.
    frames: None (crops only), True (allocate n full frames) or a preallocated int32 [slots, H, pitch_words] ring.
    plan: (meta, crop_off, total_crop_words) from paste_plan() — possibly a slice of a larger plan whose crop offsets index
    the shared `crops_out` buffer; given a plan the call does not synchronise.
    ctas_per_sm: resident CTAs per SM of the paste kernel (0 = default); a smaller grid leaves room for kernels of
    another stream."""
    lib = _lib.load()
    dev = probs.device
    n = int(probs.shape[0])
    assert probs.dtype in (torch.float32, torch.float16) and boxes.dtype == torch.float32 and probs.is_contiguous() and boxes.is_contiguous()
    st = _stream()
    if probs.dtype == torch.float16 and (variant != 2 or ((W + 31) // 32 + 1) * 32 > 2112):
        probs = probs.to(torch.float32)          # only the variant-2 kernel (frames up to 2048 px wide) reads halves directly
    f16 = (1 << 16) if probs.dtype == torch.float16 else 0      # EMIA_PASTE_PROBS_F16: AMP heads, widened exactly in the kernel
    if plan is None:
        meta, crop_off = paste_plan(boxes, H, W, scale_x, scale_y)
        total = buffer_len(crop_off[n:], n)
    else:
        meta, crop_off, total = plan
        assert meta.shape[0] == n and crop_off.numel() == n + 1 and meta.is_contiguous() and crop_off.is_contiguous()
    if crops_out is not None:
        assert crops_out.numel() >= max(total, 1)
        crops = crops_out
    else:
        crops = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
    bbox = torch.empty((n, 4), dtype=torch.int32, device=dev)
    area = torch.empty(n, dtype=torch.int32, device=dev)
    pw = pitch_words_for(W)
    if frames is True:
        frames = torch.empty((max(n, 1), H, pw), dtype=torch.int32, device=dev)
    slots = int(frames.shape[0]) if frames is not None else 1
    if frames is not None:
        assert frames.shape[1] == H and frames.shape[2] == pw and frames.is_contiguous()
    with _stage("k1_paste"):
        _lib.check(lib.emia_paste_threshold_bitpack(_ptr(probs), _ptr(boxes), _ptr(meta), _ptr(crop_off), n, scale_x, scale_y, H, W,
                                                    _ptr(frames), slots, pw, _ptr(crops), _ptr(bbox), _ptr(area),
                                                    int(variant) | (int(ctas_per_sm) << 8) | f16, _ptr(abort), st),
                   "emia_paste_threshold_bitpack")
    LAUNCHES["count"] += 1
    return InstanceSet(n=n, H=H, W=W, meta=meta, crop_off=crop_off, crops=crops, bbox=bbox, area=area, scores=scores,
                       classes=classes, frames=frames, total_crop_words=total)


def from_masks(masks, scores=None, classes=None):
    """Import n byte masks [n,H,W] (uint8/bool device tensor, non-zero = set) as an InstanceSet (bbox crops)."""
    lib = _lib.load()
    dev = masks.device
    if masks.dtype == torch.bool:
        masks = masks.view(torch.uint8)
    assert masks.dtype == torch.uint8 and masks.is_contiguous() and masks.dim() == 3
    n, H, W = (int(s) for s in masks.shape)
    meta = torch.empty((n, 8), dtype=torch.int32, device=dev)
    crop_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    bbox = torch.empty((n, 4), dtype=torch.int32, device=dev)
    area = torch.empty(n, dtype=torch.int32, device=dev)
    st = _stream()
    _lib.check(lib.emia_mask_bbox(_ptr(masks), n, H, W, _ptr(meta), _ptr(crop_off), _ptr(bbox), _ptr(area), st), "emia_mask_bbox")
    exclusive_scan_(crop_off)
    total = buffer_len(crop_off[n:], n)
    crops = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
    _lib.check(lib.emia_mask_pack(_ptr(masks), n, H, W, _ptr(meta), _ptr(crop_off), _ptr(crops), st), "emia_mask_pack")
    LAUNCHES["count"] += 2
    return InstanceSet(n=n, H=H, W=W, meta=meta, crop_off=crop_off, crops=crops, bbox=bbox, area=area, scores=scores,
                       classes=classes, total_crop_words=total)


def unpack_masks(iset, idx=None):
    """Full-frame byte masks [k,H,W] (0/1) of the selected instances (drop-in list-of-arrays surface)."""
    lib = _lib.load()
    dev = iset.device
    if idx is None:
        k = iset.n
        idx_t = None
    else:
        idx_t = torch.as_tensor(idx, dtype=torch.int32, device=dev).contiguous()
        k = int(idx_t.numel())
    out = torch.empty((k, iset.H, iset.W), dtype=torch.uint8, device=dev)
    _lib.check(lib.emia_mask_unpack(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(idx_t), k, iset.H, iset.W,
                                    _ptr(out), _stream()), "emia_mask_unpack")
    LAUNCHES["count"] += 1
    return out


MORPH_FILL, MORPH_ERODE, MORPH_DILATE = 1, 2, 3


def _pad_plan(iset, arena=None, tag="k2"):
    """Global work planes of the K2 kernels: only instances whose padded plane exceeds 1024 words need them (the others use
    shared memory), so the buffer is usually empty.  With an arena nothing is read back (capacity + device-side guard)."""
    cached = iset.extra.get("pad_plan")
    if cached is not None:
        return cached
    lib = _lib.load()
    pad_off = torch.empty(iset.n + 1, dtype=torch.int64, device=iset.device)
    _lib.check(lib.emia_morph_plan(_ptr(iset.meta), iset.n, _ptr(pad_off), _stream()), "emia_morph_plan")
    exclusive_scan_(pad_off)
    LAUNCHES["count"] += 1
    total = buffer_len(pad_off[iset.n:], iset.n, arena, tag + ".work", 1 << 18, iset.meta)
    work = torch.empty(int(lib.emia_morph_scratch_words()) + 3 * total + 1, dtype=torch.int32, device=iset.device)
    iset.extra["pad_plan"] = (pad_off, work)
    return pad_off, work


def _derived(iset, crops, geometry=None, bbox=None, area=None):
    """A new InstanceSet with new crop bits in the geometry (meta, crop_off, total words) of `iset` or the given one; bbox/area
    as computed by the producing kernel, or recomputed here."""
    lib = _lib.load()
    meta, crop_off, total = geometry if geometry is not None else (iset.meta, iset.crop_off, iset.total_crop_words)
    if bbox is None:
        bbox = torch.empty_like(iset.bbox)
        area = torch.empty_like(iset.area)
        _lib.check(lib.emia_crop_stats(_ptr(crops), _ptr(meta), _ptr(crop_off), iset.n, _ptr(bbox), _ptr(area), _stream()),
                   "emia_crop_stats")
        LAUNCHES["count"] += 1
    out = InstanceSet(n=iset.n, H=iset.H, W=iset.W, meta=meta, crop_off=crop_off, crops=crops, bbox=bbox, area=area,
                      scores=iset.scores, classes=iset.classes, total_crop_words=total)
    if geometry is None and "pad_plan" in iset.extra:
        out.extra["pad_plan"] = iset.extra["pad_plan"]
    return out


def morph(iset, ops, apply=None, arena=None, tag="k2", ops_b=None):
    """K2: apply `ops` (MORPH_FILL / MORPH_ERODE / MORPH_DILATE, 3x3 cross, at most 4) to every instance (apply: optional int32
    selector per instance, 0 = pass through unchanged, 1 = `ops`, 2 = `ops_b`).  The result has the geometry of the input, or — a chain that dilates
    first — the crop grown by one pixel.  bbox / area of the result come from the same kernel.  With an arena: no host sync."""
    lib = _lib.load()
    chains = [list(ops)] + ([list(ops_b)] if ops_b is not None else [])
    grows = False
    for ch in chains:
        structuring = [int(o) for o in ch if int(o) != MORPH_FILL]
        grows = grows or (bool(structuring) and structuring[0] == MORPH_DILATE)
    if ops_b is not None:
        ops = list(ops) + [0] * (4 - len(ops)) + list(ops_b)
    ops = np.ascontiguousarray(ops, dtype=np.int32)
    pad_off, work = _pad_plan(iset, arena, tag)
    geometry = None
    meta_out = crop_off_out = None
    if grows and iset.n:
        # closing / dilation: the result may be one pixel larger (always for a dilation; for a closing next to the frame border)
        meta_out = torch.empty_like(iset.meta)
        crop_off_out = torch.empty(iset.n + 1, dtype=torch.int64, device=iset.device)
        _lib.check(lib.emia_morph_grow_plan(_ptr(iset.meta), iset.n, iset.H, iset.W, _ptr(meta_out), _ptr(crop_off_out), _stream()),
                   "emia_morph_grow_plan")
        exclusive_scan_(crop_off_out)
        LAUNCHES["count"] += 1
        total = buffer_len(crop_off_out[iset.n:], iset.n, arena, tag + ".grown", int(iset.total_crop_words * 1.5) + 4 * iset.n + 1024,
                           meta_out)
        geometry = (meta_out, crop_off_out, total)
        crops = torch.empty(max(total, 1), dtype=torch.int32, device=iset.device)
    else:
        crops = torch.empty_like(iset.crops)
    bbox = torch.empty_like(iset.bbox)
    area = torch.empty_like(iset.area)
    if iset.n:
        with _stage("k2_morph"):
            _lib.check(lib.emia_morph(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), iset.n, iset.H, iset.W, ops.ctypes.data,
                                      len(ops), _ptr(pad_off), _ptr(work), _ptr(meta_out), _ptr(crop_off_out), _ptr(crops),
                                      _ptr(apply), _ptr(bbox), _ptr(area), _stream()), "emia_morph")
        LAUNCHES["count"] += 1
    return _derived(iset, crops, geometry, bbox, area)


def overlap_first_come(iset, groups, arena=None, tag="k2"):
    """Tail of postprocess_masks (src/utils/mask_utils.py:77-82): list member k loses the pixels earlier members cover, then is
    zeroed if it has more than one 8-connected component.  Members keep their list position (Q6); instances outside the
    lists are unchanged."""
    lib = _lib.load()
    pad_off, work = _pad_plan(iset, arena, tag)
    crops = iset.crops.clone()
    bbox = iset.bbox.clone()
    area = iset.area.clone()
    if iset.n and groups.total_cap:
        with _stage("k2_overlap_first_come"):
            _lib.check(lib.emia_overlap_first_come(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(iset.bbox),
                                                   _ptr(groups.cap_off), groups.G, groups.total_cap, _ptr(groups.length),
                                                   _ptr(groups.idx), _ptr(pad_off), _ptr(work), _ptr(crops), _ptr(bbox), _ptr(area),
                                                   _stream()),
                       "emia_overlap_first_come")
        LAUNCHES["count"] += 1
    return _derived(iset, crops, None, bbox, area)


def filter_area(iset, groups, min_area, out=None):
    """List members with area >= min_area (`np.sum(final_mask) >= min_crys_size`, src/functions/inference.py:1800).  Areas are
    integers, so a fractional threshold is rounded UP (area >= 5.5 <=> area >= 6)."""
    lib = _lib.load()
    out = out if out is not None else _new_groups_like(groups)
    _lib.check(lib.emia_group_filter_area(_ptr(groups.cap_off), groups.G, _ptr(groups.length), _ptr(groups.idx), _ptr(iset.area),
                                          int(math.ceil(min_area)), _ptr(out.length), _ptr(out.idx), _stream()), "emia_group_filter_area")
    LAUNCHES["count"] += 1
    return out


def column_gate(iset, groups, min_size):
    lib = _lib.load()
    out = _new_groups_like(groups)
    # `column total > min_size` on integers: a fractional threshold is rounded DOWN (total > 5.5 <=> total > 5)
    _lib.check(lib.emia_column_gate(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(groups.cap_off), groups.G,
                                    _ptr(groups.length), _ptr(groups.idx), iset.W, int(math.floor(min_size)), _ptr(out.length), _ptr(out.idx),
                                    _stream()), "emia_column_gate")
    LAUNCHES["count"] += 1
    return out


def filter_heads(iset, groups, target_class, min_score, zero_score_empties=False, out=None):
    """The class / confidence filter of the flows (src/functions/inference.py:1411-1420, :1519-1523, :2146-2151) on every list:
    members that survived Boxes.nonempty(), have class == target_class (None: any) and score >= min_score (float32 compare, as
    numpy does for a float32 array against a Python float).  zero_score_empties: postprocess_masks' `ori_score.all() < 0.5`
    early exit (src/utils/mask_utils.py:59) — a list that still holds a score of exactly 0 becomes empty."""
    lib = _lib.load()
    out = out if out is not None else _new_groups_like(groups)
    _lib.check(lib.emia_group_filter_heads(_ptr(groups.cap_off), groups.G, _ptr(groups.length), _ptr(groups.idx), _ptr(iset.meta),
                                           _ptr(iset.classes), _ptr(iset.scores), -1 if target_class is None else int(target_class),
                                           float(np.float32(min_score)), 1 if zero_score_empties else 0, _ptr(out.length), _ptr(out.idx),
                                           _stream()), "emia_group_filter_heads")
    LAUNCHES["count"] += 1
    return out


def mark_members(iset, groups, min_len, value=1, into=None):
    """int32 [n] flag: `value` for the members of lists longer than min_len (the `len(processed_masks) > 2` gate of
    process_masks_parallel, src/functions/inference.py:1443), 0 elsewhere; `into`: add to an existing flag array."""
    lib = _lib.load()
    flag = into if into is not None else torch.empty(max(iset.n, 1), dtype=torch.int32, device=iset.device)
    _lib.check(lib.emia_group_mark_members(_ptr(groups.cap_off), groups.G, groups.total_cap, _ptr(groups.length), _ptr(groups.idx),
                                           int(min_len), int(value), 1 if into is not None else 0, _ptr(flag), iset.n, _stream()),
               "emia_group_mark_members")
    LAUNCHES["count"] += 2 if into is None else 1
    return flag


def postprocess_masks(iset, groups, min_crys_size=2, arena=None, tag="k2"):
    """postprocess_masks (src/utils/mask_utils.py:38-84) on every group: column gate (Q5) -> fill holes -> closing ->
    first-come overlap removal -> multi-component masks zeroed (kept in the list, Q6).  Returns (InstanceSet, Groups)."""
    gated = column_gate(iset, groups, min_crys_size)
    closed = morph(iset, [MORPH_FILL, MORPH_DILATE, MORPH_ERODE], arena=arena, tag=tag + ".close")
    return overlap_first_come(closed, gated, arena=arena, tag=tag + ".ofc"), gated


def process_masks_parallel(iset, apply=None, arena=None, tag="k2"):
    """process_masks_parallel (src/functions/inference.py:170-213): fill holes -> erosion(disk 1) -> dilation(disk 1)."""
    return morph(iset, [MORPH_FILL, MORPH_ERODE, MORPH_DILATE], apply=apply, arena=arena, tag=tag + ".open")


def postprocess_masks_universal(iset, groups, is_small_class, min_crys_size=None, arena=None, tag="k2", out=None):
    """postprocess_masks_universal (src/functions/inference.py:1739-1813).  Returns (InstanceSet, Groups of survivors)."""
    if min_crys_size is None:
        a = iset.H * iset.W
        min_crys_size = max(3, int(a * 0.000005)) if is_small_class else max(25, int(a * 0.0001))
    res = morph(iset, [MORPH_FILL, MORPH_ERODE] if is_small_class else [MORPH_FILL, MORPH_ERODE, MORPH_DILATE], arena=arena,
                tag=tag + ".univ")
    return res, filter_area(res, groups, min_crys_size, out=out)


CAP_CONTOURS = 8   # contours per instance held by the single-pass slab layout


def default_min_area(H, W):
    """Contour-area gate of the measurement loop (src/functions/inference.py:1178-1184)."""
    return max(5, H * W * 0.000005 * 0.05)


def trace(iset, single_pass=True, marks=None, arena=None, tag="k5", pt_cap=None):
    """K5a: external contours of every instance.  Leaves on the device: vertex lists (pts, cstart), the number of contours and
    the hull scratch size per instance, and perim0 = arcLength(contours[0]) (the compactness pre-filter of
    deduplicate_masks_smart needs it).  single_pass follows every border once into bounded per-instance slabs; an overflow
    (counter in extra["overflow"]) is detected by the next measure*() call, which re-traces exactly.  The vertex buffer of
    the single pass is sized by buffer_len() (capacity tag + ".pts" of the arena), or takes pt_cap when the caller already
    knows the exact size."""
    lib = _lib.load()
    dev = iset.device
    n = iset.n
    st = _stream()
    if marks is None:     # 2 bit planes per crop word, addressed by the (possibly shared) crop offsets
        marks = torch.empty(max(2 * iset.total_crop_words, 1), dtype=torch.int32, device=dev)
    perim0 = torch.empty(max(n, 1), dtype=torch.float64, device=dev)
    sizes = torch.empty((3, n + 1), dtype=torch.int64, device=dev)     # rows: n_contours, pt offsets, scratch bytes
    if single_pass and n:
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        with _stage("k5_plan+scan"):
            _lib.check(lib.emia_contour_trace_plan(_ptr(iset.meta), n, _ptr(sizes[1]), st), "emia_contour_trace_plan")
            exclusive_scan_(sizes[1])
        # the size is a pure function of the crop sizes: 4 * (sum ch + 32 * sum cw) + 32 * n_live
        cap_total = pt_cap if pt_cap is not None else buffer_len(sizes[1, n:], n, arena, tag + ".pts", n * 1536 + 65536)
        pts = torch.empty(max(cap_total, 1), dtype=torch.int32, device=dev)
        cstart = torch.empty(n * (CAP_CONTOURS + 1) + 1, dtype=torch.int32, device=dev)
        with _stage("k5_trace"):
            _lib.check(lib.emia_contour_trace_slab(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), n, _ptr(marks), _ptr(sizes[1]),
                                                   CAP_CONTOURS, _ptr(pts), _ptr(cstart), _ptr(sizes[0]), _ptr(sizes[2]), _ptr(flag),
                                                   _ptr(perim0), _ptr(arena.abort) if arena is not None else 0, st),
                       "emia_contour_trace_slab")
        LAUNCHES["count"] += 2
        iset.cstart_stride = CAP_CONTOURS + 1
        iset.extra["overflow"] = flag
        iset.cont_off = None
    else:
        with _stage("k5_count"):
            _lib.check(lib.emia_contour_count(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), n, _ptr(marks), _ptr(sizes[0]),
                                              _ptr(sizes[1]), _ptr(sizes[2]), st), "emia_contour_count")
        cont_off = sizes[0].clone()
        with _stage("k5_scans"):
            exclusive_scan_(cont_off)
            exclusive_scan_(sizes[1])
        totals = [int(cont_off[n].item()), int(sizes[1, n].item())] if n else [0, 0]
        pts = torch.empty(max(totals[1], 1), dtype=torch.int32, device=dev)
        cstart = torch.empty(totals[0] + n + 1, dtype=torch.int32, device=dev)
        with _stage("k5_trace"):
            _lib.check(lib.emia_contour_store(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), n, _ptr(marks), _ptr(cont_off),
                                              _ptr(sizes[1]), _ptr(pts), _ptr(cstart), _ptr(perim0), st), "emia_contour_store")
        LAUNCHES["count"] += 2
        iset.cstart_stride = 0
        iset.extra.pop("overflow", None)
        iset.cont_off = cont_off
    iset.pt_off, iset.pts, iset.cstart, iset.perim0 = sizes[1], pts, cstart, perim0
    iset.extra["n_contours"] = sizes[0]
    iset.extra["scratch_bytes"] = sizes[2]
    return iset


@dataclass
class Measurements:
    """Morphometry records of the members of G lists: the rows of list slot s are records[rec_off[s]:rec_off[s+1]]
    (OpenCV contour order); rec_inst[r] = instance id of row r; a row counts when records[r, REC_MEASURED] == 1."""
    records: torch.Tensor     # float64 [R, 16]
    rec_inst: torch.Tensor    # int32 [R]
    rec_off: torch.Tensor     # int64 [L + 1]
    n_records: Optional[int]  # None: sized by capacity, call finalize()
    groups: "Groups"
    totals: object = None     # (records, scratch bytes): host ints, or a device tensor until finalize()

    def finalize(self):
        """Read the totals back (one host synchronisation) and trim the capacity-sized buffers."""
        if self.n_records is None:
            n_rec, n_scr = (int(v) for v in self.totals.tolist())
            self.totals = (n_rec, n_scr)
            self.n_records = n_rec
            self.records, self.rec_inst = self.records[:n_rec], self.rec_inst[:n_rec]
        return self

    def rows_to_host(self):
        """Per group: list of (instance id, float64 [k,16] rows) in list order (host copies)."""
        rec = self.records.cpu().numpy(); off = self.rec_off.cpu().numpy()
        ln = self.groups.length.cpu().numpy(); idx = self.groups.idx.cpu().numpy()
        co = self.groups.cap_off_host
        return [[(int(idx[co[g] + k]), rec[off[co[g] + k]: off[co[g] + k + 1]]) for k in range(int(ln[g]))]
                for g in range(self.groups.G)]


def _measure_order(iset, item_inst, rec_off, L):
    """The K5 work order of a list of L slots, or None below MEASURE_ORDER_MIN_SLOTS."""
    if not (MEASURE_ORDER and L >= MEASURE_ORDER_MIN_SLOTS):
        return None
    # work order: slots sorted by vertex count (a warp of the morphometry kernel is as slow as its longest contour).  Measured:
    # 1 M slots -0.80 ms, 128 K slots -0.04 ms, 8 K - 44 K slots (the batched flows) +0.06 ... +0.17 ms (three more graph
    # nodes and a scattered hull pass for a stage that is only 0.1 ms there) - hence the threshold
    lib = _lib.load()
    dev = iset.device
    order = torch.empty(L, dtype=torch.int32, device=dev)
    bins = torch.empty(128, dtype=torch.int32, device=dev)
    with _stage("k5_order"):
        _lib.check(lib.emia_list_measure_order(L, _ptr(item_inst), _ptr(rec_off), _ptr(iset.cont_off), _ptr(iset.cstart),
                                               iset.cstart_stride, _ptr(order), _ptr(bins), _stream()), "emia_list_measure_order")
    LAUNCHES["count"] += 2
    return order


def measure_list(iset, groups, um_pix=1.0, min_area=None, arena=None, tag="k5"):
    """K5b: morphometry of the members of `groups` only (what the reference's measurement loop sees).  Needs trace().
    Returns None when the single-pass trace overflowed (the caller re-traces with single_pass=False).
    With an arena there is no host synchronisation: the buffers take the arena's capacities tag + ".records" and
    tag + ".scratch" (bytes), its abort flag is raised on the device when the actual totals (or a slab) overflow, and nothing
    is written then; the returned Measurements has n_records = None until finalize()."""
    lib = _lib.load()
    dev = iset.device
    assert iset.pts is not None, "run trace() first"
    if min_area is None:
        min_area = default_min_area(iset.H, iset.W)
    L = groups.total_cap
    st = _stream()
    item_inst = torch.empty(max(L, 1), dtype=torch.int32, device=dev)
    offs = torch.zeros((2, L + 1), dtype=torch.int64, device=dev)
    with _stage("k5_list_plan+scans"):
        _lib.check(lib.emia_list_measure_plan(_ptr(groups.cap_off), groups.G, L, _ptr(groups.length), _ptr(groups.idx),
                                              _ptr(iset.extra["n_contours"]), _ptr(iset.extra["scratch_bytes"]), _ptr(item_inst),
                                              _ptr(offs[0]), _ptr(offs[1]), st), "emia_list_measure_plan")
        exclusive_scan_(offs[0])
        exclusive_scan_(offs[1])
    LAUNCHES["count"] += 1
    flag = iset.extra.get("overflow")
    if arena is not None:
        # device-side checks, stream-ordered before the kernels that honour the flag (a slab overflow of the trace counts too)
        n_rec = buffer_len(offs[0, L:], L, arena, tag + ".records", L + L // 8 + 64)
        n_scr = buffer_len(offs[1, L:], L, arena, tag + ".scratch", L * 4096 + 65536)
        if flag is not None:
            arena.abort.logical_or_(flag)
    else:
        # one read for both totals and the slab overflow flag
        tot = torch.stack([offs[0, L], offs[1, L], flag[0].to(torch.int64) if flag is not None else offs[0, 0]]).tolist()
        n_rec, n_scr, overflow = int(tot[0]), int(tot[1]), int(tot[2])
        if overflow:
            return None
    records = torch.empty((max(n_rec, 1), REC_FIELDS), dtype=torch.float64, device=dev)
    rec_inst = torch.empty(max(n_rec, 1), dtype=torch.int32, device=dev)
    scratch = torch.empty(max(n_scr, 16), dtype=torch.uint8, device=dev)
    if L:
        order = _measure_order(iset, item_inst, offs[0], L)
        with _stage("k5_measure"):
            _lib.check(lib.emia_contour_measure_list(L, _ptr(item_inst), _ptr(offs[0]), _ptr(offs[1]), _ptr(iset.cont_off),
                                                     _ptr(iset.pt_off), _ptr(iset.cstart), iset.cstart_stride, float(um_pix),
                                                     float(min_area), _ptr(iset.pts), _ptr(records), _ptr(rec_inst), _ptr(scratch),
                                                     _ptr(arena.abort) if arena is not None else 0, _ptr(order) if order is not None else 0,
                                                     st), "emia_contour_measure_list")
        LAUNCHES["count"] += 2
    if arena is not None:
        return Measurements(records=records, rec_inst=rec_inst, rec_off=offs[0], n_records=None, groups=groups,
                            totals=torch.stack([offs[0, L], offs[1, L]]))
    return Measurements(records=records[:n_rec], rec_inst=rec_inst[:n_rec], rec_off=offs[0], n_records=n_rec, groups=groups,
                        totals=(n_rec, n_scr))


SHAPE_FIELDS = 10   # EMIA_S_COUNT: area, convex area, solidity, convex perimeter, convexity, max / min Feret, Feret angle, centroid x / y


def shape_list(iset, meas, um_pix=1.0):
    """Shape descriptors float64 [R, SHAPE_FIELDS] of the records of `meas`, an exact measure_list result on `iset` (row r belongs to
    meas.records[r]; NaN rows for records below the area gate): area, convex hull area, solidity, convex hull perimeter, convexity,
    max / min Feret diameter, max-Feret angle in degrees [0, 180) with y up (areas and lengths scaled by um_pix), and the centroid in
    frame pixels (core/emia_shape.cuh, oracle/shape.py).  The hull scratch of measure_list is sized again (one host
    synchronisation); the slots take the K5 work order from MEASURE_ORDER_MIN_SLOTS on."""
    lib = _lib.load()
    dev = iset.device
    if meas.n_records is None:
        raise ValueError("shape_list needs an exact measure_list result: call finalize() first")
    R = int(meas.n_records)
    shape = torch.empty((max(R, 1), SHAPE_FIELDS), dtype=torch.float64, device=dev)
    groups = meas.groups
    L = groups.total_cap
    if R == 0 or L == 0:
        return shape[:0]
    st = _stream()
    item_inst = torch.empty(L, dtype=torch.int32, device=dev)
    offs = torch.zeros((2, L + 1), dtype=torch.int64, device=dev)
    with _stage("shape_plan+scan"):
        _lib.check(lib.emia_list_measure_plan(_ptr(groups.cap_off), groups.G, L, _ptr(groups.length), _ptr(groups.idx),
                                              _ptr(iset.extra["n_contours"]), _ptr(iset.extra["scratch_bytes"]), _ptr(item_inst),
                                              _ptr(offs[0]), _ptr(offs[1]), st), "emia_list_measure_plan")
        exclusive_scan_(offs[1])
    LAUNCHES["count"] += 1
    scratch = torch.empty(max(buffer_len(offs[1, L:], L), 16), dtype=torch.uint8, device=dev)
    order = _measure_order(iset, item_inst, meas.rec_off, L)
    records = meas.records.contiguous()
    with _stage("shape"):
        _lib.check(lib.emia_contour_shape_list(L, _ptr(item_inst), _ptr(meas.rec_off), _ptr(offs[1]), _ptr(iset.cont_off), _ptr(iset.pt_off),
                                               _ptr(iset.cstart), iset.cstart_stride, float(um_pix), _ptr(iset.pts), _ptr(records),
                                               _ptr(scratch), _ptr(order) if order is not None else 0, _ptr(shape), st),
                   "emia_contour_shape_list")
    LAUNCHES["count"] += 1
    return shape[:R]


def shape_descriptors(iset):
    """shape_list over every record of a set after measure(): float64 [n_records, SHAPE_FIELDS], row for row with iset.records, at
    the um_pix of that measure() call."""
    assert iset.records is not None, "run measure() first"
    ident = groups_from_offsets([0, iset.n], iset.device)
    meas = Measurements(records=iset.records, rec_inst=iset.rec_inst, rec_off=iset.cont_off, n_records=iset.n_records, groups=ident)
    return shape_list(iset, meas, iset.extra["um_pix"])


def measure(iset, um_pix=1.0, min_area=None, single_pass=True):
    """K5 over EVERY instance of the set: trace() + measure_list() on the identity list.  Records of instance i are
    iset.records[cont_off[i]:cont_off[i+1]]."""
    if min_area is None:
        min_area = default_min_area(iset.H, iset.W)
    trace(iset, single_pass=single_pass)
    ident = groups_from_offsets([0, iset.n], iset.device)
    m = measure_list(iset, ident, um_pix, min_area)
    if m is None:
        trace(iset, single_pass=False)
        m = measure_list(iset, ident, um_pix, min_area)
    if iset.cont_off is None:
        iset.cont_off = m.rec_off
    iset.records, iset.rec_inst, iset.n_records = m.records, m.rec_inst, m.n_records
    iset.extra["um_pix"] = um_pix
    iset.extra["min_area"] = min_area
    return iset


def measure_contours(contours, um_pix=1.0, device=None):
    """Morphometry records [n,16] (float64, device) of n explicit contours (each an int array [K,2] or OpenCV's [K,1,2]):
    the kernel behind calculate_measurements (src/utils/measurements.py:114-233) for callers that hold contours."""
    return _measure_contours(contours, um_pix, device)[0]


def shape_contours(contours, um_pix=1.0, device=None):
    """Shape descriptors [n, SHAPE_FIELDS] (float64, device; shape_list's columns) of n explicit contours, measured without an area
    gate."""
    lib = _lib.load()
    records, n, d_cont, d_pt, d_cs, d_scr, d_pts, scratch = _measure_contours(contours, um_pix, device)
    dev = records.device
    shape = torch.empty((max(n, 1), SHAPE_FIELDS), dtype=torch.float64, device=dev)
    item_inst = torch.arange(max(n, 1), dtype=torch.int32, device=dev)
    _lib.check(lib.emia_contour_shape_list(n, _ptr(item_inst), _ptr(d_cont), _ptr(d_scr), _ptr(d_cont), _ptr(d_pt), _ptr(d_cs), 0,
                                           float(um_pix), _ptr(d_pts), _ptr(records), _ptr(scratch), 0, _ptr(shape), _stream()),
               "emia_contour_shape_list")
    LAUNCHES["count"] += 1
    return shape[:n]


def _measure_contours(contours, um_pix, device):
    """measure_contours: (records [n, 16], n, and the device list it measured: cont_off, pt_off, cstart, scratch offsets, points,
    scratch)."""
    lib = _lib.load()
    dev = _need_cuda(device)
    n = len(contours)
    lens = np.array([len(c) for c in contours], np.int64)
    pt_off = np.zeros(n + 1, np.int64); pt_off[1:] = np.cumsum(lens)
    flat = (np.concatenate([np.asarray(c).reshape(-1, 2) for c in contours]) if n and pt_off[-1] else np.zeros((0, 2), np.int64))
    if flat.size and (flat.min() < 0 or flat.max() > 0xFFFF):
        raise _lib.EmiaError("contour coordinates must lie in [0, 65535]")
    packed = (flat[:, 0].astype(np.uint32) | (flat[:, 1].astype(np.uint32) << 16)).astype(np.uint32)
    cont_off = np.arange(n + 1, dtype=np.int64)
    cstart = np.zeros(2 * n + 1, np.int32)
    cstart[1:2 * n:2] = lens.astype(np.int32)           # instance i: entries (0, len_i) at cont_off[i] + i = 2 i
    scr = ((28 * lens + 64 + 15) // 16) * 16
    scr_off = np.zeros(n + 1, np.int64); scr_off[1:] = np.cumsum(scr)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev)
    d_pts = t(packed.view(np.int32)) if packed.size else torch.zeros(1, dtype=torch.int32, device=dev)
    d_cont, d_pt, d_cs, d_scr = t(cont_off), t(pt_off), t(cstart), t(scr_off)
    records = torch.empty((max(n, 1), REC_FIELDS), dtype=torch.float64, device=dev)
    rec_inst = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    perim0 = torch.empty(max(n, 1), dtype=torch.float64, device=dev)
    scratch = torch.empty(max(int(scr_off[-1]), 16), dtype=torch.uint8, device=dev)
    dummy_meta = torch.zeros((max(n, 1), 8), dtype=torch.int32, device=dev)
    _lib.check(lib.emia_contour_measure_stored(_ptr(dummy_meta), n, _ptr(d_cont), _ptr(d_pt), _ptr(d_cs), 0, _ptr(d_scr), float(um_pix), 0.0,
                                               _ptr(d_pts), _ptr(records), _ptr(rec_inst), _ptr(perim0), _ptr(scratch), _stream()),
               "emia_contour_measure_stored")
    LAUNCHES["count"] += 2
    return records[:n], n, d_cont, d_pt, d_cs, d_scr, d_pts, scratch


def contours_to_host(iset):
    """Host copy of the contour vertex lists: list (per instance) of lists (OpenCV order) of int32 [k,2] arrays."""
    pts = iset.pts.cpu().numpy().view(np.uint32)
    ncont = iset.extra["n_contours"].cpu().numpy()
    cont_off = np.concatenate([[0], np.cumsum(ncont[:iset.n])])
    pt_off = iset.pt_off.cpu().numpy(); cstart = iset.cstart.cpu().numpy()
    out = []
    for i in range(iset.n):
        nc = int(ncont[i])
        base = i * iset.cstart_stride if iset.cstart_stride else cont_off[i] + i
        cs = cstart[base: base + nc + 1]
        cl = []
        for j in range(nc):
            k = nc - 1 - j
            p = pts[pt_off[i] + cs[k]: pt_off[i] + cs[k + 1]]
            cl.append(np.stack([p & 0xFFFF, p >> 16], 1).astype(np.int32))
        out.append(cl)
    return out


@dataclass
class Groups:
    """G lists of instance ids (one per image / tile / de-dup call)."""
    cap_off_host: np.ndarray      # int32 [G+1]
    cap_off: torch.Tensor         # int32 [G+1] (device)
    length: torch.Tensor          # int32 [G]
    idx: torch.Tensor             # int32 [cap_off[G]]

    @property
    def G(self):
        return len(self.cap_off_host) - 1

    @property
    def total_cap(self):
        return int(self.cap_off_host[-1])

    @property
    def max_cap(self):
        return int(np.diff(self.cap_off_host).max()) if self.G else 0

    @property
    def fused_cap(self):
        """Largest group capacity handed to the K4 entry points (0 = unknown -> staged kernels); FUSED_K4 = False forces the
        staged global-memory path (tests compare both)."""
        return self.max_cap if FUSED_K4 else 0

    def to_lists(self):
        ln = self.length.cpu().numpy()
        ix = self.idx.cpu().numpy()
        return [ix[self.cap_off_host[g]: self.cap_off_host[g] + ln[g]].tolist() for g in range(self.G)]


def groups_from_offsets(offsets, device):
    """Identity lists: group g = instances [offsets[g], offsets[g+1])."""
    off = np.asarray(offsets, dtype=np.int32)
    cap_off = torch.as_tensor(off, device=device)
    length = torch.as_tensor(np.diff(off).astype(np.int32), device=device)
    idx = torch.arange(int(off[-1]), dtype=torch.int32, device=device) + int(off[0])
    off0 = (off - off[0]).astype(np.int32)
    return Groups(cap_off_host=off0, cap_off=torch.as_tensor(off0, device=device), length=length, idx=idx)


def groups_from_lists(lists, device):
    off = np.zeros(len(lists) + 1, np.int32)
    off[1:] = np.cumsum([len(l) for l in lists])
    flat = np.concatenate([np.asarray(l, np.int32) for l in lists]) if off[-1] else np.zeros(0, np.int32)
    return Groups(cap_off_host=off, cap_off=torch.as_tensor(off, device=device),
                  length=torch.as_tensor(np.diff(off).astype(np.int32), device=device),
                  idx=torch.as_tensor(flat, device=device))


class GroupSpace:
    """One (length, idx) allocation shared by several SECTIONS of groups (e.g. the full-image lists and the tile lists of a
    batch).  Each section is an ordinary Groups object over views of the shared arrays, so the last kernel of a flow stage can
    write its surviving lists straight into the space, and flatten() can then concatenate lists of different sections
    (`full_image_masks + all_tile_masks`, src/functions/inference.py:2452) without moving any instance data."""

    def __init__(self, section_caps, device):
        self.dev = torch.device(device)
        caps = [np.asarray(c, dtype=np.int64).reshape(-1) for c in section_caps]
        self.g0 = np.concatenate([[0], np.cumsum([len(c) for c in caps])]).astype(np.int64)
        allc = np.concatenate(caps) if caps else np.zeros(0, np.int64)
        self.cap_abs = np.concatenate([[0], np.cumsum(allc)]).astype(np.int32)
        G, L = len(allc), int(self.cap_abs[-1])
        self.length = torch.zeros(max(G, 1), dtype=torch.int32, device=self.dev)
        self.idx = torch.empty(max(L, 1), dtype=torch.int32, device=self.dev)
        self.cap_off = torch.as_tensor(self.cap_abs, device=self.dev)
        self._sections = {}

    def fresh(self):
        """The same layout with new (length, idx) arrays (a new run of the flow); the device offset tables are shared."""
        o = object.__new__(GroupSpace)
        o.dev, o.g0, o.cap_abs, o.cap_off = self.dev, self.g0, self.cap_abs, self.cap_off
        o.length = torch.zeros_like(self.length)
        o.idx = torch.empty_like(self.idx)
        o._sections = {}
        o._rebased = self._rebased_tables()
        return o

    def _rebased_tables(self):
        r = getattr(self, "_rebased", None)
        if r is None:
            r = {}
            self._rebased = r
        return r

    def section(self, k):
        sec = self._sections.get(k)
        if sec is None:
            a, b = int(self.g0[k]), int(self.g0[k + 1])
            l0, l1 = int(self.cap_abs[a]), int(self.cap_abs[b])
            host = (self.cap_abs[a:b + 1] - self.cap_abs[a]).astype(np.int32)
            tabs = self._rebased_tables()
            dev_tab = tabs.get(k)
            if dev_tab is None:
                dev_tab = torch.as_tensor(host, device=self.dev)
                tabs[k] = dev_tab
            sec = Groups(cap_off_host=host, cap_off=dev_tab, length=self.length[a:max(b, a + 1)] if b > a else self.length[a:a],
                         idx=self.idx[l0:max(l1, l0 + 1)] if l1 > l0 else self.idx[l0:l0])
            self._sections[k] = sec
        return sec

    def range(self, k0, k1):
        """Sections k0 .. k1-1 as ONE Groups object (their groups are contiguous in the space)."""
        key = ("range", k0, k1)
        sec = self._sections.get(key)
        if sec is None:
            a, b = int(self.g0[k0]), int(self.g0[k1])
            l0, l1 = int(self.cap_abs[a]), int(self.cap_abs[b])
            host = (self.cap_abs[a:b + 1] - self.cap_abs[a]).astype(np.int32)
            tabs = self._rebased_tables()
            dev_tab = tabs.get(key)
            if dev_tab is None:
                dev_tab = torch.as_tensor(host, device=self.dev)
                tabs[key] = dev_tab
            sec = Groups(cap_off_host=host, cap_off=dev_tab, length=self.length[a:b], idx=self.idx[l0:max(l1, l0 + 1)])
            self._sections[key] = sec
        return sec

    def group_index(self, k, j=0):
        return int(self.g0[k]) + j


def flatten(space, grp_lists, id_add=None, cache=None):
    """New Groups with one list per entry of grp_lists: list s = the members of the space's groups grp_lists[s] (global group
    indices, in that order) one after the other.  id_add: per group of the space, added to its member ids (host int array)."""
    lib = _lib.load()
    dev = space.dev
    key = None if cache is None else "flatten"
    tabs = None if cache is None else cache.get(key)
    if tabs is None:
        seg = np.zeros(len(grp_lists) + 1, np.int32)
        seg[1:] = np.cumsum([len(g) for g in grp_lists])
        flat = np.concatenate([np.asarray(g, np.int32) for g in grp_lists]) if seg[-1] else np.zeros(1, np.int32)
        caps = np.array([int(sum(int(space.cap_abs[g + 1] - space.cap_abs[g]) for g in gl)) for gl in grp_lists], np.int64)
        out_off = np.concatenate([[0], np.cumsum(caps)]).astype(np.int32)
        tabs = (seg, torch.as_tensor(seg, device=dev), torch.as_tensor(flat, device=dev), out_off, torch.as_tensor(out_off, device=dev),
                None if id_add is None else torch.as_tensor(np.asarray(id_add, np.int32), device=dev))
        if cache is not None:
            cache[key] = tabs
    seg, seg_t, flat_t, out_off, out_off_t, add_t = tabs
    S = len(seg) - 1
    out = Groups(cap_off_host=out_off, cap_off=out_off_t, length=torch.empty(max(S, 1), dtype=torch.int32, device=dev),
                 idx=torch.empty(max(int(out_off[-1]), 1), dtype=torch.int32, device=dev))
    _lib.check(lib.emia_group_flatten(_ptr(space.cap_off), len(space.cap_abs) - 1, _ptr(space.length), _ptr(space.idx), _ptr(flat_t),
                                      _ptr(seg_t), S, _ptr(add_t), _ptr(out_off_t), _ptr(out.length), _ptr(out.idx), _stream()),
               "emia_group_flatten")
    LAUNCHES["count"] += 1
    return out


_ws_cache = {}


def _workspace(groups, device):
    lib = _lib.load()
    key = (groups.cap_off_host.tobytes(), str(device))
    nbytes = _ws_cache.get(key)
    if nbytes is None:
        host = np.ascontiguousarray(groups.cap_off_host, dtype=np.int32)
        nbytes = int(lib.emia_group_workspace_bytes(host.ctypes.data, groups.G))
        if len(_ws_cache) > 256:
            _ws_cache.clear()
        _ws_cache[key] = nbytes
    return torch.empty(nbytes, dtype=torch.uint8, device=device), nbytes


def _new_groups_like(g):
    return Groups(cap_off_host=g.cap_off_host, cap_off=g.cap_off, length=torch.empty_like(g.length), idx=torch.empty_like(g.idx))


def dedup_smart(iset, groups, iou_threshold=0.4, max_aspect_ratio=None, out=None):
    """deduplicate_masks_smart (src/functions/inference.py:2552) on every group.  Needs measure() first (compactness)."""
    lib = _lib.load()
    assert iset.perim0 is not None, "run trace() before dedup_smart (the pre-filter needs contour perimeters)"
    ws, nb = _workspace(groups, iset.device)
    out = out if out is not None else _new_groups_like(groups)
    ncont = iset.extra["n_contours"]
    with _stage("k4_dedup_smart"):
      _lib.check(lib.emia_dedup_smart(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(iset.bbox), _ptr(iset.area),
                                    _ptr(iset.perim0), _ptr(ncont), _ptr(iset.scores), _ptr(iset.classes), _ptr(groups.cap_off),
                                    groups.G, groups.total_cap, groups.fused_cap, _ptr(groups.length), _ptr(groups.idx), float(iou_threshold),
                                    float(max_aspect_ratio) if max_aspect_ratio else 0.0, _ptr(out.length), _ptr(out.idx),
                                    _ptr(ws), nb, _stream()), "emia_dedup_smart")
    LAUNCHES["count"] += 6
    return out


def dedup_inorder(iset, groups, iou_threshold, out=None):
    """Greedy in-order de-dup with iou() (src/functions/inference.py:1453-1459)."""
    lib = _lib.load()
    ws, nb = _workspace(groups, iset.device)
    out = out if out is not None else _new_groups_like(groups)
    _lib.check(lib.emia_dedup_inorder(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(iset.bbox), _ptr(iset.area),
                                      _ptr(groups.cap_off), groups.G, groups.total_cap, groups.fused_cap, _ptr(groups.length), _ptr(groups.idx),
                                      float(iou_threshold), _ptr(out.length), _ptr(out.idx), _ptr(ws), nb, _stream()),
               "emia_dedup_inorder")
    LAUNCHES["count"] += 6
    return out


def dedup_sorted(iset, groups, iou_threshold, out=None):
    """Score-sorted greedy de-dup with iou() (run_adaptive_multiscale_inference, src/functions/inference.py:1964-1978)."""
    lib = _lib.load()
    ws, nb = _workspace(groups, iset.device)
    out = out if out is not None else _new_groups_like(groups)
    _lib.check(lib.emia_dedup_sorted(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(iset.bbox), _ptr(iset.area),
                                     _ptr(iset.scores), _ptr(groups.cap_off), groups.G, groups.total_cap, groups.fused_cap,
                                     _ptr(groups.length), _ptr(groups.idx), float(iou_threshold), _ptr(out.length), _ptr(out.idx),
                                     _ptr(ws), nb, _stream()), "emia_dedup_sorted")
    LAUNCHES["count"] += 1 if groups.fused_cap and groups.fused_cap <= 1024 else 6
    return out


def filter_flag(groups, flag, keep_value=0, out=None):
    """List members whose flag[inst] == keep_value (e.g. the edge filter of the tile pipeline)."""
    lib = _lib.load()
    out = out if out is not None else _new_groups_like(groups)
    _lib.check(lib.emia_group_filter_flag(_ptr(groups.cap_off), groups.G, _ptr(groups.length), _ptr(groups.idx), _ptr(flag),
                                          int(keep_value), _ptr(out.length), _ptr(out.idx), _stream()), "emia_group_filter_flag")
    LAUNCHES["count"] += 1
    return out


def resize_place(iset, th, tw, Hd, Wd, off_xy=None, tile_size=None, overlap_ratio=None):
    """K3: cv2.resize(mask, (tw, th), INTER_NEAREST) of every instance of `iset` (frame iset.H x iset.W), placed at
    off_xy[i] = (x_offset, y_offset) of an Hd x Wd frame with the reference's clipping (src/functions/inference.py:2399-2420;
    :2044-2054 with th, tw = Hd, Wd and no offsets).  Returns (InstanceSet in the destination frame, edge_flag or None):
    edge_flag[i] = is_edge_mask(resized mask, tile_size, overlap_ratio) (inference.py:2522-2549)."""
    lib = _lib.load()
    dev = iset.device
    n = iset.n
    meta = torch.empty((n, 8), dtype=torch.int32, device=dev)
    crop_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    if off_xy is not None:
        off_xy = torch.as_tensor(off_xy, dtype=torch.int32, device=dev).contiguous()
        assert off_xy.shape == (n, 2)
    st = _stream()
    _lib.check(lib.emia_resize_place_plan(_ptr(iset.bbox), n, iset.H, iset.W, th, tw, _ptr(off_xy), 0, Hd, Wd, _ptr(meta), _ptr(crop_off), st),
               "emia_resize_place_plan")
    exclusive_scan_(crop_off)
    total = buffer_len(crop_off[n:], n)
    crops = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
    bbox = torch.empty((n, 4), dtype=torch.int32, device=dev)
    area = torch.empty(n, dtype=torch.int32, device=dev)
    edge = None
    edge_width = ts = 0
    if tile_size is not None:
        edge = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
        ts = int(tile_size)
        edge_width = int(tile_size * overlap_ratio / 2)
    _lib.check(lib.emia_resize_nearest_place(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(iset.bbox), n, iset.H, iset.W,
                                             th, tw, _ptr(off_xy), Hd, Wd, edge_width, ts, _ptr(meta), _ptr(crop_off), _ptr(crops),
                                             _ptr(bbox), _ptr(area), _ptr(edge), 0, st), "emia_resize_nearest_place")
    LAUNCHES["count"] += 2
    out = InstanceSet(n=n, H=Hd, W=Wd, meta=meta, crop_off=crop_off, crops=crops, bbox=bbox, area=area, scores=iset.scores,
                      classes=iset.classes, total_crop_words=total)
    return out, edge


class Combined:
    """A destination InstanceSet assembled by K3 from several source sets (the full-image pass and every tile of a micrograph;
    every scale of a multi-scale pass; every model of an ensemble), all back-projected into ONE H x W frame.  The reference
    allocates one full-frame array per instance for this (src/functions/inference.py:2413); here every part writes its
    word-aligned crops into a slice of shared arrays: plan all parts -> one scan -> (guarded) crop buffer -> place all parts.
    Part p owns the instance ids [start[p], start[p + 1])."""

    def __init__(self, part_sizes, H, W, device):
        dev = torch.device(device)
        self.H, self.W, self.dev = H, W, dev
        self.start = np.concatenate([[0], np.cumsum(part_sizes)]).astype(np.int64)
        n = int(self.start[-1])
        self.n = n
        self.meta = torch.empty((n, 8), dtype=torch.int32, device=dev)
        self.crop_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        self.bbox = torch.empty((n, 4), dtype=torch.int32, device=dev)
        self.area = torch.empty(n, dtype=torch.int32, device=dev)
        self.scores = torch.empty(n, dtype=torch.float32, device=dev)
        self.classes = torch.empty(n, dtype=torch.int32, device=dev)
        self.edge = torch.zeros(max(n, 1), dtype=torch.int32, device=dev)
        self.crops = None
        self.total = 0
        self._parts = []

    def plan(self, p, src, th, tw, off_xy=None, alive=None):
        """Part p <- cv2.resize(mask, (tw, th), INTER_NEAREST) of every instance of `src`, placed at off_xy[i] (int32 [n,2] device
        tensor of (x, y) offsets, or None).  alive (optional int32 [n]): instances with 0 are no longer in any list and are not
        resampled.  Only the geometry is computed here."""
        lib = _lib.load()
        a, b = int(self.start[p]), int(self.start[p + 1])
        assert b - a == src.n
        if src.n:
            _lib.check(lib.emia_resize_place_plan(_ptr(src.bbox), src.n, src.H, src.W, th, tw, _ptr(off_xy), _ptr(alive), self.H, self.W,
                                                  _ptr(self.meta[a:]), _ptr(self.crop_off[a:]), _stream()), "emia_resize_place_plan")
            LAUNCHES["count"] += 1
        self._parts.append((p, src, th, tw, off_xy, alive))

    def place(self, arena=None, tag="k3", edge=None):
        """Scan the crop sizes of all planned parts, size the crop buffer (exactly, or arena capacity + device-side guard) and
        run the placement kernels.  edge: {part: (tile_size, overlap_ratio)} -> is_edge_mask flags in self.edge."""
        lib = _lib.load()
        n = self.n
        exclusive_scan_(self.crop_off)
        total = buffer_len(self.crop_off[n:], n, arena, tag + ".crops",
                           sum(int(part[1].total_crop_words) for part in self._parts) + 64 * n + 1024, self.meta)
        self.total = total
        self.crops = torch.empty(max(total, 1), dtype=torch.int32, device=self.dev)
        st = _stream()
        for p, src, th, tw, off_xy, alive in self._parts:
            a = int(self.start[p])
            if not src.n:
                continue
            ew = ts = 0
            ef = None
            if edge and p in edge:
                ts = int(edge[p][0])
                ew = int(edge[p][0] * edge[p][1] / 2)
                ef = self.edge[a:]
            with _stage("k3_resize_place"):
                _lib.check(lib.emia_resize_nearest_place(_ptr(src.crops), _ptr(src.meta), _ptr(src.crop_off), _ptr(src.bbox), src.n, src.H,
                                                         src.W, th, tw, _ptr(off_xy), self.H, self.W, ew, ts, _ptr(self.meta[a:]),
                                                         _ptr(self.crop_off[a:]), _ptr(self.crops), _ptr(self.bbox[a:]), _ptr(self.area[a:]),
                                                         _ptr(ef), _ptr(alive), st), "emia_resize_nearest_place")
            LAUNCHES["count"] += 1
            if src.scores is not None:
                self.scores[a:a + src.n].copy_(src.scores)
            if src.classes is not None:
                self.classes[a:a + src.n].copy_(src.classes)
        return InstanceSet(n=n, H=self.H, W=self.W, meta=self.meta, crop_off=self.crop_off, crops=self.crops, bbox=self.bbox,
                           area=self.area, scores=self.scores, classes=self.classes, total_crop_words=total)


def unit_broadcast(unit_off_t, U, n, vals_t, k):
    """int32 [n, k]: the per-unit constants vals_t [U, k] expanded to the instances of every unit (device)."""
    lib = _lib.load()
    out = torch.empty((max(n, 1), k), dtype=torch.int32, device=vals_t.device)
    _lib.check(lib.emia_unit_broadcast_i32(_ptr(unit_off_t), U, n, _ptr(vals_t), k, _ptr(out), _stream()), "emia_unit_broadcast_i32")
    LAUNCHES["count"] += 1
    return out


def scale_scores(scores, weight, out=None):
    """score * weight in float32 (run_ensemble_inference, src/functions/inference.py:1553)."""
    lib = _lib.load()
    out = out if out is not None else torch.empty_like(scores)
    _lib.check(lib.emia_scale_f32(_ptr(scores), float(np.float32(weight)), scores.numel(), _ptr(out), _stream()), "emia_scale_f32")
    LAUNCHES["count"] += 1
    return out


def _gather_into(src, idx_t, k, meta, crop_off, a):
    """Plan step of a gather: geometry of src[idx] into rows [a, a + k) of (meta, crop_off-as-sizes)."""
    lib = _lib.load()
    if k:
        _lib.check(lib.emia_gather_plan(_ptr(src.meta), _ptr(idx_t), k, _ptr(meta[a:]), _ptr(crop_off[a:]), _stream()), "emia_gather_plan")
        LAUNCHES["count"] += 1


def _gather_copy(src, idx_t, k, dst, a):
    lib = _lib.load()
    if not k:
        return
    _lib.check(lib.emia_gather_crops(_ptr(src.crops), _ptr(src.crop_off), _ptr(src.bbox), _ptr(src.area), _ptr(idx_t), k, _ptr(dst.meta[a:]),
                                     _ptr(dst.crop_off[a:]), _ptr(dst.crops), _ptr(dst.bbox[a:]), _ptr(dst.area[a:]), _stream()),
               "emia_gather_crops")
    LAUNCHES["count"] += 1
    for name in ("scores", "classes"):
        s_, d_ = getattr(src, name), getattr(dst, name)
        if s_ is None or d_ is None:
            continue
        if idx_t is None:
            d_[a:a + k].copy_(s_[:k])
        else:
            _lib.check(lib.emia_gather_b32(_ptr(s_), _ptr(idx_t), k, _ptr(d_[a:]), _stream()), "emia_gather_b32")
            LAUNCHES["count"] += 1


def _empty_set(n, H, W, dev, scores=True, classes=True):
    return InstanceSet(n=n, H=H, W=W, meta=torch.empty((n, 8), dtype=torch.int32, device=dev),
                       crop_off=torch.zeros(n + 1, dtype=torch.int64, device=dev), crops=None,
                       bbox=torch.empty((n, 4), dtype=torch.int32, device=dev), area=torch.empty(n, dtype=torch.int32, device=dev),
                       scores=torch.empty(n, dtype=torch.float32, device=dev) if scores else None,
                       classes=torch.empty(n, dtype=torch.int32, device=dev) if classes else None)


def select(iset, idx):
    """A new InstanceSet holding instances idx (device or host int array) of `iset`, crops re-packed (emia_gather_* kernels)."""
    dev = iset.device
    idx_t = torch.as_tensor(np.asarray(idx, np.int32) if not torch.is_tensor(idx) else idx, dtype=torch.int32, device=dev).contiguous()
    k = int(idx_t.numel())
    out = _empty_set(k, iset.H, iset.W, dev, iset.scores is not None, iset.classes is not None)
    _gather_into(iset, idx_t, k, out.meta, out.crop_off, 0)
    exclusive_scan_(out.crop_off)
    total = buffer_len(out.crop_off[k:], k)
    out.crops = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
    out.total_crop_words = total
    _gather_copy(iset, idx_t, k, out, 0)
    return out


def concat(isets):
    """Concatenate InstanceSets of the same frame size (e.g. full-image pass + every tile, src/functions/inference.py:2452-2454):
    one plan launch per part, one scan, one copy launch per part."""
    isets = [s for s in isets if s is not None]
    assert isets and all(s.H == isets[0].H and s.W == isets[0].W for s in isets)
    dev = isets[0].device
    n = sum(s.n for s in isets)
    out = _empty_set(n, isets[0].H, isets[0].W, dev, all(s.scores is not None for s in isets), all(s.classes is not None for s in isets))
    a = 0
    for s_ in isets:
        _gather_into(s_, None, s_.n, out.meta, out.crop_off, a)
        a += s_.n
    exclusive_scan_(out.crop_off)
    total = buffer_len(out.crop_off[n:], n)
    out.crops = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
    out.total_crop_words = total
    a = 0
    for s_ in isets:
        _gather_copy(s_, None, s_.n, out, a)
        a += s_.n
    return out


def rle_encode(iset, idx=None):
    """K6: rle_encoding (src/utils/mask_utils.py:17-35) of every instance: (run_off int64 [n+1], runs int64 [R, 2]) on the device;
    runs[run_off[i]:run_off[i+1]] are the (start, length) pairs of instance i (column-major, 1-indexed)."""
    lib = _lib.load()
    dev = iset.device
    n = iset.n
    run_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    st = _stream()
    _lib.check(lib.emia_rle_count(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(iset.bbox), n, iset.H, _ptr(run_off), st),
               "emia_rle_count")
    exclusive_scan_(run_off)
    R = buffer_len(run_off[n:], n)
    runs = torch.empty((max(R, 1), 2), dtype=torch.int64, device=dev)
    _lib.check(lib.emia_rle_encode(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(iset.bbox), n, iset.H, _ptr(run_off),
                                   _ptr(runs), st), "emia_rle_encode")
    LAUNCHES["count"] += 2
    return run_off, runs[:R]


RLE_TEXT_CHUNK = 8192        # EMIA_RLE_TEXT_CHUNK
RLE_HEADER = b"ImageId,EncodedPixels"
RLE_STATUS = {1: "no comma separates ImageId from EncodedPixels", 2: "EncodedPixels holds a character other than a digit or a blank",
              3: "odd number of values", 4: "a value of more than 18 digits", 5: "a run with start < 1 or length < 1",
              6: "a run past pixel H * W", 7: "a run that starts at or before the end of the previous run (unsorted or overlapping)",
              8: "more than 2^31 - 1 pixels"}


def _csv_field(raw):
    """An ImageId as csv.writer wrote it: a quoted field loses its quotes and doubled inner quotes."""
    s = raw.decode("utf-8")
    if len(s) >= 2 and s[0] == '"' and s[-1] == '"':
        s = s[1:-1].replace('""', '"')
    return s


def _rle_parse(data, device=None):
    """rle_parse_csv plus the 1-based file line number of every data line (numpy int64)."""
    lib = _lib.load()
    dev = _need_cuda(device)
    data = bytes(data)
    first = data.split(b"\n", 1)[0].rstrip(b"\r ")
    if first != RLE_HEADER:
        raise _lib.EmiaError(f"rle_parse_csv: line 1: header {first[:64]!r} is not {RLE_HEADER!r}")
    nbytes = len(data)
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    host.numpy()[:] = np.frombuffer(data, np.uint8)
    st = _stream()
    with _stage("rle_h2d"):
        text = host.to(dev, non_blocking=True)
    with _stage("rle_parse"):
        chunks = (nbytes + RLE_TEXT_CHUNK - 1) // RLE_TEXT_CHUNK
        chunk_off = torch.zeros(chunks + 1, dtype=torch.int64, device=dev)
        _lib.check(lib.emia_rle_line_count(_ptr(text), nbytes, _ptr(chunk_off), st), "emia_rle_line_count")
        exclusive_scan_(chunk_off)
        L = int(chunk_off[chunks].item()) + (data[-1:] != b"\n")          # lines, the header included
        line_off = torch.empty(L + 2, dtype=torch.int64, device=dev)
        _lib.check(lib.emia_rle_line_index(_ptr(text), nbytes, _ptr(chunk_off), _ptr(line_off), st), "emia_rle_line_index")
        n = L - 1                                                          # lines after the header
        cnt = torch.zeros((2, n + 1), dtype=torch.int64, device=dev)      # rows: data lines, runs
        _lib.check(lib.emia_rle_parse_count(_ptr(text), _ptr(line_off[1:]), n, _ptr(cnt[0]), _ptr(cnt[1]), st), "emia_rle_parse_count")
        exclusive_scan_(cnt[0])
        exclusive_scan_(cnt[1])
        D, R = (int(v) for v in cnt[:, n].tolist())
        run_off = torch.zeros(D + 1, dtype=torch.int64, device=dev)
        runs = torch.empty((max(R, 1), 2), dtype=torch.int64, device=dev)
        field = torch.empty((max(D, 1), 2), dtype=torch.int64, device=dev)
        line_idx = torch.empty(max(D, 1), dtype=torch.int32, device=dev)
        status = torch.empty(max(D, 1), dtype=torch.int32, device=dev)
        _lib.check(lib.emia_rle_parse_fill(_ptr(text), _ptr(line_off[1:]), n, _ptr(cnt[0]), _ptr(cnt[1]), _ptr(run_off), _ptr(runs),
                                           _ptr(field), _ptr(line_idx), _ptr(status), st), "emia_rle_parse_fill")
    LAUNCHES["count"] += 4
    status = status[:D].cpu().numpy()
    line_no = line_idx[:D].cpu().numpy().astype(np.int64) + 2
    bad = np.nonzero(status)[0]
    if len(bad):
        k = int(bad[0])
        raise _lib.EmiaError(f"rle_parse_csv: line {line_no[k]}: {RLE_STATUS[int(status[k])]}")
    fld = field[:D].cpu().numpy()
    ids = [_csv_field(data[a:b]) for a, b in fld.tolist()]
    return ids, run_off, runs[:R], line_no


def rle_parse_csv(data, device=None):
    """The text of an R50_flip_results.csv file (bytes) -> (image_ids: list[str], run_off int64 [L+1], runs int64 [R, 2]) with the
    runs of data line k at runs[run_off[k]:run_off[k+1]] (device tensors), one H2D copy of the text and the parse in CUDA.
    Line 1 must be the header `ImageId,EncodedPixels`; empty lines are skipped; the last comma of a line separates the ImageId
    (quoted by csv.writer when it holds a comma) from EncodedPixels; an empty EncodedPixels field is an empty mask.
    Raises EmiaError naming the first malformed line (1-based line number of the file)."""
    ids, run_off, runs, _ = _rle_parse(data, device)
    return ids, run_off, runs


def _rle_decode(run_off, runs, H, W, rows=None):
    """(InstanceSet, per-instance status as numpy int32) of the lines `rows` (default: all) of (run_off, runs)."""
    lib = _lib.load()
    if not (1 <= H <= 65535 and 1 <= W <= 65535):
        raise _lib.EmiaError(f"rle_decode: frame {H} x {W} outside 1..65535 (the contour vertex packing limit)")
    dev = run_off.device
    assert run_off.dtype == torch.int64 and runs.dtype == torch.int64 and run_off.is_contiguous() and runs.is_contiguous()
    rows_t = None if rows is None else torch.as_tensor(np.asarray(rows, np.int32), device=dev)
    n = int(run_off.numel()) - 1 if rows is None else int(rows_t.numel())
    meta = torch.empty((n, 8), dtype=torch.int32, device=dev)
    crop_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    bbox = torch.empty((n, 4), dtype=torch.int32, device=dev)
    area = torch.empty(n, dtype=torch.int32, device=dev)
    status = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    st = _stream()
    rp = _ptr(runs) if runs.numel() else _ptr(run_off)      # no runs at all: never read, but the ABI wants a pointer
    with _stage("rle_decode"):
        _lib.check(lib.emia_rle_decode_plan(rp, _ptr(run_off), _ptr(rows_t), n, H, W, _ptr(meta), _ptr(crop_off), _ptr(bbox), _ptr(area),
                                            _ptr(status), st), "emia_rle_decode_plan")
        exclusive_scan_(crop_off)
        total = buffer_len(crop_off[n:], n)
        crops = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
        _lib.check(lib.emia_rle_decode(rp, _ptr(run_off), _ptr(rows_t), n, H, _ptr(meta), _ptr(crop_off), _ptr(crops), st),
                   "emia_rle_decode")
    LAUNCHES["count"] += 2
    iset = InstanceSet(n=n, H=H, W=W, meta=meta, crop_off=crop_off, crops=crops, bbox=bbox, area=area, total_crop_words=total)
    return iset, status[:n].cpu().numpy()


def rle_decode(run_off, runs, H, W):
    """Inverse of rle_encode: (run_off int64 [n+1], runs int64 [R, 2]) of an H x W frame -> InstanceSet, bit for bit the tables
    from_masks gives for the same masks (tight bbox crops), so rle_decode(*rle_encode(s), H, W) round-trips.  Runs are column-major
    and 1-indexed; one may continue from row H-1 of a column into the next columns.  Raises EmiaError naming the first instance
    with a bad run (start or length < 1, past H * W, unsorted or overlapping) or more than 2^31 - 1 pixels."""
    iset, status = _rle_decode(run_off, runs, H, W)
    bad = np.nonzero(status)[0]
    if len(bad):
        k = int(bad[0])
        raise _lib.EmiaError(f"rle_decode: instance {k}: {RLE_STATUS[int(status[k])]}")
    return iset


def csv_field(value):
    """The text csv.writer writes for `value` as one field of a row (QUOTE_MINIMAL: quoted when it holds a comma, a quote or a
    line break, inner quotes doubled; None is empty; a float is its repr)."""
    buf = io.StringIO()
    csv.writer(buf).writerow([value, ""])
    return buf.getvalue()[:-3]                     # the row ends in ",\r\n"


def _text_to_host(text, nbytes):
    """One D2H copy of text[:nbytes] into pinned memory -> bytes."""
    if nbytes == 0:
        return b""
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    host.copy_(text[:nbytes], non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return host.numpy().tobytes()


def _strings_to_device(strings, dev):
    """(UTF-8 bytes, int64 offsets [k + 1]) of k strings, on the device."""
    raw = [s.encode("utf-8") for s in strings]
    off = np.concatenate([[0], np.cumsum([len(b) for b in raw])]).astype(np.int64)
    data = torch.frombuffer(bytearray(b"".join(raw) or b"\0"), dtype=torch.uint8).to(dev)
    return data, torch.as_tensor(off, device=dev)


def _row_strings(file_name, psum, class_fields):
    """The string fields of a result row, rendered by csv_field: the Instance_ID text before and after the number, "Detected scale
    bar,File name", and "Class,Class_Name" per class-table entry."""
    ident = csv_field(f"{file_name}_1")                     # the digits never change the quoting of the whole field
    pre, suf = (ident[:-2], '"') if ident.endswith('"') else (ident[:-1], "")
    strs = [pre, suf, csv_field(psum) + "," + csv_field(file_name)]
    return strs + [csv_field(c) + "," + csv_field(name) for c, name in class_fields]


def rle_csv_text(run_off, runs, image_id):
    """The lines of R50_flip_results.csv for the instances of (run_off, runs) (rle_encode's output) of the image `image_id`: byte for
    byte what csv.writer writes for the rows (image_id, " ".join of the instance's runs), UTF-8, "\\r\\n" line ends; an empty mask
    gives `<ImageId>,`.  Formatted on the device; one host synchronisation to size the text and one D2H copy of it."""
    lib = _lib.load()
    dev = run_off.device
    assert run_off.dtype == torch.int64 and runs.dtype == torch.int64 and run_off.is_contiguous() and runs.is_contiguous()
    n = int(run_off.numel()) - 1
    if n <= 0:
        return b""
    prefix = (csv_field(image_id) + ",").encode("utf-8")
    pre = torch.frombuffer(bytearray(prefix), dtype=torch.uint8).to(dev)
    line_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    st = _stream()
    rp = _ptr(runs) if runs.numel() else _ptr(run_off)      # no runs at all: never read, but the ABI wants a pointer
    with _stage("csv_rle_count"):
        _lib.check(lib.emia_csv_rle_count(rp, _ptr(run_off), n, len(prefix), _ptr(line_off), st), "emia_csv_rle_count")
    with _stage("csv_rle_scan"):
        exclusive_scan_(line_off)
    nbytes = buffer_len(line_off[n:], n)
    text = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
    with _stage("csv_rle_write"):
        _lib.check(lib.emia_csv_rle_write(rp, _ptr(run_off), n, _ptr(pre), len(prefix), _ptr(line_off), _ptr(text), st),
                   "emia_csv_rle_write")
    LAUNCHES["count"] += 2
    with _stage("csv_rle_d2h"):
        return _text_to_host(text, nbytes)


def coco_annotations_text(iset, run_off, runs, image_id, category_ids, scores, first_id):
    """The "annotations" entries of coco_instances.json for the n instances of `iset` (with (run_off, runs) = rle_encode(iset)), joined
    by ", ": byte for byte json.dumps of the dicts oracle/coco.py defines.  Instance i gets id first_id + i, image_id, category_id
    category_ids[i], segmentation {"size": [H, W], "counts": pycocotools' compressed RLE string}, the popcount as area, the tight bbox
    [x, y, w, h] as floats and float(scores[i]) as score.  Formatted on the device; one host synchronisation to size the text and
    one D2H copy of it."""
    lib = _lib.load()
    dev = iset.device
    n = iset.n
    if n <= 0:
        return b""
    assert run_off.dtype == torch.int64 and runs.dtype == torch.int64 and run_off.is_contiguous() and runs.is_contiguous()
    assert int(run_off.numel()) == n + 1
    cat = torch.as_tensor(np.asarray([int(c) for c in category_ids], np.int32), device=dev)
    sc = torch.as_tensor(np.asarray([float(s) for s in scores], np.float64), device=dev)
    assert cat.numel() == n and sc.numel() == n
    bbox, area = iset.bbox.contiguous(), iset.area.contiguous()
    ann_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    st = _stream()
    rp = _ptr(runs) if runs.numel() else _ptr(run_off)      # no runs at all: never read, but the ABI wants a pointer
    args = (rp, _ptr(run_off), n, _ptr(bbox), _ptr(area), _ptr(sc), _ptr(cat), iset.H, iset.W, int(image_id), int(first_id))
    with _stage("coco_ann_count"):
        _lib.check(lib.emia_coco_ann_count(*args, _ptr(ann_off), st), "emia_coco_ann_count")
    with _stage("coco_ann_scan"):
        exclusive_scan_(ann_off)
    nbytes = buffer_len(ann_off[n:], n)
    text = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
    with _stage("coco_ann_write"):
        _lib.check(lib.emia_coco_ann_write(*args, _ptr(ann_off), _ptr(text), st), "emia_coco_ann_write")
    LAUNCHES["count"] += 2
    with _stage("coco_ann_d2h"):
        return _text_to_host(text, nbytes)


COCO_STATUS = {1: "counts hold a character outside '0'..'o'", 2: "counts end inside a value",
               3: "a count below 0 or above 2^31 - 1 (or a value of more than 7 characters)", 4: "counts do not add up to H * W",
               5: "more than 2^31 - 1 pixels"}


def _coco_decode(data, str_off, H, W):
    """n compressed-RLE counts strings of H x W masks (bytes `data`, string j at data[str_off[j]:str_off[j + 1]]) -> (InstanceSet of
    the n masks, per-string status as numpy int32: 0 or a COCO_STATUS key).  A rejected string gives an empty mask.  One H2D copy;
    counts -> runs on the device, then the RLE decode (tight bbox crops, as rle_decode)."""
    lib = _lib.load()
    if not (1 <= H <= 65535 and 1 <= W <= 65535):
        raise _lib.EmiaError(f"coco_decode: frame {H} x {W} outside 1..65535 (the contour vertex packing limit)")
    dev = _need_cuda(None)
    off = np.asarray(str_off, np.int64)
    n = len(off) - 1
    nbytes = len(data)
    a = (nbytes + 7) // 8 * 8                                      # the offsets follow the text, 8-byte aligned
    host = torch.zeros(a + 8 * (n + 1), dtype=torch.uint8, pin_memory=True)
    hv = host.numpy()
    hv[:nbytes] = np.frombuffer(bytes(data), np.uint8)
    hv[a:] = off.view(np.uint8)
    st = _stream()
    with _stage("coco_h2d"):
        both = host.to(dev, non_blocking=True)                    # one H2D copy of text and offsets
    text = both[:max(a, 1)]
    s_off = both[a:].view(torch.int64)
    with _stage("coco_counts"):
        run_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        status = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
        _lib.check(lib.emia_coco_counts_count(_ptr(text), _ptr(s_off), n, H, W, _ptr(run_off), _ptr(status), st), "emia_coco_counts_count")
        exclusive_scan_(run_off)
        R = buffer_len(run_off[n:], n)
        runs = torch.empty((max(R, 1), 2), dtype=torch.int64, device=dev)
        _lib.check(lib.emia_coco_counts_fill(_ptr(text), _ptr(s_off), n, H, W, _ptr(run_off), _ptr(runs), st), "emia_coco_counts_fill")
    LAUNCHES["count"] += 2
    iset, plan = _rle_decode(run_off, runs[:R], H, W)
    code = status[:n].cpu().numpy()
    code = np.where((code == 0) & (plan != 0), 5, code).astype(np.int32)     # valid counts: only the area limit remains
    return iset, code


def coco_decode(strings, H, W):
    """The compressed-RLE "counts" strings (str or bytes) of n H x W masks -> InstanceSet, bit for bit the tables rle_decode gives for
    the same masks (tight bbox crops).  Raises EmiaError naming the first rejected string (0-based) and why."""
    raw = [s.encode("utf-8") if isinstance(s, str) else bytes(s) for s in strings]
    off = np.concatenate([[0], np.cumsum([len(b) for b in raw])]).astype(np.int64)
    iset, status = _coco_decode(b"".join(raw), off, H, W)
    bad = np.nonzero(status)[0]
    if len(bad):
        k = int(bad[0])
        raise _lib.EmiaError(f"coco_decode: string {k}: {COCO_STATUS[int(status[k])]}")
    return iset


def measurements_csv_text(iset, file_name, psum, class_idx, class_fields, contrast=None, shape=None):
    """The rows of measurements_results.csv for the measured records of `iset` (after measure()), in record order: byte for byte
    what csv.writer writes for the rows of inference.measure_masks, UTF-8, "\\r\\n" line ends.  Instance i gets Instance_ID
    `<file_name>_<i + 1>` and the (Class, Class_Name) values class_fields[class_idx[i]]; psum is the Detected scale bar value;
    contrast: float64 [n, 3] d10 / d50 / d90 per instance (NaN: None), or None for empty contrast fields; shape: None, or the
    float64 [n_records, SHAPE_FIELDS] device tensor of shape_descriptors(iset), whose values follow "File name" as Python floats.
    String values are rendered once on the host (csv_field), numbers on the device; one host synchronisation to size the text,
    one D2H copy."""
    lib = _lib.load()
    dev = iset.device
    assert iset.records is not None, "run measure() first"
    R, n = int(iset.n_records), iset.n
    class_idx = np.asarray(class_idx, np.int64).reshape(-1)
    if len(class_idx) != n or (n and (class_idx.min() < 0 or class_idx.max() >= len(class_fields))):
        raise ValueError(f"measurements_csv_text: class_idx needs {n} indices into the {len(class_fields)} class_fields")
    if R == 0:
        return b""
    strs = _row_strings(file_name, psum, class_fields)
    sdata, soff = _strings_to_device(strs, dev)
    cidx = torch.as_tensor(class_idx.astype(np.int32), device=dev)
    con = None
    if contrast is not None:
        con = torch.as_tensor(np.asarray(contrast, np.float64).reshape(n, 3), device=dev).contiguous()
    if shape is not None:
        if not (isinstance(shape, torch.Tensor) and shape.device == iset.records.device and shape.dtype == torch.float64 and
                tuple(shape.shape) == (R, SHAPE_FIELDS)):
            raise ValueError(f"measurements_csv_text: shape must be a float64 [{R}, {SHAPE_FIELDS}] tensor beside the records")
        shape = shape.contiguous()
    records, rec_inst = iset.records.contiguous(), iset.rec_inst.contiguous()
    row_off = torch.empty(R + 1, dtype=torch.int64, device=dev)
    st = _stream()
    args = (_ptr(records), _ptr(rec_inst), R, _ptr(cidx), _ptr(con), _ptr(shape), _ptr(sdata), _ptr(soff), len(strs))
    with _stage("csv_measure_count"):
        _lib.check(lib.emia_csv_measure_shape_count(*args, _ptr(row_off), st), "emia_csv_measure_shape_count")
    with _stage("csv_measure_scan"):
        exclusive_scan_(row_off)
    nbytes = buffer_len(row_off[R:], R)
    text = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
    with _stage("csv_measure_write"):
        _lib.check(lib.emia_csv_measure_shape_write(*args, _ptr(row_off), _ptr(text), st), "emia_csv_measure_shape_write")
    LAUNCHES["count"] += 2
    with _stage("csv_measure_d2h"):
        return _text_to_host(text, nbytes)


def gray_hist(iset, image):
    """int32 [n,256] grey-level histograms of the image pixels under every instance (image: H x W x 3 BGR or H x W uint8)."""
    lib = _lib.load()
    img = torch.as_tensor(np.ascontiguousarray(image), device=iset.device)
    assert img.dtype == torch.uint8 and img.shape[0] == iset.H and img.shape[1] == iset.W
    ch = 1 if img.dim() == 2 else int(img.shape[2])
    out = torch.empty((max(iset.n, 1), 256), dtype=torch.int32, device=iset.device)
    _lib.check(lib.emia_gray_hist(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), iset.n, _ptr(img), iset.H, iset.W, ch, _ptr(out),
                                  _stream()), "emia_gray_hist")
    LAUNCHES["count"] += 1
    return out[:iset.n]


def image_gray_hist(image, device=None):
    """int64 [256] grey-level histogram of an H x W x 3 (BGR) or H x W uint8 image (host array or device tensor)."""
    lib = _lib.load()
    dev = _need_cuda(device)
    img = torch.as_tensor(np.ascontiguousarray(image) if isinstance(image, np.ndarray) else image, device=dev).contiguous()
    assert img.dtype == torch.uint8 and img.dim() in (2, 3)
    ch = 1 if img.dim() == 2 else int(img.shape[2])
    out = torch.empty(256, dtype=torch.int64, device=dev)
    _lib.check(lib.emia_image_gray_hist(_ptr(img), int(img.shape[0]), int(img.shape[1]), ch, _ptr(out), _stream()), "emia_image_gray_hist")
    LAUNCHES["count"] += 1
    return out


def moments01(iset):
    """(m00, m10, m01) int64 [n,3]: cv2.moments of the 0/1 mask (src/functions/inference.py:1101-1104)."""
    lib = _lib.load()
    out = torch.empty((max(iset.n, 1), 3), dtype=torch.int64, device=iset.device)
    _lib.check(lib.emia_moments01(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), iset.n, _ptr(out), _stream()), "emia_moments01")
    LAUNCHES["count"] += 1
    return out[:iset.n]


NB_VALUES = 4      # EMIA_NB_F: centroid x, centroid y, nearest-neighbour distance, edge distance
NB_INTS = 6        # EMIA_NB_I: listed, nearest neighbour, closest neighbour, touching, agglomerate, agglomerate size


@dataclass
class NeighbourResult:
    """Relations of the instances of one image (neighbours()): values float64 [n, NB_VALUES] (centroid x / y in frame pixels, the
    nearest-neighbour and edge distances scaled by um_pix; NaN without a candidate) and ints int32 [n, NB_INTS] (listed, nearest and
    closest neighbour index or -1, touching count, agglomerate index (-1: not listed), agglomerate size), device tensors."""
    values: torch.Tensor
    ints: torch.Tensor

    @property
    def listed(self):
        return self.ints[:, 0] != 0


def neighbour_cell_size(H, W, n):
    """Grid cell side of neighbours(): about one instance per cell (frame area over instance count), at least 16 pixels."""
    return max(16, int(math.ceil(math.sqrt(H * W / max(n, 1)))))


def neighbours(iset, class_idx, um_pix=1.0):
    """Nearest neighbour, closest neighbour, edge distance, touching count and agglomerate of every instance of one image after
    measure() (definitions: oracle/neighbours.py).  Listed instances are those with a measured record; candidates are listed
    instances with the same class_idx (an index per instance into the class table of measurements_csv_text).  One host
    synchronisation sizes the grid's cell lists (buffer_len)."""
    lib = _lib.load()
    dev = iset.device
    assert iset.records is not None, "run measure() first"
    n = iset.n
    cidx = np.asarray(class_idx, np.int64).reshape(-1)
    if len(cidx) != n or (n and cidx.min() < 0):
        raise ValueError(f"neighbours: class_idx needs {n} non-negative class-table indices")
    values = torch.empty((max(n, 1), NB_VALUES), dtype=torch.float64, device=dev)
    ints = torch.empty((max(n, 1), NB_INTS), dtype=torch.int32, device=dev)
    if n == 0:
        return NeighbourResult(values[:0], ints[:0])
    n_class = int(cidx.max()) + 1
    cs = neighbour_cell_size(iset.H, iset.W, n)
    ncells = n_class * ((iset.W + cs - 1) // cs) * ((iset.H + cs - 1) // cs)
    cls = torch.as_tensor(cidx.astype(np.int32), device=dev)
    with _stage("nb_moments"):
        mom = moments01(iset)
    cell_off = torch.empty(ncells + 1, dtype=torch.int64, device=dev)
    bbox = iset.bbox.contiguous()
    st = _stream()
    with _stage("nb_plan"):
        _lib.check(lib.emia_neighbour_plan(_ptr(iset.records.contiguous()), _ptr(iset.cont_off), _ptr(bbox), _ptr(mom), _ptr(cls), n,
                                           n_class, iset.H, iset.W, cs, _ptr(values), _ptr(ints), _ptr(cell_off), st),
                   "emia_neighbour_plan")
    with _stage("nb_scan"):
        exclusive_scan_(cell_off)
    n_ent = buffer_len(cell_off[ncells:], ncells)
    ent = torch.empty(max(n_ent, 1), dtype=torch.int32, device=dev)
    work = torch.empty(n + ncells, dtype=torch.int32, device=dev)
    with _stage("nb_search"):
        _lib.check(lib.emia_neighbour_search(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(bbox), _ptr(cls), n, n_class,
                                             iset.H, iset.W, cs, _ptr(cell_off), _ptr(ent), float(um_pix), _ptr(values), _ptr(ints),
                                             _ptr(work), st), "emia_neighbour_search")
    LAUNCHES["count"] += 5
    return NeighbourResult(values[:n], ints[:n])


def neighbours_csv_text(iset, nb, file_name, psum, class_idx, class_fields):
    """The rows of neighbours_results.csv for the listed instances of `iset` (nb = neighbours(iset, class_idx, ...)), in instance
    order: byte for byte what csv.writer writes for inference.neighbour_rows, UTF-8, "\\r\\n" line ends.  Instance_ID, Class,
    Class_Name, Detected scale bar and File name as in measurements_csv_text.  One host synchronisation to size the text, one D2H
    copy."""
    lib = _lib.load()
    dev = iset.device
    n = iset.n
    class_idx = np.asarray(class_idx, np.int64).reshape(-1)
    if len(class_idx) != n or (n and (class_idx.min() < 0 or class_idx.max() >= len(class_fields))):
        raise ValueError(f"neighbours_csv_text: class_idx needs {n} indices into the {len(class_fields)} class_fields")
    if tuple(nb.values.shape) != (n, NB_VALUES) or tuple(nb.ints.shape) != (n, NB_INTS):
        raise ValueError(f"neighbours_csv_text: nb must be the neighbours() result of this {n}-instance set")
    if n == 0:
        return b""
    strs = _row_strings(file_name, psum, class_fields)
    sdata, soff = _strings_to_device(strs, dev)
    cidx = torch.as_tensor(class_idx.astype(np.int32), device=dev)
    values, ints = nb.values.contiguous(), nb.ints.contiguous()
    row_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    st = _stream()
    args = (_ptr(values), _ptr(ints), n, _ptr(cidx), _ptr(sdata), _ptr(soff), len(strs))
    with _stage("csv_nb_count"):
        _lib.check(lib.emia_csv_neighbour_count(*args, _ptr(row_off), st), "emia_csv_neighbour_count")
    with _stage("csv_nb_scan"):
        exclusive_scan_(row_off)
    nbytes = buffer_len(row_off[n:], n)
    text = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
    with _stage("csv_nb_write"):
        _lib.check(lib.emia_csv_neighbour_write(*args, _ptr(row_off), _ptr(text), st), "emia_csv_neighbour_write")
    LAUNCHES["count"] += 2
    with _stage("csv_nb_d2h"):
        return _text_to_host(text, nbytes)


MOMENT_NAMES = ("m00", "m10", "m01", "m20", "m11", "m02", "m30", "m21", "m12", "m03", "mu20", "mu11", "mu02", "mu30", "mu21", "mu12",
                "mu03", "nu20", "nu11", "nu02", "nu30", "nu21", "nu12", "nu03")


def moments(iset):
    """float64 [n, 24]: every entry of cv2.moments(mask.astype(np.uint8)) (src/functions/inference.py:1101) in MOMENT_NAMES order —
    raw moments exact, central / normalised ones with OpenCV's arithmetic."""
    lib = _lib.load()
    out = torch.empty((max(iset.n, 1), len(MOMENT_NAMES)), dtype=torch.float64, device=iset.device)
    _lib.check(lib.emia_moments(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), iset.n, _ptr(out), _stream()), "emia_moments")
    LAUNCHES["count"] += 1
    return out[:iset.n]


def color_sums(iset, image):
    """int64 [n, 4]: (sum B, sum G, sum R, pixel count) of the BGR image pixels under every instance."""
    lib = _lib.load()
    img = torch.as_tensor(np.ascontiguousarray(image) if isinstance(image, np.ndarray) else image, device=iset.device).contiguous()
    assert img.dtype == torch.uint8 and img.dim() == 3 and img.shape[2] == 3 and img.shape[0] == iset.H and img.shape[1] == iset.W
    out = torch.empty((max(iset.n, 1), 4), dtype=torch.int64, device=iset.device)
    _lib.check(lib.emia_color_sums(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), iset.n, _ptr(img), iset.H, iset.W, _ptr(out),
                                   _stream()), "emia_color_sums")
    LAUNCHES["count"] += 1
    return out[:iset.n]


# ---- row f3: scale-bar line detection (src/utils/scalebar_ocr.py:140-249), batched -------------------------------------------
def hough_tables(W, H, rho=1.0, theta=np.pi / 180):
    """(trig float32 [2 * numangle], numangle, numrho) exactly as cv2.HoughLinesP builds them (float rho / theta parameters,
    computeNumangle(0, pi, theta), (float)(cos((double)n * theta) / rho))."""
    rho32, theta32 = np.float32(rho), np.float32(theta)
    th = float(theta32)
    numangle = int(math.floor(math.pi / th)) + 1
    if numangle > 1 and abs(math.pi - (numangle - 1) * th) < th / 2:
        numangle -= 1
    irho = float(np.float32(1) / rho32)
    numrho = int(np.rint(np.float32((W + H) * 2 + 1) / rho32))
    trig = np.empty(2 * numangle, np.float32)
    for a in range(numangle):
        trig[2 * a] = np.float32(math.cos(a * th) * irho)
        trig[2 * a + 1] = np.float32(math.sin(a * th) * irho)
    return trig, numangle, numrho


def scalebar_edges(images, roi, low=50, high=150):
    """images: uint8 [B,H,W,3] (BGR) or [B,H,W] (host array or device tensor); roi = (x0, y0, x1, y1) inside the images.
    Returns (gray, edges) uint8 device tensors [B, y1-y0, x1-x0]: cv2.cvtColor(BGR2GRAY) and cv2.Canny(gray, low, high)."""
    lib = _lib.load()
    dev = images.device if isinstance(images, torch.Tensor) and images.is_cuda else _need_cuda(None)
    img = torch.as_tensor(np.ascontiguousarray(images) if isinstance(images, np.ndarray) else images, device=dev).contiguous()
    assert img.dtype == torch.uint8 and img.dim() in (3, 4)
    B, H, W = (int(v) for v in img.shape[:3])
    ch = 1 if img.dim() == 3 else int(img.shape[3])
    x0, y0, x1, y1 = (int(v) for v in roi)
    rw, rh = x1 - x0, y1 - y0
    gray = torch.empty((B, max(rh, 0), max(rw, 0)), dtype=torch.uint8, device=dev)
    edges = torch.empty_like(gray)
    _lib.check(lib.emia_scalebar_edges(_ptr(img), B, H, W, ch, x0, y0, rw, rh, int(math.floor(low)), int(math.floor(high)), _ptr(gray),
                                       _ptr(edges), _stream()), "emia_scalebar_edges")
    LAUNCHES["count"] += 3
    return gray, edges


def hough_lines_p(edges, rho=1.0, theta=np.pi / 180, threshold=50, min_line_length=20, max_line_gap=10, max_lines=1024):
    """cv2.HoughLinesP on every image of edges [B,H,W] (uint8 device tensor): (lines int32 [B,max_lines,4], n_lines int32 [B]),
    lines in OpenCV's output order."""
    lib = _lib.load()
    assert edges.is_cuda and edges.dtype == torch.uint8 and edges.dim() == 3 and edges.is_contiguous()
    B, H, W = (int(v) for v in edges.shape)
    dev = edges.device
    trig, numangle, numrho = hough_tables(W, H, rho, theta)
    trig_t = torch.as_tensor(trig, device=dev)
    lines = torch.zeros((B, max_lines, 4), dtype=torch.int32, device=dev)
    n_lines = torch.zeros(max(B, 1), dtype=torch.int32, device=dev)
    nbytes = int(lib.emia_hough_workspace_bytes(B, H, W, numangle, numrho))
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
    _lib.check(lib.emia_hough_lines_p(_ptr(edges), B, H, W, _ptr(trig_t), numangle, numrho, int(threshold), int(min_line_length),
                                      int(max_line_gap), int(max_lines), _ptr(lines), _ptr(n_lines), _ptr(ws), nbytes, _stream()),
               "emia_hough_lines_p")
    LAUNCHES["count"] += 1
    return lines, n_lines[:B]


def line_means(gray, lines, n_lines):
    """int64 [B,max_lines,2] = (sum of gray, pixel count) under cv2.line(mask, p1, p2, 255, 2) of every line; the reference's
    cv2.mean(gray_roi, mask=line_mask)[0] is sum * (1.0 / count)."""
    lib = _lib.load()
    assert gray.is_cuda and gray.dtype == torch.uint8 and gray.dim() == 3 and gray.is_contiguous()
    B, H, W = (int(v) for v in gray.shape)
    out = torch.zeros((B, int(lines.shape[1]), 2), dtype=torch.int64, device=gray.device)
    _lib.check(lib.emia_line_mean(_ptr(gray), B, H, W, _ptr(lines), _ptr(n_lines), int(lines.shape[1]), _ptr(out), _stream()),
               "emia_line_mean")
    LAUNCHES["count"] += 1
    return out


_rule_cache = {}


def overlap_rules(iset, groups, rules):
    """filter_by_overlap_rules (src/utils/spatial_constraints.py:192).  rules: {class: {allow_overlap, max_iou_threshold}}."""
    lib = _lib.load()
    if not rules:
        return groups
    ncls = max(int(c) for c in rules) + 1
    active = np.zeros(ncls, np.int32)
    max_iou = np.zeros(ncls, np.float64)
    for c, r in rules.items():
        allow = r.get('allow_overlap', True)
        mi = r.get('max_iou_threshold', 0.5)
        if allow and mi >= 0.9:
            continue
        active[int(c)] = 1
        max_iou[int(c)] = mi
    dev = iset.device
    key = (active.tobytes(), max_iou.tobytes(), str(dev))
    cached = _rule_cache.get(key)
    if cached is None:       # the upload from pageable memory synchronises: do it once per rule set
        cached = (torch.as_tensor(active, device=dev), torch.as_tensor(max_iou, device=dev))
        _rule_cache[key] = cached
    act_t, mi_t = cached
    ws, nb = _workspace(groups, dev)
    out = _new_groups_like(groups)
    with _stage("k4_overlap_rules"):
      _lib.check(lib.emia_overlap_rules(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(iset.bbox), _ptr(iset.area),
                                      _ptr(iset.scores), _ptr(iset.classes), _ptr(groups.cap_off), groups.G, groups.total_cap, groups.fused_cap,
                                      _ptr(groups.length), _ptr(groups.idx), _ptr(act_t), _ptr(mi_t), ncls, _ptr(out.length),
                                      _ptr(out.idx), _ptr(ws), nb, _stream()), "emia_overlap_rules")
    LAUNCHES["count"] += 6
    return out


def containment_rules(iset, groups, rules, threshold=0.95):
    """filter_by_containment_rules (src/utils/spatial_constraints.py:280).  rules: {child_class: parent_class} (ordered)."""
    lib = _lib.load()
    if not rules:
        return groups
    child = np.asarray([int(c) for c in rules.keys()], np.int32)
    parent = np.asarray([int(p) for p in rules.values()], np.int32)
    ws, nb = _workspace(groups, iset.device)
    out = _new_groups_like(groups)
    with _stage("k4_containment"):
      _lib.check(lib.emia_containment_rules(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(iset.bbox), _ptr(iset.area),
                                          _ptr(iset.classes), _ptr(groups.cap_off), groups.G, groups.total_cap, groups.fused_cap, _ptr(groups.length),
                                          _ptr(groups.idx), child.ctypes.data, parent.ctypes.data, len(child), float(threshold),
                                          _ptr(out.length), _ptr(out.idx), _ptr(ws), nb, _stream()), "emia_containment_rules")
    LAUNCHES["count"] += 1 + 2 * len(child)
    return out


def apply_spatial_constraints(iset, groups, rules):
    """apply_spatial_constraints (src/utils/spatial_constraints.py:401) with an explicit rule dict."""
    if not rules or not rules.get('enabled', False):
        return groups
    g = overlap_rules(iset, groups, rules.get('overlap_rules', {}))
    return containment_rules(iset, g, rules.get('containment_rules', {}), rules.get('containment_threshold', 0.95))


def pair_counts(iset, pa, pb):
    """(intersection, area_a, area_b) int64 [k,3] for explicit instance pairs."""
    lib = _lib.load()
    dev = iset.device
    pa = torch.as_tensor(pa, dtype=torch.int32, device=dev).contiguous()
    pb = torch.as_tensor(pb, dtype=torch.int32, device=dev).contiguous()
    out = torch.empty((pa.numel(), 3), dtype=torch.int64, device=dev)
    _lib.check(lib.emia_pair_counts(_ptr(iset.crops), _ptr(iset.meta), _ptr(iset.crop_off), _ptr(iset.area), _ptr(pa), _ptr(pb),
                                    pa.numel(), _ptr(out), _stream()), "emia_pair_counts")
    LAUNCHES["count"] += 1
    return out


def run_tiles(probs, boxes, scores, classes, tile_offsets, H, W, um_pix=0.5, rules=None, dedup_iou=0.7, frames=None,
              variant=2, scale_x=1.0, scale_y=1.0):
    """The fused hot path over many tiles at once (BASELINE configs 2 and 5): paste -> external contours ->
    deduplicate_masks_smart -> spatial constraints -> morphometry of the survivors (the order of the reference:
    src/functions/inference.py:859, :868, :1148).  Everything stays on the device.
    Returns (InstanceSet, Groups of kept instances, Measurements of the kept instances)."""
    iset = paste(probs, boxes, H, W, scores=scores, classes=classes, scale_x=scale_x, scale_y=scale_y, frames=frames,
                 variant=variant)
    kept, meas, _ = _post_paste(iset, groups_from_offsets(tile_offsets, iset.device), um_pix, rules, dedup_iou)
    return iset, kept, meas


def _post_paste(iset, groups, um_pix, rules, dedup_iou, marks=None, pt_cap=None, arena=None):
    """trace -> deduplicate_masks_smart -> spatial constraints -> morphometry of the survivors.  Without an arena the sizes
    are read back and a contour slab that overflowed is traced again with exact sizes.  Returns (kept, meas, retraced)."""
    single_pass = True
    while True:
        trace(iset, single_pass=single_pass, marks=marks, arena=arena, pt_cap=pt_cap)
        kept = dedup_smart(iset, groups, iou_threshold=dedup_iou)
        kept = apply_spatial_constraints(iset, kept, rules)
        meas = measure_list(iset, kept, um_pix=um_pix, arena=arena)
        if meas is not None:
            return kept, meas, not single_pass
        single_pass = False      # a slab overflowed: follow the borders again with exact sizes


class TilePipeline:
    """The fused hot path over a shard of tiles, software-pipelined over tile batches on three CUDA streams:

        copy  : (host inputs only) H2D of batch b's 28x28 probabilities from pinned memory
        paste : K1 of batch b (HBM-write bound)
        post  : contours -> de-dup -> spatial constraints -> morphometry of batch b-1 (latency bound) [+ D2H of its results]

    so the latency-bound kernels run in the shadow of the bandwidth-bound paste (and, end to end, of the PCIe copy).
    The first run of a batch count is exact: the plan (crop geometry, vertex capacities) of the WHOLE shard is computed
    first, with one small device->host read of the per-batch totals; each batch then needs one more read (record/scratch
    totals) on the post stream only.  Its totals are fitted into an Arena of that batch count (margin hint_margin), and
    later runs are enqueued sync-free against those capacities (see aborted()).
    Batches see slices of shard-wide arrays; list indices stay shard-global."""

    def __init__(self, H, W, um_pix=1.0, rules=None, dedup_iou=0.7, frames=None, variant=2, batches=8, paste_ctas_per_sm=0,
                 device=None, sync_free=True, hint_margin=1.05):
        self.H, self.W, self.um_pix, self.rules, self.dedup_iou = H, W, um_pix, rules, dedup_iou
        self.frames, self.variant, self.batches, self.paste_ctas = frames, variant, batches, paste_ctas_per_sm
        self.dev = _need_cuda(device)
        lo, hi = torch.cuda.Stream.priority_range()
        self.s_copy = torch.cuda.Stream(device=self.dev)
        self.s_paste = torch.cuda.Stream(device=self.dev, priority=lo)
        self.s_post = torch.cuda.Stream(device=self.dev, priority=hi)
        self._groups_cache = {}
        self._pinned = {}
        self.k1_events = []
        # capacities per batch count, fitted to an exact run: the next run of that count is enqueued without reading anything back
        self.sync_free, self.hint_margin = sync_free, hint_margin
        self._arenas, self._ib_cache, self._abort, self._last_batches = {}, {}, None, None
        self.exact_runs = 0      # runs that read sizes back (host synchronisations); the others are enqueued sync-free

    def _groups(self, offs):
        key = offs.tobytes()
        g = self._groups_cache.get(key)
        if g is None:
            if len(self._groups_cache) > 1024:
                self._groups_cache.clear()
            g = groups_from_offsets(offs, self.dev)
            self._groups_cache[key] = g
        # length / idx are never written by the K4 stages (they produce new lists), so the cached identity lists are reusable
        return g

    def run(self, probs, boxes, scores, classes, tile_offsets, to_host=False, time_k1=False):
        """probs [n,28,28] f32, boxes [n,4] f32, scores [n] f32, classes [n] i32: device tensors, or pinned HOST tensors (then
        the copies are part of the pipeline).  tile_offsets: host int array [T+1].
        Returns a list over batches of dicts {tiles: (t0, t1), iset, kept, meas[, host: {...}]}."""
        dev = self.dev
        main = torch.cuda.current_stream(dev)
        offs = np.asarray(tile_offsets, dtype=np.int64)
        T = len(offs) - 1
        n = int(offs[-1])
        B = max(1, min(self.batches, T))
        tb = np.unique(np.linspace(0, T, B + 1).round().astype(np.int64))
        B = len(tb) - 1
        ib = offs[tb]
        host_in = not probs.is_cuda
        ev_copy = []
        if host_in:
            d_boxes = boxes.to(dev, non_blocking=True); d_scores = scores.to(dev, non_blocking=True)
            d_classes = classes.to(dev, non_blocking=True)
            d_probs = torch.empty(tuple(probs.shape), dtype=probs.dtype, device=dev)
            self.s_copy.wait_stream(main)
            with torch.cuda.stream(self.s_copy):
                for b in range(B):
                    d_probs[ib[b]:ib[b + 1]].copy_(probs[ib[b]:ib[b + 1]], non_blocking=True)
                    e = torch.cuda.Event(); e.record(self.s_copy); ev_copy.append(e)
        else:
            d_probs, d_boxes, d_scores, d_classes = probs, boxes, scores, classes
        # ---- shard-wide plan: crop geometry + vertex capacities, one read of the per-batch totals
        lib = _lib.load()
        meta, crop_off = paste_plan(d_boxes, self.H, self.W)
        # Sizes: read back once (the first run of this batch count, or after a guard tripped); afterwards the buffers take the
        # arena's CAPACITIES (fitted to that exact run, independent of the exact per-tile instance counts) and the real totals
        # are only CHECKED on the device: the whole step is enqueued without a single host synchronisation, the abort flag is
        # looked at when the results are consumed (aborted()).  A tripped guard makes the paste / trace / measure kernels write
        # nothing; the caller re-runs, which takes the exact-size path again and fits new capacities.
        arena = self._arenas.get(B) if self.sync_free else None
        ikey = offs.tobytes()
        ib_t = self._ib_cache.get(ikey)           # batch boundaries as a device array (an upload, not a size read-back)
        if ib_t is None:
            if len(self._ib_cache) > 256:
                self._ib_cache.clear()
            ib_t = torch.as_tensor(ib, device=dev)
            self._ib_cache[ikey] = ib_t
        cap_off = None
        if arena is None:
            self.exact_runs += 1
            abort = torch.zeros(1, dtype=torch.int32, device=dev)      # never raised: callers OR every run's flag
            cap_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
            _lib.check(lib.emia_contour_trace_plan(_ptr(meta), n, _ptr(cap_off), _stream()), "emia_contour_trace_plan")
            exclusive_scan_(cap_off)
            LAUNCHES["count"] += 1
            bounds = torch.stack([crop_off[ib_t], cap_off[ib_t]]).cpu().numpy()
            total_words = int(bounds[0, -1])
            pt_caps = [int(bounds[1, b + 1] - bounds[1, b]) for b in range(B)]
        else:
            abort, _ = arena.begin()
            total_words = buffer_len(crop_off[n:], n, arena, "k1.crops")
            pt_caps = [None] * B
        crops = torch.empty(max(total_words, 1), dtype=torch.int32, device=dev)
        marks = torch.empty(max(2 * total_words, 1), dtype=torch.int32, device=dev)
        # under CUDA-graph capture with device inputs (one batch: nothing to overlap) everything runs on the caller's stream: the
        # captured step is a single chain of kernel nodes
        capturing = torch.cuda.is_current_stream_capturing()
        single = capturing and not host_in          # host inputs keep the three-stream pipeline: captured as parallel graph branches
        s_paste = main if single else self.s_paste
        s_post = main if single else self.s_post
        if capturing:
            assert arena is not None, "capture needs the sync-free path: run the shard once eagerly first"
            time_k1 = False
        s_paste.wait_stream(main); s_post.wait_stream(main)
        isets, ev_paste = [], []
        self.k1_events = []
        with torch.cuda.stream(s_paste):
            for b in range(B):
                i0, i1 = int(ib[b]), int(ib[b + 1])
                if host_in:
                    s_paste.wait_event(ev_copy[b])
                if time_k1:
                    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record(s_paste)
                it = paste(d_probs[i0:i1], d_boxes[i0:i1], self.H, self.W, scores=d_scores[i0:i1], classes=d_classes[i0:i1],
                           frames=self.frames, variant=self.variant, crops_out=crops,
                           plan=(meta[i0:i1], crop_off[i0:i1 + 1], total_words), ctas_per_sm=self.paste_ctas,
                           abort=arena.abort if arena is not None else None)
                if time_k1:
                    e1.record(s_paste); self.k1_events.append((e0, e1))
                e = torch.cuda.Event(); e.record(s_paste); ev_paste.append(e)
                isets.append(it)
        out, retraced = [], False
        with torch.cuda.stream(s_post):
            for b in range(B):
                it = isets[b]
                s_post.wait_event(ev_paste[b])
                groups = self._groups(offs[tb[b]:tb[b + 1] + 1] - ib[b])
                kept, meas, again = _post_paste(it, groups, self.um_pix, self.rules, self.dedup_iou, marks=marks, pt_cap=pt_caps[b],
                                                arena=arena)
                retraced |= again
                res = {"tiles": (int(tb[b]), int(tb[b + 1])), "inst0": int(ib[b]), "iset": it, "kept": kept, "meas": meas}
                if to_host:
                    res["host"] = {k: self._pinned_like(b, k, v).copy_(v, non_blocking=True)
                                   for k, v in (("records", meas.records), ("rec_inst", meas.rec_inst), ("rec_off", meas.rec_off),
                                                ("kept_len", kept.length), ("kept_idx", kept.idx))}
                out.append(res)
        main.wait_stream(s_post); main.wait_stream(s_paste)
        if host_in:
            main.wait_stream(self.s_copy)
        self._keep = (crops, marks, meta, crop_off, cap_off, d_probs)
        self._abort = abort
        if arena is None and self.sync_free and not retraced:
            arena = Arena(dev, margin=self.hint_margin)
            arena.fit("k1.crops", total_words)
            arena.fit("k5.pts", max(pt_caps))
            arena.fit("k5.records", max(r["meas"].totals[0] for r in out))
            arena.fit("k5.scratch", max(r["meas"].totals[1] for r in out))
            self._arenas[B] = arena
        self._last_batches = B
        return out

    def aborted(self):
        """True when a capacity guard (or a contour slab) tripped in the last sync-free run(): its results are invalid, the arena
        of that batch count is dropped and the caller runs again (exact-size path).  One host synchronisation."""
        if self._abort is None or not bool(self._abort.item()):
            return False
        self._arenas.pop(self._last_batches, None)      # the next run re-measures and fits new capacities
        return True

    def _pinned_like(self, b, name, t):
        """Persistent pinned result buffers (one per batch and result array, grown on demand): page-locking memory inside
        the pipeline would serialise it.  The views handed out are overwritten by the next run()."""
        key = (b, name)
        buf = self._pinned.get(key)
        if buf is None or buf.numel() < t.numel() or buf.dtype != t.dtype:
            buf = torch.empty(max(int(t.numel() * 1.25), 16), dtype=t.dtype, pin_memory=True)
            self._pinned[key] = buf
        return buf[:t.numel()].view(t.shape)

    def k1_ms(self):
        """Sum over batches of the CUDA-event duration of the K1 launches of the last run(time_k1=True) (after a synchronize)."""
        return float(sum(a.elapsed_time(b) for a, b in self.k1_events))
