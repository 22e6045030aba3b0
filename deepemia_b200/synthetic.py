"""Synthetic micrograph instances (SURVEY.md §8d): star-polygon particles as full-frame masks or as Mask R-CNN head
outputs (28x28 probability map + box).  Host-side numpy/OpenCV; used by tests, bench.py and the golden generator."""
import cv2
import numpy as np

MASK_SIDE = 28


def star_polygon(rng, cx, cy, r):
    k = int(rng.integers(5, 13))
    ang = np.sort(rng.uniform(0, 2 * np.pi, k))
    rad = r * rng.uniform(0.6, 1.0, k)
    return np.stack([cx + rad * np.cos(ang), cy + rad * np.sin(ang)], 1)


def particle_field(rng, n, H, W, rmin=8.0, rmax=30.0, margin=40):
    """n star polygons (float vertices) with centres uniform inside the margin."""
    polys = []
    for _ in range(n):
        r = rng.uniform(rmin, rmax)
        cx = rng.uniform(margin, W - margin)
        cy = rng.uniform(margin, H - margin)
        polys.append(star_polygon(rng, cx, cy, r))
    return polys


def masks_from_polys(polys, H, W):
    out = []
    for p in polys:
        m = np.zeros((H, W), np.uint8)
        cv2.fillPoly(m, [np.round(p).astype(np.int32)], 1)
        out.append(m)
    return out


def head_from_poly(rng, poly):
    """(prob 28x28 float32 fp16-representable, box xyxy float32) for one particle."""
    x0, y0 = poly.min(0) - rng.uniform(0, 2, 2)
    x1, y1 = poly.max(0) + rng.uniform(0, 2, 2)
    sx, sy = MASK_SIDE / (x1 - x0), MASK_SIDE / (y1 - y0)
    q = np.stack([(poly[:, 0] - x0) * sx, (poly[:, 1] - y0) * sy], 1)
    m = np.zeros((MASK_SIDE, MASK_SIDE), np.float32)
    cv2.fillPoly(m, [np.round(q * 16).astype(np.int32)], 1.0, lineType=cv2.LINE_AA, shift=4)
    m = cv2.GaussianBlur(m, (0, 0), 1.0)
    m = np.clip(m, 0, 1).astype(np.float16).astype(np.float32)
    return m, np.array([x0, y0, x1, y1], np.float32)


def distinct_scores(rng, n, lo=0.05, hi=1.0):
    s = rng.uniform(lo, hi, n).astype(np.float32)
    while len(np.unique(s)) != n:
        s = rng.uniform(lo, hi, n).astype(np.float32)
    return s


def synthetic_heads(seed, n, H, W, duplicate_frac=0.0, **kw):
    """n head outputs for one H x W tile: probs (n,28,28) f32, boxes (n,4) f32, scores (n,) f32 distinct, classes (n,) i32.
    duplicate_frac > 0 re-detects that fraction of particles with a small box jitter (work for the de-dup step)."""
    rng = np.random.default_rng(seed)
    n_base = max(1, int(round(n / (1.0 + duplicate_frac))))
    polys = particle_field(rng, n_base, H, W, **kw)
    while len(polys) < n:
        src = polys[int(rng.integers(0, n_base))]
        polys.append(src + rng.uniform(-1.5, 1.5, 2))
    probs = np.zeros((n, MASK_SIDE, MASK_SIDE), np.float32)
    boxes = np.zeros((n, 4), np.float32)
    for i, p in enumerate(polys):
        probs[i], boxes[i] = head_from_poly(rng, p)
    scores = distinct_scores(rng, n)
    classes = (rng.random(n) < 0.5).astype(np.int32)
    return probs, boxes, scores, classes


# spatial rules of config/datasets/polyhipes_tommy.yaml:41-58 (class 1 must lie inside class 0; max IoU 0.30 / 0.50)
POLYHIPES_RULES = {
    'enabled': True,
    'containment_rules': {1: 0},
    'containment_threshold': 0.95,
    'overlap_rules': {0: {'allow_overlap': False, 'allow_touch': True, 'max_iou_threshold': 0.30},
                      1: {'allow_overlap': False, 'allow_touch': True, 'max_iou_threshold': 0.50}},
}


class FakeHeadPredictor:
    """A deterministic stand-in for the Mask R-CNN heads (Detectron2 is absent; SURVEY §8b): the head outputs of an image are a
    pure function of the image bytes (CRC32 -> seed), so the reference functions (fed the Detectron2-paste oracle of these heads)
    and the CUDA mirror (fed the raw heads) see the same detections for every image, tile, and rescaled image they derive.
    Test / golden-vector infrastructure."""

    def __init__(self, base_seed=0, n=28, duplicate_frac=0.35, rmin=5.0, rmax=15.0, margin=6, input_scale=1.0, zero_score=False):
        self.base_seed, self.n, self.dup, self.rmin, self.rmax, self.margin = base_seed, n, duplicate_frac, rmin, rmax, margin
        self.input_scale, self.zero_score = input_scale, zero_score
        self.calls = 0

    def raw_heads(self, image):
        """(probs [n,28,28] f32, boxes [n,4] f32 in model-input coordinates, scores, classes int64, (in_h, in_w))."""
        import zlib
        H, W = image.shape[:2]
        seed = (zlib.crc32(np.ascontiguousarray(image).tobytes()) ^ (self.base_seed * 2654435761)) & 0x7FFFFFFF
        n = self.n + int(seed % 7)
        r_hi = min(self.rmax, max(self.rmin + 1.0, min(H, W) / 6.0))
        probs, boxes, scores, classes = synthetic_heads(seed, n, H, W, duplicate_frac=self.dup, rmin=self.rmin, rmax=r_hi,
                                                        margin=self.margin)
        rng = np.random.default_rng(seed + 1)
        # a few degenerate / out-of-frame boxes exercise Boxes.nonempty() and the clipping
        boxes[0] = [W + 5.0, 3.0, W + 20.0, 18.0]
        boxes[1, 2] = boxes[1, 0]
        boxes[2] += np.array([-boxes[2, 0] - 4.0, 0.0, -boxes[2, 0] - 4.0, 0.0], np.float32)      # hangs over the left edge
        if self.zero_score:
            scores[3] = 0.0
        in_h, in_w = int(round(H * self.input_scale)), int(round(W * self.input_scale))
        boxes = boxes * np.array([in_w / W, in_h / H, in_w / W, in_h / H], np.float32)
        _ = rng
        self.calls += 1
        return probs, boxes.astype(np.float32), scores.astype(np.float32), classes.astype(np.int64), (in_h, in_w)

    def heads(self, image):
        """The pre-paste hook of deepemia_b200.functions.inference (CUDA tensors)."""
        import torch
        from .functions.inference import HeadOutputs
        probs, boxes, scores, classes, in_size = self.raw_heads(image)
        dev = torch.device("cuda", torch.cuda.current_device())
        t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev)
        return HeadOutputs(t(probs), t(boxes), t(scores), t(classes), in_size)


# =================================================================================================================
# BASELINE configs 3 and 4 as concrete synthetic inputs (SURVEY.md section 8d).  Host-side numpy; bench.py, tests.
# =================================================================================================================
def _tile_origins(h, w, tile_size, overlap_ratio):
    stride = int(tile_size * (1 - overlap_ratio))
    return [(x, y) for y in range(0, h, stride) for x in range(0, w, stride)]


def _make_distinct(sc):
    """float32 scores made pairwise distinct: ties are pushed up by single ulps in sorted order (order otherwise unchanged)."""
    sc = np.asarray(sc, np.float32).copy()
    o = np.argsort(sc, kind="stable")
    v = sc[o]
    for k in range(1, len(v)):
        if v[k] <= v[k - 1]:
            v[k] = np.nextafter(v[k - 1], np.float32(2.0))
    sc[o] = v
    return sc


def micrograph_heads(seed, h, w, n_particles, tile_size, overlap_ratio, upscale, cap=100, rmin=8.0, rmax=30.0):
    """Config 3: one particle field cut into tiles.  Every particle has ONE 28 x 28 probability map (so its re-detections in
    overlapping tiles and in the full-image pass are near-identical masks), a class and a base score.  A tile detects the
    particles whose centre lies inside it (at most `cap`, highest score first — Detectron2 returns its detections sorted by
    score and capped at DETECTIONS_PER_IMAGE); boxes are given in the UPSCALED tile's coordinates with a sub-pixel jitter and
    every detection gets its own distinct score.  The full-image pass sees the `cap` highest-scoring particles.
    Returns dict(full=(probs, boxes, scores, classes, unit_off), tiles=(...), tile_xy [T, 2], hw=(h, w))."""
    rng = np.random.default_rng(seed)
    polys = particle_field(rng, n_particles, h, w, rmin=rmin, rmax=rmax, margin=int(rmax) + 4)
    protos = np.zeros((n_particles, MASK_SIDE, MASK_SIDE), np.float32)
    pbox = np.zeros((n_particles, 4), np.float32)
    for i, p in enumerate(polys):
        protos[i], pbox[i] = head_from_poly(rng, p)
    base = rng.uniform(0.3, 0.95, n_particles)
    classes = (rng.random(n_particles) < 0.5).astype(np.int32)
    cx, cy = 0.5 * (pbox[:, 0] + pbox[:, 2]), 0.5 * (pbox[:, 1] + pbox[:, 3])
    origins = _tile_origins(h, w, tile_size, overlap_ratio)

    def detections(ids, ox, oy, s):
        k = len(ids)
        b = (pbox[ids] - np.array([ox, oy, ox, oy], np.float32)) * np.float32(s) + rng.uniform(-0.4, 0.4, (k, 4)).astype(np.float32)
        sc = (base[ids] + rng.uniform(-0.04, 0.04, k)).astype(np.float32)
        order = np.argsort(-sc, kind="stable")[:cap]
        return ids[order], b[order].astype(np.float32), sc[order]

    t_ids, t_boxes, t_scores, t_off = [], [], [], [0]
    for (x, y) in origins:
        inside = np.nonzero((cx >= x) & (cx < x + tile_size) & (cy >= y) & (cy < y + tile_size))[0]
        ids, b, sc = detections(inside, x, y, upscale)
        t_ids.append(ids); t_boxes.append(b); t_scores.append(sc); t_off.append(t_off[-1] + len(ids))
    f_ids, f_boxes, f_scores = detections(np.arange(n_particles), 0.0, 0.0, 1.0)
    # distinct scores over the whole micrograph (ties would make the reference's argsort order platform-dependent)
    all_sc = np.concatenate(t_scores + [f_scores])
    all_sc = _make_distinct(all_sc)
    # keep every unit sorted by its (now final) scores, descending
    pos = 0
    for k in range(len(t_ids) + 1):
        ids, b = (t_ids[k], t_boxes[k]) if k < len(t_ids) else (f_ids, f_boxes)
        sc = all_sc[pos:pos + len(ids)]
        pos += len(ids)
        o = np.argsort(-sc, kind="stable")
        if k < len(t_ids):
            t_ids[k], t_boxes[k], t_scores[k] = ids[o], b[o], sc[o]
        else:
            f_ids, f_boxes, f_scores = ids[o], b[o], sc[o]
    tid = np.concatenate(t_ids) if t_ids else np.zeros(0, np.int64)
    tiles = (protos[tid], np.concatenate(t_boxes).astype(np.float32), np.concatenate(t_scores).astype(np.float32), classes[tid],
             np.asarray(t_off, np.int64))
    full = (protos[f_ids], f_boxes.astype(np.float32), f_scores.astype(np.float32), classes[f_ids], np.array([0, len(f_ids)], np.int64))
    return dict(full=full, tiles=tiles, tile_xy=np.asarray(origins, np.int32).reshape(-1, 2), hw=(h, w), n_particles=n_particles)


def ensemble_multiscale_heads(seed0, n_images, h, w, n_particles=100, scales=(0.7, 1.0, 1.5), n_models=2, cap=100):
    """Config 4: per image one particle set; model m sees a jittered copy of it (box jitter +-1.5 px, score jitter, 10 % of the
    particles dropped) and every scale s the same detections in the frame int(h * s) x int(w * s).
    Returns {scale: [(probs, boxes, scores, classes, unit_off) per model]}, unit = image."""
    out = {float(s): [[[], [], [], [], [0]] for _ in range(n_models)] for s in scales}
    for i in range(n_images):
        rng = np.random.default_rng(seed0 + i)
        polys = particle_field(rng, n_particles, h, w)
        protos = np.zeros((n_particles, MASK_SIDE, MASK_SIDE), np.float32)
        pbox = np.zeros((n_particles, 4), np.float32)
        for k, p in enumerate(polys):
            protos[k], pbox[k] = head_from_poly(rng, p)
        base = rng.uniform(0.3, 0.95, n_particles)
        classes = (rng.random(n_particles) < 0.5).astype(np.int32)
        for m in range(n_models):
            keep = np.nonzero(rng.random(n_particles) >= 0.1)[0]
            jit = rng.uniform(-1.5, 1.5, (len(keep), 4)).astype(np.float32)
            for s in scales:
                sh, sw = int(h * s), int(w * s)
                b = (pbox[keep] + jit) * np.array([sw / w, sh / h, sw / w, sh / h], np.float32)
                sc = _make_distinct((base[keep] + rng.uniform(-0.05, 0.05, len(keep))).astype(np.float32))
                o = np.argsort(-sc, kind="stable")[:cap]
                rec = out[float(s)][m]
                rec[0].append(protos[keep][o]); rec[1].append(b[o].astype(np.float32)); rec[2].append(sc[o]); rec[3].append(classes[keep][o])
                rec[4].append(rec[4][-1] + len(o))
    res = {}
    for s, per_model in out.items():
        res[s] = [(np.concatenate(r[0]), np.concatenate(r[1]), np.concatenate(r[2]).astype(np.float32), np.concatenate(r[3]),
                   np.asarray(r[4], np.int64)) for r in per_model]
    return res


def scalebar_strips(seed, B, rh=92, W=1024, x0=512):
    """B info strips [B, rh, W, 3] (BGR uint8) of SEM frames — the rows a scale-bar ROI covers (row f3 bench / tests): dark band with
    detector noise, one to three white bars, a caption and a few stray annotation lines right of x0; micrograph texture left of it."""
    import cv2
    rng = np.random.default_rng(seed)
    out = np.empty((B, rh, W, 3), np.uint8)
    for b in range(B):
        g = np.clip(20 + rng.integers(-4, 5, (rh, W)), 0, 255).astype(np.uint8)
        tex = cv2.resize(rng.integers(30, 200, (rh // 6 + 1, x0 // 6 + 1), dtype=np.uint8), (x0, rh), interpolation=cv2.INTER_CUBIC)
        g[:, :x0] = tex
        for _ in range(int(rng.integers(1, 4))):
            bx, by = x0 + int(rng.integers(20, (W - x0) // 2)), int(rng.integers(12, rh - 30))
            g[by:by + int(rng.integers(3, 6)), bx:bx + int(rng.integers(40, (W - x0) // 2 - 30))] = 255
        cv2.putText(g, f"{int(rng.integers(1, 900))} nm", (x0 + int(rng.integers(30, 200)), rh - 12), cv2.FONT_HERSHEY_SIMPLEX, 0.5, 255, 1)
        for _ in range(int(rng.integers(0, 4))):
            cv2.line(g, (x0 + int(rng.integers(0, W - x0)), int(rng.integers(0, rh))), (x0 + int(rng.integers(0, W - x0)), int(rng.integers(0, rh))),
                     int(rng.integers(120, 256)), int(rng.integers(1, 3)))
        out[b] = g[:, :, None]
    return out

