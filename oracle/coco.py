"""Oracle: coco_instances.json, COCO instance JSON with compressed RLE (numpy / Python; test infrastructure only).

A DEFINITION, not a restatement of the reference: the reference writes no such file.  The counts strings restate pycocotools'
common/maskApi.c, which is not a dependency of the project (nothing here has been checked against pycocotools itself):

  rle_encode      rleEncode: column-major (Fortran order) counts of one H x W mask, starting with the background count (0 when
                  pixel 0 is set); the last run is always emitted, so an empty mask is [H*W] and a full one [0, H*W].
  rle_to_string   rleToString: count i, for i > 2 its difference to count i - 2, in 5-bit groups, least significant first; a group
                  gets 0x20 when more follow; the loop stops when the rest is 0, or -1 for a group with 0x10; each group is
                  the character 48 + group.
  rle_fr_string   rleFrString: the inverse, sign-extending each value from bit 0x10 of its last group.

The file (``coco_file``) is ``json.dumps(d)`` with default separators and ensure_ascii for

  {"images": [{"id": j + 1, "file_name": name, "height": H, "width": W} for every image of the run, in run order],
   "annotations": [one per instance of an image's final set (a line of R50_flip_results.csv), ids 1, 2, ... over the file],
   "categories": [{"id": k, "name": thing_classes[k]}] + [{"id": c, "name": f"class_{c}"} for other classes that occur, ascending]}

with annotation {"id", "image_id", "category_id": the Class of measurements_results.csv (no shift), "segmentation": {"size":
[H, W], "counts"}, "area": popcount, "bbox": [x_min, y_min, x_max - x_min + 1, y_max - y_min + 1] as floats ([0.0] * 4 for an
empty mask), "iscrowd": 0, "score": float(score)}.  The bbox is the tight box of the pixels: pycocotools' toBbox widens it to the
full height when a run wraps from row H-1 of one column into the next, this definition does not.
"""
import json

import numpy as np

OK, BAD_CHAR, OPEN_VALUE, RANGE, SUM = range(5)
MAX_CHARS = 7


def rle_encode(mask):
    """maskApi.c rleEncode of one H x W mask (non-zero = set) -> list of int counts."""
    flat = np.asarray(mask).astype(bool).ravel(order="F")
    edges = np.flatnonzero(flat[1:] != flat[:-1]) + 1
    bounds = np.concatenate([[0], edges, [flat.size]])
    counts = np.diff(bounds).tolist()
    return [0] + counts if flat.size and flat[0] else counts


def counts_from_runs(runs, H, W):
    """The counts of a mask from its K6 runs ((start, length) pairs, 1-indexed, column-major, maximal)."""
    out, end = [], 0
    for s, n in np.asarray(runs, np.int64).reshape(-1, 2).tolist():
        out += [s - 1 - end, n]
        end = s - 1 + n
    if end < H * W or not out:
        out.append(H * W - end)
    return out


def rle_to_string(counts):
    """maskApi.c rleToString."""
    s = []
    for i, c in enumerate(counts):
        x = int(c) - (int(counts[i - 2]) if i > 2 else 0)
        more = True
        while more:
            g = x & 0x1f
            x >>= 5
            more = x != -1 if g & 0x10 else x != 0
            if more:
                g |= 0x20
            s.append(chr(48 + g))
    return "".join(s)


def rle_fr_string(s):
    """maskApi.c rleFrString (for a well-formed string) -> list of counts."""
    cnts, p = [], 0
    while p < len(s):
        x, k, more = 0, 0, True
        while more:
            c = ord(s[p]) - 48
            x |= (c & 0x1f) << (5 * k)
            more = bool(c & 0x20)
            p += 1
            k += 1
            if not more and c & 0x10:
                x |= -1 << (5 * k)
        if len(cnts) > 2:
            x += cnts[-2]
        cnts.append(x)
    return cnts


def counts_status(s, H, W):
    """The status the decoder reports for counts string s of an H x W mask: the first error in string order of a character outside
    '0'..'o' (BAD_CHAR), a value of more than 7 characters or a count outside [0, 2^31 - 1] (RANGE); then a string that ends inside
    a value (OPEN_VALUE) and counts that do not add up to H * W (SUM)."""
    cnts, start = [], 0
    for p, ch in enumerate(s):
        c = ord(ch)
        if not 48 <= c <= 111:
            return BAD_CHAR
        if (c - 48) & 0x20:
            continue
        if p - start + 1 > MAX_CHARS:
            return RANGE
        v = rle_fr_string(s[start:p + 1])[0] + (cnts[-2] if len(cnts) > 2 else 0)
        if not 0 <= v <= 2 ** 31 - 1:
            return RANGE
        cnts.append(v)
        start = p + 1
    if start != len(s):
        return OPEN_VALUE
    return OK if sum(cnts) == H * W else SUM


def runs_from_counts(counts):
    """(start, length) runs (1-indexed) of the non-empty foreground counts."""
    out, pos = [], 0
    for i, c in enumerate(counts):
        if i & 1 and c > 0:
            out.append((pos + 1, c))
        pos += c
    return out


def mask_bbox(mask):
    ys, xs = np.nonzero(mask)
    if not len(ys):
        return [0.0, 0.0, 0.0, 0.0]
    return [float(xs.min()), float(ys.min()), float(xs.max() - xs.min() + 1), float(ys.max() - ys.min() + 1)]


def annotation(ann_id, image_id, category_id, mask, score):
    H, W = mask.shape
    return {"id": ann_id, "image_id": image_id, "category_id": int(category_id),
            "segmentation": {"size": [H, W], "counts": rle_to_string(rle_encode(mask))},
            "area": int(np.count_nonzero(mask)), "bbox": mask_bbox(mask), "iscrowd": 0, "score": float(score)}


def coco_file(images, thing_classes):
    """images: [(file name, H, W, [(mask, class, score), ...]), ...] in run order -> the bytes of coco_instances.json."""
    imgs, anns, seen = [], [], set()
    for j, (name, H, W, insts) in enumerate(images):
        imgs.append({"id": j + 1, "file_name": name, "height": H, "width": W})
        for mask, cls, score in insts:
            anns.append(annotation(len(anns) + 1, j + 1, cls, mask, score))
            seen.add(int(cls))
    cats = [{"id": k, "name": n} for k, n in enumerate(thing_classes)]
    cats += [{"id": c, "name": f"class_{c}"} for c in sorted(seen) if c >= len(thing_classes)]
    return json.dumps({"images": imgs, "annotations": anns, "categories": cats}).encode()
